// Training-step kernels either side of the two hot paths (SURVEY.md section 8f, rows N2-N4):
//   * OHEM cross-entropy        -- OhemCELoss2D, seg18/utils/losses.py:16-40
//   * key-encoder momentum (EMA) update + bf16 key-weight shadow -- PixPro._momentum_update_key_encoder,
//     PixPro_swin_v5.py:258-289
//   * LARS-scaled SGD step + bf16 weight shadow -- contrast/lars.py:109-152 (+ torch.optim.SGD it wraps)
//   * Adam step + bf16 weight shadow -- torch.optim.Adam of seg18/train_swin.py
// All three are HBM-bound element streams: 16-byte accesses, grids sized from the SM count or the
// element count, no host synchronisation (every data-dependent decision is taken on the device).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <initializer_list>

#include "common.cuh"
#include "host_util.h"
#include "kernels.h"

namespace stswin {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------
// OHEM cross-entropy
// ------------------------------------------------------------------------------------------------
constexpr int kBins = 2048;

struct OhemWs {                     // device workspace, zeroed at the start of every forward
  double sum_gt;                    // sum / count of per-pixel losses above the threshold
  unsigned long long cnt_gt;
  double sum_sel;                   // top-n_min case: sum / count of losses above the n_min-th largest value
  unsigned long long cnt_sel;
  unsigned int done;                // blocks finished in the final kernel
  unsigned int pad;
  unsigned int hist[3][kBins];      // radix-select histograms: key bits 31..21, 20..10, 9..0
};

template <typename T, int VEC>
struct Vec;
template <>
struct Vec<float, 4> {
  static __device__ __forceinline__ void load(const float* p, float (&x)[4]) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&x)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(x[0], x[1], x[2], x[3]);
  }
};
template <>
struct Vec<float, 1> {
  static __device__ __forceinline__ void load(const float* p, float (&x)[1]) { x[0] = __ldg(p); }
  static __device__ __forceinline__ void store(float* p, const float (&x)[1]) { *p = x[0]; }
};
template <>
struct Vec<__nv_bfloat16, 4> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&x)[4]) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    x[0] = __uint_as_float(v.x << 16); x[1] = __uint_as_float(v.x & 0xffff0000u);
    x[2] = __uint_as_float(v.y << 16); x[3] = __uint_as_float(v.y & 0xffff0000u);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&x)[4]) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(x[0], x[1]), b = __floats2bfloat162_rn(x[2], x[3]);
    uint2 v;
    v.x = *reinterpret_cast<const uint32_t*>(&a);
    v.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = v;
  }
};
template <>
struct Vec<__nv_bfloat16, 1> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&x)[1]) { x[0] = __bfloat162float(*p); }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&x)[1]) { *p = __float2bfloat16_rn(x[0]); }
};

template <int VEC>
__device__ __forceinline__ void load_labels(const int64_t* p, long long (&lab)[VEC]) {
  if constexpr (VEC == 4) {
    const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(p));
    const longlong2 b = __ldg(reinterpret_cast<const longlong2*>(p) + 1);
    lab[0] = a.x; lab[1] = a.y; lab[2] = b.x; lab[3] = b.y;
  } else {
    lab[0] = __ldg(p);
  }
}

// log-sum-exp over the K classes of VEC neighbouring pixels in one pass over the logits: classes go four at a
// time (four independent loads in flight per thread, one rescale of the running sum per group);
// xl = the logit of the pixel's own label
template <typename T, int VEC>
__device__ __forceinline__ void pixel_lse(const T* base, int K, long HW, const long long (&lab)[VEC], float (&m)[VEC],
                                          float (&s)[VEC], float (&xl)[VEC]) {
#pragma unroll
  for (int v = 0; v < VEC; ++v) { m[v] = -INFINITY; s[v] = 0.f; xl[v] = 0.f; }
  int k = 0;
  for (; k + 4 <= K; k += 4) {
    float x[4][VEC];
#pragma unroll
    for (int c = 0; c < 4; ++c) Vec<T, VEC>::load(base + (long)(k + c) * HW, x[c]);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const float mn = fmaxf(fmaxf(m[v], fmaxf(x[0][v], x[1][v])), fmaxf(x[2][v], x[3][v]));
      s[v] = s[v] * __expf(m[v] - mn) + ((__expf(x[0][v] - mn) + __expf(x[1][v] - mn)) + (__expf(x[2][v] - mn) + __expf(x[3][v] - mn)));
      m[v] = mn;
      const long long rel = lab[v] - k;
      if (rel == 0) xl[v] = x[0][v];
      if (rel == 1) xl[v] = x[1][v];
      if (rel == 2) xl[v] = x[2][v];
      if (rel == 3) xl[v] = x[3][v];
    }
  }
  for (; k < K; ++k) {
    float x[VEC];
    Vec<T, VEC>::load(base + (long)k * HW, x);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const float mn = fmaxf(m[v], x[v]);
      s[v] = s[v] * __expf(m[v] - mn) + __expf(x[v] - mn);
      m[v] = mn;
      if (lab[v] == k) xl[v] = x[v];
    }
  }
}

// per-pixel cross-entropy (nn.CrossEntropyLoss(reduction='none', ignore_index), losses.py:23,33) + the count and
// sum of the losses above the OHEM threshold (losses.py:36-37)
template <typename T, int VEC>
__global__ void __launch_bounds__(kThreads) ohem_px_kernel(const T* __restrict__ logits, const int64_t* __restrict__ labels,
                                                           int B, int K, long HW, int ignore, float thresh,
                                                           float* __restrict__ loss_px, OhemWs* ws) {
  const long gpi = HW / VEC, total = (long)B * gpi;
  float lsum = 0.f;
  unsigned int lcnt = 0;
  for (long g = (long)blockIdx.x * kThreads + threadIdx.x; g < total; g += (long)gridDim.x * kThreads) {
    const long b = g / gpi, p = (g - b * gpi) * VEC;
    long long lab[VEC];
    load_labels<VEC>(labels + b * HW + p, lab);
    float m[VEC], s[VEC], xl[VEC], loss[VEC];
    pixel_lse<T, VEC>(logits + (b * K) * HW + p, K, HW, lab, m, s, xl);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      loss[v] = lab[v] == ignore ? 0.f : (m[v] - xl[v]) + logf(s[v]);      // >= 0 by construction
      if (loss[v] > thresh) { lsum += loss[v]; ++lcnt; }
    }
    Vec<float, VEC>::store(loss_px + b * HW + p, loss);
  }
  __shared__ float s_sum[kThreads / 32];
  __shared__ unsigned int s_cnt[kThreads / 32];
  lsum = warp_sum(lsum);
  lcnt = __reduce_add_sync(0xffffffffu, lcnt);
  if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = lsum; s_cnt[threadIdx.x >> 5] = lcnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    unsigned long long c = 0;
    for (int i = 0; i < kThreads / 32; ++i) { t += s_sum[i]; c += s_cnt[i]; }
    if (c != 0) { atomicAdd(&ws->sum_gt, t); atomicAdd(&ws->cnt_gt, c); }
  }
}

// find the bin holding the k-th largest key of a histogram (k is 1-based, counted from the top bin); returns the bin
// and leaves the rank inside that bin in k.  Whole block (suffix sums by warp shuffles); the result is block-uniform.
__device__ int pick_bin(const unsigned int* hist, int bins, unsigned long long& k, unsigned int* s_part, int* s_res,
                        unsigned long long* s_k) {
  const int per = bins / kThreads;              // 8 or 4 bins per thread
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned int h[8], part = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    h[i] = i < per ? hist[threadIdx.x * per + i] : 0u;
    part += h[i];
  }
  unsigned int incl = part;                     // -> sum over the threads at or above this one
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int v = __shfl_down_sync(0xffffffffu, incl, o);
    if (lane + o < 32) incl += v;
  }
  if (lane == 0) s_part[warp] = incl;
  __syncthreads();
  for (int w = warp + 1; w < kThreads / 32; ++w) incl += s_part[w];
  const unsigned long long above = incl - part;
  if (above < k && k <= incl) {                 // exactly one thread: its bins hold the k-th key
    unsigned long long kk = k - above;
    int res = 0;
    bool found = false;
#pragma unroll
    for (int i = 7; i >= 0; --i) {
      if (i < per && !found) {
        if (kk <= h[i] || i == 0) { res = i; found = true; } else kk -= h[i];
      }
    }
    *s_res = threadIdx.x * per + res;
    *s_k = kk;
  }
  __syncthreads();
  k = *s_k;
  const int bin = *s_res;
  __syncthreads();
  return bin;
}

// PASS 0..2: histogram of the next key digit over the losses that match the digits found so far.
// Does nothing when more than n_min losses are above the threshold (the other branch of losses.py:36).
template <int PASS>
__global__ void __launch_bounds__(kThreads) ohem_hist_kernel(const float* __restrict__ loss_px, long M, long n_min, OhemWs* ws) {
  if (ws->cnt_gt > (unsigned long long)n_min) return;
  __shared__ unsigned int s_hist[kBins];
  __shared__ unsigned int s_part[kThreads / 32];
  __shared__ int s_res;
  __shared__ unsigned long long s_k;
  unsigned int prefix = 0;
  unsigned long long k = (unsigned long long)n_min;
  if (PASS >= 1) prefix = pick_bin(ws->hist[0], kBins, k, s_part, &s_res, &s_k);
  if (PASS >= 2) prefix = (prefix << 11) | pick_bin(ws->hist[1], kBins, k, s_part, &s_res, &s_k);
  constexpr int shift = PASS == 0 ? 21 : (PASS == 1 ? 10 : 0);
  constexpr int pshift = PASS == 1 ? 21 : 10;           // where the known prefix starts
  constexpr unsigned int mask = PASS == 2 ? 1023u : 2047u;
  for (int i = threadIdx.x; i < kBins; i += kThreads) s_hist[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  auto count = [&](unsigned int key, bool valid) {
    if (PASS == 0) {
      // the top digit (sign, exponent, two mantissa bits) is shared by most losses: one shared-memory atomic per
      // distinct bin of the warp
      const unsigned int bin = valid ? (key >> shift) & mask : 0xffffffffu;
      const unsigned int peers = __match_any_sync(0xffffffffu, bin);
      if (valid && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], (unsigned int)__popc(peers));
    } else if (valid && (key >> pshift) == prefix) {    // few keys survive the prefix filter
      atomicAdd(&s_hist[(key >> shift) & mask], 1u);
    }
  };
  const long M4 = M >> 2;                               // loss_px is 16-byte aligned (our own buffer)
  const long warp0 = (long)blockIdx.x * kThreads + (threadIdx.x & ~31);
  for (long i0 = warp0; i0 < M4; i0 += (long)gridDim.x * kThreads) {
    const long i = i0 + lane;
    const bool valid = i < M4;
    const float4 v = valid ? __ldg(reinterpret_cast<const float4*>(loss_px) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    count(__float_as_uint(v.x), valid);
    count(__float_as_uint(v.y), valid);
    count(__float_as_uint(v.z), valid);
    count(__float_as_uint(v.w), valid);
  }
  if (blockIdx.x == 0 && threadIdx.x < 32) {            // the last M % 4 losses
    const long i = (M4 << 2) + lane;
    const bool valid = i < M;
    count(valid ? __float_as_uint(loss_px[i]) : 0u, valid);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBins; i += kThreads)
    if (s_hist[i] != 0) atomicAdd(&ws->hist[PASS][i], s_hist[i]);
}

// loss value and the selection rule for the backward: sel = {cut, weight of a loss above cut, weight of a loss
// equal to cut}.  losses.py:36-40: more than n_min losses above thresh -> mean of those; else mean of the n_min largest.
__global__ void __launch_bounds__(kThreads) ohem_final_kernel(const float* __restrict__ loss_px, long M, long n_min, float thresh,
                                                              OhemWs* ws, float* __restrict__ loss, float* __restrict__ sel) {
  if (ws->cnt_gt > (unsigned long long)n_min) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      const double c = (double)ws->cnt_gt;
      *loss = (float)(ws->sum_gt / c);
      sel[0] = thresh; sel[1] = (float)(1.0 / c); sel[2] = 0.f;
    }
    return;
  }
  __shared__ unsigned int s_part[kThreads / 32];
  __shared__ int s_res;
  __shared__ unsigned long long s_k;
  __shared__ float s_sum[kThreads / 32];
  __shared__ unsigned int s_cnt[kThreads / 32];
  unsigned long long k = (unsigned long long)n_min;
  unsigned int key = pick_bin(ws->hist[0], kBins, k, s_part, &s_res, &s_k);
  key = (key << 11) | pick_bin(ws->hist[1], kBins, k, s_part, &s_res, &s_k);
  const int last = pick_bin(ws->hist[2], 1024, k, s_part, &s_res, &s_k);
  key = (key << 10) | last;
  const float cut = __uint_as_float(key);            // the n_min-th largest loss
  float lsum = 0.f;
  unsigned int lcnt = 0;
  const long M4 = M >> 2;
  for (long i = (long)blockIdx.x * kThreads + threadIdx.x; i < M4; i += (long)gridDim.x * kThreads) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(loss_px) + i);
    if (v.x > cut) { lsum += v.x; ++lcnt; }
    if (v.y > cut) { lsum += v.y; ++lcnt; }
    if (v.z > cut) { lsum += v.z; ++lcnt; }
    if (v.w > cut) { lsum += v.w; ++lcnt; }
  }
  if (blockIdx.x == 0 && threadIdx.x < (M & 3)) {
    const float v = loss_px[(M4 << 2) + threadIdx.x];
    if (v > cut) { lsum += v; ++lcnt; }
  }
  lsum = warp_sum(lsum);
  lcnt = __reduce_add_sync(0xffffffffu, lcnt);
  if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = lsum; s_cnt[threadIdx.x >> 5] = lcnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    unsigned long long c = 0;
    for (int i = 0; i < kThreads / 32; ++i) { t += s_sum[i]; c += s_cnt[i]; }
    if (c != 0) { atomicAdd(&ws->sum_sel, t); atomicAdd(&ws->cnt_sel, c); }
    __threadfence();
    if (atomicAdd(&ws->done, 1u) == gridDim.x - 1) {             // last block: every partial sum has landed
      __threadfence();
      const double tot = atomicAdd(&ws->sum_sel, 0.0);
      const unsigned long long above = atomicAdd(&ws->cnt_sel, 0ull);
      const double ties_taken = (double)((unsigned long long)n_min - above);     // of the losses equal to cut
      const double ties = (double)ws->hist[2][last];
      *loss = (float)((tot + ties_taken * (double)cut) / (double)n_min);
      sel[0] = cut; sel[1] = (float)(1.0 / (double)n_min); sel[2] = (float)(ties_taken / ties / (double)n_min);
    }
  }
}

// d logits = weight(pixel) * (softmax - onehot) * d_loss; unselected pixels only write zeros (no logit read)
template <typename T, int VEC>
__global__ void __launch_bounds__(kThreads) ohem_bwd_kernel(const T* __restrict__ logits, const int64_t* __restrict__ labels, int B,
                                                            int K, long HW, int ignore, const float* __restrict__ loss_px,
                                                            const float* __restrict__ sel, const float* __restrict__ d_loss,
                                                            T* __restrict__ d_logits) {
  const float cut = sel[0], dl = *d_loss;
  const float w_above = sel[1] * dl, w_tie = sel[2] * dl;
  const long gpi = HW / VEC, total = (long)B * gpi;
  for (long g = (long)blockIdx.x * kThreads + threadIdx.x; g < total; g += (long)gridDim.x * kThreads) {
    const long b = g / gpi, p = (g - b * gpi) * VEC;
    long long lab[VEC];
    load_labels<VEC>(labels + b * HW + p, lab);
    float lp[VEC], w[VEC];
    Vec<float, VEC>::load(loss_px + b * HW + p, lp);
    bool any = false;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      w[v] = lab[v] == ignore ? 0.f : (lp[v] > cut ? w_above : (lp[v] == cut ? w_tie : 0.f));
      any |= w[v] != 0.f;
    }
    const T* src = logits + (b * K) * HW + p;
    T* dst = d_logits + (b * K) * HW + p;
    if (!any) {
      float z[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) z[v] = 0.f;
      for (int k = 0; k < K; ++k) Vec<T, VEC>::store(dst + (long)k * HW, z);
      continue;
    }
    float m[VEC], s[VEC], xl[VEC];
    pixel_lse<T, VEC>(src, K, HW, lab, m, s, xl);
#pragma unroll
    for (int v = 0; v < VEC; ++v) m[v] += logf(s[v]);       // log-sum-exp
    for (int k = 0; k < K; ++k) {
      float x[VEC], d[VEC];
      Vec<T, VEC>::load(src + (long)k * HW, x);             // second read of the line: L1 / L2
#pragma unroll
      for (int v = 0; v < VEC; ++v) d[v] = w[v] * (__expf(x[v] - m[v]) - (lab[v] == k ? 1.f : 0.f));
      Vec<T, VEC>::store(dst + (long)k * HW, d);
    }
  }
}

int stream_grid(long work_items) {
  const long want = (work_items + kThreads - 1) / kThreads;
  const long cap = (long)num_sms() * 8;
  return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

// ------------------------------------------------------------------------------------------------
// multi-tensor element streams (EMA, LARS, Adam, SGD, gather): up to MT_MAX tensors per launch, described in the kernel
// parameters (no device-side table to upload, safe under stream capture); a block owns MT_CHUNK elements of one tensor
// ------------------------------------------------------------------------------------------------
constexpr int MT_MAX = 48;
constexpr int MT_CHUNK = kThreads * 64;

struct MtTable {
  void* ptr[4][MT_MAX];              // up to four tensors per entry, in the order each kernel names them
  __nv_bfloat16* shadow[MT_MAX];     // bf16 shadow of the updated weight ptr[0] (null: none)
  long numel[MT_MAX];
  int block_start[MT_MAX + 1];
  unsigned char flag[MT_MAX];        // the tensor's first step with momentum: buf = g
  int n;
};

// the block's tensor (binary search over block_start) and its element range [base, end)
struct MtBlock {
  int ti;
  long base, end;
};
__device__ __forceinline__ MtBlock mt_block(const MtTable& t) {
  int lo = 0, hi = t.n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (t.block_start[mid] <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const long base = (long)(blockIdx.x - t.block_start[lo]) * MT_CHUNK;
  return {lo, base, base + MT_CHUNK < t.numel[lo] ? base + MT_CHUNK : t.numel[lo]};
}

// gradients: fp32 (p.grad) or bf16 (the buckets of a bf16 all-reduce, widened exactly)
__device__ __forceinline__ float4 load4(const float* g) { return *reinterpret_cast<const float4*>(g); }
__device__ __forceinline__ float4 load4(const __nv_bfloat16* g) {
  const uint2 raw = *reinterpret_cast<const uint2*>(g);
  const float2 a = unpack_bf16(raw.x), b = unpack_bf16(raw.y);
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float load1(const float* g) { return *g; }
__device__ __forceinline__ float load1(const __nv_bfloat16* g) { return __bfloat162float(*g); }
// fp32 stores, and bf16 stores rounded to nearest (the weight shadows, the bf16 gradient bucket)
__device__ __forceinline__ void store4(float* d, float4 v) { *reinterpret_cast<float4*>(d) = v; }
__device__ __forceinline__ void store4(__nv_bfloat16* d, float4 v) {
  *reinterpret_cast<uint2*>(d) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
}
__device__ __forceinline__ void store1(float* d, float v) { *d = v; }
__device__ __forceinline__ void store1(__nv_bfloat16* d, float v) { *d = __float2bfloat16_rn(v); }
template <typename G>
constexpr uintptr_t vec_align_mask() { return sizeof(G) == 4 ? 15 : 7; }

// The element loop of the streams but the EMA (ema_kernel) over one block's range: when the fp32 pointers (or-ed into
// f32_ptrs) are 16-byte aligned, g is aligned for 4-element accesses of G and the shadow sh (null: none) on 8 bytes,
// vec(i) updates the four elements [i, i + 4) of each group below the last multiple of four of the range, U groups per
// thread in flight, and one(i) the remaining elements; otherwise one(i) updates every element.  LARS rounds
// differently on the two paths (lars_sgd_kernel), so this split is part of its result.
template <int U, typename G, class Vec, class One>
__device__ __forceinline__ void mt_stream(const MtBlock& b, uintptr_t f32_ptrs, const G* g, const __nv_bfloat16* sh,
                                          Vec&& vec, One&& one) {
  long i = b.base + threadIdx.x;
  if (((f32_ptrs & 15) | ((uintptr_t)g & vec_align_mask<G>()) | ((uintptr_t)sh & 7)) == 0) {
    const long end4 = b.base + ((b.end - b.base) & ~3L);
#pragma unroll U
    for (i = b.base + threadIdx.x * 4; i < end4; i += kThreads * 4) vec(i);
    i = end4 + threadIdx.x;
  }
  for (; i < b.end; i += kThreads) one(i);
}

// param_k = param_k * m + param_q * (1 - m), rounded like the three eager ops of PixPro_swin_v5.py:266-267; (m, 1 - m)
// from m_dev[0..1] when m_dev is non-null (a schedule under graph replay); shadow = bf16_rn(param_k).  8 blocks per SM:
// without the bound the shadow store takes the kernel to 38 registers and 6 blocks.
__global__ void __launch_bounds__(kThreads, 8) ema_kernel(const __grid_constant__ MtTable t, float m, float om,
                                                       const float* __restrict__ m_dev) {
  if (m_dev != nullptr) { m = __ldg(m_dev); om = __ldg(m_dev + 1); }
  const MtBlock b = mt_block(t);
  float* __restrict__ k = static_cast<float*>(t.ptr[0][b.ti]);
  const float* __restrict__ q = static_cast<const float*>(t.ptr[1][b.ti]);
  __nv_bfloat16* __restrict__ sh = t.shadow[b.ti];
  auto ema = [&](float kv, float qv) { return __fadd_rn(__fmul_rn(kv, m), __fmul_rn(qv, om)); };
  // its own loop rather than mt_stream: with all eight 16-byte loads of a thread issued before any store, the EMA
  // measures about 2 % faster on the B200 than the shared loop, whose compiled body loads one group at a time
  long i = b.base;
  if ((((uintptr_t)k | (uintptr_t)q) & 15) == 0 && (((uintptr_t)sh) & 7) == 0) {
    constexpr int U = 4;
    for (; i + U * kThreads * 4 <= b.end; i += U * kThreads * 4) {
      float4 kv[U], qv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long j = i + (long)(u * kThreads + threadIdx.x) * 4;
        kv[u] = *reinterpret_cast<const float4*>(k + j);
        qv[u] = __ldg(reinterpret_cast<const float4*>(q + j));
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long j = i + (long)(u * kThreads + threadIdx.x) * 4;
        const float4 r = make_float4(ema(kv[u].x, qv[u].x), ema(kv[u].y, qv[u].y), ema(kv[u].z, qv[u].z), ema(kv[u].w, qv[u].w));
        store4(k + j, r);
        if (sh != nullptr) store4(sh + j, r);
      }
    }
  }
  for (long j = i + threadIdx.x; j < b.end; j += kThreads) {
    const float v = ema(k[j], q[j]);
    k[j] = v;
    if (sh != nullptr) store1(sh + j, v);
  }
}

// sum p^2 and sum (g + wd p)^2 per tensor (lars.py:121-127), fp64 accumulators norms[2*t], norms[2*t+1].  Every
// rounding is spelled out (the contraction the fp32-only kernel had from nvcc), so it does not depend on the
// gradient type or on the compiler's choices.
__device__ __forceinline__ float sumsq4(float a, float b, float c, float d) {
  return __fmaf_rn(d, d, __fmaf_rn(c, c, __fmaf_rn(a, a, __fmul_rn(b, b))));
}

template <typename G>
__global__ void __launch_bounds__(kThreads) lars_norm_kernel(const __grid_constant__ MtTable t, float wd, double* __restrict__ norms) {
  const MtBlock b = mt_block(t);
  const float* __restrict__ p = static_cast<const float*>(t.ptr[0][b.ti]);
  const G* __restrict__ g = static_cast<const G*>(t.ptr[1][b.ti]);
  float sp = 0.f, sg = 0.f;
  mt_stream<4>(b, (uintptr_t)p, g, nullptr,
      [&](long i) {
        const float4 pv = __ldg(reinterpret_cast<const float4*>(p + i));
        const float4 gv = load4(g + i);
        const float g0 = __fmaf_rn(wd, pv.x, gv.x), g1 = __fmaf_rn(wd, pv.y, gv.y), g2 = __fmaf_rn(wd, pv.z, gv.z),
                    g3 = __fmaf_rn(wd, pv.w, gv.w);
        sp = __fadd_rn(sumsq4(pv.x, pv.y, pv.z, pv.w), sp);
        sg = __fadd_rn(sumsq4(g0, g1, g2, g3), sg);
      },
      [&](long i) {
        const float pv = p[i], gg = __fmaf_rn(wd, pv, load1(g + i));
        sp = __fmaf_rn(pv, pv, sp); sg = __fmaf_rn(gg, gg, sg);
      });
  __shared__ float s_p[kThreads / 32], s_g[kThreads / 32];
  sp = warp_sum(sp); sg = warp_sum(sg);
  if ((threadIdx.x & 31) == 0) { s_p[threadIdx.x >> 5] = sp; s_g[threadIdx.x >> 5] = sg; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, c = 0.0;
    for (int i = 0; i < kThreads / 32; ++i) { a += s_p[i]; c += s_g[i]; }
    atomicAdd(&norms[2 * b.ti], a);
    atomicAdd(&norms[2 * b.ti + 1], c);
  }
}

struct LarsHp {
  float lr, momentum, dampening, wd, trust, eps;
  int nesterov, lars;
  int store_grad;                    // fp32 gradients only: grad <- the decayed / scaled gradient (the p.grad contract)
  const float* lr_dev;               // device scalar read instead of lr when non-null (a schedule under graph replay)
};

// g = grad + wd p; g *= trust |p| / (|g| + eps) (LARS group); grad = g (store_grad); buf = momentum buf + (1 - dampening) g
// (buf = g on a tensor's first step); p -= lr * buf; shadow = bf16_rn(p)
// (lars.py:109-135 then torch.optim.SGD with wd 0, :137-152).  Each rounding is spelled out as nvcc contracted the
// fp32-only kernel: fma(wd, p, grad), one product by the LARS factor, fma(momentum, buf, g) for nesterov,
// fma(-lr, d, p), and the momentum update as fma(1 - dampening, g, momentum * buf) on the 16-byte path but
// fma(momentum, buf, (1 - dampening) * g) on the scalar tails and the unaligned path, so that every element keeps
// the value that kernel gave it.
template <typename G>
__global__ void __launch_bounds__(kThreads) lars_sgd_kernel(const __grid_constant__ MtTable t, const LarsHp a,
                                                            const double* __restrict__ norms) {
  const MtBlock b = mt_block(t);
  float* __restrict__ p = static_cast<float*>(t.ptr[0][b.ti]);
  G* __restrict__ g = static_cast<G*>(t.ptr[1][b.ti]);
  float* __restrict__ buf = static_cast<float*>(t.ptr[2][b.ti]);
  __nv_bfloat16* __restrict__ sh = t.shadow[b.ti];
  const bool first = t.flag[b.ti] != 0;
  const float neg_lr = -(a.lr_dev != nullptr ? __ldg(a.lr_dev) : a.lr);
  const float one_minus_damp = __fsub_rn(1.f, a.dampening);
  float alr = 1.f;
  if (a.lars) {
    const float pn = (float)sqrt(norms[2 * b.ti]), gn = (float)sqrt(norms[2 * b.ti + 1]);
    if (pn > 0.f && gn > 0.f) alr = __fdiv_rn(__fmul_rn(a.trust, pn), __fadd_rn(gn, a.eps));
  }
  const bool has_buf = a.momentum != 0.f;
  constexpr bool kF32 = sizeof(G) == 4;
  const bool store_grad = kF32 && a.store_grad;
  auto one = [&](float pv, float gv, float& bv, float& g_out, bool vec) -> float {
    float gg = a.wd > 0.f ? __fmaf_rn(a.wd, pv, gv) : gv;
    if (a.lars) gg = __fmul_rn(gg, alr);
    g_out = gg;
    float d = gg;
    if (has_buf) {
      bv = first ? gg
           : vec ? __fmaf_rn(one_minus_damp, gg, __fmul_rn(a.momentum, bv))
                 : __fmaf_rn(a.momentum, bv, __fmul_rn(one_minus_damp, gg));
      d = a.nesterov ? __fmaf_rn(a.momentum, bv, gg) : bv;
    }
    return __fmaf_rn(neg_lr, d, pv);
  };
  mt_stream<2>(b, (uintptr_t)p | (uintptr_t)buf, g, sh,
      [&](long i) {
        float4 pv = *reinterpret_cast<const float4*>(p + i);
        float4 gv = load4(g + i);
        float4 bv = (has_buf && !first) ? *reinterpret_cast<const float4*>(buf + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        pv.x = one(pv.x, gv.x, bv.x, gv.x, true);
        pv.y = one(pv.y, gv.y, bv.y, gv.y, true);
        pv.z = one(pv.z, gv.z, bv.z, gv.z, true);
        pv.w = one(pv.w, gv.w, bv.w, gv.w, true);
        store4(p + i, pv);
        if constexpr (kF32) {
          if (store_grad) store4(g + i, gv);
        }
        if (has_buf) store4(buf + i, bv);
        if (sh != nullptr) store4(sh + i, pv);
      },
      [&](long i) {
        float bv = (has_buf && !first) ? buf[i] : 0.f, gv;
        const float pv = one(p[i], load1(g + i), bv, gv, false);
        p[i] = pv;
        if constexpr (kF32) {
          if (store_grad) g[i] = gv;
        }
        if (has_buf) buf[i] = bv;
        if (sh != nullptr) store1(sh + i, pv);
      });
}
// the whole argument block of the largest of these launches stays within the 4 KB kernel-parameter limit
static_assert(sizeof(MtTable) + sizeof(LarsHp) + sizeof(double*) <= 4096, "lars_sgd_kernel parameters exceed 4 KB");

// ------------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam semantics, no amsgrad) as a multi-tensor stream that also emits the bf16 shadow of the
// weights the Swin kernels consume: one pass instead of the optimizer's own pass plus one cast kernel per weight
// and step.  The step count lives on the device (CUDA-graph capturable).
struct AdamHp {
  float lr, beta1, beta2, eps, wd, grad_scale;
  const float* step;                 // device scalar: the step being taken (>= 1)
};

__global__ void adam_tick_kernel(float* step) { *step += 1.0f; }

// p, g, m, v in ptr[0..3].  Each rounding is spelled out as nvcc contracted the kernel before it was a template on
// the gradient type: g = rn(grad * grad_scale), then fma(wd, p, g) when wd != 0; m = fma(rn(g - m), rn(1 - beta1), m);
// v = fma(v, beta2, rn(rn(rn(1 - beta2) * g) * g)); denom = fma(sqrt_rn(v), rsqrtf(bc2), eps);
// p = fma(-step_size, rn(m / denom), p) with step_size = rn(lr / rn(1 - powf(beta1, t))), bc2 = rn(1 - powf(beta2, t)).
template <typename G>
__global__ void __launch_bounds__(kThreads) adam_kernel(const __grid_constant__ MtTable t, const AdamHp a) {
  pdl_wait();
  pdl_launch_dependents();
  const MtBlock b = mt_block(t);
  float* __restrict__ p = static_cast<float*>(t.ptr[0][b.ti]);
  const G* __restrict__ g = static_cast<const G*>(t.ptr[1][b.ti]);
  float* __restrict__ m = static_cast<float*>(t.ptr[2][b.ti]);
  float* __restrict__ v = static_cast<float*>(t.ptr[3][b.ti]);
  __nv_bfloat16* __restrict__ sh = t.shadow[b.ti];
  const float stepf = __ldg(a.step);
  const float bc1 = __fsub_rn(1.0f, powf(a.beta1, stepf)), bc2 = __fsub_rn(1.0f, powf(a.beta2, stepf));
  const float neg_step_size = -__fdiv_rn(a.lr, bc1), inv_sqrt_bc2 = rsqrtf(bc2);
  const float one_minus_b1 = __fsub_rn(1.0f, a.beta1), one_minus_b2 = __fsub_rn(1.0f, a.beta2);
  auto one = [&](float pv, float gv, float& mv, float& vv) -> float {
    gv = __fmul_rn(gv, a.grad_scale);
    if (a.wd != 0.f) gv = __fmaf_rn(a.wd, pv, gv);
    mv = __fmaf_rn(__fsub_rn(gv, mv), one_minus_b1, mv);                 // lerp(m, g, 1 - beta1)
    vv = __fmaf_rn(vv, a.beta2, __fmul_rn(__fmul_rn(one_minus_b2, gv), gv));
    const float denom = __fmaf_rn(__fsqrt_rn(vv), inv_sqrt_bc2, a.eps);
    return __fmaf_rn(neg_step_size, __fdiv_rn(mv, denom), pv);
  };
  mt_stream<2>(b, (uintptr_t)p | (uintptr_t)m | (uintptr_t)v, g, sh,
      [&](long i) {
        float4 pv = *reinterpret_cast<const float4*>(p + i);
        float4 mv = *reinterpret_cast<const float4*>(m + i);
        float4 vv = *reinterpret_cast<const float4*>(v + i);
        const float4 gv = load4(g + i);
        pv.x = one(pv.x, gv.x, mv.x, vv.x);
        pv.y = one(pv.y, gv.y, mv.y, vv.y);
        pv.z = one(pv.z, gv.z, mv.z, vv.z);
        pv.w = one(pv.w, gv.w, mv.w, vv.w);
        store4(p + i, pv);
        store4(m + i, mv);
        store4(v + i, vv);
        if (sh != nullptr) store4(sh + i, pv);
      },
      [&](long i) {
        float mv = m[i], vv = v[i];
        const float pv = one(p[i], load1(g + i), mv, vv);
        p[i] = pv; m[i] = mv; v[i] = vv;
        if (sh != nullptr) store1(sh + i, pv);
      });
}

// ------------------------------------------------------------------------------------------------
// torch.optim.SGD (momentum, dampening, nesterov, weight decay, maximize) as a multi-tensor stream that also emits the
// bf16 shadow of the weights.  Each operation is rounded where the eager single-tensor step of torch rounds it --
// add(alpha=) is one fma of alpha * other onto self, mul_ one product, every eager op its own rounding -- so the result
// is bit-identical with it and does not depend on the compiler's contraction choices.  p.grad is not written.
struct SgdHp {
  float lr, momentum, one_minus_dampening, wd, grad_scale;
  int nesterov, maximize;
  const float* lr_dev;               // device scalar read instead of lr when non-null (a schedule under graph replay)
};

// p, g, momentum buffer in ptr[0..2] (buffers all null when momentum == 0)
template <typename G>
__global__ void __launch_bounds__(kThreads) sgd_kernel(const __grid_constant__ MtTable t, const SgdHp a) {
  pdl_wait();
  pdl_launch_dependents();
  const MtBlock b = mt_block(t);
  float* __restrict__ p = static_cast<float*>(t.ptr[0][b.ti]);
  const G* __restrict__ g = static_cast<const G*>(t.ptr[1][b.ti]);
  float* __restrict__ buf = static_cast<float*>(t.ptr[2][b.ti]);
  __nv_bfloat16* __restrict__ sh = t.shadow[b.ti];
  const bool has_buf = a.momentum != 0.f, first = t.flag[b.ti] != 0;
  const float neg_lr = -(a.lr_dev != nullptr ? __ldg(a.lr_dev) : a.lr);
  auto one = [&](float pv, float gv, float& bv) -> float {
    float gg = __fmul_rn(gv, a.grad_scale);
    if (a.maximize) gg = -gg;
    if (a.wd != 0.f) gg = __fmaf_rn(a.wd, pv, gg);                                    // grad.add(param, alpha=wd)
    float d = gg;
    if (has_buf) {
      bv = first ? gg : __fmaf_rn(a.one_minus_dampening, gg, __fmul_rn(bv, a.momentum));  // buf.mul_(m).add_(g, alpha=1-damp)
      d = a.nesterov ? __fmaf_rn(a.momentum, bv, gg) : bv;                            // grad.add(buf, alpha=m)
    }
    return __fmaf_rn(neg_lr, d, pv);                                                  // param.add_(d, alpha=-lr)
  };
  mt_stream<2>(b, (uintptr_t)p | (uintptr_t)buf, g, sh,
      [&](long i) {
        float4 pv = *reinterpret_cast<const float4*>(p + i);
        const float4 gv = load4(g + i);
        float4 bv = (has_buf && !first) ? *reinterpret_cast<const float4*>(buf + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        pv.x = one(pv.x, gv.x, bv.x);
        pv.y = one(pv.y, gv.y, bv.y);
        pv.z = one(pv.z, gv.z, bv.z);
        pv.w = one(pv.w, gv.w, bv.w);
        store4(p + i, pv);
        if (has_buf) store4(buf + i, bv);
        if (sh != nullptr) store4(sh + i, pv);
      },
      [&](long i) {
        float bv = (has_buf && !first) ? buf[i] : 0.f;
        const float pv = one(p[i], load1(g + i), bv);
        p[i] = pv;
        if (has_buf) buf[i] = bv;
        if (sh != nullptr) store1(sh + i, pv);
      });
}

// dst[t] = cast(src[t]) for a list of fp32 tensors (dst in ptr[0], src in ptr[1]): gathers the gradients of a backward
// segment into the flat bucket a data-parallel all-reduce sends (D = bf16 on the wire, or fp32)
template <typename D>
__global__ void __launch_bounds__(kThreads) mt_gather_kernel(const __grid_constant__ MtTable t) {
  const MtBlock b = mt_block(t);
  D* __restrict__ dst = static_cast<D*>(t.ptr[0][b.ti]);
  const float* __restrict__ src = static_cast<const float*>(t.ptr[1][b.ti]);
  mt_stream<4>(b, (uintptr_t)src, dst, nullptr,
      [&](long i) { store4(dst + i, __ldg(reinterpret_cast<const float4*>(src + i))); },
      [&](long i) { store1(dst + i, src[i]); });
}

// every entry of each given table slot (null: a slot the stream does not use) must be a tensor
int mt_check(const char* who, int n_tensors, std::initializer_list<const void* const*> slots) {
  for (const void* const* s : slots)
    for (int i = 0; s != nullptr && i < n_tensors; ++i) STSWIN_CHECK_ARG(s[i] != nullptr, "%s: null tensor %d", who, i);
  return kOk;
}

// Runs a stream over n_tensors tensors, MT_MAX per launch.  Entry t of table slot k is slots[k][t]: a slot given as
// null stays null, and every entry of a given slot must be non-null.  shadow and flag come from shadows / flags (null:
// none).  launch(table, blocks, t0) enqueues the kernels of the launch that starts at tensor t0 and has `blocks` blocks;
// a launch of only empty tensors is skipped.
template <class Launch>
int mt_launch(const char* who, int n_tensors, std::initializer_list<const void* const*> slots, void* const* shadows,
              const int64_t* numels, const uint8_t* flags, Launch&& launch) {
  if (const int st = mt_check(who, n_tensors, slots)) return st;
  for (int t0 = 0; t0 < n_tensors; t0 += MT_MAX) {
    MtTable t;
    t.n = n_tensors - t0 < MT_MAX ? n_tensors - t0 : MT_MAX;
    int blocks = 0;
    for (int i = 0; i < t.n; ++i) {
      int k = 0;
      for (const void* const* s : slots) t.ptr[k++][i] = s != nullptr ? const_cast<void*>(s[t0 + i]) : nullptr;
      t.shadow[i] = shadows != nullptr ? static_cast<__nv_bfloat16*>(shadows[t0 + i]) : nullptr;
      t.numel[i] = numels[t0 + i];
      t.flag[i] = flags != nullptr ? flags[t0 + i] : 0;
      t.block_start[i] = blocks;
      blocks += (int)((numels[t0 + i] + MT_CHUNK - 1) / MT_CHUNK);
    }
    t.block_start[t.n] = blocks;
    if (blocks > 0) STSWIN_CUDA(launch(t, blocks, t0));
  }
  STSWIN_CUDA(cudaGetLastError());
  return kOk;
}

}  // namespace

long ohem_ws_bytes() { return (long)sizeof(OhemWs); }

int ohem_ce_fwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, long HW, int ignore_index,
                float thresh, long n_min, float* loss_px, void* ws, float* loss, float* sel, cudaStream_t stream) {
  STSWIN_CHECK_ARG(logits && labels && loss_px && ws && loss && sel, "ohem_ce_fwd: null pointer");
  STSWIN_CHECK_ARG(B > 0 && K > 0 && HW > 0, "ohem_ce_fwd: empty input");
  const long M = (long)B * HW;
  // losses.py:36 reads loss[n_min] of the sorted vector (an IndexError in the reference when out of range)
  STSWIN_CHECK_ARG(n_min >= 1 && n_min < M, "ohem_ce_fwd: n_min must be in [1, B*H*W)");
  OhemWs* w = static_cast<OhemWs*>(ws);
  STSWIN_CUDA(cudaMemsetAsync(w, 0, sizeof(OhemWs), stream));
  const bool vec = HW % 4 == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(labels) & 15) == 0 && (reinterpret_cast<uintptr_t>(loss_px) & 15) == 0;
  const int grid = stream_grid(vec ? M / 4 : M);
  if (logits_is_f32) {
    if (vec) ohem_px_kernel<float, 4><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(logits), labels, B, K, HW, ignore_index, thresh, loss_px, w);
    else ohem_px_kernel<float, 1><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(logits), labels, B, K, HW, ignore_index, thresh, loss_px, w);
  } else {
    if (vec) ohem_px_kernel<__nv_bfloat16, 4><<<grid, kThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(logits), labels, B, K, HW, ignore_index, thresh, loss_px, w);
    else ohem_px_kernel<__nv_bfloat16, 1><<<grid, kThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(logits), labels, B, K, HW, ignore_index, thresh, loss_px, w);
  }
  STSWIN_CHECK_ARG((reinterpret_cast<uintptr_t>(loss_px) & 15) == 0, "ohem_ce_fwd: loss_px must be 16-byte aligned");
  int g2 = stream_grid(M / 4);
  if (g2 > 2 * num_sms()) g2 = 2 * num_sms();        // fixed per-block cost (histogram clear / flush, digit picks)
  ohem_hist_kernel<0><<<g2, kThreads, 0, stream>>>(loss_px, M, n_min, w);
  ohem_hist_kernel<1><<<g2, kThreads, 0, stream>>>(loss_px, M, n_min, w);
  ohem_hist_kernel<2><<<g2, kThreads, 0, stream>>>(loss_px, M, n_min, w);
  ohem_final_kernel<<<g2, kThreads, 0, stream>>>(loss_px, M, n_min, thresh, w, loss, sel);
  STSWIN_CUDA(cudaGetLastError());
  return kOk;
}

int ohem_ce_bwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, long HW, int ignore_index,
                const float* loss_px, const float* sel, const float* d_loss, void* d_logits, cudaStream_t stream) {
  STSWIN_CHECK_ARG(logits && labels && loss_px && sel && d_loss && d_logits, "ohem_ce_bwd: null pointer");
  STSWIN_CHECK_ARG(B > 0 && K > 0 && HW > 0, "ohem_ce_bwd: empty input");
  const long M = (long)B * HW;
  const bool vec = HW % 4 == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(labels) & 15) == 0 && (reinterpret_cast<uintptr_t>(loss_px) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(d_logits) & 15) == 0;
  const int grid = stream_grid(vec ? M / 4 : M);
  if (logits_is_f32) {
    if (vec) ohem_bwd_kernel<float, 4><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(logits), labels, B, K, HW, ignore_index, loss_px, sel, d_loss, static_cast<float*>(d_logits));
    else ohem_bwd_kernel<float, 1><<<grid, kThreads, 0, stream>>>(static_cast<const float*>(logits), labels, B, K, HW, ignore_index, loss_px, sel, d_loss, static_cast<float*>(d_logits));
  } else {
    if (vec) ohem_bwd_kernel<__nv_bfloat16, 4><<<grid, kThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(logits), labels, B, K, HW, ignore_index, loss_px, sel, d_loss, static_cast<__nv_bfloat16*>(d_logits));
    else ohem_bwd_kernel<__nv_bfloat16, 1><<<grid, kThreads, 0, stream>>>(static_cast<const __nv_bfloat16*>(logits), labels, B, K, HW, ignore_index, loss_px, sel, d_loss, static_cast<__nv_bfloat16*>(d_logits));
  }
  STSWIN_CUDA(cudaGetLastError());
  return kOk;
}

int ema_update(void* const* k_params, const void* const* q_params, void* const* k_shadows, const int64_t* numels,
               int n_tensors, float m, float one_minus_m, const float* m_dev, cudaStream_t stream) {
  STSWIN_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || (k_params && q_params && numels)), "ema_update: null table");
  return mt_launch("ema_update", n_tensors, {k_params, q_params}, k_shadows, numels, nullptr,
                   [&](const MtTable& t, int blocks, int) {
                     ema_kernel<<<blocks, kThreads, 0, stream>>>(t, m, one_minus_m, m_dev);
                     return cudaGetLastError();
                   });
}

int lars_sgd_step(void* const* params, void* const* grads, void* const* bufs, void* const* shadows, const int64_t* numels,
                  const uint8_t* first_step, int n_tensors, int grads_are_bf16, int write_grads, float lr,
                  const float* lr_dev, float momentum, float dampening, int nesterov, float weight_decay, int lars,
                  float trust_coef, float eps, double* norms_ws, cudaStream_t stream) {
  STSWIN_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || (params && grads && numels)), "lars_sgd_step: null table");
  STSWIN_CHECK_ARG(momentum == 0.f || bufs != nullptr, "lars_sgd_step: momentum needs momentum buffers");
  STSWIN_CHECK_ARG(!lars || norms_ws != nullptr, "lars_sgd_step: the LARS group needs a [2*n_tensors] fp64 workspace");
  STSWIN_CHECK_ARG(!nesterov || (momentum > 0.f && dampening == 0.f), "lars_sgd_step: nesterov needs momentum and zero dampening");
  STSWIN_CHECK_ARG(!(grads_are_bf16 && write_grads), "lars_sgd_step: bf16 gradients are read-only (write_grads needs fp32)");
  if (n_tensors == 0) return kOk;
  if (lars) STSWIN_CUDA(cudaMemsetAsync(norms_ws, 0, sizeof(double) * 2 * (size_t)n_tensors, stream));
  const LarsHp a{lr, momentum, dampening, weight_decay, trust_coef, eps, nesterov, lars, write_grads, lr_dev};
  return mt_launch("lars_sgd_step", n_tensors, {params, grads, momentum != 0.f ? bufs : nullptr}, shadows, numels,
                   first_step, [&](const MtTable& t, int blocks, int t0) {
                     double* nw = norms_ws ? norms_ws + 2 * t0 : nullptr;
                     if (grads_are_bf16) {
                       if (lars) lars_norm_kernel<__nv_bfloat16><<<blocks, kThreads, 0, stream>>>(t, weight_decay, nw);
                       lars_sgd_kernel<__nv_bfloat16><<<blocks, kThreads, 0, stream>>>(t, a, nw);
                     } else {
                       if (lars) lars_norm_kernel<float><<<blocks, kThreads, 0, stream>>>(t, weight_decay, nw);
                       lars_sgd_kernel<float><<<blocks, kThreads, 0, stream>>>(t, a, nw);
                     }
                     return cudaGetLastError();
                   });
}

int adam_step(void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
              void* const* shadows, const int64_t* numels, int n_tensors, int grads_are_bf16, float lr, float beta1,
              float beta2, float eps, float weight_decay, float grad_scale, float* step, cudaStream_t stream) {
  STSWIN_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || (params && grads && exp_avg && exp_avg_sq && numels)), "adam_step: null table");
  STSWIN_CHECK_ARG(step != nullptr, "adam_step: null step counter");
  STSWIN_CHECK_ARG(beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f && eps >= 0.f, "adam_step: bad hyper-parameters");
  if (n_tensors == 0) return kOk;
  const std::initializer_list<const void* const*> slots{params, grads, exp_avg, exp_avg_sq};
  if (const int st = mt_check("adam_step", n_tensors, slots)) return st;      // a refused step leaves the count alone
  adam_tick_kernel<<<1, 1, 0, stream>>>(step);
  const AdamHp a{lr, beta1, beta2, eps, weight_decay, grad_scale, step};
  return mt_launch("adam_step", n_tensors, slots, shadows, numels, nullptr,
                   [&](const MtTable& t, int blocks, int) {
                     return grads_are_bf16 ? launch_pdl(adam_kernel<__nv_bfloat16>, dim3(blocks), dim3(kThreads), 0, stream, t, a)
                                           : launch_pdl(adam_kernel<float>, dim3(blocks), dim3(kThreads), 0, stream, t, a);
                   });
}

int sgd_step(void* const* params, const void* const* grads, void* const* momentum_bufs, void* const* shadows,
             const int64_t* numels, const uint8_t* first_step, int n_tensors, int grads_are_bf16, float lr, const float* lr_dev,
             float momentum, float one_minus_dampening, int nesterov, int maximize, float weight_decay, float grad_scale,
             cudaStream_t stream) {
  STSWIN_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || (params && grads && numels)), "sgd_step: null table");
  STSWIN_CHECK_ARG(momentum == 0.f || momentum_bufs != nullptr, "sgd_step: momentum needs momentum buffers");
  STSWIN_CHECK_ARG(!nesterov || (momentum > 0.f && one_minus_dampening == 1.f),
                   "sgd_step: nesterov needs momentum and zero dampening");
  if (n_tensors == 0) return kOk;
  const SgdHp a{lr, momentum, one_minus_dampening, weight_decay, grad_scale, nesterov, maximize, lr_dev};
  return mt_launch("sgd_step", n_tensors, {params, grads, momentum != 0.f ? momentum_bufs : nullptr}, shadows, numels,
                   first_step, [&](const MtTable& t, int blocks, int) {
                     return grads_are_bf16 ? launch_pdl(sgd_kernel<__nv_bfloat16>, dim3(blocks), dim3(kThreads), 0, stream, t, a)
                                           : launch_pdl(sgd_kernel<float>, dim3(blocks), dim3(kThreads), 0, stream, t, a);
                   });
}

int gather_cast(void* const* dst, const void* const* src, const int64_t* numels, int n_tensors, int dst_is_bf16,
                cudaStream_t stream) {
  STSWIN_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || (dst && src && numels)), "gather_cast: null table");
  return mt_launch("gather_cast", n_tensors, {dst, src}, nullptr, numels, nullptr, [&](const MtTable& t, int blocks, int) {
    if (dst_is_bf16) mt_gather_kernel<__nv_bfloat16><<<blocks, kThreads, 0, stream>>>(t);
    else mt_gather_kernel<float><<<blocks, kThreads, 0, stream>>>(t);
    return cudaGetLastError();
  });
}

}  // namespace stswin
