// Geometry shared by the window-attention forward and backward kernels.
//
// A "tile" is 128 token rows = G consecutive windows of L = T*ws*ws tokens each.  Window g of the tile
// starts at row g * slot: slot = L for L <= 16, else L rounded up to a power of two (49 -> 64, 25 -> 32,
// 98 -> 128), G = 128 / slot; rows slot*g + [L, slot) and rows >= G*slot are padding and stay zero.  A warp of
// the row-per-thread groups (32 rows) then never straddles two windows with more than 16 tokens, which is what
// the compile-time column maps below need.
// Work item = (tile, head).  Each operand chunk is [128 rows x 64 channels] bf16 in the
// 128B-swizzled K-major layout, filled by TMA boxes taken straight from the un-rolled,
// un-partitioned [B, T, H, W, channels] tensor: the cyclic shift and the window partition
// (swin_512.py:210-218) are the box coordinates; window_reverse + the inverse roll (:224-231)
// are the same coordinates on the store side.  A window that wraps around the image border
// (last window row / column of a shifted block) is moved as four quadrant boxes, which changes
// the order of its tokens inside the tile; the per-row geometry below (`row_geom`) is the single
// place that knows the order, and bias / mask lookups go through it.
#pragma once

#include "common.cuh"
#include "host_util.h"

namespace stswin {

constexpr int SLOT_BYTES = 128 * 128;          // one operand chunk: 128 rows x 64 bf16
constexpr int TAB_MAX = 15 * 15;               // (2*ws-1)^2 for ws <= 8
constexpr float kMaskLog2e = -100.0f * 1.4426950408889634f;

// Timeline tracing for tools/trace_attn.py (debug builds with -DSTSWIN_TRACE only): CTA 0 records
// clock64() at named points of its first 64 work items.
#ifdef STSWIN_TRACE
#define STSWIN_TRACE_DECL(name) __device__ long long* name = nullptr;
#define WTRACE(sym, it, id)                                                           \
  do {                                                                                \
    if (blockIdx.x == 0 && (it) < 64 && sym != nullptr) sym[(it) * 16 + (id)] = clock64(); \
  } while (0)
#else
#define STSWIN_TRACE_DECL(name)
#define WTRACE(sym, it, id) do { } while (0)
#endif

struct WinGeom {
  int B, T, H, W, C, nH, ws, shift;
  int hd, N, L, G, nWh, nWw, nW, total_windows, num_tiles, nc;   // nc = 64-channel chunks per head group
  int slot;           // tile rows from one window of the tile to the next (>= L, see above)
  int SH, ngrp, gch;   // head_dim >= 64: SH = 1, a "head group" is one head (gch = hd channels).
                       // head_dim 32  : SH = 2 heads share one 64-channel chunk (gch = 64); S / dP use
                       // the head's 32-channel K sub-range of the chunk, the output products run over
                       // the whole chunk and only the head's own 32 columns are kept.
  float scale_log2e;                                              // hd^-0.5 * log2(e)
  float scale;                                                    // hd^-0.5
  int ra, rb;         // a shifted window that wraps is moved as 2x2 rectangles of (ws-shift | shift) rows x columns
  int roff[5];        // first tile row of rectangle k inside its window's L rows (roff[4] = L)
  int general;        // 1: L is not 16/32/64/128, or (backward) a shift with unequal rectangles: see select_variant
  const float* mask;  // optional dense additive mask [mask_nw, N, N] (WindowAttention.forward's `mask`
  int mask_nw;        //   argument, swin_512.py:127-131), applied ON TOP of the closed-form shift mask; or null
  unsigned long long mg_nW, mg_nWw;   // ceil(2^32 / nW), ceil(2^32 / nWw): exact division of window indices by multiply-shift
  int perm;           // 1 (backward, shifted): window indices are enumerated interior-windows-first (see window_coords)
  int uniform_quad;   // always 0: only the windows that wrap use quadrant order.  Kept with quad_order(): without this
                      //   run-time select, ptxas spills the backward kernel's head group in winattn_bwd_kernel<32,4,2,1,...>
};

struct RowGeom {
  int g;       // window slot inside the tile
  int rr, cc;  // token coordinates inside its window (shifted frame)
  int id;      // shift-mask region id 0..8 (swin_512.py:173-184), 0 when unshifted
  int canon;   // g*L + t*N + rr*ws + cc : position in the reference's own window-token order
  int gw;      // global window index b*nW + win in the natural order (clamped for padding windows)
  long tok;    // index of the source token in the natural [B*T, H, W] order (roll + partition undone)
  bool wraps;  // window crosses the image border (the only windows with a non-zero mask)
  bool valid;  // false for rows of a padding window in the last tile, and for padding rows
  bool inrange; // false for the padding rows of a tile (behind a window's L tokens in its slot, or behind the last slot)
};

struct WinMaps {     // tensor maps over one [B*T, H, W, channels] tensor
  CUtensorMap full;      // box = whole window (ws x ws x T)
  CUtensorMap rect[4];   // boxes of the 2x2 rectangle decomposition of a wrapping window
};

__device__ __forceinline__ bool quad_order(const WinGeom& gm, bool wraps) {
  return gm.uniform_quad ? (gm.shift > 0) : wraps;
}

// Window index -> (image, window row, window column).  With gm.perm the indices enumerate the interior
// windows of every image first and the windows that wrap around the border (last window row / column
// of a shifted block) after them: a CTA that walks its items in increasing order then changes token
// order (row-major <-> quadrant) once instead of at every third item, which is what the backward
// kernel's per-row register state (bias values, bias-gradient sums) wants.
__device__ __forceinline__ void window_coords(const WinGeom& gm, int gw, int& b, int& wh, int& ww, bool& wraps) {
  if (gm.perm) {
    const int ni = (gm.nWh - 1) * (gm.nWw - 1);       // interior windows per image
    const int n_int = gm.B * ni;
    if (gw < n_int) {
      b = gw / ni;
      const int r = gw - b * ni;
      wh = r / (gm.nWw - 1);
      ww = r - wh * (gm.nWw - 1);
      wraps = false;
    } else {
      const int nwr = gm.nWh + gm.nWw - 1;            // wrapping windows per image
      int r = gw - n_int;
      b = r / nwr;
      r -= b * nwr;
      if (r < gm.nWw) { wh = gm.nWh - 1; ww = r; }
      else            { wh = r - gm.nWw; ww = gm.nWw - 1; }
      wraps = gm.shift > 0;
    }
    return;
  }
  b = gw / gm.nW;
  const int win = gw - b * gm.nW;
  wh = win / gm.nWw;
  ww = win - wh * gm.nWw;
  wraps = gm.shift > 0 && (wh == gm.nWh - 1 || ww == gm.nWw - 1);
}

__device__ __forceinline__ int region_band(int p, int extent, int ws, int shift) {
  return (p >= extent - ws ? 1 : 0) + (p >= extent - shift ? 1 : 0);
}

// rectangle k (0..3) of the 2x2 decomposition: offsets / extents along h (k>>1) and w (k&1)
__device__ __forceinline__ void rect_dims(const WinGeom& gm, int k, int& h_off, int& w_off, int& h_ext, int& w_ext) {
  h_off = (k >> 1) ? gm.ra : 0;  h_ext = (k >> 1) ? gm.rb : gm.ra;
  w_off = (k & 1) ? gm.ra : 0;   w_ext = (k & 1) ? gm.rb : gm.ra;
}

// geometry of tile row r of tile `tile`
__device__ __forceinline__ RowGeom row_geom(const WinGeom& gm, int tile, int r) {
  RowGeom o;
  o.g = r / gm.slot;
  o.inrange = o.g < gm.G && r - o.g * gm.slot < gm.L;
  if (o.g > gm.G - 1) o.g = gm.G - 1;
  const int rem = o.inrange ? r - o.g * gm.slot : 0;
  int gw = tile * gm.G + o.g;
  o.valid = o.inrange && gw < gm.total_windows;
  if (gw > gm.total_windows - 1) gw = gm.total_windows - 1;
  int b, wh, ww, t;
  window_coords(gm, gw, b, wh, ww, o.wraps);
  o.gw = b * gm.nW + wh * gm.nWw + ww;        // the window's index in the natural (un-permuted) order
  if (!quad_order(gm, o.wraps)) {
    t = rem / gm.N;
    const int pos = rem - t * gm.N;
    o.rr = pos / gm.ws;
    o.cc = pos - o.rr * gm.ws;
  } else {
    int k = 0;
    while (k < 3 && rem >= gm.roff[k + 1]) ++k;
    int h_off, w_off, h_ext, w_ext;
    rect_dims(gm, k, h_off, w_off, h_ext, w_ext);
    const int r2 = rem - gm.roff[k], area = h_ext * w_ext;
    t = r2 / area;
    const int p = r2 - t * area;
    o.rr = h_off + p / w_ext;
    o.cc = w_off + p % w_ext;
  }
  o.canon = o.g * gm.L + t * gm.N + o.rr * gm.ws + o.cc;
  {
    const int hs = (wh * gm.ws + o.rr + gm.shift) % gm.H, wsrc = (ww * gm.ws + o.cc + gm.shift) % gm.W;
    o.tok = ((long)(b * gm.T + t) * gm.H + hs) * gm.W + wsrc;
  }
  o.id = 0;
  if (gm.shift > 0)
    o.id = 3 * region_band(wh * gm.ws + o.rr, gm.H, gm.ws, gm.shift) +
           region_band(ww * gm.ws + o.cc, gm.W, gm.ws, gm.shift);
  return o;
}

// Compile-time column maps of the fast-path geometries.  WS is the window size; L the tile rows one
// window slot spans (a power of two, <= 128); the window really holds LW = T*WS*WS tokens:
// LW = L for ws 8 / 4; 49 of 64 / 98 of 128 rows for 7x7 windows with one / two frames, 25 of 32 / 50 of 64
// for 5x5 (rows / columns >= LW of a slot are padding).  Shift is 0 or WS/2, so a window that wraps splits into 2x2 rectangles of
// RA = ceil(WS/2) and RB = WS - RA rows / columns (quadrants when WS is even).
// Column j (< LW) of a window, in row-major order (QUAD = false: t, row, column) or rectangle order
// (QUAD = true: rectangle, t, row, column inside the rectangle):
//   col_rect : rectangle index 0..3 (0 in row-major order)
//   col_pos  : spatial position rr*WS + cc of the token
//   col_key  : rr*(2*WS-1) + cc, so that key_i - col_key(j) indexes the relative-position bias table
template <int LW, int WS>
__host__ __device__ constexpr int rect_off(int k) {    // first column of rectangle k (k = 4: LW)
  constexpr int W1 = WS > 0 ? WS : 1, T = LW / (W1 * W1) > 0 ? LW / (W1 * W1) : 1;
  constexpr int RA = (W1 + 1) / 2, RB = W1 - RA;
  int off = 0;
  for (int q = 0; q < k; ++q) off += ((q >> 1) ? RB : RA) * ((q & 1) ? RB : RA) * T;
  return off;
}
template <int LW, int WS, bool QUAD>
__host__ __device__ constexpr int col_rect(int j) {
  // loop-free (the optimiser must fold this to a constant for every unrolled column)
  constexpr int o1 = rect_off<LW, WS>(1), o2 = rect_off<LW, WS>(2), o3 = rect_off<LW, WS>(3);
  return QUAD ? (j >= o1 ? 1 : 0) + (j >= o2 ? 1 : 0) + (j >= o3 ? 1 : 0) : 0;
}
template <int LW, int WS, bool QUAD>
__host__ __device__ constexpr int col_pos(int j) {
  constexpr int W1 = WS > 0 ? WS : 1, N = W1 * W1, RA = (W1 + 1) / 2, RB = W1 - RA;
  constexpr int o1 = rect_off<LW, WS>(1), o2 = rect_off<LW, WS>(2), o3 = rect_off<LW, WS>(3);
  if (!QUAD) return j % N;
  const int k = col_rect<LW, WS, true>(j);
  const int hext = (k >> 1) ? RB : RA, wext = (k & 1) ? RB : RA;
  const int off = k == 0 ? 0 : (k == 1 ? o1 : (k == 2 ? o2 : o3));
  const int p = (j - off) % (hext * wext);
  return (((k >> 1) ? RA : 0) + p / wext) * W1 + ((k & 1) ? RA : 0) + p % wext;
}
template <int LW, int WS, bool QUAD>
__host__ __device__ constexpr int col_key(int j) {
  constexpr int W1 = WS > 0 ? WS : 1;
  const int pos = col_pos<LW, WS, QUAD>(j);
  return (pos / W1) * (2 * W1 - 1) + pos % W1;
}

// n / d for 0 <= n * d < 2^32 with mg = ceil(2^32 / d) (checked on the host in fill_geom)
__device__ __forceinline__ int fast_div(int n, unsigned long long mg) {
  return int((static_cast<unsigned long long>(static_cast<unsigned>(n)) * mg) >> 32);
}

// row_geom for the fast-path geometries: slot L, tokens per window LW, ws compile-time (shifts / constant divisions),
// shift 0 or ws/2.  ORDER 0: row-major.  2: quadrant order for the windows that wrap.
template <int L, int WS, int ORDER, int LW>
__device__ __forceinline__ RowGeom row_geom_fast(const WinGeom& gm, int tile, int r) {
  static_assert(ORDER == 0 || ORDER == 2, "ORDER 0 (unshifted) or 2 (shifted)");
  constexpr int N = WS * WS, G = 128 / L, RA = (WS + 1) / 2, RB = WS - RA;
  RowGeom o;
  o.g = r / L;
  const int rin = r % L;
  o.inrange = rin < LW;                       // LW < L: the tail rows of the slot are padding
  const int rem = o.inrange ? rin : 0;
  int gw = tile * G + o.g;
  o.valid = o.inrange && gw < gm.total_windows;
  if (gw > gm.total_windows - 1) gw = gm.total_windows - 1;
  int b, wh, ww;
  if (gm.perm) {
    window_coords(gm, gw, b, wh, ww, o.wraps);
  } else {
    b = fast_div(gw, gm.mg_nW);
    const int win = gw - b * gm.nW;
    wh = fast_div(win, gm.mg_nWw);
    ww = win - wh * gm.nWw;
    o.wraps = ORDER != 0 && (wh == gm.nWh - 1 || ww == gm.nWw - 1);
  }
  o.gw = b * gm.nW + wh * gm.nWw + ww;        // the window's index in the natural (un-permuted) order
  int t;
  if (ORDER == 0 || !o.wraps) {
    t = rem / N;
    const int pos = rem % N;
    o.rr = pos / WS;
    o.cc = pos % WS;
  } else {
    int k = 0;
#pragma unroll
    for (int q = 1; q < 4; ++q) k += (rem >= rect_off<LW, WS>(q)) ? 1 : 0;
    const int hext = (k >> 1) ? RB : RA, wext = (k & 1) ? RB : RA, area = hext * wext;
    const int r2 = rem - ((k == 0) ? 0 : (k == 1) ? rect_off<LW, WS>(1) : (k == 2) ? rect_off<LW, WS>(2) : rect_off<LW, WS>(3));
    t = r2 / area;
    const int p = r2 - t * area;
    o.rr = ((k >> 1) ? RA : 0) + p / wext;
    o.cc = ((k & 1) ? RA : 0) + p % wext;
  }
  o.canon = o.g * LW + t * N + o.rr * WS + o.cc;
  const int shift = ORDER == 0 ? 0 : WS / 2;
  int hs = wh * WS + o.rr + shift, wsrc = ww * WS + o.cc + shift;
  if (hs >= gm.H) hs -= gm.H;
  if (wsrc >= gm.W) wsrc -= gm.W;
  o.tok = ((long)(b * gm.T + t) * gm.H + hs) * gm.W + wsrc;
  o.id = 0;
  if (ORDER != 0)
    o.id = 3 * region_band(wh * WS + o.rr, gm.H, WS, WS / 2) + region_band(ww * WS + o.cc, gm.W, WS, WS / 2);
  return o;
}

// Issue the TMA boxes that fill (LOAD) or drain (STORE) one [128 x 64ch] chunk buffer for `tile`.
//   ch0 : first channel of the chunk in the global tensor
// Called by all 32 lanes of one warp; box k of the chunk is issued by lane k % 32.
template <bool LOAD>
__device__ __forceinline__ void tile_boxes(const WinGeom& gm, int tile, int ch0, uint8_t* buf, const WinMaps* tm,
                                           uint64_t* bar, int lane) {
  for (int k = lane; k < gm.G * 4; k += 32) {
    const int g = k >> 2, q = k & 3;
    int gw = tile * gm.G + g;
    if (gw >= gm.total_windows) {
      if (!LOAD) continue;            // nothing to store for a padding window
      gw = gm.total_windows - 1;      // loads: finite filler data, never stored
    }
    int b, wh, ww;
    bool wraps;
    window_coords(gm, gw, b, wh, ww, wraps);
    uint8_t* dst = buf + (g * gm.slot) * 128;
    if (!quad_order(gm, wraps)) {
      if (q != 0) continue;
      const int w0 = ww * gm.ws + gm.shift, h0 = wh * gm.ws + gm.shift;
      if (LOAD) tma_load_4d(dst, &tm->full, bar, ch0, w0, h0, b * gm.T);
      else      tma_store_4d(&tm->full, dst, ch0, w0, h0, b * gm.T);
    } else {
      int h_off, w_off, h_ext, w_ext;
      rect_dims(gm, q, h_off, w_off, h_ext, w_ext);
      const int h0 = (wh * gm.ws + gm.shift + h_off) % gm.H;
      const int w0 = (ww * gm.ws + gm.shift + w_off) % gm.W;
      uint8_t* d = dst + gm.roff[q] * 128;
      if (LOAD) tma_load_4d(d, &tm->rect[q], bar, ch0, w0, h0, b * gm.T);
      else      tma_store_4d(&tm->rect[q], d, ch0, w0, h0, b * gm.T);
    }
  }
}

// bytes one chunk load brings in (only the G*L real rows of the 128-row buffer; padding rows are never written)
__device__ __forceinline__ uint32_t chunk_tx_bytes(const WinGeom& gm) { return uint32_t(gm.G * gm.L) * 128u; }

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// Load this thread's CH = min(L, 32) columns [col0 + cb*CH, +CH) of TMEM row `t_lane` into v[0..CH).
// tcgen05.ld is warp-collective and needs a warp-uniform address: for L == 16 two windows share a
// warp, so the warp loads its 32-column band and each half-warp keeps its own 16 columns.
template <int L>
__device__ __forceinline__ void tmem_ld_row_chunk(uint32_t tmem_mat, uint32_t t_lane, int col0, int cb, int wq, int lane,
                                                  uint32_t (&v)[32]) {
  if (L >= 32) {
    tmem_ld32(tmem_mat + t_lane + col0 + cb * 32, v);
    tmem_ld_wait();
  } else {
    tmem_ld32(tmem_mat + t_lane + wq * 32, v);
    tmem_ld_wait();
    if (lane >= 16) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = v[j + 16];
    }
  }
}

// Write a block held one row per lane ([32 rows] x [NB x 16 bytes]) to global memory with whole-line
// stores: the rows go through a per-warp 4 KB staging area (128B-swizzled, conflict-free both ways) and
// come back 8 lanes per row, so one store instruction covers 4 complete 128-byte lines instead of 32
// partial ones (a row-per-lane st.global is bound by the LSU: 32 lines per instruction).
//   rowp[i] : global address of the block's first byte for row i*4 + lane/8, or nullptr to skip the row
template <int NB>
__device__ __forceinline__ void warp_store_rows(uint8_t* stage, const uint4 (&vals)[NB], uint8_t* const (&rowp)[8],
                                                int lane) {
  __syncwarp();                      // the previous block has been read out
#pragma unroll
  for (int j = 0; j < NB; ++j) *reinterpret_cast<uint4*>(stage + sw128_offset(lane, j)) = vals[j];
  __syncwarp();
  const int ch = lane & 7;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3);
    if (ch < NB && rowp[i] != nullptr)
      *reinterpret_cast<uint4*>(rowp[i] + ch * 16) = *reinterpret_cast<const uint4*>(stage + sw128_offset(r, ch));
  }
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- host side of both directions

// Checks the geometry and fills *gm.  qk_scale > 0 replaces head_dim^-0.5; mask: optional dense additive mask
// [mask_windows, N, N], or null.
int fill_geom(WinGeom* gm, int B, int T, int H, int W, int C, int nH, int ws, int shift, float qk_scale,
              const float* mask, int mask_windows);
// tensor maps over a [B*T, H, W, channels] bf16 tensor: whole-window box and the four rectangle boxes
int make_window_tmaps(WinMaps* maps, const void* base, const WinGeom& gm, int channels);

// Every kernel instantiation of the forward and of the backward, X(L, WS, ORDER, GEN, LWT) (the template parameters
// of winattn_fwd_kernel); the backward instantiates each one for SHT = 1 and 2 heads per 64-channel group.
#define STSWIN_WINATTN_VARIANTS(X)                                                                  \
  X(128, 7, 0, false, 98) X(128, 7, 2, false, 98) X(64, 7, 0, false, 49) X(64, 7, 2, false, 49)   \
  X(64, 5, 0, false, 50) X(64, 5, 2, false, 50) X(32, 5, 0, false, 25) X(32, 5, 2, false, 25)     \
  X(32, 0, 0, true, 32) X(128, 0, 0, true, 128)                                                   \
  X(128, 8, 0, false, 128) X(128, 8, 2, false, 128) X(64, 8, 0, false, 64) X(64, 8, 2, false, 64) \
  X(32, 4, 0, false, 32) X(32, 4, 2, false, 32)                                                   \
  X(16, 0, 0, false, 16) X(32, 0, 0, false, 32) X(64, 0, 0, false, 64) X(128, 0, 0, false, 128)

struct WinVariant {
  int L, WS, ORDER;
  bool GEN;
  int LWT;
};

// The instantiation that runs a geometry.  Every variant computes the same result; the choice decides only speed.
// backward: sets the backward kernel's gm.general and gm.perm first.
inline WinVariant select_variant(WinGeom& gm, bool backward) {
  if (backward) {
    if (gm.shift > 0 && gm.ra != gm.rb) gm.general = 1;   // unequal rectangles: no static column -> position fold
    gm.perm = gm.shift > 0 && gm.nWh > 1 && gm.nWw > 1;   // interior windows first: one token-order switch per CTA
  }
  const int ws = gm.ws, L = gm.L;
  // token order of a shifted block: quadrant order only for the windows that wrap (one box per interior window
  // measured faster than four quadrant boxes for every window, at every L)
  const int order = gm.shift == 0 ? 0 : 2;
  // compile-time column maps need shift 0 or ws/2 (rectangles of ceil(ws/2) and ws/2) and no dense mask
  const bool maps = gm.mask == nullptr && (gm.shift == 0 || gm.shift == ws / 2);
  // odd windows in padded slots (7x7 and 5x5 with one or two frames: 49 of 64 / 98 of 128 / 25 of 32 / 50 of 64 rows)
  if (maps && ((ws == 7 && (L == 49 || L == 98)) || (ws == 5 && (L == 25 || L == 50))))
    return {gm.slot, ws, order, false, L};
  // look-up table with window tags: the warp's 32-column band for windows of 4 / 8 tokens, else the whole row
  if (gm.general) return gm.slot <= 8 && 32 % gm.slot == 0 ? WinVariant{32, 0, 0, true, 32} : WinVariant{128, 0, 0, true, 128};
  // the shipped geometries: ws 8 or 4, one or two frames per window
  if (maps && ((ws == 8 && (L == 128 || L == 64)) || (ws == 4 && L == 32))) return {L, ws, order, false, L};
  return {L, 0, 0, false, L};   // look-up table per column
}

template <int L_, int WS_, int ORDER_, bool GEN_, int LWT_>
struct WinKernel {
  static constexpr int L = L_, WS = WS_, ORDER = ORDER_, LWT = LWT_;
  static constexpr bool GEN = GEN_;
};

// launch(WinKernel<v's template parameters>{}) for a listed variant v
template <typename F>
int dispatch_variant(const WinVariant& v, F&& launch) {
#define STSWIN_DISPATCH(L_, WS_, ORDER_, GEN_, LWT_)                                          \
  if (v.L == L_ && v.WS == WS_ && v.ORDER == ORDER_ && v.GEN == GEN_ && v.LWT == LWT_) \
    return launch(WinKernel<L_, WS_, ORDER_, GEN_, LWT_>{});
  STSWIN_WINATTN_VARIANTS(STSWIN_DISPATCH)
#undef STSWIN_DISPATCH
  return set_error(kErrUnsupported, "winattn: no kernel instantiation L=%d WS=%d ORDER=%d GEN=%d LWT=%d", v.L, v.WS,
                   v.ORDER, int(v.GEN), v.LWT);
}

// CTAs of a launch: at most one per SM, and a multiple of the head groups (every CTA keeps one head group: its bias
// tables live in shared memory).  The work items are a multiple of the head groups, so the grid holds at least one
// of each unless there are more head groups than SMs.
inline int winattn_grid(const WinGeom& gm, int* grid) {
  const int items = gm.num_tiles * gm.ngrp;
  *grid = items < num_sms() ? items : num_sms();
  *grid -= *grid % gm.ngrp;
  if (*grid < gm.ngrp) return set_error(kErrUnsupported, "winattn: %d head groups exceed the SM count", gm.ngrp);
  return kOk;
}

template <typename... KArgs, typename... Args>
int launch_winattn(void (*kern)(KArgs...), const WinGeom& gm, int threads, int smem, cudaStream_t stream, Args... args) {
  int grid, rc;
  if ((rc = winattn_grid(gm, &grid)) != kOk) return rc;
  STSWIN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  STSWIN_CUDA(launch_pdl(kern, dim3(grid), dim3(threads), (size_t)smem, stream, args...));
  STSWIN_CUDA(cudaGetLastError());
  return kOk;
}

}  // namespace stswin
