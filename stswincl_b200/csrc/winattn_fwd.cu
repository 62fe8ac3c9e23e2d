// K3 forward: spatio-temporal shifted-window attention core.
//
// Replaces, in one kernel (reference: seg18/net/Ours/swin_512.py)
//   torch.roll(-s) + window_partition + view/permute           :210-218   -> TMA box coordinates
//   q*scale, q @ k^T                                            :119-120   -> tcgen05 (S in TMEM)
//   relative_position_bias gather + repeat(1,T,T), + mask       :122-131   -> registers
//   softmax                                                     :132-134   -> registers (exp2)
//   attn @ v, transpose/reshape                                 :138       -> tcgen05 (O in TMEM)
//   window_reverse + torch.roll(+s)                             :224-231   -> TMA store coordinates
//
// Input  qkv [B, T, H, W, 3C] bf16 (un-rolled token order; channel = which*C + head*hd + d, :116)
// Output out [B, T, H, W, C]  bf16 (same token order), lse2 [num_tiles, nH, 128] fp32
//        (base-2 log-sum-exp of every tile row, consumed by the backward kernel).
//
// CTA = 3 warpgroups: warp 0 TMA producer, warp 1 MMA issuer (warp-uniform control flow, one
// elected lane issues), warps 4-7 softmax, warps 8-11 epilogue (thread <-> tile row <-> TMEM lane in
// both; a softmax and an epilogue warp share each SM sub-partition, so the MUFU-heavy softmax of
// item k overlaps the TMEM / store-heavy drain of item k-1).  Operand chunks stream through a ring
// of 16 KB slots.  The tensor core runs one item ahead: S(k+1) is issued before P V(k).
#include <type_traits>

#include "winattn_common.cuh"
#include "host_util.h"

namespace stswin {

namespace {

constexpr int NQK = 6;                         // ring of Q / K chunks (consumed by S = Q K^T)
constexpr int NV = 4;                          // ring of V chunks (consumed by O = P V)
constexpr int NSLOT = NQK + NV;
constexpr int P_BYTES = 2 * SLOT_BYTES;        // P [128 x 128] bf16 as two K-major halves
constexpr int STG_BYTES = 4 * 4096;             // per-warp output transposition areas (epilogue warps)
constexpr int NUM_THREADS = 384;               // warpgroup 0: producer, MMA issuer (+2 idle); 1: softmax; 2: epilogue
constexpr int SMEM_BYTES = 1024 + NSLOT * SLOT_BYTES + P_BYTES + STG_BYTES + 128 * 4 + 2 * (TAB_MAX + 1) * 4 + 512 * 4 + 256;
STSWIN_TRACE_DECL(g_trace_fwd)

// L   : window columns a thread walks (16/32/64/128).  GEN: the tile holds G windows of gm.L tokens with gm.L not
//       16/32/64/128 (e.g. 3x3x2 = 18); every thread then walks the whole 128-column row (L = 128) -- or, when the
//       windows have 4 / 8 tokens and never straddle a warp, the 32-column band of its warp (L = 32) -- and keeps only
//       the columns tagged with its own window.
//
// WS > 0 selects the fast softmax (compile-time geometry: slot L, LWT = T*WS*WS <= L tokens per window; ORDER 0
// unshifted, 2 shifted: quadrant order for the windows that wrap, row-major for the others).  The
// column -> (relative-position key, quadrant) map is then a compile-time function of the column,
// so the bias is one LDS at an immediate offset and the shift mask is one additive constant per
// quadrant.  WS == 0 is the generic path (look-up table per column: dense mask, L = 16, GEN).
// STSWIN_WINATTN_VARIANTS lists the instantiations and select_variant picks one (winattn_common.cuh).
template <int L, int WS, int ORDER, bool GEN, int LWT>
__global__ void __launch_bounds__(NUM_THREADS, 1)
winattn_fwd_kernel(const __grid_constant__ WinMaps tm_qkv, __nv_bfloat16* __restrict__ out,
                   const float* __restrict__ bias_table, float* __restrict__ lse2, const WinGeom gm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* s_ring = smem;
  uint8_t* s_p = s_ring + NSLOT * SLOT_BYTES;
  uint8_t* s_stage = s_p + P_BYTES;                                      // 4 warps x 4 KB output transposition
  uint32_t* s_lut = reinterpret_cast<uint32_t*>(s_stage + STG_BYTES);    // [128] key | id<<8 | pos<<16 | tag<<24
  float* s_tab = reinterpret_cast<float*>(s_lut + 128);                   // [2][TAB_MAX + 1] bias * log2e per head of the group
  float* s_inv = s_tab + 2 * (TAB_MAX + 1);                               // [2 item parities][2 heads][128] 1 / rowsum
  static_assert(((128 + 2 * (TAB_MAX + 1) + 512) * 4) % 8 == 0, "mbarriers need 8-byte alignment");
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_inv + 512);
  uint64_t* full_bar = bars;                  // [NSLOT]: Q/K ring slots first, then the V ring slots
  uint64_t* empty_bar = bars + NSLOT;
  uint64_t* s_full = bars + 2 * NSLOT;
  uint64_t* s_free = s_full + 1;
  uint64_t* p_full = s_full + 2;
  uint64_t* o_full = s_full + 3;
  uint64_t* o_free = s_full + 4;
  uint64_t* pv_done = s_full + 5;
  uint64_t* inv_full = s_full + 6;            // [2] 1/rowsum of every head of an item published (per item parity)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 8);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_items = gm.num_tiles * gm.ngrp;     // work item = (tile, head group)
  const int nc = gm.nc;
  const int SH = gm.SH;
  const int hg = blockIdx.x % gm.ngrp;              // constant per CTA: gridDim.x % ngrp == 0
  const int n_local = (num_items - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x);   // items of this CTA
  const int n_units = n_local * SH;                 // unit = (item, head of the group)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_qkv.full);
    for (int i = 0; i < NSLOT; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(s_free, 128);
    mbar_init(p_full, 128);
    mbar_init(o_full, 1);
    mbar_init(o_free, 128);
    mbar_init(pv_done, 1);
    mbar_init(&inv_full[0], 128);
    mbar_init(&inv_full[1], 128);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  // P buffer: entries outside a row's own window stay zero for the whole kernel.  Ring: the padding
  // rows of a tile (general mode) are never written by TMA and must read as zero.
  for (int i = threadIdx.x; i < (NSLOT * SLOT_BYTES + P_BYTES) / 16; i += NUM_THREADS)
    reinterpret_cast<uint4*>(s_ring)[i] = make_uint4(0, 0, 0, 0);
  // bias table(s) of this CTA's head group, pre-scaled by log2(e)
  pdl_wait();                // programmatic dependent launch: everything above overlapped the previous kernel's tail
  pdl_launch_dependents();
  {
    const int nbias = (2 * gm.ws - 1) * (2 * gm.ws - 1);
    for (int i = threadIdx.x; i < SH * nbias; i += NUM_THREADS) {
      const int sub = i / nbias, k = i - sub * nbias;
      s_tab[sub * (TAB_MAX + 1) + k] = __ldg(bias_table + k * gm.nH + hg * SH + sub) * 1.4426950408889634f;
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base;          // 128 columns
  const uint32_t tmem_O = tmem_base + 128;    // nc*64 columns (<= 256), or SH*64 when two heads share a chunk

  // register budget per warpgroup (setmaxnreg): the softmax warps hold a whole 128-column row in registers
  if (warp < 4) {
   asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
   if (warp == 0 || warp == 2) {
    // ---------------------------------------------------------------- TMA producers
    // warp 0 feeds the Q/K ring (Q0 K0 Q1 K1 ... per item), warp 2 the V ring: two independent rings,
    // so a V chunk waiting for its P never holds back the Q/K chunks of the next item (with one
    // shared ring the slot dependencies formed a loop of two HBM latencies per two items).
    const bool is_v = (warp == 2);
    const int nslot = is_v ? NV : NQK;
    uint8_t* ring = s_ring + (is_v ? NQK * SLOT_BYTES : 0);
    uint64_t* fullb = full_bar + (is_v ? NQK : 0);
    uint64_t* emptyb = empty_bar + (is_v ? NQK : 0);
    int slot = 0;
    uint32_t phase = 0;
    for (int k = 0; k < n_local; ++k) {
      const int item = int(blockIdx.x) + k * int(gridDim.x);
      const int tile = item / gm.ngrp;
      if (lane == 0) WTRACE(g_trace_fwd, k, is_v ? 1 : 0);
      for (int step = 0; step < (is_v ? nc : 2 * nc); ++step) {
        const int which = is_v ? 2 : (step & 1), c = is_v ? step : (step >> 1);
        mbar_wait(&emptyb[slot], phase ^ 1);
        if (lane == 0) mbar_arrive_expect_tx(&fullb[slot], chunk_tx_bytes(gm));
        __syncwarp();
        tile_boxes<true>(gm, tile, which * gm.C + hg * gm.gch + c * 64, ring + slot * SLOT_BYTES, &tm_qkv,
                         &fullb[slot], lane);
        if (++slot == nslot) { slot = 0; phase ^= 1; }
      }
    }
   } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    // The whole warp runs the control flow (so slot indices and descriptors stay in uniform registers);
    // one elected lane issues the tcgen05 instructions.
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128, 0, 0);
    constexpr uint32_t idesc_o = umma_idesc_bf16(128, 64, 0, 1);
    const uint32_t p_addr = smem_u32(s_p), ring_addr = smem_u32(s_ring);
    uint32_t seq_qk = 0, seq_v = 0, base_qk = 0, base_v = 0;     // running chunk counters of the two rings
    auto issue_S = [&](int u) {            // S = Q K^T (SH == 2: over the 32-channel K sub-range of head `sub`)
      const int sub = (SH == 1) ? 0 : (u & 1);
      mbar_wait(s_free, (u & 1) ^ 1);      // pass 1 of the previous unit has S in registers
      tc_fence_after();
      if (sub == 0) { base_qk = seq_qk; seq_qk += 2 * nc; }
      const int k0 = (SH == 1) ? 0 : sub * 2, k1 = (SH == 1) ? 4 : sub * 2 + 2;
      for (int c = 0; c < nc; ++c) {
        const uint32_t nq = base_qk + 2 * c, nk = nq + 1;
        const uint32_t sq = nq % NQK, sk = nk % NQK;
        if (sub == 0) {
          mbar_wait(&full_bar[sq], (nq / NQK) & 1);
          mbar_wait(&full_bar[sk], (nk / NQK) & 1);
        }
        tc_fence_after();
        const uint32_t qa = ring_addr + sq * SLOT_BYTES, ka = ring_addr + sk * SLOT_BYTES;
        if (leader) {
          for (int kk = k0; kk < k1; ++kk)
            umma_bf16(tmem_S, umma_smem_desc(qa + kk * 32, 16, 1024), umma_smem_desc(ka + kk * 32, 16, 1024), idesc_s,
                      (c > 0 || kk > k0) ? 1u : 0u);
          if (sub == SH - 1) {               // last reader of these chunks
            umma_commit(&empty_bar[sq]);
            umma_commit(&empty_bar[sk]);
          }
        }
      }
      if (leader) {
        umma_commit(s_full);
        WTRACE(g_trace_fwd, (SH == 1 ? u : u >> 1), 2);
      }
      __syncwarp();
    };
    auto issue_PV = [&](int u) {           // O = P V (SH == 2: whole 64-column chunk; the epilogue keeps the head's own 32)
      const int sub = (SH == 1) ? 0 : (u & 1);
      const int k = (SH == 1) ? u : (u >> 1);
      mbar_wait(p_full, u & 1);
      if (sub == 0) {
        mbar_wait(o_free, (k & 1) ^ 1);    // the previous item's O has been drained
        base_v = seq_v; seq_v += nc;
      }
      tc_fence_after();
      if (leader) WTRACE(g_trace_fwd, k, 3);
      for (int c = 0; c < nc; ++c) {
        const uint32_t nv = base_v + c, sv = NQK + nv % NV;
        if (sub == 0) mbar_wait(&full_bar[sv], (nv / NV) & 1);
        tc_fence_after();
        const uint32_t va = ring_addr + sv * SLOT_BYTES;
        if (leader) {
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const uint64_t adesc = umma_smem_desc(p_addr + (kk >> 2) * SLOT_BYTES + (kk & 3) * 32, 16, 1024);
            const uint64_t bdesc = umma_smem_desc(va + kk * 2048, SLOT_BYTES, 1024);
            umma_bf16(tmem_O + (SH == 1 ? c : sub) * 64, adesc, bdesc, idesc_o, kk > 0 ? 1u : 0u);
          }
          if (sub == SH - 1) umma_commit(&empty_bar[sv]);
        }
      }
      if (leader) {
        umma_commit(pv_done);              // P may be overwritten
        if (sub == SH - 1) umma_commit(o_full);
        WTRACE(g_trace_fwd, k, 4);
      }
      __syncwarp();
    };
    // S of unit u+1 is issued before P V of unit u (the softmax of u+1 then never waits for a tensor-core round trip).
    if (n_units > 0) issue_S(0);
    for (int u = 0; u < n_units; ++u) {
      if (u + 1 < n_units) issue_S(u + 1);
      issue_PV(u);
    }
   }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    // ---------------------------------------------------------------- softmax warps (group A)
    // thread <-> tile row <-> TMEM lane.  Per unit: S -> registers (+ bias, mask), row max, P = exp2(.)
    // -> smem (bf16) for the P V product; 1/rowsum goes to smem for the epilogue warps.
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const uint32_t t_lane = uint32_t(wq * 32) << 16;
    const bool tr = (threadIdx.x == 128);
    (void)tr;
    RowGeom rg;
    int key_i = 0, col0 = 0;
    for (int u = 0; u < n_units; ++u) {
      const int sub = (SH == 1) ? 0 : (u & 1);
      const int k = (SH == 1) ? u : (u >> 1);
      const int item = int(blockIdx.x) + k * int(gridDim.x);
      const int tile = item / gm.ngrp;
      const int head = hg * SH + sub;
      if (sub == 0) {
        if (tr) WTRACE(g_trace_fwd, k, 5);
        if constexpr (WS > 0) rg = row_geom_fast<L, WS, ORDER, LWT>(gm, tile, row);
        else                  rg = row_geom(gm, tile, row);
        key_i = (rg.rr + gm.ws - 1) * (2 * gm.ws - 1) + rg.cc + gm.ws - 1;
        col0 = GEN ? (L == 128 ? 0 : (row / L) * L) : rg.g * L;   // GEN with L = 32: the warp's own 32-column band
        if (tr) WTRACE(g_trace_fwd, k, 6);
      }
      const float* tab = s_tab + sub * (TAB_MAX + 1);
      float s[L];
      float mx = -INFINITY;
      float sum = 0.f;
      constexpr int CH = (L >= 32) ? 32 : 16;
      if constexpr (WS > 0) {
        // ---- fast path: compile-time column map, instantiated per token order of the row's window
        auto softmax_fast = [&](auto quad_tag) {
          constexpr bool QUAD = decltype(quad_tag)::value;
          constexpr int NQ = QUAD ? 4 : 1;
          constexpr int LW = LWT;                      // real columns of the window (e.g. 98 of 128 for 7x7x2)
          constexpr int RA = (WS + 1) / 2;             // rows / columns of the first rectangle pair
          const float* tp = tab + key_i;
          float mq[NQ];
#pragma unroll
          for (int q = 0; q < NQ; ++q) mq[q] = -INFINITY;
          mbar_wait(s_full, u & 1);
          tc_fence_after();
          if (tr) WTRACE(g_trace_fwd, k, 7);
#pragma unroll
          for (int cb = 0; cb < L / CH; ++cb) {
            uint32_t v[32];
            tmem_ld_row_chunk<L>(tmem_S, t_lane, col0, cb, wq, lane, v);
#pragma unroll
            for (int jj = 0; jj < CH; ++jj) {
              const int j = cb * CH + jj;
              if (j < LW) {                            // compile-time: padding columns are never touched
                const float x = fmaf(__uint_as_float(v[jj]), gm.scale_log2e, tp[-col_key<LW, WS, QUAD>(j)]);
                s[j] = x;
                mq[col_rect<LW, WS, QUAD>(j)] = fmaxf(mq[col_rect<LW, WS, QUAD>(j)], x);
              }
            }
          }
          // S is in registers: the next unit's QK^T may overwrite TMEM now
          tc_fence_before();
          mbar_arrive(s_free);
          if (tr) WTRACE(g_trace_fwd, k, 8);
          // shift mask (swin_512.py:171-192): a window of the last window row / column holds two bands
          // per wrapping axis; tokens of different bands get -100.  In quadrant order the band pair
          // of a token IS its quadrant, so the mask is one additive constant per quadrant of columns.
          float nq[NQ];
          if constexpr (QUAD) {
            const int q_i = (rg.rr >= RA ? 2 : 0) | (rg.cc >= RA ? 1 : 0);
            const int wm = (rg.id >= 3 ? 2 : 0) | (rg.id % 3 != 0 ? 1 : 0);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              nq[q] = ((q ^ q_i) & wm) ? kMaskLog2e : 0.f;
              mx = fmaxf(mx, mq[q] + nq[q]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) nq[q] -= mx;
          } else {
            mx = mq[0];
            nq[0] = -mx;
          }
          mbar_wait(pv_done, (u & 1) ^ 1);        // the previous P V product has finished reading P
          if (tr) WTRACE(g_trace_fwd, k, 9);
          if (LW < L && !rg.inrange) return;      // padding row of the slot: its P row stays zero
#pragma unroll
          for (int j8 = 0; j8 < (LW + 7) / 8; ++j8) {
            uint32_t w[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const int j = j8 * 8 + 2 * h;
              float p0 = 0.f, p1 = 0.f;
              if (j < LW) p0 = fast_exp2(s[j] + nq[col_rect<LW, WS, QUAD>(j)]);
              if (j + 1 < LW) p1 = fast_exp2(s[j + 1] + nq[col_rect<LW, WS, QUAD>(j + 1)]);
              sum += p0 + p1;
              w[h] = pack_bf16(p0, p1);
            }
            const int col = col0 + j8 * 8;
            *reinterpret_cast<uint4*>(s_p + (col >> 6) * SLOT_BYTES + sw128_offset(row, (col & 63) >> 3)) =
                make_uint4(w[0], w[1], w[2], w[3]);
          }
        };
        // a warp never straddles two windows for L >= 32, so the branch is warp-uniform
        if (ORDER == 0 || !rg.wraps) softmax_fast(std::false_type{});
        else                         softmax_fast(std::true_type{});
      } else {
        // ---- generic path: per-column look-up table (any order, dense mask, window tags)
        named_bar_sync(1, 128);                  // everybody is done with the previous LUT
        const uint32_t my_tag = rg.inrange ? uint32_t(rg.g + 1) : 0u;
        s_lut[row] = uint32_t(rg.rr * (2 * gm.ws - 1) + rg.cc) | (uint32_t(rg.id) << 8) |
                     (uint32_t(rg.rr * gm.ws + rg.cc) << 16) | (my_tag << 24);
        named_bar_sync(1, 128);
        const bool use_mask = rg.wraps;
        // dense mask row of this query token (stand-alone WindowAttention with an explicit mask tensor)
        const float* mask_row =
            gm.mask ? gm.mask + ((size_t)(rg.gw % gm.mask_nw) * gm.N + (rg.rr * gm.ws + rg.cc)) * gm.N : nullptr;
        mbar_wait(s_full, u & 1);
        tc_fence_after();
#pragma unroll
        for (int cb = 0; cb < L / CH; ++cb) {
          uint32_t v[32];
          tmem_ld_row_chunk<L>(tmem_S, t_lane, col0, cb, wq, lane, v);
#pragma unroll
          for (int jj = 0; jj < CH; ++jj) {
            const uint32_t lj = s_lut[col0 + cb * CH + jj];
            float x = fmaf(__uint_as_float(v[jj]), gm.scale_log2e, tab[key_i - int(lj & 0xff)]);
            if (use_mask && ((lj >> 8) & 0xffu) != uint32_t(rg.id)) x += kMaskLog2e;
            if (mask_row != nullptr) x = fmaf(__ldg(mask_row + ((lj >> 16) & 0xffu)), 1.4426950408889634f, x);
            if (GEN && (lj >> 24) != my_tag) x = -1.0e30f;        // another window's column, or padding
            s[cb * CH + jj] = x;
            mx = fmaxf(mx, x);
          }
        }
        tc_fence_before();
        mbar_arrive(s_free);
        mbar_wait(pv_done, (u & 1) ^ 1);
#pragma unroll
        for (int j8 = 0; j8 < L / 8; ++j8) {
          uint32_t w[4];
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            float p0 = fast_exp2(s[j8 * 8 + 2 * h] - mx);
            float p1 = fast_exp2(s[j8 * 8 + 2 * h + 1] - mx);
            if (GEN && !rg.inrange) { p0 = 0.f; p1 = 0.f; }          // padding row: keep P finite and empty
            sum += p0 + p1;
            w[h] = pack_bf16(p0, p1);
          }
          const int col = col0 + j8 * 8;
          *reinterpret_cast<uint4*>(s_p + (col >> 6) * SLOT_BYTES + sw128_offset(row, (col & 63) >> 3)) =
              make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
      // 1/rowsum for the epilogue warps: slot (item parity, head of the group), read after p_full
      s_inv[((k & 1) * 2 + sub) * 128 + row] = !rg.inrange ? 0.f : 1.0f / sum;     // padding rows of a slot: nothing to scale
      if (sub == SH - 1) mbar_arrive(&inv_full[k & 1]);
      fence_proxy_async_smem();
      mbar_arrive(p_full);
      if (tr) WTRACE(g_trace_fwd, k, 10);
      if (rg.inrange) lse2[((size_t)tile * gm.nH + head) * 128 + rg.canon] = mx + log2f(sum);
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 160;");
    // ---------------------------------------------------------------- epilogue warps (group B)
    // drain O of every item: O * (1/rowsum) -> bf16 -> whole 128-byte lines of `out` at the un-rolled
    // token index of each row (window_reverse + inverse roll, swin_512.py:224-231)
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const uint32_t t_lane = uint32_t(wq * 32) << 16;
    uint8_t* stage = s_stage + (warp - 8) * 4096;
    const bool tr = (threadIdx.x == 256);
    (void)tr;
    for (int k = 0; k < n_local; ++k) {
      const int item = int(blockIdx.x) + k * int(gridDim.x);
      const int tile = item / gm.ngrp;
      RowGeom rg;
      if constexpr (WS > 0) rg = row_geom_fast<L, WS, ORDER, LWT>(gm, tile, row);
      else                  rg = row_geom(gm, tile, row);
      const long tok = rg.valid ? rg.tok : -1;
      uint8_t* rowp[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long t = __shfl_sync(0xffffffffu, tok, i * 4 + (lane >> 3));
        rowp[i] = t < 0 ? nullptr : reinterpret_cast<uint8_t*>(out + t * gm.C + hg * gm.gch);
      }
      // 1/rowsum of every head of this item (the softmax warps cannot overwrite the slot before the
      // P V of item k+1 starts, which waits for this warp's o_free)
      mbar_wait(&inv_full[k & 1], (k >> 1) & 1);
      const float inv0 = s_inv[((k & 1) * 2 + 0) * 128 + row];
      const float inv1 = s_inv[((k & 1) * 2 + (SH - 1)) * 128 + row];
      mbar_wait(o_full, k & 1);
      tc_fence_after();
      if (tr) WTRACE(g_trace_fwd, k, 11);
      for (int c = 0; c < nc; ++c) {
        uint32_t v0[32], v1[32];
        // SH == 1: columns [c*64, +64) of this head.  SH == 2: columns [0,32) of head 0's product
        // and columns [32,64) of head 1's product (each product spans the whole 64-channel chunk).
        tmem_ld32(tmem_O + t_lane + (SH == 1 ? c * 64 : 0), v0);
        tmem_ld32(tmem_O + t_lane + (SH == 1 ? c * 64 + 32 : 64 + 32), v1);
        tmem_ld_wait();
        if (c == nc - 1) {
          tc_fence_before();
          mbar_arrive(o_free);
        }
        uint4 vals[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          vals[j] = make_uint4(pack_bf16(__uint_as_float(v0[8 * j + 0]) * inv0, __uint_as_float(v0[8 * j + 1]) * inv0),
                               pack_bf16(__uint_as_float(v0[8 * j + 2]) * inv0, __uint_as_float(v0[8 * j + 3]) * inv0),
                               pack_bf16(__uint_as_float(v0[8 * j + 4]) * inv0, __uint_as_float(v0[8 * j + 5]) * inv0),
                               pack_bf16(__uint_as_float(v0[8 * j + 6]) * inv0, __uint_as_float(v0[8 * j + 7]) * inv0));
          vals[4 + j] = make_uint4(pack_bf16(__uint_as_float(v1[8 * j + 0]) * inv1, __uint_as_float(v1[8 * j + 1]) * inv1),
                                   pack_bf16(__uint_as_float(v1[8 * j + 2]) * inv1, __uint_as_float(v1[8 * j + 3]) * inv1),
                                   pack_bf16(__uint_as_float(v1[8 * j + 4]) * inv1, __uint_as_float(v1[8 * j + 5]) * inv1),
                                   pack_bf16(__uint_as_float(v1[8 * j + 6]) * inv1, __uint_as_float(v1[8 * j + 7]) * inv1));
        }
        uint8_t* rp[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) rp[i] = rowp[i] ? rowp[i] + c * 128 : nullptr;
        warp_store_rows<8>(stage, vals, rp, lane);
      }
      if (tr) WTRACE(g_trace_fwd, k, 12);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace

int fill_geom(WinGeom* gm, int B, int T, int H, int W, int C, int nH, int ws, int shift, float qk_scale,
              const float* mask, int mask_windows) {
  STSWIN_CHECK_ARG(B > 0 && T > 0 && H > 0 && W > 0 && C > 0 && nH > 0 && ws > 0, "winattn: non-positive dimension");
  STSWIN_CHECK_ARG(H % ws == 0 && W % ws == 0, "winattn: H=%d, W=%d must be multiples of the window size %d", H, W, ws);
  STSWIN_CHECK_ARG(C % nH == 0, "winattn: C=%d not divisible by num_heads=%d", C, nH);
  gm->B = B; gm->T = T; gm->H = H; gm->W = W; gm->C = C; gm->nH = nH; gm->ws = ws; gm->shift = shift;
  gm->hd = C / nH;
  gm->N = ws * ws;
  gm->L = T * ws * ws;
  if (!((gm->hd % 64 == 0 && gm->hd <= 256) || (gm->hd == 32 && nH % 2 == 0)))
    return set_error(kErrUnsupported, "winattn: head_dim %d unsupported (need 32 or a multiple of 64, <= 256)", gm->hd);
  if (gm->L > 128 || gm->L < 1)
    return set_error(kErrUnsupported, "winattn: T*ws*ws = %d tokens per window unsupported (need <= 128)", gm->L);
  if (shift < 0 || shift >= ws)
    return set_error(kErrInvalidArg, "winattn: shift %d must be in [0, window_size = %d)", shift, ws);
  if (ws > 8) return set_error(kErrUnsupported, "winattn: window size %d > 8 unsupported", ws);
  gm->general = !(gm->L == 16 || gm->L == 32 || gm->L == 64 || gm->L == 128);
  // rows per window slot of a tile: windows of more than 16 tokens start at a power-of-two row (49 -> 64, 25 -> 32, 98 -> 128)
  gm->slot = gm->L;
  if (gm->L > 16) { gm->slot = 32; while (gm->slot < gm->L) gm->slot *= 2; }
  gm->G = 128 / gm->slot;
  gm->nWh = H / ws; gm->nWw = W / ws; gm->nW = gm->nWh * gm->nWw;
  gm->total_windows = B * gm->nW;
  gm->num_tiles = (gm->total_windows + gm->G - 1) / gm->G;
  gm->SH = gm->hd >= 64 ? 1 : 64 / gm->hd;
  gm->ngrp = nH / gm->SH;
  gm->gch = gm->SH * gm->hd;
  gm->nc = gm->gch / 64;
  gm->scale_log2e = qk_scale > 0.f ? qk_scale * 1.4426950408889634f : 1.4426950408889634f / sqrtf((float)gm->hd);
  gm->scale = qk_scale > 0.f ? qk_scale : 1.0f / sqrtf((float)gm->hd);
  gm->ra = ws - shift; gm->rb = shift;
  {
    int off = 0;
    for (int k = 0; k < 4; ++k) {
      gm->roff[k] = off;
      off += ((k >> 1) ? gm->rb : gm->ra) * ((k & 1) ? gm->rb : gm->ra) * T;
    }
    gm->roff[4] = off;       // == L
  }
  gm->uniform_quad = 0;
  gm->perm = 0;
  gm->mask = mask; gm->mask_nw = mask_windows;
  // exact multiply-shift division of window indices (row_geom_fast)
  if ((unsigned long long)gm->total_windows * (unsigned long long)gm->nW >= (1ull << 32))
    return set_error(kErrUnsupported, "winattn: %d windows exceed the supported index range", gm->total_windows);
  gm->mg_nW = ((1ull << 32) + gm->nW - 1) / gm->nW;
  gm->mg_nWw = ((1ull << 32) + gm->nWw - 1) / gm->nWw;
  STSWIN_CHECK_ARG(mask == nullptr || mask_windows > 0, "winattn: mask given with mask_windows <= 0");
  return kOk;
}

// tensor maps over a [B*T, H, W, channels] bf16 tensor: whole-window box and the four rectangle boxes
int make_window_tmaps(WinMaps* maps, const void* base, const WinGeom& gm, int channels) {
  uint64_t dims[4] = {(uint64_t)channels, (uint64_t)gm.W, (uint64_t)gm.H, (uint64_t)gm.B * gm.T};
  uint64_t str[3] = {(uint64_t)channels * 2, (uint64_t)gm.W * channels * 2, (uint64_t)gm.H * gm.W * channels * 2};
  uint32_t box_full[4] = {64, (uint32_t)gm.ws, (uint32_t)gm.ws, (uint32_t)gm.T};
  int rc = make_tmap(&maps->full, TmapDtype::BF16, 4, base, dims, str, box_full, true);
  if (rc != kOk) return rc;
  for (int k = 0; k < 4; ++k) {
    maps->rect[k] = maps->full;
    if (gm.shift > 0) {
      uint32_t box[4] = {64, (uint32_t)((k & 1) ? gm.rb : gm.ra), (uint32_t)((k >> 1) ? gm.rb : gm.ra), (uint32_t)gm.T};
      if ((rc = make_tmap(&maps->rect[k], TmapDtype::BF16, 4, base, dims, str, box, true)) != kOk) return rc;
    }
  }
  return kOk;
}

long winattn_lse_elems(int B, int T, int H, int W, int C, int nH, int ws) {
  WinGeom gm;
  if (fill_geom(&gm, B, T, H, W, C, nH, ws, 0, 0.f, nullptr, 0) != kOk) return -1;
  return (long)gm.num_tiles * gm.nH * 128;
}

#ifdef STSWIN_TRACE
extern "C" int stswin_debug_trace_fwd(long long* buf) {
  return cudaMemcpyToSymbol(g_trace_fwd, &buf, sizeof(buf)) == cudaSuccess ? 0 : -1;
}
#endif

// see include/stswin_b200.h : stswin_winattn_fwd
int winattn_fwd(const void* qkv, const float* bias_table, void* out, float* lse2, int B, int T, int H, int W, int C,
                int nH, int ws, int shift, float qk_scale, const float* mask, int mask_windows, cudaStream_t stream) {
  STSWIN_CHECK_ARG(qkv && bias_table && out && lse2, "winattn_fwd: null pointer");
  WinGeom gm;
  int rc = fill_geom(&gm, B, T, H, W, C, nH, ws, shift, qk_scale, mask, mask_windows);
  if (rc != kOk) return rc;
  STSWIN_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 15) == 0, "winattn_fwd: out must be 16-byte aligned");
  WinMaps tq;
  if ((rc = make_window_tmaps(&tq, qkv, gm, 3 * C)) != kOk) return rc;
  return dispatch_variant(select_variant(gm, false), [&](auto v) {
    using V = decltype(v);
    return launch_winattn(winattn_fwd_kernel<V::L, V::WS, V::ORDER, V::GEN, V::LWT>, gm, NUM_THREADS, SMEM_BYTES, stream,
                          tq, static_cast<__nv_bfloat16*>(out), bias_table, lse2, gm);
  });
}

}  // namespace stswin
