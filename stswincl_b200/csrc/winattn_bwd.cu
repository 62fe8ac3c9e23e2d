// K3 backward: gradient of the spatio-temporal shifted-window attention core.
//
// Autograd twin of winattn_fwd.cu for the op sequence seg18/net/Ours/swin_512.py:119-138 wrapped
// by the gather/scatter of :210-231.  Per (tile, head), with S2 = scale*log2e*QK^T + (bias+mask)*log2e:
//   P  = exp2(S2 - lse2)                    (recomputed, never stored between passes)
//   dP = dO V^T
//   dS = P o (dP - rowsum(P o dP))
//   dV = P^T dO      dQ = scale * dS K      dK = scale * dS^T Q
//   d relative_position_bias_table[idx(i,j), head] += dS[i,j]       (:122-125, summed over windows,
//                                                                     batch and the TxT tiling)
// Inputs  qkv [B,T,H,W,3C] bf16, d_out [B,T,H,W,C] bf16, lse2 from the forward.
// Outputs d_qkv [B,T,H,W,3C] bf16 (scattered to the un-rolled coordinates by TMA),
//         d_table [(2ws-1)^2, nH] fp32 (+=), optional d_qkv_colsum [3C] fp32 (+=, the qkv bias grad).
//
// Streaming: operand chunks [128 rows x 64 ch] flow through 16 KB ring slots twice -- once from
// HBM for S and dP (ring H, producer warp 0), once more from L2 for the three output products
// (ring L, producer warp 2).  (One shared in-order ring was tried twice: it chains the two passes into
// one HBM/L2 latency after the other on the MMA warp's critical path.)  S, two dP buffers and two
// 64-column output accumulators live in TMEM.
// Four warpgroups (setmaxnreg): producers + MMA issuer (warp-uniform control flow, one elected lane
// issues) / softmax-backward (one thread per tile row, 232 registers) / two drain groups that
// alternate the output products (TMEM -> bf16 -> 256-bit stores to the row's own line of d_qkv:
// the scatter is the row's token index, no staging buffer).
// The bias-table gradient needs the sum of dS over every item this CTA processes: on the fast path
// each softmax-backward thread (= query row) keeps N = ws*ws fp32 running sums, one per key position
// (the TxT tiling folds onto the same entry), together with the row's N bias values, and bins them by
// relative position into shared memory whenever the row's own position changes (windows that wrap
// use quadrant token order, interior windows row-major) and at the end -- no per-element atomics in
// the main loop and no bf16 rounding inside a sum that cancels heavily; every CTA sees ONE head
// group (grid % ngrp == 0).  Generic / general paths: shared-memory atomics per element.
// (A first version accumulated bf16 dS on the tensor core through an identity tile; its rounding
// noise reached 6% of the gradient for a 6-window batch.)
#include <type_traits>

#include "winattn_common.cuh"
#include "host_util.h"
#include "kernels.h"

namespace stswin {

namespace {

constexpr int NRH = 5;                         // ring H: first-pass chunks, streamed from HBM
constexpr int NRL = 4;                         // ring L: second-pass chunks, re-read from L2
constexpr int PD_BYTES = 2 * SLOT_BYTES;       // [128 x 128] bf16 as two K-major halves
constexpr int NUM_THREADS = 512;               // warpgroup 0: producers H / L, MMA issuer; 1: softmax backward; 2, 3: drain
constexpr int SMEM_BYTES = 1024 + (NRH + NRL) * SLOT_BYTES + 2 * PD_BYTES + 128 * 4 +
                           4 * (TAB_MAX + 1) * 4 + 256;
STSWIN_TRACE_DECL(g_trace_bwd)

// L, WS, ORDER, GEN, LWT as in the forward kernel, with the same instantiations; WS > 0 also sums the
// bias-table gradient in registers.  SHT: heads per 64-channel group (2 when head_dim is 32).
template <int L, int WS, int ORDER, int SHT, bool GEN, int LWT>
__global__ void __launch_bounds__(NUM_THREADS, 1)
winattn_bwd_kernel(const __grid_constant__ WinMaps tm_qkv, const __grid_constant__ WinMaps tm_do,
                   __nv_bfloat16* __restrict__ d_qkv, const float* __restrict__ bias_table, const float* __restrict__ lse2, float* __restrict__ d_table,
                   float* __restrict__ d_colsum, const WinGeom gm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint8_t* s_ringh = smem;
  uint8_t* s_ringl = s_ringh + NRH * SLOT_BYTES;
  uint8_t* s_p = s_ringl + NRL * SLOT_BYTES;
  uint8_t* s_ds = s_p + PD_BYTES;
  uint32_t* s_lut = reinterpret_cast<uint32_t*>(s_ds + PD_BYTES);
  float* s_tab = reinterpret_cast<float*>(s_lut + 128);   // [2][TAB_MAX + 1] bias * log2e, one table per head of the group
  float* s_bacc = s_tab + 2 * (TAB_MAX + 1);              // [2][TAB_MAX + 1] bias-table gradient bins of this CTA
  static_assert(((128 + 4 * (TAB_MAX + 1)) * 4) % 8 == 0, "mbarriers need 8-byte alignment");
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_bacc + 2 * (TAB_MAX + 1));
  uint64_t* fullh = bars;
  uint64_t* emptyh = fullh + NRH;
  uint64_t* fulll = emptyh + NRH;
  uint64_t* emptyl = fulll + NRL;
  uint64_t* sdp_full = emptyl + NRL;    // S and dP of a unit complete (tensor core)
  uint64_t* s_free = sdp_full + 1;      // S read out (after pass 1)
  uint64_t* dp_free = sdp_full + 2;     // [2] dP buffer read out (after pass 2)
  uint64_t* pds_full = sdp_full + 4;    // P and dS of a unit in shared memory
  uint64_t* p_free = sdp_full + 5;      // the dV products have read P
  uint64_t* ds_free = sdp_full + 6;     // the dQ / dK products have read dS
  uint64_t* obuf_full = sdp_full + 7;   // [2]
  uint64_t* obuf_free = sdp_full + 9;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sdp_full + 11);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_items = gm.num_tiles * gm.ngrp;     // work item = (tile, head group)
  const int nc = gm.nc;
  const int hg = blockIdx.x % gm.ngrp;          // head group, constant per CTA: gridDim.x % ngrp == 0
  constexpr int SH = SHT;                       // heads per group (2 when head_dim is 32)
  const int n_local = (num_items - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x);
  const int n_units = n_local * SH;             // unit = (item, head of the group)
  const int nbias = (2 * gm.ws - 1) * (2 * gm.ws - 1);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_qkv.full);
    tma_prefetch_desc(&tm_do.full);
    for (int i = 0; i < NRH; ++i) {
      mbar_init(&fullh[i], 1);
      mbar_init(&emptyh[i], 1);
    }
    for (int i = 0; i < NRL; ++i) {
      mbar_init(&fulll[i], 1);
      mbar_init(&emptyl[i], 1);
    }
    mbar_init(sdp_full, 1);
    mbar_init(s_free, 128);
    mbar_init(&dp_free[0], 128);
    mbar_init(&dp_free[1], 128);
    mbar_init(pds_full, 128);
    mbar_init(p_free, 1);
    mbar_init(ds_free, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&obuf_full[i], 1);
      mbar_init(&obuf_free[i], 128);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  // P / dS: entries outside a row's own window stay zero.  Rings: the padding rows of a tile (general
  // mode) are never written by TMA and must read as zero.
  for (int i = threadIdx.x; i < ((NRH + NRL) * SLOT_BYTES + 2 * PD_BYTES) / 16; i += NUM_THREADS)
    reinterpret_cast<uint4*>(s_ringh)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 2 * (TAB_MAX + 1); i += NUM_THREADS) s_bacc[i] = 0.f;
  pdl_wait();                // programmatic dependent launch: everything above overlapped the previous kernel's tail
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < SH * nbias; i += NUM_THREADS) {
    const int sub = i / nbias, k = i - sub * nbias;
    s_tab[sub * (TAB_MAX + 1) + k] = __ldg(bias_table + k * gm.nH + hg * SH + sub) * 1.4426950408889634f;
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base;            // 128 columns
  const uint32_t tmem_dP = tmem_base + 128;     // two 128-column buffers (units alternate)
  const uint32_t tmem_out = tmem_base + 384;    // two 64-column output accumulators

  if (warp < 4) {
   asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
   if (warp == 0 || warp == 2) {
    // ---------------------------------------------------------------- TMA producers (all lanes issue boxes)
    // ring H (warp 0): per 64-channel chunk c: Q_c K_c dO_c V_c      -> S, dP
    // ring L (warp 2): dO_0.. (dV), then per c: K_c (dQ_c) Q_c (dK_c) -> re-read from L2
    const bool ring_h = (warp == 0);
    uint8_t* ring = ring_h ? s_ringh : s_ringl;
    uint64_t* fullb = ring_h ? fullh : fulll;
    uint64_t* emptyb = ring_h ? emptyh : emptyl;
    const int nslot = ring_h ? NRH : NRL;
    int slot = 0;
    uint32_t phase = 0;
    auto load = [&](int tile, bool from_do, int ch0) {
      mbar_wait(&emptyb[slot], phase ^ 1);
      if (lane == 0) mbar_arrive_expect_tx(&fullb[slot], chunk_tx_bytes(gm));
      __syncwarp();
      tile_boxes<true>(gm, tile, ch0, ring + slot * SLOT_BYTES, from_do ? &tm_do : &tm_qkv, &fullb[slot], lane);
      if (++slot == nslot) { slot = 0; phase ^= 1; }
    };
    for (int k = 0; k < n_local; ++k) {
      const int item = int(blockIdx.x) + k * int(gridDim.x);
      const int tile = item / gm.ngrp;
      const int hq = hg * gm.gch;
      if (lane == 0) WTRACE(g_trace_bwd, k, ring_h ? 0 : 2);
      if (ring_h) {
        for (int c = 0; c < nc; ++c) {
          load(tile, false, 0 * gm.C + hq + c * 64);   // Q_c
          load(tile, false, 1 * gm.C + hq + c * 64);   // K_c
          load(tile, true, hq + c * 64);               // dO_c
          load(tile, false, 2 * gm.C + hq + c * 64);   // V_c
        }
      } else {
        for (int c = 0; c < nc; ++c) load(tile, true, hq + c * 64);   // dO_c -> dV_c
        for (int c = 0; c < nc; ++c) {
          load(tile, false, 1 * gm.C + hq + c * 64);   // K_c  -> dQ_c
          load(tile, false, 0 * gm.C + hq + c * 64);   // Q_c  -> dK_c
        }
      }
      if (lane == 0) WTRACE(g_trace_bwd, k, ring_h ? 1 : 3);
    }
   } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    // warp-uniform control flow (descriptors stay in uniform registers); one elected lane issues.
    const bool leader = elect_one();
    constexpr uint32_t idesc_kk = umma_idesc_bf16(128, 128, 0, 0);   // S, dP
    constexpr uint32_t idesc_kn = umma_idesc_bf16(128, 64, 0, 1);    // dQ = dS K
    constexpr uint32_t idesc_nn = umma_idesc_bf16(128, 64, 1, 1);    // dV = P^T dO, dK = dS^T Q
    const uint32_t p_addr = smem_u32(s_p), ds_addr = smem_u32(s_ds);
    const uint32_t rh_addr = smem_u32(s_ringh), rl_addr = smem_u32(s_ringl);
    uint32_t seq_h = 0, seq_l = 0, base_h = 0, base_l = 0;   // running chunk counters of the two rings
    uint32_t nout = 0;                                        // output products issued so far (buffer = nout & 1)
    auto issue_SdP = [&](int u) {
      const int sub = (SH == 1) ? 0 : (u & 1);
      const int b = u & 1;                                    // dP buffer of this unit
      mbar_wait(s_free, (u & 1) ^ 1);                         // pass 1 of the previous unit has read S
      mbar_wait(&dp_free[b], ((u >> 1) & 1) ^ 1);             // pass 2 of unit u-2 has read this dP buffer
      tc_fence_after();
      if (sub == 0) { base_h = seq_h; seq_h += 4 * nc; }
      // with two heads per chunk only the head's 32-channel K range (two k-steps)
      const int k0 = (SH == 1) ? 0 : sub * 2, k1 = (SH == 1) ? 4 : sub * 2 + 2;
      for (int c = 0; c < nc; ++c) {
#pragma unroll
        for (int pair = 0; pair < 2; ++pair) {     // (Q_c, K_c) -> S ; (dO_c, V_c) -> dP
          const uint32_t na = base_h + 4 * c + 2 * pair, nb = na + 1;
          const uint32_t sa = na % NRH, sb = nb % NRH;
          if (sub == 0) {
            mbar_wait(&fullh[sa], (na / NRH) & 1);
            mbar_wait(&fullh[sb], (nb / NRH) & 1);
          }
          tc_fence_after();
          const uint32_t aa = rh_addr + sa * SLOT_BYTES, ba = rh_addr + sb * SLOT_BYTES;
          if (leader) {
            for (int kk = k0; kk < k1; ++kk)
              umma_bf16(pair == 0 ? tmem_S : tmem_dP + b * 128, umma_smem_desc(aa + kk * 32, 16, 1024),
                        umma_smem_desc(ba + kk * 32, 16, 1024), idesc_kk, (c > 0 || kk > k0) ? 1u : 0u);
            if (sub == SH - 1) {
              umma_commit(&emptyh[sa]);
              umma_commit(&emptyh[sb]);
            }
          }
        }
      }
      if (leader) {
        umma_commit(sdp_full);
        WTRACE(g_trace_bwd, (SH == 1 ? u : u >> 1), 4);
      }
      __syncwarp();
    };
    auto issue_out = [&](int u) {
      const int sub = (SH == 1) ? 0 : (u & 1);
      mbar_wait(pds_full, u & 1);
      tc_fence_after();
      if (leader) WTRACE(g_trace_bwd, (SH == 1 ? u : u >> 1), 5);
      if (sub == 0) { base_l = seq_l; seq_l += 3 * nc; }
      // products in ring-L order: dV_0 .. dV_{nc-1}, then dQ_c, dK_c per chunk (whole 64-channel chunks)
      for (int n = 0; n < 3 * nc; ++n) {
        const int o = n < nc ? 0 : 1 + ((n - nc) & 1);        // 0: dV, 1: dQ, 2: dK
        const uint32_t nl = base_l + n, sl = nl % NRL;
        const uint32_t ob = nout & 1;
        if (sub == 0) mbar_wait(&fulll[sl], (nl / NRL) & 1);
        mbar_wait(&obuf_free[ob], ((nout >> 1) & 1) ^ 1);     // the drain warps have emptied this accumulator
        tc_fence_after();
        const uint32_t xa = rl_addr + sl * SLOT_BYTES;
        const uint32_t dst = tmem_out + ob * 64;
        if (leader) {
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const uint64_t bdesc = umma_smem_desc(xa + kk * 2048, SLOT_BYTES, 1024);   // [rows x 64ch], MN-major
            if (o == 0)        // dV = P^T dO : A = P viewed MN-major (m = key), k = query
              umma_bf16(dst, umma_smem_desc(p_addr + kk * 2048, SLOT_BYTES, 1024), bdesc, idesc_nn, kk > 0);
            else if (o == 1)   // dQ = dS K   : A = dS K-major, k = key
              umma_bf16(dst, umma_smem_desc(ds_addr + (kk >> 2) * SLOT_BYTES + (kk & 3) * 32, 16, 1024), bdesc,
                        idesc_kn, kk > 0);
            else               // dK = dS^T Q : A = dS viewed MN-major
              umma_bf16(dst, umma_smem_desc(ds_addr + kk * 2048, SLOT_BYTES, 1024), bdesc, idesc_nn, kk > 0);
          }
          if (sub == SH - 1) umma_commit(&emptyl[sl]);
          umma_commit(&obuf_full[ob]);
          if (n == nc - 1) umma_commit(p_free);               // P may be overwritten by the next unit's pass 1
        }
        ++nout;
      }
      if (leader) {
        umma_commit(ds_free);                                 // dS may be overwritten by the next unit's pass 2
        WTRACE(g_trace_bwd, (SH == 1 ? u : u >> 1), 6);
      }
      __syncwarp();
    };
    // S / dP of unit u+1 are issued before the output products of unit u: they run on the tensor
    // core while the softmax-backward warps are in pass 2 of unit u.
    if (n_units > 0) issue_SdP(0);
    for (int u = 0; u < n_units; ++u) {
      if (u + 1 < n_units) issue_SdP(u + 1);
      issue_out(u);
    }
   }
  } else if (warp < 8) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    // ---------------------------------------------------------------- softmax-backward warps (group A)
    // thread <-> tile row <-> TMEM lane.  pass 1: P = exp2(S2 - lse2) -> smem, delta = sum_j P dP.
    // pass 2: dS = P o (dP - delta) -> smem, bias-table gradient sums.
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const int cm_tid = threadIdx.x - 128;
    const uint32_t t_lane = uint32_t(wq * 32) << 16;
    const bool tr = (threadIdx.x == 128);
    (void)tr;
    constexpr int CH = (L >= 32) ? 32 : 16;
    constexpr int NCHUNK = L / CH;
    // fast path: per-row running sums of dS over every item of this CTA, one per key position (the TxT
    // tiling folds onto the same entry).  They are binned by relative position whenever the row's own
    // position changes (token order switch) and at the end of the kernel.  Two heads per group (SH == 2):
    // one set per head; the units alternate between the heads, so the two register arrays are SWAPPED
    // after every unit and the code always addresses `bacc` (no dynamic register indexing, one body).
    // The row's bias values are kept in registers too when there is one head per group.
    constexpr bool REG_BACC = (WS > 0);
    constexpr bool REG_BIAS = (WS > 0 && SH == 1);
    constexpr int NPOS = REG_BACC ? WS * WS : 1;
    constexpr int NPOS2 = (REG_BACC && SH == 2) ? NPOS : 1;
    constexpr int NBIAS = REG_BIAS ? NPOS : 1;
    float bacc[NPOS];                        // sums of the head of the current unit
    float bacc_o[NPOS2];                     // SH == 2: sums of the other head
    float breg[NBIAS];                       // bias * log2e of this row against every key position
#pragma unroll
    for (int i = 0; i < NPOS; ++i) bacc[i] = 0.f;
#pragma unroll
    for (int i = 0; i < NPOS2; ++i) bacc_o[i] = 0.f;
#pragma unroll
    for (int i = 0; i < NBIAS; ++i) breg[i] = 0.f;
    int bacc_key = -1;                       // key_i the sums / bias values belong to (-1: none)
    // (called between items, i.e. with `bacc` = head 0 and `bacc_o` = head 1)
    auto flush_bacc = [&]() {
      if constexpr (REG_BACC) {
        if (bacc_key >= 0) {
#pragma unroll
          for (int pos = 0; pos < NPOS; ++pos) {
            const int key = (pos / WS) * (2 * WS - 1) + pos % WS;
            if (bacc[pos] != 0.f) atomicAdd(&s_bacc[bacc_key - key], bacc[pos]);
            bacc[pos] = 0.f;
            if constexpr (SH == 2) {
              if (bacc_o[pos] != 0.f) atomicAdd(&s_bacc[(TAB_MAX + 1) + bacc_key - key], bacc_o[pos]);
              bacc_o[pos] = 0.f;
            }
          }
        }
      }
    };
    RowGeom rg;
    int key_i = 0, col0 = 0;
    for (int u = 0; u < n_units; ++u) {
      const int sub = (SH == 1) ? 0 : (u & 1);
      const int k = (SH == 1) ? u : (u >> 1);
      const int item = int(blockIdx.x) + k * int(gridDim.x);
      const int tile = item / gm.ngrp;
      const int head = hg * SH + sub;
      const uint32_t tmem_dPu = tmem_dP + (u & 1) * 128;
      if (sub == 0) {
        if (tr) WTRACE(g_trace_bwd, k, 7);
        if constexpr (WS > 0) rg = row_geom_fast<L, WS, ORDER, LWT>(gm, tile, row);
        else                  rg = row_geom(gm, tile, row);
        key_i = (rg.rr + gm.ws - 1) * (2 * gm.ws - 1) + rg.cc + gm.ws - 1;
        col0 = GEN ? (L == 128 ? 0 : (row / L) * L) : rg.g * L;   // GEN with L = 32: the warp's own 32-column band
        if constexpr (REG_BACC) {
          if (key_i != bacc_key) {           // the row's own position changed (token-order switch)
            flush_bacc();
            bacc_key = key_i;
            if constexpr (REG_BIAS) {
#pragma unroll
              for (int pos = 0; pos < NPOS; ++pos) breg[pos] = s_tab[key_i - ((pos / WS) * (2 * WS - 1) + pos % WS)];
            }
          }
        }
      }
      const float* tab = s_tab + sub * (TAB_MAX + 1);
      float* bins = s_bacc + sub * (TAB_MAX + 1);
      // lse2 is indexed by the forward's tiling (natural window order): tile = window / G, row = (window % G)*L + ...
      // (fetching it one item ahead was measured: no gain -- the S / dP wait takes the stall over -- and 44-144 bytes of spills)
      const float lse_i = !rg.inrange ? 0.f
                          : lse2[((size_t)(rg.gw / gm.G) * gm.nH + head) * 128 + (rg.gw % gm.G) * gm.L + (rg.canon - rg.g * gm.L)];
      float delta = 0.f;

      if constexpr (WS > 0) {
        // ---- fast path: compile-time column map, instantiated per token order of the row's window
        auto softmax_bwd_fast = [&](auto quad_tag) {
          constexpr bool QUAD = decltype(quad_tag)::value;
          constexpr int LW = LWT;                      // real columns of the window (e.g. 98 of 128 for 7x7x2)
          constexpr int RA = (WS + 1) / 2;             // rows / columns of the first rectangle pair
          const float* tp = tab + key_i;
          // shift mask: one additive constant per quadrant of columns (see the forward kernel); folded with -lse
          float nq[4];
          if constexpr (QUAD) {
            const int q_i = (rg.rr >= RA ? 2 : 0) | (rg.cc >= RA ? 1 : 0);
            const int wm = (rg.id >= 3 ? 2 : 0) | (rg.id % 3 != 0 ? 1 : 0);
#pragma unroll
            for (int q = 0; q < 4; ++q) nq[q] = (((q ^ q_i) & wm) ? kMaskLog2e : 0.f) - lse_i;
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) nq[q] = -lse_i;
          }
          mbar_wait(sdp_full, u & 1);
          tc_fence_after();
          if (tr) WTRACE(g_trace_bwd, k, 8);
          // Both passes walk the row's L columns in pieces of CW columns.  With two frames per 8x8 window
          // the columns of frame 1 repeat the key positions of frame 0 (row-major: 64 columns later;
          // quadrant order: 16 columns later inside each 32-column quadrant), so the frame loop stays ROLLED
          // and only half of the columns exist as straight-line code: the fully unrolled 128-column bodies did
          // not fit the instruction cache (30 % of this warp's stall samples were instruction fetch).
          constexpr bool ROLL = (L == 128 && WS == 8);
          constexpr int CW = (ROLL && QUAD) ? 16 : 32;          // columns per piece (one TMEM load)
          constexpr int NPIECE = ROLL ? (64 / CW) : NCHUNK;     // unrolled pieces per frame (ROLL) / per row
          constexpr int NFR = ROLL ? 2 : 1;                     // rolled iterations
          // piece pc of rolled iteration fr: first column in the row, and the column the compile-time maps use
          auto piece_col = [](int fr, int pc) { return !ROLL ? pc * 32 : (QUAD ? pc * 32 + fr * 16 : fr * 64 + pc * 32); };
          auto piece_map = [](int pc) { return (ROLL && QUAD) ? pc * 32 : pc * 32; };
          static_assert(L >= 32, "fast path: 32-column chunks");
          // pass 1
#pragma unroll 1
          for (int fr = 0; fr < NFR; ++fr)
#pragma unroll
          for (int pc = 0; pc < NPIECE; ++pc) {
            const int cc0 = piece_col(fr, pc);                 // runtime when rolled
            const int jb = piece_map(pc);                      // compile-time
            uint32_t v[CW], w[CW];
            if constexpr (CW == 32) {
              tmem_ld32(tmem_S + t_lane + col0 + cc0, v);      // both loads in flight, one wait
              tmem_ld32(tmem_dPu + t_lane + col0 + cc0, w);
            } else {
              tmem_ld16(tmem_S + t_lane + col0 + cc0, v);
              tmem_ld16(tmem_dPu + t_lane + col0 + cc0, w);
            }
            tmem_ld_wait();
            if (fr == 0 && pc == 0) {
              mbar_wait(p_free, (u & 1) ^ 1);                  // the previous unit's dV products have read P
              if (tr) WTRACE(g_trace_bwd, k, 13);
            }
#pragma unroll
            for (int j8 = 0; j8 < CW / 8; ++j8) {
              uint32_t pk[4];
#pragma unroll
              for (int h = 0; h < 4; ++h) {
                float pv[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const int jj = j8 * 8 + 2 * h + e, j = jb + jj;
                  pv[e] = 0.f;
                  if (j < LW) {                        // compile-time: padding columns stay zero
                    const float bias = REG_BIAS ? breg[REG_BIAS ? col_pos<LW, WS, QUAD>(j) : 0] : tp[-col_key<LW, WS, QUAD>(j)];
                    const float x = fmaf(__uint_as_float(v[jj]), gm.scale_log2e, bias);
                    pv[e] = fast_exp2(x + nq[col_rect<LW, WS, QUAD>(j)]);
                    if (LW < L && !rg.inrange) pv[e] = 0.f;    // padding row of the slot
                    delta = fmaf(pv[e], __uint_as_float(w[jj]), delta);
                  }
                }
                pk[h] = pack_bf16(pv[0], pv[1]);
              }
              const int col = col0 + cc0 + j8 * 8;
              *reinterpret_cast<uint4*>(s_p + (col >> 6) * SLOT_BYTES + sw128_offset(row, (col & 63) >> 3)) =
                  make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
          }
          tc_fence_before();
          mbar_arrive(s_free);            // S may be overwritten by the next unit
          if (tr) WTRACE(g_trace_bwd, k, 9);
          // pass 2
          mbar_wait(ds_free, (u & 1) ^ 1);                     // the previous unit's dQ / dK products have read dS
          if (tr) WTRACE(g_trace_bwd, k, 14);
#pragma unroll 1
          for (int fr = 0; fr < NFR; ++fr)
#pragma unroll
          for (int pc = 0; pc < NPIECE; ++pc) {
            const int cc0 = piece_col(fr, pc);
            const int jb = piece_map(pc);
            uint32_t w[CW];
            if constexpr (CW == 32) tmem_ld32(tmem_dPu + t_lane + col0 + cc0, w);
            else                    tmem_ld16(tmem_dPu + t_lane + col0 + cc0, w);
            tmem_ld_wait();
#pragma unroll
            for (int j8 = 0; j8 < CW / 8; ++j8) {
              const int col = col0 + cc0 + j8 * 8;
              const uint32_t off = (col >> 6) * SLOT_BYTES + sw128_offset(row, (col & 63) >> 3);
              const uint4 pq = *reinterpret_cast<const uint4*>(s_p + off);
              const uint32_t pw[4] = {pq.x, pq.y, pq.z, pq.w};
              uint32_t dk[4];
#pragma unroll
              for (int h = 0; h < 4; ++h) {
                const int jj = j8 * 8 + 2 * h, j = jb + jj;
                const float2 pf = unpack_bf16(pw[h]);
                // rows of a padding window hold filler data: keep them out of the bias-table sum
                const float d0 = rg.valid ? pf.x * (__uint_as_float(w[jj]) - delta) : 0.f;
                const float d1 = rg.valid ? pf.y * (__uint_as_float(w[jj + 1]) - delta) : 0.f;
                dk[h] = pack_bf16(d0, d1);
                if constexpr (REG_BACC) {
                  if (j < LW) bacc[col_pos<LW, WS, QUAD>(j < LW ? j : 0)] += d0;
                  if (j + 1 < LW) bacc[col_pos<LW, WS, QUAD>(j + 1 < LW ? j + 1 : 0)] += d1;
                } else {
                  if (j < LW && d0 != 0.f) atomicAdd(&bins[key_i - col_key<LW, WS, QUAD>(j < LW ? j : 0)], d0);
                  if (j + 1 < LW && d1 != 0.f) atomicAdd(&bins[key_i - col_key<LW, WS, QUAD>(j + 1 < LW ? j + 1 : 0)], d1);
                }
              }
              *reinterpret_cast<uint4*>(s_ds + off) = make_uint4(dk[0], dk[1], dk[2], dk[3]);
            }
          }
        };
        // a warp never straddles two windows for L >= 32, so the branch is warp-uniform
        if (ORDER == 0 || !rg.wraps) softmax_bwd_fast(std::false_type{});
        else                         softmax_bwd_fast(std::true_type{});
      } else {
        // ---- generic path: per-column look-up table (any order, dense mask, window tags); the
        //      bias-table gradient goes through the shared bins (no static column -> position map)
        named_bar_sync(1, 128);                     // everybody is done with the previous LUT
        const uint32_t my_tag = rg.inrange ? uint32_t(rg.g + 1) : 0u;
        s_lut[row] = uint32_t(rg.rr * (2 * gm.ws - 1) + rg.cc) | (uint32_t(rg.id) << 8) |
                     (uint32_t(rg.rr * gm.ws + rg.cc) << 16) | (my_tag << 24);
        named_bar_sync(1, 128);
        const bool use_mask = rg.wraps;
        // dense mask row of this query token (stand-alone WindowAttention with an explicit mask tensor)
        const float* mask_row =
            gm.mask ? gm.mask + ((size_t)(rg.gw % gm.mask_nw) * gm.N + (rg.rr * gm.ws + rg.cc)) * gm.N : nullptr;
        mbar_wait(sdp_full, u & 1);
        tc_fence_after();
#pragma unroll
        for (int cb = 0; cb < NCHUNK; ++cb) {
          uint32_t v[32], w[32];
          tmem_ld_row_chunk<L>(tmem_S, t_lane, col0, cb, wq, lane, v);
          tmem_ld_row_chunk<L>(tmem_dPu, t_lane, col0, cb, wq, lane, w);
          if (cb == 0) mbar_wait(p_free, (u & 1) ^ 1);
#pragma unroll
          for (int j8 = 0; j8 < CH / 8; ++j8) {
            uint32_t pk[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              float pv[2];
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const int jj = j8 * 8 + 2 * h + e;
                const uint32_t lj = s_lut[col0 + cb * CH + jj];
                float x = fmaf(__uint_as_float(v[jj]), gm.scale_log2e, tab[key_i - int(lj & 0xff)]);
                if (use_mask && ((lj >> 8) & 0xffu) != uint32_t(rg.id)) x += kMaskLog2e;
                if (mask_row != nullptr) x = fmaf(__ldg(mask_row + ((lj >> 16) & 0xffu)), 1.4426950408889634f, x);
                pv[e] = fast_exp2(x - lse_i);
                // general geometry: columns of another window (or padding) of this tile do not attend
                if (GEN && ((lj >> 24) != my_tag || my_tag == 0u)) pv[e] = 0.f;
                delta = fmaf(pv[e], __uint_as_float(w[jj]), delta);
              }
              pk[h] = pack_bf16(pv[0], pv[1]);
            }
            const int col = col0 + cb * CH + j8 * 8;
            *reinterpret_cast<uint4*>(s_p + (col >> 6) * SLOT_BYTES + sw128_offset(row, (col & 63) >> 3)) =
                make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
        tc_fence_before();
        mbar_arrive(s_free);
        mbar_wait(ds_free, (u & 1) ^ 1);
#pragma unroll
        for (int cb = 0; cb < NCHUNK; ++cb) {
          uint32_t w[32];
          tmem_ld_row_chunk<L>(tmem_dPu, t_lane, col0, cb, wq, lane, w);
#pragma unroll
          for (int j8 = 0; j8 < CH / 8; ++j8) {
            const int col = col0 + cb * CH + j8 * 8;
            const uint32_t off = (col >> 6) * SLOT_BYTES + sw128_offset(row, (col & 63) >> 3);
            const uint4 pq = *reinterpret_cast<const uint4*>(s_p + off);
            const uint32_t pw[4] = {pq.x, pq.y, pq.z, pq.w};
            uint32_t dk[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const int jj = j8 * 8 + 2 * h;
              const float2 pf = unpack_bf16(pw[h]);
              const float d0 = rg.valid ? pf.x * (__uint_as_float(w[jj]) - delta) : 0.f;
              const float d1 = rg.valid ? pf.y * (__uint_as_float(w[jj + 1]) - delta) : 0.f;
              dk[h] = pack_bf16(d0, d1);
              const uint32_t l0 = s_lut[col0 + cb * CH + jj], l1 = s_lut[col0 + cb * CH + jj + 1];
              if (d0 != 0.f) atomicAdd(&bins[key_i - int(l0 & 0xff)], d0);
              if (d1 != 0.f) atomicAdd(&bins[key_i - int(l1 & 0xff)], d1);
            }
            *reinterpret_cast<uint4*>(s_ds + off) = make_uint4(dk[0], dk[1], dk[2], dk[3]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&dp_free[u & 1]);     // this dP buffer may be overwritten (by unit u+2)
      fence_proxy_async_smem();
      mbar_arrive(pds_full);            // P / dS visible to the tensor core
      if (tr) WTRACE(g_trace_bwd, k, 10);
      if constexpr (REG_BACC && SH == 2) {   // the next unit belongs to the other head
#pragma unroll
        for (int pos = 0; pos < NPOS; ++pos) { const float t = bacc[pos]; bacc[pos] = bacc_o[pos]; bacc_o[pos] = t; }
      }
    }
    // ---- bias-table gradient: bin what is left in registers, then one global atomic per bin, CTA and head
    flush_bacc();
    named_bar_sync(1, 128);
    for (int i = cm_tid; i < SH * nbias; i += 128) {
      const int sub = i / nbias, bin = i - sub * nbias;
      atomicAdd(d_table + bin * gm.nH + hg * SH + sub, s_bacc[sub * (TAB_MAX + 1) + bin]);
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 112;");
    // ---------------------------------------------------------------- drain warps (groups B0 / B1)
    // Output product n of the CTA lands in TMEM accumulator n % 2, which is group (n % 2)'s to drain:
    // TMEM -> bf16 -> the row's own line of d_qkv (window_reverse + inverse roll = the token index of
    // the row) with 256-bit stores, one full 32-byte sector per lane and instruction: no shared-memory
    // staging (the SM's shared-memory port is the scarce resource of this kernel), plus the qkv-bias
    // gradient column sums.  32 columns at a time.
    const int bg = (warp - 8) >> 2;               // 0: warps 8-11, 1: warps 12-15
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const uint32_t t_lane = uint32_t(wq * 32) << 16;
    const bool tr = (threadIdx.x == 256);
    (void)tr;
    uint32_t nout = 0;                            // products of the CTA so far
    for (int k = 0; k < n_local; ++k) {
      const int item = int(blockIdx.x) + k * int(gridDim.x);
      const int tile = item / gm.ngrp;
      RowGeom rg;
      if constexpr (WS > 0) rg = row_geom_fast<L, WS, ORDER, LWT>(gm, tile, row);
      else                  rg = row_geom(gm, tile, row);
      __nv_bfloat16* row_out = d_qkv + rg.tok * (3 * gm.C) + hg * gm.gch;
#pragma unroll 1
      for (int sub = 0; sub < SH; ++sub) {
#pragma unroll 1
        for (int n = 0; n < 3 * nc; ++n, ++nout) {
          if (int(nout & 1) != bg) continue;
          const int o = n < nc ? 0 : 1 + ((n - nc) & 1);        // 0: dV, 1: dQ, 2: dK
          const int c = n < nc ? n : ((n - nc) >> 1);
          const int which = (o == 0) ? 2 : (o == 1 ? 0 : 1);
          const float m2 = !rg.valid ? 0.f : (o == 0 ? 1.0f : gm.scale);
          mbar_wait(&obuf_full[bg], (nout >> 1) & 1);
          tc_fence_after();
          if (tr && n == 0) WTRACE(g_trace_bwd, k, 11);
          // two heads per chunk (SH == 2): only columns [sub*32, +32) of the product belong to this head
          constexpr int NHALF = (SH == 1) ? 2 : 1;
#pragma unroll 1
          for (int half = 0; half < NHALF; ++half) {     // rolled: small code (instruction cache)
            const int cofs = (SH == 1) ? half * 32 : sub * 32;     // first column inside the 64-channel chunk
            float a[32];
            {
              uint32_t v[32];
              tmem_ld32(tmem_out + bg * 64 + t_lane + cofs, v);
              tmem_ld_wait();
#pragma unroll
              for (int q = 0; q < 32; ++q) a[q] = __uint_as_float(v[q]) * m2;
            }
            if (half == NHALF - 1) {
              tc_fence_before();
              mbar_arrive(&obuf_free[bg]);
            }
            const int ch0 = which * gm.C + c * 64 + cofs;          // relative to the head group's first channel
            if (rg.valid) {
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                uint32_t w8[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) w8[e] = pack_bf16(a[16 * j + 2 * e], a[16 * j + 2 * e + 1]);
                st_global_v8(row_out + ch0 + 16 * j, w8);
              }
            }
            if (d_colsum != nullptr) {
              warp_colsum<32>(a, lane);        // lane l: column l summed over this warp's 32 rows
              atomicAdd(d_colsum + ch0 + hg * gm.gch + lane, a[0]);
            }
          }
        }
      }
      if (tr) WTRACE(g_trace_bwd, k, 12);
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

#ifdef STSWIN_TRACE
extern "C" int stswin_debug_trace_bwd(long long* buf) {
  return cudaMemcpyToSymbol(g_trace_bwd, &buf, sizeof(buf)) == cudaSuccess ? 0 : -1;
}
#endif

// see include/stswin_b200.h : stswin_winattn_bwd
int winattn_bwd(const void* qkv, const float* bias_table, const float* lse2, const void* d_out, void* d_qkv,
                float* d_table, float* d_qkv_colsum, int B, int T, int H, int W, int C, int nH, int ws, int shift,
                float qk_scale, const float* mask, int mask_windows, cudaStream_t stream) {
  STSWIN_CHECK_ARG(qkv && bias_table && lse2 && d_out && d_qkv && d_table, "winattn_bwd: null pointer");
  WinGeom gm;
  int rc = fill_geom(&gm, B, T, H, W, C, nH, ws, shift, qk_scale, mask, mask_windows);
  if (rc != kOk) return rc;
  WinMaps tq, td;
  if ((rc = make_window_tmaps(&tq, qkv, gm, 3 * C)) != kOk) return rc;
  if ((rc = make_window_tmaps(&td, d_out, gm, C)) != kOk) return rc;
  STSWIN_CHECK_ARG((reinterpret_cast<uintptr_t>(d_qkv) & 31) == 0, "winattn_bwd: d_qkv must be 32-byte aligned");
  return dispatch_variant(select_variant(gm, true), [&](auto v) {
    using V = decltype(v);
    auto launch = [&](auto kern) {
      return launch_winattn(kern, gm, NUM_THREADS, SMEM_BYTES, stream, tq, td, static_cast<__nv_bfloat16*>(d_qkv),
                            bias_table, lse2, d_table, d_qkv_colsum, gm);
    };
    if (gm.SH == 1) return launch(winattn_bwd_kernel<V::L, V::WS, V::ORDER, 1, V::GEN, V::LWT>);
    return launch(winattn_bwd_kernel<V::L, V::WS, V::ORDER, 2, V::GEN, V::LWT>);
  });
}

}  // namespace stswin
