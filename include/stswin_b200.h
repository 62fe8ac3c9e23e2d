/* stswin_b200 -- C ABI of the B200-native (sm_100a) STswinCL hot paths.
 *
 * The reference (YuemingJin/STswinCL) is pure Python/PyTorch and has no FFI of its own; its
 * boundary for these paths is the nn.Module / function API (SURVEY.md section 8b).  This header
 * is the C boundary underneath the drop-in Python modules of `stswincl_b200/`: each entry point
 * names the reference op sequence it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch) unless stated otherwise;
 *   - `stream` is a cudaStream_t passed as void*; functions only enqueue work and never synchronise;
 *   - return value 0 = success, negative = error (STSWIN_ERR_*); the message of the last error of
 *     the calling thread is available from stswin_last_error();
 *   - activations are bf16 (uint16 storage), statistics / gradients of parameters are fp32;
 *   - no global mutable state besides per-device read-only attribute caches.
 */
#ifndef STSWIN_B200_H_
#define STSWIN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STSWIN_OK 0
#define STSWIN_ERR_INVALID_ARG (-1)
#define STSWIN_ERR_UNSUPPORTED (-2)
#define STSWIN_ERR_CUDA (-3)
#define STSWIN_ERR_DRIVER (-4)

/* ABI version of this header; bumped on any signature change. */
int stswin_abi_version(void);
/* Text of the last error raised on the calling thread ("" if none). */
const char* stswin_last_error(void);
/* Bind the calling thread to `device` (cudaSetDevice in this library's runtime).  Call before the
 * other entry points from any thread that has not used the device yet -- e.g. an autograd worker
 * or an nn.DataParallel replica thread (seg18/train_swin.py:131-135): tensor-map encoding is a
 * driver call and needs the device's context current on the thread. */
int stswin_set_device(int device);

/* ---------------------------------------------------------------------------------------------
 * Dense layers: D[M,N] = sum_k A[m,k] * B[n,k]   (bf16 x bf16 -> fp32 accumulate, tcgen05)
 *
 * Replaces nn.Linear forward/backward inside the block:
 *   qkv   seg18/net/Ours/swin_512.py:116     proj  :139     fc1/fc2  :18,22 (Mlp.forward)
 *   PatchMerging.reduction :275
 *
 *   a_major / b_major : 0 = K-major  (A is [M,K] row-major with leading dim lda; B is [N,K], ldb)
 *                       1 = MN-major (A is [K,M] row-major;                      B is [K,N])
 *                       (1,0) is not provided.
 *   mode : STSWIN_EPI_*.  `bias` ([N] fp32) may be NULL.  `colsum` ([N] fp32, may be NULL)
 *          receives += the column sums of the bf16-rounded D (bias gradient of the producer).
 *   STSWIN_EPI_F32_REDUCE: D is fp32 [M,N] with leading dim ldd and receives += the product;
 *          the K range is split `k_splits` ways across CTAs (weight gradients reduce over tokens).
 */
#define STSWIN_EPI_BIAS 0          /* D = acc + bias                                  */
#define STSWIN_EPI_BIAS_RES 1      /* D = acc + bias + aux            (residual add)  */
#define STSWIN_EPI_BIAS_GELU 2     /* u = acc + bias ; D = gelu_erf(u) ; D2 = gelu_erf'(u) */
/* The two x-aux modes add `bias` (when not NULL) before the product: D = (acc + bias) * aux.  The block's dgrad passes
 * NULL; the term is kept because it is free in the epilogue and is what a Linear followed by an elementwise gate needs. */
#define STSWIN_EPI_MUL_AUX 3       /* D = (acc + bias) * aux     (dgrad through GELU: aux = D2, bias NULL) */
#define STSWIN_EPI_F32_REDUCE 4    /* D(fp32) += acc, split-K                          */
#define STSWIN_EPI_BIAS_GELU_FWD 5 /* D = gelu_erf(acc + bias)      (inference: no D2) */
/* The derivative is only ever a multiplier of the backward and lies in [-0.13, 1.13]: the two modes below keep it as ONE
 * byte per element (D2 / aux are uint8 [M,N] with the leading dimension of D / ld_aux in bytes; N and the leading dimensions
 * multiples of 16): q = round((gelu'(u) + 0.14) * 255 / 1.28), i.e. a step of 0.005 (|error| <= 0.0025, the bf16 rounding of
 * a value near 1 is 0.002-0.004).  fc1 + GELU writes 1.28 GB per stage-1 launch in the bf16 form and is HBM-write bound. */
#define STSWIN_EPI_BIAS_GELU_Q8 6  /* D = gelu_erf(acc + bias) ; D2(uint8) = quantised gelu_erf'(acc + bias) */
#define STSWIN_EPI_MUL_AUX_Q8 7    /* D = (acc + bias) * dequant(aux)  (aux = the uint8 D2 of mode 6) */

int stswin_gemm_bf16(const void* A, int a_major, int64_t lda,
                     const void* B, int b_major, int64_t ldb,
                     void* D, int64_t ldd, void* D2,
                     const void* aux, int64_t ld_aux,
                     const float* bias, float* colsum,
                     int M, int N, int K, int mode, int k_splits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Spatio-temporal shifted-window attention core (K1+K3+K5 of SURVEY.md section 2c).
 *
 * Replaces, for one SwinTransformerBlock call (seg18/net/Ours/swin_512.py):
 *   torch.roll + window_partition + permute   :210-218      (gather = TMA box coordinates)
 *   q*scale, q@k^T, bias gather, mask, softmax, attn@v      :119-138 (WindowAttention.forward)
 *   window_reverse + torch.roll               :224-231      (scatter = TMA store coordinates)
 *
 *   qkv        [B, T, H, W, 3C] bf16, tokens in natural (un-rolled) order, channel =
 *              which*C + head*(C/nH) + d  (the layout nn.Linear(dim, 3*dim) produces, :116)
 *   bias_table [(2*ws-1)^2, nH] fp32   (relative_position_bias_table, :81-82; the relative
 *              position index :88-99 and the shift mask :171-192 are closed forms in-kernel)
 *   out        [B, T, H, W, C] bf16, same token order
 *   lse2       [stswin_winattn_lse_elems(...)] fp32 workspace written by fwd, read by bwd
 *   shift      0 <= shift < ws (the reference uses 0 and ws/2).  ws <= 8 and T*ws*ws <= 128 (any value,
 *              e.g. 98 for ws 7); H, W multiples of ws; C/nH = 32 or a multiple of 64, <= 256.
 *   qk_scale   multiplier of q (WindowAttention's `qk_scale`, :79); <= 0 selects (C/nH)^-0.5
 *   mask       optional dense additive mask [mask_windows, N, N] fp32 (N = ws*ws), the `mask` argument of
 *              WindowAttention.forward (:127-131): window w uses mask[w % mask_windows], tiled over the
 *              frame pair.  NULL for the normal case -- the block's shift mask is a closed form of
 *              (H, W, ws, shift) and is rebuilt in-kernel.
 */
int64_t stswin_winattn_lse_elems(int B, int T, int H, int W, int C, int nH, int ws);
int stswin_winattn_fwd(const void* qkv, const float* bias_table, void* out, float* lse2,
                       int B, int T, int H, int W, int C, int nH, int ws, int shift, float qk_scale,
                       const float* mask, int mask_windows, void* stream);
/* Backward of the same op sequence (what autograd derives for swin_512.py:119-138 + :210-231).
 *   d_out        [B, T, H, W, C]  bf16  gradient w.r.t. `out`
 *   d_qkv        [B, T, H, W, 3C] bf16  written (every element)
 *   d_bias_table [(2*ws-1)^2, nH] fp32  += (zero it for a fresh gradient)
 *   d_qkv_colsum [3C] fp32 or NULL      += column sums of d_qkv (= gradient of qkv.bias)
 */
int stswin_winattn_bwd(const void* qkv, const float* bias_table, const float* lse2, const void* d_out,
                       void* d_qkv, float* d_bias_table, float* d_qkv_colsum,
                       int B, int T, int H, int W, int C, int nH, int ws, int shift, float qk_scale,
                       const float* mask, int mask_windows, void* stream);

/* ---------------------------------------------------------------------------------------------
 * LayerNorm (eps inside the rsqrt, fp32 statistics) over rows of `row_len` bf16 channels.
 * Replaces nn.LayerNorm at swin_512.py:235 (norm2, norm1) and, with pm = 1, the PatchMerging
 * prologue  x[:,0::2,0::2] | x[:,1::2,0::2] | x[:,0::2,1::2] | x[:,1::2,1::2] -> cat -> norm
 * (swin_512.py:266-274): logical row r of the normalised matrix is then the 2x2 neighbourhood
 * of output token r, gathered from x [BT, H, W, C] with row_len = 4*C (H, W, C describe x).
 *   fwd: y [M,row_len] bf16 (dense), mean/rstd [M] fp32
 *   bwd: dx has the layout of x (scattered through the same 2x2 map when pm = 1);
 *        dres (optional, same layout as dy) is added to dx (residual branch);
 *        dgamma/dbeta [row_len] fp32 +=; dx_colsum [row_len] fp32 += column sums of dx or NULL
 */
int stswin_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                         int64_t M, int row_len, float eps, int pm, int H, int W, int C, void* stream);
int stswin_layernorm_bwd(const void* dy, const void* x, const float* mean, const float* rstd, const float* gamma,
                         const void* dres, void* dx, float* dgamma, float* dbeta, float* dx_colsum,
                         int64_t M, int row_len, int pm, int H, int W, int C, void* stream);

/* [batch, R, Cc] -> [batch, Cc, R] with dtype conversion (1 = fp32, 0 = bf16 on either side).
 * Replaces permute(0,1,3,4,2).contiguous() / permute(0,1,3,2) of SwinTransformerLayerv5.forward
 * (swin_512.py:314,319,326). */
int stswin_transpose(const void* in, int in_is_f32, void* out, int out_is_f32, int64_t batch, int R, int Cc, void* stream);

/* out[c] += sum_r x[r, c] for a dense bf16 matrix x [R, C] (C a multiple of 8): the bias gradient of nn.Linear
 * (proj.bias when WindowAttention runs stand-alone, swin_512.py:139; Mlp.fc2.bias, :22).  out is fp32 [C]. */
int stswin_colsum(const void* x, float* out, int64_t R, int C, void* stream);

/* Batched strided copy: dst[b*dst_stride + i] = src[b*src_stride + i] for i < bytes, b < batches (all in bytes;
 * pointers, strides and `bytes` multiples of 16).  Moves the frame slices of the middle Swin layer
 * (x[:, 1:3] in, cat([x[:, :1], y, x[:, 3:]]) out, swin_512.py:302-307) at copy bandwidth. */
int stswin_copy_strided(void* dst, int64_t dst_stride, const void* src, int64_t src_stride, int64_t bytes, int batches,
                        void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pixel-level contrastive loss (K7).  Replaces regression_loss / posMask / negMask of
 * pixcontrast_18/contrast/models/PixPro_swin_v5.py:48-129, the F.normalize(dim=1) calls feeding it
 * (:330,362,400,432,463,494,526,557) and the tail of ConsistencyLoss.forward (:584-597: nearest
 * down-sampling of the six label maps, two symmetric regression_loss calls sharing four key sets).
 *
 * One loss STEP evaluates Q <= 2 "queries" (one regression_loss call each), every query against S <= 64
 * key sets.  The embedding maps and label maps of a step live in SLOTS of caller-owned workspaces; host
 * tables say which slot each query / key set uses, so a map shared by both queries is prepared once.
 * With HW = H*W pixels per map, HWp = HW rounded up to 256, GLp = HWp/32 rounded up to 16:
 *
 *   xn         [slots, N, C, HW]   bf16  prepared maps: query maps in pixel order, key maps in LABEL order
 *   inv_norm   [slots, N, HW]      fp32  1 / max(|x|, 1e-12) per pixel (pixel order)
 *   ksum       [slots, N, C]       fp32  per-channel sums of a key map over its pixels
 *   lab_nat    [lslots, N, HWp]    u8    labels in pixel order (255 = padding / out of range)
 *   lab_sorted [lslots, N, HWp]    u8    labels in sorted (key) order
 *   glab       [lslots, N, GLp]    u8    label of each group of 32 sorted keys (254 = mixed, 255 = padding)
 *   perm       [lslots, N, HW]     u16   sorted position of pixel j (stable counting sort by label)
 *   hist       [lslots, N, 256]    i32   pixels per label
 *   ctl        [2]                 i32   [0] |= 1 when a label is outside [0, class_num) -- the loss is then
 *                                        NaN (the reference's F.one_hot raises, :54-55); [1] finalize ticket
 *
 * stswin_pixloss_labels : label maps labels[i] ([N,1,Hs,Ws], dtypes[i]: 0 u8, 1 f32, 2 i64, 3 i32, 4 bf16,
 *     5 f16; HOST arrays of n_labels device pointers / codes) -> slots slot_off.. of the label workspaces:
 *     F.interpolate(mode='nearest') to H x W (:585-590), .long() (:54), range check, counting sort.
 *     slot_off == 0 also clears ctl.  1 <= class_num <= 254; H*W a multiple of 8, <= 8192.
 * stswin_pixloss_prepare: maps[i] ([N,C,HW], dtypes[i]: 0 bf16, 1 f32, 2 f16) -> slots slot_off.. of xn /
 *     inv_norm / ksum: x / max(|x|_2 over C, 1e-12) when do_normalize (else a plain cast), stored in the
 *     order of label slot label_slots[i] (key maps) or in pixel order (label_slots[i] = -1, query maps).
 *     C a multiple of 64, <= 256.
 * stswin_pixloss_fwd    : qmap/qlab [Q], kmap/klab [Q*S] (HOST int arrays): map slot and label slot of
 *     every query and of its key sets, ordered (k, adj1, adj2, adj3, neg3, extra sets...) like the
 *     reference's arguments (extra sets extend the positive pool and the negative sum).
 *     stats [Q,N,HW,S,2,2] fp32 workspace; loss: device scalar = sum over queries of
 *     -mean log(e^P/(e^P+e^N)+1e-6); loss_per_query [Q] or NULL; coef [Q,N,HW,1+S] fp32 (NULL when no
 *     gradient is needed): per-row dloss/dz coefficients for the backward; partial: fp32 scratch of
 *     Q*ceil(N*HW/64) elements; ticket = &ctl[1].
 * stswin_pixloss_bwd    : dq_out[q] (HOST array of Q device pointers, [N,C,HW], out_dtype 0 bf16 / 1 f32 /
 *     2 f16) = d_loss * dloss/d(query map q); with inv_norm != NULL through the Jacobian of the fused
 *     normalisation.  dq32 [Q,N,HW,C] fp32 scratch; d_loss: device scalar (the upstream gradient).
 *     Keys receive no gradient (they are built under no_grad in the reference, :366).
 *
 * Launch chaining: the kernels of a step are launched with programmatic dependent launch (each one's prologue -- barrier
 * initialisation, TMEM allocation, descriptor prefetch -- overlaps its predecessor's tail; STSWIN_PDL=0 disables it), and
 * buffer clears ride on neighbouring kernels instead of memset nodes: stswin_pixloss_labels (slot_off == 0) clears
 * ksum_to_clear[0 .. ksum_elems) -- stswin_pixloss_prepare ACCUMULATES into ksum and expects it cleared --, and
 * stswin_pixloss_prepare clears f32_to_clear[0 .. f32_elems) (may be NULL; the [Q,N,HW,C] fp32 accumulator of a backward
 * that is then called with dq32_is_clear = 1).
 *
 * fp32-accurate mode (loss value and gradient <= 1e-3 against the reference's fp32 run): stswin_pixloss_prepare with
 * lo_slot_off > 0 also stores the second bf16 term x - bf16(x) of every map in slot (slot + lo_slot_off) and sums the
 * channels in fp32; the row sums are linear in the similarities, so stswin_pixloss_fwd takes n_terms = 3 tables
 * (qmap [n_terms*Q], kmap [n_terms*Q*S]: (q_hi,k_hi), (q_hi,k_lo), (q_lo,k_hi); stats then holds n_terms copies) and
 * stswin_pixloss_bwd n_terms = 2 key tables (k_hi, k_lo) with qmap_lo [Q] naming the queries' second terms (NULL in
 * the bf16 mode).  n_terms = 1 is the bf16 mode.
 */
int stswin_pixloss_labels(const void* const* labels, const int* dtypes, int n_labels, int slot_off,
                          int N, int Hs, int Ws, int H, int W, int class_num,
                          uint8_t* lab_nat, uint8_t* lab_sorted, uint8_t* glab, uint16_t* perm, int32_t* hist,
                          int32_t* ctl, float* ksum_to_clear, int64_t ksum_elems, void* stream);
int stswin_pixloss_prepare(const void* const* maps, const int* dtypes, const int* label_slots, int n_maps, int slot_off,
                           int N, int C, int HW, int do_normalize, int lo_slot_off, const uint16_t* perm,
                           void* xn, float* inv_norm, float* ksum, float* f32_to_clear, int64_t f32_elems, void* stream);
int stswin_pixloss_fwd(const void* xn, int n_slots, int n_label_slots,
                       const uint8_t* lab_nat, const uint8_t* lab_sorted, const uint8_t* glab, const int32_t* hist,
                       const int* qmap, const int* qlab, const int* kmap, const int* klab,
                       int n_terms, int Q, int S, int N, int C, int HW,
                       float* stats, float* loss, float* loss_per_query, float* coef,
                       const int32_t* ctl, float* partial, uint32_t* ticket, void* stream);
int stswin_pixloss_bwd(const void* xn, int n_slots, int n_label_slots,
                       const uint8_t* lab_nat, const uint8_t* lab_sorted, const uint8_t* glab,
                       const int* qmap, const int* qmap_lo, const int* qlab, const int* kmap, const int* klab,
                       int n_terms, int Q, int S, int N, int C, int HW,
                       const float* coef, const float* ksum, const float* d_loss, float* dq32, int dq32_is_clear,
                       const float* inv_norm, void* const* dq_out, int out_dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training-step kernels either side of the two hot paths (SURVEY.md section 8f, rows N2-N4).
 *
 * OHEM cross-entropy.  Replaces OhemCELoss2D.forward (seg18/utils/losses.py:16-40): per-pixel
 * cross_entropy(reduction='none', ignore_index) :33, the full descending sort :34 and the
 * `loss[n_min] > thresh` branch :36-39, without the sort and without a host read:
 *   more than n_min losses above thresh -> mean of the losses above thresh,
 *   otherwise                           -> mean of the n_min largest (k-th value by a 3-pass radix select).
 *   logits  [B, K, HW] fp32 (logits_is_f32) or bf16, class-major as the decoder emits (NCHW)
 *   labels  [B, HW] int64; a label equal to ignore_index contributes loss 0 (and no gradient)
 *   thresh  the loss threshold -log(0.7) of :26;   1 <= n_min < B*HW (:36 indexes loss[n_min])
 *   loss_px [B*HW] fp32 per-pixel losses (kept for the backward);  ws: stswin_ohem_ws_bytes() bytes
 *   loss    device scalar;  sel [4] fp32: {cut, gradient weight of a loss above cut, weight of a loss
 *           equal to cut (ties at the n_min-th value share the remaining weight), unused}
 * stswin_ohem_ce_bwd: d_logits (dtype of logits, every element written) =
 *           weight(pixel) * (softmax - onehot) * d_loss   (d_loss: device scalar)
 */
int64_t stswin_ohem_ws_bytes(void);
int stswin_ohem_ce_fwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, int64_t HW,
                       int ignore_index, float thresh, int64_t n_min, float* loss_px, void* ws, float* loss, float* sel,
                       void* stream);
int stswin_ohem_ce_bwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, int64_t HW,
                       int ignore_index, const float* loss_px, const float* sel, const float* d_loss, void* d_logits,
                       void* stream);

/* Momentum (EMA) update of the key encoder as one multi-tensor stream.  Replaces the ~600 per-parameter
 * `param_k.data = param_k.data * m + param_q.data * (1. - m)` of PixPro._momentum_update_key_encoder
 * (pixcontrast_18/contrast/models/PixPro_swin_v5.py:258-289); bit-exact with the eager expression
 * (two rounded products, one rounded sum).  k_params / q_params / numels are HOST arrays of n_tensors
 * device pointers (fp32 tensors, contiguous) and element counts. */
int stswin_ema_update(void* const* k_params, const void* const* q_params, const int64_t* numels, int n_tensors, float m,
                      float one_minus_m, void* stream);

/* LARS-scaled SGD step of one parameter group.  Replaces LARS.apply_adaptive_lrs + the wrapped
 * torch.optim.SGD.step (pixcontrast_18/contrast/lars.py:109-152): per tensor
 *   g = grad + weight_decay * p (:121-122); if `lars`: g *= trust_coef * |p| / (|g| + eps) when both norms
 *   are positive (:125-135); grad <- g (the reference rebinds p.grad); buf = g on a tensor's first step
 *   (first_step[t] != 0) else momentum * buf + (1 - dampening) * g; p -= lr * (nesterov ? g + momentum * buf : buf).
 * The norms are reduced on the device (no .norm() host reads, :127-133).  params / grads / momentum_bufs /
 * numels / first_step are HOST arrays over the group's tensors (fp32, contiguous); momentum_bufs may be NULL
 * when momentum == 0; norms_ws: device [2 * n_tensors] fp64 scratch (only when `lars`). */
int stswin_lars_sgd_step(void* const* params, void* const* grads, void* const* momentum_bufs, const int64_t* numels,
                         const uint8_t* first_step, int n_tensors, float lr, float momentum, float dampening,
                         int nesterov, float weight_decay, int lars, float trust_coef, float eps, double* norms_ws,
                         void* stream);

/* Adam step over a list of tensors (the optimiser of seg18/train_swin.py: torch.optim.Adam, no amsgrad), emitting the
 * bf16 copy of the updated weights that the Swin kernels consume (replaces the optimiser's own pass plus one cast
 * kernel per weight tensor and step).  Per element, with t = *step after the increment this call performs:
 *   g = grad_scale * grad + weight_decay * p;  m = m + (1 - beta1) (g - m);  v = beta2 v + (1 - beta2) g^2;
 *   p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps);  shadow = bf16(p)
 * params / exp_avg / exp_avg_sq: fp32; grads: fp32, or bf16 when grads_are_bf16 (gradients that arrive from a bf16
 * all-reduce); shadows: bf16 or NULL (whole array or per tensor).  All tables are HOST arrays of n_tensors device
 * pointers; step is a device float (the step count, kept on the device so that the call is graph-capturable). */
int stswin_adam_step(void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                     void* const* shadows, const int64_t* numels, int n_tensors, int grads_are_bf16, float lr, float beta1,
                     float beta2, float eps, float weight_decay, float grad_scale, float* step, void* stream);

/* dst[t] = cast(src[t]) over a list of fp32 tensors (HOST arrays of n_tensors device pointers / element counts):
 * gathers the gradients a backward segment produced into the flat bucket of the data-parallel all-reduce (SURVEY.md
 * section 8e, C1), rounding to bf16 when dst_is_bf16 (bytes on the wire halved) -- one launch per 48 tensors. */
int stswin_gather_cast(void* const* dst, const void* const* src, const int64_t* numels, int n_tensors, int dst_is_bf16,
                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * fp32-accurate mode of the window-attention path: the reference's fp32 (no-AMP) run of
 * seg18/net/Ours/swin_512.py:109-141,196-237 at <= 1e-3 relative error (BASELINE.json north_star).
 * Activations stay fp32.  Dense layers go through stswin_gemm_bf16 with both fp32 operands split into two bf16 terms
 * concatenated along the reduction dimension (K' = 3K, STSWIN_EPI_F32_REDUCE onto a bias / residual-initialised D):
 *
 * stswin_f32_split : x fp32 [R, C] -> bf16 [R, 3C] (layout 0, reduction over columns) or [3R, C] (layout 1, reduction
 *     over rows); pattern 0 = (hi, hi, lo) for the A operand, 1 = (hi, lo, hi) for the B operand, so that
 *     A'.B' = hi*hi + hi*lo + lo*hi; op 1 splits gelu_erf(x) instead of x (Mlp activation, swin_512.py:19).
 * stswin_f32_rowop : mode 0: out[r,c] = bias[c] + res[r,c] (either may be NULL) -- the value a D += acc GEMM starts
 *     from (nn.Linear bias, residual add :232-235); mode 1: out = res * gelu_erf'(aux) (GELU backward).
 * stswin_f32_colsum: out[c] += sum_r x[r,c] (bias gradients).
 * stswin_f32_layernorm_fwd / _bwd: nn.LayerNorm in fp32 with the same pm (PatchMerging gather, :266-274) convention as
 *     stswin_layernorm_*; bwd: dx (+= dres), dgamma / dbeta += .
 * stswin_winattn_f32_fwd / _bwd: the attention core of stswin_winattn_* (roll + partition + QK^T + bias + shift mask
 *     + softmax + PV + reverse, and its gradient) on fp32 qkv [B,T,H,W,3C] -> out [B,T,H,W,C], as fp32 SIMT kernels
 *     (the core is 4 % of a block's FLOPs).  lse and delta_ws: fp32 [B * (H/ws) * (W/ws) * nH * T*ws*ws] each;
 *     T*ws*ws <= 128, head_dim a multiple of 8; d_bias_table += . */
int stswin_f32_split(const float* x, void* out, int64_t R, int C, int layout, int pattern, int op, void* stream);
int stswin_f32_rowop(float* out, const float* bias, const float* res, const float* aux, int64_t R, int C, int mode, void* stream);
int stswin_f32_colsum(const float* x, float* out, int64_t R, int C, void* stream);
int stswin_f32_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd,
                             int64_t M, int row_len, float eps, int pm, int H, int W, int C, void* stream);
int stswin_f32_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                             const float* dres, float* dx, float* dgamma, float* dbeta, int64_t M, int row_len, int pm, int H,
                             int W, int C, void* stream);
int stswin_winattn_f32_fwd(const float* qkv, const float* bias_table, float* out, float* lse, int B, int T, int H, int W, int C,
                           int nH, int ws, int shift, float qk_scale, const float* mask, int mask_windows, void* stream);
int stswin_winattn_f32_bwd(const float* qkv, const float* bias_table, const float* out, const float* lse, const float* d_out,
                           float* d_qkv, float* d_bias_table, float* delta_ws, int B, int T, int H, int W, int C, int nH, int ws,
                           int shift, float qk_scale, const float* mask, int mask_windows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STSWIN_B200_H_ */
