// extern "C" surface of libstswin_b200.so -- see include/stswin_b200.h
#include "../../include/stswin_b200.h"
#include "host_util.h"
#include "kernels.h"

extern "C" {

int stswin_abi_version(void) { return 6; }
const char* stswin_last_error(void) { return stswin::last_error(); }
int stswin_set_device(int device) {
  STSWIN_CUDA(cudaSetDevice(device));
  return stswin::kOk;
}

int stswin_gemm_bf16(const void* A, int a_major, int64_t lda, const void* B, int b_major, int64_t ldb, void* D,
                     int64_t ldd, void* D2, const void* aux, int64_t ld_aux, const float* bias, float* colsum, int M,
                     int N, int K, int mode, int k_splits, void* stream) {
  return stswin::gemm_bf16(A, a_major, lda, B, b_major, ldb, D, ldd, D2, aux, ld_aux, bias, colsum, M, N, K, mode,
                           k_splits, static_cast<cudaStream_t>(stream));
}

int64_t stswin_winattn_lse_elems(int B, int T, int H, int W, int C, int nH, int ws) {
  return stswin::winattn_lse_elems(B, T, H, W, C, nH, ws);
}
int stswin_winattn_fwd(const void* qkv, const float* bias_table, void* out, float* lse2, int B, int T, int H, int W,
                       int C, int nH, int ws, int shift, float qk_scale, const float* mask, int mask_windows, void* stream) {
  return stswin::winattn_fwd(qkv, bias_table, out, lse2, B, T, H, W, C, nH, ws, shift, qk_scale, mask, mask_windows,
                             static_cast<cudaStream_t>(stream));
}

int stswin_winattn_bwd(const void* qkv, const float* bias_table, const float* lse2, const void* d_out, void* d_qkv,
                       float* d_bias_table, float* d_qkv_colsum, int B, int T, int H, int W, int C, int nH, int ws,
                       int shift, float qk_scale, const float* mask, int mask_windows, void* stream) {
  return stswin::winattn_bwd(qkv, bias_table, lse2, d_out, d_qkv, d_bias_table, d_qkv_colsum, B, T, H, W, C, nH, ws,
                             shift, qk_scale, mask, mask_windows, static_cast<cudaStream_t>(stream));
}

int stswin_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                         int64_t M, int row_len, float eps, int pm, int H, int W, int C, void* stream) {
  return stswin::layernorm_fwd(x, gamma, beta, y, mean, rstd, M, row_len, eps, pm, H, W, C,
                               static_cast<cudaStream_t>(stream));
}
int stswin_layernorm_bwd(const void* dy, const void* x, const float* mean, const float* rstd, const float* gamma,
                         const void* dres, void* dx, float* dgamma, float* dbeta, float* dx_colsum, int64_t M,
                         int row_len, int pm, int H, int W, int C, void* stream) {
  return stswin::layernorm_bwd(dy, x, mean, rstd, gamma, dres, dx, dgamma, dbeta, dx_colsum, M, row_len, pm, H, W, C,
                               static_cast<cudaStream_t>(stream));
}
int stswin_transpose(const void* in, int in_is_f32, void* out, int out_is_f32, int64_t batch, int R, int Cc,
                     void* stream) {
  return stswin::transpose_cvt(in, in_is_f32, out, out_is_f32, batch, R, Cc, static_cast<cudaStream_t>(stream));
}
int stswin_colsum(const void* x, float* out, int64_t R, int C, void* stream) {
  return stswin::colsum_bf16(x, out, R, C, static_cast<cudaStream_t>(stream));
}
int stswin_copy_strided(void* dst, int64_t dst_stride, const void* src, int64_t src_stride, int64_t bytes, int batches,
                        void* stream) {
  return stswin::copy_strided(dst, dst_stride, src, src_stride, bytes, batches, static_cast<cudaStream_t>(stream));
}

int stswin_pixloss_labels(const void* const* labels, const int* dtypes, int n_labels, int slot_off, int N, int Hs, int Ws,
                          int H, int W, int class_num, uint8_t* lab_nat, uint8_t* lab_sorted, uint8_t* glab, uint16_t* perm,
                          int32_t* hist, int32_t* err_flag, float* ksum_to_clear, int64_t ksum_elems, void* stream) {
  return stswin::pixloss_labels(labels, dtypes, n_labels, slot_off, N, Hs, Ws, H, W, class_num, lab_nat, lab_sorted, glab,
                                perm, hist, err_flag, ksum_to_clear, ksum_elems, static_cast<cudaStream_t>(stream));
}
int stswin_pixloss_prepare(const void* const* maps, const int* dtypes, const int* label_slots, int n_maps, int slot_off,
                           int N, int C, int HW, int do_normalize, int lo_slot_off, const uint16_t* perm, void* xn,
                           float* inv_norm, float* ksum, float* f32_to_clear, int64_t f32_elems, void* stream) {
  return stswin::pixloss_prepare(maps, dtypes, label_slots, n_maps, slot_off, N, C, HW, do_normalize, lo_slot_off, perm, xn,
                                 inv_norm, ksum, f32_to_clear, f32_elems, static_cast<cudaStream_t>(stream));
}
int stswin_pixloss_fwd(const void* xn, int n_slots, int n_label_slots, const uint8_t* lab_nat, const uint8_t* lab_sorted,
                       const uint8_t* glab, const int32_t* hist, const int* qmap, const int* qlab, const int* kmap,
                       const int* klab, int n_terms, int Q, int S, int N, int C, int HW, float* stats, float* loss,
                       float* loss_per_query,
                       float* coef, const int32_t* err_flag, float* partial, uint32_t* ticket, void* stream) {
  return stswin::pixloss_fwd(xn, n_slots, n_label_slots, lab_nat, lab_sorted, glab, hist, qmap, qlab, kmap, klab, n_terms, Q, S, N,
                             C, HW, stats, loss, loss_per_query, coef, err_flag, partial, ticket, static_cast<cudaStream_t>(stream));
}
int stswin_pixloss_bwd(const void* xn, int n_slots, int n_label_slots, const uint8_t* lab_nat, const uint8_t* lab_sorted,
                       const uint8_t* glab, const int* qmap, const int* qmap_lo, const int* qlab, const int* kmap,
                       const int* klab, int n_terms, int Q, int S, int N, int C, int HW, const float* coef, const float* ksum, const float* d_loss, float* dq32,
                       int dq32_is_clear, const float* inv_norm, void* const* dq_out, int out_dtype, void* stream) {
  return stswin::pixloss_bwd(xn, n_slots, n_label_slots, lab_nat, lab_sorted, glab, qmap, qmap_lo, qlab, kmap, klab, n_terms, Q, S, N, C, HW,
                             coef, ksum, d_loss, dq32, dq32_is_clear, inv_norm, dq_out, out_dtype, static_cast<cudaStream_t>(stream));
}

int64_t stswin_ohem_ws_bytes(void) { return stswin::ohem_ws_bytes(); }
int stswin_ohem_ce_fwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, int64_t HW,
                       int ignore_index, float thresh, int64_t n_min, float* loss_px, void* ws, float* loss, float* sel,
                       void* stream) {
  return stswin::ohem_ce_fwd(logits, logits_is_f32, labels, B, K, HW, ignore_index, thresh, n_min, loss_px, ws, loss, sel,
                             static_cast<cudaStream_t>(stream));
}
int stswin_ohem_ce_bwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, int64_t HW,
                       int ignore_index, const float* loss_px, const float* sel, const float* d_loss, void* d_logits,
                       void* stream) {
  return stswin::ohem_ce_bwd(logits, logits_is_f32, labels, B, K, HW, ignore_index, loss_px, sel, d_loss, d_logits,
                             static_cast<cudaStream_t>(stream));
}
int stswin_ema_update(void* const* k_params, const void* const* q_params, void* const* k_shadows, const int64_t* numels,
                      int n_tensors, float m, float one_minus_m, const float* m_dev, void* stream) {
  return stswin::ema_update(k_params, q_params, k_shadows, numels, n_tensors, m, one_minus_m, m_dev,
                            static_cast<cudaStream_t>(stream));
}
int stswin_lars_sgd_step(void* const* params, void* const* grads, void* const* momentum_bufs, void* const* shadows,
                         const int64_t* numels, const uint8_t* first_step, int n_tensors, int grads_are_bf16,
                         int write_grads, float lr, const float* lr_dev, float momentum, float dampening, int nesterov,
                         float weight_decay, int lars, float trust_coef, float eps, double* norms_ws, void* stream) {
  return stswin::lars_sgd_step(params, grads, momentum_bufs, shadows, numels, first_step, n_tensors, grads_are_bf16,
                               write_grads, lr, lr_dev, momentum, dampening, nesterov, weight_decay, lars, trust_coef, eps,
                               norms_ws, static_cast<cudaStream_t>(stream));
}

int stswin_adam_step(void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                     void* const* shadows, const int64_t* numels, int n_tensors, int grads_are_bf16, float lr, float beta1,
                     float beta2, float eps, float weight_decay, float grad_scale, float* step, void* stream) {
  return stswin::adam_step(params, grads, exp_avg, exp_avg_sq, shadows, numels, n_tensors, grads_are_bf16, lr, beta1, beta2,
                           eps, weight_decay, grad_scale, step, static_cast<cudaStream_t>(stream));
}

int stswin_sgd_step(void* const* params, const void* const* grads, void* const* momentum_bufs, void* const* shadows,
                    const int64_t* numels, const uint8_t* first_step, int n_tensors, int grads_are_bf16, float lr,
                    const float* lr_dev, float momentum, float one_minus_dampening, int nesterov, int maximize,
                    float weight_decay, float grad_scale, void* stream) {
  return stswin::sgd_step(params, grads, momentum_bufs, shadows, numels, first_step, n_tensors, grads_are_bf16, lr, lr_dev,
                          momentum, one_minus_dampening, nesterov, maximize, weight_decay, grad_scale,
                          static_cast<cudaStream_t>(stream));
}

int stswin_gather_cast(void* const* dst, const void* const* src, const int64_t* numels, int n_tensors, int dst_is_bf16,
                       void* stream) {
  return stswin::gather_cast(dst, src, numels, n_tensors, dst_is_bf16, static_cast<cudaStream_t>(stream));
}

int stswin_f32_split(const float* x, void* out, int64_t R, int C, int layout, int pattern, int op, void* stream) {
  return stswin::f32_split(x, out, R, C, layout, pattern, op, static_cast<cudaStream_t>(stream));
}
int stswin_f32_rowop(float* out, const float* bias, const float* res, const float* aux, int64_t R, int C, int mode, void* stream) {
  return stswin::f32_rowop(out, bias, res, aux, R, C, mode, static_cast<cudaStream_t>(stream));
}
int stswin_f32_colsum(const float* x, float* out, int64_t R, int C, void* stream) {
  return stswin::f32_colsum(x, out, R, C, static_cast<cudaStream_t>(stream));
}
int stswin_f32_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd,
                             int64_t M, int row_len, float eps, int pm, int H, int W, int C, void* stream) {
  return stswin::f32_layernorm_fwd(x, gamma, beta, y, mean, rstd, M, row_len, eps, pm, H, W, C, static_cast<cudaStream_t>(stream));
}
int stswin_f32_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                             const float* dres, float* dx, float* dgamma, float* dbeta, int64_t M, int row_len, int pm, int H,
                             int W, int C, void* stream) {
  return stswin::f32_layernorm_bwd(dy, x, mean, rstd, gamma, dres, dx, dgamma, dbeta, M, row_len, pm, H, W, C,
                                   static_cast<cudaStream_t>(stream));
}
int stswin_winattn_f32_fwd(const float* qkv, const float* bias_table, float* out, float* lse, int B, int T, int H, int W, int C,
                           int nH, int ws, int shift, float qk_scale, const float* mask, int mask_windows, void* stream) {
  return stswin::winattn_f32_fwd(qkv, bias_table, out, lse, B, T, H, W, C, nH, ws, shift, qk_scale, mask, mask_windows,
                                 static_cast<cudaStream_t>(stream));
}
int stswin_winattn_f32_bwd(const float* qkv, const float* bias_table, const float* out, const float* lse, const float* d_out,
                           float* d_qkv, float* d_bias_table, float* delta_ws, int B, int T, int H, int W, int C, int nH, int ws,
                           int shift, float qk_scale, const float* mask, int mask_windows, void* stream) {
  return stswin::winattn_f32_bwd(qkv, bias_table, out, lse, d_out, d_qkv, d_bias_table, delta_ws, B, T, H, W, C, nH, ws, shift,
                                 qk_scale, mask, mask_windows, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
