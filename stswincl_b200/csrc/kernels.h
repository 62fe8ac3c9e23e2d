// Internal C++ declarations of the launchers behind the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace stswin {

int gemm_bf16(const void* A, int a_major, long lda, const void* B, int b_major, long ldb, void* D, long ldd, void* D2,
              const void* aux, long ld_aux, const float* bias, float* colsum, int M, int N, int K, int mode,
              int k_splits, cudaStream_t stream);

int winattn_fwd(const void* qkv, const float* bias_table, void* out, float* lse2, int B, int T, int H, int W, int C,
                int nH, int ws, int shift, float qk_scale, const float* mask, int mask_windows, cudaStream_t stream);
int winattn_bwd(const void* qkv, const float* bias_table, const float* lse2, const void* d_out, void* d_qkv,
                float* d_table, float* d_qkv_colsum, int B, int T, int H, int W, int C, int nH, int ws, int shift,
                float qk_scale, const float* mask, int mask_windows, cudaStream_t stream);
long winattn_lse_elems(int B, int T, int H, int W, int C, int nH, int ws);

int layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, long M,
                  int Ctot, float eps, int pm, int H, int W, int C, cudaStream_t stream);
int layernorm_bwd(const void* dy, const void* x, const float* mean, const float* rstd, const float* gamma,
                  const void* dres, void* dx, float* dgamma, float* dbeta, float* dx_colsum, long M, int Ctot, int pm,
                  int H, int W, int C, cudaStream_t stream);
int transpose_cvt(const void* in, int in_f32, void* out, int out_f32, long batch, int R, int Cc, cudaStream_t stream);
int colsum_bf16(const void* x, float* out, long R, int C, cudaStream_t stream);
int copy_strided(void* dst, long dst_stride, const void* src, long src_stride, long bytes, int batches, cudaStream_t stream);

int pixloss_labels(const void* const* labels, const int* dtypes, int n_labels, int slot_off, int N, int Hs, int Ws, int H,
                   int W, int class_num, uint8_t* lab_nat, uint8_t* lab_sorted, uint8_t* glab, uint16_t* perm, int* hist,
                   int* err_flag, float* ksum_to_clear, long ksum_elems, cudaStream_t stream);
int pixloss_prepare(const void* const* maps, const int* dtypes, const int* label_slots, int n_maps, int slot_off, int N,
                    int C, int HW, int do_normalize, int lo_slot_off, const uint16_t* perm, void* xn, float* inv_norm,
                    float* ksum, float* f32_to_clear, long f32_elems, cudaStream_t stream);
int pixloss_fwd(const void* xn, int n_slots, int n_label_slots, const uint8_t* lab_nat, const uint8_t* lab_sorted,
                const uint8_t* glab, const int* hist, const int* qmap, const int* qlab, const int* kmap, const int* klab,
                int n_terms, int Q, int S, int N, int C, int HW, float* stats, float* loss, float* loss_per_query, float* coef, const int* err_flag,
                float* partial, unsigned int* ticket, cudaStream_t stream);
int pixloss_bwd(const void* xn, int n_slots, int n_label_slots, const uint8_t* lab_nat, const uint8_t* lab_sorted,
                const uint8_t* glab, const int* qmap, const int* qmap_lo, const int* qlab, const int* kmap, const int* klab,
                int n_terms, int Q, int S, int N, int C, int HW, const float* coef, const float* ksum, const float* d_loss, float* dq32,
                int dq32_is_clear, const float* inv_norm, void* const* dq_out, int out_dtype, cudaStream_t stream);

// training-step kernels around the hot paths (trainaux.cu)
long ohem_ws_bytes();
int ohem_ce_fwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, long HW, int ignore_index,
                float thresh, long n_min, float* loss_px, void* ws, float* loss, float* sel, cudaStream_t stream);
int ohem_ce_bwd(const void* logits, int logits_is_f32, const int64_t* labels, int B, int K, long HW, int ignore_index,
                const float* loss_px, const float* sel, const float* d_loss, void* d_logits, cudaStream_t stream);
int ema_update(void* const* k_params, const void* const* q_params, void* const* k_shadows, const int64_t* numels,
               int n_tensors, float m, float one_minus_m, const float* m_dev, cudaStream_t stream);
int lars_sgd_step(void* const* params, void* const* grads, void* const* bufs, void* const* shadows, const int64_t* numels,
                  const uint8_t* first_step, int n_tensors, int grads_are_bf16, int write_grads, float lr,
                  const float* lr_dev, float momentum, float dampening, int nesterov, float weight_decay, int lars,
                  float trust_coef, float eps, double* norms_ws, cudaStream_t stream);

int adam_step(void* const* params, const void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
              void* const* shadows, const int64_t* numels, int n_tensors, int grads_are_bf16, float lr, float beta1,
              float beta2, float eps, float weight_decay, float grad_scale, float* step, cudaStream_t stream);
int sgd_step(void* const* params, const void* const* grads, void* const* momentum_bufs, void* const* shadows,
             const int64_t* numels, const uint8_t* first_step, int n_tensors, int grads_are_bf16, float lr, const float* lr_dev,
             float momentum, float one_minus_dampening, int nesterov, int maximize, float weight_decay, float grad_scale,
             cudaStream_t stream);
int gather_cast(void* const* dst, const void* const* src, const int64_t* numels, int n_tensors, int dst_is_bf16,
                cudaStream_t stream);

// fp32-accurate mode (f32path.cu)
int f32_split(const float* x, void* out, long R, int C, int layout, int pattern, int op, cudaStream_t stream);
int f32_rowop(float* out, const float* bias, const float* res, const float* aux, long R, int C, int mode, cudaStream_t stream);
int f32_colsum(const float* x, float* out, long R, int C, cudaStream_t stream);
int f32_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd, long M,
                      int row_len, float eps, int pm, int H, int W, int C, cudaStream_t stream);
int f32_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                      const float* dres, float* dx, float* dgamma, float* dbeta, long M, int row_len, int pm, int H, int W,
                      int C, cudaStream_t stream);
int winattn_f32_fwd(const float* qkv, const float* bias_table, float* out, float* lse, int B, int T, int H, int W, int C, int nH,
                    int ws, int shift, float qk_scale, const float* mask, int mask_windows, cudaStream_t stream);
int winattn_f32_bwd(const float* qkv, const float* bias_table, const float* out, const float* lse, const float* d_out,
                    float* d_qkv, float* d_bias_table, float* delta_ws, int B, int T, int H, int W, int C, int nH, int ws,
                    int shift, float qk_scale, const float* mask, int mask_windows, cudaStream_t stream);

}  // namespace stswin
