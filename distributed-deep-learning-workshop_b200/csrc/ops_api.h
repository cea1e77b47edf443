// Plain (torch-free) launch interface of the bandwidth-bound kernels and fused optimizers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

void bn_finalize(float* sum, float* sqsum, double count, const float* gamma, const float* beta, float* running_mean,
                 float* running_var, float momentum, float eps, float* mean, float* invstd, float* scale,
                 float* shift, int C, bool training, cudaStream_t s);
void bn_apply(const void* y, const float* scale, const float* shift, const void* res, const float* res_scale,
              const float* res_shift, void* out, void* mask, int64_t M, int C, bool relu, cudaStream_t s);
void channel_stats(const void* y, float* sum, float* sqsum, int64_t M, int C, cudaStream_t s);
void bn_bwd_reduce(int mode, const void* g1, const void* g2, const void* outp, const void* y, const float* scale,
                   const float* shift, void* dz_out, float* sum_dz, float* sum_dzy, int64_t M, int C, cudaStream_t s);
void bn_bwd_coeffs(float* sum_dz, float* sum_dzy, const float* gamma, const float* mean, const float* invstd,
                   double count, float* dgamma, float* dbeta, float* cA, float* cB, float* cC, int C, cudaStream_t s);
void bn_bwd_apply(const void* g, const void* y, const float* scale, const float* shift, const float* cA,
                  const float* cB, const float* cC, void* dy, int64_t M, int C, cudaStream_t s);
void maxpool_fwd(const void* x, void* out, void* idx, int N, int H, int W, int C, cudaStream_t s);
void bn_relu_maxpool_fwd(const void* y, const float* scale, const float* shift, void* out, void* idx, int N, int H,
                         int W, int C, cudaStream_t s);
void maxpool_bwd(const void* idx, const void* g1, const void* g2, void* dx, int N, int H, int W, int C,
                 cudaStream_t s);
void gap_fwd(const void* x, void* out, int N, int HW, int C, float drop_p, uint64_t seed, cudaStream_t s);
void gap_bwd(const void* dout, void* dx, int N, int HW, int C, float drop_p, uint64_t seed, cudaStream_t s);
void softmax_ce(const float* logits, const int64_t* labels, float* dlogits, float* loss_rows, float* stats, int B,
                int K, float grad_scale, cudaStream_t s);
void softmax_ce_head(const void* logits16, int ld, const float* bias, const int64_t* labels, float* logits32,
                     void* dlogits16, float* loss_rows, float* stats, int B, int K, float grad_scale, cudaStream_t s);
void fc_bias_grad(const void* dlogits16, int ld, float* dbias, int B, int K, cudaStream_t s);
void pack_stem_weight(const float* w, void* out, cudaStream_t s);
void mbv2_stem(const uint8_t* x, const float* w, const float* scale, const float* shift, void* out, int N, int H, int W,
               int ldc, float mul, float add, cudaStream_t s);
void dwconv3x3(const void* x, const float* w, const float* scale, const float* shift, void* out, int N, int H, int W, int C,
               int stride, int tile_w, cudaStream_t s);
void resize_bilinear_u8(const uint8_t* x, uint8_t* out, int N, int H, int W, int OH, int OW, bool planar, cudaStream_t s);
void weight_prep(const float* w, void* wf, void* wd, int taps, int cout, int cin, cudaStream_t s);
void weight_prep_batched(const float* params, void* wd, const int64_t* table, int layers, int64_t total,
                         cudaStream_t s);

// Fused flat-buffer optimizers.  `hyper` is a DEVICE array (so LR schedules do not invalidate CUDA graphs):
//   [0] lr  [1] momentum/beta1  [2] beta2/rho  [3] eps  [4] weight_decay  [5] grad_scale  [6] bias_corr1  [7] bias_corr2
constexpr int kHyperLen = 8;
void sgd_step(float* p, const float* g, float* mom, void* p16, int64_t n, const float* hyper, bool nesterov,
              cudaStream_t s);
void adam_step(float* p, const float* g, float* m, float* v, void* p16, int64_t n, const float* hyper, cudaStream_t s);
void adadelta_step(float* p, const float* g, float* sq, float* acc, void* p16, int64_t n, const float* hyper,
                   cudaStream_t s);
void cast_f32_to_bf16(const float* x, void* out, int64_t n, cudaStream_t s);

}  // namespace b200
