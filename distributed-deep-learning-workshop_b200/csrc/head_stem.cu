// Classifier-head and stem-weight kernels (SURVEY.md K11, K14, K15): the bandwidth-bound glue around the two GEMM-shaped
// ends of the network.  The FC layer itself runs on the tcgen05 implicit-GEMM kernels (a 1x1 "convolution" over a 1x1
// image, csrc/conv_igemm.cuh / conv_wgrad.cu); what lives here is everything the reference's Dense + softmax head
// (P1/02:175) needs besides the GEMMs:
//   * softmax_ce_head: bf16 logits + fp32 bias -> loss, accuracy, bf16 dlogits (padded columns zero) in one pass;
//   * fc_bias_grad: column sums of dlogits;
//   * pack_stem_weight: fp32 [49, 64, 3] master -> bf16 [64, 192] GEMM operand.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ops_api.h"

namespace b200 {

// ------------------------------------------------------------------------------------------------ softmax CE head
// One warp per row.  logit[k] = bf16 logits16[row, k] + bias[k] for k < K (row pitch ld >= K, padded columns ignored).
__global__ void softmax_ce_head_kernel(const __nv_bfloat16* __restrict__ logits16, int ld,
                                       const float* __restrict__ bias, const int64_t* __restrict__ labels,
                                       float* __restrict__ logits32, __nv_bfloat16* __restrict__ dlogits16,
                                       float* __restrict__ loss_rows, float* __restrict__ stats, int B, int K,
                                       float grad_scale) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B) return;
  const __nv_bfloat16* row = logits16 + (int64_t)warp * ld;
  const int label = (int)labels[warp];
  float mx = -3.0e38f;
  int amax = 0;
  for (int k = lane; k < K; k += 32) {
    const float v = __bfloat162float(row[k]) + bias[k];
    if (logits32 != nullptr) logits32[(int64_t)warp * K + k] = v;
    if (v > mx) { mx = v; amax = k; }
  }
  for (int o = 16; o; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, amax, o);
    if (om > mx || (om == mx && oa < amax)) { mx = om; amax = oa; }
  }
  float se = 0.f;
  for (int k = lane; k < K; k += 32) se += __expf(__bfloat162float(row[k]) + bias[k] - mx);
  for (int o = 16; o; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  const float lse = mx + __logf(se);
  const float inv = 1.f / se;
  if (dlogits16 != nullptr) {
    __nv_bfloat16* drow = dlogits16 + (int64_t)warp * ld;
    for (int k = lane; k < ld; k += 32) {
      float d = 0.f;
      if (k < K) {
        const float pk = __expf(__bfloat162float(row[k]) + bias[k] - mx) * inv;
        d = (pk - (k == label ? 1.f : 0.f)) * grad_scale;
      }
      drow[k] = __float2bfloat16(d);
    }
  }
  if (lane == 0) {
    const float l = lse - (__bfloat162float(row[label]) + bias[label]);
    if (loss_rows != nullptr) loss_rows[warp] = l;
    atomicAdd(stats, l);
    atomicAdd(stats + 1, amax == label ? 1.f : 0.f);
  }
}
void softmax_ce_head(const void* logits16, int ld, const float* bias, const int64_t* labels, float* logits32,
                     void* dlogits16, float* loss_rows, float* stats, int B, int K, float grad_scale, cudaStream_t s) {
  const int threads = 128;
  const int blocks = (B * 32 + threads - 1) / threads;
  softmax_ce_head_kernel<<<blocks, threads, 0, s>>>((const __nv_bfloat16*)logits16, ld, bias, labels, logits32,
                                                    (__nv_bfloat16*)dlogits16, loss_rows, stats, B, K, grad_scale);
}

// dbias[k] = sum_b dlogits16[b, k]   (thread per column: coalesced across k for every row)
__global__ void fc_bias_grad_kernel(const __nv_bfloat16* __restrict__ dl, int ld, float* __restrict__ dbias, int B, int K) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int b = 0;
  for (; b + 4 <= B; b += 4) {
    a0 += __bfloat162float(dl[(int64_t)(b + 0) * ld + k]);
    a1 += __bfloat162float(dl[(int64_t)(b + 1) * ld + k]);
    a2 += __bfloat162float(dl[(int64_t)(b + 2) * ld + k]);
    a3 += __bfloat162float(dl[(int64_t)(b + 3) * ld + k]);
  }
  for (; b < B; ++b) a0 += __bfloat162float(dl[(int64_t)b * ld + k]);
  dbias[k] = (a0 + a1) + (a2 + a3);
}
void fc_bias_grad(const void* dlogits16, int ld, float* dbias, int B, int K, cudaStream_t s) {
  fc_bias_grad_kernel<<<(K + 127) / 128, 128, 0, s>>>((const __nv_bfloat16*)dlogits16, ld, dbias, B, K);
}

// ------------------------------------------------------------------------------------------------ stem weight pack
// fp32 [49, 64, 3] (tap, co, c) -> bf16 [64, 192] with k = tap*3 + c (columns 147.. are zero)
__global__ void pack_stem_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 192) return;
  const int co = i / 192, k = i - co * 192;
  float v = 0.f;
  if (k < 147) v = w[((k / 3) * 64 + co) * 3 + (k % 3)];
  out[i] = __float2bfloat16(v);
}
void pack_stem_weight(const float* w, void* out, cudaStream_t s) {
  pack_stem_weight_kernel<<<(64 * 192 + 255) / 256, 256, 0, s>>>(w, (__nv_bfloat16*)out);
}

}  // namespace b200
