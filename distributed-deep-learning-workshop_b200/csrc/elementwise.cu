// Bandwidth-bound kernels of the image-classifier stack (SURVEY.md K10-K15, K17), NHWC bf16, fp32 math.
// Every kernel moves 16 bytes per thread per access (8 bf16 channels) and is written so one pass does as much
// as possible: BN-apply+ReLU+residual in one pass; BN-backward = one reduce pass + one apply pass that also
// emits the masked gradient for the skip connection; softmax-CE forward+backward+accuracy in one kernel.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ops_api.h"

namespace b200 {

struct alignas(16) bf16x8 {
  __nv_bfloat162 v[4];
};

__device__ __forceinline__ void unpack8(const bf16x8& p, float (&f)[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(p.v[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ bf16x8 pack8(const float (&f)[8]) {
  bf16x8 p;
#pragma unroll
  for (int i = 0; i < 4; ++i) p.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return p;
}
__device__ __forceinline__ bf16x8 ld8(const __nv_bfloat16* p) { return *reinterpret_cast<const bf16x8*>(p); }
__device__ __forceinline__ void st8(__nv_bfloat16* p, const bf16x8& v) { *reinterpret_cast<bf16x8*>(p) = v; }
__device__ __forceinline__ void ldf8(const float* p, float (&f)[8]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
  f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

static inline int grid_for(int64_t work, int threads, int max_blocks = 148 * 16) {
  int64_t b = (work + threads - 1) / threads;
  if (b > max_blocks) b = max_blocks;
  if (b < 1) b = 1;
  return (int)b;
}

// ------------------------------------------------------------------------------------------------ BN finalize
// sum/sqsum (accumulated by the conv epilogue or channel_stats) -> mean, invstd, scale, shift; running stats
// update; the accumulators are zeroed for the next step.
__global__ void bn_finalize_kernel(float* __restrict__ sum, float* __restrict__ sqsum, float inv_count,
                                   float unbias, const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* __restrict__ running_mean, float* __restrict__ running_var, float momentum,
                                   float eps, float* __restrict__ mean, float* __restrict__ invstd,
                                   float* __restrict__ scale, float* __restrict__ shift, int C, int training) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float m, var;
  if (training) {
    m = sum[c] * inv_count;
    var = fmaxf(sqsum[c] * inv_count - m * m, 0.f);
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * m;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * unbias;
  } else {
    m = running_mean[c];
    var = running_var[c];
  }
  sum[c] = 0.f;  // the conv epilogue accumulates into these in both modes
  sqsum[c] = 0.f;
  float is = rsqrtf(var + eps);
  mean[c] = m;
  invstd[c] = is;
  float sc = gamma[c] * is;
  scale[c] = sc;
  shift[c] = beta[c] - m * sc;
}

void bn_finalize(float* sum, float* sqsum, double count, const float* gamma, const float* beta, float* running_mean,
                 float* running_var, float momentum, float eps, float* mean, float* invstd, float* scale,
                 float* shift, int C, bool training, cudaStream_t s) {
  float unbias = count > 1 ? (float)(count / (count - 1.0)) : 1.f;
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, s>>>(sum, sqsum, (float)(1.0 / count), unbias, gamma, beta,
                                                      running_mean, running_var, momentum, eps, mean, invstd, scale,
                                                      shift, C, training ? 1 : 0);
}

// ------------------------------------------------------------------------------------------------ BN apply
// out = [relu]( y*scale + shift  [+ res | + res*res_scale + res_shift] )
// Column-resident: a thread owns one 8-channel column vector and walks down the rows, so the per-channel
// parameters are loaded into registers once instead of once per element (L1 traffic was 5x the payload).
template <bool RELU, int RES>  // RES: 0 none, 1 identity residual, 2 residual with its own BN
__global__ void __launch_bounds__(256, 1)
bn_apply_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                const float* __restrict__ shift, const __nv_bfloat16* __restrict__ res,
                const float* __restrict__ res_scale, const float* __restrict__ res_shift,
                __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ mask, int64_t M, int C) {
  const int cvec = C / 8;
  const int lanes = cvec < (int)blockDim.x ? cvec : blockDim.x;
  const int rpb = blockDim.x / lanes;
  const int cx = threadIdx.x % lanes;
  const int ry = threadIdx.x / lanes;
  if (ry >= rpb) return;
  for (int cv = cx; cv < cvec; cv += lanes) {
    float sc[8], sh[8], rs[8], rh[8];
    ldf8(scale + cv * 8, sc);
    ldf8(shift + cv * 8, sh);
    if (RES == 2) {
      ldf8(res_scale + cv * 8, rs);
      ldf8(res_shift + cv * 8, rh);
    }
    const int64_t rstep = (int64_t)gridDim.x * rpb;
    for (int64_t r = (int64_t)blockIdx.x * rpb + ry; r < M; r += rstep) {
      const int64_t off = r * C + cv * 8;
      const bf16x8 yraw = ld8(y + off);
      bf16x8 rraw;
      if (RES >= 1) rraw = ld8(res + off);
      float f[8];
      unpack8(yraw, f);
#pragma unroll
      for (int k = 0; k < 8; ++k) f[k] = fmaf(f[k], sc[k], sh[k]);
      if (RES >= 1) {
        float q[8];
        unpack8(rraw, q);
        if (RES == 2) {
#pragma unroll
          for (int k = 0; k < 8; ++k) q[k] = fmaf(q[k], rs[k], rh[k]);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] += q[k];
      }
      if (RELU) {
        if (mask != nullptr) {  // 1 bit per element: the backward pass reads this instead of the activation
          uint32_t mbits = 0;
#pragma unroll
          for (int k = 0; k < 8; ++k) mbits |= (f[k] > 0.f ? 1u : 0u) << k;
          mask[r * cvec + cv] = (uint8_t)mbits;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = fmaxf(f[k], 0.f);
      }
      st8(out + off, pack8(f));
    }
  }
}

static inline int rows_grid(int64_t M, int C, int threads) {
  const int cvec = C / 8;
  const int lanes = cvec < threads ? cvec : threads;
  const int rpb = threads / lanes;
  int64_t b = (M + rpb - 1) / rpb;
  const int64_t cap = 148 * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

void bn_apply(const void* y, const float* scale, const float* shift, const void* res, const float* res_scale,
              const float* res_shift, void* out, void* mask, int64_t M, int C, bool relu, cudaStream_t s) {
  const int threads = 256;
  const int blocks = rows_grid(M, C, threads);
  auto Y = (const __nv_bfloat16*)y;
  auto R = (const __nv_bfloat16*)res;
  auto O = (__nv_bfloat16*)out;
  auto MK = (uint8_t*)mask;
  const int rmode = res == nullptr ? 0 : (res_scale == nullptr ? 1 : 2);
  const auto kernel = relu ? (rmode == 0   ? bn_apply_kernel<true, 0>
                              : rmode == 1 ? bn_apply_kernel<true, 1>
                                           : bn_apply_kernel<true, 2>)
                           : (rmode == 0   ? bn_apply_kernel<false, 0>
                              : rmode == 1 ? bn_apply_kernel<false, 1>
                                           : bn_apply_kernel<false, 2>);
  kernel<<<blocks, threads, 0, s>>>(Y, scale, shift, R, res_scale, res_shift, O, MK, M, C);
}

// ------------------------------------------------------------------------------------------------ channel stats
// Column reductions over a [M, C] bf16 matrix.
//   MODE 0: sum(y), sum(y^2)                                   (BatchNorm statistics of a conv we did not run)
//   MODE 1: dz = (g1 [+ g2]) * (out > 0)      [dz optionally stored]   -> sum(dz), sum(dz*y)   (block-final BN)
//   MODE 2: dz = g1 * (y*scale + shift > 0)   (mask recomputed from y) -> sum(dz), sum(dz*y)   (BN + ReLU, no residual)
//   MODE 3: dz = g1                                                     -> sum(dz), sum(dz*y)   (BN without ReLU)
//   MODE 4: like MODE 1 but the ReLU mask is the 1-bit/element bitmap written by bn_apply (outp = uint8 [M, C/8])
template <int MODE>
__global__ void __launch_bounds__(256)
col_reduce_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ g2,
                  const __nv_bfloat16* __restrict__ outp, const __nv_bfloat16* __restrict__ y,
                  const float* __restrict__ scale, const float* __restrict__ shift,
                  __nv_bfloat16* __restrict__ dz_out, float* __restrict__ r0, float* __restrict__ r1, int64_t M, int C) {
  extern __shared__ float red[];  // [2][rows_per_block][C]
  const int cvec = C / 8;
  const int lanes = cvec < (int)blockDim.x ? cvec : blockDim.x;  // threads along channels
  const int rpb = blockDim.x / lanes;                            // rows processed concurrently
  const int cx = threadIdx.x % lanes;
  const int ry = threadIdx.x / lanes;
  const int64_t rows_per_block = (M + gridDim.x - 1) / gridDim.x;
  const int64_t r_begin = blockIdx.x * rows_per_block;
  const int64_t r_end = r_begin + rows_per_block < M ? r_begin + rows_per_block : M;
  float t0[8], t1[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) t0[k] = t1[k] = 0.f;
  if (ry < rpb && cx < cvec) {
    float sc[8], sh[8];
    if (MODE == 2) {
      ldf8(scale + cx * 8, sc);
      ldf8(shift + cx * 8, sh);
    }
    for (int64_t r = r_begin + ry; r < r_end; r += rpb) {
      const int64_t off = r * C + cx * 8;
      float f[8];
      unpack8(ld8(a + off), f);
      if (MODE == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          t0[k] += f[k];
          t1[k] = fmaf(f[k], f[k], t1[k]);
        }
      } else {
        float yy[8];
        unpack8(ld8(y + off), yy);
        if (MODE == 1 || MODE == 4) {
          if (g2 != nullptr) {
            float h[8];
            unpack8(ld8(g2 + off), h);
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] += h[k];
          }
          if (MODE == 1) {
            float o[8];
            unpack8(ld8(outp + off), o);
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] = o[k] > 0.f ? f[k] : 0.f;
          } else {
            const uint32_t mbits = reinterpret_cast<const uint8_t*>(outp)[r * cvec + cx];
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] = ((mbits >> k) & 1u) ? f[k] : 0.f;
          }
          if (dz_out != nullptr) st8(dz_out + off, pack8(f));
        } else if (MODE == 2) {
#pragma unroll
          for (int k = 0; k < 8; ++k) f[k] = fmaf(yy[k], sc[k], sh[k]) > 0.f ? f[k] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          t0[k] += f[k];
          t1[k] = fmaf(f[k], yy[k], t1[k]);
        }
      }
    }
  }
  // reduce across the rpb row-lanes through shared memory, then one atomic per channel per block
  float* sm0 = red;
  float* sm1 = red + rpb * C;
  if (ry < rpb && cx < cvec) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      sm0[ry * C + cx * 8 + k] = t0[k];
      sm1[ry * C + cx * 8 + k] = t1[k];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a0 = 0.f, a1 = 0.f;
    for (int r = 0; r < rpb; ++r) {
      a0 += sm0[r * C + c];
      a1 += sm1[r * C + c];
    }
    atomicAdd(r0 + c, a0);
    atomicAdd(r1 + c, a1);
  }
}

static void col_reduce_launch(int mode, const void* a, const void* g2, const void* outp, const void* y,
                              const float* scale, const float* shift, void* dz_out, float* r0, float* r1, int64_t M,
                              int C, cudaStream_t s) {
  const int threads = 256;
  int blocks = (int)((M + 31) / 32);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  const int cvec = C / 8;
  const int lanes = cvec < threads ? cvec : threads;
  const int rpb = threads / lanes;
  const size_t smem = (size_t)2 * rpb * C * sizeof(float);
  auto A = (const __nv_bfloat16*)a;
  auto G2 = (const __nv_bfloat16*)g2;
  auto O = (const __nv_bfloat16*)outp;
  auto Y = (const __nv_bfloat16*)y;
  auto DZ = (__nv_bfloat16*)dz_out;
  switch (mode) {
    case 0: col_reduce_kernel<0><<<blocks, threads, smem, s>>>(A, G2, O, Y, scale, shift, DZ, r0, r1, M, C); break;
    case 1: col_reduce_kernel<1><<<blocks, threads, smem, s>>>(A, G2, O, Y, scale, shift, DZ, r0, r1, M, C); break;
    case 2: col_reduce_kernel<2><<<blocks, threads, smem, s>>>(A, G2, O, Y, scale, shift, DZ, r0, r1, M, C); break;
    case 4: col_reduce_kernel<4><<<blocks, threads, smem, s>>>(A, G2, O, Y, scale, shift, DZ, r0, r1, M, C); break;
    default: col_reduce_kernel<3><<<blocks, threads, smem, s>>>(A, G2, O, Y, scale, shift, DZ, r0, r1, M, C); break;
  }
}

void channel_stats(const void* y, float* sum, float* sqsum, int64_t M, int C, cudaStream_t s) {
  col_reduce_launch(0, y, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, sum, sqsum, M, C, s);
}
// mode 1: mask from `outp` (g2 optional, dz_out optional);  mode 2: mask from y*scale+shift;  mode 3: no mask
void bn_bwd_reduce(int mode, const void* g1, const void* g2, const void* outp, const void* y, const float* scale,
                   const float* shift, void* dz_out, float* sum_dz, float* sum_dzy, int64_t M, int C, cudaStream_t s) {
  col_reduce_launch(mode, g1, g2, outp, y, scale, shift, dz_out, sum_dz, sum_dzy, M, C, s);
}

// ------------------------------------------------------------------------------------------------ BN bwd coeffs
// dy = A*dz + B*y + Cc   with  A = gamma*invstd,  B = -A*invstd*dgamma/M,  Cc = -A*dbeta/M - B*mean
__global__ void bn_bwd_coeffs_kernel(float* __restrict__ sum_dz, float* __restrict__ sum_dzy,
                                     const float* __restrict__ gamma, const float* __restrict__ mean,
                                     const float* __restrict__ invstd, float inv_count, float* __restrict__ dgamma,
                                     float* __restrict__ dbeta, float* __restrict__ cA, float* __restrict__ cB,
                                     float* __restrict__ cC, int C) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float db = sum_dz[c];
  const float dzy = sum_dzy[c];
  sum_dz[c] = 0.f;
  sum_dzy[c] = 0.f;
  const float m = mean[c], is = invstd[c];
  const float dg = is * (dzy - m * db);
  dgamma[c] = dg;
  dbeta[c] = db;
  const float A = gamma[c] * is;
  const float B = -A * is * dg * inv_count;
  cA[c] = A;
  cB[c] = B;
  cC[c] = -A * db * inv_count - B * m;
}
void bn_bwd_coeffs(float* sum_dz, float* sum_dzy, const float* gamma, const float* mean, const float* invstd,
                   double count, float* dgamma, float* dbeta, float* cA, float* cB, float* cC, int C,
                   cudaStream_t s) {
  bn_bwd_coeffs_kernel<<<(C + 127) / 128, 128, 0, s>>>(sum_dz, sum_dzy, gamma, mean, invstd, (float)(1.0 / count),
                                                        dgamma, dbeta, cA, cB, cC, C);
}

// dy = A*dz + B*y + Cc  with dz either read as-is (MASK=false: stored dz / BN without ReLU) or recomputed as
// g * (y*scale + shift > 0) (MASK=true).  Column-resident like bn_apply_kernel.
template <bool MASK>
__global__ void __launch_bounds__(256, 1)
bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ g, const __nv_bfloat16* __restrict__ y,
                    const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ cA, const float* __restrict__ cB,
                    const float* __restrict__ cC, __nv_bfloat16* __restrict__ dy, int64_t M, int C) {
  const int cvec = C / 8;
  const int lanes = cvec < (int)blockDim.x ? cvec : blockDim.x;
  const int rpb = blockDim.x / lanes;
  const int cx = threadIdx.x % lanes;
  const int ry = threadIdx.x / lanes;
  if (ry >= rpb) return;
  for (int cv = cx; cv < cvec; cv += lanes) {
    float A[8], B[8], Cc[8], sc[8], sh[8];
    ldf8(cA + cv * 8, A);
    ldf8(cB + cv * 8, B);
    ldf8(cC + cv * 8, Cc);
    if (MASK) {
      ldf8(scale + cv * 8, sc);
      ldf8(shift + cv * 8, sh);
    }
    const int64_t rstep = (int64_t)gridDim.x * rpb;
    for (int64_t r = (int64_t)blockIdx.x * rpb + ry; r < M; r += rstep) {
      const int64_t off = r * C + cv * 8;
      const bf16x8 graw = ld8(g + off);
      const bf16x8 yraw = ld8(y + off);
      float gg[8], yy[8];
      unpack8(graw, gg);
      unpack8(yraw, yy);
      if (MASK) {
#pragma unroll
        for (int k = 0; k < 8; ++k) gg[k] = fmaf(yy[k], sc[k], sh[k]) > 0.f ? gg[k] : 0.f;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) gg[k] = fmaf(A[k], gg[k], fmaf(B[k], yy[k], Cc[k]));
      st8(dy + off, pack8(gg));
    }
  }
}
void bn_bwd_apply(const void* g, const void* y, const float* scale, const float* shift, const float* cA,
                  const float* cB, const float* cC, void* dy, int64_t M, int C, cudaStream_t s) {
  const int threads = 256;
  const int blocks = rows_grid(M, C, threads);
  const auto kernel = scale != nullptr ? bn_bwd_apply_kernel<true> : bn_bwd_apply_kernel<false>;
  kernel<<<blocks, threads, 0, s>>>((const __nv_bfloat16*)g, (const __nv_bfloat16*)y, scale, shift, cA, cB, cC,
                                    (__nv_bfloat16*)dy, M, C);
}

// ------------------------------------------------------------------------------------------------ max pool 3x3 s2 p1
// Forward also stores the window position (0..8, first maximum in row-major scan order = torch's tie rule) so
// that backward is a pure gather: every input pixel checks the <= 4 windows that contain it.
__global__ void maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                   uint8_t* __restrict__ idx, int N, int H, int W, int C, int Ho, int Wo) {
  const int cvec = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * cvec;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % cvec);
    int64_t p = i / cvec;
    const int wo = (int)(p % Wo);
    p /= Wo;
    const int ho = (int)(p % Ho);
    const int n = (int)(p / Ho);
    float m[8];
    uint32_t am[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      m[k] = -3.0e38f;
      am[k] = 0;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int h = 2 * ho - 1 + r;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int w = 2 * wo - 1 + q;
        if (w < 0 || w >= W) continue;
        float f[8];
        unpack8(ld8(x + (((int64_t)n * H + h) * W + w) * C + cv * 8), f);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          if (f[k] > m[k]) {
            m[k] = f[k];
            am[k] = r * 3 + q;
          }
        }
      }
    }
    st8(out + i * 8, pack8(m));
    if (idx != nullptr) {
      uint2 pk;
      pk.x = am[0] | (am[1] << 8) | (am[2] << 16) | (am[3] << 24);
      pk.y = am[4] | (am[5] << 8) | (am[6] << 16) | (am[7] << 24);
      *reinterpret_cast<uint2*>(idx + i * 8) = pk;
    }
  }
}
void maxpool_fwd(const void* x, void* out, void* idx, int N, int H, int W, int C, cudaStream_t s) {
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  const int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  maxpool_fwd_kernel<<<grid_for(total, 256), 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)out, (uint8_t*)idx,
                                                          N, H, W, C, Ho, Wo);
}

// Stem tail in one pass: out = maxpool3x3/2( relu( y*scale + shift ) ) + argmax; the 112x112 post-ReLU activation is
// never materialised (its backward needs only y, the BN affine and the argmax).
__global__ void __launch_bounds__(256)
bn_relu_maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale,
                           const float* __restrict__ shift, __nv_bfloat16* __restrict__ out,
                           uint8_t* __restrict__ idx, int N, int H, int W, int C, int Ho, int Wo) {
  const int cvec = C / 8;
  const int64_t total = (int64_t)N * Ho * Wo * cvec;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % cvec);
    int64_t p = i / cvec;
    const int wo = (int)(p % Wo);
    p /= Wo;
    const int ho = (int)(p % Ho);
    const int n = (int)(p / Ho);
    float sc[8], sh[8], m[8];
    uint32_t am[8];
    ldf8(scale + cv * 8, sc);
    ldf8(shift + cv * 8, sh);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      m[k] = -3.0e38f;
      am[k] = 0;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int h = 2 * ho - 1 + r;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int w = 2 * wo - 1 + q;
        if (w < 0 || w >= W) continue;
        float f[8];
        unpack8(ld8(y + (((int64_t)n * H + h) * W + w) * C + cv * 8), f);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          // same rounding as the materialised path: bf16(relu(fma))
          const float a = __bfloat162float(__float2bfloat16(fmaxf(fmaf(f[k], sc[k], sh[k]), 0.f)));
          if (a > m[k]) {
            m[k] = a;
            am[k] = r * 3 + q;
          }
        }
      }
    }
    st8(out + i * 8, pack8(m));
    if (idx != nullptr) {
      uint2 pk;
      pk.x = am[0] | (am[1] << 8) | (am[2] << 16) | (am[3] << 24);
      pk.y = am[4] | (am[5] << 8) | (am[6] << 16) | (am[7] << 24);
      *reinterpret_cast<uint2*>(idx + i * 8) = pk;
    }
  }
}
void bn_relu_maxpool_fwd(const void* y, const float* scale, const float* shift, void* out, void* idx, int N, int H,
                         int W, int C, cudaStream_t s) {
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  const int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  bn_relu_maxpool_fwd_kernel<<<grid_for(total, 256), 256, 0, s>>>((const __nv_bfloat16*)y, scale, shift,
                                                                  (__nv_bfloat16*)out, (uint8_t*)idx, N, H, W, C, Ho, Wo);
}

// dx[h, w] = sum over windows (ho, wo) containing (h, w) whose argmax is this position of (g1 [+ g2])[ho, wo].
__global__ void maxpool_bwd_kernel(const uint8_t* __restrict__ idx, const __nv_bfloat16* __restrict__ g1,
                                   const __nv_bfloat16* __restrict__ g2, __nv_bfloat16* __restrict__ dx, int N, int H,
                                   int W, int C, int Ho, int Wo) {
  const int cvec = C / 8;
  const int64_t total = (int64_t)N * H * W * cvec;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % cvec);
    int64_t p = i / cvec;
    const int w = (int)(p % W);
    p /= W;
    const int h = (int)(p % H);
    const int n = (int)(p / H);
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    // windows containing (h, w): 2*ho-1 <= h <= 2*ho+1  <=>  ho in [h/2, (h+1)/2]
    for (int ho = h / 2; ho <= (h + 1) / 2; ++ho) {
      if (ho >= Ho) continue;
      const int r = h - (2 * ho - 1);
      for (int wo = w / 2; wo <= (w + 1) / 2; ++wo) {
        if (wo >= Wo) continue;
        const uint32_t pos = r * 3 + (w - (2 * wo - 1));
        const int64_t o = ((((int64_t)n * Ho + ho) * Wo + wo) * C) + cv * 8;
        const uint2 pk = *reinterpret_cast<const uint2*>(idx + o);
        float gv[8];
        unpack8(ld8(g1 + o), gv);
        if (g2 != nullptr) {
          float hv[8];
          unpack8(ld8(g2 + o), hv);
#pragma unroll
          for (int k = 0; k < 8; ++k) gv[k] += hv[k];
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint32_t a = ((k < 4 ? pk.x : pk.y) >> (8 * (k & 3))) & 0xFFu;
          acc[k] += (a == pos) ? gv[k] : 0.f;
        }
      }
    }
    st8(dx + i * 8, pack8(acc));
  }
}
void maxpool_bwd(const void* idx, const void* g1, const void* g2, void* dx, int N, int H, int W, int C,
                 cudaStream_t s) {
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  const int64_t total = (int64_t)N * H * W * (C / 8);
  maxpool_bwd_kernel<<<grid_for(total, 256), 256, 0, s>>>((const uint8_t*)idx, (const __nv_bfloat16*)g1,
                                                          (const __nv_bfloat16*)g2, (__nv_bfloat16*)dx, N, H, W, C, Ho,
                                                          Wo);
}

// ------------------------------------------------------------------------------------------------ global avg pool
// x [N, HW, C] -> out [N, C]  (optionally with inverted-dropout mask from a counter-based hash RNG)
__device__ __forceinline__ uint32_t hash_u32(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t h = a * 0x9E3779B1u ^ (b + 0x7F4A7C15u) * 0x85EBCA77u ^ (c + 0x165667B1u) * 0xC2B2AE3Du;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
  return h;
}
__global__ void gap_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out, int N, int HW,
                               int C, float keep_scale, uint32_t keep_thresh, uint32_t seed_lo, uint32_t seed_hi) {
  const int cvec = C / 8;
  const int64_t total = (int64_t)N * cvec;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % cvec);
    const int n = (int)(i / cvec);
    float a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = 0.f;
    for (int p = 0; p < HW; ++p) {
      float f[8];
      unpack8(ld8(x + ((int64_t)n * HW + p) * C + cv * 8), f);
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] += f[k];
    }
    const float inv = 1.f / HW;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float v = a[k] * inv;
      if (keep_thresh != 0xFFFFFFFFu) {
        const uint32_t r = hash_u32(seed_lo, seed_hi, (uint32_t)(i * 8 + k));
        v = (r <= keep_thresh) ? v * keep_scale : 0.f;
      }
      a[k] = v;
    }
    st8(out + i * 8, pack8(a));
  }
}
void gap_fwd(const void* x, void* out, int N, int HW, int C, float drop_p, uint64_t seed, cudaStream_t s) {
  const int64_t total = (int64_t)N * (C / 8);
  uint32_t thresh = 0xFFFFFFFFu;
  float ks = 1.f;
  if (drop_p > 0.f) {
    thresh = (uint32_t)((1.0 - (double)drop_p) * 4294967295.0);
    ks = 1.f / (1.f - drop_p);
  }
  gap_fwd_kernel<<<grid_for(total, 128), 128, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)out, N, HW, C, ks,
                                                      thresh, (uint32_t)seed, (uint32_t)(seed >> 32));
}
__global__ void gap_bwd_kernel(const __nv_bfloat16* __restrict__ dout, __nv_bfloat16* __restrict__ dx, int N, int HW,
                               int C, float keep_scale, uint32_t keep_thresh, uint32_t seed_lo, uint32_t seed_hi) {
  const int cvec = C / 8;
  const int64_t total = (int64_t)N * HW * cvec;
  const float inv = 1.f / HW;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % cvec);
    const int n = (int)(i / ((int64_t)HW * cvec));
    const int64_t j = (int64_t)n * cvec + cv;
    float g[8];
    unpack8(ld8(dout + j * 8), g);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float v = g[k] * inv;
      if (keep_thresh != 0xFFFFFFFFu) {
        const uint32_t r = hash_u32(seed_lo, seed_hi, (uint32_t)(j * 8 + k));
        v = (r <= keep_thresh) ? v * keep_scale : 0.f;
      }
      g[k] = v;
    }
    st8(dx + i * 8, pack8(g));
  }
}
void gap_bwd(const void* dout, void* dx, int N, int HW, int C, float drop_p, uint64_t seed, cudaStream_t s) {
  const int64_t total = (int64_t)N * HW * (C / 8);
  uint32_t thresh = 0xFFFFFFFFu;
  float ks = 1.f;
  if (drop_p > 0.f) {
    thresh = (uint32_t)((1.0 - (double)drop_p) * 4294967295.0);
    ks = 1.f / (1.f - drop_p);
  }
  gap_bwd_kernel<<<grid_for(total, 256), 256, 0, s>>>((const __nv_bfloat16*)dout, (__nv_bfloat16*)dx, N, HW, C, ks,
                                                      thresh, (uint32_t)seed, (uint32_t)(seed >> 32));
}

// ------------------------------------------------------------------------------------------------ softmax CE
// One warp per row.  logits fp32 [B, K] -> per-row loss, dlogits = (softmax - onehot) * grad_scale,
// and the running (sum loss, correct count) pair in stats[0..1] via atomics.
__global__ void softmax_ce_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                  float* __restrict__ dlogits, float* __restrict__ loss_rows,
                                  float* __restrict__ stats, int B, int K, float grad_scale) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= B) return;
  const float* row = logits + (int64_t)warp * K;
  const int label = (int)labels[warp];
  float mx = -3.0e38f;
  int amax = 0;
  for (int k = lane; k < K; k += 32) {
    const float v = row[k];
    if (v > mx) { mx = v; amax = k; }
  }
  for (int o = 16; o; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, amax, o);
    if (om > mx || (om == mx && oa < amax)) { mx = om; amax = oa; }
  }
  float se = 0.f;
  for (int k = lane; k < K; k += 32) se += __expf(row[k] - mx);
  for (int o = 16; o; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  const float lse = mx + __logf(se);
  const float inv = 1.f / se;
  if (dlogits != nullptr) {
    float* drow = dlogits + (int64_t)warp * K;
    for (int k = lane; k < K; k += 32) {
      const float pk = __expf(row[k] - mx) * inv;
      drow[k] = (pk - (k == label ? 1.f : 0.f)) * grad_scale;
    }
  }
  if (lane == 0) {
    const float l = lse - row[label];
    if (loss_rows != nullptr) loss_rows[warp] = l;
    atomicAdd(stats, l);
    atomicAdd(stats + 1, amax == label ? 1.f : 0.f);
  }
}
void softmax_ce(const float* logits, const int64_t* labels, float* dlogits, float* loss_rows, float* stats, int B,
                int K, float grad_scale, cudaStream_t s) {
  const int threads = 128;
  const int blocks = (B * 32 + threads - 1) / threads;
  softmax_ce_kernel<<<blocks, threads, 0, s>>>(logits, labels, dlogits, loss_rows, stats, B, K, grad_scale);
}

// Bilinear resize (half-pixel centres, like tf.image.resize) of one uint8 image batch to [N, OH, OW, 3] uint8 (HWC).
// PLANAR: the input is [N, 3, H, W] (what nvJPEG / torchvision.io.decode_jpeg produce), otherwise [N, H, W, 3].
template <bool PLANAR>
__global__ void resize_bilinear_u8_kernel(const uint8_t* __restrict__ x, uint8_t* __restrict__ out, int N, int H,
                                          int W, int OH, int OW) {
  const int64_t total = (int64_t)N * OH * OW;
  const float sy = (float)H / OH, sx = (float)W / OW;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ow = (int)(i % OW);
    const int oh = (int)((i / OW) % OH);
    const int n = (int)(i / ((int64_t)OW * OH));
    float fy = (oh + 0.5f) * sy - 0.5f, fx = (ow + 0.5f) * sx - 0.5f;
    fy = fminf(fmaxf(fy, 0.f), (float)(H - 1));
    fx = fminf(fmaxf(fx, 0.f), (float)(W - 1));
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
    const float wy = fy - y0, wx = fx - x0;
    const uint8_t* b = x + (int64_t)n * H * W * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float v00, v01, v10, v11;
      if (PLANAR) {
        const uint8_t* pc = b + (int64_t)c * H * W;
        v00 = pc[(int64_t)y0 * W + x0]; v01 = pc[(int64_t)y0 * W + x1];
        v10 = pc[(int64_t)y1 * W + x0]; v11 = pc[(int64_t)y1 * W + x1];
      } else {
        v00 = b[((int64_t)y0 * W + x0) * 3 + c]; v01 = b[((int64_t)y0 * W + x1) * 3 + c];
        v10 = b[((int64_t)y1 * W + x0) * 3 + c]; v11 = b[((int64_t)y1 * W + x1) * 3 + c];
      }
      const float v = (v00 * (1 - wx) + v01 * wx) * (1 - wy) + (v10 * (1 - wx) + v11 * wx) * wy;
      out[i * 3 + c] = (uint8_t)fminf(fmaxf(v + 0.5f, 0.f), 255.f);
    }
  }
}
void resize_bilinear_u8(const uint8_t* x, uint8_t* out, int N, int H, int W, int OH, int OW, bool planar, cudaStream_t s) {
  if (planar)
    resize_bilinear_u8_kernel<true><<<grid_for((int64_t)N * OH * OW, 256), 256, 0, s>>>(x, out, N, H, W, OH, OW);
  else
    resize_bilinear_u8_kernel<false><<<grid_for((int64_t)N * OH * OW, 256), 256, 0, s>>>(x, out, N, H, W, OH, OW);
}

// ------------------------------------------------------------------------------------------------ weight layouts
// fp32 master [taps][Cout][Cin] -> bf16 forward copy (same layout) and bf16 dgrad copy [taps][Cin][Cout]
// (per-tap transpose; the dgrad plan pairs tap t with the mirrored pixel offset).
__global__ void weight_prep_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                                   __nv_bfloat16* __restrict__ wd, int taps, int cout, int cin) {
  const int64_t total = (int64_t)taps * cout * cin;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ci = (int)(i % cin);
    const int co = (int)((i / cin) % cout);
    const int t = (int)(i / ((int64_t)cin * cout));
    const __nv_bfloat16 v = __float2bfloat16(w[i]);
    if (wf != nullptr) wf[i] = v;
    if (wd != nullptr) wd[((int64_t)t * cin + ci) * cout + co] = v;
  }
}
void weight_prep(const float* w, void* wf, void* wd, int taps, int cout, int cin, cudaStream_t s) {
  weight_prep_kernel<<<grid_for((int64_t)taps * cout * cin, 256, 148 * 4), 256, 0, s>>>(
      w, (__nv_bfloat16*)wf, (__nv_bfloat16*)wd, taps, cout, cin);
}


// All filters in one launch: table rows = (src offset in the flat fp32 master, dst offset in the flat bf16 dgrad buffer,
// taps, cout, cin, first TILE index of the row).  Every tap matrix [cout, cin] fp32 is transposed to [cin, cout] bf16
// through 64x32 shared-memory tiles: 128-byte coalesced reads (32 floats of one co row) and 128-byte coalesced writes
// (64 bf16 of one ci row).  The element-wise version it replaces wrote 2-byte values at a cout-element stride and spent
// ~0.29 ms per step on 141 MB of traffic (~20 us at HBM speed).  cout % 64 == 0 and cin % 32 == 0 (host-checked).
__global__ void __launch_bounds__(256)
weight_prep_batched_kernel(const float* __restrict__ params, __nv_bfloat16* __restrict__ wd,
                           const int64_t* __restrict__ table, int layers, int64_t total_tiles) {
  __shared__ int64_t t[128 * 6];
  __shared__ float tile[64][33];
  for (int i = threadIdx.x; i < layers * 6; i += blockDim.x) t[i] = table[i];
  __syncthreads();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int64_t tid = blockIdx.x; tid < total_tiles; tid += gridDim.x) {
    int lo = 0, hi = layers - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (t[mid * 6 + 5] <= tid) lo = mid; else hi = mid - 1;
    }
    const int64_t* L = t + lo * 6;
    const int cout = (int)L[3], cin = (int)L[4];
    const int tiles_ci = cin >> 5, tiles_co = cout >> 6;
    int64_t j = tid - L[5];
    const int tci = (int)(j % tiles_ci);
    j /= tiles_ci;
    const int tco = (int)(j % tiles_co);
    const int tp = (int)(j / tiles_co);
    const float* src = params + L[0] + ((int64_t)tp * cout + tco * 64) * cin + tci * 32;
    __nv_bfloat16* dst = wd + L[1] + ((int64_t)tp * cin + tci * 32) * cout + tco * 64;
    __syncthreads();  // previous tile fully written out
#pragma unroll
    for (int r = ty; r < 64; r += 8) tile[r][tx] = src[(int64_t)r * cin + tx];
    __syncthreads();
#pragma unroll
    for (int c = ty; c < 32; c += 8) {
      const __nv_bfloat162 v = __floats2bfloat162_rn(tile[2 * tx][c], tile[2 * tx + 1][c]);
      *reinterpret_cast<__nv_bfloat162*>(dst + (int64_t)c * cout + 2 * tx) = v;
    }
  }
}
void weight_prep_batched(const float* params, void* wd, const int64_t* table, int layers, int64_t total_tiles,
                         cudaStream_t s) {
  int64_t grid = total_tiles < 148 * 16 ? total_tiles : 148 * 16;
  if (grid < 1) grid = 1;
  weight_prep_batched_kernel<<<(int)grid, 256, 0, s>>>(params, (__nv_bfloat16*)wd, table, layers, total_tiles);
}

}  // namespace b200
