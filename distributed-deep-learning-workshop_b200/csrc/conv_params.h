// Kernel parameter blocks shared by device code and the (torch-facing) host code.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace b200 {

constexpr int kMaxTaps = 16;
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 bf16 = 128 B = one SWIZZLE_128B row

struct ConvParams {
  int mode;      // 0 = flat, 1 = box
  int taps;      // number of filter taps (1, 9, ...)
  int kblocks;   // Cin / 64
  int n_blocks;  // Cout / BLOCK_N
  int cout;
  int m_tiles;
  int num_tiles;   // m_tiles * n_blocks
  int valid_rows;  // rows of the 128-row tile that hold real pixels (box mode may use < 128)
  int bw, bh, bn;  // box extents
  int tiles_w, tiles_h;
  int8_t tap_map[kMaxTaps];  // which A tensor map the tap reads
  int8_t tap_dw[kMaxTaps];   // coordinate offsets (in the view's pixel grid)
  int8_t tap_dh[kMaxTaps];
  float* stat_sum;    // [Cout] or nullptr   (mode 2: sum dz)
  float* stat_sqsum;  // [Cout] or nullptr   (mode 2: sum dz*y)
  const float* bn_scale;  // mode 2: forward BN affine of the activation whose gradient this GEMM produces
  const float* bn_shift;
  // Halo mode (3x3 stride 1, full-width pixel boxes, resident filter): ONE [bw x (bh+2)] box per horizontal tap offset
  // (tensor map 1 of the A array) serves the three vertical taps at row offsets 0, bw, 2*bw of the stage.
  int halo;              // 0 off, 1 vertical halo (3 loads per tile), 2 two-dimensional halo (1 load per tile, bw == 8)
  int halo_bytes;        // bw * (bh + 2) * 128
  int8_t halo_dw[3];     // horizontal offset of stage s
  int8_t halo_dh0;       // vertical offset of row-shift 0 (normally -1)
  int8_t halo_tap[9];    // filter tap index of (stage s, row shift r) at [s * 3 + r]
  // kStats == 3 (flat mode): dz = (acc + add_src) * relu_mask is stored; sums of dz, dz*y go to stat_sum / stat_sqsum
  const __nv_bfloat16* add_src;  // skip gradient: dense [M, Cout] (add_mode 0) or compact [N, H/2, W/2, Cout] (add_mode 1)
  const uint8_t* relu_mask;      // 1 bit per element, [M, Cout / 8]
  int add_mode;
  int add_h, add_w;              // add_mode 1: spatial extent of the OUTPUT grid (rows decode to (n, h, w))
  int64_t m_rows;                // number of real rows (pixels) of the flat problem
  // kStats == 4 (inference epilogue): out = act(acc * ep_scale[c] + ep_shift[c] [+ add_src]);  act: 0 none, 1 ReLU, 2 ReLU6
  const float* ep_scale;
  const float* ep_shift;
  int ep_act;
};

// Weight-gradient GEMM:  dW[tap][co][ci] += sum_px dY[px, co] * X_tap[px, ci]
struct WgradParams {
  int mode;          // 0 = flat (2-D [M, C] maps), 1 = box (4-D NHWC maps)
  int P;             // pixels per k-iteration (multiple of 16, <= 128)
  int a_chunks;      // 64-channel chunks of dY per unit (1 if Cout == 64, else 2)
  int G;             // 64-channel chunks of X per unit (1..6), ordered (ci-block, s)
  int acc_chunks;    // chunks per accumulator: MMA N = 64 * acc_chunks
  int S;             // filter width; a unit covers one filter row r (taps r*S .. r*S+S-1)
  int cb_per_group;  // ci 64-blocks per unit
  int cgroups;       // (Cin/64) / cb_per_group
  int groups;        // R * cgroups
  int co_blocks;     // ceil(Cout / 128)
  int px_chunks;     // split-K factor over pixels
  int iters_total;   // number of pixel boxes
  int iters_per_chunk;
  int stages;
  int cout, cin;
  int bw, bh, bn, tiles_w, tiles_h;
  int num_units;
  int8_t tap_map[kMaxTaps];
  int8_t tap_dw[kMaxTaps];
  int8_t tap_dh[kMaxTaps];
  float* dw;  // [taps][Cout][Cin] fp32, accumulated with vector atomics
};

// ResNet stem (7x7/2 conv over a uint8 image), forward and weight gradient (csrc/stem.cu)
struct StemParams {
  const uint8_t* x;  // [N, H, W, 3] uint8
  int N, H, W, Ho, Wo;
  int64_t M;         // N * Ho * Wo output pixels
  int num_tiles;     // ceil(M / 128)
  float mul, add;    // input normalisation: v = u8 * mul + add
  float* stat_sum;   // forward: [64] BatchNorm statistics (nullable)
  float* stat_sqsum;
  float* dw;         // wgrad: fp32 [49][64][3], accumulated with atomics
};

}  // namespace b200
