// Implicit-GEMM convolution (forward and data-gradient) for sm_100a.
//
//   D[m, n] = sum_{tap, c} A_tap[m, c] * B[tap][n][c]            (bf16 x bf16 -> fp32 in TMEM -> bf16)
//
// * A is an NHWC bf16 activation.  An M-tile is either 128 consecutive pixels of the flattened
//   [N*H*W, C] view ("flat", 1x1 stride-1 convs) or a TMA box (bw x bh x bn pixels, <=128) of the 4-D tensor
//   ("box", 3x3 / strided convs).  A filter tap is a coordinate offset of the box; zero padding is the TMA
//   out-of-bounds fill, so there is no im2col buffer.  Strided convs pass up to 4 "parity" views of the input (each a
//   strided NHWC view) and a tap table that says which view + offset each tap reads.
// * B is the filter as a [taps*Cout, Cin] K-major matrix.
// * Warp-specialised, persistent: warp0 = TMA producer, warp1 = tcgen05.mma issuer (both ONE thread chosen with
//   elect.sync on a shuffle-broadcast warp index, integer smem addresses, descriptors built once), warp2 = TMEM allocator,
//   warps4-7 = epilogue (tcgen05.ld -> bf16 -> swizzled smem -> TMA store), double-buffered TMEM accumulator so the
//   epilogue of tile i overlaps the main loop of tile i+1.
// * kStats = 1: warps 8-11 reduce per-channel sum / sum-of-squares of the staged bf16 output tile (register accumulators
//   across tiles, one global atomic per channel per CTA) - no separate BatchNorm statistics pass (SURVEY.md K10).
//   kStats = 2: the same warps do the BatchNorm-BACKWARD reduction inside a dgrad GEMM (sum dz, sum dz*y with
//   dz = g * [y*scale + shift > 0]; the pre-BN tile y arrives by an extra TMA load).
// * kResB: the CTA's whole filter slice (<= 9 tiles of 8 KB, single N-block of 64 channels) stays resident in shared
//   memory.  kHalo (on top of kResB; 3x3 stride 1, full-width single-image boxes): one [bw x (bh+2)] box per
//   horizontal tap offset; its three vertical taps read the same stage 0 / bw / 2*bw rows in (row-shifted SWIZZLE_128B
//   descriptors, exact with base_offset 0 - umma_probe.cu).  Why: the stage ring is latency-bound per slot
//   (tma_probe.cu), so fewer and larger loads win; see profiles/README.md 2.1b.
#pragma once
#include "conv_params.h"
#include "ptx.cuh"

namespace b200 {

// kStats: 0 = plain epilogue, 1 = forward BatchNorm statistics (sum y, sum y^2), 2 = BatchNorm-backward reduction
// fused into a dgrad GEMM: the output tile is g = dL/d(activation); with the activation's pre-BN tensor y (extra TMA
// load per chunk) the statistics warps accumulate sum(dz), sum(dz*y) for dz = g * [y*scale + shift > 0].
// kStats = 3 (flat 1x1 dgrad of a residual block's first conv): the whole gradient merge of the PREVIOUS block's output
// happens in the epilogue - dz = (acc + skip_gradient) * relu_bitmask is what gets stored, and the statistics warps
// accumulate sum(dz), sum(dz*y3) for that block's final BatchNorm.  The separate reduce pass (4 tensor reads + 1 write of
// the widest activation of the block) and the store / re-read of the main-path gradient disappear.
// kStats = 4 (inference): per-channel affine (folded BatchNorm: y*scale + shift) + optional residual add (flat mode) +
// ReLU / ReLU6 applied in the epilogue - the convolution writes the block's activation directly, no BatchNorm pass at all.
// The (up to four) parity views of the A operand as ONE kernel parameter: the per-tap choice is an index.
struct TmapArray4 {
  CUtensorMap m[4];
};

// kResB: the whole filter slice this CTA needs (taps * kblocks tiles of [BLOCK_N x 64]) stays resident in shared memory
// (loaded once per CTA) and the pipeline stages carry only the A tile.  The 3x3 64->64 @56^2 layer moves ~90 % of the
// measured L2 -> SM cap (~42.6 B/clk/SM) with a third of those bytes being the same 72 KB of weights re-read per tile.
constexpr int kResBBytes = 9 * 64 * kBlockK * 2;  // 72 KB = nine [64 x 64] bf16 filter tiles (taps * kblocks <= 9)

constexpr int kHaloRows = 224;  // largest halo box: bw * (bh + 2) pixels (56 x 4); 28 KB per stage

template <int BLOCK_N, int kStats = 0, bool kResB = false, bool kHalo = false>
struct ConvSmem {
  // Two pre-BN tile buffers, loaded at the start of their own chunk.  (Four buffers prefetched two chunks ahead were tried:
  // the statistics warps already run a chunk behind the epilogue, so the load latency was hidden, and the extra 32 KB cost
  // a pipeline stage - the block-gradient kernel went from 302 to 353 us.  profiles/README.md, r2 negative results.)
  static constexpr int kYBufs = 2;
  static constexpr int kYBytes = (kStats == 2 || kStats == 3) ? kYBufs * kBlockM * 128 : 0;  // 128x64 bf16 tiles of y
  static constexpr int kABytes = kBlockM * kBlockK * 2;
  static constexpr int kASlot = kHalo ? kHaloRows * 128 : kABytes;     // bytes of A per pipeline stage
  static constexpr int kBBytes = BLOCK_N * kBlockK * 2;
  static constexpr int kStageBytes = kResB ? kASlot : kASlot + kBBytes;
  static constexpr int kResBytes = kResB ? kResBBytes : 0;
  static constexpr int kStagingBytes = 2 * kBlockM * 128;  // two 128x64 bf16 store buffers
  static constexpr int kBarBytes = 256;
  static constexpr int kStatBytes = 2 * BLOCK_N * 4;
  static constexpr int kFixed = kResBytes + kStagingBytes + kYBytes + kBarBytes + kStatBytes;
  static constexpr int kFit = (232448 - kFixed) / kStageBytes;   // stages that fit beside the fixed buffers
  static constexpr int kCap = kResB ? 8 : ((BLOCK_N == 256) ? 4 : (BLOCK_N == 128 ? 5 : 6));
  static constexpr int kStages = kFit > kCap ? kCap : kFit;
  static constexpr int kTotal = kStages * kStageBytes + kFixed;
  static_assert(!kResB || BLOCK_N == 64, "resident filter: BLOCK_N == 64 only");
  static_assert(!kHalo || kResB, "halo mode builds on the resident filter");
  static_assert(kStages >= 2 && 2 * kStages + 9 <= kBarBytes / 8, "pipeline depth / barrier area");
  static_assert(kTotal <= 232448, "exceeds 227 KB of shared memory");
};

template <int BLOCK_N, int kStats, bool kResB = false, bool kHalo = false>
__global__ void __launch_bounds__((kStats >= 1 && kStats <= 3) ? 384 : 256, 1)
conv_igemm_kernel(const __grid_constant__ TmapArray4 tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmY,
                  const __grid_constant__ ConvParams p) {
  using L = ConvSmem<BLOCK_N, kStats, kResB, kHalo>;
  constexpr int kStages = L::kStages;
  constexpr bool kStatWarps = kStats >= 1 && kStats <= 3;  // warps 8-11 exist and consume the staged tiles
  constexpr bool kHasY = kStats == 2 || kStats == 3;       // a pre-BN tile accompanies every output chunk
  constexpr bool kAffine = kStats == 4;                    // epilogue: acc*scale + shift (+ residual) -> activation
  constexpr bool kRowAdd = kStats == 3 || kStats == 4;     // per-row global loads of an additive tensor in the epilogue
  constexpr uint32_t kTmemCols = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64 ? 64 : (2 * BLOCK_N <= 128 ? 128 : (2 * BLOCK_N <= 256 ? 256 : 512)));

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem) & 1023u) != 0) __trap();  // SWIZZLE_128B tiles need 1024 B alignment
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStages * L::kASlot;  // per-stage B tiles, or (kResB) the resident filter slice
  uint8_t* sStage = smem + kStages * L::kStageBytes + L::kResBytes;
  uint8_t* sY = sStage + L::kStagingBytes;  // kStats == 2 only
  uint64_t* bars = reinterpret_cast<uint64_t*>(sY + L::kYBytes);
  uint64_t* full_bar = bars;                     // [kStages]
  uint64_t* empty_bar = bars + kStages;          // [kStages]
  uint64_t* tfull_bar = bars + 2 * kStages;      // [2]
  uint64_t* tempty_bar = bars + 2 * kStages + 2; // [2]
  uint64_t* y_bar = bars + 2 * kStages + 4;      // [4] (kStats >= 2)
  uint64_t* bres_bar = bars + 2 * kStages + 8;   // resident filter loaded (kResB)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 9);
  float* sStat = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + L::kBarBytes);  // [2][BLOCK_N]

  // Provably warp-uniform (the compiler cannot see that threadIdx.x >> 5 is): together with elect.sync for the
  // single-thread roles this keeps tcgen05 / TMA / mbarrier instructions free of per-instruction serialisation loops.
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA.m[0]);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmD);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 4);
    }
    for (int i = 0; i < 4; ++i) mbar_init(&y_bar[i], 1);
    mbar_init(bres_bar, 1);
    fence_barrier_init();
  }
  if (kStatWarps) {
    for (int i = threadIdx.x; i < 2 * BLOCK_N; i += blockDim.x) sStat[i] = 0.f;
  }
  if (kHasY) {
    // rows past the pixel box are never written by TMA: keep them finite (0 * NaN would poison the sums)
    for (int i = threadIdx.x; i < L::kYBytes / 16; i += blockDim.x) reinterpret_cast<uint4*>(sY)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int k_iters = p.taps * p.kblocks;
  const uint32_t a_bytes = (p.mode == 0 ? kBlockM : p.valid_rows) * 128;
  const uint32_t stage_tx = kHalo ? static_cast<uint32_t>(p.halo_bytes) : (kResB ? a_bytes : a_bytes + L::kBBytes);

  // The two single-thread roles below were the bottleneck of the small-K / small-N layers (ncu, 3x3 64->64 @56^2: tensor
  // pipe 22 %, L2 32 %, both role threads busy ~90 % of the time executing ~70-100 dependent instructions per 24 KB
  // stage).  Hence: one elect.sync around each loop, integer smem addresses and UMMA descriptors built once, kernel
  // parameters hoisted into registers, per-tap work hoisted out of the k-block loop.
  if (warp == 0) {
    if (elect_one()) {
      // ---------------------------------------------------------------- TMA producer (one elected thread)
      const int taps = p.taps, kblocks = p.kblocks, n_blocks = p.n_blocks, num_tiles = p.num_tiles, cout = p.cout;
      const bool flat = p.mode == 0;
      const int tiles_w = p.tiles_w, tiles_h = p.tiles_h, bw = p.bw, bh = p.bh, bn = p.bn;
      const uint32_t sA0 = smem_u32(sA), sB0 = smem_u32(sB);
      const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
      if (kResB && static_cast<int>(blockIdx.x) < num_tiles) {
        // n_blocks == 1 (host-checked): every tile of this CTA uses the same taps * kblocks filter tiles, tile
        // (t, kb) at index t * kblocks + kb.
        mbar_arrive_expect_tx_u32(smem_u32(bres_bar), static_cast<uint32_t>(taps * kblocks) * L::kBBytes);
        for (int t = 0; t < taps; ++t)
          for (int kb = 0; kb < kblocks; ++kb)
            tma_load_2d_u32(sB0 + (t * kblocks + kb) * L::kBBytes, &tmB, smem_u32(bres_bar), kb * kBlockK, t * cout);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_tile = tile / n_blocks;
        const int nb = tile - m_tile * n_blocks;
        int w0 = 0, h0 = 0, n0 = 0;
        if (!flat) {
          const int tw = m_tile % tiles_w;
          const int rest = m_tile / tiles_w;
          const int th = rest % tiles_h;
          w0 = tw * bw;
          h0 = th * bh;
          n0 = (rest / tiles_h) * bn;
        }
        if (kHalo && p.halo == 2) {
          // 2-D halo: ONE [(bw+2) x (bh+2)] box per tile (and k-block) serves all nine taps
          for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait_u32(empty0 + stage * 8, phase ^ 1);
            const uint32_t fb = full0 + stage * 8;
            mbar_arrive_expect_tx_u32(fb, stage_tx);
            tma_load_4d_u32(sA0 + stage * L::kASlot, &tmA.m[1], fb, kb * kBlockK, w0 - 1, h0 - 1, n0);
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
          continue;
        }
        if (kHalo) {
          // one [bw x (bh+2)] box per horizontal tap offset; rows above / below / beside the image are zero-filled
          for (int hs = 0; hs < 3; ++hs) {
            const int cw = w0 + p.halo_dw[hs];
            const int ch = h0 + p.halo_dh0;
            for (int kb = 0; kb < kblocks; ++kb) {
              mbar_wait_u32(empty0 + stage * 8, phase ^ 1);
              const uint32_t fb = full0 + stage * 8;
              mbar_arrive_expect_tx_u32(fb, stage_tx);
              tma_load_4d_u32(sA0 + stage * L::kASlot, &tmA.m[1], fb, kb * kBlockK, cw, ch, n0);
              if (++stage == kStages) {
                stage = 0;
                phase ^= 1;
              }
            }
          }
          continue;
        }
        const int m0 = m_tile * kBlockM;
        const int brow = nb * BLOCK_N;
        for (int t = 0; t < taps; ++t) {
          const CUtensorMap* am = &tmA.m[p.tap_map[t]];
          const int cw = w0 + p.tap_dw[t];
          const int ch = h0 + p.tap_dh[t];
          const int b1 = t * cout + brow;
          for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait_u32(empty0 + stage * 8, phase ^ 1);
            const uint32_t fb = full0 + stage * 8;
            mbar_arrive_expect_tx_u32(fb, stage_tx);
            if (flat)
              tma_load_2d_u32(sA0 + stage * L::kASlot, am, fb, kb * kBlockK, m0);
            else
              tma_load_4d_u32(sA0 + stage * L::kASlot, am, fb, kb * kBlockK, cw, ch, n0);
            if (!kResB) tma_load_2d_u32(sB0 + stage * L::kBBytes, &tmB, fb, kb * kBlockK, b1);
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      // ---------------------------------------------------------------- MMA issuer (one elected thread)
      constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, BLOCK_N, 0, 0);
      const int num_tiles = p.num_tiles;
      const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
      const uint32_t tfull0 = smem_u32(tfull_bar), tempty0 = smem_u32(tempty_bar);
      // descriptors differ only in the 14-bit start-address field (addr >> 4): build once, add per stage / k-step
      const uint64_t da0 = umma_desc_sw128(smem_u32(sA), 16, 1024);
      const uint64_t db0 = umma_desc_sw128(smem_u32(sB), 16, 1024);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      if (kResB && static_cast<int>(blockIdx.x) < num_tiles) mbar_wait_u32(smem_u32(bres_bar), 0);
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait_u32(tempty0 + acc * 8, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        if (kHalo && p.halo == 2) {
          // 2-D halo (bw == 8): the stage holds a [(bh+2) x (bw+2)] pixel tile, row-major.  Output pixel (g, r) of the
          // 8-wide box is accumulator row 8g + r, so the M = 128 operand is 16 groups of 8 consecutive tile rows at a
          // stride of (bw+2) rows = 1280 B (the descriptor's stride-byte-offset) and tap (dw, dh) starts
          // (dh+1)*(bw+2) + (dw+1) rows in.  Any 128-byte-multiple group stride and row shift is exact (umma_probe.cu);
          // groups past bh read rows whose accumulator lanes are discarded.
          const int kblocks = p.kblocks, taps = p.taps;
          const uint32_t hw = static_cast<uint32_t>(p.bw) + 2;
          const uint64_t da2 = umma_desc_sw128(smem_u32(sA), 16, hw * 128);
          for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait_u32(full0 + stage * 8, phase);
            tc_fence_after();
            const uint64_t da_s = da2 + static_cast<uint32_t>(stage * (L::kASlot >> 4));
            for (int t = 0; t < taps; ++t) {
              const uint32_t shift16 = ((p.tap_dh[t] + 1) * hw + (p.tap_dw[t] + 1)) * 8;  // rows of 128 B in the (addr >> 4) field
              const uint64_t da = da_s + shift16;
              const uint64_t db = db0 + static_cast<uint32_t>((t * kblocks + kb) * (L::kBBytes >> 4));
              umma_bf16(d_tmem, da, db, idesc, (kb | t) != 0 ? 1u : 0u);
#pragma unroll
              for (int k = 1; k < kBlockK / 16; ++k) umma_bf16_acc(d_tmem, da + 2 * k, db + 2 * k, idesc);
            }
            umma_commit_u32(empty0 + stage * 8);
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        } else if (kHalo) {
          const int kblocks = p.kblocks;
          const uint32_t shift16 = static_cast<uint32_t>(p.bw) * 8;  // bw rows of 128 B, in the (addr >> 4) field
          for (int hs = 0; hs < 3; ++hs) {
            for (int kb = 0; kb < kblocks; ++kb) {
              mbar_wait_u32(full0 + stage * 8, phase);
              tc_fence_after();
              const uint64_t da_s = da0 + static_cast<uint32_t>(stage * (L::kASlot >> 4));
#pragma unroll
              for (int r = 0; r < 3; ++r) {
                // vertical tap r reads the same stage bw * r rows further down (row-shifted SWIZZLE_128B start address
                // with base_offset 0 is exact - csrc/umma_probe.cu); rows past the pixel box feed discarded lanes
                const uint64_t da = da_s + r * shift16;
                const uint64_t db = db0 + static_cast<uint32_t>((p.halo_tap[hs * 3 + r] * kblocks + kb) * (L::kBBytes >> 4));
                umma_bf16(d_tmem, da, db, idesc, (hs | kb | r) != 0 ? 1u : 0u);
#pragma unroll
                for (int k = 1; k < kBlockK / 16; ++k) umma_bf16_acc(d_tmem, da + 2 * k, db + 2 * k, idesc);
              }
              umma_commit_u32(empty0 + stage * 8);
              if (++stage == kStages) {
                stage = 0;
                phase ^= 1;
              }
            }
          }
        }
        for (int it = 0; it < (kHalo ? 0 : k_iters); ++it) {
          mbar_wait_u32(full0 + stage * 8, phase);
          tc_fence_after();
          const uint64_t da = da0 + static_cast<uint32_t>(stage * (L::kASlot >> 4));
          const uint64_t db = db0 + static_cast<uint32_t>((kResB ? it : stage) * (L::kBBytes >> 4));
          // 16 bf16 = 32 B along K inside the 128 B swizzle row: +2 in the (addr >> 4) field per k-step
          umma_bf16(d_tmem, da, db, idesc, it != 0 ? 1u : 0u);
#pragma unroll
          for (int k = 1; k < kBlockK / 16; ++k) umma_bf16_acc(d_tmem, da + 2 * k, db + 2 * k, idesc);
          umma_commit_u32(empty0 + stage * 8);  // frees the smem slot when these MMAs retire
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_u32(tfull0 + acc * 8);  // accumulator complete -> epilogue
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ------------------------------------------------------------------ epilogue (128 threads)
    const int ew = warp - 4;           // TMEM lane quarter == warp_id % 4
    const int row = ew * 32 + lane;    // tile row owned by this thread
    const int etid = threadIdx.x - 128;
    int acc = 0;
    uint32_t acc_phase = 0;
    int chunk_ctr = 0;
    // kStats 2 / 3: the pre-BN tile of CTA-local output chunk g (tile g / kChunks of this CTA, 64-column chunk g % kChunks)
    // goes to Y buffer g & 1; it is issued at the start of chunk g, after the barrier that says the statistics warps are
    // done with chunk g - 2 (which used the same buffer).
    auto issue_y = [&](int g) {
      constexpr int kChunksE = BLOCK_N / 64;
      const int lt = g / kChunksE, c = g - lt * kChunksE;
      const int tl = static_cast<int>(blockIdx.x) + lt * static_cast<int>(gridDim.x);
      if (tl >= p.num_tiles) return;
      const int mt = tl / p.n_blocks, nbb = tl - mt * p.n_blocks;
      const int b = g & 1;
      mbar_arrive_expect_tx(&y_bar[b], static_cast<uint32_t>(p.valid_rows) * 128u);
      if (p.mode == 0) {
        tma_load_2d(sY + b * (kBlockM * 128), &tmY, &y_bar[b], nbb * BLOCK_N + c * 64, mt * kBlockM);
      } else {
        const int tw = mt % p.tiles_w;
        const int rest = mt / p.tiles_w;
        const int th = rest % p.tiles_h;
        tma_load_4d(sY + b * (kBlockM * 128), &tmY, &y_bar[b], nbb * BLOCK_N + c * 64, tw * p.bw, th * p.bh,
                    (rest / p.tiles_h) * p.bn);
      }
    };
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int m_tile = tile / p.n_blocks;
      const int nb = tile - m_tile * p.n_blocks;
      int w0 = 0, h0 = 0, n0 = 0;
      if (p.mode == 1) {
        const int tw = m_tile % p.tiles_w;
        const int rest = m_tile / p.tiles_w;
        const int th = rest % p.tiles_h;
        w0 = tw * p.bw;
        h0 = th * p.bh;
        n0 = (rest / p.tiles_h) * p.bn;
      }
      // kStats == 3: this thread's row of the skip gradient / ReLU bitmask (flat mode: tile row == pixel index).
      // The 64 B + 4 B per 32-column half are prefetched one half ahead (slot = h), the first one before the
      // accumulator wait, so the global-load latency hides behind the TMEM wait and the previous half's packing.
      const __nv_bfloat16* arow = nullptr;
      const uint8_t* mrow = nullptr;
      // Two STATICALLY indexed slots (slot = h, the 32-column half inside a 64-column chunk): half i is consumed from slot
      // i & 1 while half i + 1 loads into the other one.  (A rotating queue - "gq[0] = gq[1]" - was tried for a deeper
      // prefetch: the register move needs the value, so every rotation waited for the load that had just been issued and
      // the kernel went from 302 to 353 us.  Prefetch slots must never be moved.)
      uint4 gq[2][4];
      uint32_t mq[2] = {0u, 0u};
      if (kAffine) {
        // per-channel scale / shift of this tile's N-block -> shared memory (read back as float4 broadcasts); every thread
        // passed the previous tile's last staging barrier after its last read, and the first chunk barrier below publishes
        for (int i = etid; i < BLOCK_N; i += 128) {
          sStat[i] = p.ep_scale[nb * BLOCK_N + i];
          sStat[BLOCK_N + i] = p.ep_shift[nb * BLOCK_N + i];
        }
      }
      if (kRowAdd) {
#pragma unroll
        for (int j = 0; j < 4; ++j) gq[0][j] = gq[1][j] = make_uint4(0u, 0u, 0u, 0u);
      }
      if (kRowAdd && (kStats == 3 || (p.add_src != nullptr && p.mode == 0))) {
        const int64_t grow = static_cast<int64_t>(m_tile) * kBlockM + row;
        if (grow < p.m_rows) {
          if (kStats == 3) mrow = p.relu_mask + grow * (p.cout >> 3) + ((nb * BLOCK_N) >> 3);
          if (p.add_mode == 0) {
            arow = p.add_src + grow * p.cout + nb * BLOCK_N;
          } else {
            // compact skip gradient of a stride-2 1x1 projection: only even (h, w) positions carry a value
            const int wq = static_cast<int>(grow % p.add_w);
            const int64_t t = grow / p.add_w;
            const int hq = static_cast<int>(t % p.add_h);
            const int64_t nq = t / p.add_h;
            if (((wq | hq) & 1) == 0)
              arow = p.add_src + ((nq * (p.add_h >> 1) + (hq >> 1)) * (p.add_w >> 1) + (wq >> 1)) * p.cout + nb * BLOCK_N;
          }
        }
        if (arow != nullptr) {
#pragma unroll
          for (int j = 0; j < 4; ++j) gq[0][j] = __ldg(reinterpret_cast<const uint4*>(arow) + j);
        }
        if (mrow != nullptr) mq[0] = __ldg(reinterpret_cast<const uint32_t*>(mrow));
      }
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BLOCK_N;

#pragma unroll 1
      for (int c64 = 0; c64 < BLOCK_N / 64; ++c64, ++chunk_ctr) {
        uint8_t* sbuf = sStage + (chunk_ctr & 1) * (kBlockM * 128);
        if (etid == 0) tma_store_wait_read<1>();  // the store that used this buffer two chunks ago is done
        if (kStatWarps)
          named_bar_sync(4 + (chunk_ctr & 1), 256);  // ... and the statistics warps are done reading it
        else
          named_bar_sync(1, 128);
        if (kHasY && etid == 0) issue_y(chunk_ctr);  // pre-BN tile of this chunk (see issue_y)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t r[32];
          if (kRowAdd) {
            // prefetch the next half (h ^ 1 of this chunk, or h = 0 of the next chunk) into the other slot
            const int nxt = c64 * 64 + h * 32 + 32;
            if (nxt < BLOCK_N) {
              if (arow != nullptr) {
#pragma unroll
                for (int j = 0; j < 4; ++j) gq[h ^ 1][j] = __ldg(reinterpret_cast<const uint4*>(arow + nxt) + j);
              }
              if (mrow != nullptr) mq[h ^ 1] = __ldg(reinterpret_cast<const uint32_t*>(mrow + (nxt >> 3)));
            }
          }
          tmem_ld_32x32b_x32(taddr + c64 * 64 + h * 32, r);
          tmem_ld_wait();
          if (kAffine) {
            // out = act(acc * scale[c] + shift[c] [+ residual])
            const float4* sc4 = reinterpret_cast<const float4*>(sStat + c64 * 64 + h * 32);
            const float4* sh4 = reinterpret_cast<const float4*>(sStat + BLOCK_N + c64 * 64 + h * 32);
            const int act = p.ep_act;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t gw[4] = {gq[h][j].x, gq[h][j].y, gq[h][j].z, gq[h][j].w};
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const float4 sc = sc4[2 * j + e], sh = sh4[2 * j + e];
                const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const int col = 8 * j + 4 * e + q;
                  const uint32_t gword = gw[(4 * e + q) >> 1];
                  const float res = __uint_as_float(((4 * e + q) & 1) ? (gword & 0xFFFF0000u) : (gword << 16));
                  float f = fmaf(__uint_as_float(r[col]), scv[q], shv[q]) + res;
                  if (act >= 1) f = fmaxf(f, 0.f);
                  if (act == 2) f = fminf(f, 6.f);
                  r[col] = __float_as_uint(f);
                }
              }
            }
          }
          if (kStats == 3) {
            // dz = (main-path gradient + skip gradient) * [block output > 0]
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t gw[4] = {gq[h][j].x, gq[h][j].y, gq[h][j].z, gq[h][j].w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float lo = __uint_as_float(r[8 * j + 2 * e]) + __uint_as_float(gw[e] << 16);
                const float hi = __uint_as_float(r[8 * j + 2 * e + 1]) + __uint_as_float(gw[e] & 0xFFFF0000u);
                r[8 * j + 2 * e] = ((mq[h] >> (8 * j + 2 * e)) & 1u) ? __float_as_uint(lo) : 0u;
                r[8 * j + 2 * e + 1] = ((mq[h] >> (8 * j + 2 * e + 1)) & 1u) ? __float_as_uint(hi) : 0u;
              }
            }
          }
          if (c64 == BLOCK_N / 64 - 1 && h == 1) {
            // all TMEM reads of this accumulator are done: hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
          }
          // bf16 pack + swizzled smem write (16 B chunk j of row r lives at chunk j ^ (r & 7))
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 v;
            v.x = pack_bf16x2(__uint_as_float(r[8 * j + 0]), __uint_as_float(r[8 * j + 1]));
            v.y = pack_bf16x2(__uint_as_float(r[8 * j + 2]), __uint_as_float(r[8 * j + 3]));
            v.z = pack_bf16x2(__uint_as_float(r[8 * j + 4]), __uint_as_float(r[8 * j + 5]));
            v.w = pack_bf16x2(__uint_as_float(r[8 * j + 6]), __uint_as_float(r[8 * j + 7]));
            if (kStatWarps && row >= p.valid_rows) v = make_uint4(0u, 0u, 0u, 0u);  // rows past the pixel box: no statistics
            const int chunk = (h * 4 + j) ^ (row & 7);
            *reinterpret_cast<uint4*>(sbuf + row * 128 + chunk * 16) = v;
          }
        }
        fence_proxy_async_smem();
        named_bar_sync(2, 128);
        if (kStatWarps) named_bar_arrive(6 + (chunk_ctr & 1), 256);  // staged tile is complete: wake the statistics warps
        if (etid == 0) {
          const int ccol = nb * BLOCK_N + c64 * 64;
          if (p.mode == 0)
            tma_store_2d(&tmD, sbuf, ccol, m_tile * kBlockM);
          else
            tma_store_4d(&tmD, sbuf, ccol, w0, h0, n0);
          tma_store_commit();
        }
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (etid == 0) tma_store_wait_all<0>();
  } else if (kStatWarps && warp >= 8) {
    // ------------------------------------------------------------------ BatchNorm statistics warps (128 threads)
    // Column sums / sums of squares of the bf16 tile the epilogue just staged (exactly the values BatchNorm will
    // read), concurrent with the epilogue's next chunk.  Thread = (column pair cp, 32-row group rg): one
    // conflict-free LDS.32 per row with precomputed swizzled offsets, accumulators live in registers across tiles
    // and are flushed with global atomics only when the CTA moves to another n-block.
    // Named barriers 4/5 = "staging buffer b is free", 6/7 = "staging buffer b is full".
    const int stid = threadIdx.x - 256;
    const int cp = stid & 31;
    const int rg = stid >> 5;
    uint32_t xoff[8];  // byte offset of this thread's column pair in a row with (row & 7) == j
#pragma unroll
    for (int j = 0; j < 8; ++j) xoff[j] = ((((cp >> 2) ^ j) << 4) + ((cp & 3) << 2)) + rg * 32 * 128;
    constexpr int kChunks = BLOCK_N / 64;
    float acc[kChunks][4];
#pragma unroll
    for (int c = 0; c < kChunks; ++c) acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0.f;
    named_bar_arrive(4, 256);
    named_bar_arrive(5, 256);
    int chunk_ctr = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int nb = tile % p.n_blocks;
#pragma unroll
      for (int c64 = 0; c64 < kChunks; ++c64, ++chunk_ctr) {
        const int b = chunk_ctr & 1;
        const uint8_t* sbuf = sStage + b * (kBlockM * 128);
        named_bar_sync(6 + b, 256);
        float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
        if (kStats == 1) {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(sbuf + xoff[i & 7] + i * 128);
            const float lo = __uint_as_float(w << 16);
            const float hi = __uint_as_float(w & 0xFFFF0000u);
            s0 += lo;
            s1 += hi;
            q0 = fmaf(lo, lo, q0);
            q1 = fmaf(hi, hi, q1);
          }
        } else if (kStats == 3) {
          // the staged tile already is dz (merged + masked by the epilogue): accumulate sum(dz) and sum(dz * y)
          const uint8_t* ybuf = sY + (chunk_ctr & 1) * (kBlockM * 128);
          mbar_wait(&y_bar[chunk_ctr & 1], (chunk_ctr >> 1) & 1);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(sbuf + xoff[i & 7] + i * 128);
            const uint32_t v = *reinterpret_cast<const uint32_t*>(ybuf + xoff[i & 7] + i * 128);
            const float y0 = __uint_as_float(v << 16), y1 = __uint_as_float(v & 0xFFFF0000u);
            const float g0 = __uint_as_float(w << 16), g1 = __uint_as_float(w & 0xFFFF0000u);
            s0 += g0;
            s1 += g1;
            q0 = fmaf(g0, y0, q0);
            q1 = fmaf(g1, y1, q1);
          }
        } else {
          // dz = g * [y*scale + shift > 0];  accumulate sum(dz) and sum(dz * y)
          const int col = nb * BLOCK_N + c64 * 64 + cp * 2;
          const float sc0 = p.bn_scale[col], sc1 = p.bn_scale[col + 1];
          const float sh0 = p.bn_shift[col], sh1 = p.bn_shift[col + 1];
          const uint8_t* ybuf = sY + (chunk_ctr & 1) * (kBlockM * 128);
          mbar_wait(&y_bar[chunk_ctr & 1], (chunk_ctr >> 1) & 1);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(sbuf + xoff[i & 7] + i * 128);
            const uint32_t v = *reinterpret_cast<const uint32_t*>(ybuf + xoff[i & 7] + i * 128);
            const float y0 = __uint_as_float(v << 16), y1 = __uint_as_float(v & 0xFFFF0000u);
            const float g0 = fmaf(y0, sc0, sh0) > 0.f ? __uint_as_float(w << 16) : 0.f;
            const float g1 = fmaf(y1, sc1, sh1) > 0.f ? __uint_as_float(w & 0xFFFF0000u) : 0.f;
            s0 += g0;
            s1 += g1;
            q0 = fmaf(g0, y0, q0);
            q1 = fmaf(g1, y1, q1);
          }
        }
        named_bar_arrive(4 + b, 256);  // done reading the staging buffer
        acc[c64][0] += s0;
        acc[c64][1] += s1;
        acc[c64][2] += q0;
        acc[c64][3] += q1;
      }
      const int next = tile + gridDim.x;
      const bool flush = (next >= p.num_tiles) || ((next % p.n_blocks) != nb);
      if (flush) {
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
          const int col = nb * BLOCK_N + c * 64 + cp * 2;
          atomicAdd(p.stat_sum + col, acc[c][0]);
          atomicAdd(p.stat_sum + col + 1, acc[c][1]);
          atomicAdd(p.stat_sqsum + col, acc[c][2]);
          atomicAdd(p.stat_sqsum + col + 1, acc[c][3]);
          acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0.f;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace b200
