// pybind layer for the tcgen05 convolution kernels: validates tensors, derives the tiling, encodes the TMA
// descriptors once, and exposes launchable plan objects (static buffers => plans are reused under CUDA graphs).
#include <ATen/cuda/CUDAContext.h>
#include <torch/extension.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "conv_api.h"

namespace b200 {

static void check_nhwc_view(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == at::kBFloat16, name, " must be bf16");
  TORCH_CHECK(t.dim() == 4, name, " must be 4-D (N,H,W,C)");
  TORCH_CHECK(t.stride(3) == 1, name, " must be channel-contiguous (NHWC)");
  TORCH_CHECK(reinterpret_cast<uintptr_t>(t.data_ptr()) % 16 == 0, name, " must be 16-byte aligned");
  TORCH_CHECK((t.stride(2) * 2) % 16 == 0 && (t.stride(1) * 2) % 16 == 0 && (t.stride(0) * 2) % 16 == 0, name,
              " strides must be multiples of 16 bytes");
}

// 4-D map over a (possibly strided) NHWC view: dims (C, W, H, N).
static CUtensorMap map_nhwc(const at::Tensor& t, int box_c, int bw, int bh, int bn) {
  uint64_t dims[4] = {(uint64_t)t.size(3), (uint64_t)t.size(2), (uint64_t)t.size(1), (uint64_t)t.size(0)};
  uint64_t strides[3] = {(uint64_t)t.stride(2) * 2, (uint64_t)t.stride(1) * 2, (uint64_t)t.stride(0) * 2};
  uint32_t box[4] = {(uint32_t)box_c, (uint32_t)bw, (uint32_t)bh, (uint32_t)bn};
  return encode_bf16(t.data_ptr(), 4, dims, strides, box);
}
// 2-D map over a row-major [rows, cols] matrix with given row pitch (elements).
static CUtensorMap map_2d(void* ptr, int64_t rows, int64_t cols, int64_t pitch, int box_cols, int box_rows) {
  uint64_t dims[2] = {(uint64_t)cols, (uint64_t)rows};
  uint64_t strides[1] = {(uint64_t)pitch * 2};
  uint32_t box[2] = {(uint32_t)box_cols, (uint32_t)box_rows};
  return encode_bf16(ptr, 2, dims, strides, box);
}

static int sm_count() { return at::cuda::getCurrentDeviceProperties()->multiProcessorCount; }

struct ConvPlan {
  ConvPlanRaw raw;
  std::vector<at::Tensor> keep;
  int64_t launches = 0;

  // views:  1..4 NHWC (possibly strided) input views on one pixel grid (N, Hv, Wv, Cin)
  // weight: bf16 [taps*Cout, Cin];  out: NHWC view (N, Ho, Wo, Cout)
  // tap_map/dw/dh: per tap view index + pixel offset;  bw/bh/bn: pixel box (0 => flat 1x1 mode)
  ConvPlan(std::vector<at::Tensor> views, at::Tensor weight, at::Tensor out, std::vector<int64_t> tap_map,
           std::vector<int64_t> tap_dw, std::vector<int64_t> tap_dh, int64_t bw, int64_t bh, int64_t bn,
           c10::optional<at::Tensor> stat_sum, c10::optional<at::Tensor> stat_sqsum, int64_t max_ctas,
           c10::optional<at::Tensor> bwd_y, c10::optional<at::Tensor> bn_scale, c10::optional<at::Tensor> bn_shift,
           c10::optional<at::Tensor> add_src, c10::optional<at::Tensor> relu_mask, c10::optional<at::Tensor> ep_scale,
           c10::optional<at::Tensor> ep_shift, int64_t ep_act) {
    TORCH_CHECK(!views.empty() && views.size() <= 4, "1..4 input views");
    for (auto& v : views) check_nhwc_view(v, "input view");
    check_nhwc_view(out, "out");
    const int taps = (int)tap_map.size();
    TORCH_CHECK(taps >= 1 && taps <= kMaxTaps, "1..16 taps");
    TORCH_CHECK(tap_dw.size() == tap_map.size() && tap_dh.size() == tap_map.size());
    const int64_t cin = views[0].size(3);
    const int64_t cout = out.size(3);
    TORCH_CHECK(cin % 64 == 0, "Cin must be a multiple of 64, got ", cin);
    TORCH_CHECK(cout % 64 == 0, "Cout must be a multiple of 64, got ", cout);
    TORCH_CHECK(weight.is_cuda() && weight.scalar_type() == at::kBFloat16 && weight.is_contiguous() &&
                    weight.dim() == 2 && weight.size(0) == taps * cout && weight.size(1) == cin,
                "weight must be bf16 [taps*Cout, Cin]");
    ConvParams& p = raw.p;
    std::memset(&p, 0, sizeof(p));
    raw.block_n = cout % 256 == 0 ? 256 : (cout % 128 == 0 ? 128 : 64);
    p.taps = taps;
    p.kblocks = (int)(cin / 64);
    p.cout = (int)cout;
    for (int t = 0; t < taps; ++t) {
      TORCH_CHECK(tap_map[t] >= 0 && tap_map[t] < (int64_t)views.size());
      p.tap_map[t] = (int8_t)tap_map[t];
      p.tap_dw[t] = (int8_t)tap_dw[t];
      p.tap_dh[t] = (int8_t)tap_dh[t];
    }
    const int64_t N = out.size(0), Ho = out.size(1), Wo = out.size(2);
    if (bw == 0) {
      TORCH_CHECK(views.size() == 1 && taps == 1 && tap_dw[0] == 0 && tap_dh[0] == 0, "flat mode is 1x1 only");
      TORCH_CHECK(views[0].is_contiguous() && out.is_contiguous(), "flat mode needs dense NHWC tensors");
      TORCH_CHECK(views[0].size(0) == N && views[0].size(1) == Ho && views[0].size(2) == Wo);
      const int64_t M = N * Ho * Wo;
      p.mode = 0;
      p.valid_rows = kBlockM;
      p.m_tiles = (int)((M + kBlockM - 1) / kBlockM);
      raw.tmA[0] = map_2d(views[0].data_ptr(), M, cin, cin, 64, kBlockM);
      for (int i = 1; i < 4; ++i) raw.tmA[i] = raw.tmA[0];
      raw.tmD = map_2d(out.data_ptr(), M, cout, cout, 64, kBlockM);
    } else {
      TORCH_CHECK(bw * bh * bn <= kBlockM && bw * bh * bn >= 8, "box must hold 8..128 pixels");
      // W and H must tile exactly (a partial spatial box would pick up halo pixels); the image dimension may
      // overhang: out-of-range images are zero-filled on load and clipped on store.
      TORCH_CHECK(Wo % bw == 0 && Ho % bh == 0, "box must tile the output plane exactly: out ", N, "x", Ho, "x", Wo,
                  " box ", bn, "x", bh, "x", bw);
      p.mode = 1;
      p.bw = (int)bw;
      p.bh = (int)bh;
      p.bn = (int)bn;
      p.valid_rows = (int)(bw * bh * bn);
      p.tiles_w = (int)(Wo / bw);
      p.tiles_h = (int)(Ho / bh);
      p.m_tiles = (int)(p.tiles_w * p.tiles_h * ((N + bn - 1) / bn));
      for (size_t i = 0; i < 4; ++i) {
        const at::Tensor& v = views[i < views.size() ? i : 0];
        TORCH_CHECK(v.size(0) == N && v.size(3) == cin);
        raw.tmA[i] = map_nhwc(v, 64, (int)bw, (int)bh, (int)bn);
      }
      raw.tmD = map_nhwc(out, 64, (int)bw, (int)bh, (int)bn);
    }
    // Tile width: the widest N tile re-reads the A operand least, but a persistent grid of one CTA per SM pays for whole
    // waves - e.g. 3x3 512->512 @7^2 at batch 256 is 98 M-tiles x 2 N-blocks = 196 tiles of 128x256 on 148 SMs = 2 waves at
    // 66 % fill (ncu: tensor pipe 80 % busy, 59 us vs cuDNN 47), while 392 tiles of 128x128 fill 3 waves at 88 %.  The cost
    // model is waves x tile width (the MMA time of a tile is proportional to its width); a narrower tile is taken only when
    // it wins by >= 10 %.  B200DDL_BLOCK_N=256|128|64 forces a width (A/B measurements).
    {
      const int cap_ = max_ctas > 0 ? (int)max_ctas : sm_count();
      auto cost = [&](int bn) {
        const int64_t tiles = (int64_t)p.m_tiles * (cout / bn);
        return ((tiles + cap_ - 1) / cap_) * bn;
      };
      int best = raw.block_n;
      for (int bn = raw.block_n / 2; bn >= 64; bn /= 2)
        if (cout % bn == 0 && cost(bn) * 10 <= cost(best) * 9) best = bn;
      if (const char* f = std::getenv("B200DDL_BLOCK_N")) {
        const int v = std::atoi(f);
        if ((v == 256 || v == 128 || v == 64) && cout % v == 0) best = v;
      }
      raw.block_n = best;
    }
    p.n_blocks = (int)(cout / raw.block_n);
    raw.tmB = map_2d(weight.data_ptr(), taps * cout, cin, cin, 64, raw.block_n);
    p.num_tiles = p.m_tiles * p.n_blocks;
    raw.stats = stat_sum.has_value() ? (bwd_y.has_value() ? (relu_mask.has_value() ? 3 : 2) : 1) : (ep_scale.has_value() ? 4 : 0);
    p.m_rows = N * Ho * Wo;
    // Resident filter: one N-block of 64 channels whose taps * kblocks filter tiles (8 KB each) fit in 72 KB.
    // B200DDL_NO_RESIDENT_FILTER=1 switches it off (A/B measurements).
    {
      const char* off = std::getenv("B200DDL_NO_RESIDENT_FILTER");
      raw.res_b = (raw.block_n == 64 && p.n_blocks == 1 && taps * p.kblocks <= 9 && !(off && off[0] == '1') &&
                   raw.stats != 3) ? 1 : 0;
    }
    // Halo mode: a 3x3 stride-1 conv (9 taps on ONE view forming the full {-1,0,1}^2 offset grid, in any order) over
    // full-width single-image boxes: one [bw x (bh+2)] load per horizontal offset serves its three vertical taps.
    // B200DDL_NO_HALO=1 switches it off (A/B measurements).
    raw.halo = 0;
    {
      const char* off = std::getenv("B200DDL_NO_HALO");
      // two-dimensional variant: 8-pixel-wide boxes, ONE [(bw+2) x (bh+2)] load per tile (B200DDL_HALO2D=1 opts in)
      const char* h2 = std::getenv("B200DDL_HALO2D");
      const bool two_d = (h2 && h2[0] == '1') && bw == 8 && bh <= 16 && (bw + 2) * (bh + 2) <= 224 && Wo % 8 == 0;
      bool ok = raw.res_b && p.mode == 1 && taps == 9 && views.size() == 1 && bn == 1 && !(off && off[0] == '1') &&
                (two_d || (bw == views[0].size(2) && bw == Wo && bw * (bh + 2) <= 224));
      int8_t table[9];
      for (int i = 0; i < 9; ++i) table[i] = -1;
      for (int t = 0; ok && t < 9; ++t) {
        const int dwv = p.tap_dw[t], dhv = p.tap_dh[t];
        if (p.tap_map[t] != 0 || dwv < -1 || dwv > 1 || dhv < -1 || dhv > 1 || table[(dwv + 1) * 3 + (dhv + 1)] != -1) ok = false;
        else table[(dwv + 1) * 3 + (dhv + 1)] = (int8_t)t;
      }
      if (ok && two_d) {
        raw.halo = 2;
        p.halo = 2;
        p.halo_bytes = (int)((bw + 2) * (bh + 2) * 128);
        raw.tmA[1] = map_nhwc(views[0], 64, (int)bw + 2, (int)bh + 2, 1);
      } else if (ok) {
        raw.halo = 1;
        p.halo = 1;
        p.halo_bytes = (int)(bw * (bh + 2) * 128);
        p.halo_dh0 = -1;
        for (int hs = 0; hs < 3; ++hs) p.halo_dw[hs] = (int8_t)(hs - 1);
        for (int i = 0; i < 9; ++i) p.halo_tap[i] = table[i];
        raw.tmA[1] = map_nhwc(views[0], 64, (int)bw, (int)bh + 2, 1);
      }
    }
    raw.tmY = raw.tmD;
    if (raw.stats == 3) {
      // block-gradient merge: out = dz = (acc + add_src) * relu_mask; sums of dz, dz*y (y = bwd_y, the block's y3)
      TORCH_CHECK(p.mode == 0, "the block-gradient epilogue needs a flat (dense 1x1) plan");
      check_nhwc_view(*bwd_y, "bwd_y");
      TORCH_CHECK(bwd_y->sizes() == out.sizes() && bwd_y->is_contiguous(), "bwd_y must match the (dense) output");
      TORCH_CHECK(relu_mask->is_cuda() && relu_mask->scalar_type() == at::kByte && relu_mask->is_contiguous() &&
                      relu_mask->numel() == N * Ho * Wo * cout / 8, "relu_mask must be uint8 [M * Cout / 8]");
      TORCH_CHECK(add_src.has_value(), "the block-gradient epilogue needs the skip gradient");
      check_nhwc_view(*add_src, "add_src");
      TORCH_CHECK(add_src->is_contiguous() && add_src->size(0) == N && add_src->size(3) == cout, "add_src: dense NHWC with Cout channels");
      if (add_src->size(1) == Ho && add_src->size(2) == Wo) {
        p.add_mode = 0;
      } else {
        TORCH_CHECK(Ho % 2 == 0 && Wo % 2 == 0 && add_src->size(1) == Ho / 2 && add_src->size(2) == Wo / 2,
                    "add_src must have the output's grid or its stride-2 sub-grid");
        p.add_mode = 1;
      }
      p.add_h = (int)Ho;
      p.add_w = (int)Wo;
      p.add_src = reinterpret_cast<const __nv_bfloat16*>(add_src->data_ptr());
      p.relu_mask = relu_mask->data_ptr<uint8_t>();
      raw.tmY = map_2d(bwd_y->data_ptr(), N * Ho * Wo, cout, cout, 64, kBlockM);
      keep.push_back(*bwd_y);
      keep.push_back(*add_src);
      keep.push_back(*relu_mask);
    }
    if (raw.stats == 4) {
      // inference epilogue: out = act(acc * scale[c] + shift[c] [+ residual]); the residual needs a flat (dense 1x1) plan
      TORCH_CHECK(ep_shift.has_value() && ep_scale->is_cuda() && ep_scale->scalar_type() == at::kFloat &&
                      ep_shift->scalar_type() == at::kFloat && ep_scale->numel() >= cout && ep_shift->numel() >= cout &&
                      ep_scale->is_contiguous() && ep_shift->is_contiguous(), "epilogue scale/shift: fp32 CUDA vectors of Cout");
      TORCH_CHECK(ep_act >= 0 && ep_act <= 2, "epilogue activation: 0 none, 1 relu, 2 relu6");
      p.ep_scale = ep_scale->data_ptr<float>();
      p.ep_shift = ep_shift->data_ptr<float>();
      p.ep_act = (int)ep_act;
      keep.push_back(*ep_scale);
      keep.push_back(*ep_shift);
      if (add_src.has_value()) {
        TORCH_CHECK(p.mode == 0, "an epilogue residual needs a flat (dense 1x1) plan");
        check_nhwc_view(*add_src, "add_src");
        TORCH_CHECK(add_src->is_contiguous() && add_src->sizes() == out.sizes(), "the residual must have the output's dense shape");
        p.add_mode = 0;
        p.add_src = reinterpret_cast<const __nv_bfloat16*>(add_src->data_ptr());
        keep.push_back(*add_src);
      }
    }
    if (raw.stats == 2) {
      // fused BatchNorm-backward reduction: y has exactly the output's shape / layout
      TORCH_CHECK(bn_scale.has_value() && bn_shift.has_value(), "bwd stats need the forward BN scale/shift");
      check_nhwc_view(*bwd_y, "bwd_y");
      TORCH_CHECK(bwd_y->sizes() == out.sizes() && bwd_y->strides() == out.strides(), "bwd_y must match the output");
      TORCH_CHECK(bn_scale->scalar_type() == at::kFloat && bn_shift->scalar_type() == at::kFloat &&
                  bn_scale->numel() >= cout && bn_shift->numel() >= cout);
      p.bn_scale = bn_scale->data_ptr<float>();
      p.bn_shift = bn_shift->data_ptr<float>();
      if (bw == 0) raw.tmY = map_2d(bwd_y->data_ptr(), N * Ho * Wo, cout, cout, 64, kBlockM);
      else raw.tmY = map_nhwc(*bwd_y, 64, (int)bw, (int)bh, (int)bn);
      keep.push_back(*bwd_y);
      keep.push_back(*bn_scale);
      keep.push_back(*bn_shift);
    }
    if (raw.stats >= 1 && raw.stats <= 3) {
      TORCH_CHECK(stat_sqsum.has_value());
      TORCH_CHECK(stat_sum->is_cuda() && stat_sum->scalar_type() == at::kFloat && stat_sum->numel() >= cout);
      TORCH_CHECK(stat_sqsum->is_cuda() && stat_sqsum->scalar_type() == at::kFloat && stat_sqsum->numel() >= cout);
      p.stat_sum = stat_sum->data_ptr<float>();
      p.stat_sqsum = stat_sqsum->data_ptr<float>();
      keep.push_back(*stat_sum);
      keep.push_back(*stat_sqsum);
    }
    const int cap = max_ctas > 0 ? (int)max_ctas : sm_count();
    raw.grid = p.num_tiles < cap ? p.num_tiles : cap;
    for (auto& v : views) keep.push_back(v);
    keep.push_back(weight);
    keep.push_back(out);
  }
  void run() {
    conv_plan_launch(raw, at::cuda::getCurrentCUDAStream());
    ++launches;
  }
  int grid() const { return raw.grid; }
  int block_n() const { return raw.block_n; }
  int res_b() const { return raw.res_b; }
  int halo() const { return raw.halo; }
  int stats_mode() const { return raw.stats; }
};

struct WgradPlan {
  WgradPlanRaw raw;
  std::vector<at::Tensor> keep;
  int64_t launches = 0;

  // dy: NHWC view (N, Ho, Wo, Cout) bf16;  views: input views on the same pixel grid;  dw: fp32 [taps*Cout, Cin]
  WgradPlan(at::Tensor dy, std::vector<at::Tensor> views, at::Tensor dw, int64_t R, int64_t S,
            std::vector<int64_t> tap_map, std::vector<int64_t> tap_dw, std::vector<int64_t> tap_dh, int64_t bw,
            int64_t bh, int64_t bn, int64_t px_chunks, int64_t max_ctas, int64_t smem_budget) {
    check_nhwc_view(dy, "dy");
    TORCH_CHECK(!views.empty() && views.size() <= 4);
    for (auto& v : views) check_nhwc_view(v, "input view");
    const int taps = (int)(R * S);
    TORCH_CHECK(taps >= 1 && taps <= kMaxTaps && (int)tap_map.size() == taps && (int)tap_dw.size() == taps &&
                (int)tap_dh.size() == taps);
    const int64_t cout = dy.size(3), cin = views[0].size(3);
    TORCH_CHECK(cin % 64 == 0 && (cout == 64 || cout % 128 == 0), "wgrad: Cin % 64 == 0 and Cout == 64 or % 128 == 0");
    TORCH_CHECK(dw.is_cuda() && dw.scalar_type() == at::kFloat && dw.is_contiguous() && dw.numel() == taps * cout * cin,
                "dw must be fp32 [taps*Cout, Cin]");
    TORCH_CHECK(S >= 1 && S <= 4, "filter width 1..4");
    WgradParams& p = raw.p;
    std::memset(&p, 0, sizeof(p));
    p.cout = (int)cout;
    p.cin = (int)cin;
    p.S = (int)S;
    p.a_chunks = cout == 64 ? 1 : 2;
    p.co_blocks = (int)((cout + 127) / 128);
    const int cin_blocks = (int)(cin / 64);
    if (S == 1) {
      p.cb_per_group = cin_blocks < 4 ? cin_blocks : 4;
      while (cin_blocks % p.cb_per_group) --p.cb_per_group;
      p.acc_chunks = p.cb_per_group;
    } else {
      p.cb_per_group = (cin_blocks >= 2 && S * 2 <= 6) ? 2 : 1;
      p.acc_chunks = (int)S;
    }
    p.G = (int)S * p.cb_per_group;
    p.cgroups = cin_blocks / p.cb_per_group;
    p.groups = (int)R * p.cgroups;
    for (int t = 0; t < taps; ++t) {
      TORCH_CHECK(tap_map[t] >= 0 && tap_map[t] < (int64_t)views.size());
      p.tap_map[t] = (int8_t)tap_map[t];
      p.tap_dw[t] = (int8_t)tap_dw[t];
      p.tap_dh[t] = (int8_t)tap_dh[t];
    }
    const int64_t N = dy.size(0), Ho = dy.size(1), Wo = dy.size(2);
    if (bw == 0) {
      TORCH_CHECK(views.size() == 1 && taps == 1 && dy.is_contiguous() && views[0].is_contiguous());
      const int64_t M = N * Ho * Wo;
      p.mode = 0;
      p.P = 64;
      TORCH_CHECK(M % p.P == 0, "flat wgrad needs pixels % 64 == 0");
      p.iters_total = (int)(M / p.P);
      raw.tmDY = map_2d(dy.data_ptr(), M, cout, cout, 64, p.P);
      raw.tmX[0] = map_2d(views[0].data_ptr(), M, cin, cin, 64, p.P);
      for (int i = 1; i < 4; ++i) raw.tmX[i] = raw.tmX[0];
    } else {
      const int64_t P = bw * bh * bn;
      TORCH_CHECK(P % 16 == 0 && P <= 128, "wgrad pixel box must hold a multiple of 16 pixels (<= 128), got ", P);
      TORCH_CHECK(Wo % bw == 0 && Ho % bh == 0, "box must tile the dy plane exactly");
      p.mode = 1;
      p.P = (int)P;
      p.bw = (int)bw;
      p.bh = (int)bh;
      p.bn = (int)bn;
      p.tiles_w = (int)(Wo / bw);
      p.tiles_h = (int)(Ho / bh);
      p.iters_total = (int)(p.tiles_w * p.tiles_h * ((N + bn - 1) / bn));
      raw.tmDY = map_nhwc(dy, 64, (int)bw, (int)bh, (int)bn);
      for (size_t i = 0; i < 4; ++i) {
        const at::Tensor& v = views[i < views.size() ? i : 0];
        TORCH_CHECK(v.size(0) == N && v.size(3) == cin);
        raw.tmX[i] = map_nhwc(v, 64, (int)bw, (int)bh, (int)bn);
      }
    }
    const int stage_bytes = (p.a_chunks + p.G) * p.P * 128;
    // smem_budget < 227 KB leaves room for bandwidth-bound kernels to co-reside when wgrad runs on a side stream
    const int budget = (smem_budget > 0 && smem_budget < 232448) ? (int)smem_budget : 232448;
    p.stages = (budget - 256) / stage_bytes;
    if (p.stages > 8) p.stages = 8;
    TORCH_CHECK(p.stages >= 2, "wgrad stage does not fit shared memory");
    const int combos = p.co_blocks * p.groups;
    const int cap = max_ctas > 0 ? (int)max_ctas : sm_count();
    // one wave of units: every extra pixel chunk costs a full accumulator flush of fp32 atomics
    int64_t pc = px_chunks > 0 ? px_chunks : cap / combos;
    if (pc < 1) pc = 1;
    if (pc > p.iters_total) pc = p.iters_total;
    p.iters_per_chunk = (int)((p.iters_total + pc - 1) / pc);
    p.px_chunks = (p.iters_total + p.iters_per_chunk - 1) / p.iters_per_chunk;
    p.num_units = p.px_chunks * combos;
    p.dw = dw.data_ptr<float>();
    raw.grid = p.num_units < cap ? p.num_units : cap;
    keep.push_back(dy);
    for (auto& v : views) keep.push_back(v);
    keep.push_back(dw);
  }
  void run() {
    wgrad_plan_launch(raw, at::cuda::getCurrentCUDAStream());
    ++launches;
  }
  int grid() const { return raw.grid; }
  int units() const { return raw.p.num_units; }
  int stages() const { return raw.p.stages; }
};

struct StemPlan {
  StemPlanRaw raw;
  std::vector<at::Tensor> keep;
  int64_t launches = 0;
  bool is_wgrad;

  // forward: y = conv7x7s2(x_u8 * mul + add, w) (+ BN statistics);  wgrad: dw += dy (x) patches
  StemPlan(at::Tensor x_u8, c10::optional<at::Tensor> w16, at::Tensor y_or_dy, c10::optional<at::Tensor> dw,
           c10::optional<at::Tensor> stat_sum, c10::optional<at::Tensor> stat_sqsum, double mul, double add,
           int64_t max_ctas) {
    TORCH_CHECK(x_u8.is_cuda() && x_u8.scalar_type() == at::kByte && x_u8.is_contiguous() && x_u8.dim() == 4 &&
                x_u8.size(3) == 3, "x must be uint8 [N, H, W, 3]");
    TORCH_CHECK(y_or_dy.is_cuda() && y_or_dy.scalar_type() == at::kBFloat16 && y_or_dy.is_contiguous() &&
                y_or_dy.dim() == 4 && y_or_dy.size(3) == 64, "y/dy must be bf16 [N, Ho, Wo, 64]");
    std::memset(&raw.p, 0, sizeof(raw.p));
    StemParams& p = raw.p;
    p.x = x_u8.data_ptr<uint8_t>();
    p.N = (int)x_u8.size(0);
    p.H = (int)x_u8.size(1);
    p.W = (int)x_u8.size(2);
    p.Ho = (int)y_or_dy.size(1);
    p.Wo = (int)y_or_dy.size(2);
    TORCH_CHECK(p.Ho == (p.H + 6 - 7) / 2 + 1 && p.Wo == (p.W + 6 - 7) / 2 + 1 && y_or_dy.size(0) == p.N,
                "stem output shape mismatch");
    TORCH_CHECK(p.Wo <= 128 && p.W % 16 == 0 && p.W <= 256, "stem kernel needs W % 16 == 0 and W <= 256");
    p.M = (int64_t)p.N * p.Ho * p.Wo;
    p.num_tiles = p.N * p.Ho;  // one output row per tile
    p.mul = (float)mul;
    p.add = (float)add;
    is_wgrad = dw.has_value();
    raw.tmY = map_2d(y_or_dy.data_ptr(), p.M, 64, 64, 64, p.Wo);
    if (is_wgrad) {
      TORCH_CHECK(dw->is_cuda() && dw->scalar_type() == at::kFloat && dw->is_contiguous() && dw->numel() == 49 * 64 * 3);
      p.dw = dw->data_ptr<float>();
      raw.tmW = raw.tmY;
      keep.push_back(*dw);
    } else {
      TORCH_CHECK(w16.has_value() && w16->is_cuda() && w16->scalar_type() == at::kBFloat16 && w16->is_contiguous() &&
                  w16->dim() == 2 && w16->size(0) == 64 && w16->size(1) == 192, "stem weight must be bf16 [64, 192]");
      raw.tmW = map_2d(w16->data_ptr(), 64, 192, 192, 64, 64);
      keep.push_back(*w16);
      if (stat_sum.has_value()) {
        TORCH_CHECK(stat_sqsum.has_value() && stat_sum->scalar_type() == at::kFloat && stat_sum->numel() >= 64);
        p.stat_sum = stat_sum->data_ptr<float>();
        p.stat_sqsum = stat_sqsum->data_ptr<float>();
        keep.push_back(*stat_sum);
        keep.push_back(*stat_sqsum);
      }
    }
    const int cap = max_ctas > 0 ? (int)max_ctas : sm_count();
    raw.grid = p.num_tiles < cap ? p.num_tiles : cap;
    keep.push_back(x_u8);
    keep.push_back(y_or_dy);
  }
  void run() {
    if (is_wgrad) stem_wgrad_launch(raw, at::cuda::getCurrentCUDAStream());
    else stem_fwd_launch(raw, at::cuda::getCurrentCUDAStream());
    ++launches;
  }
};

}  // namespace b200

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  namespace py = pybind11;
  m.doc() = "b200ddl tcgen05/TMA implicit-GEMM convolution kernels (sm_100a)";
  py::class_<b200::ConvPlan>(m, "ConvPlan")
      .def(py::init<std::vector<at::Tensor>, at::Tensor, at::Tensor, std::vector<int64_t>, std::vector<int64_t>,
                    std::vector<int64_t>, int64_t, int64_t, int64_t, c10::optional<at::Tensor>,
                    c10::optional<at::Tensor>, int64_t, c10::optional<at::Tensor>, c10::optional<at::Tensor>,
                    c10::optional<at::Tensor>, c10::optional<at::Tensor>, c10::optional<at::Tensor>, c10::optional<at::Tensor>,
                    c10::optional<at::Tensor>, int64_t>(),
           py::arg("views"), py::arg("weight"), py::arg("out"), py::arg("tap_map"), py::arg("tap_dw"),
           py::arg("tap_dh"), py::arg("bw"), py::arg("bh"), py::arg("bn"), py::arg("stat_sum") = c10::nullopt,
           py::arg("stat_sqsum") = c10::nullopt, py::arg("max_ctas") = 0, py::arg("bwd_y") = c10::nullopt,
           py::arg("bn_scale") = c10::nullopt, py::arg("bn_shift") = c10::nullopt, py::arg("add_src") = c10::nullopt,
           py::arg("relu_mask") = c10::nullopt, py::arg("ep_scale") = c10::nullopt, py::arg("ep_shift") = c10::nullopt,
           py::arg("ep_act") = 0)
      .def("run", &b200::ConvPlan::run)
      .def_readonly("launches", &b200::ConvPlan::launches)
      .def_property_readonly("grid", &b200::ConvPlan::grid)
      .def_property_readonly("block_n", &b200::ConvPlan::block_n)
      .def_property_readonly("resident_filter", &b200::ConvPlan::res_b)
      .def_property_readonly("halo", &b200::ConvPlan::halo)
      .def_property_readonly("stats_mode", &b200::ConvPlan::stats_mode);
  py::class_<b200::WgradPlan>(m, "WgradPlan")
      .def(py::init<at::Tensor, std::vector<at::Tensor>, at::Tensor, int64_t, int64_t, std::vector<int64_t>,
                    std::vector<int64_t>, std::vector<int64_t>, int64_t, int64_t, int64_t, int64_t, int64_t, int64_t>(),
           py::arg("dy"), py::arg("views"), py::arg("dw"), py::arg("R"), py::arg("S"), py::arg("tap_map"),
           py::arg("tap_dw"), py::arg("tap_dh"), py::arg("bw"), py::arg("bh"), py::arg("bn"),
           py::arg("px_chunks") = 0, py::arg("max_ctas") = 0, py::arg("smem_budget") = 0)
      .def("run", &b200::WgradPlan::run)
      .def_readonly("launches", &b200::WgradPlan::launches)
      .def_property_readonly("grid", &b200::WgradPlan::grid)
      .def_property_readonly("units", &b200::WgradPlan::units)
      .def_property_readonly("stages", &b200::WgradPlan::stages);
  py::class_<b200::StemPlan>(m, "StemPlan")
      .def(py::init<at::Tensor, c10::optional<at::Tensor>, at::Tensor, c10::optional<at::Tensor>,
                    c10::optional<at::Tensor>, c10::optional<at::Tensor>, double, double, int64_t>(),
           py::arg("x_u8"), py::arg("w16"), py::arg("y_or_dy"), py::arg("dw") = c10::nullopt,
           py::arg("stat_sum") = c10::nullopt, py::arg("stat_sqsum") = c10::nullopt, py::arg("mul") = 1.0 / 127.5,
           py::arg("add") = -1.0, py::arg("max_ctas") = 0)
      .def("run", &b200::StemPlan::run)
      .def_readonly("launches", &b200::StemPlan::launches);
}
