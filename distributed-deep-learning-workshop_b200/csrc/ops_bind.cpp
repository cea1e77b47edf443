// pybind layer for the bandwidth-bound kernels and fused optimizers (tensor checks + raw-pointer dispatch).
#include <ATen/cuda/CUDAContext.h>
#include <torch/extension.h>

#include <cstdint>

#include "ops_api.h"

namespace {

using at::Tensor;
using OptT = c10::optional<at::Tensor>;

int64_t g_launches = 0;  // number of kernels of ours launched through this module (bench.py reports it)

inline cudaStream_t cur() { return at::cuda::getCurrentCUDAStream(); }
inline void chk(const Tensor& t, at::ScalarType ty, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be CUDA");
  TORCH_CHECK(t.scalar_type() == ty, name, " has wrong dtype");
  TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}
inline const float* fp(const OptT& t) { return t.has_value() ? t->data_ptr<float>() : nullptr; }
inline const void* vp(const OptT& t) { return t.has_value() ? t->data_ptr() : nullptr; }
inline void after() {
  ++g_launches;
  C10_CUDA_KERNEL_LAUNCH_CHECK();
}

void bn_finalize(Tensor sum, Tensor sqsum, double count, Tensor gamma, Tensor beta, Tensor rmean, Tensor rvar,
                 double momentum, double eps, Tensor mean, Tensor invstd, Tensor scale, Tensor shift, bool training) {
  const int C = (int)gamma.numel();
  for (auto* t : {&sum, &sqsum, &gamma, &beta, &rmean, &rvar, &mean, &invstd, &scale, &shift}) chk(*t, at::kFloat, "bn tensor");
  b200::bn_finalize(sum.data_ptr<float>(), sqsum.data_ptr<float>(), count, gamma.data_ptr<float>(),
                    beta.data_ptr<float>(), rmean.data_ptr<float>(), rvar.data_ptr<float>(), (float)momentum,
                    (float)eps, mean.data_ptr<float>(), invstd.data_ptr<float>(), scale.data_ptr<float>(),
                    shift.data_ptr<float>(), C, training, cur());
  after();
}

void bn_apply(Tensor y, Tensor scale, Tensor shift, OptT res, OptT res_scale, OptT res_shift, Tensor out, bool relu,
              OptT mask) {
  chk(y, at::kBFloat16, "y");
  chk(out, at::kBFloat16, "out");
  const int C = (int)y.size(-1);
  const int64_t M = y.numel() / C;
  TORCH_CHECK(C % 8 == 0 && scale.numel() == C && shift.numel() == C && out.numel() == y.numel());
  if (res.has_value()) { chk(*res, at::kBFloat16, "res"); TORCH_CHECK(res->numel() == y.numel()); }
  if (mask.has_value()) { chk(*mask, at::kByte, "mask"); TORCH_CHECK(mask->numel() * 8 == y.numel()); }
  b200::bn_apply(y.data_ptr(), scale.data_ptr<float>(), shift.data_ptr<float>(), vp(res), fp(res_scale),
                 fp(res_shift), out.data_ptr(), mask.has_value() ? mask->data_ptr() : nullptr, M, C, relu, cur());
  after();
}

void channel_stats(Tensor y, Tensor sum, Tensor sqsum) {
  chk(y, at::kBFloat16, "y");
  const int C = (int)y.size(-1);
  TORCH_CHECK(C % 8 == 0 && C <= 2048);
  b200::channel_stats(y.data_ptr(), sum.data_ptr<float>(), sqsum.data_ptr<float>(), y.numel() / C, C, cur());
  after();
}

// mode: 1 = ReLU mask from `outp` (g2 / dz_out optional), 2 = mask from y*scale+shift, 3 = no mask
void bn_bwd_reduce(int64_t mode, Tensor g1, OptT g2, OptT outp, Tensor y, OptT scale, OptT shift, OptT dz_out,
                   Tensor sum_dz, Tensor sum_dzy) {
  chk(g1, at::kBFloat16, "g1");
  chk(y, at::kBFloat16, "y");
  const int C = (int)y.size(-1);
  TORCH_CHECK(C % 8 == 0 && C <= 2048 && g1.numel() == y.numel());
  TORCH_CHECK(mode >= 1 && mode <= 4);
  TORCH_CHECK((mode != 1 && mode != 4) || outp.has_value(), "modes 1/4 need the activation output / bitmask");
  TORCH_CHECK(mode != 2 || (scale.has_value() && shift.has_value()), "mode 2 needs scale/shift");
  b200::bn_bwd_reduce((int)mode, g1.data_ptr(), vp(g2), vp(outp), y.data_ptr(), fp(scale), fp(shift),
                      dz_out.has_value() ? dz_out->data_ptr() : nullptr, sum_dz.data_ptr<float>(),
                      sum_dzy.data_ptr<float>(), y.numel() / C, C, cur());
  after();
}

void bn_bwd_coeffs(Tensor sum_dz, Tensor sum_dzy, Tensor gamma, Tensor mean, Tensor invstd, double count,
                   Tensor dgamma, Tensor dbeta, Tensor cA, Tensor cB, Tensor cC) {
  const int C = (int)gamma.numel();
  b200::bn_bwd_coeffs(sum_dz.data_ptr<float>(), sum_dzy.data_ptr<float>(), gamma.data_ptr<float>(),
                      mean.data_ptr<float>(), invstd.data_ptr<float>(), count, dgamma.data_ptr<float>(),
                      dbeta.data_ptr<float>(), cA.data_ptr<float>(), cB.data_ptr<float>(), cC.data_ptr<float>(), C,
                      cur());
  after();
}

// dy = A*dz + B*y + C;  dz = g (scale absent) or g * (y*scale+shift > 0)
void bn_bwd_apply(Tensor g, Tensor y, OptT scale, OptT shift, Tensor cA, Tensor cB, Tensor cC, Tensor dy) {
  chk(g, at::kBFloat16, "g");
  chk(y, at::kBFloat16, "y");
  chk(dy, at::kBFloat16, "dy");
  const int C = (int)y.size(-1);
  b200::bn_bwd_apply(g.data_ptr(), y.data_ptr(), fp(scale), fp(shift), cA.data_ptr<float>(), cB.data_ptr<float>(),
                     cC.data_ptr<float>(), dy.data_ptr(), y.numel() / C, C, cur());
  after();
}

void maxpool_fwd(Tensor x, Tensor out, OptT idx) {
  chk(x, at::kBFloat16, "x");
  chk(out, at::kBFloat16, "out");
  if (idx.has_value()) { chk(*idx, at::kByte, "idx"); TORCH_CHECK(idx->numel() == out.numel()); }
  b200::maxpool_fwd(x.data_ptr(), out.data_ptr(), idx.has_value() ? idx->data_ptr() : nullptr, (int)x.size(0),
                    (int)x.size(1), (int)x.size(2), (int)x.size(3), cur());
  after();
}
void bn_relu_maxpool_fwd(Tensor y, Tensor scale, Tensor shift, Tensor out, OptT idx) {
  chk(y, at::kBFloat16, "y");
  chk(out, at::kBFloat16, "out");
  chk(scale, at::kFloat, "scale");
  chk(shift, at::kFloat, "shift");
  if (idx.has_value()) { chk(*idx, at::kByte, "idx"); TORCH_CHECK(idx->numel() == out.numel()); }
  b200::bn_relu_maxpool_fwd(y.data_ptr(), scale.data_ptr<float>(), shift.data_ptr<float>(), out.data_ptr(),
                            idx.has_value() ? idx->data_ptr() : nullptr, (int)y.size(0), (int)y.size(1),
                            (int)y.size(2), (int)y.size(3), cur());
  after();
}
void maxpool_bwd(Tensor idx, Tensor g1, OptT g2, Tensor dx) {
  chk(idx, at::kByte, "idx");
  chk(g1, at::kBFloat16, "g1");
  chk(dx, at::kBFloat16, "dx");
  b200::maxpool_bwd(idx.data_ptr(), g1.data_ptr(), vp(g2), dx.data_ptr(), (int)dx.size(0), (int)dx.size(1),
                    (int)dx.size(2), (int)dx.size(3), cur());
  after();
}
void gap_fwd(Tensor x, Tensor out, double drop_p, int64_t seed) {
  chk(x, at::kBFloat16, "x");
  chk(out, at::kBFloat16, "out");
  const int N = (int)x.size(0), C = (int)x.size(-1);
  b200::gap_fwd(x.data_ptr(), out.data_ptr(), N, (int)(x.numel() / N / C), C, (float)drop_p, (uint64_t)seed, cur());
  after();
}
void gap_bwd(Tensor dout, Tensor dx, double drop_p, int64_t seed) {
  chk(dout, at::kBFloat16, "dout");
  chk(dx, at::kBFloat16, "dx");
  const int N = (int)dx.size(0), C = (int)dx.size(-1);
  b200::gap_bwd(dout.data_ptr(), dx.data_ptr(), N, (int)(dx.numel() / N / C), C, (float)drop_p, (uint64_t)seed, cur());
  after();
}
void softmax_ce(Tensor logits, Tensor labels, OptT dlogits, OptT loss_rows, Tensor stats, double grad_scale) {
  chk(logits, at::kFloat, "logits");
  chk(labels, at::kLong, "labels");
  chk(stats, at::kFloat, "stats");
  b200::softmax_ce(logits.data_ptr<float>(), labels.data_ptr<int64_t>(),
                   dlogits.has_value() ? dlogits->data_ptr<float>() : nullptr,
                   loss_rows.has_value() ? loss_rows->data_ptr<float>() : nullptr, stats.data_ptr<float>(),
                   (int)logits.size(0), (int)logits.size(1), (float)grad_scale, cur());
  after();
}
// classifier head: bf16 logits [B, ld] (first K columns real) + fp32 bias -> loss / accuracy / bf16 dlogits [B, ld]
void softmax_ce_head(Tensor logits16, Tensor bias, Tensor labels, OptT logits32, OptT dlogits16, OptT loss_rows,
                     Tensor stats, double grad_scale) {
  chk(logits16, at::kBFloat16, "logits16");
  chk(bias, at::kFloat, "bias");
  chk(labels, at::kLong, "labels");
  chk(stats, at::kFloat, "stats");
  TORCH_CHECK(logits16.dim() == 2 && bias.numel() <= logits16.size(1) && labels.numel() == logits16.size(0));
  const int B = (int)logits16.size(0), ld = (int)logits16.size(1), K = (int)bias.numel();
  if (logits32.has_value()) { chk(*logits32, at::kFloat, "logits32"); TORCH_CHECK(logits32->numel() == (int64_t)B * K); }
  if (dlogits16.has_value()) { chk(*dlogits16, at::kBFloat16, "dlogits16"); TORCH_CHECK(dlogits16->numel() == logits16.numel()); }
  b200::softmax_ce_head(logits16.data_ptr(), ld, bias.data_ptr<float>(), labels.data_ptr<int64_t>(),
                        logits32.has_value() ? logits32->data_ptr<float>() : nullptr,
                        dlogits16.has_value() ? dlogits16->data_ptr() : nullptr,
                        loss_rows.has_value() ? loss_rows->data_ptr<float>() : nullptr, stats.data_ptr<float>(), B, K,
                        (float)grad_scale, cur());
  after();
}
void fc_bias_grad(Tensor dlogits16, Tensor dbias) {
  chk(dlogits16, at::kBFloat16, "dlogits16");
  chk(dbias, at::kFloat, "dbias");
  TORCH_CHECK(dlogits16.dim() == 2 && dbias.numel() <= dlogits16.size(1));
  b200::fc_bias_grad(dlogits16.data_ptr(), (int)dlogits16.size(1), dbias.data_ptr<float>(), (int)dlogits16.size(0),
                     (int)dbias.numel(), cur());
  after();
}
void pack_stem_weight(Tensor w, Tensor out) {
  chk(w, at::kFloat, "w");
  chk(out, at::kBFloat16, "out");
  TORCH_CHECK(w.numel() == 49 * 64 * 3 && out.numel() == 64 * 192);
  b200::pack_stem_weight(w.data_ptr<float>(), out.data_ptr(), cur());
  after();
}
// cudaMemsetAsync on the current stream (a memset node under graph capture, not a kernel)
void zero_(Tensor t) {
  TORCH_CHECK(t.is_cuda() && t.is_contiguous());
  C10_CUDA_CHECK(cudaMemsetAsync(t.data_ptr(), 0, t.numel() * t.element_size(), cur()));
}
// MobileNetV2 stem: uint8 [N,H,W,3] -> bf16 [N,H/2,W/2,ldc] (32 real channels), relu6(conv3x3/2(x*mul+add) * scale + shift)
void mbv2_stem(Tensor x, Tensor w, Tensor scale, Tensor shift, Tensor out, double mul, double add) {
  chk(x, at::kByte, "x");
  chk(w, at::kFloat, "w");
  chk(scale, at::kFloat, "scale");
  chk(shift, at::kFloat, "shift");
  chk(out, at::kBFloat16, "out");
  TORCH_CHECK(x.dim() == 4 && x.size(3) == 3 && x.size(1) % 2 == 0 && x.size(2) % 2 == 0, "stem input: uint8 [N, H, W, 3], even H / W");
  TORCH_CHECK(w.numel() == 27 * 32 && scale.numel() >= 32 && shift.numel() >= 32);
  TORCH_CHECK(out.dim() == 4 && out.size(0) == x.size(0) && out.size(1) == x.size(1) / 2 && out.size(2) == x.size(2) / 2 &&
              out.size(3) >= 32 && out.size(3) % 8 == 0);
  b200::mbv2_stem(x.data_ptr<uint8_t>(), w.data_ptr<float>(), scale.data_ptr<float>(), shift.data_ptr<float>(), out.data_ptr(),
                  (int)x.size(0), (int)x.size(1), (int)x.size(2), (int)out.size(3), (float)mul, (float)add, cur());
  after();
}
// depthwise 3x3 (pad 1, stride 1 / 2) + folded BatchNorm + ReLU6;  x bf16 [N,H,W,C], w fp32 [9, C], out bf16 [N,Ho,Wo,C]
void dwconv3x3(Tensor x, Tensor w, Tensor scale, Tensor shift, Tensor out, int64_t stride, int64_t tile_w) {
  chk(x, at::kBFloat16, "x");
  chk(w, at::kFloat, "w");
  chk(scale, at::kFloat, "scale");
  chk(shift, at::kFloat, "shift");
  chk(out, at::kBFloat16, "out");
  TORCH_CHECK((stride == 1 || stride == 2) && (tile_w == 1 || tile_w == 4));
  const int C = (int)x.size(3), H = (int)x.size(1), W = (int)x.size(2);
  TORCH_CHECK(x.dim() == 4 && C % 8 == 0 && w.numel() == 9 * C && scale.numel() == C && shift.numel() == C);
  TORCH_CHECK(out.dim() == 4 && out.size(0) == x.size(0) && out.size(3) == C && out.size(1) == (H - 1) / stride + 1 &&
              out.size(2) == (W - 1) / stride + 1, "dwconv3x3 output shape");
  b200::dwconv3x3(x.data_ptr(), w.data_ptr<float>(), scale.data_ptr<float>(), shift.data_ptr<float>(), out.data_ptr(),
                  (int)x.size(0), H, W, C, (int)stride, (int)tile_w, cur());
  after();
}
// x: uint8 [N, H, W, 3] (planar = false) or [N, 3, H, W] (planar = true, the nvJPEG layout);  out: uint8 [N, OH, OW, 3]
void resize_bilinear_u8(Tensor x, Tensor out, bool planar) {
  chk(x, at::kByte, "x");
  chk(out, at::kByte, "out");
  TORCH_CHECK(x.dim() == 4 && out.dim() == 4 && out.size(3) == 3 && x.size(0) == out.size(0));
  TORCH_CHECK(planar ? x.size(1) == 3 : x.size(3) == 3, "resize_bilinear_u8: 3-channel images");
  const int H = (int)(planar ? x.size(2) : x.size(1)), W = (int)(planar ? x.size(3) : x.size(2));
  b200::resize_bilinear_u8(x.data_ptr<uint8_t>(), out.data_ptr<uint8_t>(), (int)x.size(0), H, W, (int)out.size(1),
                           (int)out.size(2), planar, cur());
  after();
}
void weight_prep(Tensor w, OptT wf, OptT wd, int64_t taps, int64_t cout, int64_t cin) {
  chk(w, at::kFloat, "w");
  TORCH_CHECK(w.numel() == taps * cout * cin);
  b200::weight_prep(w.data_ptr<float>(), wf.has_value() ? wf->data_ptr() : nullptr,
                    wd.has_value() ? wd->data_ptr() : nullptr, (int)taps, (int)cout, (int)cin, cur());
  after();
}
// table: int64 [layers, 6] on the device = (src_off, dst_off, taps, cout, cin, first_tile_index); a tile = 64 co x 32 ci
void weight_prep_batched(Tensor params, Tensor wd, Tensor table, int64_t total) {
  chk(params, at::kFloat, "params");
  chk(wd, at::kBFloat16, "wd");
  chk(table, at::kLong, "table");
  TORCH_CHECK(table.dim() == 2 && table.size(1) == 6 && table.size(0) <= 128);
  b200::weight_prep_batched(params.data_ptr<float>(), wd.data_ptr(), table.data_ptr<int64_t>(), (int)table.size(0),
                            total, cur());
  after();
}
void sgd_step(Tensor p, Tensor g, Tensor mom, OptT p16, Tensor hyper, bool nesterov) {
  chk(p, at::kFloat, "p"); chk(g, at::kFloat, "g"); chk(mom, at::kFloat, "mom"); chk(hyper, at::kFloat, "hyper");
  TORCH_CHECK(p.numel() % 4 == 0 && g.numel() == p.numel() && mom.numel() == p.numel() && hyper.numel() >= b200::kHyperLen);
  b200::sgd_step(p.data_ptr<float>(), g.data_ptr<float>(), mom.data_ptr<float>(),
                 p16.has_value() ? p16->data_ptr() : nullptr, p.numel(), hyper.data_ptr<float>(), nesterov, cur());
  after();
}
void adam_step(Tensor p, Tensor g, Tensor m, Tensor v, OptT p16, Tensor hyper) {
  chk(p, at::kFloat, "p"); chk(g, at::kFloat, "g"); chk(m, at::kFloat, "m"); chk(v, at::kFloat, "v");
  TORCH_CHECK(p.numel() % 4 == 0 && g.numel() == p.numel() && hyper.numel() >= b200::kHyperLen);
  b200::adam_step(p.data_ptr<float>(), g.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                  p16.has_value() ? p16->data_ptr() : nullptr, p.numel(), hyper.data_ptr<float>(), cur());
  after();
}
void adadelta_step(Tensor p, Tensor g, Tensor sq, Tensor acc, OptT p16, Tensor hyper) {
  chk(p, at::kFloat, "p"); chk(g, at::kFloat, "g");
  TORCH_CHECK(p.numel() % 4 == 0 && g.numel() == p.numel() && hyper.numel() >= b200::kHyperLen);
  b200::adadelta_step(p.data_ptr<float>(), g.data_ptr<float>(), sq.data_ptr<float>(), acc.data_ptr<float>(),
                      p16.has_value() ? p16->data_ptr() : nullptr, p.numel(), hyper.data_ptr<float>(), cur());
  after();
}
void cast_bf16(Tensor x, Tensor out) {
  chk(x, at::kFloat, "x"); chk(out, at::kBFloat16, "out");
  TORCH_CHECK(x.numel() % 4 == 0 && out.numel() == x.numel());
  b200::cast_f32_to_bf16(x.data_ptr<float>(), out.data_ptr(), x.numel(), cur());
  after();
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  namespace py = pybind11;
  m.doc() = "b200ddl bandwidth-bound sm_100a kernels and fused optimizers";
  m.def("bn_finalize", &bn_finalize);
  m.def("bn_apply", &bn_apply, py::arg("y"), py::arg("scale"), py::arg("shift"), py::arg("res") = c10::nullopt,
        py::arg("res_scale") = c10::nullopt, py::arg("res_shift") = c10::nullopt, py::arg("out"), py::arg("relu") = true,
        py::arg("mask") = c10::nullopt);
  m.def("channel_stats", &channel_stats);
  m.def("bn_bwd_reduce", &bn_bwd_reduce);
  m.def("bn_bwd_coeffs", &bn_bwd_coeffs);
  m.def("bn_bwd_apply", &bn_bwd_apply);
  m.def("maxpool_fwd", &maxpool_fwd);
  m.def("maxpool_bwd", &maxpool_bwd);
  m.def("bn_relu_maxpool_fwd", &bn_relu_maxpool_fwd);
  m.def("gap_fwd", &gap_fwd);
  m.def("gap_bwd", &gap_bwd);
  m.def("softmax_ce", &softmax_ce);
  m.def("softmax_ce_head", &softmax_ce_head, py::arg("logits16"), py::arg("bias"), py::arg("labels"),
        py::arg("logits32") = c10::nullopt, py::arg("dlogits16") = c10::nullopt, py::arg("loss_rows") = c10::nullopt,
        py::arg("stats"), py::arg("grad_scale") = 1.0);
  m.def("fc_bias_grad", &fc_bias_grad);
  m.def("pack_stem_weight", &pack_stem_weight);
  m.def("zero_", &zero_);
  m.def("mbv2_stem", &mbv2_stem);
  m.def("dwconv3x3", &dwconv3x3, pybind11::arg("x"), pybind11::arg("w"), pybind11::arg("scale"), pybind11::arg("shift"),
        pybind11::arg("out"), pybind11::arg("stride"), pybind11::arg("tile_w") = 4);
  m.def("resize_bilinear_u8", &resize_bilinear_u8, py::arg("x"), py::arg("out"), py::arg("planar") = false);
  m.def("weight_prep", &weight_prep);
  m.def("weight_prep_batched", &weight_prep_batched);
  m.def("sgd_step", &sgd_step);
  m.def("adam_step", &adam_step);
  m.def("adadelta_step", &adadelta_step);
  m.def("cast_bf16", &cast_bf16);
  m.def("launch_count", [] { return g_launches; });
  m.def("reset_launch_count", [] { g_launches = 0; });
}
