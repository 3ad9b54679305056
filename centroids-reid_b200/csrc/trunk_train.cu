// Train-mode trunk behind the C ABI (SURVEY 8b, the "train fwd/bwd variants" of the whole-trunk entry points): what torch
// autograd does through ResNet.forward / ResNet_IBN.forward in train mode (modelling/backbones/resnet.py:67-87,122-133,
// resnet_ibn_a.py:18-32,126-141) and Baseline.forward's global average pool (modelling/baseline.py:91-96), as ONE forward
// call and ONE backward call on an opaque handle.  A host that is not Python runs a training step as
//   ctl_trainer_bind -> ctl_train_forward -> (its loss on global_feat, ctl_ctl_loss_step) -> ctl_train_backward ->
//   ctl_adam_multi_step
// without re-implementing modelling/backbones/engine_train.py.  The launches are the same C entry points engine_train.py
// issues, in the same order, on the same shapes -- the two drivers produce the same bits (tests/test_train_gpu.py).
//
// Memory: everything lives in the caller's workspace of ctl_train_workspace_bytes(...) bytes, carved by a bump allocator
// that is walked once "dry" (no launches) to size it.  The forward keeps y (raw conv output) and z (normalised output) of
// every conv + BatchNorm; the backward ping-pongs the block-boundary gradient between two buffers and resets a scratch
// region after every bottleneck.
#include <string.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.h"
#include "umma.cuh"

namespace ctl {

static constexpr float TT_BN_EPS = 1e-5f;
static constexpr int TT_PACK_CHUNK = 8192;  // == PACK_CHUNK of train.cu

// conv1.weight [64][3][7][7] fp32 -> the tensor-core stem's operand [64][192] fp16, k = (c*7 + r)*8 + s (s = 7, k >= 168 zero)
__global__ void stem_train_pack_kernel(const float* __restrict__ w, __half* __restrict__ w192) {
  const int o = blockIdx.x;
  for (int i = threadIdx.x; i < 192; i += blockDim.x) {
    float v = 0.f;
    if (i < 168 && (i & 7) < 7) v = w[(size_t)o * 147 + (i >> 3) * 7 + (i & 7)];
    w192[(size_t)o * 192 + i] = __float2half_rn(v);
  }
}

// dw [64][192] fp32 (im2col GEMM order) -> conv1.weight's gradient [64][3][7][7], times 1 / loss-scale
__global__ void stem_train_unpack_kernel(const float* __restrict__ dw192, float inv_scale, float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 147) return;
  const int o = i / 147, j = i - o * 147, cr = j / 7, s = j - cr * 7;
  dw[i] = __fmul_rn(dw192[(size_t)o * 192 + cr * 8 + s], inv_scale);
}

// per-image InstanceNorm parameter gradients [n][half] -> [half]: images summed in index order (double accumulator)
__global__ void sum_images_kernel(const float* __restrict__ part, int n, int half, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= half) return;
  double t = 0.0;
  for (int i = 0; i < n; ++i) t += (double)part[(size_t)i * half + c];
  out[c] = (float)t;
}

struct Bump {
  char* base = nullptr;
  size_t off = 0, cap = 0, high = 0;
  bool dry = true;
  void* take(size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) & ~(size_t)255;
    if (off > high) high = off;
    return dry ? nullptr : base + at;
  }
  template <typename T>
  T* take_n(size_t count) {
    return static_cast<T*>(take(count * sizeof(T)));
  }
};

struct ConvSpec {
  std::string conv, bn;
  int cin = 0, cout = 0, k = 1, stride = 1, relu = 1, in_half = 0;  // in_half > 0: IBN (InstanceNorm on [0, half))
  // bound parameters / gradients (device pointers into the host framework's tensors)
  const float *w = nullptr, *gamma = nullptr, *beta = nullptr, *in_gamma = nullptr, *in_beta = nullptr;
  float *rmean = nullptr, *rvar = nullptr;
  float *dw = nullptr, *dgamma = nullptr, *dbeta = nullptr, *din_gamma = nullptr, *din_beta = nullptr;
  __half *wf = nullptr, *wd = nullptr;  // packed forward / data-gradient operands (handle-owned arena)
  // saved by the forward
  const void* a = nullptr;
  void *y = nullptr, *z = nullptr;
  float *mean = nullptr, *invstd = nullptr, *in_mean = nullptr, *in_invstd = nullptr;
  int n = 0, h = 0, w_in = 0, ho = 0, wo = 0;
};

struct TrainBlock {
  ConvSpec c1, c2, c3, down;
  bool has_down = false;
};

}  // namespace ctl

struct ctl_trainer {
  int ibn = 0, last_stride = 1;
  float momentum = 0.1f;
  bool bound = false, forwarded = false;
  std::vector<ctl::TrainBlock> blocks;
  // stem
  const float *w0 = nullptr, *g0 = nullptr, *b0 = nullptr;
  float *rm0 = nullptr, *rv0 = nullptr, *dw0 = nullptr, *dg0 = nullptr, *db0 = nullptr;
  __half* stem_w192 = nullptr;
  void *y0 = nullptr, *z0 = nullptr, *arg0 = nullptr, *pool0 = nullptr;
  float *m0 = nullptr, *i0 = nullptr;
  const float* x = nullptr;
  int n = 0, H = 0, W = 0;
  size_t fwd_mark = 0;  // workspace offset where the backward's scratch starts
  size_t lay_bn = 0, lay_wg = 0, lay_total = 0;  // workspace layout of the last forward (the backward reuses it)
  const void* fwd_workspace = nullptr;
  void* last = nullptr;
  int last_h = 0, last_w = 0;
  // packed operands
  __half* arena = nullptr;
  void* table = nullptr;
  int n_packed = 0;
  long long n_chunks = 0;
  float* zero_bias = nullptr;
  std::vector<void*> owned;
};

namespace ctl {

struct Ref {
  float* data;
  long long numel;
};
using RefMap = std::unordered_map<std::string, Ref>;

static float* lookup(const RefMap& m, const std::string& name, long long numel, bool required, const char* what, int* rc) {
  auto it = m.find(name);
  if (it == m.end() || it->second.data == nullptr) {
    if (required) {
      set_error("ctl_trainer_bind: %s '%s' is missing", what, name.c_str());
      *rc = CTL_ERR_INVALID_ARGUMENT;
    }
    return nullptr;
  }
  if (it->second.numel != numel) {
    set_error("ctl_trainer_bind: %s '%s' has %lld elements, expected %lld", what, name.c_str(), it->second.numel, numel);
    *rc = CTL_ERR_INVALID_ARGUMENT;
    return nullptr;
  }
  return it->second.data;
}

static int bind_conv(ConvSpec& c, const RefMap& p, const RefMap& g) {
  int rc = 0;
  c.w = lookup(p, c.conv + ".weight", (long long)c.cout * c.cin * c.k * c.k, true, "parameter", &rc);
  c.dw = lookup(g, c.conv + ".weight", (long long)c.cout * c.cin * c.k * c.k, true, "gradient", &rc);
  const int nbn = c.cout - c.in_half;
  const std::string bn = c.in_half ? c.bn + ".BN" : c.bn;
  c.gamma = lookup(p, bn + ".weight", nbn, true, "parameter", &rc);
  c.beta = lookup(p, bn + ".bias", nbn, true, "parameter", &rc);
  c.rmean = lookup(p, bn + ".running_mean", nbn, false, "buffer", &rc);
  c.rvar = lookup(p, bn + ".running_var", nbn, false, "buffer", &rc);
  c.dgamma = lookup(g, bn + ".weight", nbn, true, "gradient", &rc);
  c.dbeta = lookup(g, bn + ".bias", nbn, true, "gradient", &rc);
  if (c.in_half) {
    c.in_gamma = lookup(p, c.bn + ".IN.weight", c.in_half, true, "parameter", &rc);
    c.in_beta = lookup(p, c.bn + ".IN.bias", c.in_half, true, "parameter", &rc);
    c.din_gamma = lookup(g, c.bn + ".IN.weight", c.in_half, true, "gradient", &rc);
    c.din_beta = lookup(g, c.bn + ".IN.bias", c.in_half, true, "gradient", &rc);
  }
  if (!rc && (c.rmean == nullptr) != (c.rvar == nullptr)) {
    set_error("ctl_trainer_bind: '%s' needs running_mean and running_var together (or neither)", bn.c_str());
    rc = CTL_ERR_INVALID_ARGUMENT;
  }
  return rc;
}

// conv (raw fp16 output) -> batch statistics -> z = [relu](gamma * xhat + beta [+ residual])   (engine_train.py::_conv_bn)
static int conv_bn_forward(ctl_trainer* t, ConvSpec& c, Bump& ws, void* bn_ws, size_t bn_ws_bytes, size_t* bn_need, const void* a, int n,
                           int h, int w, const void* residual, cudaStream_t st) {
  const int pad = c.k == 3 ? 1 : 0;
  c.n = n;
  c.h = h;
  c.w_in = w;
  c.ho = (h + 2 * pad - c.k) / c.stride + 1;
  c.wo = (w + 2 * pad - c.k) / c.stride + 1;
  c.a = a;
  const long long rows = (long long)n * c.ho * c.wo;
  c.y = ws.take((size_t)rows * c.cout * 2);
  c.z = ws.take((size_t)rows * c.cout * 2);
  const int nbn = c.cout - c.in_half;
  c.mean = ws.take_n<float>(nbn);
  c.invstd = ws.take_n<float>(nbn);
  if (c.in_half) {
    c.in_mean = ws.take_n<float>((size_t)n * c.in_half);
    c.in_invstd = ws.take_n<float>((size_t)n * c.in_half);
  }
  const size_t need = ctl_bn_workspace_bytes(rows, nbn);
  if (need > *bn_need) *bn_need = need;
  if (ws.dry) return 0;
  int rc = ctl_conv2d_nhwc_f16(a, n, h, w, c.cin, c.wf, t->zero_bias, nullptr, c.y, c.cout, c.k, c.stride, 0, 0, st);
  if (rc) return rc;
  if (!c.in_half)
    return ctl_bn_train_forward_nhwc_f16(c.y, rows, c.cout, c.cout, c.gamma, c.beta, TT_BN_EPS, t->momentum, c.rmean, c.rvar, residual,
                                         c.relu, bn_ws, bn_ws_bytes, c.mean, c.invstd, c.z, st);
  // IBN (resnet_ibn_a.py:18-32): InstanceNorm on channels [0, half), batch-statistics BatchNorm on [half, C); ReLU
  rc = ctl_instnorm_train_forward_nhwc_f16(c.y, n, c.ho * c.wo, c.cout, c.in_half, c.in_gamma, c.in_beta, TT_BN_EPS, c.in_mean,
                                           c.in_invstd, c.z, st);
  if (rc) return rc;
  return ctl_bn_train_forward_nhwc_f16(static_cast<const __half*>(c.y) + c.in_half, rows, nbn, c.cout, c.gamma, c.beta, TT_BN_EPS,
                                       t->momentum, c.rmean, c.rvar, nullptr, 1, bn_ws, bn_ws_bytes, c.mean, c.invstd,
                                       static_cast<__half*>(c.z) + c.in_half, st);
}

// BatchNorm (+ ReLU mask) backward of `c`: dz -> dy (new scratch), parameter gradients; with relu_mask dz becomes g = dz * mask
static int bn_backward(ctl_trainer* t, ConvSpec& c, Bump& ws, void* bn_ws, size_t bn_ws_bytes, void* dz, bool relu_mask, float inv_scale,
                       void** dy_out, cudaStream_t st) {
  const long long rows = (long long)c.n * c.ho * c.wo;
  void* dy = ws.take((size_t)rows * c.cout * 2);
  *dy_out = dy;
  float *dgp = nullptr, *dbp = nullptr;
  if (c.in_half) {
    dgp = ws.take_n<float>((size_t)c.n * c.in_half);
    dbp = ws.take_n<float>((size_t)c.n * c.in_half);
  }
  if (ws.dry) return 0;
  if (!c.in_half)
    return ctl_bn_train_backward_nhwc_f16(dz, relu_mask ? c.z : nullptr, c.y, rows, c.cout, c.cout, c.gamma, c.mean, c.invstd, inv_scale,
                                          bn_ws, bn_ws_bytes, relu_mask ? dz : nullptr, c.dgamma, c.dbeta, dy, st);
  int rc = ctl_instnorm_train_backward_nhwc_f16(dz, c.z, c.y, c.n, c.ho * c.wo, c.cout, c.in_half, c.in_gamma, c.in_mean, c.in_invstd,
                                                inv_scale, dgp, dbp, dy, st);
  if (rc) return rc;
  sum_images_kernel<<<(c.in_half + 127) / 128, 128, 0, st>>>(dgp, c.n, c.in_half, c.din_gamma);
  sum_images_kernel<<<(c.in_half + 127) / 128, 128, 0, st>>>(dbp, c.n, c.in_half, c.din_beta);
  CTL_LAUNCH_CHECK();
  const int nbn = c.cout - c.in_half;
  __half* dzb = static_cast<__half*>(dz) + c.in_half;
  return ctl_bn_train_backward_nhwc_f16(dzb, static_cast<const __half*>(c.z) + c.in_half, static_cast<const __half*>(c.y) + c.in_half, rows,
                                        nbn, c.cout, c.gamma, c.mean, c.invstd, inv_scale, bn_ws, bn_ws_bytes, dzb, c.dgamma, c.dbeta,
                                        static_cast<__half*>(dy) + c.in_half, st);
}

// weight gradient of `c` (parameter layout, un-scaled) and, when `dx_out`, the data gradient w.r.t. its input (+ residual)
// written to *dx_out (a caller buffer) or fresh scratch (engine_train.py::_conv_bwd)
static int conv_backward(ctl_trainer* t, ConvSpec& c, Bump& ws, void* wg_ws, size_t wg_ws_bytes, size_t* wg_need, const void* dy,
                         float inv_scale, bool need_dx, const void* residual, void* dx_buffer, void** dx_out, cudaStream_t st) {
  const size_t need = ctl_conv2d_wgrad_workspace_bytes(c.n, c.h, c.w_in, c.cin, c.cout, c.k, c.stride);
  if (need > *wg_need) *wg_need = need;
  int rc = 0;
  if (!ws.dry) {
    rc = ctl_conv2d_wgrad_nhwc_f16_ex(c.a, c.n, c.h, c.w_in, c.cin, dy, c.cout, c.k, c.stride, wg_ws, wg_ws_bytes, c.dw, inv_scale, 1, st);
    if (rc) return rc;
  }
  if (!need_dx) return 0;
  const size_t in_bytes = (size_t)c.n * c.h * c.w_in * c.cin * 2;
  void* dx = dx_buffer ? dx_buffer : ws.take(in_bytes);
  *dx_out = dx;
  if (c.stride == 1) {
    if (ws.dry) return 0;
    return ctl_conv2d_nhwc_f16(dy, c.n, c.ho, c.wo, c.cout, c.wd, t->zero_bias, residual, dx, c.cin, c.k, 1, 0, 0, st);
  }
  if (c.k == 1) {  // strided 1x1: low-resolution GEMM, then zero-insertion (+ residual)
    void* low = ws.take((size_t)c.n * c.ho * c.wo * c.cin * 2);
    if (ws.dry) return 0;
    rc = ctl_conv2d_nhwc_f16(dy, c.n, c.ho, c.wo, c.cout, c.wd, t->zero_bias, nullptr, low, c.cin, 1, 1, 0, 0, st);
    if (rc) return rc;
    return ctl_upsample2_zero_nhwc_f16(low, c.n, c.ho, c.wo, c.cin, residual, dx, st);
  }
  void* up = ws.take((size_t)c.n * c.h * c.w_in * c.cout * 2);  // strided 3x3: zero-insert dy, then the stride-1 transposed conv
  if (ws.dry) return 0;
  rc = ctl_upsample2_zero_nhwc_f16(dy, c.n, c.ho, c.wo, c.cout, nullptr, up, st);
  if (rc) return rc;
  return ctl_conv2d_nhwc_f16(up, c.n, c.h, c.w_in, c.cout, c.wd, t->zero_bias, residual, dx, c.cin, 3, 1, 0, 0, st);
}

struct Plan {
  size_t bn_need = 0, wg_need = 0;
};

// The forward walk.  dry: sizes only.  Returns 0 or an error code.
static int forward_walk(ctl_trainer* t, Bump& ws, Plan& plan, void* bn_ws, size_t bn_ws_bytes, const float* x, int n, int H, int W,
                        float* out_feat, cudaStream_t st) {
  int rc = 0;
  const int h = (H + 6 - 7) / 2 + 1, w = (W + 6 - 7) / 2 + 1;
  const int hp = (h + 2 - 3) / 2 + 1, wp = (w + 2 - 3) / 2 + 1;
  const long long rows0 = (long long)n * h * w;
  t->y0 = ws.take((size_t)rows0 * 64 * 2);
  t->z0 = ws.take((size_t)rows0 * 64 * 2);
  t->m0 = ws.take_n<float>(64);
  t->i0 = ws.take_n<float>(64);
  t->pool0 = ws.take((size_t)n * hp * wp * 64 * 2);
  t->arg0 = ws.take((size_t)n * hp * wp * 64);
  plan.bn_need = std::max(plan.bn_need, ctl_bn_workspace_bytes(rows0, 64));
  if (!ws.dry) {
    // stem: raw 7x7/2 conv -> BatchNorm (ReLU only in the IBN-a variant, resnet.py:125 / resnet_ibn_a.py:129) -> max-pool
    stem_train_pack_kernel<<<64, 192, 0, st>>>(t->w0, t->stem_w192);
    CTL_LAUNCH_CHECK();
    if ((rc = ctl_stem_conv7x7_tc(x, n, H, W, t->stem_w192, t->zero_bias, 0, t->y0, st))) return rc;
    if ((rc = ctl_bn_train_forward_nhwc_f16(t->y0, rows0, 64, 64, t->g0, t->b0, TT_BN_EPS, t->momentum, t->rm0, t->rv0, nullptr, t->ibn,
                                            bn_ws, bn_ws_bytes, t->m0, t->i0, t->z0, st)))
      return rc;
    if ((rc = ctl_maxpool3x3s2_argmax_nhwc_f16(t->z0, n, h, w, 64, t->pool0, t->arg0, st))) return rc;
    if ((rc = ctl_train_pack_weights(t->table, t->n_packed, t->n_chunks, st))) return rc;
  }
  const void* a = t->pool0;
  int hh = hp, ww = wp;
  for (TrainBlock& b : t->blocks) {
    if ((rc = conv_bn_forward(t, b.c1, ws, bn_ws, bn_ws_bytes, &plan.bn_need, a, n, hh, ww, nullptr, st))) return rc;
    if ((rc = conv_bn_forward(t, b.c2, ws, bn_ws, bn_ws_bytes, &plan.bn_need, b.c1.z, n, b.c1.ho, b.c1.wo, nullptr, st))) return rc;
    const void* res = a;
    if (b.has_down) {
      if ((rc = conv_bn_forward(t, b.down, ws, bn_ws, bn_ws_bytes, &plan.bn_need, a, n, hh, ww, nullptr, st))) return rc;
      res = b.down.z;
    }
    if ((rc = conv_bn_forward(t, b.c3, ws, bn_ws, bn_ws_bytes, &plan.bn_need, b.c2.z, n, b.c2.ho, b.c2.wo, res, st))) return rc;
    a = b.c3.z;
    hh = b.c3.ho;
    ww = b.c3.wo;
  }
  t->last = const_cast<void*>(a);
  t->last_h = hh;
  t->last_w = ww;
  if (!ws.dry) rc = ctl_gap_bn_nhwc_f16(a, n, hh * ww, 2048, nullptr, nullptr, out_feat, nullptr, st);
  return rc;
}

static int backward_walk(ctl_trainer* t, Bump& ws, Plan& plan, void* bn_ws, size_t bn_ws_bytes, void* wg_ws, size_t wg_ws_bytes,
                         const float* dfeat, float grad_scale, cudaStream_t st) {
  int rc = 0;
  const int n = t->n;
  const float inv_scale = (float)(1.0 / (double)grad_scale);
  // the block-boundary gradient ping-pongs between two buffers of the largest block input
  size_t edge = 0;
  for (const TrainBlock& b : t->blocks) edge = std::max(edge, (size_t)n * b.c1.h * b.c1.w_in * b.c1.cin * 2);
  edge = std::max(edge, (size_t)n * t->last_h * t->last_w * 2048 * 2);
  void* pp[2] = {ws.take(edge), ws.take(edge)};
  int cur = 0;
  if (!ws.dry)
    if ((rc = ctl_gap_backward_nhwc_f16(dfeat, n, t->last_h * t->last_w, 2048, (float)((double)grad_scale / (double)(t->last_h * t->last_w)), pp[0], st)))
      return rc;
  const size_t mark = ws.off;
  for (size_t bi = t->blocks.size(); bi-- > 0;) {
    TrainBlock& b = t->blocks[bi];
    ws.off = mark;
    void* dz = pp[cur];
    void *dy3, *d2, *dy2, *d1, *dy1, *dyd, *shortcut = dz, *unused;
    if ((rc = bn_backward(t, b.c3, ws, bn_ws, bn_ws_bytes, dz, true, inv_scale, &dy3, st))) return rc;  // dz becomes g3
    if ((rc = conv_backward(t, b.c3, ws, wg_ws, wg_ws_bytes, &plan.wg_need, dy3, inv_scale, true, nullptr, nullptr, &d2, st))) return rc;
    if ((rc = bn_backward(t, b.c2, ws, bn_ws, bn_ws_bytes, d2, true, inv_scale, &dy2, st))) return rc;
    if ((rc = conv_backward(t, b.c2, ws, wg_ws, wg_ws_bytes, &plan.wg_need, dy2, inv_scale, true, nullptr, nullptr, &d1, st))) return rc;
    if ((rc = bn_backward(t, b.c1, ws, bn_ws, bn_ws_bytes, d1, true, inv_scale, &dy1, st))) return rc;
    if (b.has_down) {
      if ((rc = bn_backward(t, b.down, ws, bn_ws, bn_ws_bytes, dz, false, inv_scale, &dyd, st))) return rc;
      if ((rc = conv_backward(t, b.down, ws, wg_ws, wg_ws_bytes, &plan.wg_need, dyd, inv_scale, true, nullptr, nullptr, &shortcut, st)))
        return rc;
    }
    if ((rc = conv_backward(t, b.c1, ws, wg_ws, wg_ws_bytes, &plan.wg_need, dy1, inv_scale, true, shortcut, pp[cur ^ 1], &unused, st)))
      return rc;
    cur ^= 1;
  }
  ws.off = mark;
  // stem: max-pool -> BatchNorm (ReLU mask only for IBN-a) -> 7x7 weight gradient through the im2col GEMM
  const int h = (t->H + 6 - 7) / 2 + 1, w = (t->W + 6 - 7) / 2 + 1;
  const long long rows0 = (long long)n * h * w;
  void* dz0 = ws.take((size_t)rows0 * 64 * 2);
  void* dy0 = ws.take((size_t)rows0 * 64 * 2);
  void* col = ws.take((size_t)rows0 * 192 * 2);
  float* dw192 = ws.take_n<float>(64 * 192);
  plan.wg_need = std::max(plan.wg_need, ctl_conv2d_wgrad_workspace_bytes(n, h, w, 192, 64, 1, 1));
  if (ws.dry) return 0;
  if ((rc = ctl_maxpool3x3s2_backward_argmax_nhwc_f16(t->arg0, pp[cur], n, h, w, 64, dz0, st))) return rc;
  if ((rc = ctl_bn_train_backward_nhwc_f16(dz0, t->ibn ? t->z0 : nullptr, t->y0, rows0, 64, 64, t->g0, t->m0, t->i0, inv_scale, bn_ws,
                                           bn_ws_bytes, t->ibn ? dz0 : nullptr, t->dg0, t->db0, dy0, st)))
    return rc;
  if ((rc = ctl_stem_im2col_f16(t->x, n, t->H, t->W, col, st))) return rc;
  if ((rc = ctl_conv2d_wgrad_nhwc_f16_ex(col, n, h, w, 192, dy0, 64, 1, 1, wg_ws, wg_ws_bytes, dw192, 1.0f, 0, st))) return rc;
  stem_train_unpack_kernel<<<(64 * 147 + 255) / 256, 256, 0, st>>>(dw192, inv_scale, t->dw0);
  CTL_LAUNCH_CHECK();
  return 0;
}

// workspace = [bn scratch | wgrad scratch | forward arena | backward arena]; the plan is the dry walk of both passes
struct Layout {
  size_t bn_bytes = 0, wg_bytes = 0, total = 0;
};

static int plan_layout(const ctl_trainer* t, int n, int H, int W, Layout* out) {
  // the dry walk runs on a COPY of the handle: it overwrites the per-layer saved pointers and shapes, which a real
  // forward may have left for the backward of the same step
  ctl_trainer tmp = *t;
  tmp.n = n;
  tmp.H = H;
  tmp.W = W;
  Bump dry;
  Plan plan;
  int rc = forward_walk(&tmp, dry, plan, nullptr, 0, nullptr, n, H, W, nullptr, nullptr);
  if (rc) return rc;
  // the backward of a stride-2 layer needs its input map even: the weight gradient (ctl_conv2d_wgrad_nhwc_f16) and the
  // zero-insertion data gradient (ctl_upsample2_zero_nhwc_f16 writes a [2 ho][2 wo] map) both assume it
  for (const TrainBlock& b : tmp.blocks)
    for (const ConvSpec* c : {&b.c1, &b.c2, &b.c3, &b.down})
      if (c->stride == 2 && (c->h % 2 || c->w_in % 2)) {
        set_error("%s: a training step needs an even input map at every stride-2 layer, got %dx%d (input %dx%d)",
                  c->conv.c_str(), c->h, c->w_in, H, W);
        return CTL_ERR_INVALID_ARGUMENT;
      }
  rc = backward_walk(&tmp, dry, plan, nullptr, 0, nullptr, 0, nullptr, 1.f, nullptr);
  if (rc) return rc;
  out->bn_bytes = (plan.bn_need + 255) & ~(size_t)255;
  out->wg_bytes = (plan.wg_need + 255) & ~(size_t)255;
  out->total = out->bn_bytes + out->wg_bytes + dry.high;
  return 0;
}

template <typename T>
static T* t_alloc(ctl_trainer* h, size_t count) {
  void* p = nullptr;
  if (cudaMalloc(&p, count * sizeof(T)) != cudaSuccess) return nullptr;
  h->owned.push_back(p);
  return static_cast<T*>(p);
}

}  // namespace ctl

using namespace ctl;

extern "C" {

int ctl_trainer_create(ctl_trainer** out, int32_t ibn, int32_t last_stride, float momentum) {
  CTL_CHECK_ARG(out != nullptr, "null pointer");
  CTL_CHECK_ARG(last_stride == 1 || last_stride == 2, "last_stride must be 1 or 2 (config/defaults.py:24)");
  CTL_CHECK_ARG(momentum > 0.f && momentum <= 1.f, "momentum must be in (0, 1]");
  ctl_trainer* t = new ctl_trainer();
  t->ibn = ibn ? 1 : 0;
  t->last_stride = last_stride;
  t->momentum = momentum;
  const int planes[4] = {64, 128, 256, 512}, nblk[4] = {3, 4, 6, 3};
  int inplanes = 64;
  for (int li = 0; li < 4; ++li)
    for (int bi = 0; bi < nblk[li]; ++bi) {
      TrainBlock b;
      const std::string p = "layer" + std::to_string(li + 1) + "." + std::to_string(bi);
      const int stride0 = li == 0 ? 1 : (li == 3 ? last_stride : 2);
      b.c1.conv = p + ".conv1";
      b.c1.bn = p + ".bn1";
      b.c1.cin = inplanes;
      b.c1.cout = planes[li];
      b.c1.in_half = (t->ibn && planes[li] != 512) ? planes[li] / 2 : 0;  // resnet_ibn_a.py:116-119
      b.c2.conv = p + ".conv2";
      b.c2.bn = p + ".bn2";
      b.c2.cin = b.c2.cout = planes[li];
      b.c2.k = 3;
      b.c2.stride = bi == 0 ? stride0 : 1;
      b.c3.conv = p + ".conv3";
      b.c3.bn = p + ".bn3";
      b.c3.cin = planes[li];
      b.c3.cout = planes[li] * 4;
      b.has_down = bi == 0;
      if (b.has_down) {
        b.down.conv = p + ".downsample.0";
        b.down.bn = p + ".downsample.1";
        b.down.cin = inplanes;
        b.down.cout = planes[li] * 4;
        b.down.stride = b.c2.stride;
        b.down.relu = 0;
      }
      inplanes = planes[li] * 4;
      t->blocks.push_back(b);
    }
  *out = t;
  return 0;
}

void ctl_trainer_destroy(ctl_trainer* t) {
  if (!t) return;
  for (void* p : t->owned) cudaFree(p);
  delete t;
}

int ctl_trainer_bind(ctl_trainer* t, const ctl_named_tensor* params, int32_t n_params, const ctl_named_buffer* grads, int32_t n_grads) {
  CTL_CHECK_ARG(t && params && grads && n_params > 0 && n_grads > 0, "bad arguments");
  int rc = ctl_device_check();
  if (rc) return rc;
  RefMap p, g;
  for (int i = 0; i < n_params; ++i) {
    CTL_CHECK_ARG(params[i].name != nullptr, "parameter %d has no name", i);
    p[params[i].name] = Ref{const_cast<float*>(params[i].data), (long long)params[i].numel};
  }
  for (int i = 0; i < n_grads; ++i) {
    CTL_CHECK_ARG(grads[i].name != nullptr, "gradient %d has no name", i);
    g[grads[i].name] = Ref{grads[i].data, (long long)grads[i].numel};
  }
  t->bound = false;
  t->forwarded = false;
  t->w0 = lookup(p, "conv1.weight", 64 * 147, true, "parameter", &rc);
  t->g0 = lookup(p, "bn1.weight", 64, true, "parameter", &rc);
  t->b0 = lookup(p, "bn1.bias", 64, true, "parameter", &rc);
  t->rm0 = lookup(p, "bn1.running_mean", 64, false, "buffer", &rc);
  t->rv0 = lookup(p, "bn1.running_var", 64, false, "buffer", &rc);
  t->dw0 = lookup(g, "conv1.weight", 64 * 147, true, "gradient", &rc);
  t->dg0 = lookup(g, "bn1.weight", 64, true, "gradient", &rc);
  t->db0 = lookup(g, "bn1.bias", 64, true, "gradient", &rc);
  if (rc) return rc;
  CTL_CHECK_ARG((t->rm0 == nullptr) == (t->rv0 == nullptr), "bn1 needs running_mean and running_var together (or neither)");
  size_t total = 0;
  int n_convs = 0;
  for (TrainBlock& b : t->blocks) {
    ConvSpec* cs[4] = {&b.c1, &b.c2, &b.c3, b.has_down ? &b.down : nullptr};
    for (ConvSpec* c : cs) {
      if (!c) continue;
      if ((rc = bind_conv(*c, p, g))) return rc;
      total += (size_t)c->cout * c->cin * c->k * c->k;
      ++n_convs;
    }
  }
  // packed fp16 operands: [forward arena | data-gradient arena], refreshed by ctl_train_pack_weights every forward
  if (!t->arena) {
    t->arena = t_alloc<__half>(t, 2 * total);
    t->table = t_alloc<long long>(t, (size_t)n_convs * 6);
    t->stem_w192 = t_alloc<__half>(t, 64 * 192);
    t->zero_bias = t_alloc<float>(t, 2048);
    if (!t->arena || !t->table || !t->stem_w192 || !t->zero_bias) {
      set_error("ctl_trainer_bind: out of device memory");
      return (int)cudaErrorMemoryAllocation;
    }
    CTL_CUDA(cudaMemset(t->zero_bias, 0, 2048 * sizeof(float)));
  }
  std::vector<long long> rows;
  rows.reserve((size_t)n_convs * 6);
  size_t off = 0;
  long long chunks = 0;
  for (TrainBlock& b : t->blocks) {
    // table order == engine_train.py's (state_dict order: conv1, conv2, conv3, downsample.0)
    ConvSpec* cs[4] = {&b.c1, &b.c2, &b.c3, b.has_down ? &b.down : nullptr};
    for (ConvSpec* c : cs) {
      if (!c) continue;
      const size_t numel = (size_t)c->cout * c->cin * c->k * c->k;
      c->wf = t->arena + off;
      c->wd = t->arena + total + off;
      rows.push_back((long long)reinterpret_cast<uintptr_t>(c->w));
      rows.push_back((long long)reinterpret_cast<uintptr_t>(c->wf));
      rows.push_back((long long)reinterpret_cast<uintptr_t>(c->wd));
      rows.push_back((long long)c->cout | ((long long)c->cin << 32));
      rows.push_back((long long)c->k);
      rows.push_back(chunks);
      chunks += (long long)((numel + TT_PACK_CHUNK - 1) / TT_PACK_CHUNK);
      off += numel;
    }
  }
  CTL_CUDA(cudaMemcpy(t->table, rows.data(), rows.size() * sizeof(long long), cudaMemcpyHostToDevice));
  t->n_packed = n_convs;
  t->n_chunks = chunks;
  t->bound = true;
  return 0;
}

size_t ctl_train_workspace_bytes(const ctl_trainer* t, int32_t n, int32_t height, int32_t width) {
  if (!t || n < 1 || height < 32 || width < 32) {
    set_error("ctl_train_workspace_bytes: bad arguments (n=%d, %dx%d; n >= 1 and sides >= 32 needed)", n, height, width);
    return 0;
  }
  Layout l;
  if (plan_layout(t, n, height, width, &l)) return 0;
  return l.total;
}

int ctl_train_forward(ctl_trainer* t, const float* x_nchw, int32_t n, int32_t height, int32_t width, float* out_feat, void* workspace,
                      size_t workspace_bytes, ctl_stream_t stream) {
  CTL_CHECK_ARG(t && x_nchw && out_feat && workspace, "null pointer");
  CTL_CHECK_ARG(t->bound, "ctl_trainer_bind has not been called on this handle");
  CTL_CHECK_ARG(n >= 1 && height >= 32 && width >= 32, "bad input shape");
  CTL_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255u) == 0, "workspace must be 256-byte aligned");
  Layout l;
  int rc = plan_layout(t, n, height, width, &l);
  if (rc) return rc;
  if (workspace_bytes < l.total) {
    set_error("workspace too small: need %zu bytes, have %zu", l.total, workspace_bytes);
    return CTL_ERR_WORKSPACE;
  }
  if ((rc = ctl_device_check())) return rc;
  char* base = static_cast<char*>(workspace);
  Bump ws;
  ws.base = base + l.bn_bytes + l.wg_bytes;
  ws.cap = l.total - l.bn_bytes - l.wg_bytes;
  ws.dry = false;
  Plan plan;
  t->forwarded = false;
  t->x = x_nchw;
  t->n = n;
  t->H = height;
  t->W = width;
  rc = forward_walk(t, ws, plan, base, l.bn_bytes, x_nchw, n, height, width, out_feat, (cudaStream_t)stream);
  if (rc) return rc;
  t->fwd_mark = ws.off;
  t->lay_bn = l.bn_bytes;
  t->lay_wg = l.wg_bytes;
  t->lay_total = l.total;
  t->fwd_workspace = workspace;
  t->forwarded = true;
  return 0;
}

int ctl_train_backward(ctl_trainer* t, const float* dfeat, float grad_scale, void* workspace, size_t workspace_bytes, ctl_stream_t stream) {
  CTL_CHECK_ARG(t && dfeat && workspace, "null pointer");
  CTL_CHECK_ARG(t->forwarded, "ctl_train_backward needs the ctl_train_forward of the same step (same workspace, same input)");
  CTL_CHECK_ARG(grad_scale > 0.f, "grad_scale must be positive");
  CTL_CHECK_ARG(workspace == t->fwd_workspace && workspace_bytes >= t->lay_total,
                "ctl_train_backward must get the workspace of the forward (it holds the saved activations)");
  int rc = ctl_device_check();
  if (rc) return rc;
  char* base = static_cast<char*>(workspace);
  Bump ws;
  ws.base = base + t->lay_bn + t->lay_wg;
  ws.cap = t->lay_total - t->lay_bn - t->lay_wg;
  ws.off = ws.high = t->fwd_mark;
  ws.dry = false;
  Plan plan;
  t->forwarded = false;  // dz buffers are consumed in place: one backward per forward
  return backward_walk(t, ws, plan, base, t->lay_bn, base + t->lay_bn, t->lay_wg, dfeat, grad_scale, (cudaStream_t)stream);
}

}  // extern "C"
