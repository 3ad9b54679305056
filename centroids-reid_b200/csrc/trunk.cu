// Whole-trunk entry points of the C ABI (SURVEY 8b: ctl_weights_pack + ctl_embed_forward): the layer graph of the eval
// embedding path -- ResNet.forward / ResNet_IBN.forward (modelling/backbones/resnet.py:122-133, resnet_ibn_a.py:126-141),
// Baseline.forward's global average pool (modelling/baseline.py:91-96) and the eval BatchNorm1d of
// ModelBase.validation_step (modelling/bases.py:169-177) -- behind an opaque handle, so that a host that is not Python can
// run `bn(backbone(x))` without re-implementing modelling/backbones/engine.py.
//
// The handle owns the PACKED operands: [Cout][kh][kw][Cin] fp16 weights with the eval BatchNorm folded in and fp32
// biases, produced on the device from the reference's fp32 state_dict tensors (fold_pack_kernel: exactly the arithmetic
// of engine.py::_fold, operation by operation, so both paths produce the same bits), the K-concatenated [W3 | Wd]
// matrices of every first block, the two stem layouts, and the zero-bordered staging buffer of the fused stem.
// Activations live in a caller-provided workspace.  The launches are the same C entry points engine.py calls.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.h"
#include "umma.cuh"

namespace ctl {

static constexpr float TRUNK_BN_EPS = 1e-5f;

// w [cout][cin][k][k] fp32 (+ BatchNorm gamma/beta/mean/var of `nbn` channels starting at channel c0; nullptr = no fold)
//   -> out [cout][k][k][cin] fp16 rows of pitch `pitch` elements at column offset `col0`;
//   bias[c] (= beta - mean * scale) written, or ADDED when `accumulate` (the [W3 | Wd] pair shares one bias vector).
__global__ void fold_pack_kernel(const float* __restrict__ w, int cout, int cin, int k, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, const float* __restrict__ mean,
                                 const float* __restrict__ var, int c0, __half* __restrict__ out, long long pitch, int col0,
                                 float* __restrict__ bias, int accumulate) {
  const int co = blockIdx.x;
  float scale = 1.f, b = 0.f;
  if (gamma != nullptr && co >= c0) {
    const int j = co - c0;
    scale = __fdiv_rn(gamma[j], __fsqrt_rn(__fadd_rn(var[j], TRUNK_BN_EPS)));
    b = __fsub_rn(beta[j], __fmul_rn(mean[j], scale));
  }
  const int kk = k * k;
  for (int i = threadIdx.x; i < cin * kk; i += blockDim.x) {
    const int ci = i % cin, rs = i / cin;  // output order (r, s, ci)
    const float v = w[((size_t)co * cin + ci) * kk + rs];
    out[(size_t)co * pitch + col0 + (size_t)rs * cin + ci] = __float2half_rn(__fmul_rn(v, scale));
  }
  if (threadIdx.x == 0 && bias != nullptr) bias[co] = accumulate ? __fadd_rn(bias[co], b) : b;
}

// stem layouts from the folded [64][3][7][7] weights (engine.py: stem_w = [64][192], k = (c*7 + r)*8 + s, s = 7 and
// k >= 168 zero;  pack_stem_fused = [28][64][8], chunk = r*4 + s/2, element = (s%2)*4 + ch, ch == 3 and s == 7 zero)
__global__ void stem_pack_kernel(const float* __restrict__ w, const float* __restrict__ gamma, const float* __restrict__ beta,
                                 const float* __restrict__ mean, const float* __restrict__ var, __half* __restrict__ w192,
                                 __half* __restrict__ w3, float* __restrict__ bias) {
  const int o = blockIdx.x;
  const float scale = __fdiv_rn(gamma[o], __fsqrt_rn(__fadd_rn(var[o], TRUNK_BN_EPS)));
  if (threadIdx.x == 0) bias[o] = __fsub_rn(beta[o], __fmul_rn(mean[o], scale));
  for (int i = threadIdx.x; i < 192; i += blockDim.x) {
    float v = 0.f;
    if (i < 168) {
      const int cr = i / 8, s = i % 8;
      if (s < 7) v = __fmul_rn(w[(size_t)o * 147 + cr * 7 + s], scale);
    }
    w192[(size_t)o * 192 + i] = __float2half_rn(v);
  }
  for (int i = threadIdx.x; i < 28 * 8; i += blockDim.x) {
    const int chunk = i / 8, e = i % 8, r = chunk / 4, s = (chunk % 4) * 2 + e / 4, ch = e % 4;
    float v = 0.f;
    if (s < 7 && ch < 3) v = __fmul_rn(w[(size_t)o * 147 + (ch * 7 + r) * 7 + s], scale);
    w3[((size_t)chunk * 64 + o) * 8 + e] = __float2half_rn(v);
  }
}

__global__ void head_pack_kernel(const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                                 const float* __restrict__ var, int n, float* __restrict__ scale, float* __restrict__ shift) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = __fdiv_rn(gamma[i], __fsqrt_rn(__fadd_rn(var[i], TRUNK_BN_EPS)));
  scale[i] = s;
  shift[i] = __fsub_rn(beta[i], __fmul_rn(mean[i], s));
}

struct PackedConv {
  __half* w = nullptr;
  float* b = nullptr;
  int cin = 0, cout = 0, k = 1, stride = 1, relu = 1, relu_from = 0;
};
struct TrunkBlock {
  PackedConv c1, c2, c3, down;
  bool has_down = false, has_in = false;
  int in_half = 0;
  float *in_gamma = nullptr, *in_beta = nullptr;
  __half* dual_w = nullptr;
  float* dual_b = nullptr;
};

}  // namespace ctl

struct ctl_trunk {
  int ibn = 0, last_stride = 1;
  bool packed = false, has_head = false;
  std::vector<ctl::TrunkBlock> blocks;
  __half *stem_w192 = nullptr, *stem_w3 = nullptr;
  float* stem_b = nullptr;
  float *head_scale = nullptr, *head_shift = nullptr;
  void* stem_pad = nullptr;
  size_t stem_pad_bytes = 0;
  int pad_n = 0, pad_h = 0, pad_w = 0;
  std::vector<void*> owned;  // every cudaMalloc of this handle
};

namespace ctl {

template <typename T>
static T* dev_alloc(ctl_trunk* h, size_t count) {
  void* p = nullptr;
  if (cudaMalloc(&p, count * sizeof(T)) != cudaSuccess) return nullptr;
  h->owned.push_back(p);
  return static_cast<T*>(p);
}

struct TensorRef {
  const float* data;
  long long numel;
};
using TensorMap = std::unordered_map<std::string, TensorRef>;

static const float* need(const TensorMap& m, const std::string& name, long long numel, int* rc) {
  auto it = m.find(name);
  if (it == m.end() || it->second.data == nullptr) {
    set_error("ctl_weights_pack: tensor '%s' is missing", name.c_str());
    *rc = CTL_ERR_INVALID_ARGUMENT;
    return nullptr;
  }
  if (it->second.numel != numel) {
    set_error("ctl_weights_pack: tensor '%s' has %lld elements, expected %lld", name.c_str(), it->second.numel, numel);
    *rc = CTL_ERR_INVALID_ARGUMENT;
    return nullptr;
  }
  return it->second.data;
}

// packs conv `conv` with BatchNorm `bn` (bn empty: raw weights); ibn_half > 0: BN folds channels [ibn_half, cout) only
static int pack_conv(ctl_trunk* h, const TensorMap& m, const std::string& conv, const std::string& bn, int cout, int cin, int k,
                     int ibn_half, PackedConv* out, cudaStream_t st) {
  int rc = 0;
  const float* w = need(m, conv + ".weight", (long long)cout * cin * k * k, &rc);
  if (rc) return rc;
  const int nbn = cout - ibn_half;
  const float *g = need(m, bn + ".weight", nbn, &rc), *b = need(m, bn + ".bias", nbn, &rc),
              *mu = need(m, bn + ".running_mean", nbn, &rc), *va = need(m, bn + ".running_var", nbn, &rc);
  if (rc) return rc;
  if (!out->w) out->w = dev_alloc<__half>(h, (size_t)cout * cin * k * k);
  if (!out->b) out->b = dev_alloc<float>(h, cout);
  if (!out->w || !out->b) {
    set_error("ctl_weights_pack: out of device memory");
    return (int)cudaErrorMemoryAllocation;
  }
  out->cin = cin;
  out->cout = cout;
  out->k = k;
  fold_pack_kernel<<<cout, 256, 0, st>>>(w, cout, cin, k, g, b, mu, va, ibn_half, out->w, (long long)cin * k * k, 0, out->b, 0);
  CTL_LAUNCH_CHECK();
  return 0;
}

}  // namespace ctl

using namespace ctl;

extern "C" {

int ctl_trunk_create(ctl_trunk** out, int32_t ibn, int32_t last_stride) {
  CTL_CHECK_ARG(out != nullptr, "null pointer");
  CTL_CHECK_ARG(last_stride == 1 || last_stride == 2, "last_stride must be 1 or 2 (config/defaults.py:24)");
  ctl_trunk* h = new ctl_trunk();
  h->ibn = ibn ? 1 : 0;
  h->last_stride = last_stride;
  const int planes[4] = {64, 128, 256, 512}, nblk[4] = {3, 4, 6, 3};
  int inplanes = 64;
  for (int li = 0; li < 4; ++li)
    for (int bi = 0; bi < nblk[li]; ++bi) {
      TrunkBlock blk;
      const int stride0 = li == 0 ? 1 : (li == 3 ? last_stride : 2);
      blk.c1.cin = inplanes;
      blk.c1.cout = planes[li];
      blk.c2.cin = blk.c2.cout = planes[li];
      blk.c2.k = 3;
      blk.c2.stride = bi == 0 ? stride0 : 1;
      blk.c3.cin = planes[li];
      blk.c3.cout = planes[li] * 4;
      blk.has_down = bi == 0;
      if (blk.has_down) {
        blk.down.cin = inplanes;
        blk.down.cout = planes[li] * 4;
        blk.down.stride = blk.c2.stride;
        blk.down.relu = 0;
        inplanes = planes[li] * 4;
      }
      blk.has_in = h->ibn && planes[li] != 512;  // resnet_ibn_a.py:116-119
      blk.in_half = blk.has_in ? planes[li] / 2 : 0;
      h->blocks.push_back(blk);
    }
  *out = h;
  return 0;
}

void ctl_trunk_destroy(ctl_trunk* h) {
  if (!h) return;
  for (void* p : h->owned) cudaFree(p);
  if (h->stem_pad) cudaFree(h->stem_pad);
  delete h;
}

int ctl_weights_pack(ctl_trunk* h, const ctl_named_tensor* tensors, int32_t n_tensors, ctl_stream_t stream) {
  CTL_CHECK_ARG(h && tensors && n_tensors > 0, "bad arguments");
  int rc = ctl_device_check();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  TensorMap m;
  for (int i = 0; i < n_tensors; ++i) {
    CTL_CHECK_ARG(tensors[i].name != nullptr, "tensor %d has no name", i);
    m[tensors[i].name] = TensorRef{tensors[i].data, (long long)tensors[i].numel};
  }
  // ---- stem ----
  {
    const float* w = need(m, "conv1.weight", 64 * 147, &rc);
    const float *g = need(m, "bn1.weight", 64, &rc), *b = need(m, "bn1.bias", 64, &rc), *mu = need(m, "bn1.running_mean", 64, &rc),
                *va = need(m, "bn1.running_var", 64, &rc);
    if (rc) return rc;
    if (!h->stem_w192) {
      h->stem_w192 = dev_alloc<__half>(h, 64 * 192);
      h->stem_w3 = dev_alloc<__half>(h, 28 * 64 * 8);
      h->stem_b = dev_alloc<float>(h, 64);
    }
    if (!h->stem_w192 || !h->stem_w3 || !h->stem_b) {
      set_error("ctl_weights_pack: out of device memory");
      return (int)cudaErrorMemoryAllocation;
    }
    stem_pack_kernel<<<64, 128, 0, st>>>(w, g, b, mu, va, h->stem_w192, h->stem_w3, h->stem_b);
    CTL_LAUNCH_CHECK();
  }
  // ---- bottlenecks ----
  const int nblk[4] = {3, 4, 6, 3};
  size_t idx = 0;
  for (int li = 0; li < 4; ++li)
    for (int bi = 0; bi < nblk[li]; ++bi, ++idx) {
      TrunkBlock& blk = h->blocks[idx];
      const std::string p = "layer" + std::to_string(li + 1) + "." + std::to_string(bi);
      if (blk.has_in) {
        // IBN: channels [0, half) keep the raw convolution (InstanceNorm + ReLU follow as their own kernel), the
        // BatchNorm half is folded; ReLU in the conv epilogue only from channel `half` on
        if ((rc = pack_conv(h, m, p + ".conv1", p + ".bn1.BN", blk.c1.cout, blk.c1.cin, 1, blk.in_half, &blk.c1, st))) return rc;
        blk.c1.relu_from = blk.in_half;
        const float *ig = need(m, p + ".bn1.IN.weight", blk.in_half, &rc), *ib = need(m, p + ".bn1.IN.bias", blk.in_half, &rc);
        if (rc) return rc;
        if (!blk.in_gamma) {
          blk.in_gamma = dev_alloc<float>(h, blk.in_half);
          blk.in_beta = dev_alloc<float>(h, blk.in_half);
        }
        CTL_CUDA(cudaMemcpyAsync(blk.in_gamma, ig, blk.in_half * sizeof(float), cudaMemcpyDeviceToDevice, st));
        CTL_CUDA(cudaMemcpyAsync(blk.in_beta, ib, blk.in_half * sizeof(float), cudaMemcpyDeviceToDevice, st));
      } else {
        if ((rc = pack_conv(h, m, p + ".conv1", p + ".bn1", blk.c1.cout, blk.c1.cin, 1, 0, &blk.c1, st))) return rc;
      }
      const int s2 = blk.c2.stride;
      if ((rc = pack_conv(h, m, p + ".conv2", p + ".bn2", blk.c2.cout, blk.c2.cin, 3, 0, &blk.c2, st))) return rc;
      blk.c2.stride = s2;
      if ((rc = pack_conv(h, m, p + ".conv3", p + ".bn3", blk.c3.cout, blk.c3.cin, 1, 0, &blk.c3, st))) return rc;
      if (blk.has_down) {
        const int sd = blk.down.stride;
        if ((rc = pack_conv(h, m, p + ".downsample.0", p + ".downsample.1", blk.down.cout, blk.down.cin, 1, 0, &blk.down, st))) return rc;
        blk.down.stride = sd;
        blk.down.relu = 0;
        // [W3 | Wd] and bias3 + bias_d for the single-GEMM form of conv3 + shortcut (ctl_conv1x1_dual_nhwc_f16)
        const int kt = blk.c3.cin + blk.down.cin;
        if (!blk.dual_w) {
          blk.dual_w = dev_alloc<__half>(h, (size_t)blk.c3.cout * kt);
          blk.dual_b = dev_alloc<float>(h, blk.c3.cout);
        }
        if (!blk.dual_w || !blk.dual_b) {
          set_error("ctl_weights_pack: out of device memory");
          return (int)cudaErrorMemoryAllocation;
        }
        CTL_CUDA(cudaMemcpy2DAsync(blk.dual_w, (size_t)kt * 2, blk.c3.w, (size_t)blk.c3.cin * 2, (size_t)blk.c3.cin * 2, blk.c3.cout,
                                   cudaMemcpyDeviceToDevice, st));
        CTL_CUDA(cudaMemcpy2DAsync(blk.dual_w + blk.c3.cin, (size_t)kt * 2, blk.down.w, (size_t)blk.down.cin * 2,
                                   (size_t)blk.down.cin * 2, blk.c3.cout, cudaMemcpyDeviceToDevice, st));
        // bias3 + bias_d in fp32, like engine.py (c3.b + cd.b)
        CTL_CUDA(cudaMemcpyAsync(blk.dual_b, blk.c3.b, blk.c3.cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
        const std::string d = p + ".downsample.1";
        int rc2 = 0;
        fold_pack_kernel<<<blk.c3.cout, 32, 0, st>>>(need(m, p + ".downsample.0.weight", (long long)blk.down.cout * blk.down.cin, &rc2), blk.down.cout, 0, 1,
                                                     need(m, d + ".weight", blk.down.cout, &rc2), need(m, d + ".bias", blk.down.cout, &rc2),
                                                     need(m, d + ".running_mean", blk.down.cout, &rc2),
                                                     need(m, d + ".running_var", blk.down.cout, &rc2), 0, blk.down.w, 0, 0, blk.dual_b, 1);
        CTL_LAUNCH_CHECK();
        if (rc2) return rc2;
      }
    }
  // ---- optional BatchNorm1d head (ModelBase.bn, modelling/bases.py:83) ----
  h->has_head = m.count("bn_head.weight") != 0;
  if (h->has_head) {
    const float *g = need(m, "bn_head.weight", 2048, &rc), *b = need(m, "bn_head.bias", 2048, &rc),
                *mu = need(m, "bn_head.running_mean", 2048, &rc), *va = need(m, "bn_head.running_var", 2048, &rc);
    if (rc) return rc;
    if (!h->head_scale) {
      h->head_scale = dev_alloc<float>(h, 2048);
      h->head_shift = dev_alloc<float>(h, 2048);
    }
    head_pack_kernel<<<8, 256, 0, st>>>(g, b, mu, va, 2048, h->head_scale, h->head_shift);
    CTL_LAUNCH_CHECK();
  }
  h->packed = true;
  return 0;
}

// Bytes of one of the five activation buffers of ctl_embed_forward: the largest activation of the trunk, found by a dry
// walk of the layer shapes with the forward's own ceil formulas.  With even sides that is the stem's conv output
// [n, H/2, W/2, 64] (== layer1's output [n, H/4, W/4, 256]).  When the stem output has an odd side the max-pool rounds
// up and layer1's output is the larger one; at tiny inputs (8x8) a 1-pixel map of 1024 or 2048 channels is.
static size_t trunk_act_bytes(const ctl_trunk* h, int n, int hgt, int wid) {
  int hh = (hgt + 6 - 7) / 2 + 1, ww = (wid + 6 - 7) / 2 + 1;
  size_t px_ch = (size_t)hh * ww * 64;  // stem conv output
  hh = (hh + 2 - 3) / 2 + 1;
  ww = (ww + 2 - 3) / 2 + 1;
  for (const TrunkBlock& blk : h->blocks) {
    const int s = blk.c2.stride;
    const int h2 = (hh + 2 - 3) / s + 1, w2 = (ww + 2 - 3) / s + 1;
    px_ch = std::max(px_ch, (size_t)hh * ww * blk.c1.cout);
    px_ch = std::max(px_ch, (size_t)h2 * w2 * std::max(blk.c2.cout, blk.c3.cout));
    if (blk.has_down) px_ch = std::max(px_ch, (size_t)h2 * w2 * blk.down.cout);
    hh = h2;
    ww = w2;
  }
  return ((size_t)n * px_ch * 2 + 255) & ~(size_t)255;
}

size_t ctl_embed_workspace_bytes(const ctl_trunk* h, int32_t n, int32_t hgt, int32_t wid) {
  if (!h || n < 1 || hgt < 8 || wid < 8) return 0;
  return 5 * trunk_act_bytes(h, n, hgt, wid);
}

static int run_conv(const PackedConv& c, const void* x, int n, int hh, int ww, const void* residual, void* out, cudaStream_t st) {
  return ctl_conv2d_nhwc_f16(x, n, hh, ww, c.cin, c.w, c.b, residual, out, c.cout, c.k, c.stride, c.relu, c.relu_from, st);
}

int ctl_embed_forward(ctl_trunk* h, const float* x_nchw, int32_t n, int32_t hgt, int32_t wid, float* out_feat, float* out_emb,
                      void* workspace, size_t workspace_bytes, ctl_stream_t stream) {
  CTL_CHECK_ARG(h && x_nchw && workspace && (out_feat || out_emb), "null pointer");
  CTL_CHECK_ARG(h->packed, "ctl_weights_pack has not been called on this handle");
  CTL_CHECK_ARG(n >= 1 && hgt >= 8 && wid >= 8, "bad input shape");
  CTL_CHECK_ARG(out_emb == nullptr || h->has_head, "out_emb needs the bn_head.* tensors in ctl_weights_pack");
  const size_t act = trunk_act_bytes(h, n, hgt, wid);
  if (workspace_bytes < 5 * act) {
    set_error("workspace too small: need %zu bytes, have %zu", 5 * act, workspace_bytes);
    return CTL_ERR_WORKSPACE;
  }
  int rc = ctl_device_check();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = static_cast<char*>(workspace);
  void* buf[5] = {ws, ws + act, ws + 2 * act, ws + 3 * act, ws + 4 * act};
  int hh = (hgt + 6 - 7) / 2 + 1, ww = (wid + 6 - 7) / 2 + 1;
  const int hp = (hh + 2 - 3) / 2 + 1, wp = (ww + 2 - 3) / 2 + 1;
  void* a = buf[0];
  if (hgt % 4 == 0 && wid % 2 == 0 && wid <= 128) {
    if (h->pad_n != n || h->pad_h != hgt || h->pad_w != wid) {
      if (h->stem_pad) CTL_CUDA(cudaFree(h->stem_pad));
      h->stem_pad = nullptr;
      h->stem_pad_bytes = ctl_stem_pad_bytes(n, hgt, wid);
      CTL_CUDA(cudaMalloc(&h->stem_pad, h->stem_pad_bytes));
      CTL_CUDA(cudaMemsetAsync(h->stem_pad, 0, h->stem_pad_bytes, st));  // the zero border is written once
      h->pad_n = n;
      h->pad_h = hgt;
      h->pad_w = wid;
    }
    if ((rc = ctl_stem_pool_fused(x_nchw, n, hgt, wid, h->stem_pad, h->stem_w3, h->stem_b, h->ibn, a, st))) return rc;
  } else {
    if ((rc = ctl_stem_conv7x7_tc(x_nchw, n, hgt, wid, h->stem_w192, h->stem_b, h->ibn, buf[1], st))) return rc;
    if ((rc = ctl_maxpool3x3s2_nhwc_f16(buf[1], n, hh, ww, 64, a, st))) return rc;
  }
  hh = hp;
  ww = wp;
  int cur = 0;  // index of the buffer holding the block input
  for (const TrunkBlock& blk : h->blocks) {
    void* o1 = buf[(cur + 1) % 5];
    void* o2 = buf[(cur + 2) % 5];
    void* res = buf[(cur + 3) % 5];
    void* out = buf[(cur + 4) % 5];
    if ((rc = run_conv(blk.c1, a, n, hh, ww, nullptr, o1, st))) return rc;
    if (blk.has_in)
      if ((rc = ctl_instnorm_relu_nhwc_f16(o1, n, hh * ww, blk.c1.cout, blk.in_half, blk.in_gamma, blk.in_beta, TRUNK_BN_EPS, st)))
        return rc;
    const int s = blk.c2.stride;
    const int h2 = (hh + 2 - 3) / s + 1, w2 = (ww + 2 - 3) / s + 1;
    if ((rc = run_conv(blk.c2, o1, n, hh, ww, nullptr, o2, st))) return rc;
    if (blk.has_down && hh % s == 0 && ww % s == 0) {
      if ((rc = ctl_conv1x1_dual_nhwc_f16(o2, blk.c3.cin, a, hh, ww, blk.down.cin, s, n, blk.dual_w, blk.dual_b, out, blk.c3.cout, 1, st)))
        return rc;
    } else {
      const void* r = a;
      if (blk.has_down) {
        if ((rc = run_conv(blk.down, a, n, hh, ww, nullptr, res, st))) return rc;
        r = res;
      }
      if ((rc = run_conv(blk.c3, o2, n, h2, w2, r, out, st))) return rc;
    }
    a = out;
    cur = (cur + 4) % 5;
    hh = h2;
    ww = w2;
  }
  return ctl_gap_bn_nhwc_f16(a, n, hh * ww, 2048, out_emb ? h->head_scale : nullptr, out_emb ? h->head_shift : nullptr, out_feat,
                             out_emb, st);
}

}  // extern "C"
