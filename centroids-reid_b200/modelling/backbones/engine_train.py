"""Train-mode ResNet-50 trunk on the B200 kernels: forward with batch-statistics BatchNorm and the full backward
(what autograd does through modelling/backbones/resnet.py:67-87,122-133 + baseline.py:91-96 in the reference).

Per conv+BN of the forward:   conv (tcgen05 implicit GEMM, raw fp16 output y)  ->  batch statistics  ->
z = [relu](gamma * xhat + beta [+ shortcut])  (fp16).  The backward walks the blocks in reverse:
BN/ReLU backward (masked grad g, dgamma, dbeta, dy), weight gradient (tcgen05 GEMM over the pixel dimension),
data gradient = the forward conv kernel on dy with the transposed / flipped weights (stride-2 layers through
zero-insertion upsampling), shortcut gradients folded into conv1's data gradient through the kernel's residual
input.  Activations and activation gradients are fp16, every reduction and all parameter gradients fp32.

Gradients are computed on `grad_scale * dfeat` (a fixed loss scale against fp16 underflow, the role of the AMP
GradScaler in the reference's PL trainer) and un-scaled in fp32.  `ibn=True` runs the IBN-a variant
(resnet_ibn_a.py): ReLU after the stem, and bn1 of layer1-3 = InstanceNorm on the first half of the channels
(per-image statistics) + batch-statistics BatchNorm on the rest, both through channel-slice (row pitch) kernels.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch

from ... import _native as N

BN_EPS = 1e-5
R50_LAYERS = (3, 4, 6, 3)


class _Saved:
    __slots__ = ("a", "y", "z", "mean", "invstd", "shape_in", "shape_out", "conv", "bn", "k", "stride", "relu", "ibn")


class TrunkTrainer:
    """`params`: name -> tensor with the reference's `base.*`-stripped names (conv weights [Cout, Cin, k, k], BN
    weight / bias fp32 on the device; BN running_mean / running_var are updated in place)."""

    def __init__(self, device, last_stride: int = 1, layers=R50_LAYERS, grad_scale: float = 1024.0,
                 momentum: float = 0.1, graphs: bool = False, ibn: bool = False):
        self.device = torch.device(device)
        self.ibn = ibn  # resnet_ibn_a.py: ReLU after the stem, IBN (InstanceNorm half + BatchNorm half) as bn1 of layer1-3
        self.last_stride, self.layers, self.grad_scale, self.momentum = last_stride, layers, float(grad_scale), momentum
        self._zero_bias = torch.zeros(2048, device=self.device)
        self._ws_bn = None
        self._ws_wg = None
        self.saved: List[_Saved] = []
        self.launches = 0
        # graphs=True: forward and backward are captured once per (input shape, parameter storage) into two CUDA
        # graphs and replayed (the ~540 launches and ~300 torch glue ops of a step cost more CPU time than the GPU
        # needs to run them); the stored activations live in the graphs' private pool
        self.graphs = graphs
        self._graph = None

    # ---------------------------------------------------------------- helpers
    def _bn_ws(self, rows, c):
        need = N.lib().ctl_bn_workspace_bytes(rows, c)
        if self._ws_bn is None or self._ws_bn.numel() < need:
            self._ws_bn = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws_bn

    def _conv(self, a, n, h, w, wf, cout, k, stride, residual=None):
        cin = a.shape[-1]
        pad = 1 if k == 3 else 0
        ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
        out = torch.empty(n, ho, wo, cout, dtype=torch.float16, device=self.device)
        N.check(N.lib().ctl_conv2d_nhwc_f16(a.data_ptr(), n, h, w, cin, wf.data_ptr(), self._zero_bias.data_ptr(),
                                            N.ptr(residual), out.data_ptr(), cout, k, stride, 0, 0, N.stream_ptr()))
        self.launches += 1
        return out, ho, wo

    def _pack_weights(self, params):
        """Forward ([Cout][k][k][Cin]) and data-gradient ([Cin][k][k][Cout], flipped taps) fp16 operands of EVERY
        bottleneck convolution in ONE launch (ctl_train_pack_weights) -- round 1 ran a permute / contiguous / half (/ flip)
        chain of torch kernels per layer and direction, ~1 ms of launch-bound glue per step."""
        import numpy as np

        names = [k[:-7] for k in params if k.endswith(".weight") and params[k].dim() == 4 and k != "conv1.weight"]
        key = tuple((nm, params[nm + ".weight"].data_ptr()) for nm in names)
        if getattr(self, "_pack_key", None) != key:
            total = sum(params[nm + ".weight"].numel() for nm in names)
            arena = torch.empty(2 * total, dtype=torch.float16, device=self.device)
            rows, off, chunks, packs = [], 0, 0, {}
            for nm in names:
                wt = params[nm + ".weight"]
                if wt.dtype != torch.float32 or not wt.is_contiguous():
                    raise TypeError(f"{nm}.weight must be a contiguous fp32 tensor")
                cout, cin, k, _ = wt.shape
                fwd, dgr = arena[off:off + wt.numel()], arena[total + off:total + off + wt.numel()]
                packs[nm] = (fwd, dgr)
                rows.append([wt.data_ptr(), fwd.data_ptr(), dgr.data_ptr(), cout | (cin << 32), k, chunks])
                chunks += (wt.numel() + 8191) // 8192
                off += wt.numel()
            self._pack_table = torch.from_numpy(np.asarray(rows, dtype=np.int64)).to(self.device)
            self._pack_meta, self._pack_arena, self._packs, self._pack_key = (len(rows), chunks), arena, packs, key
        N.check(N.lib().ctl_train_pack_weights(self._pack_table.data_ptr(), self._pack_meta[0], self._pack_meta[1], N.stream_ptr()))
        self.launches += 1

    def _conv_bn(self, a, n, h, w, params, conv, bn, k, stride, relu, residual=None, ibn=False):
        wt = params[conv + ".weight"]
        cout = wt.shape[0]
        wf = self._packs[conv][0]  # forward operand [Cout][k][k][Cin] fp16 (ctl_train_pack_weights)
        y, ho, wo = self._conv(a, n, h, w, wf, cout, k, stride)
        rows = n * ho * wo
        z = torch.empty_like(y)
        L = N.lib()
        s = _Saved()
        if not ibn:
            mean = torch.empty(cout, device=self.device)
            invstd = torch.empty(cout, device=self.device)
            ws = self._bn_ws(rows, cout)
            rm, rv = params.get(bn + ".running_mean"), params.get(bn + ".running_var")
            N.check(L.ctl_bn_train_forward_nhwc_f16(
                y.data_ptr(), rows, cout, cout, params[bn + ".weight"].data_ptr(), params[bn + ".bias"].data_ptr(), BN_EPS,
                self.momentum, N.ptr(rm), N.ptr(rv), N.ptr(residual), int(relu), ws.data_ptr(), ws.numel(),
                mean.data_ptr(), invstd.data_ptr(), z.data_ptr(), N.stream_ptr()))
            self.launches += 3
            s.ibn = None
        else:
            # IBN (resnet_ibn_a.py:18-32): InstanceNorm on channels [0, half), batch-stat BatchNorm on [half, C); ReLU
            half = cout // 2
            im = torch.empty(n, half, device=self.device)
            ii = torch.empty(n, half, device=self.device)
            N.check(L.ctl_instnorm_train_forward_nhwc_f16(
                y.data_ptr(), n, ho * wo, cout, half, params[bn + ".IN.weight"].data_ptr(),
                params[bn + ".IN.bias"].data_ptr(), BN_EPS, im.data_ptr(), ii.data_ptr(), z.data_ptr(), N.stream_ptr()))
            mean = torch.empty(cout - half, device=self.device)
            invstd = torch.empty(cout - half, device=self.device)
            ws = self._bn_ws(rows, cout - half)
            off = half * 2  # bytes
            N.check(L.ctl_bn_train_forward_nhwc_f16(
                y.data_ptr() + off, rows, cout - half, cout, params[bn + ".BN.weight"].data_ptr(),
                params[bn + ".BN.bias"].data_ptr(), BN_EPS, self.momentum, N.ptr(params.get(bn + ".BN.running_mean")),
                N.ptr(params.get(bn + ".BN.running_var")), None, 1, ws.data_ptr(), ws.numel(), mean.data_ptr(),
                invstd.data_ptr(), z.data_ptr() + off, N.stream_ptr()))
            self.launches += 4
            s.ibn = (half, im, ii)
        s.a, s.y, s.z, s.mean, s.invstd = a, y, z, mean, invstd
        s.shape_in, s.shape_out, s.conv, s.bn, s.k, s.stride, s.relu = (n, h, w), (n, ho, wo), conv, bn, k, stride, relu
        self.saved.append(s)
        return z, ho, wo, s

    # ---------------------------------------------------------------- forward
    def check_input_size(self, H: int, W: int):
        """ValueError unless every stride-2 layer sees an even map at an H x W input: the backward of a stride-2 layer
        (weight gradient, zero-insertion data gradient) needs it.  Same rule and message as ctl_train_workspace_bytes."""
        h, w = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
        h, w = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
        for li in (2, 3, 4) if self.last_stride == 2 else (2, 3):
            if h % 2 or w % 2:
                raise ValueError(f"layer{li}.0.conv2: a training step needs an even input map at every stride-2 layer, "
                                 f"got {h}x{w} (input {H}x{W})")
            h, w = h // 2, w // 2

    def forward(self, x: torch.Tensor, params: Dict[str, torch.Tensor]) -> torch.Tensor:
        """x: [B, 3, H, W] fp32 NCHW on the device -> global_feat [B, 2048] fp32; keeps what backward needs."""
        if x.dim() != 4:
            raise ValueError(f"expected [B, 3, H, W], got {tuple(x.shape)}")
        self.check_input_size(int(x.shape[2]), int(x.shape[3]))
        if not self.graphs:
            return self._forward_impl(x, params)
        N.require_cuda(x)
        key = (tuple(x.shape), tuple(sorted((k, v.data_ptr()) for k, v in params.items())))
        g = self._graph
        if g is None or g["key"] != key:
            g = self._capture(x, params, key)
        g["x"].copy_(x)
        g["fwd"].replay()
        return g["feat"].clone()

    def backward(self, dfeat: torch.Tensor) -> Dict[str, torch.Tensor]:
        """dfeat: [B, 2048] fp32 = dLoss/dglobal_feat -> {param name: fp32 gradient in the reference's layout}."""
        if not self.graphs:
            return self._backward_impl(dfeat)
        g = self._graph
        g["dfeat"].copy_(dfeat)
        g["bwd"].replay()
        return {k: v.clone() for k, v in g["grads"].items()}

    def _capture(self, x, params, key):
        self._graph = None
        sx = x.detach().float().contiguous().clone()
        running = {k: v.clone() for k, v in params.items() if "running" in k}
        sdf = torch.zeros(x.shape[0], 2048, device=self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):  # eager warm-up: function attributes, workspaces, allocator pools
            self._forward_impl(sx, params)
            self._backward_impl(sdf)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        fwd, bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(fwd):
            feat = self._forward_impl(sx, params)
        with torch.cuda.graph(bwd, pool=fwd.pool()):
            grads = self._backward_impl(sdf)
        for k, v in running.items():  # the warm-up and capture passes must not count as training steps
            params[k].copy_(v)
        self._graph = {"key": key, "x": sx, "dfeat": sdf, "fwd": fwd, "bwd": bwd, "feat": feat, "grads": grads}
        return self._graph

    def _forward_impl(self, x: torch.Tensor, params: Dict[str, torch.Tensor]) -> torch.Tensor:
        N.require_cuda(x)
        x = x.float().contiguous()
        n, _, H, W = x.shape
        L = N.lib()
        self.saved, self.launches = [], 0
        self._params = params
        self._x = x
        with torch.cuda.device(self.device):
            # stem: raw 7x7/2 conv (tensor-core stem, zero bias, no ReLU) -> BN (no ReLU, resnet.py:125) -> max-pool
            w0 = params["conv1.weight"].detach()
            wk = torch.zeros(64, 21, 8, device=self.device)
            wk[:, :, :7] = w0.reshape(64, 21, 7)
            stem_w = torch.cat((wk.reshape(64, 168), torch.zeros(64, 24, device=self.device)), 1).half().contiguous()
            h, w = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
            y0 = torch.empty(n, h, w, 64, dtype=torch.float16, device=self.device)
            N.check(L.ctl_stem_conv7x7_tc(x.data_ptr(), n, H, W, stem_w.data_ptr(), self._zero_bias.data_ptr(), 0,
                                          y0.data_ptr(), N.stream_ptr()))
            rows = n * h * w
            z0 = torch.empty_like(y0)
            m0, i0 = torch.empty(64, device=self.device), torch.empty(64, device=self.device)
            ws = self._bn_ws(rows, 64)
            N.check(L.ctl_bn_train_forward_nhwc_f16(
                y0.data_ptr(), rows, 64, 64, params["bn1.weight"].data_ptr(), params["bn1.bias"].data_ptr(), BN_EPS,
                self.momentum, N.ptr(params.get("bn1.running_mean")), N.ptr(params.get("bn1.running_var")), None,
                int(self.ibn), ws.data_ptr(), ws.numel(), m0.data_ptr(), i0.data_ptr(), z0.data_ptr(), N.stream_ptr()))
            hp, wp = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
            a = torch.empty(n, hp, wp, 64, dtype=torch.float16, device=self.device)
            arg = torch.empty(n, hp, wp, 64, dtype=torch.uint8, device=self.device)
            N.check(L.ctl_maxpool3x3s2_argmax_nhwc_f16(z0.data_ptr(), n, h, w, 64, a.data_ptr(), arg.data_ptr(),
                                                       N.stream_ptr()))
            self.launches += 5
            self._stem = (y0, z0, m0, i0, (n, H, W, h, w, hp, wp), arg)
            self._pack_weights(params)
            h, w = hp, wp
            self._blocks = []
            for li, (planes, nblk) in enumerate(zip((64, 128, 256, 512), self.layers), start=1):
                stride0 = 1 if li == 1 else (self.last_stride if li == 4 else 2)
                for bi in range(nblk):
                    p = f"layer{li}.{bi}"
                    stride = stride0 if bi == 0 else 1
                    o1, h1, w1, s1 = self._conv_bn(a, n, h, w, params, p + ".conv1", p + ".bn1", 1, 1, True,
                                                   ibn=self.ibn and planes != 512)
                    o2, h2, w2, s2 = self._conv_bn(o1, n, h1, w1, params, p + ".conv2", p + ".bn2", 3, stride, True)
                    sd = None
                    res = a
                    if bi == 0:
                        res, _, _, sd = self._conv_bn(a, n, h, w, params, p + ".downsample.0", p + ".downsample.1", 1,
                                                      stride, False)
                    a, h, w, s3 = self._conv_bn(o2, n, h2, w2, params, p + ".conv3", p + ".bn3", 1, 1, True, residual=res)
                    self._blocks.append((s1, s2, s3, sd))
            c = a.shape[-1]
            feat = torch.empty(n, c, dtype=torch.float32, device=self.device)
            N.check(L.ctl_gap_bn_nhwc_f16(a.data_ptr(), n, h * w, c, None, None, feat.data_ptr(), None, N.stream_ptr()))
            self.launches += 1
            self._last = (n, h, w, c)
        return feat

    # ---------------------------------------------------------------- backward
    def _bn_bwd(self, s: _Saved, dz, relu_mask: bool, params, grads):
        n, ho, wo = s.shape_out
        c = s.y.shape[-1]
        rows = n * ho * wo
        dy = torch.empty_like(s.y)
        L = N.lib()
        if getattr(s, "ibn", None) is None:
            dg, db = torch.empty(c, device=self.device), torch.empty(c, device=self.device)
            ws = self._bn_ws(rows, c)
            N.check(L.ctl_bn_train_backward_nhwc_f16(
                dz.data_ptr(), s.z.data_ptr() if relu_mask else None, s.y.data_ptr(), rows, c, c,
                params[s.bn + ".weight"].data_ptr(), s.mean.data_ptr(), s.invstd.data_ptr(), 1.0 / self.grad_scale,
                ws.data_ptr(), ws.numel(), dz.data_ptr() if relu_mask else None, dg.data_ptr(), db.data_ptr(),
                dy.data_ptr(), N.stream_ptr()))
            self.launches += 3
            grads[s.bn + ".weight"], grads[s.bn + ".bias"] = dg, db
            return dy  # (dz now holds g = dz * mask when relu_mask)
        half, im, ii = s.ibn
        dgp, dbp = torch.empty(n, half, device=self.device), torch.empty(n, half, device=self.device)
        N.check(L.ctl_instnorm_train_backward_nhwc_f16(
            dz.data_ptr(), s.z.data_ptr(), s.y.data_ptr(), n, ho * wo, c, half, params[s.bn + ".IN.weight"].data_ptr(),
            im.data_ptr(), ii.data_ptr(), 1.0 / self.grad_scale, dgp.data_ptr(), dbp.data_ptr(), dy.data_ptr(),
            N.stream_ptr()))
        grads[s.bn + ".IN.weight"], grads[s.bn + ".IN.bias"] = dgp.sum(0), dbp.sum(0)
        cb = c - half
        dg, db = torch.empty(cb, device=self.device), torch.empty(cb, device=self.device)
        ws = self._bn_ws(rows, cb)
        off = half * 2
        N.check(L.ctl_bn_train_backward_nhwc_f16(
            dz.data_ptr() + off, s.z.data_ptr() + off, s.y.data_ptr() + off, rows, cb, c,
            params[s.bn + ".BN.weight"].data_ptr(), s.mean.data_ptr(), s.invstd.data_ptr(), 1.0 / self.grad_scale,
            ws.data_ptr(), ws.numel(), dz.data_ptr() + off, dg.data_ptr(), db.data_ptr(), dy.data_ptr() + off,
            N.stream_ptr()))
        self.launches += 6
        grads[s.bn + ".BN.weight"], grads[s.bn + ".BN.bias"] = dg, db
        return dy

    def _wgrad(self, a, shape_in, dy, cout, k, stride, param_layout=False):
        """param_layout: dw comes back un-scaled (x 1 / grad_scale) as [Cout][Cin][k][k], torch.nn.Conv2d.weight's layout
        (folded into the split-K reduction); else raw [Cout][k][k][Cin]."""
        n, h, w = shape_in
        cin = a.shape[-1]
        L = N.lib()
        need = L.ctl_conv2d_wgrad_workspace_bytes(n, h, w, cin, cout, k, stride)
        if self._ws_wg is None or self._ws_wg.numel() < need:
            self._ws_wg = torch.empty(need, dtype=torch.uint8, device=self.device)
        dw = torch.empty((cout, cin, k, k) if param_layout else (cout, k, k, cin), device=self.device)
        N.check(L.ctl_conv2d_wgrad_nhwc_f16_ex(a.data_ptr(), n, h, w, cin, dy.data_ptr(), cout, k, stride,
                                               self._ws_wg.data_ptr(), self._ws_wg.numel(), dw.data_ptr(),
                                               1.0 / self.grad_scale if param_layout else 1.0, int(param_layout),
                                               N.stream_ptr()))
        self.launches += 2
        return dw

    def _conv_bwd(self, s: _Saved, dy, params, grads, need_dx=True, residual=None):
        """weight gradient of s.conv and (optionally) the data gradient w.r.t. s.a (+ residual)."""
        wt = params[s.conv + ".weight"].detach()
        cout, cin, k = wt.shape[0], wt.shape[1], s.k
        if os.environ.get("CTL_WGRAD_NCHW", "1") == "1":
            grads[s.conv + ".weight"] = self._wgrad(s.a, s.shape_in, dy, cout, k, s.stride, param_layout=True)
        else:  # round-1 form (bisect aid): operand layout + torch permute / mul
            dw = self._wgrad(s.a, s.shape_in, dy, cout, k, s.stride)
            grads[s.conv + ".weight"] = dw.permute(0, 3, 1, 2).mul(1.0 / self.grad_scale)
        if not need_dx:
            return None
        n, h, w = s.shape_in
        _, ho, wo = s.shape_out
        wd = self._packs[s.conv][1]  # [Cin][k][k][Cout], flipped taps: the transposed convolution's operand
        L = N.lib()
        if s.stride == 1:
            dx, _, _ = self._conv(dy, n, ho, wo, wd, cin, k, 1, residual=residual)
            return dx
        if k == 1:
            low, _, _ = self._conv(dy, n, ho, wo, wd, cin, 1, 1)
            dx = torch.empty(n, h, w, cin, dtype=torch.float16, device=self.device)
            N.check(L.ctl_upsample2_zero_nhwc_f16(low.data_ptr(), n, ho, wo, cin, N.ptr(residual), dx.data_ptr(),
                                                  N.stream_ptr()))
            self.launches += 1
            return dx
        up = torch.empty(n, h, w, cout, dtype=torch.float16, device=self.device)
        N.check(L.ctl_upsample2_zero_nhwc_f16(dy.data_ptr(), n, ho, wo, cout, None, up.data_ptr(), N.stream_ptr()))
        self.launches += 1
        dx, _, _ = self._conv(up, n, h, w, wd, cin, 3, 1, residual=residual)
        return dx

    def _backward_impl(self, dfeat: torch.Tensor) -> Dict[str, torch.Tensor]:
        params, grads = self._params, {}
        L = N.lib()
        n, h, w, c = self._last
        with torch.cuda.device(self.device):
            dz = torch.empty(n, h, w, c, dtype=torch.float16, device=self.device)
            dfeat = dfeat.float().contiguous()
            N.check(L.ctl_gap_backward_nhwc_f16(dfeat.data_ptr(), n, h * w, c, self.grad_scale / (h * w), dz.data_ptr(),
                                                N.stream_ptr()))
            self.launches += 1
            for s1, s2, s3, sd in reversed(self._blocks):
                dy3 = self._bn_bwd(s3, dz, True, params, grads)  # dz becomes g3, the shortcut's gradient
                g3 = dz
                d2 = self._conv_bwd(s3, dy3, params, grads)
                dy2 = self._bn_bwd(s2, d2, True, params, grads)
                d1 = self._conv_bwd(s2, dy2, params, grads)
                dy1 = self._bn_bwd(s1, d1, True, params, grads)
                if sd is not None:
                    dyd = self._bn_bwd(sd, g3, False, params, grads)
                    shortcut = self._conv_bwd(sd, dyd, params, grads)
                else:
                    shortcut = g3
                dz = self._conv_bwd(s1, dy1, params, grads, residual=shortcut)
            # stem: max-pool -> BN (no ReLU) -> 7x7 weight gradient through the im2col GEMM
            y0, z0, m0, i0, (n, H, W, h, w, hp, wp), arg = self._stem
            dz0 = torch.empty_like(z0)
            N.check(L.ctl_maxpool3x3s2_backward_argmax_nhwc_f16(arg.data_ptr(), dz.data_ptr(), n, h, w, 64, dz0.data_ptr(),
                                                                N.stream_ptr()))
            st = _Saved()
            st.y, st.z, st.mean, st.invstd, st.bn, st.shape_out = y0, z0, m0, i0, "bn1", (n, h, w)
            st.ibn = None
            dy0 = self._bn_bwd(st, dz0, self.ibn, params, grads)  # IBN-a keeps the ReLU after the stem
            col = torch.empty(n, h, w, 192, dtype=torch.float16, device=self.device)
            N.check(L.ctl_stem_im2col_f16(self._x.data_ptr(), n, H, W, col.data_ptr(), N.stream_ptr()))
            self.launches += 2
            dw = self._wgrad(col, (n, h, w), dy0, 64, 1, 1)  # [64][1][1][192]
            grads["conv1.weight"] = dw.reshape(64, 192)[:, :168].reshape(64, 3, 7, 8)[..., :7].mul(1.0 / self.grad_scale)
        return grads


class NativeTrainer:
    """The same train-mode trunk with the LAYER GRAPH behind the C ABI (ctl_trainer_create / ctl_trainer_bind /
    ctl_train_forward / ctl_train_backward, csrc/trunk_train.cu): what a non-Python host binds.  `params` as in
    TrunkTrainer; gradients land in fp32 tensors this object owns (`grads`, the parameters' own layouts).
    Bit-identical to TrunkTrainer (tests/test_train_gpu.py::test_native_trainer_handle_matches_trunk_trainer)."""

    def __init__(self, params: Dict[str, torch.Tensor], device, last_stride: int = 1, ibn: bool = False,
                 grad_scale: float = 1024.0, momentum: float = 0.1):
        import ctypes as C

        self.device = torch.device(device)
        self.grad_scale = float(grad_scale)
        self._h = C.c_void_p()
        N.check(N.lib().ctl_trainer_create(C.byref(self._h), int(ibn), int(last_stride), float(momentum)))
        self._ws = None
        self.bind(params)

    def bind(self, params: Dict[str, torch.Tensor]):
        for k, v in params.items():
            if v.is_floating_point() and (v.dtype != torch.float32 or not v.is_contiguous() or v.device != self.device):
                raise TypeError(f"{k} must be a contiguous fp32 tensor on {self.device}")
        # the trunk's own tensors only (resnet_ibn_a.py keeps an unused ImageNet `fc` in its state_dict)
        self.params = {k: v for k, v in params.items() if v.is_floating_point() and not k.startswith("fc.")}
        self.grads = {k: torch.empty_like(v) for k, v in self.params.items() if "running" not in k}
        pa = (N.NamedTensor * len(self.params))()
        for i, (k, v) in enumerate(self.params.items()):
            pa[i].name, pa[i].data, pa[i].numel = k.encode(), v.data_ptr(), v.numel()
        ga = (N.NamedTensor * len(self.grads))()  # ctl_named_buffer has the same layout (writable data pointer)
        for i, (k, v) in enumerate(self.grads.items()):
            ga[i].name, ga[i].data, ga[i].numel = k.encode(), v.data_ptr(), v.numel()
        with torch.cuda.device(self.device):
            N.check(N.lib().ctl_trainer_bind(self._h, pa, len(self.params), ga, len(self.grads)))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        N.require_cuda(x)
        self._x = x.float().contiguous()  # the backward's stem im2col reads it again
        n, _, H, W = self._x.shape
        L = N.lib()
        need = L.ctl_train_workspace_bytes(self._h, n, H, W)
        if need == 0:
            raise ValueError(f"unsupported input shape {tuple(x.shape)}: {L.ctl_last_error().decode('utf-8', 'replace')}")
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        feat = torch.empty(n, 2048, device=self.device)
        with torch.cuda.device(self.device):
            N.check(L.ctl_train_forward(self._h, self._x.data_ptr(), n, H, W, feat.data_ptr(), self._ws.data_ptr(),
                                        self._ws.numel(), N.stream_ptr()))
        return feat

    def backward(self, dfeat: torch.Tensor) -> Dict[str, torch.Tensor]:
        dfeat = dfeat.float().contiguous()
        with torch.cuda.device(self.device):
            N.check(N.lib().ctl_train_backward(self._h, dfeat.data_ptr(), self.grad_scale, self._ws.data_ptr(),
                                               self._ws.numel(), N.stream_ptr()))
        return self.grads

    def __del__(self):
        try:
            if self._h:
                N.lib().ctl_trainer_destroy(self._h)
                self._h = None
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass
