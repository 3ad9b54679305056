"""GPU: training-side trunk kernels (weight gradient, batch-statistics BatchNorm forward/backward, ...)
against float64 torch autograd of the same fp16-rounded operands."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

WGRAD_SHAPES = [
    # n, h, w, cin, cout, k, stride
    (2, 16, 8, 64, 64, 1, 1),
    (3, 16, 8, 64, 64, 3, 1),
    (2, 16, 8, 256, 128, 1, 1),
    (2, 16, 16, 128, 128, 3, 2),
    (2, 12, 20, 64, 256, 1, 2),
    (5, 8, 4, 512, 192, 3, 1),
    (4, 32, 16, 128, 512, 1, 1),      # wide layers (layer2 expand)
    (3, 16, 8, 256, 256, 3, 1),       # layer3 3x3
    (6, 16, 8, 1024, 512, 1, 1),      # several cin chunks and cout tiles per CTA
    (2, 32, 16, 256, 512, 1, 2),      # strided shortcut (parity views)
    (2, 20, 20, 512, 256, 3, 1),      # 320x320 geometry: partial pixel tiles
]


@pytest.mark.parametrize("shape", WGRAD_SHAPES)
def test_conv_wgrad(shape):
    from ctl_b200 import _native as N

    L = N.lib()
    n, h, w, cin, cout, k, stride = shape
    g = torch.Generator().manual_seed(hash(shape) % 1000)
    pad = 1 if k == 3 else 0
    ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    x = (torch.randn(n, h, w, cin, generator=g)).half()
    dy = (torch.randn(n, ho, wo, cout, generator=g) * 0.5).half()
    ref = torch.nn.grad.conv2d_weight(x.double().permute(0, 3, 1, 2), (cout, cin, k, k), dy.double().permute(0, 3, 1, 2),
                                      stride=stride, padding=pad).permute(0, 2, 3, 1)  # [cout][k][k][cin]
    xd, dyd = x.cuda(), dy.cuda()
    nbytes = L.ctl_conv2d_wgrad_workspace_bytes(n, h, w, cin, cout, k, stride)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dw = torch.full((cout, k, k, cin), float("nan"), device="cuda")
    N.check(L.ctl_conv2d_wgrad_nhwc_f16(xd.data_ptr(), n, h, w, cin, dyd.data_ptr(), cout, k, stride, ws.data_ptr(),
                                        nbytes, dw.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    got = dw.cpu().double()
    assert torch.isfinite(got).all()
    # fp32 accumulation of exact fp16 products: error ~ sqrt(K) * 2^-24 * |terms|
    assert float((got - ref).abs().max()) <= 2e-5 * float(ref.abs().max()) + 1e-4
    # deterministic: a second call reproduces the bits
    dw2 = torch.empty_like(dw)
    N.check(L.ctl_conv2d_wgrad_nhwc_f16(xd.data_ptr(), n, h, w, cin, dyd.data_ptr(), cout, k, stride, ws.data_ptr(),
                                        nbytes, dw2.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)
    # the training engine's form: un-scaled, in torch.nn.Conv2d.weight's own layout [cout][cin][k][k]
    dw3 = torch.full((cout, cin, k, k), float("nan"), device="cuda")
    N.check(L.ctl_conv2d_wgrad_nhwc_f16_ex(xd.data_ptr(), n, h, w, cin, dyd.data_ptr(), cout, k, stride, ws.data_ptr(),
                                           nbytes, dw3.data_ptr(), 0.25, 1, N.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(dw3, dw.permute(0, 3, 1, 2) * 0.25)


@pytest.mark.parametrize("rows,c,relu,res", [(1000, 64, 1, 0), (4096, 256, 1, 1), (333, 2048, 0, 0), (20000, 128, 1, 1)])
def test_bn_train_forward_backward(rows, c, relu, res):
    from ctl_b200 import _native as N

    L = N.lib()
    g = torch.Generator().manual_seed(rows + c)
    y = (torch.randn(rows, c, generator=g) * 1.5 + 0.3).half()
    r = torch.randn(rows, c, generator=g).half() if res else None
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.2
    rm, rv = torch.randn(c, generator=g) * 0.1, torch.rand(c, generator=g) + 0.5
    dz = (torch.randn(rows, c, generator=g) * 0.1).half()
    eps, mom = 1e-5, 0.1
    # float64 reference on the fp16-rounded operands
    yd = y.double().requires_grad_(True)
    gd, bd = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    mean, var = yd.mean(0), yd.var(0, unbiased=False)
    pre = (yd - mean) / torch.sqrt(var + eps) * gd + bd + (r.double() if res else 0.0)
    zref = pre.clamp(min=0) if relu else pre
    zref16 = zref.detach().half()
    mask = (zref16 > 0).double() if relu else torch.ones_like(pre)
    (pre * (dz.double() * mask)).sum().backward()  # d/dpre = dz * mask, the engine's definition of g

    yc, dzc = y.cuda(), dz.cuda()
    rc_ = r.cuda() if res else None
    gam, bet, rmc, rvc = gamma.cuda(), beta.cuda(), rm.cuda(), rv.cuda()
    nb = L.ctl_bn_workspace_bytes(rows, c)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    sm, si = torch.empty(c, device="cuda"), torch.empty(c, device="cuda")
    out = torch.empty(rows, c, dtype=torch.float16, device="cuda")
    N.check(L.ctl_bn_train_forward_nhwc_f16(yc.data_ptr(), rows, c, c, gam.data_ptr(), bet.data_ptr(), eps, mom, rmc.data_ptr(),
                                            rvc.data_ptr(), N.ptr(rc_), relu, ws.data_ptr(), nb, sm.data_ptr(), si.data_ptr(),
                                            out.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(sm.cpu().numpy(), mean.detach().numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(si.cpu().numpy(), (1 / torch.sqrt(var + eps)).detach().numpy(), rtol=1e-5)
    np.testing.assert_allclose(rmc.cpu().numpy(), (0.9 * rm.double() + 0.1 * mean.detach()).numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(rvc.cpu().numpy(), (0.9 * rv.double() + 0.1 * yd.detach().var(0, unbiased=True)).numpy(), rtol=1e-5)
    err = (out.cpu().double() - zref.detach()).abs().max()
    assert float(err) <= float(zref.abs().max()) * 2.0 ** -10 + 1e-6  # one fp16 rounding

    dgam, dbet = torch.empty(c, device="cuda"), torch.empty(c, device="cuda")
    dy = torch.empty(rows, c, dtype=torch.float16, device="cuda")
    gbuf = torch.empty_like(dzc)
    zc = zref16.cuda()
    N.check(L.ctl_bn_train_backward_nhwc_f16(dzc.data_ptr(), zc.data_ptr() if relu else None, yc.data_ptr(), rows, c, c,
                                             gam.data_ptr(), sm.data_ptr(), si.data_ptr(), 0.5, ws.data_ptr(), nb,
                                             gbuf.data_ptr() if relu else None, dgam.data_ptr(), dbet.data_ptr(),
                                             dy.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    np.testing.assert_allclose(dgam.cpu().numpy(), 0.5 * gd.grad.numpy(), rtol=2e-4, atol=2e-4 * float(gd.grad.abs().max()))
    np.testing.assert_allclose(dbet.cpu().numpy(), 0.5 * bd.grad.numpy(), rtol=2e-4, atol=2e-4 * float(bd.grad.abs().max()))
    dyr = yd.grad
    assert float((dy.cpu().double() - dyr).abs().max()) <= float(dyr.abs().max()) * 2.0 ** -9 + 1e-7
    if relu:
        assert torch.equal(gbuf.cpu(), (dz.double() * mask).half())


def test_pool_gap_upsample_im2col_backward_helpers():
    from ctl_b200 import _native as N

    L = N.lib()
    g = torch.Generator().manual_seed(9)
    # max-pool backward vs autograd (fp16 values, including exact ties from a ReLU)
    n, h, w, c = 3, 12, 10, 64
    x = torch.randn(n, h, w, c, generator=g).clamp(min=0).half()
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    dy = torch.randn(n, ho, wo, c, generator=g).half()
    xr = x.float().permute(0, 3, 1, 2).requires_grad_(True)
    F.max_pool2d(xr, 3, 2, 1).backward(dy.float().permute(0, 3, 1, 2))
    xd, dyd = x.cuda(), dy.cuda()
    dx = torch.empty_like(xd)
    N.check(L.ctl_maxpool3x3s2_backward_nhwc_f16(xd.data_ptr(), dyd.data_ptr(), n, h, w, c, dx.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    ref = xr.grad.permute(0, 2, 3, 1)
    assert float((dx.cpu().float() - ref).abs().max()) <= 2.0 ** -9 * float(ref.abs().max())
    # training pair: forward that records the argmax tap + gather backward
    pooled = torch.empty(n, ho, wo, c, dtype=torch.float16, device="cuda")
    arg = torch.empty(n, ho, wo, c, dtype=torch.uint8, device="cuda")
    N.check(L.ctl_maxpool3x3s2_argmax_nhwc_f16(xd.data_ptr(), n, h, w, c, pooled.data_ptr(), arg.data_ptr(), N.stream_ptr()))
    dx2 = torch.empty_like(xd)
    N.check(L.ctl_maxpool3x3s2_backward_argmax_nhwc_f16(arg.data_ptr(), dyd.data_ptr(), n, h, w, c, dx2.data_ptr(),
                                                        N.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(pooled.cpu().float(), F.max_pool2d(x.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1))
    assert torch.equal(dx2.cpu(), dx.cpu())
    # global-average-pool backward
    df = torch.randn(4, 128, generator=g)
    out = torch.empty(4, 6, 128, dtype=torch.float16, device="cuda")
    dfd = df.cuda()
    N.check(L.ctl_gap_backward_nhwc_f16(dfd.data_ptr(), 4, 6, 128, 0.25, out.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(out.cpu(), (df * 0.25).half()[:, None, :].expand(4, 6, 128))
    # zero-insertion upsampling (+ add)
    xs = torch.randn(2, 3, 5, 64, generator=g).half()
    add = torch.randn(2, 6, 10, 64, generator=g).half()
    xsd, addd = xs.cuda(), add.cuda()
    up = torch.empty(2, 6, 10, 64, dtype=torch.float16, device="cuda")
    for a in (None, addd):
        N.check(L.ctl_upsample2_zero_nhwc_f16(xsd.data_ptr(), 2, 3, 5, 64, N.ptr(a), up.data_ptr(), N.stream_ptr()))
        torch.cuda.synchronize()
        ref = torch.zeros(2, 6, 10, 64)
        ref[:, ::2, ::2] = xs.float()
        if a is not None:
            ref = ref + add.float()
        assert torch.equal(up.cpu(), ref.half())
    # stem im2col: k = (c*7 + r)*8 + s
    xi = torch.randn(2, 3, 16, 12, generator=g)
    ho, wo = 8, 6
    col = torch.empty(2 * ho * wo, 192, dtype=torch.float16, device="cuda")
    xid = xi.cuda()
    N.check(L.ctl_stem_im2col_f16(xid.data_ptr(), 2, 16, 12, col.data_ptr(), N.stream_ptr()))
    torch.cuda.synchronize()
    unf = F.unfold(xi, 7, padding=3, stride=2).reshape(2, 3, 7, 7, ho * wo).permute(0, 4, 1, 2, 3)  # [n][pix][c][r][s]
    ref = torch.zeros(2, ho * wo, 3, 7, 8)
    ref[..., :7] = unf
    ref = torch.cat((ref.reshape(2 * ho * wo, 168), torch.zeros(2 * ho * wo, 24)), 1).half()
    assert torch.equal(col.cpu(), ref)


def _rel(a, b):
    return float((a.double() - b.double()).abs().max()) / (float(b.double().abs().max()) + 1e-30)


def test_trunk_train_step_against_float64_autograd():
    """Train-mode ResNet-50 forward + full backward on the B200 kernels vs float64 autograd of the same network
    with the engine's fp16 rounding points (oracle.trunk_train_fp16sim).

    (1) independent forward: features within 2e-2; gradients agree in direction and size (ReLU masks are
        discontinuous, so last-bit differences between two correct fp16 forwards show up as ~10 % max-norm
        gradient noise: cosine >= 0.98, norm within 3 %);
    (2) teacher-forced: the oracle differentiates through the ENGINE's stored activations, which isolates the
        backward arithmetic: every parameter gradient within 2e-2 (max-norm relative)."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.backbones.engine_train import TrunkTrainer

    sd = O.make_trunk_state(seed=7)
    g = torch.Generator().manual_seed(1)
    n, H, W = 8, 128, 64
    x = torch.randn(n, 3, H, W, generator=g)
    dfeat = torch.randn(n, 2048, generator=g) * 1e-3
    feat_o, grads_o, running_o = O.trunk_train_fp16sim(x, sd, dfeat)

    params = {k: v.clone().cuda() for k, v in sd.items() if v.is_floating_point()}
    tr = TrunkTrainer("cuda", grad_scale=4096.0)
    feat = tr.forward(x.cuda(), params)
    torch.cuda.synchronize()
    assert _rel(feat.cpu(), feat_o) <= 2e-2
    nchw = lambda t: t.cpu().float().permute(0, 3, 1, 2)  # noqa: E731
    forced = [(nchw(tr._stem[0]), nchw(tr._stem[1]))] + [(nchw(s.y), nchw(s.z)) for s in tr.saved]
    grads = tr.backward(dfeat.cuda())
    torch.cuda.synchronize()
    assert set(grads.keys()) == set(grads_o.keys())
    gscale = max(float(v.abs().max()) for v in grads_o.values())
    for k, go in grads_o.items():
        gk = grads[k].cpu().double()
        assert gk.shape == go.shape and torch.isfinite(gk).all(), k
        if float(go.abs().max()) < 1e-6 * gscale:  # stem bn1.bias: exactly cancelled by the next batch-stat BN
            assert float(gk.abs().max()) <= 1e-3 * gscale, k
            continue
        cos = float((gk * go).sum() / (gk.norm() * go.norm()))
        assert cos >= 0.98 and abs(float(gk.norm() / go.norm()) - 1) <= 3e-2, (k, cos)
    for k, v in running_o.items():
        assert _rel(params[k].cpu(), v) <= 2e-2, k
    # (2) teacher-forced backward check
    feat_f, grads_f, _ = O.trunk_train_fp16sim(x, sd, dfeat, forced=forced)
    assert _rel(feat.cpu(), feat_f) <= 1e-5
    bad = {}
    for k, go in grads_f.items():
        if float(go.abs().max()) < 1e-6 * gscale:
            continue
        r = _rel(grads[k].cpu(), go)
        if r > 2e-2:
            bad[k] = r
    assert not bad, f"gradient mismatch (max-norm relative): {sorted(bad.items(), key=lambda t: -t[1])[:8]}"


def test_baseline_train_mode_is_differentiable():
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.baseline import Baseline
    from test_modules_gpu import _cfg

    model = Baseline(_cfg()).cuda().train()
    model.base.load_state_dict(O.make_trunk_state(seed=2))
    x = torch.randn(4, 3, 64, 32, generator=torch.Generator().manual_seed(4)).cuda()
    rm0 = model.base.bn1.running_mean.clone()
    base_out, feat = model(x)
    assert base_out is None and feat.shape == (4, 2048) and feat.requires_grad
    (feat * 1e-3).sum().backward()
    names = [k for k, _ in model.base.named_parameters()]
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in model.base.parameters()), names
    assert float(model.base.layer4[2].conv3.weight.grad.abs().max()) > 0 and float(model.base.conv1.weight.grad.abs().max()) > 0
    assert not torch.equal(rm0, model.base.bn1.running_mean) and int(model.base.bn1.num_batches_tracked) == 1
    model.eval()
    with torch.no_grad():
        _, f2 = model(x)  # eval engine refolds the updated running statistics
    assert torch.isfinite(f2).all()


def test_ctl_training_step_end_to_end():
    """CTLModel.training_step (train_ctl_model.py:38-152): train-mode trunk -> CTL / center / xent / query-triplet
    losses -> backward through the fused loss step AND the trunk, on a P x K batch with padded (mock) rows."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.ctl_model import CTLModel
    from test_modules_gpu import _cfg

    torch.manual_seed(0)
    P_, K_ = 4, 4
    model = CTLModel(_cfg(), num_classes=16, num_query=4).cuda().train()
    sd = O.make_trunk_state(seed=9)
    model.backbone.base.load_state_dict(sd)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(P_ * K_, 3, 64, 32, generator=g)
    labels = torch.arange(P_).repeat_interleave(K_) + 3
    is_real = torch.ones(P_ * K_, dtype=torch.bool)
    is_real[K_ - 1] = False  # last slot of the first pid is a mock image (all-zero crop, datasets/bases.py:378-391)
    x[K_ - 1] = 0
    out = model.training_step((x.cuda(), labels.cuda(), torch.zeros(P_ * K_, dtype=torch.long).cuda(), is_real.cuda()), 0)
    loss = out["loss"]
    assert torch.isfinite(loss)
    loss.backward()
    for name, p in model.named_parameters():
        if name == "bn.bias":  # frozen in the reference (bases.py:83-84)
            continue
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    assert float(model.backbone.base.layer1[0].conv1.weight.grad.abs().max()) > 0
    # loss value against the oracle: fp16-sim train-mode features -> the reference's loss arithmetic
    feat_o, _, _ = O.trunk_train_fp16sim(x, sd)
    hs = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    ref = O.ctl_step_losses(feat_o.float(), labels, is_real, K_, hs["center_loss.centers"], hs["bn.weight"], hs["bn.bias"],
                            hs["fc_query.weight"])
    np.testing.assert_allclose(float(loss), float(ref["total"]), rtol=5e-3)


def test_trunk_train_cuda_graphs_reproduce_eager_bits():
    """graphs=True replays the captured forward/backward; kernels are deterministic, so features, gradients and
    running statistics are bit-identical to the eager path, step after step."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.backbones.engine_train import TrunkTrainer

    sd = O.make_trunk_state(seed=3)
    g = torch.Generator().manual_seed(8)
    xs = [torch.randn(4, 3, 64, 32, generator=g).cuda() for _ in range(2)]
    dfs = [(torch.randn(4, 2048, generator=g) * 1e-3).cuda() for _ in range(2)]
    outs = []
    for graphs in (False, True):
        params = {k: v.clone().cuda() for k, v in sd.items() if v.is_floating_point()}
        tr = TrunkTrainer("cuda", graphs=graphs)
        res = []
        for x, df in zip(xs, dfs):
            feat = tr.forward(x, params)
            grads = tr.backward(df)
            res.append((feat.clone(), {k: v.clone() for k, v in grads.items()}))
        torch.cuda.synchronize()
        outs.append((res, {k: v.clone() for k, v in params.items() if "running" in k}))
    (eager, run_e), (graph, run_g) = outs
    for (fe, ge), (fg, gg) in zip(eager, graph):
        assert torch.equal(fe, fg)
        assert all(torch.equal(ge[k], gg[k]) for k in ge)
    assert all(torch.equal(run_e[k], run_g[k]) for k in run_e)


def test_full_training_iterations_reduce_the_loss():
    """Three complete iterations (train-mode trunk -> losses -> backward -> fused Adam + center SGD) on one batch:
    finite everywhere, parameters move, the loss decreases."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.ctl_model import CTLModel
    from test_modules_gpu import _cfg

    torch.manual_seed(0)
    cfg = _cfg()
    cfg["SOLVER"].update(dict(OPTIMIZER_NAME="Adam", BASE_LR=3.5e-4, WEIGHT_DECAY=5e-4, CENTER_LR=0.5,
                              LR_SCHEDULER_NAME="multistep_lr", LR_STEPS=(40, 70), GAMMA=0.1, USE_WARMUP_LR=False,
                              WARMUP_EPOCHS=10))
    model = CTLModel(cfg, num_classes=16, num_query=4).cuda().train()
    model.backbone.base.load_state_dict(O.make_trunk_state(seed=11))
    (opt, opt_center), _ = model.configure_optimizers()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(16, 3, 64, 32, generator=g).cuda()
    labels = (torch.arange(4).repeat_interleave(4) + 1).cuda()
    batch = (x, labels, torch.zeros(16, dtype=torch.long).cuda(), torch.ones(16, dtype=torch.bool).cuda())
    w0 = model.backbone.base.layer2[0].conv2.weight.detach().clone()
    losses = []
    for _ in range(3):
        for p_ in model.parameters():
            p_.grad = None
        out = model.training_step(batch, 0)
        out["loss"].backward()
        model.optimizer_step_manual(opt, opt_center, epoch=20)
        losses.append(float(out["loss"]))
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    assert not torch.equal(w0, model.backbone.base.layer2[0].conv2.weight)
    assert all(torch.isfinite(p_).all() for p_ in model.parameters())


def test_ibn_trunk_train_step_teacher_forced():
    """ResNet50-IBN-a train step (resnet_ibn_a.py): ReLU after the stem, InstanceNorm half + BatchNorm half as bn1 of
    layer1-3 (channel-slice kernels), 80x40 crops (non-power-of-two maps, partial tiles) -- same two-level check as the
    plain trunk."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.backbones.engine_train import TrunkTrainer

    sd = O.make_trunk_state(seed=13, ibn=True)
    g = torch.Generator().manual_seed(5)
    n, H, W = 6, 160, 80
    x = torch.randn(n, 3, H, W, generator=g)
    dfeat = torch.randn(n, 2048, generator=g) * 1e-3
    params = {k: v.clone().cuda() for k, v in sd.items() if v.is_floating_point()}
    tr = TrunkTrainer("cuda", grad_scale=4096.0, ibn=True)
    feat = tr.forward(x.cuda(), params)
    torch.cuda.synchronize()
    nchw = lambda t: t.cpu().float().permute(0, 3, 1, 2)  # noqa: E731
    forced = [(nchw(tr._stem[0]), nchw(tr._stem[1]))] + [(nchw(s.y), nchw(s.z)) for s in tr.saved]
    grads = tr.backward(dfeat.cuda())
    torch.cuda.synchronize()
    feat_o, _, running_o = O.trunk_train_fp16sim(x, sd, ibn=True)
    assert _rel(feat.cpu(), feat_o) <= 2e-2
    for k, v in running_o.items():
        assert _rel(params[k].cpu(), v) <= 2e-2, k
    feat_f, grads_f, _ = O.trunk_train_fp16sim(x, sd, dfeat, forced=forced, ibn=True)
    grads_f = {k: v for k, v in grads_f.items() if v is not None}  # the unused ImageNet fc head has no gradient
    assert set(grads.keys()) == set(grads_f.keys())
    assert _rel(feat.cpu(), feat_f) <= 1e-5
    gscale = max(float(v.abs().max()) for v in grads_f.values())
    bad = {}
    for k, go in grads_f.items():
        assert torch.isfinite(grads[k]).all(), k
        if float(go.abs().max()) < 1e-6 * gscale:
            continue
        r = _rel(grads[k].cpu(), go)
        if r > 2e-2:
            bad[k] = r
    assert not bad, f"gradient mismatch (max-norm relative): {sorted(bad.items(), key=lambda t: -t[1])[:8]}"


@pytest.mark.parametrize("tag,ibn", [("r50", False), ("ibn", True)])
def test_trunk_train_matches_reference_under_autocast(tag, ibn):
    """Train-mode features and parameter gradients against the UNMODIFIED reference run under fp16 autocast with a fixed
    loss scale (tests/golden/trunk_autocast.npz, oracle/make_golden.py::gen_trunk_autocast) -- the same-precision
    checker.  Two correct fp16 train steps differ through ReLU masks (see test_trunk_train_step_against_float64_autograd),
    so gradients are compared by direction and size on the golden's evenly strided samples: cosine >= 0.97, norm within
    5 %; features within 2e-2 of the feature scale (measured values are printed)."""
    from oracle import ctl_oracle as O
    from oracle.make_golden import TRAIN_GRAD_KEYS, grad_sample
    from conftest import load_golden
    from ctl_b200.modelling.backbones.engine_train import TrunkTrainer

    g = load_golden("trunk_autocast.npz")
    sd = O.make_trunk_state(seed=17, ibn=ibn)
    gen = torch.Generator().manual_seed(23)
    x = torch.randn(4, 3, 64, 32, generator=gen)
    dfeat = torch.randn(4, 2048, generator=gen) * 1e-2
    params = {k: v.clone().cuda() for k, v in sd.items() if v.is_floating_point()}
    tr = TrunkTrainer("cuda", grad_scale=1024.0, ibn=ibn)
    feat = tr.forward(x.cuda(), params)
    grads = tr.backward(dfeat.cuda())
    torch.cuda.synchronize()
    ref_feat = torch.from_numpy(g[f"{tag}_train_feat_amp"])
    e = _rel(feat.cpu(), ref_feat)
    print(f"{tag}: train-mode features vs reference-under-autocast {e:.3e}")
    assert e <= 2e-2
    worst = (1.0, None)
    for key in TRAIN_GRAD_KEYS:
        k = key.format(bn="BN." if ibn else "")
        want = torch.from_numpy(g[f"{tag}_train_grad_{k}"])[:-2]
        got = torch.from_numpy(grad_sample(grads[k].cpu()))[:-2]
        if float(want.abs().max()) < 1e-7:
            continue
        cos = float((got * want).sum() / (got.norm() * want.norm()))
        nr = float(got.norm() / want.norm())
        if cos < worst[0]:
            worst = (cos, k)
        assert cos >= 0.97 and abs(nr - 1) <= 5e-2, (k, cos, nr)
    print(f"{tag}: worst gradient cosine vs reference-under-autocast {worst[0]:.4f} ({worst[1]})")


@pytest.mark.parametrize("ibn,shape,last_stride", [(False, (4, 64, 32), 1), (False, (3, 96, 64), 2), (True, (6, 160, 80), 1)])
def test_native_trainer_handle_matches_trunk_trainer(ibn, shape, last_stride):
    """ctl_trainer_* (csrc/trunk_train.cu, the train forward / backward behind the C ABI) issues the launches of
    engine_train.TrunkTrainer in the same order: features, every parameter gradient and the running statistics are
    bit-identical over two consecutive steps (the InstanceNorm affine gradients, which TrunkTrainer sums over the
    images with torch.sum and the handle with its own fixed-order kernel: 1e-6 relative)."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.backbones.engine_train import NativeTrainer, TrunkTrainer

    sd = O.make_trunk_state(seed=21, ibn=ibn)
    n, H, W = shape
    g = torch.Generator().manual_seed(31)
    xs = [torch.randn(n, 3, H, W, generator=g).cuda() for _ in range(2)]
    dfs = [(torch.randn(n, 2048, generator=g) * 1e-3).cuda() for _ in range(2)]
    outs = []
    for native in (False, True):
        params = {k: v.clone().cuda().contiguous() for k, v in sd.items() if v.is_floating_point()}
        tr = (NativeTrainer(params, "cuda:0", last_stride=last_stride, ibn=ibn, grad_scale=2048.0) if native
              else TrunkTrainer("cuda:0", last_stride=last_stride, ibn=ibn, grad_scale=2048.0))
        res = []
        for x, df in zip(xs, dfs):
            feat = tr.forward(x) if native else tr.forward(x, params)
            grads = tr.backward(df)
            res.append((feat.clone(), {k: v.clone() for k, v in grads.items()}))
        torch.cuda.synchronize()
        outs.append((res, {k: v.clone() for k, v in params.items() if "running" in k}))
    (py, run_p), (nat, run_n) = outs
    for (fp, gp), (fn, gn) in zip(py, nat):
        assert torch.equal(fp, fn)
        assert set(gp) == set(gn)
        for k in gp:
            assert gp[k].shape == gn[k].shape, k
            if ".IN." in k:
                assert _rel(gn[k], gp[k]) < 1e-6, k
            else:
                assert torch.equal(gp[k], gn[k]), k
    assert all(torch.equal(run_p[k], run_n[k]) for k in run_p)


def test_native_trainer_argument_errors():
    """missing tensors, a backward without its forward, and a foreign workspace are reported, not executed."""
    import ctypes as C

    from ctl_b200 import _native as N
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.backbones.engine_train import NativeTrainer

    sd = O.make_trunk_state(seed=2)
    params = {k: v.clone().cuda().contiguous() for k, v in sd.items() if v.is_floating_point()}
    broken = dict(params)
    del broken["layer2.0.downsample.1.weight"]
    with pytest.raises(ValueError, match="layer2.0.downsample.1.weight"):
        NativeTrainer(broken, "cuda:0")
    tr = NativeTrainer(params, "cuda:0")
    df = torch.zeros(2, 2048, device="cuda")
    tr._ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="forward"):
        tr.backward(df)
    tr.forward(torch.randn(2, 3, 64, 32, device="cuda"))
    other = torch.empty_like(tr._ws)
    rc = N.lib().ctl_train_backward(tr._h, df.data_ptr(), C.c_float(1024.0), other.data_ptr(), other.numel(), N.stream_ptr())
    assert rc != 0 and b"workspace of the forward" in N.lib().ctl_last_error()
    tr.backward(df)  # the right workspace still works
    torch.cuda.synchronize()


@pytest.mark.parametrize("which", ["python", "python_graphs", "native"])
def test_trainers_reject_odd_stride2_maps_before_any_launch(which):
    """A training step cannot run where a stride-2 layer would see an odd map (300x150: layer1 leaves 75x38).  Both
    trainers raise ValueError naming the layer and the map size before anything runs on the device: the BatchNorm
    running statistics they were given are unchanged."""
    from oracle import ctl_oracle as O
    from ctl_b200.modelling.backbones.engine_train import NativeTrainer, TrunkTrainer

    sd = O.make_trunk_state(seed=3)
    params = {k: v.clone().cuda().contiguous() for k, v in sd.items() if v.is_floating_point()}
    running = {k: v.clone() for k, v in params.items() if "running" in k}
    x = torch.randn(2, 3, 300, 150, generator=torch.Generator().manual_seed(1)).cuda()
    if which == "native":
        tr = NativeTrainer(params, "cuda:0")
        call = lambda: tr.forward(x)  # noqa: E731
    else:
        tr = TrunkTrainer("cuda:0", graphs=which == "python_graphs")
        call = lambda: tr.forward(x, params)  # noqa: E731
    with pytest.raises(ValueError, match=r"layer2\.0\.conv2.*75x38"):
        call()
    torch.cuda.synchronize()
    assert all(torch.equal(params[k], v) for k, v in running.items())
