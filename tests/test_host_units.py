"""CPU: host-side pieces added around the hot path (no GPU, no kernels): parameter sampling of the device transforms,
the stem weight packing, the warm-up LR rule, the pid/path index of the inference scripts."""
import numpy as np
import torch

import ctl_b200  # noqa: F401


class _C(dict):
    __getattr__ = dict.__getitem__


def test_sample_params_ranges_and_mock_rows():
    from ctl_b200.datasets.transforms import sample_params

    p = sample_params(500, 64, 32, prob_flip=0.3, pad=5, re_prob=1.0, is_real=np.r_[np.ones(499), 0],
                      rng=np.random.default_rng(1))
    assert p.dtype == np.int32 and p.shape == (500, 8)
    assert set(np.unique(p[:, 0])) <= {0, 1} and abs(p[:, 0].mean() - 0.3) < 0.08
    assert p[:, 1:3].min() >= 0 and p[:, 1:3].max() <= 10
    assert (p[:, 5] > 0).all() and (p[:, 5] < 64).all() and (p[:, 6] < 32).all()      # re_prob = 1: always erased
    assert (p[:, 3] + p[:, 5] <= 64).all() and (p[:, 4] + p[:, 6] <= 32).all()       # rectangle inside the image
    assert p[-1, 7] == 0 and p[:-1, 7].all()
    none = sample_params(50, 64, 32, re_prob=0.0, rng=np.random.default_rng(2))
    assert (none[:, 5] == 0).all()


def test_pack_stem_fused_layout_matches_the_header_definition():
    from ctl_b200.modelling.backbones.engine import pack_stem_fused

    w = torch.randn(64, 3, 7, 7, generator=torch.Generator().manual_seed(0))
    pk = pack_stem_fused(w)
    assert pk.shape == (28, 64, 8) and pk.dtype == torch.float16
    for c in (0, 5, 13, 27):
        for e in range(8):
            r, s, ch = c // 4, 2 * (c % 4) + e // 4, e % 4
            exp = w[:, ch, r, s].half() if (ch < 3 and s < 7) else torch.zeros(64, dtype=torch.float16)
            assert torch.equal(pk[c, :, e], exp), (c, e)


def test_warmup_rule_and_scheduler_names():
    from ctl_b200.solver.build import apply_warmup_lr, build_scheduler

    hp = _C(SOLVER=_C(USE_WARMUP_LR=True, WARMUP_EPOCHS=10, BASE_LR=1e-3, LR_SCHEDULER_NAME="multistep_lr", LR_STEPS=(2, 3),
                      GAMMA=0.1, MAX_EPOCHS=5, MIN_LR=1e-6))
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=1e-3)
    for epoch, exp in ((0, 1e-4), (4, 5e-4), (9, 1e-3)):
        apply_warmup_lr(opt, epoch, hp)
        assert abs(opt.param_groups[0]["lr"] - exp) < 1e-12
    opt.param_groups[0]["lr"] = 0.123
    apply_warmup_lr(opt, 10, hp)  # past the warm-up: untouched (modelling/bases.py:116)
    assert opt.param_groups[0]["lr"] == 0.123
    assert isinstance(build_scheduler(opt, hp), torch.optim.lr_scheduler.MultiStepLR)
    hp.SOLVER.LR_SCHEDULER_NAME = "cosine_annealing"
    assert isinstance(build_scheduler(opt, hp), torch.optim.lr_scheduler.CosineAnnealingLR)
    hp.SOLVER.LR_SCHEDULER_NAME = "nope"
    try:
        build_scheduler(opt, hp)
        raise AssertionError("expected NotImplementedError")
    except NotImplementedError:
        pass


def test_pid_path_index_and_no_cpu_fallback(tmp_path):
    from ctl_b200.inference import inference_utils as IU

    paths = ["a/0002_c1.jpg", "a/0001_c2.jpg", "a/0002_c3.jpg"]
    idx = IU.create_pid_path_index(paths, lambda p: p.split("/")[-1].split("_")[0])
    assert list(idx.items()) == [("0002", [0, 2]), ("0001", [1])]
    IU.save_gallery(tmp_path, np.ones((2, 4), dtype=np.float32), np.array(["x", "y"]))
    emb, pth = IU.load_gallery(tmp_path)
    assert emb.dtype == torch.float32 and list(pth) == ["x", "y"]
    try:
        IU._inference(None, (torch.zeros(1, 3, 8, 8), [""], ["p"]), use_cuda=False)
        raise AssertionError("expected RuntimeError")
    except RuntimeError as e:
        assert "no CPU path" in str(e)


def test_c_abi_argument_errors_are_reported_without_a_gpu():
    """Shape / contract violations are rejected by the C ABI before any device work (status CTL_ERR_INVALID_ARGUMENT,
    message in ctl_last_error(), mapped to ValueError by the shim) -- the reference raises on the same conditions with
    Python asserts; nothing silently falls back."""
    import ctypes as C

    import pytest

    from ctl_b200 import _native as N

    L = N.lib()
    one = C.c_void_p(16)  # a non-null, 16-byte-aligned dummy pointer: argument checks come before any dereference
    cases = [
        lambda: L.ctl_conv2d_nhwc_f16(one, 1, 8, 8, 48, one, one, None, one, 64, 1, 1, 0, 0, None),          # Cin % 64
        lambda: L.ctl_conv2d_nhwc_f16(one, 1, 8, 8, 64, one, one, None, one, 64, 5, 1, 0, 0, None),          # 5x5
        lambda: L.ctl_conv2d_nhwc_f16(one, 1, 7, 8, 64, one, one, None, one, 64, 3, 3, 0, 0, None),          # stride 3
        lambda: L.ctl_conv2d_wgrad_nhwc_f16(one, 1, 8, 8, 64, one, 96, 1, 1, one, 1 << 30, one, None),       # Cout % 64
        lambda: L.ctl_bn_train_forward_nhwc_f16(one, 10, 48, 48, one, one, 1e-5, 0.1, None, None, None, 0, one, 1 << 20,
                                                 one, one, one, None),                                         # C not a power of two
        lambda: L.ctl_bn_train_forward_nhwc_f16(one, 10, 64, 32, one, one, 1e-5, 0.1, None, None, None, 0, one, 1 << 20,
                                                 one, one, one, None),                                         # pitch < C
        lambda: L.ctl_bn_train_backward_nhwc_f16(one, one, one, 10, 64, 64, one, one, one, 1.0, one, 1 << 20, None, one, one,
                                                  one, None),                                                  # mask without g_out
        lambda: L.ctl_stem_pool_fused(one, 1, 30, 64, one, one, one, 0, one, None),                           # H % 4
        lambda: L.ctl_stem_pool_fused(one, 1, 32, 256, one, one, one, 0, one, None),                          # W > 128
        lambda: L.ctl_instnorm_train_forward_nhwc_f16(one, 1, 16, 64, 12, one, one, 1e-5, one, one, one, None),  # half % 8
        lambda: L.ctl_adam_multi_step(one, 0, 1, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, 1.0, None, None),            # no tensors
        lambda: L.ctl_loss_scale_update(one, one, one, one, 1024.0, 0.5, 0.5, 2000, None),                    # growth < 1
        lambda: L.ctl_conv1x1_dual_nhwc_f16(one, 64, one, 7, 8, 64, 2, 1, one, one, one, 256, 1, None),       # odd H2, stride 2
        lambda: L.ctl_augment_batch_u8(one, 1, 8, 8, -1, one, (C.c_float * 3)(0, 0, 0), (C.c_float * 3)(1, 1, 1), one, None),
        lambda: L.ctl_trainer_create(C.byref(C.c_void_p()), 0, 3, 0.1),                                      # LAST_STRIDE 3
        lambda: L.ctl_trainer_create(C.byref(C.c_void_p()), 0, 1, 0.0),                                      # momentum 0
    ]
    for i, call in enumerate(cases):
        rc = call()
        assert rc == -1, (i, rc, L.ctl_last_error())
        assert len(L.ctl_last_error()) > 0
        with pytest.raises(ValueError):
            N.check(rc)
    assert L.ctl_bn_workspace_bytes(10, 48) == 0 and L.ctl_conv2d_wgrad_workspace_bytes(1, 8, 8, 60, 64, 1, 1) == 0


def test_trainer_handle_plans_its_workspace_without_a_gpu():
    """ctl_train_workspace_bytes is a dry walk of the forward + backward launch sequence (no device work): it grows
    linearly with the batch and covers at least the saved activations (y and z of every conv + BatchNorm)."""
    import ctypes as C

    from ctl_b200 import _native as N

    L = N.lib()
    for ibn in (0, 1):
        h = C.c_void_p()
        assert L.ctl_trainer_create(C.byref(h), ibn, 1, 0.1) == 0
        b16, b32 = L.ctl_train_workspace_bytes(h, 16, 256, 128), L.ctl_train_workspace_bytes(h, 32, 256, 128)
        assert b16 > 0 and 1.8 < b32 / b16 < 2.05
        # saved y + z alone: ~29 MB per 256x128 image (fp16), the whole step stays below 3x that
        assert 16 * 25e6 < b16 < 16 * 90e6
        assert L.ctl_train_workspace_bytes(h, 0, 256, 128) == 0 and L.ctl_train_workspace_bytes(h, 4, 16, 16) == 0
        df = C.c_void_p(256)
        assert L.ctl_train_backward(h, df, C.c_float(1024.0), df, 1 << 30, None) == -1  # no forward yet
        assert b"forward" in L.ctl_last_error()
        L.ctl_trainer_destroy(h)


def test_identity_orders_and_encoded_ids_on_the_host():
    """retrieval.pid_order is a stable sort by identity; encode_ids(q_order=, g_order=) hands the kernels the identity
    arrays in the planes' row order (dense labels keep the identity order, so sorted rows give monotone labels -- what the
    tile-range test of ctl_dist_worklist relies on); pid_order_pays switches by problem size."""
    import numpy as np

    from ctl_b200 import retrieval as R

    rng = np.random.default_rng(3)
    q_pid, g_pid = rng.integers(100, 160, 300), rng.integers(100, 160, 2000)
    q_cam, g_cam = rng.integers(0, 6, 300), rng.integers(0, 6, 2000)
    qo, go = R.pid_order(q_pid), R.pid_order(g_pid)
    assert np.array_equal(np.sort(qo), np.arange(300)) and (np.diff(q_pid[qo]) >= 0).all()
    same = q_pid[qo][1:] == q_pid[qo][:-1]
    assert (np.diff(qo)[same] > 0).all(), "stable: equal identities keep the caller's order"
    plain = R.encode_ids(q_pid, g_pid, q_cam, g_cam, False, "cpu")
    srt = R.encode_ids(q_pid, g_pid, q_cam, g_cam, False, "cpu", q_order=qo, g_order=go)
    assert np.array_equal(srt.q_pid.numpy(), plain.q_pid.numpy()[qo]) and np.array_equal(srt.g_pid.numpy(), plain.g_pid.numpy()[go])
    assert np.array_equal(srt.q_cam.numpy(), plain.q_cam.numpy()[qo]) and np.array_equal(srt.g_mask.numpy(), plain.g_mask.numpy()[go])
    assert srt.max_pos == plain.max_pos
    assert (np.diff(srt.q_pid.numpy()) >= 0).all() and (np.diff(srt.g_pid.numpy()) >= 0).all()
    # sorted operands: few 128 x 128 tiles have intersecting identity ranges; unsorted: all of them
    def hot_fraction(qp, gp):
        qr = [(qp[i:i + 128].min(), qp[i:i + 128].max()) for i in range(0, len(qp), 128)]
        gr = [(gp[i:i + 128].min(), gp[i:i + 128].max()) for i in range(0, len(gp), 128)]
        return np.mean([not (b[1] < a[0] or b[0] > a[1]) for a in qr for b in gr])
    assert hot_fraction(srt.q_pid.numpy(), srt.g_pid.numpy()) < 0.5 < hot_fraction(plain.q_pid.numpy(), plain.g_pid.numpy())
    assert not R.pid_order_pays(3368, 15913) and R.pid_order_pays(50000, 25000)


def _trunk_walk(H, W, last_stride):
    """Layer walk of the eval trunk at an H x W input with torch.nn.Conv2d / MaxPool2d output sizes (elementwise over numpy
    arrays H, W): (elements of the largest activation per image -- stem conv, max-pool and every conv output --, and the
    input map (h, w) of every stride-2 bottleneck layer as (name, h, w))."""
    h, w = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    big = h * w * 64
    h, w = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
    big = np.maximum(big, h * w * 64)
    strided = []
    for li, (planes, nblk) in enumerate(zip((64, 128, 256, 512), (3, 4, 6, 3)), start=1):
        for bi in range(nblk):
            s = (1 if li == 1 else (last_stride if li == 4 else 2)) if bi == 0 else 1
            if s == 2:
                strided.append((f"layer{li}.{bi}.conv2", h, w))
            h2, w2 = (h - 1) // s + 1, (w - 1) // s + 1
            big = np.maximum(big, h * w * planes)            # conv1
            big = np.maximum(big, h2 * w2 * planes * 4)      # conv3 / downsample (conv2 is smaller)
            h, w = h2, w2
    return big, strided


def test_embed_workspace_covers_the_largest_activation_at_every_input_size():
    """ctl_embed_forward ping-pongs five buffers of ctl_embed_workspace_bytes / 5 bytes, so each must hold the largest
    activation of the walk.  When the stem output has an odd side the max-pool rounds up, and layer1's output
    [n, ceil(h/2), ceil(w/2), 256] outgrows the stem's conv output; at tiny inputs the 2048-channel maps do."""
    import ctypes as C

    from ctl_b200 import _native as N

    L = N.lib()
    sides = np.arange(8, 401)
    H, W = np.meshgrid(sides, sides, indexing="ij")
    H, W = H.ravel(), W.ravel()
    for ibn in (0, 1):
        for last_stride in (1, 2):
            h = C.c_void_p()
            assert L.ctl_trunk_create(C.byref(h), ibn, last_stride) == 0
            try:
                got = np.array([L.ctl_embed_workspace_bytes(h, 1, int(a), int(b)) for a, b in zip(H, W)], dtype=np.int64)
                got3 = L.ctl_embed_workspace_bytes(h, 3, 300, 150)
            finally:
                L.ctl_trunk_destroy(h)
            need = 5 * 2 * _trunk_walk(H, W, last_stride)[0]
            bad = np.nonzero(got < need)[0]
            assert bad.size == 0, (
                f"ibn={ibn} last_stride={last_stride}: {bad.size} sizes under-sized, e.g. " +
                ", ".join(f"{H[i]}x{W[i]}: {got[i] // 5} bytes per buffer < {need[i] // 5}" for i in bad[:5]))
            assert got3 >= 3 * 5 * 2 * int(_trunk_walk(300, 150, last_stride)[0])  # the buffers scale with the batch


def test_train_workspace_rejects_exactly_the_sizes_training_cannot_run():
    """A training step needs an even input map at every stride-2 layer (weight gradient and zero-insertion data
    gradient); ctl_train_workspace_bytes is 0 for exactly the other sizes, and ctl_last_error() names the first such
    layer and its map size."""
    import ctypes as C

    from ctl_b200 import _native as N

    L = N.lib()
    sides = np.r_[32:80, 96, 126, 127, 128, 150, 160, 250, 256, 300, 320, 384, 400]
    for ibn in (0, 1):
        for last_stride in (1, 2):
            h = C.c_void_p()
            assert L.ctl_trainer_create(C.byref(h), ibn, last_stride, 0.1) == 0
            try:
                for H in sides:
                    for W in sides:
                        odd = [(name, a, b) for name, a, b in _trunk_walk(int(H), int(W), last_stride)[1] if a % 2 or b % 2]
                        got = L.ctl_train_workspace_bytes(h, 2, int(H), int(W))
                        assert (got == 0) == bool(odd), (ibn, last_stride, H, W, got, odd)
                        if odd:
                            msg = L.ctl_last_error().decode()
                            name, a, b = odd[0]
                            assert name in msg and f"{a}x{b}" in msg, (H, W, msg)
            finally:
                L.ctl_trainer_destroy(h)
            # 300x150: layer1 leaves a 75x38 map, which layer2.0 would subsample
            assert L.ctl_trainer_create(C.byref(h), ibn, last_stride, 0.1) == 0
            assert L.ctl_train_workspace_bytes(h, 4, 300, 150) == 0
            assert b"layer2.0.conv2" in L.ctl_last_error() and b"75x38" in L.ctl_last_error()
            L.ctl_trainer_destroy(h)
