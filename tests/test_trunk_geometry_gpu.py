"""GPU: the eval trunk at input sizes whose feature maps go odd at a stride-2 layer (torch.nn.Conv2d and MaxPool2d round
the output up: a 300x150 crop leaves layer1 at 75x38, 8x8 shrinks to 1x1 maps).  The bench shapes keep every map even;
these points exercise the parity views of odd sides (csrc/conv.cu: encode_source), the empty views of 1-pixel maps, the
fused stem with an odd stem width and the workspace sizing of ctl_embed_forward.

Checkers as in test_trunk_gpu.py::test_full_trunk_matches_checker_and_reference_golden: oracle.trunk_forward_fp16sim
within 3e-3 of the feature scale; the unmodified reference's fp32 features (tests/golden/trunk_geometry.npz) within
1e-2.  Every other path -- the C-ABI handle, the uint8 entry, a single image, a CUDA-graph replay -- must agree with
TrunkEngine bit for bit."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from oracle import ctl_oracle as O
from oracle.make_golden import TRUNK_GEOMETRY_CASES, checksum, trunk_geometry_input

pytestmark = pytest.mark.gpu

SWEEP = [  # ibn, MODEL.LAST_STRIDE, (H, W)
    (False, 1, (300, 150)),
    (False, 2, (260, 102)),   # fused stem (H % 4 == 0, W <= 128) with a 51-pixel-wide stem output
    (True, 1, (250, 125)),
    (False, 2, (224, 112)),   # even until layer4: 14x7
    (True, 2, (100, 50)),
    (False, 2, (8, 8)),       # 1x1 maps from layer2 on: stride-2 layers over a single pixel
    (True, 1, (36, 20)),
]


def _tag(ibn, last_stride, hw):
    return f"{'ibn' if ibn else 'r50'}_s{last_stride}_{hw[0]}x{hw[1]}"


def _head():
    g = torch.Generator().manual_seed(3)
    return dict(weight=torch.rand(2048, generator=g) + 0.5, bias=torch.randn(2048, generator=g) * 0.1,
                running_mean=torch.randn(2048, generator=g) * 0.1, running_var=torch.rand(2048, generator=g) + 0.5)


@pytest.mark.parametrize("ibn,last_stride,hw", SWEEP, ids=[_tag(*c) for c in SWEEP])
def test_trunk_at_odd_geometry(ibn, last_stride, hw):
    from ctl_b200 import _native as N
    from ctl_b200.datasets.transforms import normalize_batch
    from ctl_b200.modelling.backbones.engine import GraphedForward, NativeTrunk, TrunkEngine

    tag = _tag(ibn, last_stride, hw)
    sd, x = trunk_geometry_input(ibn, hw)
    n = x.shape[0]
    head = _head()
    eng = TrunkEngine(sd, "cuda", ibn=ibn, last_stride=last_stride, bn_head=head)
    xd = x.cuda()
    out = eng.forward(xd, want_emb=True)
    feat, emb = out["global_feat"].clone(), out["emb"].clone()
    assert torch.isfinite(feat).all() and torch.isfinite(emb).all()

    # same-precision checker and the reference's own fp32 features
    with torch.no_grad():
        _, sim = O.trunk_forward_fp16sim(x, sd, last_stride=last_stride, ibn=ibn)
    scale = float(sim.abs().max())
    err_sim = float((feat.cpu() - sim).abs().max())
    print(f"{tag}: |feat|max {scale:.4f}  err vs fp16-sim {err_sim:.3e}")
    assert err_sim <= 3e-3 * scale, f"{tag}: {err_sim:.3e} vs fp16-sim (scale {scale:.4f})"
    if tag in TRUNK_GEOMETRY_CASES:
        g = load_golden("trunk_geometry.npz")
        np.testing.assert_allclose(checksum(x[:2]), g[f"{tag}_in_checksum"], rtol=1e-9)
        np.testing.assert_allclose(checksum(torch.cat([v.flatten().float() for v in sd.values()])),
                                   g[f"{tag}_w_checksum"], rtol=1e-9)
        err_ref = float((feat[:2].cpu() - torch.from_numpy(g[f"{tag}_eval_feat"])).abs().max())
        print(f"{tag}: err vs fp32 reference {err_ref:.3e}")
        assert err_ref <= 1e-2 * scale, f"{tag}: {err_ref:.3e} vs the reference's fp32 features"
    emb_ref = F.batch_norm(feat.cpu(), head["running_mean"], head["running_var"], head["weight"], head["bias"], False, 0.1,
                           1e-5)
    np.testing.assert_allclose(emb.cpu().numpy(), emb_ref.numpy(), rtol=1e-5, atol=1e-5)

    # the C-ABI handle: same bits, and nothing written past the workspace it asked for
    nat = NativeTrunk(sd, "cuda", ibn=ibn, last_stride=last_stride, bn_head=head)
    got = nat.forward(xd, want_emb=True)
    assert torch.equal(got["global_feat"], feat) and torch.equal(got["emb"], emb), f"{tag}: NativeTrunk differs"
    L = N.lib()
    need = L.ctl_embed_workspace_bytes(nat._h, n, *hw)
    canary = 1 << 20
    ws = torch.full((need + canary,), 0xA5, dtype=torch.uint8, device="cuda")
    f2, e2 = torch.empty(n, 2048, device="cuda"), torch.empty(n, 2048, device="cuda")
    N.check(L.ctl_embed_forward(nat._h, xd.data_ptr(), n, hw[0], hw[1], f2.data_ptr(), e2.data_ptr(), ws.data_ptr(), need,
                                N.stream_ptr()))
    torch.cuda.synchronize()
    tail = ws[need:]
    assert bool((tail == 0xA5).all()), f"{tag}: {int((tail != 0xA5).sum())} bytes written past the advertised workspace"
    assert torch.equal(f2, feat) and torch.equal(e2, emb)

    # uint8 entry == normalize_batch + forward
    img = torch.randint(0, 256, (n, *hw, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(4)).cuda()
    a, b = eng.forward_u8(img, want_emb=True), eng.forward(normalize_batch(img), want_emb=True)
    assert torch.equal(a["global_feat"], b["global_feat"]) and torch.equal(a["emb"], b["emb"]), f"{tag}: forward_u8 differs"

    # batch invariance: image i of the batch == image i run alone
    for i in range(n):
        one = eng.forward(xd[i:i + 1].contiguous(), want_emb=True)
        assert torch.equal(one["global_feat"][0], feat[i]) and torch.equal(one["emb"][0], emb[i]), f"{tag}: image {i}"

    # one CUDA-graph replay == eager
    graphed = GraphedForward(eng, xd, want_emb=True)()
    assert torch.equal(graphed["global_feat"], feat) and torch.equal(graphed["emb"], emb), f"{tag}: graph replay differs"

