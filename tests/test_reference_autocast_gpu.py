"""Same-precision parity AT THE BENCH SHAPES against the UNMODIFIED reference executed on a B200.

The reference's own trunk modules (modelling/backbones/resnet.py:122-133, resnet_ibn_a.py:126-141,
modelling/baseline.py:91-96) were run on a CUDA device under ``torch.autocast(dtype=float16)`` -- the precision the
reference's configs train and validate at (USE_MIXED_PRECISION -> PL native AMP, utils/misc.py:111) -- and in fp32 by
``oracle/make_golden.py --only ref_cuda_autocast``; tests/golden/ref_cuda_autocast_*.npz hold what they produced and are
the checker for

  * the eval embedding at metric M1's configuration (256 crops of 256x128, ResNet50) and at config 4's per-GPU eval shape
    (128 crops of 320x320, ResNet50-IBN-a): every image on a fixed sample of 32 feature channels, tolerance 2e-3 of the
    full feature scale (two correct fp16 evaluations of this network differ by a few 1e-4; north_star's 1e-4 is an
    fp32-vs-fp32 bound and the reference's own autocast run is 4-7e-4 away from its fp32 run,
    tests/golden/trunk_autocast.npz);
  * one training step at config 2's shape (16 ids x 16 instances of 256x128) and config 4's per-GPU shape (32 x 4 of
    320x320, IBN-a): train-mode features within 2e-2, every parameter gradient by direction and size (cosine >= 0.95 against
    BOTH the reference's autocast and fp32 gradients on a strided sample of at most 128 elements per tensor -- the whole
    tensor for the 64- and 128-channel norm parameters; measured 0.968-0.973 at worst, on layer1's 64-channel norm
    biases; sampling moves the cosine of a larger tensor by < 0.01 --, full-tensor norm within 6 %: ReLU masks make
    element-wise comparison of two fp16 backward passes meaningless).
"""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle.make_golden import (AUTOCAST_GRAD_SAMPLE, AUTOCAST_LOSS_SCALE, autocast_eval_input, autocast_train_input,
                                checksum, golden_name, grad_sample)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("tag,ibn,hw,bs", [("r50", False, (256, 128), 256), ("ibn", True, (320, 320), 128)])
def test_eval_embedding_at_bench_shape_vs_reference_cuda_autocast(tag, ibn, hw, bs):
    from ctl_b200.modelling.backbones.engine import TrunkEngine

    g = load_golden("ref_cuda_autocast_eval.npz")
    sd, x = autocast_eval_input(ibn, hw, bs)
    assert np.array_equal(checksum(x), g[f"{tag}_in_checksum"])
    feat = TrunkEngine(sd, "cuda", ibn=ibn).forward(x.cuda())["global_feat"].cpu()
    assert torch.isfinite(feat).all()
    feat = feat[:, torch.from_numpy(g["cols"])]
    amp = torch.from_numpy(g[f"{tag}_feat_amp"]).float()
    f32 = amp + torch.from_numpy(g[f"{tag}_feat_fp32_minus_amp"]).float()
    scale, own = float(g[f"{tag}_scale"]), float(g[f"{tag}_amp_vs_fp32"])
    e_amp = float((feat - amp).abs().max()) / scale
    e_f32 = float((feat - f32).abs().max()) / scale
    print(f"{tag} bs {bs} {hw}: engine vs reference CUDA-autocast {e_amp:.3e}; engine vs reference fp32 {e_f32:.3e}; "
          f"reference CUDA-autocast vs its own fp32 {own:.3e}")
    assert e_amp <= 2e-3
    assert e_f32 <= max(3.0 * own, 1.5e-3)


@pytest.mark.parametrize("tag,ibn,hw,P,K", [("r50 cfg2", False, (256, 128), 16, 16), ("ibn cfg4/gpu", True, (320, 320), 32, 4)])
def test_training_step_at_bench_shape_vs_reference_cuda_autocast(tag, ibn, hw, P, K):
    from ctl_b200.modelling.backbones.engine_train import TrunkTrainer

    g = load_golden(f"ref_cuda_autocast_train_{golden_name(tag)}.npz")
    sd, x, dfeat = autocast_train_input(ibn, hw, P * K)
    assert np.array_equal(checksum(torch.cat((x.flatten(), dfeat.flatten()))), g["in_checksum"])
    params = {k: v.clone().cuda() for k, v in sd.items() if v.is_floating_point()}
    tr = TrunkTrainer("cuda", grad_scale=AUTOCAST_LOSS_SCALE, ibn=ibn)
    feat = tr.forward(x.cuda(), params)
    grads = tr.backward(dfeat.cuda())
    torch.cuda.synchronize()
    feat = feat.cpu()[:, torch.from_numpy(g["cols"])]
    e = float((feat - torch.from_numpy(g["feat_amp"]).float()).abs().max()) / float(g["feat_scale"])

    def cos(a_, b_):
        return float(np.dot(a_, b_) / (np.linalg.norm(a_) * np.linalg.norm(b_) + 1e-300))

    worst_cos, worst_norm, unresolved = (1.0, None), (0.0, None), []
    for k, rn, rn32, own_cos, ra, rf in zip(g["keys"].tolist(), g["norm_amp"], g["norm_fp32"], g["cos_amp_fp32"],
                                           g["grad_amp"].astype(np.float64), g["grad_fp32"].astype(np.float64)):
        gk = grads[k].double().cpu()
        assert torch.isfinite(gk).all(), k
        gk_norm = float(gk.norm())
        if own_cos < 0.9:  # the reference under autocast does not reproduce its own fp32 gradient here
            unresolved.append(k)
            partner = grads.get(k[:-4] + "weight") if k.endswith("bias") else None
            bound = 3.0 * max(rn, rn32) + (2e-2 * float(partner.double().norm()) if partner is not None else 0.0)
            assert gk_norm <= bound + 1e-12, (k, gk_norm, bound)  # round-off sized, like the reference's
            continue
        gs = grad_sample(gk, AUTOCAST_GRAD_SAMPLE)[:-2]
        c = min(cos(gs, ra[:len(gs)]), cos(gs, rf[:len(gs)]))
        nr = abs(gk_norm / rn - 1)
        if c < worst_cos[0]:
            worst_cos = (c, k)
        if nr > worst_norm[0]:
            worst_norm = (nr, k)
    print(f"{tag}: gradients the reference's own autocast run does not resolve (cos < 0.9 vs its fp32 run): {unresolved}")
    assert len(unresolved) <= 4, unresolved
    print(f"{tag}: train features vs reference CUDA-autocast {e:.3e}; worst gradient cosine {worst_cos[0]:.4f} "
          f"({worst_cos[1]}), worst norm deviation {worst_norm[0]:.3e} ({worst_norm[1]}) over {len(g['keys'])} tensors")
    assert e <= 2e-2
    assert worst_cos[0] >= 0.95, worst_cos
    assert worst_norm[0] <= 6e-2, worst_norm
