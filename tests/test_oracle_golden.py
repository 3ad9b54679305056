"""CPU: the oracle restatement (oracle/ctl_oracle.py) against the golden vectors produced by
the UNMODIFIED reference (oracle/make_golden.py).  This is what pins the oracle."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import ctl_oracle as O
from oracle.make_golden import DIM, LOSS_CASES, NUM_CLASSES, checksum, head_state

RTOL = 1e-4  # north_star: fp32 embeddings / losses within 1e-4 relative


def _close(a, b, rtol=RTOL, atol=0.0):
    np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=rtol, atol=atol)


def test_masks_match_reference():
    g = load_golden("masks.npz")
    for name in ("even", "k16", "ragged"):
        masks, lists = O.create_masks_train(g[f"{name}_labels"])
        assert np.array_equal(masks, g[f"{name}_masks"])
        assert [len(x) for x in lists] == g[f"{name}_nlists"].tolist()


@pytest.mark.parametrize("name", list(LOSS_CASES))
def test_ctl_step_losses_match_reference(name):
    g = load_golden(f"loss_{name}.npz")
    P, K, pad, seed, scale = LOSS_CASES[name]
    feats, labels, is_real = O.synth_batch(P, K, DIM, NUM_CLASSES, seed, pad, scale)
    _close(checksum(feats), g["in_checksum"], 1e-12)
    assert np.array_equal(is_real.numpy(), g["is_real"])
    hs = head_state(seed)
    feats = feats.clone().requires_grad_(True)
    centers = hs["centers"].clone().requires_grad_(True)
    bn_w = hs["bn_weight"].clone().requires_grad_(True)
    fc_w = hs["fc_weight"].clone().requires_grad_(True)
    out = O.ctl_step_losses(feats, labels, is_real, K, centers, bn_w, hs["bn_bias"], fc_w)
    for key in ("total", "xent", "triplet", "center", "ctl", "dist_ap", "dist_an", "l2_centroid"):
        _close(float(out[key]), float(g[key]), 2e-5)
    out["total"].backward()
    gscale = np.abs(g["grad_feats"]).max()
    _close(feats.grad.numpy(), g["grad_feats"], 1e-4, 1e-5 * gscale)
    rows = torch.from_numpy(g["grad_centers_rows_idx"])
    # the reference rescales centers.grad by 1/CENTER_LOSS_WEIGHT (train_ctl_model.py:157-158)
    gc = centers.grad[rows].numpy() / 5e-4
    _close(gc, g["grad_centers_rows"], 1e-4, 1e-6 * np.abs(g["grad_centers_rows"]).max())
    _close(float(centers.grad.abs().sum()) / 5e-4, float(g["grad_centers_abs_sum"]), 1e-4)
    _close(bn_w.grad.numpy(), g["grad_bn_weight"], 1e-3, 1e-5 * np.abs(g["grad_bn_weight"]).max())
    _close(fc_w.grad[rows].numpy(), g["grad_fc_rows"], 1e-3, 1e-5 * np.abs(g["grad_fc_rows"]).max())


@pytest.mark.parametrize("name", ["small", "dyadic", "ties"])
def test_retrieval_small_match_reference(name):
    g = load_golden(f"retrieval_{name}.npz")
    nq, ng = int(g["num_q"]), int(g["num_g"])
    feats, pids, cams = O.synth_retrieval(nq, ng, int(g["num_ids"]), DIM, float(g["sigma"]), int(g["seed"]),
                                          dyadic=bool(g["dyadic"]))
    _close(checksum(feats), g["in_checksum"], 1e-12)
    d = O.get_euclidean(feats[:nq], feats[nq:]).numpy()
    if bool(g["dyadic"]):
        assert np.array_equal(d, g["dist"]), "dyadic fixtures are exact in fp32"
    else:
        _close(d, g["dist"], 1e-5, 1e-6)
    idx = O.rank_indices(g["dist"])
    k = g["topk_idx"].shape[1]
    assert np.array_equal(idx[:, :k], g["topk_idx"].astype(np.int64))
    cmc, mAP, topk, single = O.eval_func(idx, pids[:nq], pids[nq:], cams[:nq], cams[nq:], 50)
    assert np.array_equal(cmc, g["cmc"])
    _close(mAP, float(g["mAP"]), 1e-12)
    _close(topk, g["all_topk"], 1e-12)
    _close(single[:, 2].astype(np.float64), g["ap"], 1e-12)
    cd = O.get_cosine(feats[:nq], feats[nq:]).numpy()
    _close(cd, g["cos_dist"], 1e-5, 1e-6)
    ti, td = O.topk_similar(feats[:nq], feats[nq:], topk=k)
    if bool(g["dyadic"]):
        assert np.array_equal(ti, g["topk_idx"].astype(np.int64))
        assert np.array_equal(td, g["topk_dist"])


def test_centroids_match_reference():
    g = load_golden("centroids.npz")
    nq, ng = int(g["num_q"]), int(g["num_g"])
    feats, pids, cams = O.synth_retrieval(nq, ng, int(g["num_ids"]), DIM, 3.0, 11, num_cams=4)
    _close(checksum(feats), g["in_checksum"], 1e-12)
    for respect, tag in ((False, "nocam"), (True, "cam")):
        emb, lab, cam = O.validation_create_centroids(feats, pids, cams, nq, respect)
        _close(emb.numpy(), g[f"{tag}_emb"], 1e-6, 1e-7)
        assert np.array_equal(lab, g[f"{tag}_lab"])
        if respect:
            assert [len(c) for c in cam] == g[f"{tag}_cam_len"].tolist()
            assert np.concatenate([np.asarray(c) for c in cam]).tolist() == g[f"{tag}_cam_flat"].tolist()
        else:
            assert np.array_equal(cam, g[f"{tag}_cam"])
        cmc, mAP, topk = O.r1_map_compute(emb, lab, cam, nq, True, "euclidean", respect)
        assert np.array_equal(cmc, g[f"{tag}_cmc"])
        _close(mAP, float(g[f"{tag}_mAP"]), 1e-12)
        _close(topk, g[f"{tag}_topk"], 1e-12)
    pid_index = {}
    for i, p in enumerate(pids[nq:].tolist()):
        pid_index.setdefault(p, []).append(i)
    cents, cp = O.calculate_centroids_by_pid(feats[nq:].numpy(), pid_index)
    _close(cents, g["inf_centroids"], 1e-6, 1e-7)
    assert np.array_equal(cp, g["inf_pids"])


@pytest.mark.parametrize("tag,ibn,hw", [("r50", False, (256, 128)), ("ibn", True, (128, 64))])
def test_trunk_matches_reference(tag, ibn, hw):
    g = load_golden("trunk.npz")
    sd = O.make_trunk_state(seed=7, ibn=ibn)
    gen = torch.Generator().manual_seed(21)
    x = torch.randn(2, 3, *hw, generator=gen)
    _close(checksum(x), g[f"{tag}_in_checksum"], 1e-12)
    _close(checksum(torch.cat([v.flatten().float() for v in sd.values()])), g[f"{tag}_w_checksum"], 1e-12)
    with torch.no_grad():
        bo, gf = O.baseline_forward(x, sd, ibn=ibn, train=False)
        _, gft = O.baseline_forward(x, sd, ibn=ibn, train=True)
    _close(gf.numpy(), g[f"{tag}_eval_feat"], 1e-4, 1e-5)
    _close(checksum(bo), g[f"{tag}_eval_base_checksum"], 1e-5)
    _close(gft.numpy(), g[f"{tag}_train_feat"], 1e-4, 1e-5)


def test_retrieval_market_shape_matches_reference():
    """BASELINE config 3 (3368 x 15913 x 2048): the reference's own get_euclidean + stable
    argsort + eval_func outputs (102 s of its per-query python loop) vs the restatement."""
    g = load_golden("retrieval_market.npz")
    nq, ng = int(g["num_q"]), int(g["num_g"])
    feats, pids, cams = O.synth_retrieval(nq, ng, int(g["num_ids"]), DIM, float(g["sigma"]), int(g["seed"]))
    _close(checksum(feats), g["in_checksum"], 1e-12)
    d = O.get_euclidean(feats[:nq], feats[nq:]).numpy()
    idx = O.rank_indices(d)
    k = g["topk_idx"].shape[1]
    # same machine family, same torch -> the sgemm is bit-reproducible; if this ever fails on
    # another CPU compare epsilon-consistently instead (see tests/test_retrieval_gpu.py)
    same = (idx[:, :k] == g["topk_idx"].astype(np.int64)).mean()
    assert same > 0.999, same
    _close(np.take_along_axis(d, idx[:, :k], 1), g["topk_dist"], 1e-5, 1e-6)
    cmc, mAP, topk, single = O.eval_func(idx, pids[:nq], pids[nq:], cams[:nq], cams[nq:], 50)
    _close(cmc, g["cmc"], 0, 1e-3)
    _close(mAP, float(g["mAP"]), 1e-5)
    _close(topk, g["all_topk"], 0, 1e-3)
    assert np.array_equal(single[:, 0].astype(np.int32), g["valid_q"])


def test_oracle_augment_pinned_against_reference_random_erasing():
    """oracle.augment_batch (normalise + random erasing with given draws) against the reference's own RandomErasing
    class (datasets/transforms/random_erasing.py) driven by random.seed(seed) (tests/golden/random_erasing.npz,
    oracle/make_golden.py:gen_random_erasing)."""
    import math
    import random

    from oracle.make_golden import ERASE_MEAN, ERASE_SEEDS, ERASE_SHAPE, ERASE_STD, erase_input

    g = load_golden("random_erasing.npz")
    (H, W), pad = ERASE_SHAPE, 10
    img, _ = erase_input()
    assert np.array_equal(checksum(img), g["in_checksum"])
    for seed in range(ERASE_SEEDS):
        out_ref = torch.from_numpy(g["erased"][seed])
        random.seed(seed)  # replay the reference's draws to recover the rectangle
        random.uniform(0, 1)
        for _ in range(100):
            ta = random.uniform(0.02, 0.4) * H * W
            ar = random.uniform(0.3, 1 / 0.3)
            h, w = int(round(math.sqrt(ta * ar))), int(round(math.sqrt(ta / ar)))
            if w < W and h < H:
                x1, y1 = random.randint(0, H - h), random.randint(0, W - w)
                break
        got = O.augment_batch(img, np.array([[0, pad, pad, x1, y1, h, w, 1]]), ERASE_MEAN, ERASE_STD, pad)[0]
        assert torch.allclose(got, out_ref, rtol=0, atol=1e-6)


@pytest.mark.parametrize("tag,ibn", [("r50", False), ("ibn", True)])
def test_train_mode_oracle_pinned_against_reference_autograd(tag, ibn):
    """oracle.trunk_train_fp16sim with the storage rounding switched off IS the reference's train-mode trunk
    (batch-stat BN / IBN, autograd): features, sampled parameter gradients and running statistics against the
    reference code run in float64 (tests/golden/trunk_train.npz, oracle/make_golden.py:gen_trunk_train); with the rounding on
    (what the B200 engine is checked against) it stays within fp16 distance of the same numbers."""
    from oracle.make_golden import TRAIN_GRAD_KEYS, grad_sample

    gd = load_golden("trunk_train.npz")
    sd = O.make_trunk_state(seed=17, ibn=ibn)
    g = torch.Generator().manual_seed(23)
    x = torch.randn(4, 3, 64, 32, generator=g)
    dfeat = torch.randn(4, 2048, generator=g) * 1e-2
    assert np.array_equal(gd[f"{tag}_in_checksum"], checksum(torch.cat((x.flatten(), dfeat.flatten()))))
    keys = [k.format(bn="BN." if ibn else "") for k in TRAIN_GRAD_KEYS] + (["layer1.0.bn1.IN.weight"] if ibn else [])
    for rnd, tol in ((False, 6e-3 if ibn else 1e-7), (True, 1e-1)):  # the IBN golden is an fp32 run (see make_golden)
        feat, grads, running = O.trunk_train_fp16sim(x, sd, dfeat, ibn=ibn, round_fp16=rnd)
        ref = gd[f"{tag}_feat"]
        assert np.abs(feat.numpy() - ref).max() <= (tol if not rnd else 5e-3) * np.abs(ref).max()
        for k in keys:
            got, exp = grad_sample(grads[k]), gd[f"{tag}_grad_{k}"]
            scale = np.abs(exp[:-2]).max()
            if not rnd and not ibn:
                assert np.abs(got[:-2] - exp[:-2]).max() <= tol * scale, k
                assert abs(got[-1] - exp[-1]) <= tol * exp[-1], k
            elif not rnd:
                # fp32 golden: a handful of ReLU masks flip against the float64 oracle (isolated elements off by a few
                # per cent), everything else agrees to fp32 round-off
                err = np.abs(got[:-2] - exp[:-2])
                cos = float(np.dot(got[:-2], exp[:-2]) / (np.linalg.norm(got[:-2]) * np.linalg.norm(exp[:-2])))
                assert np.quantile(err, 0.99) <= tol * scale and cos >= 0.9995 and abs(got[-1] / exp[-1] - 1) <= tol, (k, cos)
            else:  # ReLU masks flip under fp16 rounding: direction and size only
                cos = float(np.dot(got[:-2], exp[:-2]) / (np.linalg.norm(got[:-2]) * np.linalg.norm(exp[:-2])))
                assert cos >= 0.97 and abs(got[-1] / exp[-1] - 1) <= tol, (k, cos)
        for k in ("bn1.running_mean", "layer4.2.bn3.running_var"):
            np.testing.assert_allclose(running[k].numpy(), gd[f"{tag}_run_{k}"], rtol=5e-3 if (rnd or ibn) else 1e-6, atol=1e-5 if (rnd or ibn) else 1e-9)


@pytest.mark.parametrize("tag,ibn,hw", [("r50", False, (256, 128)), ("ibn", True, (128, 64))])
def test_fp16sim_checker_pinned_against_reference_under_autocast(tag, ibn, hw):
    """The builder's same-precision checker (trunk_forward_fp16sim: fp16 operands, BN folded into fp16 weights, fp16
    activations) is itself pinned against the UNMODIFIED reference run under fp16 autocast
    (tests/golden/trunk_autocast.npz): it must sit as close to the reference-under-autocast as the reference's own fp16
    run sits to its fp32 run (a few 1e-4 of the feature scale), i.e. it is a fair stand-in at sizes the goldens do not
    cover."""
    g = load_golden("trunk_autocast.npz")
    sd = O.make_trunk_state(seed=7, ibn=ibn)
    x = torch.randn(2, 3, *hw, generator=torch.Generator().manual_seed(21))
    np.testing.assert_allclose(checksum(x), g[f"{tag}_in_checksum"], rtol=1e-9)
    with torch.no_grad():
        _, sim = O.trunk_forward_fp16sim(x, sd, ibn=ibn)
    amp, f32 = torch.from_numpy(g[f"{tag}_eval_feat_amp"]), torch.from_numpy(g[f"{tag}_eval_feat_fp32"])
    scale = float(f32.abs().max())
    d_amp = float((sim - amp).abs().max()) / scale
    d_f32 = float((sim - f32).abs().max()) / scale
    print(f"{tag}: fp16sim vs reference-autocast {d_amp:.3e}, vs reference fp32 {d_f32:.3e}, "
          f"reference autocast vs fp32 {float(g[f'{tag}_amp_vs_fp32']):.3e}")
    assert d_amp <= 2e-3 and d_f32 <= 2e-3
