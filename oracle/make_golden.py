"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED
reference (/root/reference, through oracle/ref_import.py) on seeded synthetic inputs.

    python -m oracle.make_golden [--only loss,retrieval,trunk,trunk_train,trunk_autocast,trunk_geometry,masks,...]
    python -m oracle.make_golden --only ref_cuda_autocast      (on a CUDA device: the reference at the bench shapes)

The reference has no tests and no golden vectors of its own (SURVEY.md section 4); these
files are what pins the oracle restatement (oracle/ctl_oracle.py) and, through it, the
CUDA path.  Inputs are regenerated from seeds by the shared generators in ctl_oracle
(`synth_batch`, `synth_retrieval`, `make_trunk_state`); every file stores an input checksum
so RNG drift is detected rather than silently compared against.
"""
from __future__ import annotations

import argparse
import os
import sys
import time
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ctl_oracle as O  # noqa: E402
from oracle.ref_import import default_cfg, load_reference  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

LOSS_CASES = {
    # name: (P, K, pad_fraction, seed, scale)
    "p8k4_real": (8, 4, 0.0, 1, 1.0),
    "p8k4_pad": (8, 4, 0.4, 2, 1.0),
    "p16k16_real": (16, 16, 0.0, 3, 0.5),
    "p16k16_pad": (16, 16, 0.25, 4, 0.5),
    "p32k4_pad": (32, 4, 0.25, 5, 1.0),
}
NUM_CLASSES = 751
DIM = 2048


def checksum(t):
    t = torch.as_tensor(t).double()
    return np.array([float(t.sum()), float((t * t).sum())])


class _FixedTrunk(torch.nn.Module):
    """Stands in for Baseline so that training_step sees a prescribed feature matrix."""

    def __init__(self, feats):
        super().__init__()
        self.feats = torch.nn.Parameter(feats.clone())

    def forward(self, x):
        return None, self.feats


class _Trainer:
    current_epoch = 100  # past warm-up; the LR rule is not part of the arithmetic under test


def head_state(seed, num_classes=NUM_CLASSES, dim=DIM):
    g = torch.Generator().manual_seed(1000 + seed)
    return dict(
        centers=torch.randn(num_classes, dim, generator=g),
        bn_weight=0.5 + torch.rand(dim, generator=g),
        bn_bias=torch.zeros(dim),
        fc_weight=0.02 * torch.randn(num_classes, dim, generator=g),
    )


# TripletLoss variants reachable through the config (SOLVER.DISTANCE_FUNC = 'cosine'; margin None -> SoftMarginLoss,
# losses/triplet_loss.py:127-137): name -> (base case, SOLVER overrides)
LOSS_VARIANTS = {
    "p8k4_pad_cosine": ("p8k4_pad", {"DISTANCE_FUNC": "cosine"}),
    "p8k4_pad_softmargin": ("p8k4_pad", {"MARGIN": None}),
}


def gen_loss(ref, variants=False):
    cases = {k: (LOSS_CASES[b], o) for k, (b, o) in LOSS_VARIANTS.items()} if variants else \
        {k: (v, {}) for k, v in LOSS_CASES.items()}
    for name, ((P, K, pad, seed, scale), solver_over) in cases.items():
        feats, labels, is_real = O.synth_batch(P, K, DIM, NUM_CLASSES, seed, pad, scale)
        hs = head_state(seed)
        cfg = default_cfg(ref)
        cfg.DATALOADER.NUM_INSTANCE = K
        for k_, v_ in solver_over.items():
            cfg.SOLVER[k_] = v_
        model = ref.train_ctl.CTLModel(cfg, num_classes=NUM_CLASSES, num_query=1)
        model.backbone = _FixedTrunk(feats)
        with torch.no_grad():
            model.center_loss.centers.copy_(hs["centers"])
            model.bn.weight.copy_(hs["bn_weight"])
            model.bn.bias.copy_(hs["bn_bias"])
            model.fc_query.weight.copy_(hs["fc_weight"])
        model.trainer = _Trainer()
        params = [p for n, p in model.named_parameters() if "center" not in n and p.requires_grad]
        opt = torch.optim.SGD(params, lr=0.0)
        opt_c = torch.optim.SGD(model.center_loss.parameters(), lr=0.0)
        model._ctl_optimizers = (opt, opt_c)
        model.train()
        x = torch.zeros(P * K, 3, 8, 8)
        cam = torch.zeros(P * K, dtype=torch.long)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out = model.training_step((x, labels, cam, is_real), 0)
        parts = {n: model.losses_dict[n][-1] for n in model.losses_names}
        np.savez_compressed(
            os.path.join(GOLD, f"loss_{name}.npz"),
            P=P, K=K, pad=pad, seed=seed, scale=scale,
            in_checksum=checksum(feats),
            is_real=is_real.numpy(),
            labels=labels.numpy(),
            total=float(out["loss"]),
            xent=parts["query_xent"], triplet=parts["query_triplet"],
            center=parts["query_center"], ctl=parts["centroid_triplet"],
            dist_ap=out["other"]["step_dist_ap"], dist_an=out["other"]["step_dist_an"],
            l2_centroid=out["other"]["l2_mean_centroid"],
            grad_feats=model.backbone.feats.grad.numpy(),
            # NB: after training_step the reference has multiplied centers.grad by
            # 1/CENTER_LOSS_WEIGHT (train_ctl_model.py:157-158); stored as seen by opt_center.
            grad_centers_rows=model.center_loss.centers.grad[labels.unique()].numpy(),
            grad_centers_rows_idx=labels.unique().numpy(),
            grad_centers_abs_sum=float(model.center_loss.centers.grad.abs().sum()),
            grad_bn_weight=model.bn.weight.grad.numpy(),
            grad_fc_rows=model.fc_query.weight.grad[labels.unique()].numpy(),
            grad_fc_checksum=checksum(model.fc_query.weight.grad),
            bn_running_mean=model.bn.running_mean.numpy(),
            bn_running_var=model.bn.running_var.numpy(),
        )
        print(f"loss_{name}: total={float(out['loss']):.6f} parts={parts}")


def gen_masks(ref):
    cases = {
        "even": np.repeat(np.arange(5), 4),
        "k16": np.repeat(np.array([7, 3, 9]), 16),
        "ragged": np.array([4, 4, 4, 2, 2, 9, 9, 9, 9, 1, 1]),
    }
    out = {}
    for name, labels in cases.items():
        masks, labels_list = ref.bases.ModelBase.create_masks_train(torch.from_numpy(labels))
        out[f"{name}_labels"] = labels
        out[f"{name}_masks"] = masks.numpy()
        out[f"{name}_nlists"] = np.array([len(x) for x in labels_list])
    np.savez_compressed(os.path.join(GOLD, "masks.npz"), **out)
    print("masks done")


def _ref_eval(ref, distmat, q_pids, g_pids, q_cam, g_cam, respect=False):
    idx = np.argsort(distmat, axis=1, kind="stable")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        cmc, mAP, topk, single = ref.eval_reid.eval_func(idx, q_pids, g_pids, q_cam, g_cam, 50, respect)
    return idx, cmc, mAP, topk, single


def gen_retrieval(ref, name, num_q, num_g, num_ids, sigma, seed, dyadic=False, store_dist=True, topk=100):
    feats, pids, cams = O.synth_retrieval(num_q, num_g, num_ids, DIM, sigma, seed, dyadic=dyadic)
    qf, gf = feats[:num_q], feats[num_q:]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        t0 = time.time()
        dist = ref.reid_metric.get_euclidean(qf, gf).numpy()
        cosd = ref.reid_metric.get_cosine(qf, gf).numpy() if num_q * num_g <= 1 << 20 else None
    t1 = time.time()
    idx, cmc, mAP, topk_hits, single = _ref_eval(ref, dist, pids[:num_q], pids[num_q:], cams[:num_q], cams[num_q:])
    t2 = time.time()
    k = min(topk, num_g)
    idt = np.int16 if num_g < 32768 else np.int32
    data = dict(
        num_q=num_q, num_g=num_g, num_ids=num_ids, sigma=sigma, seed=seed, dyadic=dyadic,
        in_checksum=checksum(feats),
        topk_idx=idx[:, :k].astype(idt),
        topk_dist=np.take_along_axis(dist, idx[:, :k], 1),
        cmc=cmc, mAP=mAP, all_topk=topk_hits, ap=single[:, 2].astype(np.float64),
        valid_q=single[:, 0].astype(np.int32),
        t_dist=t1 - t0, t_eval=t2 - t1,
    )
    if store_dist:
        data["dist"] = dist
        if cosd is not None:
            data["cos_dist"] = cosd
            ci = np.argsort(cosd, axis=1, kind="stable")
            data["cos_topk_idx"] = ci[:, :k].astype(idt)
    np.savez_compressed(os.path.join(GOLD, f"retrieval_{name}.npz"), **data)
    print(f"retrieval_{name}: mAP={mAP:.6f} r1={cmc[0]:.4f} dist {t1-t0:.2f}s eval {t2-t1:.2f}s")


def gen_centroids(ref):
    num_q, num_g, num_ids = 160, 1200, 80
    feats, pids, cams = O.synth_retrieval(num_q, num_g, num_ids, DIM, 3.0, 11, num_cams=4)
    cfg = default_cfg(ref)
    model = ref.train_ctl.CTLModel(cfg, num_classes=NUM_CLASSES, num_query=num_q)
    out = {"in_checksum": checksum(feats), "num_q": num_q, "num_g": num_g, "num_ids": num_ids}
    for respect in (False, True):
        emb, lab, cam = model.validation_create_centroids(feats, pids, cams, respect_camids=respect)
        tag = "cam" if respect else "nocam"
        out[f"{tag}_emb"] = emb.numpy()
        out[f"{tag}_lab"] = np.asarray(lab)
        if respect:
            out[f"{tag}_cam_len"] = np.array([len(c) for c in cam])
            out[f"{tag}_cam_flat"] = np.concatenate([np.asarray(c) for c in cam])
            cam_arr = np.empty(len(cam), dtype=object)
            for i, c in enumerate(cam):
                cam_arr[i] = c
        else:
            out[f"{tag}_cam"] = np.asarray(cam)
            cam_arr = np.asarray(cam)
        # downstream metric on the centroid set (R1_mAP.compute internals, reid_metric.py:112-136)
        f = torch.nn.functional.normalize(emb.float(), dim=1, p=2)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            dist = ref.reid_metric.get_euclidean(f[:num_q], f[num_q:]).numpy()
            idx = np.argsort(dist, axis=1, kind="stable")
            cmc, mAP, topk, single = ref.eval_reid.eval_func(
                idx, np.asarray(lab[:num_q]), np.asarray(lab[num_q:]), cam_arr[:num_q], cam_arr[num_q:], 50, respect)
        out[f"{tag}_cmc"], out[f"{tag}_mAP"], out[f"{tag}_topk"] = cmc, mAP, topk
        out[f"{tag}_ap"] = single[:, 2].astype(np.float64)
        print(f"centroids {tag}: n_cent={emb.shape[0]-num_q} mAP={mAP:.6f}")
    # inference_utils.calculate_centroids (inference/inference_utils.py:147-159)
    pid_index = {}
    for i, p in enumerate(pids[num_q:].tolist()):
        pid_index.setdefault(p, []).append(i)
    cents, cp = ref.inference_utils.calculate_centroids(feats[num_q:].numpy(), pid_index)
    out["inf_centroids"], out["inf_pids"] = cents, np.asarray(cp)
    np.savez_compressed(os.path.join(GOLD, "centroids.npz"), **out)


def gen_trunk(ref):
    out = {}
    for ibn, mname, hw in ((False, "resnet50", (256, 128)), (True, "resnet50_ibn_a", (128, 64))):
        tag = "ibn" if ibn else "r50"
        sd = O.make_trunk_state(seed=7, ibn=ibn)
        cfg = default_cfg(ref)
        cfg.MODEL.NAME = mname
        base = ref.baseline.Baseline(cfg)
        base.base.load_state_dict(sd, strict=True)
        g = torch.Generator().manual_seed(21)
        x = torch.randn(2, 3, *hw, generator=g)
        base.eval()
        with torch.no_grad():
            bo, gf = base(x)
        out[f"{tag}_in_checksum"] = checksum(x)
        out[f"{tag}_w_checksum"] = checksum(torch.cat([v.flatten().float() for v in sd.values()]))
        out[f"{tag}_eval_feat"] = gf.numpy()
        out[f"{tag}_eval_base_checksum"] = checksum(bo)
        base.train()
        with torch.no_grad():
            _, gft = base(x)
        out[f"{tag}_train_feat"] = gft.numpy()
        print(f"trunk {tag}: feat mean {float(gf.mean()):.5f} std {float(gf.std()):.5f}")
    np.savez_compressed(os.path.join(GOLD, "trunk.npz"), **out)


# Eval trunk at input sizes whose feature maps go odd at some stride-2 layer (torch.nn.Conv2d rounds the output up):
# tag -> (ibn, MODEL.LAST_STRIDE, (H, W)).  tests/test_trunk_geometry_gpu.py sweeps more points; these four are pinned.
TRUNK_GEOMETRY_CASES = {
    "r50_s1_300x150": (False, 1, (300, 150)),
    "r50_s2_260x102": (False, 2, (260, 102)),
    "ibn_s1_250x125": (True, 1, (250, 125)),
    "ibn_s2_100x50": (True, 2, (100, 50)),
}


def trunk_geometry_input(ibn, hw, n=3):
    """Trunk weights and an n-image batch of one geometry point (the golden keeps the first two images)."""
    return O.make_trunk_state(seed=7, ibn=ibn), torch.randn(n, 3, *hw, generator=torch.Generator().manual_seed(31))


def gen_trunk_geometry(ref):
    """The reference's eval trunk (Baseline, fp32, CPU) at TRUNK_GEOMETRY_CASES: global_feat of two images."""
    out = {}
    for tag, (ibn, last_stride, hw) in TRUNK_GEOMETRY_CASES.items():
        sd, x = trunk_geometry_input(ibn, hw)
        x = x[:2]
        cfg = default_cfg(ref)
        cfg.MODEL.NAME = "resnet50_ibn_a" if ibn else "resnet50"
        cfg.MODEL.LAST_STRIDE = last_stride
        base = ref.baseline.Baseline(cfg)
        base.base.load_state_dict(sd, strict=True)
        base.eval()
        with torch.no_grad():
            _, gf = base(x)
        out[f"{tag}_in_checksum"] = checksum(x)
        out[f"{tag}_w_checksum"] = checksum(torch.cat([v.flatten().float() for v in sd.values()]))
        out[f"{tag}_eval_feat"] = gf.float().numpy()
        print(f"trunk geometry {tag}: feat mean {float(gf.mean()):.5f} std {float(gf.std()):.5f}")
    np.savez_compressed(os.path.join(GOLD, "trunk_geometry.npz"), **out)


TRAIN_GRAD_KEYS = ("conv1.weight", "bn1.weight", "layer1.0.conv2.weight", "layer1.0.bn1.{bn}weight", "layer2.0.downsample.0.weight",
                   "layer3.2.conv1.weight", "layer4.2.conv3.weight", "layer4.2.bn3.weight", "layer4.2.bn3.bias")


def grad_sample(t, n=4096):
    """<= n evenly strided elements of a gradient, followed by its sum and its absolute sum (keeps the fixture small)."""
    f = t.detach().flatten().double()
    stride = max(1, f.numel() // n)
    return torch.cat((f[::stride][:n], f.sum()[None], f.abs().sum()[None])).numpy()


def gen_trunk_train(ref):
    """The reference's own trunk in TRAIN mode (batch-statistics BatchNorm, IBN) under torch autograd on the CPU
    (float64 for the plain ResNet; fp32 for IBN-a, whose InstanceNorm over 8 positions amplifies fp32 round-off to
    ~3e-3): global_feat, a sample of parameter gradients of
    sum(global_feat * dfeat), and updated running statistics."""
    out = {}
    for ibn, mname in ((False, "resnet50"), (True, "resnet50_ibn_a")):
        tag = "ibn" if ibn else "r50"
        sd = O.make_trunk_state(seed=17, ibn=ibn)
        cfg = default_cfg(ref)
        cfg.MODEL.NAME = mname
        base = ref.baseline.Baseline(cfg)
        base.base.load_state_dict(sd, strict=True)
        # plain ResNet: float64 run of the same code; IBN-a casts its InstanceNorm input to fp32 itself
        # (resnet_ibn_a.py:29), so that variant can only run in fp32
        dt = torch.float32 if ibn else torch.float64
        base.to(dt).train()
        g = torch.Generator().manual_seed(23)
        x = torch.randn(4, 3, 64, 32, generator=g)
        dfeat = torch.randn(4, 2048, generator=g) * 1e-2
        _, feat = base(x.to(dt))
        (feat * dfeat.to(dt)).sum().backward()
        params = dict(base.base.named_parameters())
        out[f"{tag}_in_checksum"] = checksum(torch.cat((x.flatten(), dfeat.flatten())))
        out[f"{tag}_feat"] = feat.detach().numpy()
        for key in TRAIN_GRAD_KEYS:
            k = key.format(bn="BN." if ibn else "")
            out[f"{tag}_grad_{k}"] = grad_sample(params[k].grad)
        if ibn:
            out[f"{tag}_grad_layer1.0.bn1.IN.weight"] = grad_sample(params["layer1.0.bn1.IN.weight"].grad)
        bufs = dict(base.base.named_buffers())
        for k in ("bn1.running_mean", "layer4.2.bn3.running_var"):
            out[f"{tag}_run_{k}"] = bufs[k].numpy()
        print(f"trunk train {tag}: feat std {float(feat.std()):.4f}, |dW conv1| {float(params['conv1.weight'].grad.abs().max()):.4e}")
    np.savez_compressed(os.path.join(GOLD, "trunk_train.npz"), **out)


def gen_trunk_autocast(ref):
    """The reference's own trunk at the precision its configs actually run at: torch fp16 autocast
    (USE_MIXED_PRECISION -> PL native AMP, utils/misc.py:111), executed here with the CPU autocast backend (fp16 conv /
    linear outputs, fp32 BatchNorm statistics, IBN's InstanceNorm in fp32 by its own cast, resnet_ibn_a.py:29).
    Eval: R50 2x256x128 (the inputs of trunk.npz), IBN-a 2x320x320 (config 4 geometry) and 2x128x64, each stored next to
    the fp32 run of the same module so that the reference's OWN fp16-vs-fp32 distance is on record.
    Train: R50 / IBN-a 4x64x32 (the inputs of trunk_train.npz), features and a sample of parameter gradients of
    sum(feat * dfeat) * 1024 (a fixed loss scale, unscaled afterwards) under autocast."""
    out = {}
    cases = (("r50", False, "resnet50", (256, 128)), ("ibn320", True, "resnet50_ibn_a", (320, 320)),
             ("ibn", True, "resnet50_ibn_a", (128, 64)))
    for tag, ibn, mname, hw in cases:
        sd = O.make_trunk_state(seed=7, ibn=ibn)
        cfg = default_cfg(ref)
        cfg.MODEL.NAME = mname
        base = ref.baseline.Baseline(cfg)
        base.base.load_state_dict(sd, strict=True)
        base.eval()
        x = torch.randn(2, 3, *hw, generator=torch.Generator().manual_seed(21))
        with torch.no_grad():
            _, f32 = base(x)
            with torch.autocast("cpu", dtype=torch.float16):
                _, f16 = base(x)
        out[f"{tag}_in_checksum"] = checksum(x)
        out[f"{tag}_eval_feat_fp32"] = f32.float().numpy()
        out[f"{tag}_eval_feat_amp"] = f16.float().numpy()
        rel = float((f16.float() - f32).abs().max() / f32.abs().max())
        out[f"{tag}_amp_vs_fp32"] = rel
        print(f"trunk autocast {tag}: reference fp16-autocast vs its own fp32: {rel:.3e} of the feature scale")
    scale = 1024.0
    for ibn, mname in ((False, "resnet50"), (True, "resnet50_ibn_a")):
        tag = "ibn" if ibn else "r50"
        sd = O.make_trunk_state(seed=17, ibn=ibn)
        cfg = default_cfg(ref)
        cfg.MODEL.NAME = mname
        base = ref.baseline.Baseline(cfg)
        base.base.load_state_dict(sd, strict=True)
        base.train()
        g = torch.Generator().manual_seed(23)
        x = torch.randn(4, 3, 64, 32, generator=g)
        dfeat = torch.randn(4, 2048, generator=g) * 1e-2
        with torch.autocast("cpu", dtype=torch.float16):
            _, feat = base(x)
        ((feat.float() * dfeat).sum() * scale).backward()
        params = dict(base.base.named_parameters())
        out[f"{tag}_train_in_checksum"] = checksum(torch.cat((x.flatten(), dfeat.flatten())))
        out[f"{tag}_train_feat_amp"] = feat.detach().float().numpy()
        for key in TRAIN_GRAD_KEYS:
            k = key.format(bn="BN." if ibn else "")
            out[f"{tag}_train_grad_{k}"] = grad_sample(params[k].grad / scale)
        print(f"trunk autocast train {tag}: feat std {float(feat.float().std()):.4f}")
    np.savez_compressed(os.path.join(GOLD, "trunk_autocast.npz"), **out)


TRIPLET_VARIANTS = ((None, "euclidean"), (0.3, "cosine"), (None, "cosine"))
TRIPLET_GRAD_ELEMS = np.sort(np.random.default_rng(0).choice(40 * 384, 2048, replace=False))  # of the flattened gradient


def triplet_variant_batch():
    feats, labels, is_real = O.synth_batch(10, 4, 384, 100, seed=4, pad_fraction=0.2)
    return feats * 0.3 + 0.05, labels, is_real


def gen_triplet_variants(ref):
    """The reference's own TripletLoss (losses/triplet_loss.py) with a soft margin and with cosine distances: loss value
    and a fixed sample of the input gradient on one batch."""
    feats, labels, _ = triplet_variant_batch()
    out = {"in_checksum": checksum(feats)}
    for margin, dist in TRIPLET_VARIANTS:
        fr = feats.clone().requires_grad_(True)
        loss, _, _ = ref.triplet_loss.TripletLoss(margin, dist)(fr, labels)
        loss.backward()
        out[f"{dist}_{margin}_loss"] = loss.item()
        out[f"{dist}_{margin}_grad"] = fr.grad.flatten()[TRIPLET_GRAD_ELEMS].numpy()
        out[f"{dist}_{margin}_grad_absmax"] = float(fr.grad.abs().max())
    np.savez_compressed(os.path.join(GOLD, "triplet_variants.npz"), **out)
    print("triplet variants done")


ERASE_SHAPE, ERASE_SEEDS = (32, 20), 5
ERASE_MEAN, ERASE_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def erase_input():
    """One uint8 HWC image and its normalised CHW tensor (ToTensor + Normalize)."""
    H, W = ERASE_SHAPE
    img = torch.from_numpy(np.random.default_rng(1).integers(0, 256, (1, H, W, 3), dtype=np.uint8))
    norm = (img[0].permute(2, 0, 1).float() / 255.0 - torch.tensor(ERASE_MEAN)[:, None, None]) / torch.tensor(ERASE_STD)[:, None, None]
    return img, norm


def gen_random_erasing(ref):
    """The reference's own RandomErasing (datasets/transforms/random_erasing.py) on one normalised image, driven by
    random.seed(s) for s in range(ERASE_SEEDS)."""
    import importlib.util
    import random

    from oracle.ref_import import REFERENCE_ROOT

    spec = importlib.util.spec_from_file_location(
        "ref_random_erasing", os.path.join(REFERENCE_ROOT, "datasets", "transforms", "random_erasing.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    img, norm = erase_input()
    outs = []
    for seed in range(ERASE_SEEDS):
        random.seed(seed)
        outs.append(mod.RandomErasing(probability=1.0, mean=ERASE_MEAN)(norm.clone()).numpy())
    np.savez_compressed(os.path.join(GOLD, "random_erasing.npz"), in_checksum=checksum(img), erased=np.stack(outs))
    print("random erasing done")


# The reference's trunk on a CUDA device under fp16 autocast at the bench shapes (tests/test_reference_autocast_gpu.py).
# Whole outputs would not fit a small fixture, so every image is kept on a fixed sample of feature channels, and every
# parameter gradient as a strided sample (grad_sample, in float16 over its largest magnitude: the test takes cosines of
# it) next to the full tensor's norm and its fp16-vs-fp32 cosine.  The autocast features are fp16 values: stored exactly.
AUTOCAST_EVAL_CASES = (("r50", False, (256, 128), 256), ("ibn", True, (320, 320), 128))
AUTOCAST_TRAIN_CASES = (("r50 cfg2", False, (256, 128), 16, 16), ("ibn cfg4/gpu", True, (320, 320), 32, 4))
AUTOCAST_FEAT_COLS = np.sort(np.random.default_rng(0).choice(2048, 32, replace=False))
AUTOCAST_GRAD_SAMPLE = 128
AUTOCAST_LOSS_SCALE = 1024.0


def autocast_eval_input(ibn, hw, bs):
    return O.make_trunk_state(seed=7, ibn=ibn), torch.randn(bs, 3, *hw, generator=torch.Generator().manual_seed(77))


def autocast_train_input(ibn, hw, n):
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(n, 3, *hw, generator=gen)
    return O.make_trunk_state(seed=17, ibn=ibn), x, torch.randn(n, 2048, generator=gen) * 1e-3


def golden_name(tag):
    return tag.split()[0]


def _ref_base_cuda(ref, ibn, sd):
    cfg = default_cfg(ref)
    cfg.MODEL.NAME = "resnet50_ibn_a" if ibn else "resnet50"
    base = ref.baseline.Baseline(cfg)
    base.base.load_state_dict(sd, strict=True)
    return base.cuda()


def gen_ref_cuda_autocast(ref):
    """Needs a CUDA device.  Eval: global features of the eval trunk under torch.autocast(float16) and in fp32.  Train: one
    train-mode step of sum(feat * dfeat) * AUTOCAST_LOSS_SCALE under autocast (features, unscaled gradients) and the
    gradients of the same module in fp32."""
    cols = torch.from_numpy(AUTOCAST_FEAT_COLS)
    out = {"cols": AUTOCAST_FEAT_COLS}
    for tag, ibn, hw, bs in AUTOCAST_EVAL_CASES:
        sd, x = autocast_eval_input(ibn, hw, bs)
        base = _ref_base_cuda(ref, ibn, sd).eval()
        with torch.no_grad():
            _, f32 = base(x.cuda())
            with torch.autocast("cuda", dtype=torch.float16):
                _, amp = base(x.cuda())
        f32, amp = f32.float().cpu(), amp.float().cpu()
        scale = float(f32.abs().max())
        out[f"{tag}_in_checksum"] = checksum(x)
        out[f"{tag}_scale"] = scale
        out[f"{tag}_amp_vs_fp32"] = float((amp - f32).abs().max()) / scale
        out[f"{tag}_feat_amp"] = amp[:, cols].half().numpy()
        # fp32 features as their (small) distance to the autocast ones: fp16 keeps it to < 1e-6 of the feature scale
        out[f"{tag}_feat_fp32_minus_amp"] = (f32 - amp)[:, cols].half().numpy()
        print(f"ref cuda autocast eval {tag}: autocast vs fp32 {out[f'{tag}_amp_vs_fp32']:.3e}")
        del base
    np.savez_compressed(os.path.join(GOLD, "ref_cuda_autocast_eval.npz"), **out)
    for tag, ibn, hw, P, K in AUTOCAST_TRAIN_CASES:
        sd, x, dfeat = autocast_train_input(ibn, hw, P * K)
        x, dfeat_d = x.cuda(), dfeat.cuda()
        base = _ref_base_cuda(ref, ibn, sd).train()
        with torch.autocast("cuda", dtype=torch.float16):
            _, rfeat = base(x)
        ((rfeat.float() * dfeat_d).sum() * AUTOCAST_LOSS_SCALE).backward()
        rgrads = {k: (p.grad / AUTOCAST_LOSS_SCALE).cpu() for k, p in base.base.named_parameters() if p.grad is not None}
        rfeat = rfeat.detach().float().cpu()
        base.zero_grad(set_to_none=True)
        base.base.load_state_dict(sd, strict=True)  # the first pass moved the running statistics
        _, rfeat32 = base(x)
        (rfeat32 * dfeat_d).sum().backward()
        rgrads32 = {k: p.grad.cpu() for k, p in base.base.named_parameters() if p.grad is not None}
        del base, rfeat32
        torch.cuda.empty_cache()
        keys = list(rgrads)
        amp64, f64 = [rgrads[k].double() for k in keys], [rgrads32[k].double() for k in keys]
        out = {"cols": AUTOCAST_FEAT_COLS, "in_checksum": checksum(torch.cat((x.cpu().flatten(), dfeat.flatten()))),
               "feat_scale": float(rfeat.abs().max()), "feat_amp": rfeat[:, cols].half().numpy(), "keys": np.array(keys),
               "norm_amp": np.array([float(a.norm()) for a in amp64]), "norm_fp32": np.array([float(b.norm()) for b in f64]),
               "cos_amp_fp32": np.array([float((a * b).sum() / (a.norm() * b.norm() + 1e-300)) for a, b in zip(amp64, f64)])}
        for name, grads in (("grad_amp", rgrads), ("grad_fp32", rgrads32)):
            rows = np.zeros((len(keys), AUTOCAST_GRAD_SAMPLE), dtype=np.float16)  # row i: the sample of keys[i], zero-padded
            for i, k in enumerate(keys):
                s = grad_sample(grads[k], AUTOCAST_GRAD_SAMPLE)[:-2]
                rows[i, :len(s)] = s / max(float(np.abs(s).max()), 1e-300)
            out[name] = rows
        np.savez_compressed(os.path.join(GOLD, f"ref_cuda_autocast_train_{golden_name(tag)}.npz"), **out)
        print(f"ref cuda autocast train {tag}: {len(keys)} gradients, worst autocast-vs-fp32 cosine "
              f"{out['cos_amp_fp32'].min():.4f}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="loss,loss_variants,masks,retrieval,centroids,trunk,trunk_train,trunk_autocast,market,"
                                      "triplet_variants,random_erasing,trunk_geometry")
    args = ap.parse_args()
    only = set(args.only.split(","))
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    ref = load_reference()
    if "masks" in only:
        gen_masks(ref)
    if "loss" in only:
        gen_loss(ref)
    if "loss_variants" in only:
        gen_loss(ref, variants=True)
    if "retrieval" in only:
        gen_retrieval(ref, "small", 64, 512, 40, 3.0, 0)
        gen_retrieval(ref, "dyadic", 96, 1000, 60, 0.0, 5, dyadic=True)
        gen_retrieval(ref, "ties", 32, 300, 10, 0.0, 6, dyadic=True)
    if "centroids" in only:
        gen_centroids(ref)
    if "trunk" in only:
        gen_trunk(ref)
    if "trunk_train" in only:
        gen_trunk_train(ref)
    if "trunk_autocast" in only:
        gen_trunk_autocast(ref)
    if "market" in only:
        # BASELINE config 3 shape; the reference's per-query python loop takes ~80 s here
        gen_retrieval(ref, "market", 3368, 15913, 751, 3.0, 0, store_dist=False)
    if "triplet_variants" in only:
        gen_triplet_variants(ref)
    if "random_erasing" in only:
        gen_random_erasing(ref)
    if "trunk_geometry" in only:
        gen_trunk_geometry(ref)
    if "ref_cuda_autocast" in only:  # needs a CUDA device; not in the default list
        gen_ref_cuda_autocast(ref)


if __name__ == "__main__":
    main()
