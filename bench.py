#!/usr/bin/env python
"""Benchmark of the B200-native centroid-triplet re-ID hot path (driver contract: ONE JSON line).

    python bench.py --gpus N --steps K --warmup W                      (our CUDA path)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference [--workload embed|retrieval|train] (the reference on the host cores)
    python bench.py ... --dump-outputs DIR                             (+ the last timed step's embeddings, DIR/*.npy)

Primary metric (BASELINE.json): embeddings/sec @256x128 -- one "step" = one pass of the eval embedding path (trunk ->
global average pool -> BatchNorm1d, modelling/bases.py:169-177) over one batch of 256 synthetic 256x128 crops per GPU,
fp16 activations / fp32 accumulation, random-init ResNet50 weights of the reference architecture.  At N > 1 every rank
embeds its own batches and the per-rank embeddings are all-gathered ONCE after extraction over NCCL (SURVEY 8e), inside
the timed region (weak scaling).

Nested in the same line (every BASELINE config has a driver-visible record):
  retrieval   N = 1: config 3 (3368 x 15913 x 2048, top-100 + CMC/mAP);  N > 1: config 5's shape with the gallery axis
              sharded (50 000 queries x 25 000*N gallery rows, top-100 + CMC/mAP; N = 8 is config 5), checked against a
              single-GPU run of a sub-problem in the same process group
  train_step  N = 1: config 2 (ResNet50 256x128, 16 ids x 16 instances);  N > 1: config 4's per-GPU shape
              (ResNet50-IBN-a 320x320, 32 ids x 4 instances per GPU, NCCL gradient all-reduce; N = 8 is config 4)
  cpu_baseline legs (rank 0, N = 1): the UNMODIFIED reference (oracle/_ref, vendored by oracle/vendor_ref.py) on the host
              cores -- its validation_step for M1, its training_step for config 1, get_euclidean + argsort + eval_func
              for M2; the oracle port only when the vendored copy is absent (kind says which).

Only the cpu_baseline legs and `--impl reference` execute anything under oracle/.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH = 256
H, W = 256, 128
GFLOP_PER_IMG = 8.1065       # SURVEY 8d: sum over the 53 convolutions, ResNet50 256x128, last_stride 1
GFLOP_PER_IMG_IBN320 = 25.333  # SURVEY 8d: ResNet50-IBN-a 320x320
RET_Q, RET_G, RET_D, RET_K, RET_IDS = 3368, 15913, 2048, 100, 751
C5_Q, C5_G_PER_RANK, C5_IDS = 50_000, 25_000, 20_000
CPU_BATCH = 128              # BASELINE.md section 3: the CPU reference legs run B = 128


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed regions (B200_PROFILING.md).  The sampler
    process is started once (nvidia-smi needs ~0.5 s to come up) and polls every 20 ms; `window()`
    marks the wall-clock intervals of the timed loops and only samples inside them are summarised."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc, self.windows = gpu_index, [], None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.7)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def window(self):
        sampler = self

        class _W:
            def __enter__(self):
                self.t0 = time.time()

            def __exit__(self, *exc):
                sampler.windows.append((self.t0, time.time()))
                return False

        return _W()

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        sm, mx, pw, reasons = [], [], [], set()
        for t, r in self.rows:
            if self.windows and not any(a - 0.01 <= t <= b + 0.03 for a, b in self.windows):
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvidia-smi sample inside the timed windows"],
                    "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": statistics.median(pw) if pw else None}


def dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


def max_over_ranks(v, world, dev):
    if world == 1:
        return v
    import torch.distributed as dist

    t = torch.tensor([v], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


DUMP_BYTES = 63 << 20  # the arrays of --dump-outputs; the row lists of a sampled output fit in the rest of 64 MB


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: each array as out_dir/<name>.npy in float32.  If they exceed DUMP_BYTES in all, each keeps a
    fixed, seeded sample of its rows (the same rows in every run), listed in out_dir/<name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            rows = np.sort(np.random.default_rng(0).choice(len(a), max(1, len(a) * DUMP_BYTES // total), replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def timed_steps(step_fn, steps, warmup, world, finish_fn=None):
    """W warm-ups, then EXACTLY `steps` steps (+ `finish_fn`, the one collective after extraction) between
    barrier + synchronize; device time via CUDA events on the launching stream, max over ranks."""
    import torch.distributed as dist

    for i in range(warmup):
        step_fn(i)
    if finish_fn is not None and warmup:
        finish_fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step_fn(warmup + i)
    if finish_fn is not None:
        finish_fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    return max_over_ranks(e0.elapsed_time(e1), world, torch.device("cuda", torch.cuda.current_device()))


# ----------------------------------------------------------------------------------------------
# embedding workload (metric M1)
# ----------------------------------------------------------------------------------------------

def build_engine(device):
    import ctl_b200  # noqa: F401
    from ctl_b200 import synth
    from ctl_b200.modelling.backbones.engine import TrunkEngine

    return TrunkEngine(synth.make_trunk_state(seed=0), device, ibn=False, last_stride=1, bn_head=synth.make_head_bn(0))


def run_embed(args, world, rank, local):
    import torch.distributed as dist

    from ctl_b200.modelling.backbones.engine import GraphedCall, GraphedForward

    dev = torch.device("cuda", local)
    eng = build_engine(dev)
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)
    n_rot = 4  # 4 x 100.7 MB of inputs > 126 MB L2; activations (hundreds of MB per layer) never fit anyway
    dev_in = [torch.randn(BATCH, 3, H, W, generator=gen).to(dev) for _ in range(n_rot)]
    graphs = [GraphedForward(eng, d, want_emb=True) for d in dev_in]  # one CUDA graph per rotating input
    steps = args.steps
    # extraction buffer of this rank + ONE all-gather after the last batch (SURVEY 8e; the reference embeds the whole
    # validation set before it computes anything on it, modelling/bases.py:264-280)
    local_emb = torch.empty(steps, BATCH, 2048, device=dev)
    gathered = torch.empty(world, steps, BATCH, 2048, device=dev) if world > 1 else None

    def step(i):
        emb = graphs[i % n_rot]()["emb"]
        local_emb[i % steps].copy_(emb, non_blocking=True)
        return emb

    def finish():
        if world > 1:
            dist.all_gather_into_tensor(gathered, local_emb)

    clk = ClockSampler(local)
    clk.__enter__()
    for i in range(args.warmup):
        step(i)
    finish()
    with clk.window():
        ms = timed_steps(step, steps, 0, world, finish)
    if args.dump_outputs and rank == 0:  # before the e2e runs below reuse local_emb
        emb = gathered[:, steps - 1].reshape(world * BATCH, 2048) if world > 1 else local_emb[steps - 1]
        dump_outputs(args.dump_outputs, {"emb": emb, "global_feat": graphs[(steps - 1) % n_rot].out["global_feat"]})
    launches = (graphs[0].launches + 1) * steps
    value = world * BATCH * steps / (ms / 1e3)

    # ---- end to end through the public API, HOST buffers: pinned uint8 crops -> H2D -> device normalise
    # (datasets/transforms.normalize_batch = the reference's ToTensor + Normalize, transforms/build.py:29-33) -> trunk ->
    # D2H of the embeddings; double-buffered so the copy of step i+1 overlaps the compute of step i.
    def e2e_run(kind):
        copy_stream = torch.cuda.Stream(device=dev)   # H2D of the next batch
        d2h_stream = torch.cuda.Stream(device=dev)    # D2H of the finished embeddings (off the compute stream)
        g8 = torch.Generator().manual_seed(99 + rank)
        if kind == "u8":
            host = [torch.randint(0, 256, (BATCH, H, W, 3), dtype=torch.uint8, generator=g8).pin_memory() for _ in range(n_rot)]
            stage_in = [torch.empty(BATCH, H, W, 3, dtype=torch.uint8, device=dev) for _ in range(2)]
        else:
            host = [torch.randn(BATCH, 3, H, W, generator=g8).pin_memory() for _ in range(n_rot)]
            stage_in = [torch.empty(BATCH, 3, H, W, device=dev) for _ in range(2)]
        out_host = [torch.empty(BATCH, 2048).pin_memory() for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]      # staging buffer b holds the next batch
        done = [torch.cuda.Event() for _ in range(2)]       # the forward that read staging buffer b has finished
        emb_ready = [torch.cuda.Event() for _ in range(2)]  # graph b's output tensor holds this step's embeddings
        d2h_done = [torch.cuda.Event() for _ in range(2)]   # ... and has been copied out (graph b may overwrite it)

        def fwd(b):  # uint8 crops: ToTensor + Normalize run inside the fused stem's packing kernel (forward_u8)
            return eng.forward_u8(stage_in[b], want_emb=True) if kind == "u8" else eng.forward(stage_in[b], want_emb=True)

        stage_graphs = [GraphedCall(lambda b=b: fwd(b), dev) for b in range(2)]

        def prefetch(i):
            b = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[b])  # the forward that last read this staging buffer
                stage_in[b].copy_(host[i % n_rot], non_blocking=True)
                ready[b].record(copy_stream)

        def loop(n_steps, first):
            prefetch(first)
            cur = torch.cuda.current_stream()
            for j in range(n_steps):
                i = first + j
                b = i % 2
                if j + 1 < n_steps:
                    prefetch(i + 1)
                cur.wait_event(ready[b])
                cur.wait_event(d2h_done[b])  # the previous embeddings of this graph have left the device
                emb = stage_graphs[b]()["emb"]
                done[b].record()
                local_emb[i % steps].copy_(emb, non_blocking=True)
                emb_ready[b].record()
                with torch.cuda.stream(d2h_stream):
                    d2h_stream.wait_event(emb_ready[b])
                    out_host[b].copy_(emb, non_blocking=True)
                    d2h_done[b].record(d2h_stream)
            finish()
            cur.wait_stream(d2h_stream)

        for b in range(2):
            done[b].record()
            d2h_done[b].record()
        loop(args.warmup, 0)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        with clk.window():
            loop(steps, args.warmup)
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        dt = max_over_ranks(time.perf_counter() - t0, world, dev)
        return world * BATCH * steps / dt, host[0].numel() * host[0].element_size()

    v8, b8 = e2e_run("u8")
    v32, b32 = e2e_run("f32")
    clk.__exit__(None, None, None)
    e2e = {"value": v8, "unit": "embeddings/s", "h2d_bytes_per_step": b8, "d2h_bytes_per_step": BATCH * 2048 * 4,
           "input": "pinned uint8 HWC crops; ToTensor + Normalize folded into the fused stem's input packing "
                    "(TrunkEngine.forward_u8 == forward(normalize_batch(x)) bit for bit); H2D of step i+1 overlaps the compute "
                    "of step i",
           "fp32_input": {"value": v32, "unit": "embeddings/s", "h2d_bytes_per_step": b32,
                          "input": "pinned fp32 NCHW crops already normalised on the host (the tensor the reference's "
                                   "forward takes)"}}

    # ---- roofline of the dominant kernels (48 conv_gemm / conv3x3 launches), GRAPH MODE: the step's graph time minus the
    # graph time of the stem segment and of the tail segment (each captured alone and replayed the same way) ----
    roof = None
    if rank == 0:
        a_stat, n_, h_, w_ = eng.stem(dev_in[0])
        a_out, h2_, w2_ = eng.bottlenecks(a_stat, n_, h_, w_)
        seg = {"stem": GraphedCall(lambda: eng.stem(dev_in[0]), dev),
               "convs": GraphedCall(lambda: eng.bottlenecks(a_stat, n_, h_, w_), dev),
               "tail": GraphedCall(lambda: eng.tail(a_out, n_, h2_, w2_, False, True), dev)}
        seg_ms = {}
        for name, gcall in seg.items():
            for _ in range(3):
                gcall()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(20):
                gcall()
            e1.record()
            torch.cuda.synchronize()
            seg_ms[name] = e0.elapsed_time(e1) / 20
        step_ms = ms / steps
        # the conv kernels' time INSIDE the timed region: the step minus its two other segments (each replayed alone right
        # after the region).  Never the stand-alone convs segment: in a long run the timed region is power-capped while
        # a 20-replay segment still runs at burst clocks.
        conv_ms = step_ms - seg_ms["stem"] - seg_ms["tail"] if step_ms > seg_ms["stem"] + seg_ms["tail"] else seg_ms["convs"]
        # algorithmic work of the 52 bottleneck convolutions (the stem's 7x7 conv is timed in the stem segment)
        stem_gflop = 2.0 * (H // 2) * (W // 2) * 64 * 147 / 1e9
        conv_flops = (GFLOP_PER_IMG - stem_gflop) * 1e9 * BATCH
        pk = peaks()
        ach = conv_flops / (conv_ms * 1e-3) / 1e12
        traffic = conv_traffic()
        roof = {"kernel": "conv_gemm_pair / conv_gemm / conv3x3_c64 (48 launches per step: conv + folded BN + shortcut + ReLU)",
                "bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": ach / pk["tf_sust"],
                "frac_of_burst_peak": ach / pk["tf_burst"], "peak_burst": pk["tf_burst"],
                "peak_source": pk["src"] + ": bf16 sustained (cuBLAS back to back for 4 s, 1000 W cap); the burst figure "
                                           "(best of 10 short GEMMs) is the like-for-like denominator for a 50 ms timed region",
                "traffic": traffic, "conv_ms": round(conv_ms, 4), "ms_per_step": round(step_ms, 4),
                "share_of_step": conv_ms / step_ms,
                "segments_graph_ms": {k: round(v, 4) for k, v in seg_ms.items()},
                "method": "CUDA-graph replay of the step and of its three segments (stem | 48 conv launches | GAP+BN); "
                          "conv_ms = step - stem - tail",
                "whole_step_tflops": GFLOP_PER_IMG * BATCH / step_ms, "hbm_achieved_gbs": (traffic / (conv_ms * 1e-3) / 1e9) if traffic else None,
                "hbm_peak_gbs": pk["hbm"]}
    return ms, value, launches, e2e, roof, clk.summary()


def _json_metric(name, key):
    path = os.path.join(ROOT, "profiles", name)
    try:
        with open(path) as f:
            return json.load(f)[key]
    except (OSError, KeyError, ValueError):
        return None


def conv_traffic():
    """DRAM bytes (read + write) of the conv launches of one bs-256 forward, from the committed ncu metrics
    pass (profiles/conv_traffic.json, written by tools/launchlist.py on the GPU box); None if absent."""
    return _json_metric("conv_traffic.json", "dram_bytes_per_step")


# ----------------------------------------------------------------------------------------------
# training step (configs 2 and 4)
# ----------------------------------------------------------------------------------------------

def _train_cfg(K, model_name="resnet50"):
    class _C(dict):
        __getattr__ = dict.__getitem__

    return _C(MODEL=_C(NAME=model_name, LAST_STRIDE=1, PRETRAINED=False, PRETRAIN_PATH="", BACKBONE_EMB_SIZE=2048,
                       USE_CENTROIDS=False, KEEP_CAMID_CENTROIDS=True, RESUME_TRAINING=False),
              SOLVER=_C(MARGIN=0.5, DISTANCE_FUNC="euclidean", CENTER_LOSS_WEIGHT=5e-4, QUERY_XENT_WEIGHT=1.0,
                        QUERY_CONTRASTIVE_WEIGHT=1.0, CENTROID_CONTRASTIVE_WEIGHT=1.0, OPTIMIZER_NAME="Adam",
                        BASE_LR=1e-4, WEIGHT_DECAY=5e-4, CENTER_LR=0.5, LR_SCHEDULER_NAME="multistep_lr",
                        LR_STEPS=(40, 70), GAMMA=0.1, USE_WARMUP_LR=True, WARMUP_EPOCHS=10),
              DATALOADER=_C(NUM_INSTANCE=K), TEST=_C(FEAT_NORM=True, ONLY_TEST=False, VISUALIZE="no"),
              USE_MIXED_PRECISION=True)


def run_train_step(local, steps=5, warmup=2, model_name="resnet50", size=(256, 128), P=16, K=16, world=1):
    """BASELINE config 2 (and, with model_name="resnet50_ibn_a", size=(320, 320), P=32, K=4, world=8, config 4):
    one complete CTL training iteration per step -- train-mode trunk forward (batch-stat BN) -> fused
    CTL/center/xent/triplet loss step -> backward through the loss and the trunk (all parameter gradients) ->
    [world > 1: NCCL mean all-reduce of the gradients] -> fused Adam + center-SGD step.
    Every rank trains on its own P x K batch (weak scaling, like the reference's DDP).  Device-timed with CUDA
    events; max over ranks."""
    import ctl_b200  # noqa: F401
    from ctl_b200 import parallel
    from ctl_b200.modelling.ctl_model import CTLModel

    dev = torch.device("cuda", local)
    torch.manual_seed(0)
    model = CTLModel(_train_cfg(K, model_name), num_classes=751, num_query=0).to(dev).train()
    g = torch.Generator().manual_seed(1234 + local)
    x = torch.randn(P * K, 3, size[0], size[1], generator=g).to(dev)
    labels = torch.arange(P).repeat_interleave(K).to(dev)
    cam = torch.zeros(P * K, dtype=torch.long, device=dev)
    is_real = torch.ones(P * K, dtype=torch.bool, device=dev)
    (opt, opt_center), _ = model.configure_optimizers()
    reducer = parallel.GradientReducer(model.parameters()) if world > 1 else None

    def step():
        for p_ in model.parameters():
            p_.grad = None
        out = model.training_step((x, labels, cam, is_real), 0)
        out["loss"].backward()
        if reducer is not None:
            reducer.allreduce_mean()  # NCCL, flat fp32 buckets reduced in place
        model.optimizer_step_manual(opt, opt_center, epoch=0)  # fused Adam + center SGD (solver/build.py)
        return out["loss"]

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1) / steps, world, dev)
    gflop = GFLOP_PER_IMG if (model_name == "resnet50" and tuple(size) == (256, 128)) else (
        GFLOP_PER_IMG_IBN320 if (model_name == "resnet50_ibn_a" and tuple(size) == (320, 320)) else None)
    pk = peaks()
    tfl = (3 * P * K * gflop / ms) if gflop else None  # per GPU
    return {"metric": f"CTL training step images/sec ({model_name} {size[0]}x{size[1]}, {P} ids x {K} instances per GPU, "
                      "fwd+loss+bwd+optimizer)",
            "value": world * P * K / ms * 1e3, "unit": "images/s", "ms_per_step": ms, "steps": steps, "n_gpus": world,
            "loss": float(loss.detach()),
            "config": {"workload": ("BASELINE config 2" if model_name == "resnet50" else "BASELINE config 4 per-GPU shape"),
                       "global_batch": world * P * K},
            "roofline": ({"kernel": "whole training step (forward + data-gradient + weight-gradient convolutions)",
                          "bound": "tensor", "achieved": tfl, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                          "frac": tfl / pk["tf_sust"], "peak_source": pk["src"] + ", bf16 sustained", "traffic": None,
                          "note": f"algorithmic 3 x {gflop} GFLOP per image (SURVEY 8d) / device-timed step, per GPU"}
                         if tfl else None),
            "note": "includes the gradient all-reduce (N > 1) and the fused Adam / center-SGD step; dynamic loss scaling on",
            "peak_mem_gib": torch.cuda.max_memory_allocated(dev) / 2 ** 30}


# ----------------------------------------------------------------------------------------------
# retrieval workload (metric M2)
# ----------------------------------------------------------------------------------------------

def run_retrieval(args, world, rank, local, steps=None, warmup=None):
    """Config 3 on ONE GPU (3368 x 15913 x 2048, top-100 + CMC/mAP).  The planes of the gallery and of the queries are
    built once per validation set (the features do not change between the top-k and the evaluation, nor between
    repeated evaluations) and cached by the API the step times (retrieval.PlaneCache)."""
    import ctypes as C

    import ctl_b200  # noqa: F401
    from ctl_b200 import _native as N
    from ctl_b200 import retrieval as R
    from ctl_b200 import synth

    steps = steps or args.steps
    warmup = warmup or args.warmup
    dev = torch.device("cuda", local)
    feats, pids, cams = synth.synth_retrieval(RET_Q, RET_G, RET_IDS, RET_D, 3.0, 0)
    qh, gh = feats[:RET_Q].contiguous().pin_memory(), feats[RET_Q:].contiguous().pin_memory()
    q, g = qh.to(dev), gh.to(dev)
    box = {}
    # Identity-ordered operands (retrieval.pid_order: pass 1 over a tile list) pay off from ~1.5e8 pairs on
    # (retrieval.pid_order_pays, measured); config 3 is below that and runs in the caller's order, config 5 above.
    sort = R.pid_order_pays(RET_Q, RET_G)
    qo, go = (R.pid_order(pids[:RET_Q]), R.pid_order(pids[RET_Q:])) if sort else (None, None)
    ids = R.encode_ids(pids[:RET_Q], pids[RET_Q:], cams[:RET_Q], cams[RET_Q:], False, dev, q_order=qo, g_order=go)

    cache = R.PlaneCache()
    # one validation set evaluated again and again: the step's launch sequence is captured once (retrieval.TopkEvalSession)
    # when the operands stay in the caller's order; identity-ordered operands (config 5 sizes) take the eager path
    sess = None if sort else R.TopkEvalSession(g, RET_Q, RET_K, pids[:RET_Q], pids[RET_Q:], cams[:RET_Q], cams[RET_Q:])

    def step(i):
        # one retrieval pass against a RESIDENT gallery: query planes from the fp32 query features, the gallery's planes
        # built once per gallery tensor (a fixed `embeddings.npy` searched by successive query sets,
        # inference/get_similar.py:104-128), two tensor-core passes, top-100 + CMC/mAP, one read-back
        if sess is not None:
            idx, dst, res = sess(q)
        else:
            qp, gp = R.build_planes(q, order=qo), cache.get(g, order=go)
            idx, dst, res = R.topk_and_eval(qp, gp, RET_K, pids[:RET_Q], pids[RET_Q:], cams[:RET_Q], cams[RET_Q:], ids=ids)
        box["res"] = res

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()  # the step ends with a host read-back (CMC/mAP), so wall time on a quiet stream == device time
    for i in range(steps):
        step(i)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps

    def e2e_step(i):
        qd, gd = qh.to(dev, non_blocking=True), gh.to(dev, non_blocking=True)
        # nothing cached: (identity orders,) planes and identity arrays are all rebuilt from the host inputs
        qp = R.build_planes(qd, order=R.pid_order(pids[:RET_Q]) if sort else None)
        gp = R.build_planes(gd, order=R.pid_order(pids[RET_Q:]) if sort else None)
        idx, dst, res = R.topk_and_eval(qp, gp, RET_K, pids[:RET_Q], pids[RET_Q:], cams[:RET_Q], cams[RET_Q:])
        return idx.cpu(), dst.cpu(), res

    for i in range(2):
        e2e_step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        e2e_step(i)
    torch.cuda.synchronize()
    dte = (time.perf_counter() - t0) / steps
    # GEMM kernel alone (one pass)
    qp, gp = R.build_planes(q), R.build_planes(g)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gmin = torch.empty(RET_Q, (RET_G + 15) // 16, device=dev)
    desc = N.PassDesc(gmin=gmin.data_ptr())
    for _ in range(2):
        N.check(N.lib().ctl_dist_pass(qp.ptr, RET_Q, gp.ptr, RET_G, RET_D, qp.flags, C.byref(desc), N.stream_ptr()))
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
        N.check(N.lib().ctl_dist_pass(qp.ptr, RET_Q, gp.ptr, RET_G, RET_D, qp.flags, C.byref(desc), N.stream_ptr()))
    e1.record()
    torch.cuda.synchronize()
    pass_ms = e0.elapsed_time(e1) / 5
    # pass 2 as the step runs it (candidates + bucket counts): the other half of the step's tensor work
    ids_b = R.encode_ids(pids[:RET_Q], pids[RET_Q:], cams[:RET_Q], cams[RET_Q:], False, dev)
    pcnt = torch.zeros(RET_Q, dtype=torch.int32, device=dev)
    ovf = torch.zeros(1, dtype=torch.int32, device=dev)
    pos = torch.zeros(RET_Q, ids_b.max_pos, dtype=torch.int64, device=dev)
    idk = dict(q_pid=ids_b.q_pid.data_ptr(), q_cam=ids_b.q_cam.data_ptr(), g_pid=ids_b.g_pid.data_ptr(),
               g_cammask=ids_b.g_mask.data_ptr(), max_pos=ids_b.max_pos, overflow=ovf.data_ptr())
    L = N.lib()
    N.check(L.ctl_dist_pass(qp.ptr, RET_Q, gp.ptr, RET_G, RET_D, qp.flags, C.byref(N.PassDesc(
        gmin=gmin.data_ptr(), pos_keys=pos.data_ptr(), pos_count=pcnt.data_ptr(), **idk)), N.stream_ptr()))
    tau = torch.empty(RET_Q, device=dev)
    N.check(L.ctl_select_tau(gmin.data_ptr(), RET_Q, gmin.shape[1], 1, RET_K, tau.data_ptr(), N.stream_ptr()))
    N.check(L.ctl_sort_key_rows(pos.data_ptr(), pcnt.data_ptr(), RET_Q, ids_b.max_pos, N.stream_ptr()))
    cand = torch.empty(RET_Q, 4096, dtype=torch.int64, device=dev)
    cc = torch.zeros(RET_Q, dtype=torch.int32, device=dev)
    buckets = torch.zeros(RET_Q, ids_b.max_pos + 1, dtype=torch.int32, device=dev)
    desc1 = N.PassDesc(tau=tau.data_ptr(), cand_keys=cand.data_ptr(), cand_count=cc.data_ptr(), cand_cap=4096,
                       thr_keys=pos.data_ptr(), thr_count=pcnt.data_ptr(), buckets=buckets.data_ptr(), **idk)
    times = []
    for _ in range(5):
        cc.zero_()
        e0.record()
        N.check(L.ctl_dist_pass(qp.ptr, RET_Q, gp.ptr, RET_G, RET_D, qp.flags, C.byref(desc1), N.stream_ptr()))
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    pass2_ms = sorted(times)[2]
    pk = peaks()
    flops = 2.0 * RET_Q * RET_G * RET_D  # algorithmic (SURVEY 8d: 2*D flop per pair); the kernel issues 3 fp16 products
    ach = flops / (pass_ms * 1e-3) / 1e12
    return {
        "metric": "QxG top-k pairs/sec (3368x15913x2048, top-100 + CMC/mAP)", "value": RET_Q * RET_G / dt,
        "unit": "pairs/s", "ms_per_step": dt * 1e3, "steps": steps, "n_gpus": 1, "mAP": box["res"].mAP,
        "rank1": float(box["res"].cmc[0]),
        "config": {"workload": "BASELINE config 3: 3368 query x 15913 gallery x 2048-d, L2 top-100 + CMC/mAP",
                   "planes": "`value`: gallery planes resident (built once), query features copied in and their planes built every "
                             "step, the step's launches replayed from one CUDA graph (retrieval.TopkEvalSession); `e2e`: "
                             "eager path, both operands' planes built every step from the freshly uploaded host features"},
        "e2e": {"value": RET_Q * RET_G / dte, "unit": "pairs/s", "h2d_bytes_per_step": (RET_Q + RET_G) * RET_D * 4,
                "d2h_bytes_per_step": RET_Q * RET_K * 12},
        "roofline": {"kernel": "dist_gemm_kernel (split-fp16 x3 tcgen05, one pass)", "bound": "tensor",
                     "achieved": ach, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": ach / pk["tf_burst"],
                     "peak_source": pk["src"] + ", bf16 burst (a 0.5 ms kernel timed alone)", "pass_ms": pass_ms, "pass2_ms": pass2_ms,
                     "traffic": _json_metric("dist_traffic.json", "dram_bytes_per_pass"),
                     "tensor_pipe_tflops": 3 * ach,
                     "note": "achieved = algorithmic 2*Q*G*D flop per pass; the fp32-equivalent split issues 3 fp16 "
                             "MMA products per element (tensor_pipe_tflops = 3 x achieved, %.2f of the burst peak)"
                             % (3 * ach / pk["tf_burst"])},
        "gpu_launches_per_step": 9,
    }


def run_retrieval_sharded(args, world, rank, local, steps=3, warmup=1):
    """BASELINE config 5's shape with the gallery axis sharded: 50 000 queries (each rank owns a slice, all-gathered ONCE
    over NCCL) x 25 000 gallery rows PER RANK, 2048-d, top-100 + CMC/mAP (world = 8 is config 5).  Before timing, a
    sub-problem is solved both sharded and by rank 0 alone on one GPU and the results are compared bit for bit."""
    import torch.distributed as dist

    import ctl_b200  # noqa: F401
    from ctl_b200 import retrieval as R
    from ctl_b200 import synth

    dev = torch.device("cuda", local)
    grp = dist.group.WORLD

    def make(nq, ng_rank, n_ids, seed):
        """queries (all ranks build the same ones from the same seed -- the all-gather below still runs on per-rank slices)
        and this rank's gallery shard; identities uniform over n_ids."""
        gq = torch.Generator(device=dev).manual_seed(seed)
        cent = torch.randn(n_ids, RET_D, device=dev, generator=gq)  # same on every rank
        q_pid = torch.randint(0, n_ids, (nq,), device=dev, generator=gq)
        q_cam = torch.randint(0, 6, (nq,), device=dev, generator=gq)
        qf = torch.nn.functional.normalize(cent[q_pid] + 3.0 * torch.randn(nq, RET_D, device=dev, generator=gq), dim=1)
        gg = torch.Generator(device=dev).manual_seed(seed * 1000 + 17 + rank)
        g_pid = torch.randint(0, n_ids, (ng_rank,), device=dev, generator=gg)
        g_cam = torch.randint(0, 6, (ng_rank,), device=dev, generator=gg)
        gf = torch.nn.functional.normalize(cent[g_pid] + 3.0 * torch.randn(ng_rank, RET_D, device=dev, generator=gg), dim=1)
        return qf, q_pid.cpu().numpy(), q_cam.cpu().numpy(), gf, g_pid.cpu().numpy(), g_cam.cpu().numpy()

    def prepare(q_pid, q_cam, g_pid, g_cam):
        """once per validation set (the identities do not change between evaluations -- config 3 caches its `ids` the same
        way): the identity orders of both operands and the device-resident identity arrays in those orders."""
        qo, go = R.pid_order(q_pid), R.pid_order(g_pid)  # identity order on every rank: pass 1 runs a tile list
        return qo, go, R.encode_ids_sharded(q_pid, g_pid, q_cam, g_cam, dev, grp, q_order=qo, g_order=go)

    def sharded(qf, q_pid, gf, k, prep):
        qo, go, ids = prep
        nq = qf.shape[0]
        per = (nq + world - 1) // world
        q_slice = torch.zeros(per, RET_D, device=dev)
        lo = min(rank * per, nq)
        hi = min(lo + per, nq)
        q_slice[: hi - lo] = qf[lo:hi]
        q_all = torch.empty(world * per, RET_D, device=dev)
        dist.all_gather_into_tensor(q_all, q_slice)          # the ONE embedding all-gather of config 5
        qp = R.build_planes(q_all[:nq], order=qo)
        gp = R.build_planes(gf, order=go)
        return R.topk_and_eval_sharded(qp, gp, k, ids, q_pid, rank * gf.shape[0], world * gf.shape[0], grp)

    # ---- equality with one GPU on a sub-problem ----
    sq, sg = 2048, 4096
    qf, q_pid, q_cam, gf, g_pid, g_cam = make(sq, sg, 512, 7)
    idx_s, dst_s, res_s = sharded(qf, q_pid, gf, RET_K, prepare(q_pid, q_cam, g_pid, g_cam))
    g_all = torch.empty(world * sg, RET_D, device=dev)
    dist.all_gather_into_tensor(g_all, gf)
    pid_all = [None] * world
    cam_all = [None] * world
    dist.all_gather_object(pid_all, g_pid)
    dist.all_gather_object(cam_all, g_cam)
    equal = None
    if rank == 0:
        gp_all, gc_all = np.concatenate(pid_all), np.concatenate(cam_all)
        idx_1, dst_1, res_1 = R.topk_and_eval(R.build_planes(qf), R.build_planes(g_all), RET_K, q_pid, gp_all, q_cam, gc_all)
        equal = bool(torch.equal(idx_1, idx_s) and torch.equal(dst_1, dst_s) and res_1.mAP == res_s.mAP
                     and np.array_equal(res_1.cmc, res_s.cmc) and np.array_equal(res_1.ranks[:, :1], res_s.ranks[:, :1]))
    del g_all
    # ---- config 5 shape ----
    qf, q_pid, q_cam, gf, g_pid, g_cam = make(C5_Q, C5_G_PER_RANK, C5_IDS, 11)
    box = {}
    prep = prepare(q_pid, q_cam, g_pid, g_cam)

    def step():
        box["out"] = sharded(qf, q_pid, gf, RET_K, prep)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    dt = max_over_ranks((time.perf_counter() - t0) / steps, world, dev)
    res = box["out"][2]
    G = world * C5_G_PER_RANK
    return {"metric": f"QxG top-k pairs/sec ({C5_Q}x{G}x2048, gallery sharded over {world} GPUs, top-100 + CMC/mAP)",
            "value": C5_Q * G / dt, "unit": "pairs/s", "ms_per_step": dt * 1e3, "seconds": dt, "steps": steps,
            "n_gpus": world, "scaling": "weak", "mAP": res.mAP, "rank1": float(res.cmc[0]),
            "sharded_equals_single_gpu": equal,
            "config": {"workload": f"BASELINE config 5 shape: 50 000 queries x {G} gallery rows (25 000 per GPU), 2048-d, "
                                   "queries all-gathered once, positives' keys all-gathered, bucket counts all-reduced, "
                                   "per-shard top-100 merged by integer key order",
                       "equality_check": f"{sq} x {world * sg} sub-problem: sharded == rank 0 alone on one GPU "
                                         "(indices, distances, CMC, mAP bit for bit)"},
            "note": "the timed step includes the query all-gather, building both operands' planes (in identity order), both "
                    "tensor-core passes, all collectives and the CMC/mAP reduction with its host read-back; the identity "
                    "orders and the device identity arrays are prepared once per validation set (like config 3's `ids`)"}


# ----------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the UNMODIFIED reference (oracle/_ref) on the host cores
# ----------------------------------------------------------------------------------------------

def _host_threads():
    """All the host threads torch can use productively: its own default is one per physical core;
    hyper-thread oversubscription (os.cpu_count()) was measured 19x SLOWER on the 128-thread box."""
    n = max(1, (os.cpu_count() or 2) // 2)  # torchrun exports OMP_NUM_THREADS=1: set the count explicitly
    torch.set_num_threads(n)
    return n


def _best_threads(fn):
    """The CPU arm deserves its best configuration: time `fn` once at all / half / a quarter of the physical cores
    (small-M GEMMs of the late layers do not scale to 64 threads) and keep the fastest; returns the thread count."""
    full = _host_threads()
    best, best_t = full, None
    for n in sorted({full, max(1, full // 2), max(1, full // 4)}, reverse=True):
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def _reference():
    """The reference's own modules (oracle/_ref on the GPU box, /root/reference in the build container) or None."""
    from oracle import ref_import  # bench.py's cpu legs are one of the two sanctioned users of oracle/

    if not ref_import.reference_available():
        return None
    import warnings

    warnings.filterwarnings("ignore")
    return ref_import.load_reference()


def _ref_model(ref, K=4):
    from oracle import ref_import
    from oracle import ctl_oracle as O

    cfg = ref_import.default_cfg(ref)
    cfg.DATALOADER.NUM_INSTANCE = K
    model = ref.train_ctl.CTLModel(cfg, num_classes=751, num_query=0)
    model.backbone.base.load_state_dict(O.make_trunk_state(seed=0), strict=True)
    return model


def cpu_embed(steps, warmup, budget_s=150.0):
    """Metric M1 on the host cores: the reference's own `validation_step` (eval backbone -> bn, modelling/bases.py:169-177)
    on B = 128 crops per step (BASELINE.md section 3).  Runs `warmup` + up to `steps` steps, stopping early when
    `budget_s` of timed work is used up; returns what it actually ran."""
    from oracle import ctl_oracle as O

    cores = _host_threads()
    ref = _reference()
    x = torch.randn(CPU_BATCH, 3, H, W, generator=torch.Generator().manual_seed(1))
    lab = torch.zeros(CPU_BATCH, dtype=torch.long)
    if ref is not None:
        model = _ref_model(ref).eval()
        kind = "reference"

        def fwd():
            return model.validation_step((x, lab, lab, lab), 0)["emb"]
    else:
        sd = O.make_trunk_state(seed=0)
        g = torch.Generator().manual_seed(10_000)
        bn = dict(weight=0.5 + torch.rand(2048, generator=g), bias=torch.zeros(2048),
                  running_mean=0.1 * torch.randn(2048, generator=g), running_var=0.5 + torch.rand(2048, generator=g))
        kind = "port"

        def fwd():
            with torch.no_grad():
                return O.embed_forward(x, sd, bn)
    fwd()  # first touch (allocator, oneDNN primitives)
    cores = _best_threads(fwd)
    for _ in range(max(0, warmup - 1)):
        fwd()
    done, t0 = 0, time.perf_counter()
    while done < steps and (done == 0 or time.perf_counter() - t0 < budget_s):
        fwd()
        done += 1
    dt = time.perf_counter() - t0
    return {"value": CPU_BATCH * done / dt, "unit": "embeddings/s", "cores": cores, "kind": kind,
            "sample": f"{done} step(s) of {CPU_BATCH} crops (256x128, fp32) through "
                      + ("the reference's CTLModel.validation_step (backbone -> bn)" if kind == "reference" else "oracle.embed_forward")
                      + f", {dt:.1f} s", "steps_run": done, "seconds": dt}


def cpu_train(steps, warmup, budget_s=150.0):
    """BASELINE config 1: the reference's own `CTLModel.training_step` (train_ctl_model.py:38-179: forward, the four
    losses, manual backward, Adam + center-SGD steps) on B = 128 (32 ids x 4), ResNet50 256x128, fp32, on the host cores."""
    cores = _host_threads()
    ref = _reference()
    if ref is None:
        return {"value": None, "unit": "images/s", "cores": cores, "kind": "unavailable",
                "sample": "oracle/_ref absent: the reference's training_step cannot be timed on this box"}
    P, K = 32, 4
    model = _ref_model(ref, K).train()

    class _Trainer:
        current_epoch = 0

    model.trainer = _Trainer()
    opts, _ = model.configure_optimizers()
    model._ctl_optimizers = tuple(opts)
    x = torch.randn(P * K, 3, H, W, generator=torch.Generator().manual_seed(2))
    labels = torch.arange(P).repeat_interleave(K)
    cam = torch.zeros(P * K, dtype=torch.long)
    is_real = torch.ones(P * K, dtype=torch.bool)
    model.training_step((x, labels, cam, is_real), 0)  # first touch
    cores = _best_threads(lambda: model.training_step((x, labels, cam, is_real), 0))
    done, t0 = 0, time.perf_counter()
    while done < steps and (done == 0 or time.perf_counter() - t0 < budget_s):
        out = model.training_step((x, labels, cam, is_real), 0)
        done += 1
    dt = time.perf_counter() - t0
    return {"value": P * K * done / dt, "unit": "images/s", "cores": cores, "kind": "reference",
            "sample": f"{done} step(s) of the reference's CTLModel.training_step, B = {P * K} ({P} ids x {K}), ResNet50 "
                      f"256x128 fp32, {dt / done:.2f} s/step (BASELINE config 1)", "steps_run": done, "seconds": dt,
            "loss": float(out["loss"])}


def cpu_retrieval(nq):
    """Metric M2 on the host cores: the reference's get_euclidean + np.argsort + eval_func (utils/reid_metric.py:25-33,
    :112-136, utils/eval_reid.py:25-92) on the first `nq` queries of config 3 against the whole gallery."""
    from oracle import ctl_oracle as O

    cores = _host_threads()
    ref = _reference()
    feats, pids, cams = O.synth_retrieval(RET_Q, RET_G, RET_IDS, RET_D, 3.0, 0)
    q, g = feats[:nq], feats[RET_Q:]
    t0 = time.perf_counter()
    if ref is not None:
        kind = "reference"
        dist = ref.reid_metric.get_euclidean(q, g).numpy()
        t1 = time.perf_counter()
        idx = np.argsort(dist, axis=1)
        t2 = time.perf_counter()
        ref.eval_reid.eval_func(idx, pids[:nq], pids[RET_Q:], cams[:nq], cams[RET_Q:], 50, False)
        parts = f"get_euclidean {t1 - t0:.2f} s + argsort {t2 - t1:.2f} s + eval_func {time.perf_counter() - t2:.2f} s"
    else:
        kind = "port"
        O.r1_map_compute(torch.cat((q, g)), np.concatenate((pids[:nq], pids[RET_Q:])),
                         np.concatenate((cams[:nq], cams[RET_Q:])), nq)
        parts = "oracle.r1_map_compute"
    dt = time.perf_counter() - t0
    return {"value": nq * RET_G / dt, "unit": "pairs/s", "cores": cores, "kind": kind,
            "sample": f"{nq} of {RET_Q} queries x {RET_G} gallery x 2048-d: {parts}", "seconds": dt}


def reference_arm(args, world):
    """`--impl reference`: rank 0 only; the reference's own CPU implementation of the selected workload."""
    if args.workload == "embed":
        r = cpu_embed(args.steps, min(args.warmup, 2))
        metric, name = "embeddings/sec @256x128", (f"resnet50 eval embedding forward (trunk->GAP->BN1d), {CPU_BATCH} of {BATCH} "
                                                    "synthetic 256x128 crops per step, random-init weights, fp32 on the host cores")
        per_step = CPU_BATCH
    elif args.workload == "train":
        r = cpu_train(min(args.steps, 5), 1)
        metric, name = "CTL training step images/sec", "BASELINE config 1: CTLModel.training_step, ResNet50 256x128, B = 128 (32 x 4), fp32"
        per_step = 128
    else:
        r = cpu_retrieval(256)
        r["steps_run"] = 1
        metric, name = "QxG top-k pairs/sec", f"256 of {RET_Q} queries x {RET_G} gallery (config 3 slice), top-k + CMC/mAP"
        per_step = 256 * RET_G
    done = r.get("steps_run", 1)
    line = {"metric": metric, "value": r["value"], "unit": r["unit"], "impl": "reference", "n_gpus": args.gpus,
            "steps": done, "requested_steps": args.steps, "warmup": min(args.warmup, 2),
            "ms_per_step": (per_step / r["value"] * 1e3) if r["value"] else None, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": name},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="embed", choices=["embed", "retrieval", "train"])
    ap.add_argument("--train-model", default="resnet50", choices=["resnet50", "resnet50_ibn_a"])
    ap.add_argument("--train-size", default="256x128", help="HxW of the training crops (config 4: 320x320)")
    ap.add_argument("--train-pk", default="16x16", help="ids x instances per GPU (config 4: 32x4)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the nested metrics and the CPU baselines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (emb, global_feat) as DIR/<name>.npy "
                         "(float32); the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "embed"):
        ap.error("--dump-outputs records the embed workload of --impl ours")
    args.warmup = max(args.warmup, 3)
    world, rank, local = dist_env()

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    workload_name = (f"resnet50 eval embedding forward (trunk->GAP->BN1d), {BATCH} synthetic 256x128 crops per GPU, "
                     "random-init weights")

    def guarded(fn, *a, **k):
        import contextlib

        try:
            with contextlib.redirect_stdout(sys.stderr):  # stdout carries the ONE JSON line only
                return fn(*a, **k)
        except Exception as exc:  # a failing nested metric must not take the primary line with it
            return {"error": f"{type(exc).__name__}: {exc}"}

    try:
        if args.workload == "embed":
            ms, value, launches, e2e, roof, clocks = run_embed(args, world, rank, local)
            line = {"metric": "embeddings/sec @256x128", "value": value, "unit": "embeddings/s",
                    "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
                    "data": "synthetic",
                    "config": {"workload": workload_name, "batch_per_gpu": BATCH, "global_batch": BATCH * world,
                               "model": "resnet50 last_stride=1", "gflop_per_embedding": GFLOP_PER_IMG,
                               "l2": "4 rotating input batches (403 MB) > 126 MB L2; per-layer activations 67-268 MB",
                               "parallelism": f"dp{world}: per-rank batches, ONE NCCL all_gather_into_tensor of the "
                                              "extracted embeddings inside the timed region"},
                    "tflops": value * GFLOP_PER_IMG / 1e3, "roofline": roof, "e2e": e2e, "gpu_launches": launches,
                    "clocks": clocks}
            if not args.no_secondary:
                if world == 1:
                    line["retrieval"] = guarded(run_retrieval, args, world, rank, local, steps=5, warmup=3)
                    line["train_step"] = guarded(run_train_step, local)
                    line["cpu_baseline"] = guarded(cpu_embed, 3, 1, 60.0)
                    if isinstance(line["retrieval"], dict) and "error" not in line["retrieval"]:
                        line["retrieval"]["cpu_baseline"] = guarded(cpu_retrieval, 128)
                    if isinstance(line["train_step"], dict) and "error" not in line["train_step"]:
                        line["train_step"]["cpu_baseline"] = guarded(cpu_train, 2, 1, 90.0)
                else:
                    line["retrieval"] = guarded(run_retrieval_sharded, args, world, rank, local)
                    line["train_step"] = guarded(run_train_step, local, 5, 2, "resnet50_ibn_a", (320, 320), 32, 4, world)
        elif args.workload == "train":
            hh, ww = (int(v) for v in args.train_size.split("x"))
            pp, kk = (int(v) for v in args.train_pk.split("x"))
            if world > 1:
                dist.barrier()
            with ClockSampler(local) as clk:
                with clk.window():
                    r = run_train_step(local, steps=args.steps, warmup=args.warmup, model_name=args.train_model,
                                       size=(hh, ww), P=pp, K=kk, world=world)
            line = {"metric": r["metric"], "value": r["value"], "unit": r["unit"], "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                    "config": {"workload": f"CTL training iteration, {args.train_model} {hh}x{ww}, {pp} ids x {kk} instances per GPU, "
                                           "random-init weights", "global_batch": pp * kk * world,
                               "parallelism": f"dp{world}: per-rank P x K batches, NCCL mean all-reduce of the gradients"},
                    "loss": r["loss"], "peak_mem_gib": r["peak_mem_gib"], "clocks": clk.summary(),
                    "roofline": r["roofline"], "e2e": None, "note": r["note"]}
            if rank == 0 and not args.no_secondary and world == 1:
                line["cpu_baseline"] = guarded(cpu_train, 2, 1, 90.0)
        else:
            with ClockSampler(local) as clk:
                with clk.window():
                    r = run_retrieval_sharded(args, world, rank, local, steps=args.steps, warmup=args.warmup) if world > 1 \
                        else run_retrieval(args, world, rank, local)
            line = {"metric": r["metric"], "value": r["value"], "unit": r["unit"], "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "f16x3 (fp32-equivalent split)", "data": "synthetic",
                    "config": r["config"], "roofline": r.get("roofline"), "e2e": r.get("e2e"),
                    "gpu_launches": r.get("gpu_launches_per_step", 12) * args.steps,
                    "clocks": clk.summary(), "mAP": r["mAP"], "rank1": r["rank1"]}
            if "sharded_equals_single_gpu" in r:
                line["sharded_equals_single_gpu"] = r["sharded_equals_single_gpu"]
            if rank == 0 and not args.no_secondary and world == 1:
                line["cpu_baseline"] = guarded(cpu_retrieval, 128)
        if rank == 0:
            print(json.dumps(line))
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
