#!/usr/bin/env python
"""bench.py -- images/s of the embedding-to-distance hot path (patchify -> alpha -> X -> dist).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input: hooked backbone feature maps resident
in HBM -> Z -> w -> alpha -> X -> Dmat resident in HBM (BASELINE.json metric).  `value` is the device-timed
whole-job throughput (CUDA events, max over ranks); `e2e` repeats the measurement through the public API with
HOST feature buffers (pinned) and host results, copies inside the timed region.

Workloads = BASELINE.json's configs (the default, config2, is the one the metric is quoted on):
    config1   WRN50 layer2+layer3 shape, 20 images, unsupervised tau=1
    config2   ViT-B/8 shape, 100 images x 784 patches x 4096-d, unsupervised tau=1
    config3   config-2 queries against a 200-image normal bank: supervised alpha + the 'average' mode
    config4   1210 images, ONE joint bank (every image against the other 1209), unsupervised
    config4pc 10 MVTec-object-sized categories, per-category banks (the reference's semantics, main.py:353)
    config5   ViT-S/8 at 448x448 shape (3136 patches), 64 images, 6 taus incl. 0.1 from one distance pass
At N > 1: unsupervised / supervised workloads shard the query images over the ranks (operand all-gather over NCCL,
X rows gathered back; strong scaling of the same workload); config4pc assigns whole categories to ranks (LPT, no
collective).  During warm-up rank 0 also runs the whole workload alone and compares -> `parity_ok`.
`--impl reference` times the oracle port of the reference's torch CPU path on the host cores.
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (alpha, X, Dmat, w, ...) as DIR/<name>.npy; the
synthetic inputs depend only on the arguments, so two builds can be compared output for output."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/s (patchify→alpha→X→dist)"

VITB = [(768, 28, 28, True), (768, 28, 28, True)]
MVTEC_OBJECT_SIZES = [83, 150, 132, 110, 115, 167, 160, 42, 100, 151]   # test-set sizes of the 10 object categories (info_*.pickle)

WORKLOADS = {
    "config1": dict(
        name="config1: WideResNet50 layer2+layer3 shape, 20 synthetic images x 784 patches, 1024->1024, unsupervised tau=1",
        layers=[(512, 28, 28, False), (1024, 14, 14, False)], n_img=20, Dp=1024, D=1024, taus=[1.0], mode="unsupervised"),
    "config2": dict(
        name="config2: DINO ViT-B/8 blocks.10+blocks.11 shape, 100 synthetic images x 784 patches, 2048->4096, unsupervised tau=1",
        layers=VITB, n_img=100, Dp=2048, D=4096, taus=[1.0], mode="unsupervised"),
    "config3": dict(
        name="config3: DINO ViT-B/8 shape, 100 query images against a 200-image normal bank, 2048->4096, supervised tau=1 + average mode",
        layers=VITB, n_img=100, n_bank=200, Dp=2048, D=4096, taus=[1.0], mode="supervised"),
    "config4": dict(
        name="config4 (joint bank): 1210 synthetic images x 784 patches (10 MVTec-object-sized categories), 2048->4096, unsupervised tau=1",
        layers=VITB, n_img=1210, Dp=2048, D=4096, taus=[1.0], mode="unsupervised"),
    "config4pc": dict(
        name="config4 (per-category banks): 10 MVTec-object-sized categories, 1210 synthetic images x 784 patches, 2048->4096, unsupervised tau=1",
        layers=VITB, sizes=MVTEC_OBJECT_SIZES, n_img=sum(MVTEC_OBJECT_SIZES), Dp=2048, D=4096, taus=[1.0], mode="percategory"),
    "config5": dict(
        name="config5: ViT-S/8 at 448x448 shape, 64 synthetic images x 3136 patches, 2048->4096, unsupervised, taus 0.1..10 from one distance pass",
        layers=[(384, 56, 56, True), (384, 56, 56, True)], n_img=64, Dp=2048, D=4096, taus=[0.1, 0.5, 1.0, 2.0, 5.0, 10.0],
        mode="unsupervised"),
    # CI smokes of the bench itself
    "tiny13": dict(
        name="tiny13: 2x[96,12,12] tokens, 13 images x 144 patches, 256->512 (uneven shards on 2+ ranks; CI smoke)",
        layers=[(96, 12, 12, True), (96, 12, 12, True)], n_img=13, Dp=256, D=512, taus=[1.0], mode="unsupervised"),
    "tiny": dict(
        name="tiny: 2x[96,12,12] tokens, 12 images x 144 patches, 256->512 (CI smoke of the bench itself)",
        layers=[(96, 12, 12, True), (96, 12, 12, True)], n_img=12, Dp=256, D=512, taus=[1.0], mode="unsupervised"),
    "tiny3": dict(
        name="tiny3: 2x[96,12,12] tokens, 9 query images vs a 7-image bank, 256->512, supervised + average (CI smoke)",
        layers=[(96, 12, 12, True), (96, 12, 12, True)], n_img=9, n_bank=7, Dp=256, D=512, taus=[1.0, 0.25], mode="supervised"),
    "tinypc": dict(
        name="tinypc: 2x[96,12,12] tokens, categories of 5+9+4+7 images, 256->512, per-category banks (CI smoke)",
        layers=[(96, 12, 12, True), (96, 12, 12, True)], sizes=[5, 9, 4, 7], n_img=25, Dp=256, D=512, taus=[1.0], mode="percategory"),
}


def patches_of(wl):
    return wl["layers"][0][1] * wl["layers"][0][2]     # 3x3 patches, stride 1: the patch grid is the layer-0 map


def workload_config(wl):
    """The `config` object of the JSON line -- identical for the GPU arm and the reference arm (the driver compares them);
    everything implementation-specific goes to `impl_config`."""
    P = patches_of(wl)
    maps_mb = wl["n_img"] * sum(c * h * w * 4 for c, h, w, _ in wl["layers"]) / 1e6
    cfg = {"workload": wl["name"], "mode": wl["mode"] + (" + average" if wl["mode"] == "supervised" else ""), "n_images": wl["n_img"],
           "bank_images": wl.get("n_bank"), "category_sizes": wl.get("sizes"), "patches_per_image": P, "pretrain_dim": wl["Dp"],
           "embed_dim": wl["D"], "taus": wl["taus"],
           "l2": "inputs larger than L2 (feature maps %.0f MB + embeddings %.0f MB per step vs 126 MB of L2)"
                 % (maps_mb, wl["n_img"] * P * wl["D"] * 2 / 1e6) if maps_mb > 130 else
                 "inputs fit L2: every step re-reads the same %.0f MB of feature maps (launch-bound workload, not a bandwidth claim)" % maps_mb}
    return cfg


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 1024          # allowance per file for the .npy header (np.save writes 128 bytes for these shapes)


def dump_outputs(out, directory, limit_bytes=DUMP_LIMIT_BYTES):
    """Writes the tensors of one step's result `out` ({name: tensor or list of tensors}) as <directory>/<name>.npy, a list
    as <name>_<i>.npy.  float64 stays float64, every other dtype is stored as float32.  The files hold at most
    `limit_bytes` in all: the smallest arrays are written whole, and an array larger than its share of what is left is
    replaced by a 1-D sample of its flattened elements at sorted indices drawn from np.random.default_rng(0), so the
    sample depends only on the array's shape and is the same for every build.  Returns {file name: (shape, sampled)}."""
    import numpy as np
    import torch

    items = []
    for name in sorted(out):
        v = out[name]
        items += [("%s_%d" % (name, i), t) for i, t in enumerate(v)] if isinstance(v, (list, tuple)) else [(name, v)]
    items = [(n, t, 8 if t.dtype == torch.float64 else 4) for n, t in items]
    items.sort(key=lambda it: (it[1].numel() * it[2], it[0]))
    os.makedirs(directory, exist_ok=True)
    left = limit_bytes - NPY_HEADER_BYTES * len(items)
    written = {}
    for k, (name, t, size) in enumerate(items):
        share = left // (len(items) - k)
        x = t.detach().reshape(-1)
        sampled = x.numel() * size > share
        if sampled:
            idx = np.unique(np.random.default_rng(0).integers(0, x.numel(), size=max(1, share // size)))
            x = x[torch.from_numpy(idx).to(x.device)]
        arr = x.to("cpu", torch.float64 if size == 8 else torch.float32).numpy()
        if not sampled:
            arr = arr.reshape(tuple(t.shape))
        np.save(os.path.join(directory, name + ".npy"), arr)
        left -= arr.nbytes
        written[name + ".npy"] = (tuple(t.shape), sampled)
    return written


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons DURING the timed region (B200_PROFILING.md's clocks line).
    The sampler is started BEFORE the warm-up steps (nvidia-smi needs a few hundred ms before its first line) and
    the samples are cut to the timed window by their timestamps; when the timed region is shorter than two
    sampling periods the under-load samples of warm-up + timed region are used and `window` says so.
    Never raises: a failure is reported inside the record."""

    QUERY = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 50

    def __init__(self, gpu_index: int):
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                 "-lms", str(self.PERIOD_MS)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    @staticmethod
    def parse(out: str):
        """-> list of (epoch seconds | None, sm MHz, max sm MHz, power W, set of active slowdown reasons)."""
        import datetime

        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 10:
                continue
            try:
                sm, mx, pw = float(f[2]), float(f[3]), float(f[4])
            except ValueError:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = None
            reasons = {name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10])
                       if v.lower().startswith("active")}
            rows.append((ts, sm, mx, pw, reasons))
        return rows

    @staticmethod
    def summarise(rows, t_begin=None, t_end=None):
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        window = "timed region"
        sel = [r for r in rows if r[0] is not None and t_begin is not None and t_begin <= r[0] <= t_end]
        if len(sel) < 2:
            # timed region shorter than two sampling periods (or no usable timestamps): under-load samples of the
            # whole run of the sampler (warm-up + timed region, same kernels back to back)
            top = max(r[3] for r in rows)
            sel = [r for r in rows if r[3] > 0.5 * top] or rows
            window = "warm-up + timed region (under-load samples; timed region shorter than 2 sampling periods)"
        reasons = set()
        for r in sel:
            reasons |= r[4]
        return {"sm_mhz": statistics.median(r[1] for r in sel), "sm_max_mhz": max(r[2] for r in sel),
                "power_w_max": max(r[3] for r in sel), "samples": len(sel), "window": window, "reasons": sorted(reasons)}

    def stop(self, t_begin=None, t_end=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        try:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            return self.summarise(self.parse(out), t_begin, t_end)
        except Exception as e:   # noqa: BLE001 -- the clocks record must never take the bench line down
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["sampler error: %r" % (e,)]}


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_sample_plan(wl, n_q):
    """(query images, bank images) of one bounded CPU sample.  Cost is exactly linear in query images, so the sample is
    n_q query images against the FULL bank they see in the workload (per-category: a bank of the workload's mean size)."""
    if wl["mode"] == "supervised":
        return n_q, wl["n_bank"]
    if wl["mode"] == "percategory":
        s = wl["sizes"]
        return n_q, max(2, round(sum(n * (n - 1) for n in s) / sum(s)))
    return n_q, wl["n_img"] - 1


def cpu_path_sample(wl, feats_q, Zbank, self_idx=None, want=False):
    """One bounded sample of the reference's CPU path (oracle port): embed the query images, min-distance of those images
    against the given bank, alpha per tau, X, pairwise distances.  self_idx: unsupervised, the bank index of each query
    image (its own column is dropped, utils.py:224-225); None: supervised (min over the bank, utils.py:234-236).
    The supervised workload also runs the 'average' mode (main.py:290-291).  Returns seconds (and the results if asked)."""
    import torch

    from oracle import restated

    n_q, D = feats_q[0].shape[0], wl["D"]
    t0 = time.perf_counter()
    Zq = restated.embed(feats_q, 3, 1, wl["Dp"], D).reshape(n_q, -1, D)
    dm = restated.per_image_min_dist(Zq, Zbank)            # [n_q, P, n_bank]
    if wl["mode"] == "supervised":
        w = dm.min(dim=2)[0]
    elif self_idx is not None:
        keep = torch.ones(n_q, Zbank.shape[0], dtype=torch.bool)
        keep[torch.arange(n_q), torch.as_tensor(self_idx)] = False
        w = torch.stack([dm[i][:, keep[i]].mean(dim=1) for i in range(n_q)])
    else:
        w = dm.mean(dim=2)
    outs = []
    for tau in wl["taus"]:
        alpha = restated.alpha_from_weights(w, tau, stable=True)
        X = restated.weighted_embedding(alpha, Zq)
        outs.append((alpha, X, restated.pairwise_euclidean(X)))
    if wl["mode"] == "supervised":
        Xa = restated.weighted_embedding(restated.matrix_alpha_average(n_q, Zq.shape[1]), Zq)
        restated.pairwise_euclidean(Xa)
    dt = time.perf_counter() - t0
    return (dt, w, outs) if want else dt


def oracle_embed_chunked(wl, feats, chunk=8):
    import torch

    from oracle import restated

    n = feats[0].shape[0]
    Z = torch.cat([restated.embed([f[a:a + chunk] for f in feats], 3, 1, wl["Dp"], wl["D"]) for a in range(0, n, chunk)], dim=0)
    return Z.reshape(n, -1, wl["D"])


def run_reference_arm(args, wl):
    """--impl reference: the reference's own torch CPU implementation of the path (oracle port; the reference is a Python
    script tree that cannot travel to the GPU box), all host threads.  A step is one bounded sample of the workload:
    `--cpu-sample` query images embedded and taken against the FULL, really embedded bank (embedding the bank is set-up,
    like the feature generation).  `ms_per_step` is what a step took; the extrapolation to a whole pass is its own field."""
    import torch

    from anomaly_clustering_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_q, n_bank = cpu_sample_plan(wl, max(1, args.cpu_sample))
    n_q = min(n_q, wl["n_img"])
    sup = wl["mode"] == "supervised"
    # the GPU arm's synthetic data set (same construction, generated on the CPU here).  Supervised: queries 0..n_q-1
    # against the normal images.  Unsupervised: the bank is the data set itself (n_bank + 1 images, the queries
    # included) and every query drops its own column -- "all other images", exactly utils.py:222-227.
    if sup:
        feats_q, _ = synth.planted_features_device(range(n_q), wl["layers"], seed=2023, device="cpu")
        feats_b, _ = synth.planted_features_device(range(1000, 1000 + n_bank), wl["layers"], n_classes=1, seed=2023, device="cpu")
        self_idx = None
    else:
        feats_b, _ = synth.planted_features_device(range(n_bank + 1), wl["layers"], seed=2023, device="cpu")
        feats_q = [f[:n_q] for f in feats_b]
        self_idx = list(range(n_q))
    Zbank = oracle_embed_chunked(wl, feats_b)
    del feats_b
    for _ in range(args.warmup):
        cpu_path_sample(wl, feats_q, Zbank, self_idx)
    t = [cpu_path_sample(wl, feats_q, Zbank, self_idx) for _ in range(args.steps)]
    total = sum(t)
    value = n_q * args.steps / total
    sample = ("%d query images embedded + cdist/min against the full %d-image bank (really embedded) + alpha (%d taus) + X + "
              "pdist per step" % (n_q, n_bank, len(wl["taus"])))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl),
        "impl_config": {"sample": sample, "images_per_step": n_q,
                        "ms_per_full_pass_extrapolated": 1e3 * total / args.steps * (wl["n_img"] / n_q),
                        "note": "cost is exactly linear in query images: value (images/s) is measured on the sample, the full pass is "
                                "never run on the CPU"},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="auto", choices=["auto", "f16", "bf16", "f16x3", "bf16x3", "f16r", "f32"])
    ap.add_argument("--cpu-sample", type=int, default=2, help="query images per CPU-baseline sample")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="CPU-baseline leg: repeat the sample until this much CPU time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true", help="N > 1: skip the single-rank comparison during warm-up")
    ap.add_argument("--keep-z", action="store_true",
                    help="materialise the fp32 Z (1.3 GB at config 2); default: operands only from the embed kernel, X from the feature maps")
    ap.add_argument("--z-free", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--no-symmetry", action="store_true", help="force the all-pairs distance kernel (every image pair multiplied twice)")
    ap.add_argument("--cuda-profiler", action="store_true", help="cudaProfilerStart/Stop around the timed steps (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float32 / float64, at most 64 MB")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    wl = WORKLOADS[args.workload]
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args, wl)

    # keep the real stdout for the ONE JSON line: libraries (NCCL prints its version banner) write to fd 1
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    from anomaly_clustering_b200 import distributed, ops, pipeline, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():          # (scripts/r02_multi.py runs several workloads in one process group)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not ops.device_ok(local_rank):
        raise SystemExit("device %d is not sm_100" % local_rank)
    dev = torch.device("cuda", local_rank)
    peaks = load_peaks()

    n_img, layers, Dp, D, taus, mode = wl["n_img"], wl["layers"], wl["Dp"], wl["D"], wl["taus"], wl["mode"]
    P = patches_of(wl)
    keep_z = args.keep_z
    precision = pipeline.resolve_precision(args.precision, taus)
    symmetric = (not args.no_symmetry) and precision != "f32" and mode != "supervised"
    pipeline.SYMMETRIC = symmetric

    # ---------------------------------------------------------------- this rank's share of the synthetic data set
    bank = None
    if mode == "percategory":
        sizes = wl["sizes"]
        bins = distributed.lpt_assign([float(n) * (n - 1) for n in sizes], world)   # whole categories to ranks (SURVEY 8e)
        my_cats = sorted(bins[rank])
        my_sizes = [sizes[c] for c in my_cats]
        ids = [1000 * c + i for c in my_cats for i in range(sizes[c])]
        feats, _ = synth.planted_features_device(ids, layers, seed=2023, device=dev) if ids else (None, None)
        nq_local = len(ids)
    else:
        lo_i, hi_i = distributed.shard_bounds(n_img, world)[rank]
        feats, _ = synth.planted_features_device(range(lo_i, hi_i), layers, seed=2023, device=dev)
        nq_local = hi_i - lo_i
        if mode == "supervised":
            blo, bhi = distributed.shard_bounds(wl["n_bank"], world)[rank]
            bank, _ = synth.planted_features_device(range(1000 + blo, 1000 + bhi), layers, n_classes=1, seed=2023, device=dev)
    inputs = [] if feats is None else list(feats) + (list(bank) if bank is not None else [])
    nf = 0 if feats is None else len(feats)

    def step(inp):
        """One pass over this rank's inputs -> dict of device results (what the public API returns)."""
        f, b = inp[:nf], inp[nf:]
        if mode == "unsupervised":
            if world == 1:
                r = pipeline.run_path(f, 3, 1, Dp, D, "unsupervised", taus, precision=precision, keep_z=keep_z)
                return {"alpha": r.alpha32, "X": r.X, "Dmat": r.Dmat, "w": r.w}
            a64, X, Dm, w = distributed.run_path_sharded(f, n_img, 3, 1, Dp, D, taus, precision=precision, symmetric=symmetric,
                                                         keep_z=keep_z)
            return {"alpha": a64, "X": X, "Dmat": Dm, "w": w}
        if mode == "supervised":
            if world == 1:
                r = pipeline.run_path(f, 3, 1, Dp, D, "supervised", taus, bank_features=b, precision=precision, keep_z=keep_z)
                ra = pipeline.run_path(f, 3, 1, Dp, D, "average", keep_z=False)
                return {"alpha": r.alpha32, "X": r.X, "Dmat": r.Dmat, "w": r.w, "X_avg": ra.X, "Dmat_avg": ra.Dmat}
            a64, X, Dm, w = distributed.run_path_sharded_supervised(f, n_img, b, wl["n_bank"], 3, 1, Dp, D, taus, precision=precision)
            Xa, Da = distributed.run_path_sharded_average(f, n_img, 3, 1, Dp, D)
            return {"alpha": a64, "X": X, "Dmat": Dm, "w": w, "X_avg": Xa, "Dmat_avg": Da}
        if not my_sizes:
            return {}
        rs = pipeline.run_categories(f, my_sizes, 3, 1, Dp, D, taus, precision=precision, keep_z=keep_z)
        return {"alpha": torch.cat([r.alpha32 for r in rs], dim=1), "X": torch.cat([r.X for r in rs], dim=1),
                "Dmat": [r.Dmat for r in rs], "w": torch.cat([r.w for r in rs], dim=0)}

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident timing
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # before the warm-up: nvidia-smi is slow to emit its first line
    out = None
    for _ in range(args.warmup):
        out = step(inputs)
    sync_all()

    # ---------------------------------------------------------------- N > 1: the sharded result against ONE rank running it all
    parity = None
    if world > 1 and not args.no_parity_check:
        parity = multi_rank_parity(wl, out, step, rank, world, dev, precision, symmetric, keep_z)
        sync_all()

    pipeline.PROFILE = []
    launches0 = ops.launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    if args.cuda_profiler:
        torch.cuda.profiler.start()
    t_begin = time.time()
    ev0.record()
    for _ in range(args.steps):
        out = step(inputs)
    ev1.record()
    sync_all()
    t_end = time.time()
    if args.cuda_profiler:
        torch.cuda.profiler.stop()
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    launches = ops.launches() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)       # before the untimed legs below run the path again
    elapsed_ms = ev0.elapsed_time(ev1)
    marks = pipeline.PROFILE
    pipeline.PROFILE = None
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())

    # per-kernel time of the dominant kernel (tcgen05 min-distance), CUDA events on the launch stream
    def span(tag):
        b = [e for n, e in marks if n == tag + "_begin"]
        e_ = [e for n, e in marks if n == tag + "_end"]
        return sum(x.elapsed_time(y) for x, y in zip(b, e_)) / max(1, args.steps)

    comm = {t_: span(t_) for t_ in ("gather", "exchange", "xgather")} if world > 1 else {}
    md_ms, emb_ms, refine_ms = span("mindist"), span("embed"), span("refine")
    # algorithmic FLOPs of this rank's share: self pairs excluded, no padding charged (SURVEY 8d)
    if mode == "supervised":
        flops = 2.0 * (nq_local * P) * (wl["n_bank"] * P) * D
        exec_flops = flops
    elif mode == "percategory":
        flops = sum(2.0 * n * (n - 1) * P * P * D for n in my_sizes)
        exec_flops = flops / 2 if symmetric else flops
    else:
        flops = 2.0 * (nq_local * P) * ((n_img - 1) * P) * D
        if symmetric:
            # the symmetric kernel multiplies each unordered image pair once (cdist(Zi,Zj) = cdist(Zj,Zi)^T):
            # tensor-pipe utilisation is reported on the EXECUTED flops, the algorithmic rate beside it
            owned = sum(distributed.pair_owned(i, j, n_img) for i in range(lo_i, hi_i) for j in range(n_img))
            exec_flops = 2.0 * owned * P * P * D
        else:
            exec_flops = flops
    if precision in ("f16x3", "bf16x3"):
        exec_flops *= 3          # three MMA passes per tile
    tflops = exec_flops / (md_ms * 1e-3) / 1e12 if md_ms > 0 else 0.0
    alg_tflops = flops / (md_ms * 1e-3) / 1e12 if md_ms > 0 else 0.0
    z_free = (not keep_z) and feats is not None and pipeline.z_free_supported(feats, 3, 1, Dp, D, precision) and precision not in pipeline.REFINED
    n_embedded = nq_local + (0 if bank is None else bank[0].shape[0])
    op_bytes = 0 if precision == "f32" else (4 if precision in ("f16x3", "bf16x3") else 2)
    embed_bytes = n_embedded * (sum(c * h * w * 4 for c, h, w, _ in layers) + P * D * op_bytes + P * 4) + (0 if z_free else nq_local * P * D * 4)
    embed_gbs = embed_bytes / (emb_ms * 1e-3) / 1e9 if emb_ms > 0 else 0.0
    # The same embed launch sequence timed ALONE (back to back, after an idle moment): inside a step it inherits the
    # power-capped SM clock of the tensor kernel before it and its time scales with that clock (DESIGN 5b)
    emb_iso_ms = None
    if world == 1 and mode == "unsupervised" and feats is not None:
        operand = "f32" if precision == "f32" else precision
        torch.cuda.synchronize()
        time.sleep(0.2)
        for _ in range(3):
            pipeline.embed_images(feats, 3, 1, Dp, D, operand, want_z=not z_free)
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        i0.record()
        for _ in range(20):
            pipeline.embed_images(feats, 3, 1, Dp, D, operand, want_z=not z_free)
        i1.record()
        torch.cuda.synchronize()
        emb_iso_ms = i0.elapsed_time(i1) / 20

    # ---------------------------------------------------------------- end-to-end (host buffers)
    e2e = None
    if not args.no_e2e:
        host = [f.cpu().pin_memory() for f in inputs]
        h2d = sum(f.numel() * 4 for f in host)
        res_host = None

        # Public-API streaming driver: consecutive batches are double-buffered, the H2D copy of step
        # i+1 (copy stream) overlaps the compute of step i; every step's copy and its D2H result read are
        # inside the timed region.
        copy_stream = torch.cuda.Stream()
        main_stream = torch.cuda.current_stream()
        bufs = [[torch.empty_like(f) for f in inputs] for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]

        def issue_copy(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[slot])
                for d_, h_ in zip(bufs[slot], host):
                    d_.copy_(h_, non_blocking=True)
                ready[slot].record(copy_stream)

        def flat(o):
            res = []
            for k in sorted(o):
                if k == "w":
                    continue
                v = o[k]
                res += list(v) if isinstance(v, list) else [v]
            return res

        def e2e_run(nsteps):
            nonlocal res_host
            d2h_bytes = 0
            for sl in range(2):
                freed[sl].record(main_stream)
            issue_copy(0)
            for i in range(nsteps):
                slot = i & 1
                if i + 1 < nsteps:
                    issue_copy(slot ^ 1)
                main_stream.wait_event(ready[slot])
                o = step(bufs[slot])
                freed[slot].record(main_stream)
                # every rank reads its alpha rows back; the gathered X / Dmat once (rank 0) when they are replicated
                outs = flat(o) if (rank == 0 or mode == "percategory") else [o["alpha"]]
                if res_host is None:
                    res_host = [torch.empty(x.shape, dtype=x.dtype).pin_memory() for x in outs]
                for h_, x in zip(res_host, outs):
                    h_.copy_(x, non_blocking=True)
                d2h_bytes = sum(x.numel() * x.element_size() for x in outs)
            return d2h_bytes

        # raw pinned-host -> device copy rate of this box (explains the gap between `value` and `e2e`)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        issue_copy(0); torch.cuda.synchronize()
        c0.record(copy_stream); issue_copy(0); c1.record(copy_stream); torch.cuda.synchronize()
        h2d_gbps = h2d / max(c0.elapsed_time(c1), 1e-6) * 1e3 / 1e9
        d2h = e2e_run(3)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        d2h = e2e_run(args.steps)
        e1.record()
        sync_all()
        te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        tb = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dist.all_reduce(tb, op=dist.ReduceOp.SUM)
        e2e = {"value": n_img * args.steps / (float(te.item()) * 1e-3), "unit": "images/s",
               "h2d_bytes_per_step": int(tb[0].item()), "d2h_bytes_per_step": int(tb[1].item()),
               "h2d_GBps_measured_per_gpu": h2d_gbps}
        del bufs, host

    # ---------------------------------------------------------------- CPU baseline + oracle check (rank 0, N = 1)
    cpu_baseline = None
    torch_gpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline, parity = cpu_baseline_leg(args, wl, pipeline, feats, bank, out, precision)
        torch_gpu = torch_gpu_reference_leg(wl, pipeline, feats, bank, out)

    if rank == 0:
        value = n_img * args.steps / (elapsed_ms * 1e-3)
        traffic = None
        prof = os.path.join(ROOT, "profiles", "ncu_summary.json")
        if os.path.exists(prof):
            try:
                with open(prof) as f:
                    traffic = json.load(f).get("mindist_tc_dram_bytes_per_launch", {}).get(args.workload if world == 1 else "", None)
            except Exception:
                traffic = None
        if mode == "percategory":
            par = "whole categories to ranks by LPT on n_c(n_c-1), no collective: %s" % (bins,) if world > 1 else "single GPU"
        elif world > 1:
            transport = ("symmetric-memory pulls (copy engines) + one flag-driven distance launch" if os.environ.get("AC_SHARD_TRANSPORT", "symm") == "symm"
                         else "NCCL collectives")
            par = "query-sharded x%d, operand transport: %s, X gather (NCCL)" % (world, transport)
        else:
            par = "single GPU"
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": precision, "data": "synthetic",
            "config": workload_config(wl),
            "impl_config": {"precision": precision, "precision_requested": args.precision, "symmetric_pairs": symmetric,
                            "fp32_Z_materialised": not z_free, "parallelism": par,
                            "e2e_mode": "pinned host features -> H2D (copy stream, overlapped with the previous step's compute) -> path -> "
                                        "D2H of alpha, X, Dmat"},
            "parity_ok": None if parity is None else bool(parity.get("ok")),
            "parity": parity,
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "mindist_tc_kernel (tcgen05, fused per-image row-min)",
                         "achieved": tflops, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                         "frac": tflops / peaks["bf16_sustained"], "peak_burst": peaks["bf16_burst"],
                         "frac_of_burst": tflops / peaks["bf16_burst"], "peak_source": peaks["source"] + " (sustained: kernel timed inside a long step)",
                         "ms_per_step": md_ms, "flops_per_launch": exec_flops,
                         "flops_counted": ("executed: each unordered image pair multiplied once (symmetric kernel); "
                                           "the all-pairs algorithmic count is algorithmic_flops_per_launch") if symmetric
                         else "algorithmic = executed (all-pairs kernel)",
                         "algorithmic_flops_per_launch": flops, "algorithmic_tflops": alg_tflops, "traffic": traffic},
            "stages": {"embed_ms_per_step": emb_ms, "embed_bytes_per_step": embed_bytes, "embed_GBps": embed_gbs,
                       "embed_frac_of_hbm": embed_gbs / peaks["hbm_gbs"],
                       "embed_isolated_ms": emb_iso_ms,
                       "embed_isolated_frac_of_hbm": None if not emb_iso_ms else embed_bytes / (emb_iso_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                       "mindist_ms_per_step": md_ms, "refine_ms_per_step": refine_ms,
                       "other_ms_per_step": elapsed_ms / args.steps - emb_ms - md_ms - refine_ms,
                       "comm_ms_per_step_rank0": comm},
            "cpu_baseline": cpu_baseline,
            "reference_loop_on_gpu": torch_gpu,
        }
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    os.dup2(real_stdout, 1)          # give fd 1 back (main() may be called again in this process)
    os.close(real_stdout)
    if world > 1 and os.environ.get("AC_BENCH_KEEP_PG", "0") != "1":
        dist.destroy_process_group()


def _rel(a, b):
    return float(((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item())


def multi_rank_parity(wl, out, step, rank, world, dev, precision, symmetric, keep_z):
    """N > 1 self-check (untimed, during warm-up): rank 0 runs the WHOLE workload alone through the single-GPU path and
    compares the sharded result with it -- X and Dmat of all images, w and alpha of its own rows.  Per-category workloads
    have no cross-rank arithmetic: there every rank recomputes the smallest category and the checksums must agree."""
    import torch
    import torch.distributed as dist

    from anomaly_clustering_b200 import distributed, pipeline, synth

    layers, Dp, D, taus, mode, n_img = wl["layers"], wl["Dp"], wl["D"], wl["taus"], wl["mode"], wl["n_img"]
    res = {"ok": True}
    if mode == "percategory":
        c = min(range(len(wl["sizes"])), key=lambda i: wl["sizes"][i])
        f, _ = synth.planted_features_device([1000 * c + i for i in range(wl["sizes"][c])], layers, seed=2023, device=dev)
        r = pipeline.run_path(f, 3, 1, Dp, D, "unsupervised", taus, precision=precision, keep_z=keep_z)
        cs = torch.stack([r.X.double().sum(), r.Dmat.double().sum(), r.w.double().sum()])
        lo, hi = cs.clone(), cs.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        res.update(check="every rank recomputed category %d; checksums of X, Dmat, w across ranks" % c,
                   max_spread=float((hi - lo).abs().max().item()))
        res["ok"] = bool(torch.equal(lo, hi))
        return res
    flag = torch.ones(1, device=dev)
    if rank == 0:
        lo_i, hi_i = distributed.shard_bounds(n_img, world)[0]
        allf, _ = synth.planted_features_device(range(n_img), layers, seed=2023, device=dev)
        if mode == "supervised":
            allb, _ = synth.planted_features_device(range(1000, 1000 + wl["n_bank"]), layers, n_classes=1, seed=2023, device=dev)
            ref = pipeline.run_path(allf, 3, 1, Dp, D, "supervised", taus, bank_features=allb, precision=precision, keep_z=keep_z)
        else:
            ref = pipeline.run_path(allf, 3, 1, Dp, D, "unsupervised", taus, precision=precision, keep_z=keep_z)
        e_w = float(((out["w"] - ref.w[lo_i:hi_i]).abs() / ref.w[lo_i:hi_i].abs().clamp_min(1e-6)).max().item())
        e_a = float((out["alpha"].double() - ref.alpha64[:, lo_i:hi_i]).abs().max().item())
        e_x, e_d = _rel(out["X"], ref.X), _rel(out["Dmat"], ref.Dmat)
        res.update(check="rank 0 ran all %d images alone (single-GPU path)" % n_img, w_max_rel=e_w, alpha_max_abs=e_a, X_rel_l2=e_x,
                   Dmat_rel_l2=e_d, bit_identical=bool(torch.equal(out["X"], ref.X) and torch.equal(out["Dmat"], ref.Dmat)))
        res["ok"] = e_w <= 1e-5 and e_a <= 1e-5 and e_x <= 1e-5 and e_d <= 1e-5
        flag[0] = 1.0 if res["ok"] else 0.0
        del allf, ref
        torch.cuda.empty_cache()
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return res


def cpu_baseline_leg(args, wl, pipeline, feats, bank, out, precision):
    """Rank 0 at N = 1: a bounded sample of the reference's CPU path (oracle port) on the box's host cores, and -- since the
    oracle's answer for those query images is at hand -- a comparison of the GPU step's w / alpha / X rows with it."""
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_q, n_bank = cpu_sample_plan(wl, max(1, args.cpu_sample))
    mode = wl["mode"]
    if mode == "percategory":
        n_bank = min(n_bank, wl["sizes"][0] - 1)
        src = [f[: n_bank + 1] for f in feats]           # first category
    elif mode == "supervised":
        src = bank
    else:
        src = feats
    # bank embeddings for the CPU sample: produced once on the GPU, copied to the host (inputs of the timed CPU computation)
    q = pipeline.embed_images(src, 3, 1, wl["Dp"], wl["D"], "f32", want_z=True)
    Zbank = q.Z.reshape(q.n_img, q.P, q.D).cpu()
    del q
    n_q = min(n_q, feats[0].shape[0])
    feats_q = [f[:n_q].cpu() for f in feats]
    self_idx = None if mode == "supervised" else list(range(n_q))
    cpu_path_sample(wl, [f[:1] for f in feats_q], Zbank[: max(2, len(Zbank) // 8)], None if self_idx is None else [0])  # warm-up
    tcpu, reps, last = 0.0, 0, None
    while tcpu < args.cpu_seconds and reps < 64:           # bounded sample: about args.cpu_seconds of CPU work
        dt, w, outs = cpu_path_sample(wl, feats_q, Zbank, self_idx, want=True)
        tcpu += dt
        reps += 1
        last = (w, outs)
    cpu_baseline = {"value": n_q * reps / tcpu, "unit": "images/s", "cores": cores, "kind": "port",
                    "sample": "%d x %d query images: oracle embed + cdist/min against %d bank images + alpha (%d taus) + X (%.1f s)"
                              % (reps, n_q, len(Zbank) - (0 if self_idx is None else 1), len(wl["taus"]), tcpu)}
    parity = None
    if mode != "percategory" or True:
        w, outs = last
        gw = out["w"][:n_q].cpu()
        e_w = float(((gw - w).abs() / w.abs().clamp_min(1e-6)).max().item())
        e_a = max(float((out["alpha"][ti][:n_q].cpu().double() - outs[ti][0]).abs().max().item()) for ti in range(len(wl["taus"])))
        e_x = max(_rel(out["X"][ti][:n_q].cpu(), torch.from_numpy(outs[ti][1])) for ti in range(len(wl["taus"])))
        parity = {"check": "GPU w / alpha / X rows of %d query images against the CPU oracle (north_star tolerances)" % n_q,
                  "w_max_rel": e_w, "alpha_max_abs": e_a, "X_rel_l2": e_x, "ok": e_w <= 5e-4 and e_a <= 1e-3 and e_x <= 1e-3}
    return cpu_baseline, parity


def torch_gpu_reference_leg(wl, pipeline, feats, bank, out, n_q=4):
    """Reported next to the CPU baseline (rank 0, N = 1, untimed region): the reference's OWN distance loop -- one torch.cdist +
    min(dim=1) per (query image, bank image), models/patchcore/utils.py:222-237 -- in plain torch fp32 on this GPU, which is
    how upstream runs it when a GPU is present (examples/main.py:38 picks cuda:0).  A bounded sample of query images against
    the whole bank; the embed stage and alpha / X are NOT charged to it (they are < 1 % of the reference's time), so the
    images/s figure is an upper bound for the reference on this hardware.  Not an oracle, not a product path: a baseline."""
    import torch

    mode = wl["mode"]
    if mode == "percategory":
        n0 = wl["sizes"][0]
        src_q = src_b = [f[:n0] for f in feats]                # first category
    elif mode == "supervised":
        src_q, src_b = feats, bank
    else:
        src_q = src_b = feats
    qb = pipeline.embed_images(src_b, 3, 1, wl["Dp"], wl["D"], "f32", want_z=True)
    Zb = qb.Z.reshape(qb.n_img, qb.P, qb.D)
    if src_q is src_b:
        Zq = Zb
    else:
        qq = pipeline.embed_images([f[:n_q] for f in src_q], 3, 1, wl["Dp"], wl["D"], "f32", want_z=True)
        Zq = qq.Z.reshape(qq.n_img, qq.P, qq.D)
    n_q = min(n_q, Zq.shape[0])
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False             # the reference's default: fp32 cdist

    def loop(i):
        mins = []
        for j in range(Zb.shape[0]):
            if mode != "supervised" and j == i:
                continue
            mins.append(torch.min(torch.cdist(Zq[i], Zb[j]), dim=1)[0].unsqueeze(1))
        m = torch.cat(mins, dim=1)
        return torch.min(m, dim=1)[0] if mode == "supervised" else torch.mean(m, dim=1)

    try:
        loop(0)                                                # warm-up (cuBLAS handles, autotuning)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ws = [loop(i) for i in range(n_q)]
        e1.record()
        torch.cuda.synchronize()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    ms = e0.elapsed_time(e1)
    gw = out["w"][:n_q]
    dev_w = float(((gw - torch.stack(ws)).abs() / torch.stack(ws).abs().clamp_min(1e-6)).max().item())
    return {"value": n_q / (ms / 1e3), "unit": "images/s", "kind": "torch fp32 cdist loop of the reference on this GPU (distance stage only)",
            "sample": "%d query images x %d bank images, %.1f ms" % (n_q, Zb.shape[0] - (0 if mode == "supervised" else 1), ms),
            "w_max_rel_vs_ours": dev_w}


if __name__ == "__main__":
    main()
