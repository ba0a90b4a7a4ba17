"""16-bit (bf16) against fp32 backbone feature maps, configs 1, 2 and 5 geometry: what native 16-bit reads in the embed
kernels buy, and that they change no result.

    python scripts/half_features_probe.py [--steps 10] [--reps 3]                       # legs (a) (b) (c)
    torchrun --nproc-per-node N scripts/half_features_probe.py --sharded-only            # leg (d), N > 1

(a) the embed call alone (operands + norms, the Z-free default), CUDA events over many launches, inputs larger than the
    126 MB L2, GB/s against the algorithmic bytes of each input width;
(b) the device-resident step (pipeline.run_path) on fp32 maps, bf16 maps, and bf16 maps upcast with .float() first (what a
    bf16 backbone user pays without native reads), with the embed / distance split of pipeline.PROFILE;
(c) end to end from pinned host maps, the host-to-device copies inside the timed region;
(d) config 2 end to end through run_path_sharded, each rank shipping its slice of the maps.
fp32 and bf16 runs alternate, same seeds.  Every line carries bit_identical: w, alpha, X and Dmat (or the embed outputs) of
the bf16 run against the fp32 run on the same maps upcast.  One JSON object per line on stdout and in --out."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from anomaly_clustering_b200 import distributed, ops, pipeline, synth  # noqa: E402

VITB = [(768, 28, 28, True), (768, 28, 28, True)]
CONFIGS = {   # name -> (layers, images of the step, images of leg (a), Dp, D, taus)
    "config1": ([(512, 28, 28, False), (1024, 14, 14, False)], 20, 200, 1024, 1024, [1.0]),
    "config2": (VITB, 100, 100, 2048, 4096, [1.0]),
    "config5": ([(384, 56, 56, True), (384, 56, 56, True)], 64, 64, 2048, 4096, [0.1, 0.5, 1.0, 2.0, 5.0, 10.0]),
}
L2_BYTES = 126 * 2 ** 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()}


def map_bytes(feats):
    return sum(f.numel() * f.element_size() for f in feats)


def emit(out, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


def embed_call(feats, Dp, D):
    """The Z-free default of pipeline.embed_images for f16: fp16 operands + their squared norms."""
    v = ops.feature_view(feats[0])
    h, w = ops.patch_grid(v.shape[2], v.shape[3], 3, 1)
    rows = v.shape[0] * h * w
    n2 = torch.empty(rows, dtype=torch.float32, device="cuda")
    _, hi, _, _ = ops.embed(feats, 3, 1, Dp, D, want_z=False, operand="f16", out_n2=n2)
    return hi, n2


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def path_outputs(r):
    return [t for t in (r.w, r.alpha64, r.X, r.Dmat) if t is not None]


def leg_a(out, name, layers, n, Dp, D, reps, launches):
    f32, _ = synth.planted_features_device(range(n), layers, device="cuda")
    b16 = [f.to(torch.bfloat16) for f in f32]
    up = [f.float() for f in b16]
    ident = same(embed_call(b16, Dp, D), embed_call(up, Dp, D))
    v = ops.feature_view(f32[0])
    rows = n * ops.patch_grid(v.shape[2], v.shape[3], 3, 1)[0] * ops.patch_grid(v.shape[2], v.shape[3], 3, 1)[1]
    out_bytes = rows * D * 2 + rows * 4
    t = {"fp32": [], "bf16": []}
    for _ in range(reps):                       # alternated
        t["fp32"].append(events_ms(lambda: embed_call(f32, Dp, D), launches))
        t["bf16"].append(events_ms(lambda: embed_call(b16, Dp, D), launches))
    rec = {"leg": "a_embed_kernel", "config": name, "images": n, "launches_per_rep": launches,
           "inputs_exceed_l2": {"fp32_map_MB": map_bytes(f32) / 1e6, "bf16_map_MB": map_bytes(b16) / 1e6, "l2_MB": L2_BYTES / 1e6,
                                "both_larger_than_l2": map_bytes(b16) > L2_BYTES},
           "bit_identical": ident}
    for k, feats in (("fp32", f32), ("bf16", b16)):
        ms = min(t[k])
        rec[k] = {"ms_per_call": t[k], "best_ms": ms, "algorithmic_bytes_MB": (map_bytes(feats) + out_bytes) / 1e6,
                  "GBps": (map_bytes(feats) + out_bytes) / ms / 1e6}
    rec["speedup_bf16"] = min(t["fp32"]) / min(t["bf16"])
    emit(out, rec)
    del f32, b16, up
    torch.cuda.empty_cache()


def step_split(fn, steps):
    pipeline.PROFILE = []
    ms = events_ms(fn, steps)
    marks, pipeline.PROFILE = pipeline.PROFILE, None

    def span(tag):
        b = [e for k, e in marks if k == tag + "_begin"]
        e_ = [e for k, e in marks if k == tag + "_end"]
        return sum(x.elapsed_time(y) for x, y in zip(b, e_)) / max(1, len(b))
    return ms, {"embed_ms": span("embed"), "mindist_ms": span("mindist"), "refine_ms": span("refine")}


def leg_b_c(out, name, layers, n, Dp, D, taus, steps, reps):
    f32, _ = synth.planted_features_device(range(n), layers, device="cuda")
    b16 = [f.to(torch.bfloat16) for f in f32]
    run = lambda fs: pipeline.run_path(fs, 3, 1, Dp, D, "unsupervised", taus, keep_z=False)  # noqa: E731
    ident = same(path_outputs(run(b16)), path_outputs(run([f.float() for f in b16])))
    variants = {"fp32": lambda: run(f32), "bf16": lambda: run(b16), "bf16_upcast": lambda: run([f.float() for f in b16])}
    res = {k: [] for k in variants}
    split = {}
    for _ in range(reps):
        for k, fn in variants.items():
            ms, sp = step_split(fn, steps)
            res[k].append(ms)
            split[k] = sp
    emit(out, {"leg": "b_device_step", "config": name, "images": n, "steps": steps, "ms_per_step": res,
               "best_ms": {k: min(v) for k, v in res.items()}, "stage_split_last_rep": split, "bit_identical": ident,
               "speedup_bf16_vs_bf16_upcast": min(res["bf16_upcast"]) / min(res["bf16"])})
    # (c) pinned host maps, copies in the timed region
    h32 = [f.cpu().pin_memory() for f in f32]
    h16 = [f.cpu().pin_memory() for f in b16]
    e2e = {"fp32": lambda: run([h.to("cuda", non_blocking=True) for h in h32]),
           "bf16": lambda: run([h.to("cuda", non_blocking=True) for h in h16]),
           "bf16_upcast": lambda: run([h.to("cuda", non_blocking=True).float() for h in h16])}
    ident_c = same(path_outputs(e2e["bf16"]()), path_outputs(e2e["bf16_upcast"]()))
    res = {k: [] for k in e2e}
    for _ in range(reps):
        for k, fn in e2e.items():
            res[k].append(events_ms(fn, steps))
    emit(out, {"leg": "c_end_to_end_pinned_host", "config": name, "images": n, "steps": steps, "host_map_MB": {
        "fp32": map_bytes(h32) / 1e6, "bf16": map_bytes(h16) / 1e6}, "ms_per_step": res, "best_ms": {k: min(v) for k, v in res.items()},
        "images_per_s": {k: n / min(v) * 1e3 for k, v in res.items()}, "bit_identical": ident_c})
    del f32, b16, h32, h16
    torch.cuda.empty_cache()


def leg_d(out, steps, reps):
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    layers, n, _, Dp, D, taus = CONFIGS["config2"]
    lo, hi = distributed.shard_bounds(n, world)[rank]
    f32, _ = synth.planted_features_device(range(lo, hi), layers, device="cuda")
    h32 = [f.cpu().pin_memory() for f in f32]
    h16 = [f.to(torch.bfloat16).cpu().pin_memory() for f in f32]
    run = lambda fs: distributed.run_path_sharded(fs, n, 3, 1, Dp, D, taus)  # noqa: E731
    variants = {"fp32": lambda: run([h.to("cuda", non_blocking=True) for h in h32]),
                "bf16": lambda: run([h.to("cuda", non_blocking=True) for h in h16]),
                "bf16_upcast": lambda: run([h.to("cuda", non_blocking=True).float() for h in h16])}
    ident = same(variants["bf16"](), variants["bf16_upcast"]())
    ok = torch.tensor([int(ident)], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    res = {k: [] for k in variants}
    for _ in range(reps):
        for k, fn in variants.items():
            dist.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            dist.barrier()
            res[k].append((time.perf_counter() - t0) / steps * 1e3)
    if rank == 0:
        emit(out, {"leg": "d_sharded_end_to_end", "config": "config2", "world": world, "images": n, "steps": steps,
                   "ms_per_step": res, "images_per_s": {k: n / min(v) * 1e3 for k, v in res.items()},
                   "bit_identical": bool(ok.item()), **card()})
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=20, help="leg (a): embed calls per timed repetition")
    ap.add_argument("--configs", nargs="+", default=sorted(CONFIGS))
    ap.add_argument("--sharded-only", action="store_true", help="leg (d) under torchrun")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    out = open(args.out, "a") if args.out else None
    if args.sharded_only:
        leg_d(out, args.steps, args.reps)
        return
    emit(out, {"leg": "card", **card()})
    for name in args.configs:
        layers, n, n_a, Dp, D, taus = CONFIGS[name]
        leg_a(out, name, layers, n_a, Dp, D, args.reps, args.launches)
        leg_b_c(out, name, layers, n, Dp, D, taus, args.steps, args.reps)


if __name__ == "__main__":
    main()
