"""torchrun --nproc-per-node N scripts/r02_multi.py [out_dir]: every multi-GPU measurement of round 2 in ONE process group
(one NCCL init instead of one per bench invocation; multi-GPU box time is charged N-fold):
  1. the sharded path against one GPU (default transport, NCCL collectives, all-pairs form, refined precision), uneven shards;
  2. bench.py lines (same code, same JSON) for config 2 (fp16 and f16r), configs 3, 4 (joint), 4pc, 5;
  3. a kineto timeline of three config-2 steps on rank 0 for the symmetric-memory transport and the NCCL collectives.
The NCCL collectives are forced in-process through SymmetricBank.disabled_reason."""
import io
import json
import os
import sys
import time
import contextlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402
from anomaly_clustering_b200 import distributed, pipeline, synth  # noqa: E402
from anomaly_clustering_b200.symm_transport import SymmetricBank  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "r02_multi")
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
os.environ["AC_BENCH_KEEP_PG"] = "1"
if rank == 0:
    os.makedirs(OUT, exist_ok=True)
dist.barrier()
T0 = time.time()


@contextlib.contextmanager
def nccl_collectives(on):
    """With on=True the sharded path inside the block uses the NCCL collectives instead of symmetric memory."""
    saved = SymmetricBank.disabled_reason
    if on:
        SymmetricBank.disabled_reason = "NCCL collectives forced by scripts/r02_multi.py"
    try:
        yield
    finally:
        SymmetricBank.disabled_reason = saved


def log(msg):
    if rank == 0:
        print("[%6.1fs] %s" % (time.time() - T0, msg), flush=True)
        with open(os.path.join(OUT, "log_n%d.txt" % world), "a") as f:
            f.write("[%6.1fs] %s\n" % (time.time() - T0, msg))


# ---------------------------------------------------------------- 1. correctness against one GPU
ok_all = True
for n_img, layers, Dp, D in ((13, [(96, 12, 12, True), (96, 12, 12, True)], 256, 512),
                             (29, [(768, 28, 28, True), (768, 28, 28, True)], 2048, 4096)):
    if n_img < world:
        continue
    bounds = distributed.shard_bounds(n_img, world)
    lo, hi = bounds[rank]
    feats, _ = synth.planted_features_device(range(lo, hi), layers, device="cuda")
    allf = synth.planted_features_device(range(n_img), layers, device="cuda")[0] if rank == 0 else None
    for name, prec, taus in (("default (symm)", "f16", [1.0, 2.0]), ("nccl", "f16", [1.0, 2.0]),
                             ("all-pairs", "f16", [1.0]), ("refined f16r", "auto", [0.1, 1.0])):
        try:
            with nccl_collectives(name == "nccl"):
                a64, X, Dm, w = distributed.run_path_sharded(feats, n_img, 3, 1, Dp, D, taus, precision=prec, symmetric=name != "all-pairs")
            torch.cuda.synchronize()
            if rank == 0:
                ref = pipeline.run_path(allf, 3, 1, Dp, D, "unsupervised", taus, precision=prec)
                e_w = ((w - ref.w[lo:hi]).abs() / ref.w[lo:hi]).max().item()
                e_a = (a64 - ref.alpha64[:, lo:hi]).abs().max().item()
                e_x = ((X - ref.X).norm() / ref.X.norm()).item()
                e_d = ((Dm - ref.Dmat).norm() / ref.Dmat.norm()).item()
                good = e_w < 2e-4 and e_a < 1e-3 and e_x < 1e-4 and e_d < 1e-4
                ok_all &= good
                log("check N=%d on %d ranks %s  %-12s: w rel %.1e  alpha abs %.1e  X relL2 %.1e  Dmat relL2 %.1e  bit-identical X %s  %s"
                    % (n_img, world, [b - a for a, b in bounds], name, e_w, e_a, e_x, e_d, bool(torch.equal(X, ref.X)), "OK" if good else "MISMATCH"))
        except Exception as e:  # noqa: BLE001
            ok_all = False
            log("check N=%d %s FAILED: %r" % (n_img, name, e))
        dist.barrier()
    del feats, allf
torch.cuda.empty_cache()


# ---------------------------------------------------------------- 2. bench lines
def run_bench(tag, argv):
    buf = io.StringIO()
    t0 = time.time()
    try:
        with contextlib.redirect_stdout(buf):
            bench.main(argv + ["--gpus", str(world)])
    except BaseException as e:  # noqa: BLE001
        log("bench %s FAILED: %r" % (tag, e))
    if rank == 0:
        line = [ln for ln in buf.getvalue().splitlines() if ln.startswith("{")]
        with open(os.path.join(OUT, "bench_%s_n%d.json" % (tag.replace(" ", "_"), world)), "w") as f:
            f.write("\n".join(line) + "\n")
        try:
            d = json.loads(line[-1])
            log("bench %-16s %.1f s: images/s %.0f  ms/step %.3f  parity_ok %s  e2e %s  stages %s  comm %s  roofline %.3f" % (
                tag, time.time() - t0, d["value"], d["ms_per_step"], d.get("parity_ok"), (d.get("e2e") or {}).get("value"),
                {k: round(v, 3) for k, v in d["stages"].items() if isinstance(v, float)},
                {k: round(v, 3) for k, v in d["stages"]["comm_ms_per_step_rank0"].items()}, d["roofline"]["frac"]))
            log("      parity %s" % (d.get("parity"),))
        except Exception as e:  # noqa: BLE001
            log("bench %s: no line (%r)" % (tag, e))
    torch.cuda.empty_cache()
    dist.barrier()


which = os.environ.get("AC_MULTI_WHICH", "c2,c2r,c3,c4,c4pc,c5,trace").split(",")
if "c2" in which:
    run_bench("config2 default", ["--workload", "config2", "--steps", "20", "--warmup", "5", "--no-cpu-baseline"])
if "c2r" in which:
    run_bench("config2 f16r", ["--workload", "config2", "--steps", "10", "--warmup", "3", "--no-e2e", "--precision", "f16r"])
if "c3" in which:
    run_bench("config3", ["--workload", "config3", "--steps", "5", "--warmup", "3", "--no-e2e"])
if "c4pc" in which:
    run_bench("config4pc", ["--workload", "config4pc", "--steps", "3", "--warmup", "3", "--no-e2e"])
if "c5" in which:
    run_bench("config5", ["--workload", "config5", "--steps", "3", "--warmup", "3", "--no-e2e"])
if "c4" in which:
    run_bench("config4 joint", ["--workload", "config4", "--steps", "3", "--warmup", "3", "--no-e2e"])

# ---------------------------------------------------------------- 3. timelines
if "trace" in which:
    from torch.profiler import ProfilerActivity, profile

    layers = [(768, 28, 28, True), (768, 28, 28, True)]
    lo, hi = distributed.shard_bounds(100, world)[rank]
    feats, _ = synth.planted_features_device(range(lo, hi), layers, device="cuda")
    for name in ("symm", "nccl"):
        with nccl_collectives(name == "nccl"):
            for _ in range(5):
                distributed.run_path_sharded(feats, 100, 3, 1, 2048, 4096, [1.0], precision="f16", keep_z=False)
            torch.cuda.synchronize()
            dist.barrier()
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    distributed.run_path_sharded(feats, 100, 3, 1, 2048, 4096, [1.0], precision="f16", keep_z=False)
                torch.cuda.synchronize()
            dist.barrier()
        if rank in (0, world - 1):
            path = os.path.join(OUT, "trace_%s_n%d_rank%d.json" % (name, world, rank))
            prof.export_chrome_trace(path)
            # compact digest: GPU activities in time order
            ev = json.load(open(path))["traceEvents"]
            gpu = sorted([e for e in ev if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")], key=lambda e: e["ts"])
            t0 = gpu[0]["ts"] if gpu else 0
            with open(os.path.join(OUT, "timeline_%s_n%d_rank%d.txt" % (name, world, rank)), "w") as f:
                for e in gpu:
                    f.write("%10.1f us  +%8.1f us  stream %s  %s\n" % (e["ts"] - t0, e["dur"], e.get("args", {}).get("stream"), e["name"][:110]))
            os.remove(path)
log("all checks %s" % ("OK" if ok_all else "HAD MISMATCHES"))
dist.barrier()
dist.destroy_process_group()
