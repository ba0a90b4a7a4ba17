"""Growing a config-2 category (ViT-B/8-shaped tokens, 28 x 28 patches, 2048 -> 4096, 100 images, tau 1) by 1 and by 10 images
with pipeline.GrowingCategory, against run_path from scratch on the same 101 and 110 images.

    python scripts/grow_probe.py [--reps 5] [--out profiles/grow_probe.log]

Each repetition builds a fresh category of 100 images (not timed), then times, alternately: add(+1 image), run_path on the
101 images, add(+10 images) to a second fresh category, run_path on the 110 images.  Times are CUDA events around work that
ends in a device synchronise; the first repetition is a warm-up and is not reported.  The card's name, power limit and max
SM clock are read in the same run, and each line reports the max deviation of w, alpha, X and Dmat between the add and the
from-scratch run."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from anomaly_clustering_b200 import pipeline, synth  # noqa: E402

LAYERS = [(768, 28, 28, True), (768, 28, 28, True)]
DP, D, TAUS = 2048, 4096, [1.0]


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b)


def deviation(g, r):
    rel = lambda x, y: (torch.linalg.norm((x.double() - y.double()).flatten()) / torch.linalg.norm(y.double().flatten())).item()
    return ("w max-rel %.2e  alpha64 max-abs %.2e  X rel-L2 %.2e  Dmat rel-L2 %.2e"
            % (((g.w - r.w).abs() / r.w.abs()).max().item(), (g.alpha64 - r.alpha64).abs().max().item(), rel(g.X, r.X),
               rel(g.Dmat, r.Dmat)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    if not torch.cuda.is_available():
        raise SystemExit("grow_probe needs a B200 (no CUDA device)")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    say("device: %s  (name, power limit, max SM clock: %s)" % (torch.cuda.get_device_name(), q))
    feats, _ = synth.planted_features(110, LAYERS, seed=11)
    feats = [f.cuda() for f in feats]
    say("config 2 geometry: P = 784, D = 4096, tau = 1 (precision %s), Z-free; %d repetitions after one warm-up"
        % (pipeline.resolve_precision("auto", TAUS), args.reps))

    def fresh():
        g = pipeline.GrowingCategory(3, 1, DP, D, TAUS, keep_z=False)
        g.add([f[:100] for f in feats])
        return g

    t = {k: [] for k in ("add1", "scratch101", "add10", "scratch110", "dist_add1", "dist_add10", "dist_scratch101", "dist_scratch110")}
    dev1 = dev10 = None
    for rep in range(args.reps + 1):
        stage = {}
        for n_new, key in ((1, "1"), (10, "10")):
            g = fresh()
            pipeline.PROFILE = []
            ga, ms_add = timed(lambda: g.add([f[100:100 + n_new] for f in feats]))
            marks = dict(pipeline.PROFILE)
            stage["dist_add" + key] = marks["mindist_begin"].elapsed_time(marks["mindist_end"])
            pipeline.PROFILE = []
            ra, ms_scratch = timed(lambda: pipeline.run_path([f[:100 + n_new] for f in feats], 3, 1, DP, D, "unsupervised", TAUS,
                                                             keep_z=False))
            marks = dict(pipeline.PROFILE)
            pipeline.PROFILE = None
            stage["dist_scratch1%02d" % n_new] = marks["mindist_begin"].elapsed_time(marks["mindist_end"])
            stage["add" + key], stage["scratch1%02d" % n_new] = ms_add, ms_scratch
            if key == "1":
                dev1 = deviation(ga, ra)
            else:
                dev10 = deviation(ga, ra)
            del g, ga, ra
        if rep == 0:
            continue
        for k, v in stage.items():
            t[k].append(v)
        say("rep %d: add +1 %.3f ms (distance %.3f) | scratch 101 %.3f ms (distance %.3f) | add +10 %.3f ms (distance %.3f) | "
            "scratch 110 %.3f ms (distance %.3f)" % (rep, stage["add1"], stage["dist_add1"], stage["scratch101"], stage["dist_scratch101"],
                                                       stage["add10"], stage["dist_add10"], stage["scratch110"], stage["dist_scratch110"]))
    med = {k: statistics.median(v) for k, v in t.items()}
    say("median: add +1 %.3f ms vs scratch 101 %.3f ms -> %.1fx;  add +10 %.3f ms vs scratch 110 %.3f ms -> %.1fx"
        % (med["add1"], med["scratch101"], med["scratch101"] / med["add1"], med["add10"], med["scratch110"], med["scratch110"] / med["add10"]))
    say("median distance pass: add +1 %.3f ms vs %.3f ms;  add +10 %.3f ms vs %.3f ms"
        % (med["dist_add1"], med["dist_scratch101"], med["dist_add10"], med["dist_scratch110"]))
    say("deviation +1 vs scratch 101: " + dev1)
    say("deviation +10 vs scratch 110: " + dev10)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
