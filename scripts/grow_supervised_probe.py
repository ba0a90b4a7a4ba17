"""Growing a config-3 supervised category (ViT-B-shaped tokens, 28 x 28 patches, 2048 -> 4096, tau 1, f16, Z-free; 100 queries
against a 200-image normal bank) with pipeline.GrowingSupervisedCategory, against run_path from scratch on the same images.

    python scripts/grow_supervised_probe.py [--reps 5] [--out profiles/grow_supervised_probe.log]

Each repetition times, on a freshly built category (200 normal + 100 query images, not timed), each of add(+1 query),
add(+10 queries), add_normal(+1 normal) and add_normal(+10 normals), alternated with run_path from scratch on the same images.
Times are CUDA events around work that ends in a device synchronise, and the distance pass (min_dist launch) is reported
separately from the stage marks; the first repetition is a warm-up and is not reported.  The card's name, power limit and
max SM clock are read in the same run, and each line says whether every field of the result is bit-identical to the
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
NQ, NB = 100, 200
FIELDS = ("w", "alpha64", "alpha32", "X", "Dmat")


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b)


def profiled(fn):
    """(result, ms, distance-pass ms) of one call, with the pipeline's stage marks."""
    pipeline.PROFILE = []
    out, ms = timed(fn)
    marks = dict(pipeline.PROFILE)
    pipeline.PROFILE = None
    return out, ms, marks["mindist_begin"].elapsed_time(marks["mindist_end"])


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
        raise SystemExit("grow_supervised_probe needs a B200 (no CUDA device)")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    say("device: %s  (name, power limit, max SM clock: %s)" % (torch.cuda.get_device_name(), q))
    fq, _ = synth.planted_features_device(range(NQ + 10), LAYERS, seed=31)
    fb, _ = synth.planted_features_device(range(10_000, 10_000 + NB + 10), LAYERS, n_classes=1, seed=32)
    say("config 3 geometry: P = 784, D = 4096, tau = 1 (precision %s), Z-free; %d normal + %d query images built untimed; "
        "%d repetitions after one warm-up" % (pipeline.resolve_precision("auto", TAUS), NB, NQ, args.reps))

    def fresh():
        g = pipeline.GrowingSupervisedCategory(3, 1, DP, D, TAUS, keep_z=False)
        g.add_normal([f[:NB] for f in fb])
        g.add([f[:NQ] for f in fq])
        return g

    def scratch(nq, nb):
        return profiled(lambda: pipeline.run_path([f[:nq] for f in fq], 3, 1, DP, D, "supervised", TAUS,
                                                  bank_features=[f[:nb] for f in fb], keep_z=False))

    cases = (("add +1", lambda g: g.add([f[NQ:NQ + 1] for f in fq]), NQ + 1, NB),
             ("add +10", lambda g: g.add([f[NQ:NQ + 10] for f in fq]), NQ + 10, NB),
             ("add_normal +1", lambda g: g.add_normal([f[NB:NB + 1] for f in fb]), NQ, NB + 1),
             ("add_normal +10", lambda g: g.add_normal([f[NB:NB + 10] for f in fb]), NQ, NB + 10))
    t = {name: {"grow": [], "grow_dist": [], "scratch": [], "scratch_dist": []} for name, _, _, _ in cases}
    same = {name: True for name, _, _, _ in cases}
    for rep in range(args.reps + 1):
        parts = []
        for name, call, nq, nb in cases:
            g = fresh()
            res, ms, dist = profiled(lambda: call(g))
            ref, ms_s, dist_s = scratch(nq, nb)
            ok = all(torch.equal(getattr(res, k), getattr(ref, k)) for k in FIELDS)
            del g, res, ref
            if rep == 0:
                continue
            same[name] &= ok
            for k, v in (("grow", ms), ("grow_dist", dist), ("scratch", ms_s), ("scratch_dist", dist_s)):
                t[name][k].append(v)
            parts.append("%s %.3f ms (distance %.3f) vs scratch %.3f ms (distance %.3f) bit_identical=%s"
                         % (name, ms, dist, ms_s, dist_s, str(ok).lower()))
        if rep:
            say("rep %d: " % rep + " | ".join(parts))
    for name, _, nq, nb in cases:
        m = {k: statistics.median(v) for k, v in t[name].items()}
        say("median %s (%d queries x %d normals): %.3f ms (distance %.3f) vs run_path from scratch %.3f ms (distance %.3f) -> "
            "%.1fx  bit_identical=%s" % (name, nq, nb, m["grow"], m["grow_dist"], m["scratch"], m["scratch_dist"],
                                         m["scratch"] / m["grow"], str(same[name]).lower()))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
