"""Fused single-pass embed (config-2 shape, 100 images): time per launch in isolation of the lean kernel, Z-free and with
fp32 Z, against the per-layer launches of round 1 (variant 3) and the general fused kernel -- CUDA events, L2 flushed by
the 482 MB of maps themselves."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from anomaly_clustering_b200 import _lib, ops, pipeline, synth  # noqa: E402

lib = _lib.load()
n = int(sys.argv[1]) if len(sys.argv) > 1 else 100
layers = [(768, 28, 28, True), (768, 28, 28, True)]
feats, _ = synth.planted_features_device(range(n), layers, device="cuda")
P, D = 784, 4096
maps = sum(f[:, 1:].numel() * 4 for f in feats)


def reset():
    lib.ac_debug_set(2, 0)
    lib.ac_debug_set(9, 1)


def timed(want_z, reps=20):
    for _ in range(3):
        pipeline.embed_images(feats, 3, 1, 2048, D, "f16", want_z=want_z)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        pipeline.embed_images(feats, 3, 1, 2048, D, "f16", want_z=want_z)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def line(want_z, what, ms, nbytes):
    print("want_z=%s  %s: %.3f ms  = %.0f GB/s algorithmic = %.3f of 6553.3" % (want_z, what, ms, nbytes / ms / 1e6, nbytes / ms / 1e6 / 6553.3),
          flush=True)


for want_z in (False, True):
    nbytes = maps + n * P * D * 2 + n * P * 4 + (n * P * D * 4 if want_z else 0)
    reset()
    lib.ac_debug_set(2, 3)
    line(want_z, "per-layer launches (+ statistics pass + row norms) (%.1f MB)" % (nbytes / 1e6), timed(want_z), nbytes)
    lib.ac_debug_set(2, 0)
    lib.ac_debug_set(9, 0)
    line(want_z, "general fused kernel", timed(want_z), nbytes)
    reset()
    line(want_z, "lean fused kernel", timed(want_z), nbytes)
reset()
