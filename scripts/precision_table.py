"""Measured precision / speed of every ac_min_dist precision mode at full config-2 size against the exact
fp32 SIMT kernel (AC_PREC_F32): max-abs error of w, max-abs error of alpha per tau, time per launch.
    python scripts/precision_table.py [n_images] [channel_bias]
channel_bias 1.45 gives real-data patch norms (~46) -- the hard case for the |x|^2+|y|^2-2xy form."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from anomaly_clustering_b200 import ops, pipeline, synth  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 100
bias = float(sys.argv[2]) if len(sys.argv) > 2 else 0.0
layers = [(768, 28, 28, True), (768, 28, 28, True)]
feats, _ = synth.planted_features_device(range(n), layers, device="cuda", channel_bias=bias)
taus = [0.1, 0.25, 0.5, 1.0, 2.0]
q32 = pipeline.embed_images(feats, 3, 1, 2048, 4096, "f32")
w_ex = pipeline.min_distance_weights(q32, q32, "unsupervised", "f32")
a_ex, _ = ops.alpha(w_ex, taus)
X_ex = [ops.weighted_embed(a_ex[t].float(), q32.Z.reshape(n, -1, 4096)) for t in range(len(taus))]
print("config 2 shape, N=%d, channel_bias=%g: patch norm mean %.1f, w mean %.2f, within-image w spread (max-min) mean %.2f"
      % (n, bias, q32.Z.norm(dim=1).mean().item(), w_ex.mean().item(), (w_ex.max(1)[0] - w_ex.min(1)[0]).mean().item()))
print("| mode | ms / pass (GEMM + refine) | max abs dw | max rel dw | " + " | ".join("dalpha tau=%g" % t for t in taus) + " | X rel-L2 tau=0.1 | arg-max flips (tau=0) |")
print("|---|---:|---:|---:|" + "---:|" * (len(taus) + 2))
for prec in ("f16", "bf16", "f16r", "f16r (Z-free)", "f16x3", "bf16x3"):
    zfree = prec.endswith("(Z-free)")
    mode = prec.split()[0]
    q = pipeline.embed_images(feats, 3, 1, 2048, 4096, mode, want_z=not zfree)
    w = pipeline.min_distance_weights(q, q, "unsupervised", mode)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        pipeline.min_distance_weights(q, q, "unsupervised", mode)
    e1.record()
    torch.cuda.synchronize()
    a, _ = ops.alpha(w, taus)
    da = [(a[t] - a_ex[t]).abs().max().item() for t in range(len(taus))]
    X0 = ops.weighted_embed(a[0].float(), q32.Z.reshape(n, -1, 4096))
    flips = int((w.argmax(dim=1) != w_ex.argmax(dim=1)).sum())
    print("| %s | %.1f | %.2e | %.2e | " % (prec, e0.elapsed_time(e1) / 5, (w - w_ex).abs().max().item(),
                                           ((w - w_ex).abs() / w_ex).max().item()) + " | ".join("%.1e" % x for x in da)
          + " | %.1e | %d |" % (((X0 - X_ex[0]).norm() / X_ex[0].norm()).item(), flips), flush=True)
    del q
