"""GPU: bench.py --dump-outputs writes what the timed path returned, the same arrays whatever --steps is (the inputs
depend only on the arguments), and --steps sets the number of timed steps (the library launches scale with it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _bench(steps, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", str(steps), "--warmup", "3",
                        "--no-cpu-baseline", "--no-e2e", "--dump-outputs", out_dir], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_bench_dump_outputs_and_steps(tmp_path):
    import torch

    from anomaly_clustering_b200 import pipeline, synth

    a, b = _bench(2, str(tmp_path / "a")), _bench(4, str(tmp_path / "b"))
    assert a["steps"] == 2 and b["steps"] == 4 and b["gpu_launches"] == 2 * a["gpu_launches"] > 0
    names = sorted(os.listdir(str(tmp_path / "a")))
    assert names == ["Dmat.npy", "X.npy", "alpha.npy", "w.npy"] and sorted(os.listdir(str(tmp_path / "b"))) == names
    got = {n[:-4]: np.load(str(tmp_path / "a" / n)) for n in names}
    for n in names:
        assert np.array_equal(got[n[:-4]], np.load(str(tmp_path / "b" / n))), n
    # the same workload through the library in this process, with the bench's settings
    wl = bench.WORKLOADS["tiny"]
    feats, _ = synth.planted_features_device(range(wl["n_img"]), wl["layers"], seed=2023, device="cuda")
    r = pipeline.run_path(feats, 3, 1, wl["Dp"], wl["D"], "unsupervised", wl["taus"], precision=a["dtype"], keep_z=False)
    torch.cuda.synchronize()
    for name, want in (("alpha", r.alpha32), ("X", r.X), ("Dmat", r.Dmat), ("w", r.w)):
        assert got[name].dtype == np.float32 and got[name].shape == tuple(want.shape), name
        assert np.allclose(got[name], want.float().cpu().numpy(), rtol=1e-5, atol=1e-6), name
