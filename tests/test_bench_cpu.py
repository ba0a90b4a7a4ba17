"""CPU: bench.py's host-side pieces that can be checked without a GPU -- the nvidia-smi clock sampler (parsing,
cutting the samples to the timed window, the short-run fallback) against a fake nvidia-smi, and the reference arm's
JSON contract."""
import json
import os
import stat
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def _line(ts, sm, pw, cap):
    return "%s, 0, %d, 1965, %.2f, 0x0000000000000004, Not Active, Not Active, Not Active, %s" % (
        time.strftime("%Y/%m/%d %H:%M:%S", time.localtime(ts)) + ".%03d" % int((ts % 1) * 1000), sm, pw, "Active" if cap else "Not Active")


def test_clock_samples_are_cut_to_the_timed_window():
    t0 = 1_800_000_000.0
    text = "\n".join([_line(t0 + 0.05 * i, 1965, 180.0, False) for i in range(4)]            # idle before the warm-up
                     + [_line(t0 + 0.2 + 0.05 * i, 1100, 990.0, True) for i in range(12)]    # warm-up + timed, power-capped
                     + [_line(t0 + 0.8 + 0.05 * i, 1965, 200.0, False) for i in range(3)])   # after
    rows = bench.ClockSampler.parse(text)
    assert len(rows) == 19 and rows[5][4] == {"sw_power_cap"}
    rec = bench.ClockSampler.summarise(rows, t0 + 0.4, t0 + 0.75)
    assert rec["window"] == "timed region" and rec["samples"] == 8 and rec["sm_mhz"] == 1100 and rec["reasons"] == ["sw_power_cap"]
    assert rec["sm_max_mhz"] == 1965 and rec["power_w_max"] == 990.0
    # timed region shorter than two sampling periods: under-load samples of the whole sampler run, and the record says so
    rec = bench.ClockSampler.summarise(rows, t0 + 0.41, t0 + 0.44)
    assert rec["window"].startswith("warm-up + timed") and rec["samples"] == 12 and rec["reasons"] == ["sw_power_cap"]
    assert bench.ClockSampler.summarise([], 0, 1)["reasons"] == ["no samples"]
    assert bench.ClockSampler.parse("garbage\n1,2,3\n") == []


def test_clock_sampler_against_a_fake_nvidia_smi(tmp_path, monkeypatch):
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nwhile true; do echo \"$(date '+%Y/%m/%d %H:%M:%S.%3N'), 0, 1245, 1965, 987.50, 0x4, Not Active, Not Active, "
                    "Not Active, Active\"; sleep 0.05; done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ["PATH"])
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.3)
    t_begin = time.time()
    time.sleep(0.5)
    t_end = time.time()
    rec = s.stop(t_begin, t_end)
    assert rec["window"] == "timed region" and 5 <= rec["samples"] <= 12, rec
    assert rec["sm_mhz"] == 1245 and rec["sm_max_mhz"] == 1965 and rec["reasons"] == ["sw_power_cap"]


def test_clock_sampler_without_nvidia_smi(tmp_path, monkeypatch):
    monkeypatch.setenv("PATH", str(tmp_path))
    s = bench.ClockSampler(0)
    s.start()
    assert s.stop(0.0, 1.0)["reasons"] == ["nvidia-smi unavailable"]


def test_dump_outputs_dtypes_names_and_size_cap(tmp_path):
    import numpy as np
    import torch

    gen = torch.Generator().manual_seed(0)
    out = {"alpha": torch.rand(2, 3, 50, dtype=torch.float64, generator=gen), "X": torch.rand(2, 3, 64, generator=gen).half(),
           "Dmat": [torch.rand(1, 3, 3, generator=gen), torch.rand(1, 4, 4, generator=gen)], "w": torch.rand(3, 50, generator=gen)}
    got = bench.dump_outputs(out, str(tmp_path / "full"))
    assert sorted(got) == ["Dmat_0.npy", "Dmat_1.npy", "X.npy", "alpha.npy", "w.npy"] and not any(s for _, s in got.values())
    a, X, d1 = (np.load(str(tmp_path / "full" / n)) for n in ("alpha.npy", "X.npy", "Dmat_1.npy"))
    assert a.dtype == np.float64 and np.array_equal(a, out["alpha"].numpy())
    assert X.dtype == np.float32 and np.array_equal(X, out["X"].float().numpy())
    assert d1.dtype == np.float32 and np.array_equal(d1, out["Dmat"][1].numpy())
    # over the cap: the small arrays stay whole, the large ones become fixed samples, the files stay under the cap
    big = {"X": torch.rand(400, 1000, generator=gen), "Dmat": torch.rand(300, 300, dtype=torch.float64, generator=gen),
           "w": torch.rand(10, 10, generator=gen)}
    limit = 1 << 20
    for run in ("s1", "s2"):
        got = bench.dump_outputs(big, str(tmp_path / run), limit_bytes=limit)
        assert got == {"w.npy": ((10, 10), False), "X.npy": ((400, 1000), True), "Dmat.npy": ((300, 300), True)}
        assert sum(os.path.getsize(str(tmp_path / run / n)) for n in got) <= limit
    for n in got:
        assert np.array_equal(np.load(str(tmp_path / "s1" / n)), np.load(str(tmp_path / "s2" / n)))
    # the documented rule: smallest first, each array gets what is left over the arrays still to write, and a sampled
    # array holds the elements at np.unique(default_rng(0).integers(0, numel, size=share // itemsize))
    left = limit - 3 * bench.NPY_HEADER_BYTES - 10 * 10 * 4
    for name, itemsize, n_after in (("Dmat", 8, 2), ("X", 4, 1)):
        src = big[name].numpy().ravel()
        idx = np.unique(np.random.default_rng(0).integers(0, src.size, size=(left // n_after) // itemsize))
        xs = np.load(str(tmp_path / "s1" / (name + ".npy")))
        assert xs.dtype == src.dtype and np.array_equal(xs, src[idx]), name
        left -= xs.nbytes


def test_bench_refuses_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120,
                       cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


@pytest.mark.timeout(900)
def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=800, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config",
                "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    # under torchrun the other ranks exit without work or output
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
