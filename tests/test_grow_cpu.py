"""CPU: the ownership rule of a growing category (ac_min_dist_sym_grow) and the argument checks of its entry points."""
import ctypes
import os
import random
import shutil
import subprocess

import pytest

from anomaly_clustering_b200.distributed import pair_owned, pair_owned_grow

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(0, 1), (0, 2), (0, 7), (1, 1), (5, 1), (100, 1), (100, 10), (3, 4), (9, 2)] + \
         [(random.Random(s).randint(0, 40), random.Random(s + 99).randint(1, 12)) for s in range(20)]


@pytest.mark.parametrize("n_old,M", SHAPES)
def test_every_new_pair_has_one_owner_and_no_old_pair_has_any(n_old, M):
    n = n_old + M
    for i in range(n):
        for j in range(i + 1, n):
            owners = int(pair_owned_grow(n_old, i, j, n)) + int(pair_owned_grow(n_old, j, i, n))
            assert owners == (0 if j < n_old else 1), (n_old, M, i, j)
        assert not pair_owned_grow(n_old, i, i, n)


@pytest.mark.parametrize("n", [1, 2, 3, 8, 13, 100])
def test_growth_from_nothing_is_the_symmetric_rule(n):
    for i in range(n):
        for j in range(n):
            assert pair_owned_grow(0, i, j, n) == pair_owned(i, j, n)


def test_device_rule_matches_the_host_mirror(tmp_path):
    """csrc/common.cuh: pair_owned_grow, compiled for the host, agrees with the Python mirror on every pair."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    src = tmp_path / "rule.cu"
    src.write_text('#include <cstdio>\n#include "%s"\nint main() {\n'
                   '  for (int n_old = 0; n_old <= 12; ++n_old)\n    for (int n = n_old + 1; n <= n_old + 9; ++n)\n'
                   '      for (int i = 0; i < n; ++i)\n        for (int j = 0; j < n; ++j)\n'
                   '          std::printf("%%d", (int)ac::pair_owned_grow(n_old, i, j, n));\n  return 0;\n}\n'
                   % os.path.join(ROOT, "anomaly_clustering_b200", "csrc", "common.cuh"))
    exe = tmp_path / "rule"
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-o", str(exe), str(src)], check=True, capture_output=True)
    got = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    want = "".join(str(int(pair_owned_grow(n_old, i, j, n))) for n_old in range(13) for n in range(n_old + 1, n_old + 10)
                   for i in range(n) for j in range(n))
    assert got == want


def test_growth_entry_points_refuse_bad_arguments_without_a_gpu():
    from anomaly_clustering_b200 import _lib, build

    build.build()
    lib = _lib.load()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    args = dict(Mq=3 * 64, q_img0=4, nb_img=7, P=64, D=64, n_old=4)

    def grow(**kw):
        a = dict(args, **kw)
        return lib.ac_min_dist_sym_grow(p, None, p, a["Mq"], a["q_img0"], p, None, p, a["nb_img"], a["P"], a["D"], 0, 0,
                                        a["nb_img"], 1, p, p, None, None, kw.get("groups"), a["n_old"], p, 1 << 20, None)

    assert grow(groups=p) == _lib.AC_ERR_UNSUPPORTED           # per-category batches do not grow
    assert grow(q_img0=3) == _lib.AC_ERR_INVALID               # the query window is the new images
    assert grow(Mq=2 * 64) == _lib.AC_ERR_INVALID
    assert grow(n_old=7, q_img0=7, Mq=0) == _lib.AC_ERR_INVALID    # nothing new
    assert lib.ac_accumulate_weights_grow(None, p, 1, 4, 7, 64, p, p, None) == _lib.AC_ERR_INVALID
    assert lib.ac_accumulate_weights_grow(p, p, 1, 7, 7, 64, p, p, None) == _lib.AC_ERR_INVALID
    assert lib.ac_refine_min_dist_grow(None, p, None, _lib.AC_DT_F16, 4, 7, 64, 64, p, p, p, p, p, None) == _lib.AC_ERR_INVALID


def test_growing_category_refuses_the_exact_fp32_mode():
    from anomaly_clustering_b200 import pipeline

    with pytest.raises(ValueError, match="tensor-core precision"):
        pipeline.GrowingCategory(3, 1, 256, 512, [1.0], precision="f32")
    assert pipeline.GrowingCategory(3, 1, 256, 512, [0.0, 1.0]).precision == "f16r"      # resolved once, from the taus
    assert pipeline.GrowingCategory(3, 1, 256, 512, [1.0, 2.0]).precision == "f16"
