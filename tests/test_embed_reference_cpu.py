"""CPU: the float64 stage-1 reference (oracle/restated.embed with dtype=torch.float64) that tests/test_gpu_embed_edges.py
compares the embedding kernels against, and the argument checks of the embed entry points that run before any CUDA call.

The float64 reference is pinned against the outputs of the unmodified reference (tests/golden/embed_*.npz) and against
the float32 restatement, so a GPU failure against it points at the kernel, not at the reference."""
import ctypes
import os

import numpy as np
import pytest
import torch

from anomaly_clustering_b200 import _lib, ops, pipeline
from oracle import restated

EMBED_CASES = ["embed_vit_small", "embed_wrn_small", "embed_ragged", "embed_k5s2", "embed_single"]


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False)


@pytest.mark.parametrize("name", EMBED_CASES)
def test_float64_reference_matches_reference_outputs(golden_dir, name):
    """The stored Z is the reference's own fp32 result: its rounding error (fp32 LayerNorm, unfold, two pools) is far below
    1e-5 at these unit-scale maps."""
    g = _golden(golden_dir, name)
    feats = [torch.from_numpy(g["feat%d" % i]) for i in range(int(g["L"]))]
    z = restated.embed(feats, int(g["patchsize"]), int(g["stride"]), int(g["Dp"]), int(g["D"]), dtype=torch.float64)
    assert z.dtype == torch.float64 and z.shape == g["Z"].shape
    assert np.abs(z.numpy() - g["Z"].astype(np.float64)).max() <= 1e-5


def test_default_dtype_is_bit_identical_to_float32(golden_dir):
    g = _golden(golden_dir, "embed_ragged")
    feats = [torch.from_numpy(g["feat%d" % i]) for i in range(int(g["L"]))]
    a = restated.embed(feats, 3, 1, int(g["Dp"]), int(g["D"]))
    b = restated.embed(feats, 3, 1, int(g["Dp"]), int(g["D"]), dtype=torch.float32)
    assert a.dtype == torch.float32 and torch.equal(a, b)


SEEDED = [  # (layers [(C, H, W, tokens)], B, patchsize, stride, Dp, D, layernorm)
    ([(24, 9, 9, True), (24, 9, 9, True)], 2, 3, 1, 64, 128, True),
    ([(16, 12, 10, False), (32, 6, 5, False)], 3, 3, 1, 40, 30, True),     # resampled layer, straddling Aggregator windows
    ([(5, 7, 7, False)], 2, 5, 2, 100, 50, False),                          # Dp > C*k*k, no LayerNorm
    ([(3, 1, 2, False)], 2, 7, 3, 20, 20, True),                            # map smaller than the patch
]


@pytest.mark.parametrize("case", range(len(SEEDED)))
def test_float64_reference_matches_float32_restatement(case):
    layers, B, ps, st, Dp, D, ln = SEEDED[case]
    g = torch.Generator().manual_seed(100 + case)
    feats = []
    for C, H, W, tok in layers:
        x = torch.randn(B, C, H, W, generator=g) * 1.5 + 0.5
        feats.append(torch.cat([torch.zeros(B, 1, C), x.flatten(2).transpose(1, 2)], 1) if tok else x)
    z32 = restated.embed(feats, ps, st, Dp, D, layernorm=ln)
    z64 = restated.embed(feats, ps, st, Dp, D, layernorm=ln, dtype=torch.float64)
    assert z64.dtype == torch.float64 and z64.shape == z32.shape
    # fp32 LayerNorm + pools of values of a few units: a few fp32 ulps
    assert (z32.double() - z64).abs().max().item() <= 1e-5


def test_float64_weighted_embedding_matches_explicit_loop():
    g = torch.Generator().manual_seed(7)
    Z = torch.randn(3, 5, 4, generator=g, dtype=torch.float64)
    a = torch.randn(3, 5, generator=g, dtype=torch.float64)
    X = restated.weighted_embedding64(a, Z)
    ref = torch.zeros(3, 4, dtype=torch.float64)
    for i in range(3):
        for p in range(5):
            for d in range(4):
                ref[i, d] += a[i, p] * Z[i, p, d]
    assert X.dtype == torch.float64
    assert (X - ref).abs().max().item() <= 1e-14


# --------------------------------------------------------------------------------------- argument checks before any CUDA call
M = "meta"   # the maps live on the meta device: shapes only, nothing is allocated or launched


@pytest.mark.parametrize("which,bad", [
    ("out_z", lambda r, d: torch.empty(r, d + 1, device=M)),                          # shape
    ("out_z", lambda r, d: torch.empty(r - 1, d, device=M)),
    ("out_z", lambda r, d: torch.empty(r * d, device=M)),
    ("out_z", lambda r, d: torch.empty(r, d, dtype=torch.float64, device=M)),        # dtype
    ("out_z", lambda r, d: torch.empty(d, r, device=M).T),                            # not contiguous
    ("out_z", lambda r, d: torch.empty(r, d)),                                        # device (the maps are elsewhere)
    ("out_hi", lambda r, d: torch.empty(r, d, dtype=torch.bfloat16, device=M)),      # operand dtype
    ("out_hi", lambda r, d: torch.empty(r, 2 * d, dtype=torch.float16, device=M)[:, ::2]),
    ("out_hi", lambda r, d: torch.empty(r, d, dtype=torch.float16)),
    ("out_lo", lambda r, d: torch.empty(r, d // 2, dtype=torch.float16, device=M)),
    ("out_lo", lambda r, d: torch.empty(r, d, dtype=torch.float32, device=M)),
])
def test_embed_refuses_bad_output_buffers(which, bad):
    """A buffer the kernels would write as a dense [B*P, D] array but that is not one is refused (it was written out of
    bounds or with the wrong element size)."""
    feats = [torch.empty(2, 1 + 16, 8, device=M)]      # ViT tokens: 2 images of a 4 x 4 grid, P = 16
    rows, D = 2 * 16, 32
    with pytest.raises(ValueError, match=which):
        ops.embed(feats, 3, 1, 16, D, operand="f16", want_lo=True, **{which: bad(rows, D)})


def test_embed_accepts_offset_output_buffers_in_the_checks():
    """A contiguous buffer with an odd storage offset passes the checks (the kernels take scalar stores for it)."""
    rows, D = 32, 32
    z = torch.empty(rows * D + 1, device="meta")[1:].view(rows, D)
    hi = torch.empty(rows * D + 1, dtype=torch.float16, device="meta")[1:].view(rows, D)
    ops._out_ok(z, "out_z", (rows, D), torch.float32, torch.device("meta"))
    ops._out_ok(hi, "out_hi", (rows, D), torch.float16, torch.device("meta"))


@pytest.mark.parametrize("grid,supported", [(224, True), (225, False)])
def test_z_free_supported_follows_the_alpha_tile_bound(grid, supported):
    """ac_weighted_embed_from_features stages the (h0 + 2) x (w0 + 2) fp32 alpha tile in at most 200 KB of shared memory."""
    feats = [torch.empty(1, 8, grid, grid, device="meta")]
    assert pipeline.z_free_supported(feats, 3, 1, 8, 8, "f16") is supported


@pytest.fixture(scope="module")
def lib():
    from anomaly_clustering_b200 import build

    build.build()
    return _lib.load()


@pytest.mark.parametrize("dt", [_lib.AC_DT_F32, _lib.AC_DT_F16, _lib.AC_DT_BF16])
def test_misaligned_workspace_is_invalid(lib, dt):
    """The statistics partials in the workspace are read as doubles and its scratch as 16-byte vectors."""
    arr = (_lib.AcLayer * 1)()
    arr[0] = _lib.AcLayer(4096, 64, 8, 8, 64 * 64, 1, 8 * 64, 64)   # a plausible (never dereferenced) address
    buf = ctypes.c_void_p(4096)
    for off in (1, 4, 8):
        ws = ctypes.c_void_p(4096 + off)
        assert lib.ac_embed_dt(arr, 1, dt, 2, 3, 1, 64, 64, 1, 1e-5, buf, buf, None, _lib.AC_DT_F16, None, ws, 1 << 24,
                               None) == _lib.AC_ERR_INVALID
        assert lib.ac_weighted_embed_from_features_dt(arr, 1, dt, 2, 3, 1, 64, 64, 1, 1e-5, buf, buf, ws, 1 << 24,
                                                      None) == _lib.AC_ERR_INVALID
