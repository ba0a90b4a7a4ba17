"""CPU: the oracle restatement against the committed reference outputs (tests/golden, generated
by oracle/make_golden.py from the UNMODIFIED reference) and against the reference's shipped results."""
import os

import numpy as np
import pytest
import torch

from oracle import cluster as ocluster
from oracle import make_golden, ref_import, restated

EMBED_CASES = ["embed_vit_small", "embed_wrn_small", "embed_ragged", "embed_k5s2", "embed_single"]


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False)


@pytest.mark.parametrize("name", EMBED_CASES)
def test_embed_matches_reference(golden_dir, name):
    g = load(golden_dir, name)
    feats = [torch.from_numpy(g["feat%d" % i]) for i in range(int(g["L"]))]
    z = restated.embed(feats, int(g["patchsize"]), int(g["stride"]), int(g["Dp"]), int(g["D"]))
    assert z.shape == g["Z"].shape
    assert np.abs(z.numpy() - g["Z"]).max() <= 2e-6


def test_alpha_w_X_match_reference(golden_dir):
    g = load(golden_dir, "alpha_small")
    Z, Zb = torch.from_numpy(g["Z"]), torch.from_numpy(g["Z_train"])
    wu = restated.weight_distance_unsupervised(Z)
    ws = restated.weight_distance_supervised(Z, Zb)
    assert np.abs(wu.numpy() - g["w_unsup"]).max() <= 1e-5
    assert np.abs(ws.numpy() - g["w_sup"]).max() <= 1e-5
    for t in g["taus"]:
        au = restated.alpha_from_weights(wu, float(t))
        asup = restated.alpha_from_weights(ws, float(t))
        assert np.abs(au.numpy() - g["alpha_unsup_%g" % t]).max() <= 1e-5
        assert np.abs(asup.numpy() - g["alpha_sup_%g" % t]).max() <= 1e-5
        assert np.abs(restated.weighted_embedding(au, Z) - g["X_unsup_%g" % t]).max() <= 1e-4
        # stabilised softmax == reference softmax wherever the reference is finite
        assert np.abs(restated.alpha_from_weights(wu, float(t), stable=True).numpy() - au.numpy()).max() <= 1e-12


def test_tau_zero_is_onehot_with_ties():
    w = torch.tensor([[1.0, 3.0, 3.0, 2.0]])
    a = restated.alpha_from_weights(w, 0.0)
    assert torch.allclose(a, torch.tensor([[0.0, 0.5, 0.5, 0.0]], dtype=torch.float64))


def test_reference_softmax_overflows_where_stable_does_not():
    w = torch.tensor([[800.0, 799.0]])
    assert torch.isnan(restated.alpha_from_weights(w, 1.0)).any()  # reference behaviour (utils.py:253)
    a = restated.alpha_from_weights(w, 1.0, stable=True)
    assert torch.isfinite(a).all() and abs(a.sum().item() - 1) < 1e-12


def test_patchify_pool_match_reference(golden_dir):
    g = load(golden_dir, "patchify_small")
    x = torch.from_numpy(g["x"])
    for k, s in [(3, 1), (5, 2), (1, 1)]:
        u, grid = restated.patchify(x, k, s)
        assert grid == list(g["grid_k%d_s%d" % (k, s)])
        assert np.array_equal(u.contiguous().numpy(), g["patch_k%d_s%d" % (k, s)])
    pre = restated.preprocessing_forward([torch.from_numpy(g["pre_in0"]), torch.from_numpy(g["pre_in1"])], 20)
    assert np.array_equal(pre.numpy(), g["pre_out"])
    assert np.array_equal(restated.aggregator_forward(pre, 13).numpy(), g["agg_out"])


def test_shipped_results_reproduce_published_metrics(golden_dir):
    """X -> Ward -> best_map -> NMI/ARI/F1 equals the reference's own tau_result.csv (TAU=2)."""
    g = load(golden_dir, "shipped_cluster_golden")
    for key in g["cases"]:
        key = str(key)
        nmi, ari, f1, _, _ = ocluster.metrics_from_X(g[key + "_Xlow"], [str(a) for a in g[key + "_anomaly"]])
        assert np.allclose([nmi, ari, f1], g[key + "_csv"], atol=1e-9), key
        assert np.allclose(g[key + "_alpha_rowsum"], 1.0, atol=1e-4)
        assert int(g[key + "_alpha_shape"][2]) == 784


def test_pairwise_matches_scipy():
    rng = np.random.default_rng(0)
    X = rng.normal(size=(7, 33)).astype(np.float32)
    D = restated.pairwise_euclidean(X)
    ref = np.sqrt(((X[:, None, :].astype(np.float64) - X[None, :, :]) ** 2).sum(-1))
    assert np.allclose(D, ref, atol=1e-12)


def _check_embed(g, key, seed, z, feats, tol):
    assert np.allclose(g[key + "_input_sums"], [f.double().sum().item() for f in feats], rtol=1e-12, atol=1e-9), \
        (key, "the seeded inputs changed: the fixture no longer describes these inputs")
    assert tuple(z.shape) == tuple(g[key + "_shape"]), key
    n, zmax = z.numel(), float(z.abs().max())
    z64 = z.double()
    assert abs(z64.sum().item() - g[key + "_sums"][0]) <= tol * n, key
    assert abs((z64 * z64).sum().item() - g[key + "_sums"][1]) <= tol * n * (2 * zmax + tol), key
    idx = make_golden.fuzz_sample_index(seed, n)
    assert np.abs(z.reshape(-1).numpy()[idx] - g[key + "_sample"]).max() <= tol, key


def test_oracle_matches_stored_fuzz_outputs(golden_dir):
    """The restatement on the seeded inputs of the two live-reference tests below against tests/golden/fuzz_golden.npz,
    at the same tolerances: Z of every embed geometry (shape, float64 sum and sum of squares, a fixed sample of elements)
    and alpha of every alpha case in both modes."""
    g = load(golden_dir, "fuzz_golden")
    embed, alpha = make_golden.fuzz_cases()
    for i, (k, s, feats, Dp, D) in enumerate(embed):
        _check_embed(g, "embed%d" % i, i, restated.embed(feats, k, s, Dp, D), feats, 5e-6)
    feats1, Z1 = make_golden.single_case()
    _check_embed(g, "single", len(embed), restated.embed(feats1, 3, 1, 128, 256), feats1, 2e-6)
    for i, (Z, Zt, tau) in enumerate(alpha):
        assert np.allclose(g["alpha%d_input_sums" % i], [Z.double().sum().item(), Zt.double().sum().item(), tau], rtol=1e-12, atol=1e-9), i
        assert np.abs(restated.matrix_alpha_unsupervised(tau, Z).numpy() - g["alpha%d_unsup" % i]).max() <= 1e-6, (i, tau)
        assert np.abs(restated.matrix_alpha_supervised(tau, Z, Zt).numpy() - g["alpha%d_sup" % i]).max() <= 1e-6, (i, tau)
    assert np.abs(restated.matrix_alpha_unsupervised(1.0, Z1).numpy() - g["single_alpha_unsup"]).max() <= 1e-6


@pytest.mark.skipif(not ref_import.available(), reason="AC_REFERENCE_DIR (a checkout of the original project) not set")
def test_oracle_against_live_reference():
    """Runs the imported reference on the seeded inputs of make_golden.single_case()."""
    feats, Z = make_golden.single_case()
    zr = ref_import.reference_embed(feats, 3, 1, 128, 256)
    zo = restated.embed(feats, 3, 1, 128, 256)
    assert (zr - zo).abs().max().item() <= 2e-6
    ar = ref_import.reference_alpha_unsupervised(1.0, Z)
    ao = restated.matrix_alpha_unsupervised(1.0, Z)
    assert (ar - ao).abs().max().item() <= 1e-6


@pytest.mark.skipif(not ref_import.available(), reason="AC_REFERENCE_DIR (a checkout of the original project) not set")
def test_oracle_fuzz_against_live_reference():
    """The 24 seeded random geometries of make_golden.fuzz_cases() (CNN pyramids with 1-3 layers of different grids, ViT
    token layers, patch size 1/3/5, stride 1/2, pooling up and down, aggregator windows that straddle layers)
    through the imported reference's _embed, and random-tau alpha in both modes, against the restatement."""
    embed, alpha = make_golden.fuzz_cases()
    for case, (k, s, feats, Dp, D) in enumerate(embed):
        zr = ref_import.reference_embed(feats, k, s, Dp, D)
        zo = restated.embed(feats, k, s, Dp, D)
        assert zr.shape == zo.shape, (case, zr.shape, zo.shape)
        assert (zr - zo).abs().max().item() <= 5e-6, (case, k, s, [tuple(f.shape) for f in feats], Dp, D)
    for Z, Zt, tau in alpha:
        assert (ref_import.reference_alpha_unsupervised(tau, Z) - restated.matrix_alpha_unsupervised(tau, Z)).abs().max().item() <= 1e-6
        assert (ref_import.reference_alpha_supervised(tau, Z, Zt) - restated.matrix_alpha_supervised(tau, Z, Zt)).abs().max().item() <= 1e-6
