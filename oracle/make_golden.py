"""Generate tests/golden/*.npz by running the UNMODIFIED reference.

    AC_REFERENCE_DIR=<checkout of Anomaly-Clustering> python -m oracle.make_golden

TEST INFRASTRUCTURE.  Each fixture holds seeded synthetic inputs together with the
outputs of the reference's own code (imported from AC_REFERENCE_DIR by oracle/ref_import.py):

  embed_*.npz        AnomalyClusteringCore._embed (models/patchcore/patchcore.py:355-431)
  alpha_*.npz        Matrix_Alpha_Unsupervised / _Supervised (models/patchcore/utils.py:240-277)
                     + the bmm line (examples/main.py:294-296)
  patchify_*.npz     PatchMaker.patchify / Preprocessing / Aggregator standalone
  shipped_cluster_golden.npz
                     extract of the reference's SHIPPED results (outputs/mvtec_ad/**): for a few
                     categories an isometric low-rank copy of X (all pairwise distances kept to
                     ~1e-12), the anomaly labels from info_<cat>.pickle and the NMI/ARI/F1 the
                     reference published in *_tau_result.csv (TAU=2 block).
  fuzz_golden.npz    _embed on the 24 seeded random geometries of fuzz_cases() and on single_case()
                     (shape, float64 sum and sum of squares of Z, Z at a fixed sample of positions)
                     and Matrix_Alpha_* on their seeded alpha cases; `source` says what produced it.

The restatement (oracle/restated.py, oracle/cluster.py) is asserted equal to the reference
here as well, so a fixture is only written when the oracle already agrees with it.

    python -m oracle.make_golden fuzz

writes fuzz_golden.npz alone: from the reference when AC_REFERENCE_DIR is set (after the same
agreement check), otherwise from the restatement, recorded as such in `source`.
"""
from __future__ import annotations

import csv
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import cluster as ocluster  # noqa: E402
from oracle import ref_import, restated  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def _planted_features(gen, B, C, H, W, tokens):
    """Smooth template + noise + a planted 'defect' block so distances have structure."""
    base = torch.randn(1, C, H, W, generator=gen) * 0.7
    x = base + 0.6 * torch.randn(B, C, H, W, generator=gen)
    for b in range(B):
        y0 = int(torch.randint(0, max(1, H - 3), (1,), generator=gen))
        x0 = int(torch.randint(0, max(1, W - 3), (1,), generator=gen))
        x[b, :, y0 : y0 + 3, x0 : x0 + 3] += 2.0 * torch.randn(C, 1, 1, generator=gen)
    if tokens:
        t = x.permute(0, 2, 3, 1).reshape(B, H * W, C)
        cls = torch.randn(B, 1, C, generator=gen)
        return torch.cat([cls, t], dim=1).contiguous()
    return x.contiguous()


EMBED_CASES = {
    # name: (layers [(C,H,W,tokens)], B, patchsize, stride, Dp, D)
    # same pooling ratios as BASELINE config 2 (9C/Dp = 3.375, identity aggregator)
    "embed_vit_small": ([(96, 12, 12, True), (96, 12, 12, True)], 2, 3, 1, 256, 512),
    # same ratios as BASELINE config 1 (4.5 and 9, 2:1 aggregator, 2x bilinear upsample)
    "embed_wrn_small": ([(64, 12, 12, False), (128, 6, 6, False)], 2, 3, 1, 128, 128),
    # ragged: non-integer aggregator ratio straddling layers, odd grids, 3 layers
    "embed_ragged": ([(40, 10, 10, False), (24, 5, 5, False), (17, 7, 7, False)], 3, 3, 1, 100, 77),
    # patchsize 5, stride 2
    "embed_k5s2": ([(12, 11, 11, False), (20, 6, 6, False)], 2, 5, 2, 64, 96),
    # single layer, B=1, upsampling pool (Dp > 9C)
    "embed_single": ([(8, 9, 9, False)], 1, 3, 1, 100, 50),
}


def make_embed():
    for name, (layers, B, k, s, Dp, D) in EMBED_CASES.items():
        gen = torch.Generator().manual_seed(2023)
        feats = [_planted_features(gen, B, C, H, W, tok) for (C, H, W, tok) in layers]
        z_ref = ref_import.reference_embed(feats, k, s, Dp, D)
        z_or = restated.embed(feats, k, s, Dp, D)
        err = (z_ref - z_or).abs().max().item()
        assert err < 2e-6, (name, err)
        out = {"Z": z_ref.numpy(), "patchsize": k, "stride": s, "Dp": Dp, "D": D, "L": len(feats)}
        for i, f in enumerate(feats):
            out["feat%d" % i] = f.numpy()
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
        print(name, tuple(z_ref.shape), "oracle-vs-reference max abs", err)


def make_alpha():
    gen = torch.Generator().manual_seed(2023)
    N, Nb, P, D = 5, 4, 36, 64
    base = torch.randn(1, P, D, generator=gen)
    Z = base + 0.5 * torch.randn(N, P, D, generator=gen)
    Z[1, 5:8] += 1.5
    Z[3, 20:22] -= 2.0
    Zb = base + 0.5 * torch.randn(Nb, P, D, generator=gen)
    out = {"Z": Z.numpy(), "Z_train": Zb.numpy()}
    taus = [0.0, 0.5, 1.0, 2.0]
    out["taus"] = np.array(taus)
    for t in taus:
        au = ref_import.reference_alpha_unsupervised(t, Z)
        asup = ref_import.reference_alpha_supervised(t, Z, Zb)
        ou = restated.matrix_alpha_unsupervised(t, Z)
        osup = restated.matrix_alpha_supervised(t, Z, Zb)
        assert (au - ou).abs().max().item() < 1e-5, ("unsup", t, (au - ou).abs().max().item())
        assert (asup - osup).abs().max().item() < 1e-5, ("sup", t, (asup - osup).abs().max().item())
        out["alpha_unsup_%g" % t] = au.numpy()
        out["alpha_sup_%g" % t] = asup.numpy()
        # examples/main.py:294-296
        xu = np.array(torch.bmm(au.unsqueeze(1).float(), Z).squeeze(1))
        assert np.abs(xu - restated.weighted_embedding(ou, Z)).max() < 1e-4
        out["X_unsup_%g" % t] = xu
    ref = ref_import.load()
    out["w_unsup"] = torch.stack(
        [ref.utils.Weight_Distance_Unsupervised(Z, i, torch.device("cpu")) for i in range(N)]
    ).numpy()
    out["w_sup"] = torch.stack(
        [ref.utils.Weight_Distance_Supervised(Z, Zb, i, torch.device("cpu")) for i in range(N)]
    ).numpy()
    assert np.abs(out["w_unsup"] - restated.weight_distance_unsupervised(Z).numpy()).max() < 1e-5
    assert np.abs(out["w_sup"] - restated.weight_distance_supervised(Z, Zb).numpy()).max() < 1e-5
    np.savez_compressed(os.path.join(GOLD, "alpha_small.npz"), **out)
    print("alpha_small", {k: v.shape for k, v in out.items() if hasattr(v, "shape")})


def make_patchify():
    ref = ref_import.load()
    gen = torch.Generator().manual_seed(7)
    x = torch.randn(2, 6, 7, 5, generator=gen)
    out = {"x": x.numpy()}
    for k, s in [(3, 1), (5, 2), (1, 1)]:
        pm = ref.patchcore.PatchMaker(k, stride=s)
        u, grid = pm.patchify(x, return_spatial_info=True)
        uo, go = restated.patchify(x, k, s)
        assert grid == go and torch.equal(u.contiguous(), uo.contiguous())
        out["patch_k%d_s%d" % (k, s)] = u.contiguous().numpy()
        out["grid_k%d_s%d" % (k, s)] = np.array(grid)
    feats = [torch.randn(10, 6, 3, 3, generator=gen), torch.randn(10, 9, 3, 3, generator=gen)]
    pre = ref.common.Preprocessing([6, 9], 20)(feats)
    agg = ref.common.Aggregator(target_dim=13)(pre)
    assert torch.equal(pre, restated.preprocessing_forward(feats, 20))
    assert torch.equal(agg, restated.aggregator_forward(pre, 13))
    out.update(pre_in0=feats[0].numpy(), pre_in1=feats[1].numpy(), pre_out=pre.numpy(), agg_out=agg.numpy())
    np.savez_compressed(os.path.join(GOLD, "patchify_small.npz"), **out)
    print("patchify_small ok")


def _load_pickle(path):
    import numpy

    with torch.serialization.safe_globals(
        [numpy.ndarray, numpy.dtype, numpy._core.multiarray._reconstruct, type(numpy.dtype("float32"))]
    ):
        try:
            return torch.load(path, map_location="cpu", weights_only=True)
        except Exception:
            return torch.load(path, map_location="cpu", weights_only=False)


def make_shipped():
    base = os.path.join(ref_import.OUTPUTS, "mvtec_ad")
    out = {}
    cases = [("unsupervised", c) for c in ("bottle", "cable", "tile")] + [
        ("supervised", c) for c in ("cable", "hazelnut", "leather")
    ]
    names = []
    for mode, cat in cases:
        run = os.path.join(base, "dino_vitbase8", mode, "blocks.10_blocks.11_2048_4096_2.0_1.0")
        alpha, X = _load_pickle(os.path.join(run, "matrix_alpha_X_%s_%s.pickle" % (cat, mode)))
        info = _load_pickle(os.path.join(base, "info", "info_%s.pickle" % cat))
        anomalies = [d["anomaly"][0] for d in info]
        # CSV TAU=2 block (encoding gbk, examples/test.py:255)
        csv_path = os.path.join(base, "dino_vitbase8", mode, "blocks.10_blocks.11_2048_4096_tau_result.csv")
        want = None
        with open(csv_path, encoding="gbk") as f:
            in_block = False
            for row in csv.reader(f):
                if row and row[0].startswith("TAU="):
                    in_block = row[0] == "TAU=2"
                elif in_block and row and row[0] == cat:
                    want = [float(v) for v in row[1:4]]
        assert want is not None, (mode, cat)
        X = np.asarray(X, dtype=np.float64)
        nmi, ari, f1, _, _ = ocluster.metrics_from_X(X, anomalies)
        assert np.allclose([nmi, ari, f1], want, atol=1e-9), (mode, cat, (nmi, ari, f1), want)
        # isometric low-rank copy: X - mean = U S Vt  ->  coordinates U*S keep all pairwise distances
        Xc = X - X.mean(axis=0, keepdims=True)
        U, S, _ = np.linalg.svd(Xc, full_matrices=False)
        Xlow = U * S
        nmi2, ari2, f12, _, _ = ocluster.metrics_from_X(Xlow, anomalies)
        assert np.allclose([nmi2, ari2, f12], want, atol=1e-9), (mode, cat, "lowrank")
        key = "%s_%s" % (mode, cat)
        names.append(key)
        out[key + "_Xlow"] = Xlow
        out[key + "_anomaly"] = np.array(anomalies)
        out[key + "_csv"] = np.array(want)
        a = alpha.squeeze(1).numpy()
        out[key + "_alpha_rowsum"] = a.sum(axis=1)
        out[key + "_alpha_shape"] = np.array(alpha.shape)
        print(key, X.shape, "metrics", (nmi, ari, f1), "== csv", want)
    out["cases"] = np.array(names)
    np.savez_compressed(os.path.join(GOLD, "shipped_cluster_golden.npz"), **out)


def fuzz_cases():
    """The seeded random geometries of the live fuzz test: 24 embed cases (CNN pyramids with 1-3 layers of different
    grids, ViT token layers, patch size 1/3/5, stride 1/2, pooling up and down, aggregator windows that straddle layers)
    as (k, s, feats, Dp, D), then 8 alpha cases as (Z, Z_train, tau).  One random stream feeds both lists, in this order."""
    rng = np.random.default_rng(2023)
    gen = torch.Generator().manual_seed(2023)
    embed = []
    for case in range(24):
        k = int(rng.choice([1, 3, 3, 3, 5]))
        s = int(rng.choice([1, 1, 1, 2]))
        B = int(rng.integers(1, 3))
        if case % 3 == 0:      # ViT tokens: all layers share the grid
            g = int(rng.integers(4, 9))
            feats = [torch.randn(B, 1 + g * g, int(rng.integers(8, 40)), generator=gen) for _ in range(int(rng.integers(1, 4)))]
        else:                  # CNN pyramid: grid halves per layer
            g = int(rng.choice([8, 12, 16]))
            L = int(rng.integers(1, 4))
            feats = [torch.randn(B, int(rng.integers(6, 30)), max(g >> l, k), max(g >> l, k), generator=gen) for l in range(L)]
        Dp, D = int(rng.integers(5, 70)), int(rng.integers(5, 90))
        embed.append((k, s, feats, Dp, D))
    alpha = []
    for case in range(8):
        N, P, Dd = int(rng.integers(2, 6)), int(rng.integers(4, 30)), int(rng.integers(8, 40))
        Z = torch.randn(N, P, Dd, generator=gen) * float(rng.uniform(0.5, 3.0))
        Zt = torch.randn(int(rng.integers(1, 5)), P, Dd, generator=gen)
        tau = float(rng.choice([0.0, 0.3, 1.0, 2.5, 20.0]))
        alpha.append((Z, Zt, tau))
    return embed, alpha


def single_case():
    """The seeded inputs of the single live check: two ViT token layers [1, 65, 48] (patch 3, stride 1, 128 -> 256) and a
    [4, 30, 32] Z for unsupervised alpha at tau = 1."""
    gen = torch.Generator().manual_seed(11)
    feats = [torch.randn(1, 1 + 64, 48, generator=gen), torch.randn(1, 1 + 64, 48, generator=gen)]
    return feats, torch.randn(4, 30, 32, generator=gen)


FUZZ_SAMPLE = 512       # Z elements stored per embed case, at np.unique(default_rng(seed).integers(0, Z.numel(), FUZZ_SAMPLE))


def fuzz_sample_index(seed, numel):
    return np.unique(np.random.default_rng(seed).integers(0, numel, FUZZ_SAMPLE))


def _store_embed(out, key, seed, z, feats):
    z64 = z.double()
    out[key + "_shape"] = np.array(z.shape)
    out[key + "_sums"] = np.array([z64.sum().item(), (z64 * z64).sum().item()])
    out[key + "_sample"] = z.reshape(-1).numpy()[fuzz_sample_index(seed, z.numel())]
    out[key + "_input_sums"] = np.array([f.double().sum().item() for f in feats])


def make_fuzz():
    live = ref_import.available()
    embed, alpha = fuzz_cases()
    feats1, Z1 = single_case()
    out = {"source": np.array("reference" if live else "restatement")}
    for i, (k, s, feats, Dp, D) in enumerate(embed + [(3, 1, feats1, 128, 256)]):
        z = restated.embed(feats, k, s, Dp, D)
        if live:
            zr = ref_import.reference_embed(feats, k, s, Dp, D)
            assert zr.shape == z.shape and (zr - z).abs().max().item() <= 5e-6, (i, k, s, Dp, D)
            z = zr
        _store_embed(out, "embed%d" % i if i < len(embed) else "single", i, z, feats)
    for i, (Z, Zt, tau) in enumerate(alpha):
        au, asup = restated.matrix_alpha_unsupervised(tau, Z), restated.matrix_alpha_supervised(tau, Z, Zt)
        if live:
            ru, rs = ref_import.reference_alpha_unsupervised(tau, Z), ref_import.reference_alpha_supervised(tau, Z, Zt)
            assert (ru - au).abs().max().item() <= 1e-6 and (rs - asup).abs().max().item() <= 1e-6, (i, tau)
            au, asup = ru, rs
        out["alpha%d_unsup" % i] = au.numpy()
        out["alpha%d_sup" % i] = asup.numpy()
        out["alpha%d_input_sums" % i] = np.array([Z.double().sum().item(), Zt.double().sum().item(), tau])
    a1 = restated.matrix_alpha_unsupervised(1.0, Z1)
    if live:
        r1 = ref_import.reference_alpha_unsupervised(1.0, Z1)
        assert (r1 - a1).abs().max().item() <= 1e-6
        a1 = r1
    out["single_alpha_unsup"] = a1.numpy()
    np.savez_compressed(os.path.join(GOLD, "fuzz_golden.npz"), **out)
    print("fuzz_golden from the", out["source"], "->", os.path.getsize(os.path.join(GOLD, "fuzz_golden.npz")), "bytes")


def main():
    if sys.argv[1:] == ["fuzz"]:
        return make_fuzz()
    assert ref_import.available() and ref_import.outputs_available(), "set AC_REFERENCE_DIR to a checkout of Anomaly-Clustering"
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    make_embed()
    make_alpha()
    make_patchify()
    make_shipped()
    make_fuzz()


if __name__ == "__main__":
    main()
