"""CPU: the consumer side (Ward on a distance matrix, best_map, metrics) and the on-disk format,
checked against the reference's shipped results (tests/golden/shipped_cluster_golden.npz)."""
import os

import numpy as np
import pytest
import torch

from anomaly_clustering_b200 import cluster, io
from oracle import ref_import


def test_metrics_from_distance_matrix_match_published_csv(golden_dir):
    g = np.load(os.path.join(golden_dir, "shipped_cluster_golden.npz"), allow_pickle=False)
    for key in g["cases"]:
        key = str(key)
        X = g[key + "_Xlow"]
        D = np.sqrt(np.maximum(((X[:, None, :] - X[None, :, :]) ** 2).sum(-1), 0))
        nmi, ari, f1, _, _ = cluster.calculate_metrics(D.astype(np.float32), [str(a) for a in g[key + "_anomaly"]])
        assert np.allclose([nmi, ari, f1], g[key + "_csv"], atol=1e-9), key


def test_best_map_permutation_invariance():
    rng = np.random.default_rng(0)
    lab = rng.integers(0, 4, size=60)
    perm = np.array([2, 0, 3, 1])
    assert np.array_equal(cluster.best_map(lab, perm[lab]), lab)


def test_size_weighted_mean():
    assert cluster.size_weighted_mean([1.0, 0.0], [3, 1]) == 0.75


def test_pickle_roundtrip_matches_reference_layout(tmp_path):
    alpha = torch.rand(5, 784, dtype=torch.float64)
    alpha /= alpha.sum(1, keepdim=True)
    X = np.random.default_rng(1).normal(size=(5, 64)).astype(np.float32)
    p = io.save_matrix_alpha_X(str(tmp_path), ["blocks.10", "blocks.11"], 2048, 4096, 2, 1, "bottle", "unsupervised", alpha, X)
    assert p.endswith(os.path.join("blocks.10_blocks.11_2048_4096_2.0_1.0", "matrix_alpha_X_bottle_unsupervised.pickle"))
    a, Xl = io.load_matrix_alpha_X(p)
    assert a.shape == (5, 1, 784) and a.dtype == torch.float32
    assert np.array_equal(Xl, X)


@pytest.mark.skipif(not ref_import.outputs_available(), reason="AC_REFERENCE_DIR (a checkout of the original project) not set")
def test_reads_the_reference_shipped_pickle():
    p = os.path.join(ref_import.OUTPUTS, "mvtec_ad", "dino_vitbase8", "unsupervised", "blocks.10_blocks.11_2048_4096_2.0_1.0",
                     "matrix_alpha_X_bottle_unsupervised.pickle")
    a, X = io.load_matrix_alpha_X(p)
    assert a.shape == (83, 1, 784) and X.shape == (83, 4096)


def test_result_csv_roundtrip_is_byte_identical(golden_dir, tmp_path):
    """tests/golden/shipped_tau_result_head.csv = the first three tau blocks of the reference's shipped
    unsupervised/blocks.10_blocks.11_2048_4096_tau_result.csv: parse it, write it back, same bytes."""
    src = os.path.join(golden_dir, "shipped_tau_result_head.csv")
    mode, blocks = io.read_result_csv(src)
    assert mode == "unsupervised" and [b[0] for b in blocks] == ["0", "0.2", "0.4"]
    assert [r[0] for r in blocks[0][1]] == io.OBJECT + io.TEXTURE + ["MVTec(object)", "MVTec(texture)"]
    out = io.write_result_csv(str(tmp_path / "x.csv"), mode, blocks)
    # the shipped copy went through git's end-of-line normalisation (LF); csv.writer emits CRLF like the reference's does
    assert open(out, "rb").read().replace(b"\r\n", b"\n") == open(src, "rb").read()


# MVTec AD test-set sizes without the 'combined' images, which test.py drops before clustering (cable, pill, zipper and wood
# have 11, 17, 16 and 11 of them)
MVTEC_SIZES = dict(bottle=83, cable=139, capsule=132, hazelnut=110, metal_nut=115, pill=150, screw=160, toothbrush=42, transistor=100,
                   zipper=135, carpet=117, grid=78, leather=124, tile=117, wood=68)


def test_aggregate_rows_match_the_shipped_csv(golden_dir):
    """The MVTec(object) / MVTec(texture) rows of every tau block of the shipped CSV head are size_weighted_mean of the
    category rows, weighted by the images left after dropping 'combined' ones."""
    g = np.load(os.path.join(golden_dir, "shipped_cluster_golden.npz"), allow_pickle=False)
    for key in (str(k) for k in g["cases"]):     # the sizes agree with the stored labels of the reference's info pickles
        assert MVTEC_SIZES[key.split("_", 1)[1]] == sum(str(a) != "combined" for a in g[key + "_anomaly"]), key
    _, blocks = io.read_result_csv(os.path.join(golden_dir, "shipped_tau_result_head.csv"))
    for tau, rows in blocks:
        d = {r[0]: r[1:] for r in rows}
        for c, n in MVTEC_SIZES.items():           # F1-micro is a count of correct images over n
            assert abs(d[c][2] * n - round(d[c][2] * n)) < 1e-9, (tau, c)
        for title, group in (("MVTec(object)", io.OBJECT), ("MVTec(texture)", io.TEXTURE)):
            got = [cluster.size_weighted_mean([d[c][m] for c in group], [MVTEC_SIZES[c] for c in group]) for m in range(3)]
            assert np.allclose(got, d[title], rtol=0, atol=1e-12), (tau, title, got, d[title])


def test_info_pickle_layout(tmp_path):
    info = io.make_info("bottle", ["good", "broken_large", "combined"])
    p = io.save_info(str(tmp_path), "mvtec_ad", "bottle", info)
    assert p.endswith(os.path.join("mvtec_ad", "info", "info_bottle.pickle"))
    back = io.load_info(p)
    assert io.anomaly_names(back) == ["good", "broken_large", "combined"]
    assert back[1]["classname"] == ["bottle"] and int(back[1]["is_anomaly"][0]) == 1 and int(back[0]["is_anomaly"][0]) == 0


def test_weights_roundtrip(tmp_path):
    w = torch.rand(4, 49)
    assert torch.equal(io.load_weights(io.save_weights(str(tmp_path), "bottle", "unsupervised", w)), w)


def _cpu_dmat(X):
    from scipy.spatial.distance import pdist, squareform

    return squareform(pdist(np.asarray(X, dtype=np.float64)))


def test_evaluate_runs_on_synthetic_outputs(tmp_path):
    """The test.py __main__ loop over files written by io: per-category rows, then the size-weighted aggregates;
    'combined' images are dropped before clustering (test.py:183-190)."""
    rng = np.random.default_rng(5)
    root = str(tmp_path)
    sizes = {}
    for cat, n_cls in (("bottle", 3), ("screw", 2), ("tile", 4)):
        names = []
        X = []
        for c in range(n_cls):
            for _ in range(6 + c):
                names.append("good" if c == 0 else "defect%d" % c)
                X.append(rng.normal(size=16) * 0.05 + 3.0 * np.eye(16)[c])
        names.append("combined")
        X.append(rng.normal(size=16))
        sizes[cat] = len(names) - 1
        X = np.asarray(X, dtype=np.float32)
        mode_dir = os.path.join(root, "mvtec_ad", "bb", "unsupervised")
        io.save_matrix_alpha_X(mode_dir, ["l2", "l3"], 8, 16, 1, 1, cat, "unsupervised", torch.full((len(names), 4), 0.25), X)
        io.save_info(root, "mvtec_ad", cat, io.make_info(cat, names))
    blocks = cluster.evaluate_runs(root, "mvtec_ad", "bb", "unsupervised", ["l2", "l3"], 8, 16, [1], dmat_fn=_cpu_dmat)
    (tau, rows), = blocks
    assert [r[0] for r in rows] == ["bottle", "screw", "tile", "MVTec(object)", "MVTec(texture)"]
    assert all(abs(v - 1.0) < 1e-12 for r in rows for v in r[1:])          # well-separated classes: perfect scores
    mode, back = io.read_result_csv(os.path.join(root, "mvtec_ad", "bb", "unsupervised", "l2_l3_8_16_tau_result.csv"))
    assert mode == "unsupervised" and back[0][0] == "1" and [r[0] for r in back[0][1]] == [r[0] for r in rows]


@pytest.mark.parametrize("mode", ["unsupervised", "supervised"])
def test_evaluate_runs_reproduces_the_shipped_csv_block(mode, golden_dir, tmp_path):
    """The reference's shipped results of the categories kept in tests/golden/shipped_cluster_golden.npz (X as an isometric
    copy, the anomaly labels of info_<category>.pickle), written back in the reference's on-disk layout at tau=2 -> the
    category rows of the TAU=2 block of the shipped CSV, and both aggregate rows as the means of those rows weighted as the
    shipped aggregate rows are (test_aggregate_rows_match_the_shipped_csv)."""
    g = np.load(os.path.join(golden_dir, "shipped_cluster_golden.npz"), allow_pickle=False)
    layers = ["blocks.10", "blocks.11"]
    root = str(tmp_path)
    mode_dir = os.path.join(root, "mvtec_ad", "dino_vitbase8", mode)
    want = {}
    for key in (str(k) for k in g["cases"] if str(k).startswith(mode + "_")):
        cat, names = key[len(mode) + 1:], [str(a) for a in g[key + "_anomaly"]]
        X = g[key + "_Xlow"]
        io.save_matrix_alpha_X(mode_dir, layers, 2048, 4096, 2, 1, cat, mode, torch.full((len(X), 784), 1 / 784), X)
        io.save_info(root, "mvtec_ad", cat, io.make_info(cat, names))
        want[cat] = g[key + "_csv"]
    for title, group in (("MVTec(object)", io.OBJECT), ("MVTec(texture)", io.TEXTURE)):
        cats = [c for c in group if c in want]
        want[title] = sum(want[c] * MVTEC_SIZES[c] for c in cats) / sum(MVTEC_SIZES[c] for c in cats)
    blocks = cluster.evaluate_runs(root, "mvtec_ad", "dino_vitbase8", mode, layers, 2048, 4096, [2], dmat_fn=_cpu_dmat,
                                   write_csv=False)
    got = {r[0]: r[1:] for r in blocks[0][1]}
    assert len(got) == 5 and sorted(got) == sorted(want)
    for name, vals in got.items():
        assert np.allclose(vals, want[name], atol=1e-9), (name, vals, want[name])


def test_cli_csv_and_info_collection(tmp_path):
    from anomaly_clustering_b200 import driver, main

    loader = [{"image": torch.zeros(1, 3, 4, 4), "mask": torch.zeros(1, 1, 4, 4), "anomaly": [a], "is_anomaly": torch.tensor([int(a != "good")])}
              for a in ("good", "defect1")]
    info = driver.collect_info(loader)
    assert [sorted(d) for d in info] == [["anomaly", "is_anomaly"]] * 2 and io.anomaly_names(info) == ["good", "defect1"]
    rows = [("bottle", 0.5, 0.1, 0.2, 0.3), ("bottle", 2.0, 0.4, 0.5, 0.6), ("screw", 0.5, 0.7, 0.8, 0.9)]
    p = main.write_cli_csv(str(tmp_path), ["layer2", "layer3"], 1024, 1024, "unsupervised", [0.5, 2.0], rows)
    assert os.path.basename(p) == "layer2_layer3_1024_1024_tau_result.csv"
    mode, blocks = io.read_result_csv(p)
    assert mode == "unsupervised"
    assert blocks == [("0.5", [("bottle", 0.1, 0.2, 0.3), ("screw", 0.7, 0.8, 0.9)]), ("2", [("bottle", 0.4, 0.5, 0.6)])]


def test_cli_flow_with_stubbed_device_calls(tmp_path, monkeypatch):
    """Argument handling and file layout of the CLI; the three calls that need the GPU (backbone + path inside
    make_category_data, ac_pairwise_l2) are stubbed HERE ONLY -- tests/test_gpu_dropin.py runs them for real."""
    from anomaly_clustering_b200 import driver, main, ops

    seen = {}

    def fake_make(path, category, Dp, D, backbone_names, layers, patchsize, save_path, **kw):
        seen[category] = kw
        n = len(list(kw["test_dataloader"]))
        info = driver.collect_info(kw["test_dataloader"])
        io.save_info(kw["info_root"], kw["dataset"], category, info)
        cls = {a: i for i, a in enumerate(sorted(set(io.anomaly_names(info))))}
        X = np.stack([np.eye(D, dtype=np.float32)[cls[a]] * 5 for a in io.anomaly_names(info)])
        out = []
        for t in kw["tau"]:
            io.save_matrix_alpha_X(save_path, layers, Dp, D, t, kw["train_ratio"], category, kw["supervised"], torch.full((n, 1, 9), 1 / 9), X)
            out.append((torch.full((n, 1, 9), 1 / 9), X))
        return out

    monkeypatch.setattr(main, "_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(main.backbones, "load", lambda name, **kw: torch.nn.Identity())
    monkeypatch.setattr(driver, "make_category_data", fake_make)
    monkeypatch.setattr(ops, "pairwise_l2", lambda X: torch.cdist(X.double(), X.double()).float())
    out = str(tmp_path / "outputs")
    rows = main.main(["--backbone_names", "wideresnet50", "--layers_to_extract_from", "layer2", "layer3", "--pretrain_embed_dimension", "16",
                      "--target_embed_dimension", "16", "--tau", "0.5", "2", "--output_dir", out, "--categories", "bottle", "screw",
                      "--synthetic_images", "12", "--synthetic_classes", "3"])
    assert [(r[0], r[1]) for r in rows] == [("bottle", 0.5), ("bottle", 2.0), ("screw", 0.5), ("screw", 2.0)]
    assert all(r[2:] == (1.0, 1.0, 1.0) for r in rows)
    assert seen["bottle"]["supervised"] == "unsupervised" and seen["bottle"]["tau"] == [0.5, 2.0]
    mode_dir = os.path.join(out, "synthetic", "wideresnet50-randinit", "unsupervised")
    assert os.path.exists(os.path.join(mode_dir, "layer2_layer3_16_16_2.0_1.0", "matrix_alpha_X_screw_unsupervised.pickle"))
    assert os.path.exists(os.path.join(out, "synthetic", "info", "info_bottle.pickle"))
    _, blocks = io.read_result_csv(os.path.join(mode_dir, "layer2_layer3_16_16_tau_result.csv"))
    assert [b[0] for b in blocks] == ["0.5", "2"] and [r[0] for r in blocks[1][1]] == ["bottle", "screw"]
    # ... and the offline evaluator (test.py's loop) reads the same tree back
    ev = cluster.evaluate_runs(out, "synthetic", "wideresnet50-randinit", "unsupervised", ["layer2", "layer3"], 16, 16, [0.5, 2.0],
                               objects=["bottle", "screw"], textures=[], dmat_fn=_cpu_dmat, write_csv=False)
    assert [r[0] for r in ev[0][1]] == ["bottle", "screw", "MVTec(object)"] and ev[0][1][2][1:] == (1.0, 1.0, 1.0)
