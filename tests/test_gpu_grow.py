"""B200: growing an unsupervised category (ac_min_dist_sym_grow, ac_refine_min_dist_grow, ac_accumulate_weights_grow and
pipeline.GrowingCategory) against fp64 on the same operands and against run_path from scratch on all images so far."""
import numpy as np
import pytest
import torch

from anomaly_clustering_b200 import _lib, cluster, ops, pipeline, synth
from anomaly_clustering_b200.distributed import pair_owned_grow
from oracle import restated

pytestmark = pytest.mark.gpu

SMALL = dict(layers=[(96, 12, 12, True), (96, 12, 12, True)], Dp=256, D=512)      # P = 144
CONFIG2 = dict(layers=[(768, 28, 28, True), (768, 28, 28, True)], Dp=2048, D=4096)  # P = 784 (bench config 2)
ROW_SENTINEL = -7.0
COL_SENTINEL = 3.3e38       # above every squared distance: the kernel's atomicMin would replace it where it computes


def _operands(N, P, D, precision, seed):
    gen = torch.Generator().manual_seed(seed)
    Z = (torch.randn(1, P, D, generator=gen) + 0.5 * torch.randn(N, P, D, generator=gen)).cuda()
    return pipeline.patchset_from_Z(Z, precision)


def _launch(ps, n_old, precision, grow=True, arg=False, init=0):
    """One growth launch (or, grow=False, ac_min_dist_sym_ex on the same window) into outputs pre-filled with sentinels."""
    lib = _lib.load()
    N, P, D = ps.n_img, ps.P, ps.D
    prec = _lib.PRECISIONS[precision]
    q0, Mq = n_old * P, (N - n_old) * P
    rowmin = torch.full((N, Mq), ROW_SENTINEL, dtype=torch.float32, device="cuda")
    colmin = torch.full((N - n_old, N * P), COL_SENTINEL, dtype=torch.float32, device="cuda")
    rowarg = torch.full((N, Mq), -1, dtype=torch.int32, device="cuda") if arg else None
    colkey = torch.full((N - n_old, N * P), -1, dtype=torch.int64, device="cuda") if arg else None
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, N, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    a = (ops._ptr(ps.hi[q0:]), ops._ptr(None if ps.lo is None else ps.lo[q0:]), ops._ptr(ps.n2[q0:]), Mq, n_old, ops._ptr(ps.hi),
         ops._ptr(ps.lo), ops._ptr(ps.n2), N, P, D, prec, 0, N, init, ops._ptr(rowmin), None if arg else ops._ptr(colmin),
         ops._ptr(rowarg), ops._ptr(colkey), None)
    if grow:
        rc = lib.ac_min_dist_sym_grow(*a, n_old, ops._ptr(ws), ws_bytes, ops._stream())
    else:
        rc = lib.ac_min_dist_sym_ex(*a, ops._ptr(ws), ws_bytes, ops._stream())
    _lib.check(rc, "growth launch")
    torch.cuda.synchronize()
    return rowmin, colmin, rowarg, colkey


@pytest.mark.parametrize("precision", ["f16", "bf16x3"])
@pytest.mark.parametrize("n_old,M,P,D", [(0, 5, 784, 256), (7, 1, 100, 320), (6, 3, 36, 128), (9, 2, 260, 512)])
def test_growth_launch_arithmetic(n_old, M, P, D, precision):
    """Owned entries match fp64 on the same rounded operands (tolerances of test_mindist_tensor_core_kernel_arithmetic); every
    other entry keeps the sentinel the test wrote (init = 0), so no pair outside the growth rule was computed.  P = 100 / 36 /
    260 put 256-row query blocks across image boundaries."""
    N = n_old + M
    ps = _operands(N, P, D, precision, seed=N * 100 + P)
    rowmin, colmin, _, _ = _launch(ps, n_old, precision)
    op = (ps.hi.double() + (ps.lo.double() if ps.lo is not None else 0.0)).cpu().reshape(N, P, D)
    rm, cm = rowmin.double().cpu(), colmin.double().cpu()
    want_rm = torch.full_like(rm, ROW_SENTINEL)
    want_cm = torch.full_like(cm, float(torch.tensor(COL_SENTINEL, dtype=torch.float32)))
    owned = torch.zeros_like(rm, dtype=torch.bool)
    owned_c = torch.zeros_like(cm, dtype=torch.bool)
    for i in range(n_old, N):
        r = slice((i - n_old) * P, (i - n_old + 1) * P)
        for j in range(N):
            if pair_owned_grow(n_old, i, j, N):
                d = torch.cdist(op[i], op[j])
                want_rm[j, r] = d.min(dim=1)[0]
                want_cm[i - n_old, j * P:(j + 1) * P] = d.min(dim=0)[0]
                owned[j, r] = True
                owned_c[i - n_old, j * P:(j + 1) * P] = True
    # untouched outside the rule, bit for bit
    assert torch.equal(rm[~owned], want_rm[~owned]) and torch.equal(cm[~owned_c], want_cm[~owned_c])
    tol = 5e-5 if "x3" in precision else 5e-4
    for got2, want in ((rm[owned], want_rm[owned]), (cm[owned_c], want_cm[owned_c])):
        got = got2.clamp_min(0).sqrt()
        assert (got - want).abs().max().item() <= 2e-3 * want.max().item() + 8e-2
        assert ((got - want).abs() / want.clamp_min(1e-6)).max().item() <= tol


@pytest.mark.parametrize("arg", [False, True])
@pytest.mark.parametrize("N,P,D", [(5, 784, 256), (7, 100, 320), (9, 36, 128)])
def test_growth_from_nothing_equals_the_symmetric_launch_bit_for_bit(N, P, D, arg):
    """n_old = 0 is the rule of ac_min_dist_sym: the same units of the same kernel, so every output bit is the same."""
    ps = _operands(N, P, D, "f16", seed=7 * N + P)
    got = _launch(ps, 0, "f16", grow=True, arg=arg, init=1)
    want = _launch(ps, 0, "f16", grow=False, arg=arg, init=1)
    for g, w in zip(got, want):
        if g is not None:
            assert torch.equal(g.view(torch.int32) if g.dtype == torch.float32 else g, w.view(torch.int32) if w.dtype == torch.float32 else w)


def _features(cfg, n, dtype=torch.float32, seed=5):
    feats, labels = synth.planted_features(n, cfg["layers"], n_classes=3, seed=seed)
    return [f.to(dtype).cuda() for f in feats], feats, labels


def _rel_l2(a, b):
    return (torch.linalg.norm((a.double() - b.double()).flatten()) / torch.linalg.norm(b.double().flatten())).item()


def _grow_and_compare(cfg, seq, taus, precision, keep_z, dtype, check):
    feats, feats_cpu, _ = _features(cfg, sum(seq), dtype)
    g = pipeline.GrowingCategory(3, 1, cfg["Dp"], cfg["D"], taus, precision=precision, keep_z=keep_z)
    n = 0
    for m in seq:
        res = g.add([f[n:n + m] for f in feats])
        n += m
        ref = pipeline.run_path([f[:n] for f in feats], 3, 1, cfg["Dp"], cfg["D"], "unsupervised", taus, precision=precision,
                                keep_z=keep_z)
        torch.cuda.synchronize()
        assert res.w.shape == ref.w.shape == (n, ref.w.shape[1]) and res.X.shape == ref.X.shape
        assert (res.Z is None) == (ref.Z is None)
        check(res, ref, [f[:n] for f in feats_cpu], n)


def _check_f16(res, ref, feats_cpu, n):
    assert ((res.w - ref.w).abs() / ref.w.abs()).max().item() <= 1e-5
    assert (res.alpha64 - ref.alpha64).abs().max().item() <= 1e-5
    for t in range(len(ref.taus)):
        assert _rel_l2(res.X[t], ref.X[t]) <= 1e-5
        assert _rel_l2(res.Dmat[t], ref.Dmat[t]) <= 1e-5
        if n >= 3:
            assert np.array_equal(cluster.ward_labels_from_dmat(res.Dmat[t].cpu().numpy(), 3),
                                  cluster.ward_labels_from_dmat(ref.Dmat[t].cpu().numpy(), 3))


@pytest.mark.parametrize("keep_z,dtype", [(False, torch.float32), (True, torch.float32), (False, torch.bfloat16)])
def test_growth_matches_from_scratch_f16(keep_z, dtype):
    """5, +1, +3, +1 images: Z-free (X from the feature maps), keep-Z, and bf16 feature maps."""
    _grow_and_compare(SMALL, [5, 1, 3, 1], [0.5, 1.0, 2.0], "f16", keep_z, dtype, _check_f16)


def test_growth_matches_from_scratch_f16_config2_width():
    """40, +1, +8 images at the config-2 width (P = 784, D = 4096)."""
    _grow_and_compare(CONFIG2, [40, 1, 8], [0.5, 1.0, 2.0], "f16", False, torch.float32, _check_f16)


def test_growth_matches_from_scratch_f16r():
    """The refined precision (what 'auto' picks for any tau < 1): tau = 0 arg-max positions identical to run_path, w within
    1e-4 relative, alpha within the 1e-3 north-star tolerance of the fp64 CPU oracle."""
    taus = [0.0, 0.1, 1.0]

    def check(res, ref, feats_cpu, n):
        assert torch.equal(res.alpha64[0].argmax(dim=-1), ref.alpha64[0].argmax(dim=-1))
        assert ((res.w - ref.w).abs() / ref.w.abs()).max().item() <= 1e-4
        for t, tau in enumerate(taus):
            want = restated.full_path(feats_cpu, 3, 1, SMALL["Dp"], SMALL["D"], tau, "unsupervised")[2]
            assert (res.alpha64[t].cpu() - want).abs().max().item() <= 1e-3, tau

    _grow_and_compare(SMALL, [5, 1, 3, 1], taus, "f16r", False, torch.float32, check)


@pytest.mark.parametrize("precision", ["f16", "f16r"])
def test_regrowth_gives_identical_results(precision):
    """capacity = 2 regrows the buffers twice over 2, +1, +3, +1 images (2 -> 4 -> 8): the same bits as room for all of them."""
    feats, _, _ = _features(SMALL, 7)
    out = []
    for cap in (2, 64):
        g = pipeline.GrowingCategory(3, 1, SMALL["Dp"], SMALL["D"], [0.5, 1.0], precision=precision, capacity=cap)
        n, res = 0, []
        for m in (2, 1, 3, 1):
            res.append(g.add([f[n:n + m] for f in feats]))
            n += m
        out.append((g.capacity, res))
    assert out[0][0] == 8 and out[1][0] == 64
    for a, b in zip(out[0][1], out[1][1]):
        for k in ("w", "alpha64", "X", "Dmat"):
            assert torch.equal(getattr(a, k), getattr(b, k)), k


def test_growth_refuses_mismatched_features():
    feats, _, _ = _features(SMALL, 4)
    g = pipeline.GrowingCategory(3, 1, SMALL["Dp"], SMALL["D"], [1.0])
    with pytest.raises(ValueError, match="at least 2"):
        g.add([f[:1] for f in feats])
    g.add([f[:2] for f in feats])
    other_c, _ = synth.planted_features(1, [(64, 12, 12, True), (96, 12, 12, True)], seed=1)
    other_grid, _ = synth.planted_features(1, [(96, 10, 10, True), (96, 10, 10, True)], seed=1)
    for bad in ([f[2:3] for f in feats[:1]], [f.cuda() for f in other_c], [f.cuda() for f in other_grid],
                [f[2:3].to(torch.bfloat16) for f in feats]):
        with pytest.raises(ValueError, match="differ from the first add"):
            g.add(bad)
    assert g.n_img == 2
    g.add([f[2:4] for f in feats])
    assert g.n_img == 4
