"""The float64 references of tests/test_gpu_kernel_edges.py against brute force (scipy cdist and plain loops) on tiny shapes,
so that a wrong reference fails here, without a GPU, instead of passing or failing a kernel for the wrong reason."""
import itertools

import numpy as np
import torch
from scipy.spatial.distance import cdist

import test_gpu_kernel_edges as ref
from anomaly_clustering_b200.distributed import pair_owned


def _rows(n, D, seed):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal((n, D)))


def _brute_image_min(q, b, P):
    d = cdist(q.numpy(), b.numpy())                        # [Mq, nb*P]
    nb = b.shape[0] // P
    dmin = np.array([[d[r, j * P:(j + 1) * P].min() for r in range(len(q))] for j in range(nb)])
    return d, dmin


def test_image_min_matches_cdist():
    for exact in (False, True):
        q, b = _rows(11, 5, 1), _rows(3 * 4, 5, 2)
        dmin, arg = ref.image_min(q, b, 4, exact=exact, chunk=4)          # several query chunks
        d, want = _brute_image_min(q, b, 4)
        assert np.abs(dmin.numpy() - want).max() <= 1e-12
        for j in range(3):
            for r in range(11):
                assert d[r, j * 4 + int(arg[j, r])] == d[r, j * 4:(j + 1) * 4].min()
    # explicit differences give exact zeros for equal rows (the tie checks rely on it)
    q = _rows(4, 7, 3) * 1e3
    dmin, _ = ref.image_min(q, q.clone(), 1, exact=True)
    assert (dmin.diagonal() == 0).all()


def test_selected_dist_and_arg_acceptance():
    q, b = _rows(6, 4, 4), _rows(2 * 5, 4, 5)
    arg = torch.tensor([[0, 4, 2, 1, 3, 0], [4, 4, 0, 2, 1, 3]])
    sel = ref.selected_dist(q, b, 5, arg)
    d = cdist(q.numpy(), b.numpy())
    want = np.array([[d[r, j * 5 + int(arg[j, r])] for r in range(6)] for j in range(2)])
    assert np.abs(sel.numpy() - want).max() <= 1e-12
    dmin, best = ref.image_min(q, b, 5)
    assert ref.arg_accepted(ref.selected_dist(q, b, 5, best), dmin).all()
    worst = torch.tensor(d.reshape(6, 2, 5).argmax(axis=2).T.copy())
    assert not ref.arg_accepted(ref.selected_dist(q, b, 5, worst), dmin).any()
    # a zero minimum accepts only an exact zero; a positive one accepts near-ties within 2e-3 relative
    z = torch.zeros(3, dtype=torch.float64)
    assert ref.arg_accepted(z, z).all() and not ref.arg_accepted(z + 1e-9, z).any()
    m = torch.full((2,), 10.0, dtype=torch.float64)
    assert ref.arg_accepted(m * (1 + 1.9e-3), m).all() and not ref.arg_accepted(m * (1 + 2.1e-3), m).any()


def test_grouped_ownership_covers_each_pair_once():
    for sizes in ([5], [4], [2, 3, 5, 4, 2], [3, 4, 2], [1, 6]):
        groups = ref.group_table(sizes)
        n = sum(sizes)
        for i, j in itertools.product(range(n), range(n)):
            same = groups[i] == groups[j]
            o_ij, o_ji = ref.owned(i, j, n, groups), ref.owned(j, i, n, groups)
            if i == j or not same:
                assert not o_ij and not o_ji                    # never the own image, never across categories
            else:
                assert o_ij != o_ji                             # exactly one owner per unordered pair
        if len(sizes) == 1:
            assert all(ref.owned(i, j, n, groups) == ref.owned(i, j, n) == pair_owned(i, j, n)
                       for i, j in itertools.product(range(n), range(n)))


def test_sym_expect_matches_brute_force():
    n, P, D = 5, 3, 4
    op = _rows(n * P, D, 6)
    d = cdist(op.numpy(), op.numpy())
    for q_img0, nq, groups in ((0, n, None), (2, 3, None), (1, 3, ref.group_table([2, 3]))):
        own, rowmin, colmin = ref.sym_expect(op, P, q_img0, nq, groups)
        for k in range(nq):
            i = q_img0 + k
            for j in range(n):
                assert bool(own[j, k]) == ref.owned(i, j, n, groups)
                blk = d[i * P:(i + 1) * P, j * P:(j + 1) * P]  # rows of query image i x rows of bank image j
                # matrix-product form: ~1e-8 |x| at distance 0 (the own image), 1e-12 elsewhere
                tol = 1e-6 if i == j else 1e-12
                assert np.abs(rowmin[j, k * P:(k + 1) * P].numpy() - blk.min(axis=1)).max() <= tol
                assert np.abs(colmin[k, j * P:(j + 1) * P].numpy() - blk.min(axis=0)).max() <= tol


def test_reduce_ref_matches_loops():
    nb, Pq, Mq = 6, 4, 18                                       # Mq not a multiple of Pq: a short last query image
    dmin = torch.from_numpy(np.random.default_rng(7).random((nb, Mq)) + 0.1)
    groups = ref.group_table([2, 4])
    q_self = [1, -1, 3, 0, -1]
    for mode, g in itertools.product(("mean", "min"), (None, groups)):
        w = ref.reduce_ref(dmin, Pq, q_self, g, mode)
        for r in range(Mq):
            s = q_self[r // Pq]
            js = range(nb) if (g is None or s < 0) else range(g[s][0], g[s][0] + g[s][1])
            vals = [float(dmin[j, r]) for j in js if j != s]
            want = np.mean(vals) if mode == "mean" else min(vals)
            assert abs(float(w[r]) - want) <= 1e-12
    w = ref.reduce_ref(dmin, Pq, None, None, "mean")
    assert torch.allclose(w, dmin.mean(dim=0), rtol=0, atol=1e-12)
    one = ref.reduce_ref(dmin[:1, :4], 4, [0], None, "mean"), ref.reduce_ref(dmin[:1, :4], 4, [0], None, "min")
    assert torch.isnan(one[0]).all() and torch.isinf(one[1]).all()    # nothing left to reduce over


def test_reduce_sym_ref_equals_mean_of_minima():
    """Feeding the symmetric reduction the squared minima where the ownership rule reads them (poison elsewhere) gives
    the plain mean of the per-image minima over the other images of the category."""
    n, P, D = 6, 3, 4
    op = _rows(n * P, D, 8)
    for groups in (None, ref.group_table([4, 2])):
        dmin, _ = ref.image_min(op, op, P)
        row = torch.full_like(dmin, float("nan"))
        col = torch.full_like(dmin, -1.0)
        for i, j in itertools.product(range(n), range(n)):
            rows = slice(i * P, (i + 1) * P)
            if i != j and (groups is None or groups[i] == groups[j]):
                (row if ref.owned(i, j, n, groups) else col)[j, rows] = dmin[j, rows] ** 2
        w = ref.reduce_sym_ref(row, col, P, 0, groups)
        want = ref.reduce_ref(dmin, P, list(range(n)), groups, "mean")
        assert torch.allclose(w, want, rtol=1e-12, atol=0)
        # a slice of query images reads the same entries
        ws = ref.reduce_sym_ref(row[:, 2 * P:5 * P], col[:, 2 * P:5 * P], P, 2, groups)
        assert torch.allclose(ws, want[2 * P:5 * P], rtol=1e-12, atol=0)


def test_alpha_ref():
    w = torch.tensor([[1.0, 3.0, 3.0, 2.0], [0.5, 0.25, 0.0, -1.0]])
    a0 = ref.alpha_ref(w, 0.0)
    assert np.array_equal(a0[0], [0.0, 0.5, 0.5, 0.0]) and np.array_equal(a0[1], [1.0, 0.0, 0.0, 0.0])
    x = w.double().numpy()
    for tau in (1e-3, 0.7, 50.0):
        e = np.exp(x / tau - (x / tau).max(axis=1, keepdims=True))
        assert np.abs(ref.alpha_ref(w, tau) - e / e.sum(axis=1, keepdims=True)).max() <= 1e-14


def test_structured_inputs_and_key_helpers():
    Zq, base = ref.structured(10, 4, 3, seed=1)
    Zb, base2 = ref.structured(8, 4, 3, seed=2, base=base)
    assert base2 is base and torch.allclose(Zq[5], base[1], atol=3.0) and Zq.shape == (10, 3)
    # (d2 bits << 32 | row) keys: the high half reads back as the float
    d2 = torch.tensor([0.0, 1.5, 3.0e38], dtype=torch.float32)
    key = (d2.view(torch.int32).long() << 32) | torch.tensor([7, 0, 123])
    assert torch.equal(ref._key_dist2(key), d2) and torch.equal(key & 0xFFFFFFFF, torch.tensor([7, 0, 123]))
    assert ref._key_dist2(torch.tensor([ref.COLKEY_INIT])).item() == torch.tensor([ref.COLMIN_INIT], dtype=torch.int32).view(
        torch.float32).item()
