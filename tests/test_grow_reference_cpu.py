"""The float64 references of tests/test_gpu_grow_edges.py against brute force (scipy cdist and plain loops) on tiny shapes, so
that a wrong reference fails here, without a GPU, instead of passing or failing a growth kernel for the wrong reason."""
import itertools

import numpy as np
import torch
from scipy.spatial.distance import cdist

import test_gpu_grow_edges as ref
from anomaly_clustering_b200.distributed import pair_owned, pair_owned_grow

SHAPES = [(0, 3), (0, 4), (1, 1), (1, 7), (2, 2), (9, 2), (5, 6), (40, 1), (3, 5)]   # (n_old, M), M even gives the tie


def _rows(n, D, seed):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal((n, D)))


def test_grow_owned_is_the_growth_rule():
    for n_old, M in SHAPES:
        N = n_old + M
        own = ref.grow_owned(n_old, N)
        assert own.shape == (N, M)
        for j, k in itertools.product(range(N), range(M)):
            assert bool(own[j, k]) == pair_owned_grow(n_old, n_old + k, j, N)
        # every pair with a new image has exactly one owner, a pair of two old images none
        for i, j in itertools.product(range(N), range(N)):
            o_ij, o_ji = pair_owned_grow(n_old, i, j, N), pair_owned_grow(n_old, j, i, N)
            if i == j or (i < n_old and j < n_old):
                assert not o_ij and not o_ji
            else:
                assert o_ij != o_ji
            if n_old == 0:
                assert o_ij == pair_owned(i, j, N)


def test_grow_masks_layouts():
    P = 3
    for n_old, M in SHAPES:
        N = n_old + M
        rm, cm = ref.grow_masks(n_old, N, P)
        assert rm.shape == (N, M * P) and cm.shape == (M, N * P)
        for j, r in itertools.product(range(N), range(M * P)):
            assert bool(rm[j, r]) == pair_owned_grow(n_old, n_old + r // P, j, N)      # new row r, partner j
        for k, R in itertools.product(range(M), range(N * P)):
            assert bool(cm[k, R]) == pair_owned_grow(n_old, n_old + k, R // P, N)      # new image n_old + k, row R
        # the two "read" masks cover every new (row, partner image) pair exactly once: entries of the other table are not read
        for R, j in itertools.product(range(N * P), range(N)):
            i = R // P
            in_row = i >= n_old and bool(rm[j, R - n_old * P])
            in_col = j >= n_old and bool(cm[j - n_old, R])
            new_pair = i != j and not (i < n_old and j < n_old)
            assert int(in_row) + int(in_col) == int(new_pair)


def test_grow_expect_matches_cdist():
    P, D = 3, 4
    for n_old, M in [(0, 3), (2, 2), (3, 1), (1, 4)]:
        N = n_old + M
        op = _rows(N * P, D, N + n_old)
        rowmin, colmin = ref.grow_expect(op, P, n_old)
        d = cdist(op.numpy(), op.numpy())
        assert rowmin.shape == (N, M * P) and colmin.shape == (M, N * P)
        for j, r in itertools.product(range(N), range(M * P)):
            want = d[n_old * P + r, j * P:(j + 1) * P].min()
            assert abs(float(rowmin[j, r]) - want) <= (1e-6 if j == n_old + r // P else 1e-12)   # own image: cancellation
        for k, R in itertools.product(range(M), range(N * P)):
            want = d[R, (n_old + k) * P:(n_old + k + 1) * P].min()
            assert abs(float(colmin[k, R]) - want) <= (1e-6 if R // P == n_old + k else 1e-12)


def test_refine_grow_expect_matches_loops():
    P, D = 4, 5
    rng = np.random.default_rng(3)
    for n_old, M in [(0, 3), (2, 2), (3, 1), (1, 4)]:
        N = n_old + M
        Z = _rows(N * P, D, 10 + N)
        op = _rows(N * P, D, 20 + N)
        rowarg = torch.from_numpy(rng.integers(0, P, (N, M * P)).astype(np.int32))
        colrow = torch.from_numpy(rng.integers(0, P, (M, N * P)))
        drow, dcol = ref.refine_grow_expect(Z, op, P, n_old, rowarg, colrow)
        z, b = Z.numpy(), op.numpy()
        for j, r in itertools.product(range(N), range(M * P)):
            if pair_owned_grow(n_old, n_old + r // P, j, N):
                want = np.linalg.norm(z[n_old * P + r] - b[j * P + int(rowarg[j, r])])
                assert abs(float(drow[j, r]) - want) <= 1e-12
            else:
                assert np.isnan(float(drow[j, r]))
        for k, R in itertools.product(range(M), range(N * P)):
            if pair_owned_grow(n_old, n_old + k, R // P, N):
                want = np.linalg.norm(z[R] - b[(n_old + k) * P + int(colrow[k, R])])
                assert abs(float(dcol[k, R]) - want) <= 1e-12
            else:
                assert np.isnan(float(dcol[k, R]))


def _replay_loops(rowv, colv, squared, n_old, N, P, S_prev):
    """One row at a time, one Python float (IEEE double) addition per partner image in increasing order."""
    S = np.zeros(N * P)
    for R in range(N * P):
        i = R // P
        s = float(S_prev[R]) if i < n_old else 0.0
        for j in range(n_old if i < n_old else 0, N):
            if j == i:
                continue
            v = rowv[j, R - n_old * P] if pair_owned_grow(n_old, i, j, N) else colv[j - n_old, R]
            s += float(np.sqrt(np.float32(v)) if squared else v)
        S[R] = s
    return S


def test_accumulate_replay_matches_loops():
    P = 3
    rng = np.random.default_rng(5)
    for squared in (False, True):
        S_prev = np.zeros(0)
        n_old = 0
        for m in (2, 1, 3, 2):
            N = n_old + m
            rowv, colv = ref.grow_tables(n_old, N, P, rng)
            S, w = ref.accumulate_replay(rowv, colv, squared, n_old, N, P, S_prev)
            want = _replay_loops(rowv, colv, squared, n_old, N, P, S_prev)
            assert np.array_equal(S, want)                                   # the same additions in the same order
            assert w.dtype == np.float32 and np.array_equal(w, (want / (N - 1)).astype(np.float32))
            assert not np.isnan(S).any()                                     # the NaN entries are never read
            S_prev, n_old = S, N
    S, w = ref.accumulate_replay(np.full((1, P), np.nan, np.float32), np.full((1, P), np.nan, np.float32), True, 0, 1, P, S_prev)
    assert (S == 0).all() and np.isnan(w).all()                                # one image: nothing to average


def test_replayed_growth_sequence_gives_the_mean_over_all_pairs():
    """The tables of a growth sequence (from grow_expect, in float64), composed through the replay, give the float64 mean over
    the other images of the per-image minima of the final set, whichever form (squared minima or distances) they carry."""
    P, D = 3, 4
    seq = [2, 1, 3, 1, 5, 2]
    op = _rows(sum(seq) * P, D, 9)
    d = cdist(op.numpy(), op.numpy())
    for squared in (False, True):
        S_prev = np.zeros(0)
        n_old = 0
        for m in seq:
            N = n_old + m
            rowmin, colmin = ref.grow_expect(op[:N * P], P, n_old)
            rowv, colv = rowmin.numpy(), colmin.numpy()
            if squared:
                rowv, colv = rowv ** 2, colv ** 2
            S, _ = ref.accumulate_replay(rowv, colv, squared, n_old, N, P, S_prev)
            want = np.array([np.mean([d[R, j * P:(j + 1) * P].min() for j in range(N) if j != R // P]) for R in range(N * P)])
            assert np.abs(S / (N - 1) - want).max() <= 1e-12 * want.max()
            S_prev, n_old = S, N


def test_grow_grid_covers_every_value():
    cases = ref.GROW_CASES
    assert len(cases) == 25 and cases == ref.grow_grid()                     # seeded: the same grid every run
    assert {c[0] for c in cases} == set(ref.GROW_PRECISIONS)
    assert {c[1] for c in cases} == set(ref.GROW_P)
    assert {c[2] for c in cases} == set(ref.GROW_D)
    assert {(c[3], c[4]) for c in cases} == set(ref.GROW_NM)
    assert all(c[1] >= 32 and c[2] % 8 == 0 for c in cases)                  # inside what the growth launch accepts


def test_refine_group_width():
    """Jb at config-2 width: 16 partner images with the squared norms (6.4 MB of bf16 / fp16 rows each), 8 with lo parts."""
    assert ref.refine_jb(784, 4096, False) == 16 and ref.refine_jb(784, 4096, True) == 8
    assert ref.refine_jb(37, 200, False) == 256 and ref.refine_jb(10 ** 6, 4096, True) == 4
