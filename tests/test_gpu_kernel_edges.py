"""The distance, refine and stage-3 kernels at their tiling and dispatch edges, against plain float64 CPU references.

Every expected value is computed in float64 on the CPU from the SAME rounded operands the kernel reads (hi + lo as
doubles), never from another GPU path, so a check isolates the kernel's arithmetic, tiling and masking from operand
rounding.  The shapes are the ones where a tile split, a template instantiation or a branch changes: D without a whole
64-wide K block, bank images narrower than a 16-wide N tile or straddling 256-wide tiles, query counts that are not whole
images, more than 4096 query blocks, categories, ties.  The float64 helpers at the top are themselves checked against
scipy's brute-force cdist in tests/test_kernel_edges_reference_cpu.py, which runs without a GPU.

Tolerances (each one is restated beside its assert):
  one-pass distance, other images     relative <= 5e-4   (fp32 accumulation of |q|^2 + |b|^2 - 2 q.b over K = D)
  x3 distance, other images           relative <= 5e-5
  own image (distance 0)              absolute <= 2e-3 * scale + 8e-2  (sqrt of a cancelled difference of ~|x|^2 sums)
  plain-form refine                   <= 2e-6 * d + 1e-6  (fp32 sum of (q - b)^2, no cancellation)
  dot-form refine, off the own image  <= 2e-5 * d + 1e-5  (|q|^2 + |b|^2 - 2 q.b in fp32)
An arg-min or key row is accepted when its float64 distance is <= min * (1 + 2e-3) + 1e-6; where the minimum is exactly 0
(duplicate rows), only an exact 0 is accepted.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from anomaly_clustering_b200 import _lib, ops
from anomaly_clustering_b200.distributed import pair_owned

pytestmark = pytest.mark.gpu

ARG_REL, ARG_ABS = 2e-3, 1e-6
COLMIN_INIT = 0x7F7F7F7F                   # column minima / keys start from this (huge, finite) bit pattern
COLKEY_INIT = 0x7F7F7F7F7F7F7F7F


# ----------------------------------------------------------------------------------------------- float64 references (CPU)
def cdist64(a: torch.Tensor, b: torch.Tensor, exact: bool = False) -> torch.Tensor:
    """Euclidean distances [len(a), len(b)] in float64.  exact=True sums explicit differences (equal rows give exactly 0);
    otherwise the matrix-product form, whose cancellation error (~1e-16 |x|^2) is far below every kernel tolerance."""
    mode = "donot_use_mm_for_euclid_dist" if exact else "use_mm_for_euclid_dist"
    return torch.cdist(a.double(), b.double(), compute_mode=mode)


def image_min(q: torch.Tensor, bank: torch.Tensor, P: int, exact: bool = False, chunk: int = 2048):
    """Per bank image: distance of every query row to its nearest bank row and that row's index inside the image.
    q [Mq, D], bank [nb*P, D] -> (dmin [nb, Mq] float64, arg [nb, Mq] int64)."""
    nb = bank.shape[0] // P
    Mq = q.shape[0]
    dmin = torch.empty(nb, Mq, dtype=torch.float64)
    arg = torch.empty(nb, Mq, dtype=torch.int64)
    for r0 in range(0, Mq, chunk):
        d = cdist64(q[r0:r0 + chunk], bank, exact).reshape(-1, nb, P)
        m, a = d.min(dim=2)
        dmin[:, r0:r0 + chunk] = m.T
        arg[:, r0:r0 + chunk] = a.T
    return dmin, arg


def selected_dist(q: torch.Tensor, bank: torch.Tensor, P: int, arg: torch.Tensor) -> torch.Tensor:
    """Distance of query row r to the row arg[j, r] of bank image j, from the differences (exactly 0 for equal rows).
    q [Mq, D], bank [nb*P, D], arg [nb, Mq] -> [nb, Mq] float64."""
    nb = arg.shape[0]
    b = bank.double().reshape(nb, P, -1)
    qd = q.double()
    return torch.stack([(qd - b[j][arg[j].long()]).norm(dim=1) for j in range(nb)])


def arg_accepted(sel: torch.Tensor, dmin: torch.Tensor) -> torch.Tensor:
    """The selected row is a nearest one: within 2e-3 relative of the minimum (near-ties), and exactly 0 where the minimum is 0."""
    return torch.where(dmin == 0, sel == 0, sel <= dmin * (1 + ARG_REL) + ARG_ABS)


def group_table(sizes):
    """(first image, image count) of the category of every image, categories back to back (ops.make_groups on the host)."""
    out, start = [], 0
    for n in sizes:
        out += [(start, n)] * n
        start += n
    return out


def owned(i: int, j: int, n: int, groups=None) -> bool:
    """Query image i owns the pair {i, j} (multiplies it in the symmetric form); with categories only inside j's category,
    by the same rule applied to the category (csrc/mindist_tc.cu: pair_owned_grouped)."""
    if groups is None:
        return pair_owned(i, j, n)
    g0, gn = groups[j]
    if not g0 <= i < g0 + gn:
        return False
    return pair_owned(i - g0, j - g0, gn)


def sym_expect(op: torch.Tensor, P: int, q_img0: int, nq: int, groups=None):
    """Float64 expectation of the symmetric kernel for the query images [q_img0, q_img0 + nq) of the bank op [n*P, D]:
      own     [n, nq] bool      query image q_img0 + k owns the pair with bank image j
      rowmin  [n, nq*P]         distance of each query row to its nearest row of bank image j (defined where own)
      colmin  [nq, n*P]         distance of bank row (j, c) to its nearest row of query image q_img0 + k (defined where own)
    The kernel stores squared distances; compare their square roots."""
    n = op.shape[0] // P
    q = op[q_img0 * P:(q_img0 + nq) * P]
    own = torch.tensor([[owned(q_img0 + k, j, n, groups) for k in range(nq)] for j in range(n)], dtype=torch.bool)
    rowmin, _ = image_min(q, op, P)
    colmin, _ = image_min(op, q, P)
    return own, rowmin, colmin


def reduce_ref(dmin: torch.Tensor, Pq: int, q_self=None, groups=None, mode: str = "mean") -> torch.Tensor:
    """ac_reduce_weights_ex in float64: for query row r of query image k = r // Pq, the mean (or min) of dmin[j, r] over the
    bank images j != q_self[k]; with categories, over q_self[k]'s category only (q_self[k] = -1: the whole bank).  An empty
    set gives nan (mean) or inf (min)."""
    nb, Mq = dmin.shape
    d = dmin.double()
    w = torch.empty(Mq, dtype=torch.float64)
    for k in range((Mq + Pq - 1) // Pq):
        s = -1 if q_self is None else int(q_self[k])
        j0, j1 = (groups[s][0], groups[s][0] + groups[s][1]) if (groups is not None and s >= 0) else (0, nb)
        js = [j for j in range(j0, j1) if j != s]
        rows = slice(k * Pq, min(Mq, (k + 1) * Pq))
        if not js:
            w[rows] = float("nan") if mode == "mean" else float("inf")
        elif mode == "mean":
            w[rows] = d[js, rows].mean(dim=0)
        else:
            w[rows] = d[js, rows].min(dim=0)[0]
    return w


def reduce_sym_ref(rowmin_d2: torch.Tensor, colmin_d2: torch.Tensor, Pq: int, q_img0: int, groups=None) -> torch.Tensor:
    """ac_reduce_weights_sym_ex in float64: w[r] = mean over the bank images j != i of i's category (i = q_img0 + r // Pq) of
    sqrt(rowmin_d2[j, r]) where i owns the pair, else sqrt(colmin_d2[j, r]).  Both arrays [nb, Mq]."""
    nb, Mq = rowmin_d2.shape
    w = torch.empty(Mq, dtype=torch.float64)
    for k in range(Mq // Pq):
        i = q_img0 + k
        j0, j1 = (groups[i][0], groups[i][0] + groups[i][1]) if groups is not None else (0, nb)
        rows = slice(k * Pq, (k + 1) * Pq)
        terms = [(rowmin_d2 if owned(i, j, nb, groups) else colmin_d2)[j, rows].double().sqrt() for j in range(j0, j1) if j != i]
        w[rows] = torch.stack(terms).mean(dim=0) if terms else float("nan")
    return w


def alpha_ref(w: torch.Tensor, tau: float) -> np.ndarray:
    """softmax_p(w / tau) per row in float64, max-subtracted; tau == 0: one-hot on the maximum, ties split equally."""
    x = w.double().numpy()
    m = x.max(axis=1, keepdims=True)
    e = (x == m).astype(np.float64) if tau == 0 else np.exp((x - m) / tau)
    return e / e.sum(axis=1, keepdims=True)


# ----------------------------------------------------------------------------------------------- inputs
def structured(rows: int, P: int, D: int, seed: int, base: torch.Tensor = None):
    """Row r = base[r % P] + 0.5 * noise (the structure of the suite's other distance tests: minima are not degenerate)."""
    gen = torch.Generator().manual_seed(seed)
    if base is None:
        base = torch.randn(P, D, generator=gen)
    return base[torch.arange(rows) % P] + 0.5 * torch.randn(rows, D, generator=gen), base


def operands(X: torch.Tensor, precision: str):
    """Tensor-core operands of fp32 rows X (device): (hi, lo | None, n2, float64 copy of hi + lo on the CPU)."""
    x3 = "x3" in precision
    hi, lo = ops.split_operand(X.cuda().contiguous(), "bf16" if precision.startswith("bf16") else "f16", want_lo=x3)
    n2 = ops.row_norms(hi, lo)
    op64 = hi.double().cpu() + (lo.double().cpu() if lo is not None else 0.0)
    return hi, lo, n2, op64


def dist_tol(precision: str) -> float:
    return 5e-5 if "x3" in precision else 5e-4


def check_rel(got: torch.Tensor, want: torch.Tensor, tol: float, what: str):
    rel = ((got.double() - want).abs() / want.clamp_min(1e-6)).max().item()
    assert rel <= tol, "%s: relative error %.3g > %.3g" % (what, rel, tol)


def _f32_bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int32)


def _key_dist2(key: torch.Tensor) -> torch.Tensor:
    """fp32 squared distance in the high half of (d2 bits << 32 | row) keys."""
    return (key >> 32).to(torch.int32).view(torch.float32)


# ----------------------------------------------------------------------------------------------- all-pairs kernel
# (precision, D, P, Mq, nb_img, first_image, arg): D without a whole 64-wide K block, images narrower than a 16-wide N tile
# (P < 16: one tile spans several bank images), P around the 256-wide tile split (nt 1 -> 2) and P > 1024 (nt = 5), query
# counts that are not whole images and not whole 128 / 256-row blocks, walks that start at another bank image.
AP_CASES = [
    ("f16", 8, 1, 1, 17, 0, False),
    ("bf16", 24, 7, 31, 17, 5, True),
    ("f16x3", 56, 9, 129, 2, 1, False),
    ("bf16x3", 72, 15, 257, 17, 16, True),
    ("f16", 136, 16, 128, 2, 0, True),
    ("bf16", 200, 17, 127, 17, 3, False),
    ("f16x3", 1000, 31, 255, 2, 0, True),
    ("f16", 8, 240, 256, 2, 1, False),
    ("bf16", 24, 255, 4097, 2, 0, True),
    ("f16", 56, 256, 31, 17, 9, True),
    ("f16x3", 72, 257, 129, 17, 0, False),
    ("bf16x3", 136, 272, 255, 2, 1, True),
    ("f16", 200, 513, 257, 2, 0, True),
    ("bf16", 1000, 769, 128, 2, 1, False),
    ("f16x3", 8, 1025, 4097, 2, 1, True),
    ("bf16", 72, 1025, 1, 17, 7, True),
]


@pytest.mark.parametrize("precision,D,P,Mq,nb,first,arg", AP_CASES)
def test_all_pairs_kernel_vs_fp64(precision, D, P, Mq, nb, first, arg):
    """ac_min_dist / ac_min_dist_arg: every dmin entry against float64, and the arg-min names a nearest row."""
    seed = D * 7919 + P * 31 + Mq
    Zb, base = structured(nb * P, P, D, seed)
    Zq, _ = structured(Mq, P, D, seed + 1, base)
    bhi, blo, bn2, b64 = operands(Zb, precision)
    qhi, qlo, qn2, q64 = operands(Zq, precision)
    if arg:
        dmin, am = ops.min_dist_arg(qhi, qlo, qn2, bhi, blo, bn2, nb, P, precision, first_image=first)
    else:
        dmin = ops.min_dist(qhi, qlo, qn2, bhi, blo, bn2, nb, P, precision, first_image=first)
    want, _ = image_min(q64, b64, P)
    got = dmin.cpu()
    assert torch.isfinite(got).all()
    check_rel(got, want, dist_tol(precision), "dmin")          # other images: 5e-4 one pass, 5e-5 x3
    if arg:
        a = am.cpu()
        assert int(a.min()) >= 0 and int(a.max()) < P
        assert arg_accepted(selected_dist(q64, b64, P, a), want).all()


@pytest.mark.parametrize("P,precision", [(1, "f16"), (7, "bf16x3"), (16, "f16x3"), (17, "bf16"), (31, "f16")])
def test_unsupervised_all_pairs_below_32_rows(P, precision):
    """P < 32 (no symmetric form): the all-pairs kernel against the bank itself and the mean over j != i through q_self, as
    pipeline.min_distance_weights runs it.  The own image's entries are distances 0 computed by cancellation."""
    n, D = 9, 72
    Z, _ = structured(n * P, P, D, 1000 + P)
    hi, lo, n2, op = operands(Z, precision)
    dmin = ops.min_dist(hi, lo, n2, hi, lo, n2, n, P, precision)
    q_self = torch.arange(n, dtype=torch.int32, device="cuda")
    w = ops.reduce_weights(dmin, P, q_self, "mean").cpu()
    want, _ = image_min(op, op, P)
    got = dmin.cpu()
    own = torch.zeros(n, n * P, dtype=torch.bool)
    for j in range(n):
        own[j, j * P:(j + 1) * P] = True
    assert ((got.double() - want).abs()[own] <= 2e-3 * want.max() + 8e-2).all()   # own image: cancellation, absolute
    check_rel(got[~own], want[~own], dist_tol(precision), "dmin")               # other images
    check_rel(w, reduce_ref(want, P, q_self.cpu()), dist_tol(precision), "w")   # a mean of entries within that bound


# ----------------------------------------------------------------------------------------------- symmetric kernel
def _check_sym(P, n, q_img0, nq, op, precision, got_row, got_col, got_arg=None, got_key=None, groups=None):
    """Every column minimum / key of the slice, the row minima and arg-mins of owned pairs, against float64."""
    own, rowmin, colmin = sym_expect(op, P, q_img0, nq, groups)
    tol = dist_tol(precision)
    own_rows = own.repeat_interleave(P, dim=1)                                  # [n, nq*P]
    own_cols = own.T.repeat_interleave(P, dim=1)                                # [nq, n*P]
    assert own.any()
    r = got_row.cpu()
    assert torch.isfinite(r[own_rows]).all() and (r[own_rows] >= 0).all()
    check_rel(r[own_rows].sqrt(), rowmin[own_rows], tol, "rowmin")             # owned pairs only: the rest is undefined
    q = op[q_img0 * P:(q_img0 + nq) * P]
    if got_key is None:
        c = got_col.cpu()
        check_rel(c[own_cols].sqrt(), colmin[own_cols], tol, "colmin")
        assert (_f32_bits(c)[~own_cols] == COLMIN_INIT).all()                  # nothing written outside the owned pairs
    else:
        k = got_key.cpu()
        d2 = _key_dist2(k)
        check_rel(d2[own_cols].sqrt(), colmin[own_cols], tol, "colkey distance")
        assert (k[~own_cols] == COLKEY_INIT).all()
        row = (k & 0xFFFFFFFF).long()                                           # row inside query image q_img0 + kk
        assert (row[own_cols] < P).all()
        sel = torch.empty(nq, n * P, dtype=torch.float64)
        for kk in range(nq):
            rows = op[(q_img0 + kk) * P:(q_img0 + kk + 1) * P]
            sel[kk] = (op.double() - rows.double()[row[kk].clamp(max=P - 1)]).norm(dim=1)
        assert arg_accepted(sel, colmin)[own_cols].all()
        a = got_arg.cpu().long()
        assert ((a >= 0) & (a < P))[own_rows].all()
        assert arg_accepted(selected_dist(q, op, P, a.clamp(0, P - 1)), rowmin)[own_rows].all()


# (P, N, D, precision): P from the lower bound 32 (warps straddle two images) up across the 256-wide tile split, odd and even
# N (the N/2 tie rule), D with and without a K tail
SYM_CASES = [
    (32, 2, 64, "f16"),
    (33, 3, 72, "bf16"),
    (47, 4, 128, "f16x3"),
    (63, 5, 200, "bf16x3"),
    (65, 8, 56, "f16"),
    (255, 17, 24, "f16"),
    (257, 5, 136, "bf16"),
    (32, 17, 8, "f16x3"),
    (33, 8, 1000, "f16"),
]


@pytest.mark.parametrize("P,n,D,precision", SYM_CASES)
def test_symmetric_kernel_vs_fp64(P, n, D, precision):
    """ac_min_dist_sym (float column minima) and ac_min_dist_sym_arg (keys) over the whole bank, and the weights of
    ac_reduce_weights_sym against the float64 mean over the other images."""
    Z, _ = structured(n * P, P, D, P * 131 + n * 7 + D)
    hi, lo, n2, op = operands(Z, precision)
    row, col = ops.min_dist_sym(hi, lo, n2, 0, hi, lo, n2, n, P, precision)
    _check_sym(P, n, 0, n, op, precision, row, col)
    w = ops.reduce_weights_sym(row, col, P, 0).cpu()
    want, _ = image_min(op, op, P)
    check_rel(w, reduce_ref(want, P, torch.arange(n)), dist_tol(precision), "w")   # a mean of distances within that bound
    krow, karg, key = ops.min_dist_sym_arg(hi, lo, n2, 0, hi, lo, n2, n, P, precision)
    _check_sym(P, n, 0, n, op, precision, krow, None, karg, key)


@pytest.mark.parametrize("n,P,D,a,b,windows,precision", [
    (9, 33, 72, 3, 7, [(5, 6), (2, 3)], "f16"),        # the first window wraps past the last image
    (9, 33, 72, 3, 7, [(3, 4), (7, 5)], "bf16x3"),     # the second one does
    (8, 64, 136, 5, 8, [(6, 5), (3, 3)], "f16"),       # even N, slice at the end of the bank
])
def test_symmetric_slices_with_wrapping_windows_vs_fp64(n, P, D, a, b, windows, precision):
    """What one rank of a sharded run computes: query images [a, b) of the bank, in two launches over complementary
    circular windows of bank images (init, then accumulate), in both the float and the key form."""
    Z, _ = structured(n * P, P, D, n * 17 + P + a)
    hi, lo, n2, op = operands(Z, precision)
    sl = slice(a * P, b * P)
    out = key_out = None
    for k, win in enumerate(windows):
        out = ops.min_dist_sym(hi[sl], lo[sl] if lo is not None else None, n2[sl], a, hi, lo, n2, n, P, precision,
                               bank_window=win, init=(k == 0), out=out)
        key_out = ops.min_dist_sym_arg(hi[sl], lo[sl] if lo is not None else None, n2[sl], a, hi, lo, n2, n, P, precision,
                                       bank_window=win, init=(k == 0), out=key_out)
    _check_sym(P, n, a, b - a, op, precision, out[0], out[1])
    _check_sym(P, n, a, b - a, op, precision, key_out[0], None, key_out[1], key_out[2])


# ----------------------------------------------------------------------------------------------- categories
@pytest.mark.parametrize("sizes,P,D,precision", [([2, 3, 5, 4, 2], 33, 72, "f16"), ([3, 4, 2], 784, 256, "bf16")])
def test_category_tables_vs_fp64(sizes, P, D, precision):
    """Several categories back to back (groups): row / column minima and keys under grouped ownership, the refined distances
    and the weights of every category against float64; no entry is written across a category."""
    n = sum(sizes)
    groups = group_table(sizes)
    g = ops.make_groups(sizes, "cuda")
    Z, _ = structured(n * P, P, D, sum(s * 10 ** k for k, s in enumerate(sizes)) + P)
    hi, lo, n2, op = operands(Z, precision)
    row, col = ops.min_dist_sym(hi, lo, n2, 0, hi, lo, n2, n, P, precision, groups=g)
    _check_sym(P, n, 0, n, op, precision, row, col, groups=groups)
    krow, karg, key = ops.min_dist_sym_arg(hi, lo, n2, 0, hi, lo, n2, n, P, precision, groups=g)
    _check_sym(P, n, 0, n, op, precision, krow, None, karg, key, groups=groups)
    want, _ = image_min(op, op, P)
    q_self = torch.arange(n, dtype=torch.int32)
    w_want = reduce_ref(want, P, q_self, groups)
    w = ops.reduce_weights_sym(row, col, P, 0, groups=g).cpu()
    check_rel(w, w_want, dist_tol(precision), "w")                              # a mean of distances within that bound
    # refined: distance of the selected pair in fp32 (plain form), then the per-category mean
    dex = ops.refine_min_dist(None, hi, None, hi, None, n, P, karg, colkey=key, groups=g)
    a = karg.cpu().long()
    sel_row = (key.cpu() & 0xFFFFFFFF).long()                                    # [n, n*P] = [bank image, query row] here
    dx = dex.cpu().double()
    for i in range(n):
        g0, gn = groups[i]
        rows = slice(i * P, (i + 1) * P)
        for j in range(g0, g0 + gn):
            if j == i:
                assert (dx[j, rows] == 0).all()                                  # own image
                continue
            c = a[j, rows] if owned(i, j, n, groups) else sel_row[j, rows]
            sel = (op[rows] - op[j * P:(j + 1) * P][c.clamp(0, P - 1)]).norm(dim=1)
            assert arg_accepted(sel, want[j, rows]).all()
            assert ((dx[j, rows] - sel).abs() <= 2e-6 * sel + 1e-6).all()         # plain-form refine
    w_ref = ops.reduce_weights(dex, P, torch.arange(n, dtype=torch.int32, device="cuda"), "mean", groups=g).cpu()
    check_rel(w_ref, w_want, 2e-5, "refined w")                                 # exact pairs, up to near-ties


# ----------------------------------------------------------------------------------------------- beyond 4096 query blocks
def test_symmetric_beyond_unit_table_sampled_pairs_vs_fp64():
    """N = 1025, P = 1024, D = 64: 1,049,600 query rows = 4,100 blocks of 256, past the 4,096 blocks whose image ranges the
    unit builder tabulates in shared memory.  Every owned pair must be written (row minima start as NaN, column minima
    away from the init value exactly where owned); sampled pairs of the first and last raster groups (16 blocks = 4 images)
    are compared with float64 in both orientations; every weight against a float64 reduction of the kernel's minima."""
    n, P, D = 1025, 1024, 64
    gen = torch.Generator().manual_seed(4100)
    base = torch.randn(P, D, generator=gen)
    cgen = torch.Generator(device="cuda").manual_seed(4101)
    Z = base.cuda().repeat(n, 1)
    Z.add_(torch.randn(n * P, D, generator=cgen, device="cuda"), alpha=0.5)
    hi, _ = ops.split_operand(Z, "f16", want_lo=False)
    del Z
    n2 = ops.row_norms(hi)
    Mq = n * P
    row = torch.full((n, Mq), float("nan"), dtype=torch.float32, device="cuda")
    col = torch.empty(n, Mq, dtype=torch.float32, device="cuda")
    ops.min_dist_sym(hi, None, n2, 0, hi, None, n2, n, P, "f16", out=(row, col))
    ii = torch.arange(n, device="cuda")
    dd = (ii[:, None] - ii[None, :]) % n                                        # [j, i]: (j - i) mod n
    own = (dd > 0) & (2 * dd < n)                                               # n odd: no N/2 tie
    w = ops.reduce_weights_sym(row, col, P, 0)
    step = 64
    for i0 in range(0, n, step):                                                # query images [i0, i1)
        i1 = min(n, i0 + step)
        rows = slice(i0 * P, i1 * P)
        o = own[:, i0:i1].repeat_interleave(P, dim=1)
        r_, c_ = row[:, rows], col[:, rows]
        assert torch.isfinite(r_[o]).all() and (r_[o] >= 0).all()               # every owned (row image, bank image) unit ran
        # column minima of [bank image j, query row r] = written by image j (it owns the pair with r's image) or init
        cown = own.T[:, i0:i1].repeat_interleave(P, dim=1)                      # [j, r]: j owns the pair {j, i(r)}
        assert (c_.view(torch.int32)[cown] != COLMIN_INIT).all() and (c_.view(torch.int32)[~cown] == COLMIN_INIT).all()
        sel = torch.where(o, r_, c_).double().clamp_min(0).sqrt()
        sel[torch.arange(i0, i1, device="cuda").repeat_interleave(P), torch.arange(i1 * P - i0 * P, device="cuda")] = 0.0
        w64 = sel.sum(dim=0) / (n - 1)
        # fp32 sums of 1024 square roots in four fixed quarters: ~1e-6 relative typical, 2e-5 bounds it
        assert ((w[rows].double() - w64).abs() / w64).max().item() <= 2e-5
        del o, r_, c_, sel, w64, cown
    # sampled pairs in float64 on the CPU: images of the first raster group and of the last ones
    picks = [0, 1, 3, 1021, 1023, 1024]
    for i in picks:
        for off in (1, 255, 511, 512, 513, 1024):
            j = (i + off) % n
            o_, t_ = (i, j) if pair_owned(i, j, n) else (j, i)                  # owner, other
            ro = hi[o_ * P:(o_ + 1) * P].double().cpu()
            rt = hi[t_ * P:(t_ + 1) * P].double().cpu()
            d = cdist64(ro, rt)                                                 # [rows of o_, rows of t_]
            got_row = row[t_, o_ * P:(o_ + 1) * P].cpu().double().sqrt()       # owner's rows vs the other image
            got_col = col[o_, t_ * P:(t_ + 1) * P].cpu().double().sqrt()       # the other image's rows vs the owner
            check_rel(got_row, d.min(dim=1)[0], 5e-4, "rowmin %d->%d" % (o_, t_))   # one pass, other image
            check_rel(got_col, d.min(dim=0)[0], 5e-4, "colmin %d->%d" % (o_, t_))
    del row, col


# ----------------------------------------------------------------------------------------------- refine
@pytest.mark.parametrize("D", [4096, 1024, 200])
@pytest.mark.parametrize("bank", ["lo", "norms", "plain"])
@pytest.mark.parametrize("dtype", ["f16", "bf16"])
def test_refine_instantiations_vs_fp64(dtype, bank, D):
    """All twelve refine kernels: element type x (bank as hi + lo | squared norms given -> dot form with 16 / 4 / generic
    iterations | neither -> plain form with 16 / generic iterations).  The query comes from fp32 Zq, Qhi or Qhi + Qlo;
    q_self has -1 entries (no pair skipped) and image indices (that pair is 0).  The arg-mins are arbitrary rows: the kernel
    must return the distance of exactly the named pair."""
    nb, P, Mq, Pq = 6, 24, 37, 8
    gen = torch.Generator().manual_seed(D + len(bank) + len(dtype))
    Zb = torch.randn(nb * P, D, generator=gen)
    Zq = torch.randn(Mq, D, generator=gen)
    pr = dtype + ("x3" if bank == "lo" else "")
    bhi, blo, bn2, b64 = operands(Zb, pr)
    src = {4096: "z", 1024: "hi", 200: "hilo"}[D]
    qhi, qlo = ops.split_operand(Zq.cuda(), dtype, want_lo=(src == "hilo"))
    q64 = Zq.double() if src == "z" else qhi.double().cpu() + (qlo.double().cpu() if qlo is not None else 0.0)
    arg = torch.randint(0, P, (nb, Mq), generator=gen, dtype=torch.int32)
    q_self = torch.tensor([2, -1, 0, -1, 5], dtype=torch.int32)
    dex = ops.refine_min_dist(Zq.cuda() if src == "z" else None, qhi, qlo, bhi, blo, nb, P, arg.cuda(),
                              q_self=q_self.cuda(), Pq=Pq, Bn2=bn2 if bank == "norms" else None).cpu().double()
    sel = selected_dist(q64, b64, P, arg)
    skip = torch.zeros(nb, Mq, dtype=torch.bool)
    for k, s in enumerate(q_self.tolist()):
        if s >= 0:
            skip[s, k * Pq:(k + 1) * Pq] = True
    assert (dex[skip] == 0).all()
    err = (dex - sel).abs()[~skip]
    if bank == "norms":
        assert (err <= 2e-5 * sel[~skip] + 1e-5).all(), err.max()             # dot form, off the own image
    else:
        assert (err <= 2e-6 * sel[~skip] + 1e-6).all(), err.max()             # plain form


# ----------------------------------------------------------------------------------------------- ties and degenerate data
@pytest.mark.parametrize("precision", ["f16", "bf16x3"])
def test_ties_duplicates_and_zero_rows(precision):
    """Duplicate images, duplicate rows inside an image, an image whose rows are all equal and zero rows: the minima are
    finite and >= 0, every arg-min and key row attains the exact minimum where it is 0 (a duplicate), and the plain-form
    refined distance of a duplicate is exactly 0."""
    n, P, D = 5, 40, 136
    Z, _ = structured(n * P, P, D, 77)
    Z = Z.reshape(n, P, D)
    Z[0, 5] = Z[0, 2]                        # duplicate rows inside image 0 ...
    Z[1] = Z[0]                              # ... and image 1 duplicates image 0
    Z[3] = Z[3, 0]                           # image 3: all rows equal
    Z[4, :10] = 0.0                          # zero rows (n2 = 0)
    Z[2, 7] = 0.0
    Z = Z.reshape(n * P, D)
    hi, lo, n2, op = operands(Z, precision)
    want, _ = image_min(op, op, P, exact=True)
    assert (want == 0).sum() > n * P         # the ties this test is about exist in the operands
    dmin, arg = ops.min_dist_arg(hi, lo, n2, hi, lo, n2, n, P, precision)
    d = dmin.cpu()
    assert torch.isfinite(d).all() and (d >= 0).all()
    a = arg.cpu()
    sel = selected_dist(op, op, P, a)
    assert arg_accepted(sel, want).all()
    dex = ops.refine_min_dist(None, hi, lo, hi, lo, n, P, arg).cpu()
    assert (dex[want == 0] == 0).all()       # plain form: (q - b)^2 of equal rows is exactly 0
    row, karg, key = ops.min_dist_sym_arg(hi, lo, n2, 0, hi, lo, n2, n, P, precision)
    rowf, col = ops.min_dist_sym(hi, lo, n2, 0, hi, lo, n2, n, P, precision)
    own, rowmin, colmin = sym_expect(op, P, 0, n)
    own_rows = own.repeat_interleave(P, dim=1)
    own_cols = own.T.repeat_interleave(P, dim=1)
    for r_ in (row.cpu(), rowf.cpu()):
        assert torch.isfinite(r_[own_rows]).all() and (r_[own_rows] >= 0).all()
    c = col.cpu()
    assert torch.isfinite(c).all() and (c >= 0).all()
    k = key.cpu()
    assert (_key_dist2(k)[own_cols] >= 0).all()
    selr = selected_dist(op, op, P, karg.cpu().long().clamp(0, P - 1))
    assert arg_accepted(selr, rowmin)[own_rows].all()
    kr = (k & 0xFFFFFFFF).long().clamp(max=P - 1)
    selc = torch.stack([(op.double() - op[i * P:(i + 1) * P].double()[kr[i]]).norm(dim=1) for i in range(n)])
    assert arg_accepted(selc, colmin)[own_cols].all()
    dsym = ops.refine_min_dist(None, hi, lo, hi, lo, n, P, karg, colkey=key).cpu()
    for i in range(n):
        rows = slice(i * P, (i + 1) * P)
        for j in range(n):
            z = want[j, rows] == 0
            assert (dsym[j, rows][z] == 0).all()


# ----------------------------------------------------------------------------------------------- stage 3
@pytest.mark.parametrize("N", [1, 2, 31, 33, 383, 384, 385, 417])
@pytest.mark.parametrize("D", [1, 3, 4, 129])
def test_pairwise_l2_vs_fp64(N, D):
    """Warp kernel up to N = 384, tiled kernel above (32-row tiles with tails); exact symmetry and a zero diagonal."""
    X = torch.randn(N, D, generator=torch.Generator().manual_seed(N * 1000 + D))
    Dm = ops.pairwise_l2(X.cuda()).cpu()
    assert torch.equal(Dm, Dm.T) and (Dm.diagonal() == 0).all()
    want = cdist64(X, X, exact=True)
    # fp32 sum of D rounded squared differences: <= ~D ulp relative, 1e-5 covers D = 129
    assert ((Dm.double() - want).abs() <= 1e-5 * want + 1e-6).all()


@pytest.mark.parametrize("P", [1, 255, 257, 784, 5000])
def test_alpha_64_taus_vs_fp64(P):
    """ac_alpha with the full 64-entry tau table, P past the 256-thread stride; tau = 0 with tied maxima (one-hot, ties
    split) and tiny positive taus, where exp((w - max) / tau) separates neighbouring fp32 values."""
    N = 3
    gen = torch.Generator().manual_seed(P)
    w = (10.0 + torch.rand(N, P, generator=gen)).float()
    if P > 2:
        w[0, [0, P // 2, P - 1]] = w[0].max() + 0.5        # three tied maxima
        w[1, 1] = w[1].max() + 1e-6 * 11                     # one clear maximum a few ulp above the next value
    taus = [0.0, 1e-9, 1e-6, 1e-3] + [float(t) for t in np.logspace(-2, 2, 60)]
    assert len(taus) == 64
    a64, a32 = ops.alpha(w.cuda(), taus)
    a64, a32 = a64.cpu(), a32.cpu()
    for t, tau in enumerate(taus):
        want = alpha_ref(w, tau)
        assert np.abs(a64[t].numpy() - want).max() <= 1e-12, tau
    assert torch.equal(a32, a64.float())                   # alpha32 is the float rounding of alpha64


@pytest.mark.parametrize("D", [6, 130, 256])
def test_weighted_embed_large_P_vs_fp64(D):
    """P = 13,000: the alpha row needs 52 KB of shared memory (> 48 KB: the dynamic-size attribute path), single tau and
    three taus in one pass (a group of two plus a single one); D % 4 != 0 takes the scalar loop."""
    N, P, T = 3, 13000, 3
    gen = torch.Generator().manual_seed(D)
    Z = torch.randn(N, P, D, generator=gen)
    alpha = torch.softmax(2.0 * torch.randn(T, N, P, generator=gen, dtype=torch.float64), dim=-1).float()
    X = ops.weighted_embed(alpha[0].cuda(), Z.cuda()).cpu()
    Xm = ops.weighted_embed_multi(alpha.cuda(), Z.cuda()).cpu()
    want = torch.einsum("tnp,npd->tnd", alpha.double(), Z.double())
    scale = torch.einsum("tnp,npd->tnd", alpha.double().abs(), Z.double().abs())
    # sequential fp32 sum over P: ~sqrt(P) u relative to sum |a z| typical; 4e-5 bounds it and is far below one misread term
    assert ((X.double() - want[0]).abs() <= 4e-5 * scale[0]).all()
    assert ((Xm.double() - want).abs() <= 4e-5 * scale).all()
    assert torch.equal(Xm[0], X)                           # the multi-tau form is bit-identical to the single-tau one


@pytest.mark.parametrize("mode", ["mean", "min"])
@pytest.mark.parametrize("case", ["plain", "q_self", "groups"])
def test_reduce_weights_vs_fp64(mode, case):
    """ac_reduce_weights(_ex): mean and min, q_self with -1 entries, categories, Mq not a multiple of the 256-row block."""
    nb, Pq = 9, 61
    Mq = 5 * Pq
    gen = torch.Generator().manual_seed(len(case) + len(mode))
    dmin = 0.1 + torch.rand(nb, Mq, generator=gen)
    q_self = groups = g = None
    if case != "plain":
        q_self = torch.tensor([0, -1, 3, 8, -1], dtype=torch.int32)
    if case == "groups":
        groups = group_table([2, 4, 3])
        g = ops.make_groups([2, 4, 3], "cuda")
    w = ops.reduce_weights(dmin.cuda(), Pq, q_self.cuda() if q_self is not None else None, mode, groups=g).cpu()
    want = reduce_ref(dmin, Pq, q_self, groups, mode)
    if mode == "min":
        assert torch.equal(w.double(), want)               # a min of fp32 values is exact
    else:
        assert ((w.double() - want).abs() <= 2e-6 * want).all()   # fp32 sum of <= 9 terms


@pytest.mark.parametrize("nb", [2, 3, 5, 9, 33])
def test_reduce_weights_sym_vs_fp64(nb):
    """ac_reduce_weights_sym: 4 quarters x 8-wide loads over bank-image counts that do not split evenly; entries the
    ownership rule does not select hold poison (NaN row minima, negative column minima) and must not be read."""
    P = 40
    gen = torch.Generator().manual_seed(nb)
    for q_img0, nq, sizes in ((0, nb, None), (nb // 2, nb - nb // 2, None), (0, nb, [nb // 2, nb - nb // 2] if nb > 3 else None)):
        groups = group_table(sizes) if sizes else None
        g = ops.make_groups(sizes, "cuda") if sizes else None
        Mq = nq * P
        row = 1.0 + torch.rand(nb, Mq, generator=gen)
        col = 1.0 + torch.rand(nb, Mq, generator=gen)
        for k in range(nq):
            i = q_img0 + k
            j0, j1 = (groups[i][0], groups[i][0] + groups[i][1]) if groups else (0, nb)
            for j in range(nb):
                rows = slice(k * P, (k + 1) * P)
                if j == i or not j0 <= j < j1:
                    row[j, rows], col[j, rows] = float("nan"), -1.0
                elif owned(i, j, nb, groups):
                    col[j, rows] = -1.0
                else:
                    row[j, rows] = float("nan")
        w = ops.reduce_weights_sym(row.cuda(), col.cuda(), P, q_img0, groups=g).cpu()
        want = reduce_sym_ref(row, col, P, q_img0, groups)
        assert ((w.double() - want).abs() <= 1e-5 * want).all()     # fp32 sums of <= 32 square roots


# ----------------------------------------------------------------------------------------------- misaligned pointers
def _offset_view(t: torch.Tensor, elems: int) -> torch.Tensor:
    """A contiguous copy of t that starts `elems` elements into its storage (passes every shape / contiguity check)."""
    buf = torch.empty(t.numel() + elems, dtype=t.dtype, device=t.device)
    v = buf[elems:].view(t.shape)
    v.copy_(t)
    return v


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def test_misaligned_stage3_inputs_match_aligned_bits():
    """Views that start 4 bytes into their storage: ac_weighted_embed(_multi) and ac_pairwise_l2 take the scalar loads and
    return the aligned call's bits (the float4 loads would fault on such an address)."""
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    N, P, D, T = 3, 300, 256, 3
    gen = torch.Generator().manual_seed(3)
    Z = torch.randn(N, P, D, generator=gen).cuda()
    alpha = torch.softmax(torch.randn(T, N, P, generator=gen), dim=-1).cuda()
    Zm = _offset_view(Z, 1)
    assert Zm.data_ptr() % 16 != 0
    assert torch.equal(ops.weighted_embed(alpha[0], Zm), ops.weighted_embed(alpha[0], Z))
    assert torch.equal(ops.weighted_embed_multi(alpha, Zm), ops.weighted_embed_multi(alpha, Z))
    want = ops.weighted_embed_multi(alpha, Z)
    Xm = _offset_view(torch.zeros(T, N, D, device="cuda"), 1)                  # misaligned output
    assert lib.ac_weighted_embed(_ptr(alpha), _ptr(Z), N, P, D, _ptr(Xm), st) == 0
    assert torch.equal(Xm[0], want[0])
    assert lib.ac_weighted_embed_multi(_ptr(alpha), _ptr(Z), T, N, P, D, _ptr(Xm), st) == 0
    assert torch.equal(Xm, want)
    for n in (100, 400):                                                       # warp kernel, tiled kernel
        X = torch.randn(n, D, generator=gen).cuda()
        assert torch.equal(ops.pairwise_l2(_offset_view(X, 1)), ops.pairwise_l2(X))


def test_misaligned_refine_operands_are_refused():
    """ac_refine_min_dist reads Zq, Qhi / Qlo and Bhi / Blo as 16-byte vectors: a base that is not 16-byte aligned returns
    AC_ERR_INVALID instead of faulting; an aligned view at an offset (16 bytes) gives the aligned call's bits."""
    nb, P, D, Mq = 3, 16, 64, 20
    gen = torch.Generator().manual_seed(9)
    Zb = torch.randn(nb * P, D, generator=gen).cuda()
    Zq = torch.randn(Mq, D, generator=gen).cuda()
    bhi, blo = ops.split_operand(Zb, "f16", want_lo=True)
    qhi, qlo = ops.split_operand(Zq, "f16", want_lo=True)
    arg = torch.randint(0, P, (nb, Mq), generator=gen, dtype=torch.int32).cuda()
    want = ops.refine_min_dist(Zq, None, None, bhi, blo, nb, P, arg)
    assert torch.equal(ops.refine_min_dist(_offset_view(Zq, 4), None, None, _offset_view(bhi, 8), _offset_view(blo, 8), nb, P, arg),
                       want)
    cases = [
        dict(Zq=_offset_view(Zq, 1), Qhi=None, Qlo=None, Bhi=bhi, Blo=blo),
        dict(Zq=None, Qhi=_offset_view(qhi, 4), Qlo=qlo, Bhi=bhi, Blo=None),
        dict(Zq=None, Qhi=qhi, Qlo=_offset_view(qlo, 1), Bhi=bhi, Blo=blo),
        dict(Zq=Zq, Qhi=None, Qlo=None, Bhi=_offset_view(bhi, 4), Blo=None),
        dict(Zq=Zq, Qhi=None, Qlo=None, Bhi=bhi, Blo=_offset_view(blo, 1)),
    ]
    for c in cases:
        with pytest.raises(_lib.AcError) as e:
            ops.refine_min_dist(c["Zq"], c["Qhi"], c["Qlo"], c["Bhi"], c["Blo"], nb, P, arg)
        assert e.value.code == _lib.AC_ERR_INVALID
    torch.cuda.synchronize()
