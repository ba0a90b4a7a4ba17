"""The category-growth kernels (ac_min_dist_sym_grow, ac_refine_min_dist_grow, ac_accumulate_weights_grow) and
pipeline.GrowingCategory at their tiling and dispatch edges, against plain float64 CPU references.

Every expected value is computed in float64 on the CPU from the SAME rounded operands the kernel reads (hi + lo as doubles,
fp32 Z for the refined query rows), never from another GPU path.  Outputs are pre-filled with sentinels and the launches
write into them without a reset (init = 0 unless stated), so an entry outside the growth ownership rule
(distributed.pair_owned_grow) that is written, or an owned one that is not, fails bit for bit.  The float64 helpers at the
top are checked against scipy's cdist and plain loops in tests/test_grow_reference_cpu.py, which runs without a GPU.

Layouts of one growth launch of M new images [n_old, N) joining n_old old ones (P rows per image):
  rowmin / rowarg / drow / rowv   [N, M*P]   partner image j, new row r (image n_old + r // P)    the new image owns the pair
  colmin / colkey / dcol / colv   [M, N*P]   new image n_old + k, row R of the category          n_old + k owns the pair
Each table is read (and written) only where the rule says; grow_masks gives both masks.

Tolerances (each one is restated beside its assert):
  one-pass distance                   relative <= 5e-4   (fp32 accumulation of |q|^2 + |b|^2 - 2 q.b over K = D)
  x3 distance                         relative <= 5e-5 * max(1, D / 1024): the products are exact and the error is the
                                      tensor core's fp32 accumulation over K = 3 D, whose running sum is not re-rounded to
                                      nearest, so it grows with K (8.5e-5 at D = 4096 measured on a B200; test_gpu_parity.py states
                                      0.1-0.2 absolute in d^2 ~ 1e3 at that width)
  plain-form refine (lo or neither)   <= 2e-6 * d + 1e-6  (fp32 sum of (q - b)^2, no cancellation)
  dot-form refine (norms given)       <= 2e-5 * d + 1e-5  (|q|^2 + |b|^2 - 2 q.b in fp32)
  running sums S                      bit-identical to a CPU replay of the documented order; <= 1e-12 relative of a plain
                                      float64 sum of every pair so far, in any order
  GrowingCategory, refined            w64 * (1 - 2e-5) - 1e-5 <= w <= w64 * (1 + 2e-3) + 1e-5  (refine + arg-min acceptance)
  GrowingCategory, f16                relative <= 5e-4
An arg-min or key row is accepted when its float64 distance is <= min * (1 + 2e-3) + 1e-6 (test_gpu_kernel_edges.arg_accepted).
"""
import math
import random

import numpy as np
import pytest
import torch

from anomaly_clustering_b200 import _lib, ops, pipeline, synth
from anomaly_clustering_b200.distributed import pair_owned_grow
from test_gpu_kernel_edges import arg_accepted, cdist64, check_rel, image_min, operands, selected_dist, structured

pytestmark = pytest.mark.gpu

ROW_SENTINEL = -7.0          # row minima / refined distances are plain stores: any value the kernel never writes
COL_SENTINEL = 3.3e38        # above every squared distance, below the 3.0e38 cut of the kernel's column atomicMin: kept only
                             # where nothing was computed (and not the 0x7F7F7F7F the init fill writes)
ARG_SENTINEL = -1
KEY_SENTINEL = -1            # all ones: larger than every (d2 << 32 | row) key
COLMIN_INIT = 0x7F7F7F7F     # what init = 1 writes into the column minima
REFINE_L2_MB = 128           # kRefineL2MB of csrc/refine.cu
REFINE_WPR = 4               # kWPR of csrc/refine.cu


# ----------------------------------------------------------------------------------------------- float64 references (CPU)
def grow_owned(n_old: int, N: int, device=None) -> torch.Tensor:
    """own [N, M] bool: new image n_old + k owns the pair with image j (pair_owned_grow), built with tensor ops so that it
    also serves the 10^6-row case on the device."""
    M = N - n_old
    j = torch.arange(N, device=device)[:, None]
    k = torch.arange(M, device=device)[None, :]
    jn = j - n_old
    d = (jn - k) % M                                     # circular offset among the new images
    new = (jn >= 0) & (d > 0) & ((2 * d < M) | ((2 * d == M) & (k < jn)))
    return (j < n_old) | new


def grow_masks(n_old: int, N: int, P: int):
    """(row mask [N, M*P], column mask [M, N*P]): the entries one growth launch writes, which are also the entries of the
    arg tables (rowarg, colkey low half) and value tables (rowv, colv) the refine and accumulate kernels read.  Every other
    entry is not read."""
    own = grow_owned(n_old, N)
    return own.repeat_interleave(P, dim=1), own.T.repeat_interleave(P, dim=1)


def grow_expect(op: torch.Tensor, P: int, n_old: int):
    """Float64 minima of one growth launch over the category op [N*P, D]: (rowmin [N, M*P], colmin [M, N*P]) as distances
    (the kernel stores their squares), defined for every entry; compare where grow_masks says."""
    q = op[n_old * P:]
    rowmin, _ = image_min(q, op, P)
    colmin, _ = image_min(op, q, P)
    return rowmin, colmin


def refine_grow_expect(Z: torch.Tensor, op: torch.Tensor, P: int, n_old: int, rowarg: torch.Tensor, colrow: torch.Tensor):
    """Float64 expectation of ac_refine_min_dist_grow: drow [N, M*P] = |Z[new row r] - op[j, rowarg[j, r]]| and dcol [M, N*P] =
    |Z[R] - op[n_old + k, colrow[k, R]]| where the rule reads that table, NaN elsewhere (those entries must keep whatever the
    caller put there)."""
    N = op.shape[0] // P
    rm, cm = grow_masks(n_old, N, P)
    drow = selected_dist(Z[n_old * P:], op, P, rowarg.long())
    dcol = selected_dist(Z, op[n_old * P:], P, colrow.long())
    drow[~rm] = float("nan")
    dcol[~cm] = float("nan")
    return drow, dcol


def new_pair_values(rowv: np.ndarray, colv: np.ndarray, squared: bool, n_old: int, N: int, P: int) -> np.ndarray:
    """V [N, N*P] float64: the value ac_accumulate_weights_grow adds for row R and partner image j over the new pairs of one
    growth launch (sqrt in the tables' own precision when squared), NaN for the pairs it does not add (own image, two old
    images)."""
    V = np.full((N, N * P), np.nan)
    for i in range(N):
        rows = slice(i * P, (i + 1) * P)
        for j in range(N):
            if j == i or (i < n_old and j < n_old):
                continue
            if pair_owned_grow(n_old, i, j, N):
                v = rowv[j, (i - n_old) * P:(i - n_old + 1) * P]
            else:
                v = colv[j - n_old, rows]
            V[j, rows] = (np.sqrt(v) if squared else v).astype(np.float64)
    return V


def accumulate_replay(rowv: np.ndarray, colv: np.ndarray, squared: bool, n_old: int, N: int, P: int, S_prev: np.ndarray):
    """The documented order of ac_accumulate_weights_grow on the CPU: rows of old images continue from S_prev, rows of new
    images from 0; each adds its new pairs in float64 with partner images in increasing order; w = float32(S / (N - 1)).
    Returns (S [N*P] float64, w [N*P] float32)."""
    V = new_pair_values(rowv, colv, squared, n_old, N, P)
    S = np.zeros(N * P)
    S[:n_old * P] = S_prev[:n_old * P]
    for j in range(N):                                   # partner images in increasing order, one float64 add each
        new = ~np.isnan(V[j])
        S[new] = S[new] + V[j, new]
    with np.errstate(invalid="ignore", divide="ignore"):
        w = (S / (N - 1)).astype(np.float32) if N > 1 else np.full(N * P, np.nan, dtype=np.float32)
    return S, w


def refine_jb(P: int, D: int, lo: bool) -> int:
    """Partner images per group of ac_refine_min_dist_grow (run_refine in csrc/refine.cu):
    Jb = max(4, min(256, 128e6 / (P * D * 2 * (2 if lo else 1)))) rounded down to a multiple of 4."""
    jb = int(max(float(REFINE_WPR), min(256.0, REFINE_L2_MB * 1.0e6 / (P * D * 2.0 * (2 if lo else 1)))))
    return jb - jb % REFINE_WPR


# ----------------------------------------------------------------------------------------------- launches
def _f32_bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int32)


def _bits_of(v: float) -> int:
    return int(torch.tensor([v], dtype=torch.float32).view(torch.int32))


def _outputs(n_old: int, N: int, P: int, arg: bool):
    """Sentinel-filled outputs of one growth launch: (rowmin, colmin | None, rowarg | None, colkey | None)."""
    M, dev = N - n_old, "cuda"
    rowmin = torch.full((N, M * P), ROW_SENTINEL, dtype=torch.float32, device=dev)
    if arg:
        return (rowmin, None, torch.full((N, M * P), ARG_SENTINEL, dtype=torch.int32, device=dev),
                torch.full((M, N * P), KEY_SENTINEL, dtype=torch.int64, device=dev))
    return rowmin, torch.full((M, N * P), COL_SENTINEL, dtype=torch.float32, device=dev), None, None


def _launch(hi, lo, n2, n_old: int, N: int, P: int, precision: str, out, window=None, init: int = 0):
    """ac_min_dist_sym_grow over bank window (begin, count) into the caller's outputs (no allocation, no reset unless init)."""
    lib = _lib.load()
    D = hi.shape[1]
    prec = _lib.PRECISIONS[precision]
    q0, Mq = n_old * P, (N - n_old) * P
    begin, count = window if window is not None else (0, N)
    rowmin, colmin, rowarg, colkey = out
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, N, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    rc = lib.ac_min_dist_sym_grow(ops._ptr(hi[q0:]), ops._ptr(None if lo is None else lo[q0:]), ops._ptr(n2[q0:]), Mq, n_old,
                                  ops._ptr(hi), ops._ptr(lo), ops._ptr(n2), N, P, D, prec, int(begin), int(count), int(init),
                                  ops._ptr(rowmin), ops._ptr(colmin), ops._ptr(rowarg), ops._ptr(colkey), None, n_old, ops._ptr(ws),
                                  ws_bytes, ops._stream())
    _lib.check(rc, "ac_min_dist_sym_grow")
    torch.cuda.synchronize()
    return out


def _tol(precision: str, D: int) -> float:
    return 5e-5 * max(1.0, D / 1024) if "x3" in precision else 5e-4


def _key_rows(key: torch.Tensor) -> torch.Tensor:
    return (key & 0xFFFFFFFF).long()


def _key_d2_bits(key: torch.Tensor) -> torch.Tensor:
    return (key >> 32).to(torch.int32)


# ----------------------------------------------------------------------------------------------- a. growth launch vs fp64
GROW_PRECISIONS = ["f16", "bf16", "f16x3", "bf16x3"]
GROW_P = [32, 33, 63, 255, 257, 784, 1025]
GROW_D = [8, 24, 72, 200, 1000, 4096]
GROW_NM = [(0, 3), (1, 1), (1, 7), (9, 2), (5, 6), (40, 1)]


def grow_grid(n: int = 25, seed: int = 2024):
    """A seeded sample of (precision, P, D, n_old, M) in which every value of every axis appears at least once: each axis is
    its values once, then random picks, shuffled independently of the others."""
    rng = random.Random(seed)

    def axis(vals):
        col = list(vals) + [rng.choice(vals) for _ in range(n - len(vals))]
        rng.shuffle(col)
        return col

    return [(pr, P, D, nm[0], nm[1]) for pr, P, D, nm in zip(axis(GROW_PRECISIONS), axis(GROW_P), axis(GROW_D), axis(GROW_NM))]


GROW_CASES = grow_grid()


@pytest.mark.parametrize("precision,P,D,n_old,M", GROW_CASES)
def test_growth_launch_vs_fp64(precision, P, D, n_old, M):
    """ac_min_dist_sym_grow in the float and the arg-recording form, init = 0 into sentinels: owned row and column minima
    against float64, every unowned entry of rowmin / rowarg / colmin / colkey keeps its sentinel bit for bit, every rowarg and
    key row names a nearest row, and the keys carry the float form's column minima.  P from 32 (warps straddle images) to
    1025 (5 N tiles), D with K tails and below one 64-wide K block, M even (the M/2 tie among new images), one new image
    against 40 old ones and many new images against one."""
    N = n_old + M
    Z, _ = structured(N * P, P, D, seed=P * 1009 + D * 13 + N * 7 + GROW_PRECISIONS.index(precision))
    hi, lo, n2, op = operands(Z, precision)
    own_r, own_c = grow_masks(n_old, N, P)
    want_r, want_c = grow_expect(op, P, n_old)
    tol = _tol(precision, D)

    rm, cm, _, _ = (t.cpu() if t is not None else None for t in _launch(hi, lo, n2, n_old, N, P, precision, _outputs(n_old, N, P, False)))
    assert (_f32_bits(rm)[~own_r] == _bits_of(ROW_SENTINEL)).all()           # nothing written outside the rule
    assert (_f32_bits(cm)[~own_c] == _bits_of(COL_SENTINEL)).all()
    assert (rm[own_r] >= 0).all() and torch.isfinite(rm[own_r]).all()
    check_rel(rm[own_r].double().sqrt(), want_r[own_r], tol, "rowmin")      # 5e-4 one pass, 5e-5 x3 (2e-4 at D = 4096)
    check_rel(cm[own_c].double().sqrt(), want_c[own_c], tol, "colmin")

    krm, _, karg, key = (t.cpu() if t is not None else None for t in _launch(hi, lo, n2, n_old, N, P, precision, _outputs(n_old, N, P, True)))
    assert (_f32_bits(krm)[~own_r] == _bits_of(ROW_SENTINEL)).all()
    assert (karg[~own_r] == ARG_SENTINEL).all() and (key[~own_c] == KEY_SENTINEL).all()
    check_rel(krm[own_r].double().sqrt(), want_r[own_r], tol, "rowmin (arg form)")
    a = karg.long()
    assert ((a >= 0) & (a < P))[own_r].all()
    assert arg_accepted(selected_dist(op[n_old * P:], op, P, a.clamp(0, P - 1)), want_r)[own_r].all()
    krow = _key_rows(key)
    assert (krow[own_c] < P).all()
    assert arg_accepted(selected_dist(op, op[n_old * P:], P, krow.clamp(max=P - 1)), want_c)[own_c].all()
    # the key's high half is the column minimum of the float form: the same squared distances, the same minimum
    assert torch.equal(_key_d2_bits(key)[own_c], _f32_bits(cm)[own_c])


# ----------------------------------------------------------------------------------------------- b. bank windows
@pytest.mark.parametrize("precision,n_old,M,P,D,windows", [
    ("f16", 5, 4, 33, 72, [(6, 5), (2, 4)]),                 # the first window wraps past the last image
    ("bf16x3", 3, 6, 40, 136, [(7, 4), (2, 3), (5, 2)]),     # three windows, the first wraps
    ("bf16", 4, 3, 257, 24, [(2, 3), (5, 3), (1, 1)]),       # the second wraps (5, 6, 0)
])
def test_growth_windows_equal_one_full_launch(precision, n_old, M, P, D, windows):
    """Growth launches over circular windows of bank images that together cover the category once, init on the first only,
    give the full-window launch's bits in rowmin / colmin and in rowmin / rowarg / colkey."""
    N = n_old + M
    assert sorted((b + t) % N for b, c in windows for t in range(c)) == list(range(N))
    Z, _ = structured(N * P, P, D, seed=N * 31 + P)
    hi, lo, n2, _ = operands(Z, precision)
    for arg in (False, True):
        full = _launch(hi, lo, n2, n_old, N, P, precision, _outputs(n_old, N, P, arg), init=1)
        out = _outputs(n_old, N, P, arg)
        for k, win in enumerate(windows):
            _launch(hi, lo, n2, n_old, N, P, precision, out, window=win, init=int(k == 0))
        for g, w in zip(out, full):
            if g is not None:
                assert torch.equal(g.view(torch.int32) if g.dtype == torch.float32 else g,
                                   w.view(torch.int32) if w.dtype == torch.float32 else w)


@pytest.mark.parametrize("precision,n_old,M,P,D,window", [("f16", 6, 3, 48, 64, (1, 4)), ("bf16x3", 5, 4, 257, 72, (0, 5))])
def test_growth_window_of_old_images_writes_exactly_their_pairs(precision, n_old, M, P, D, window):
    """A window of old images only: a new image owns every pair with an old one, so exactly the (new row, old image) row minima
    and the (new image, old row) column minima / keys of the window's images are written (and match float64); every other
    entry keeps its sentinel."""
    N = n_old + M
    b, c = window
    assert b + c <= n_old
    Z, _ = structured(N * P, P, D, seed=N * 37 + P)
    hi, lo, n2, op = operands(Z, precision)
    want_r, want_c = grow_expect(op, P, n_old)
    in_win = torch.zeros(N, dtype=torch.bool)
    in_win[b:b + c] = True
    wr = in_win[:, None].expand(N, M * P).clone()             # [j, r]: partner j in the window
    wc = in_win.repeat_interleave(P)[None, :].expand(M, N * P).clone()   # [k, R]: row R of an image in the window
    tol = _tol(precision, D)
    rm, cm, _, _ = _launch(hi, lo, n2, n_old, N, P, precision, _outputs(n_old, N, P, False), window=window)
    rm, cm = rm.cpu(), cm.cpu()
    assert (_f32_bits(rm)[~wr] == _bits_of(ROW_SENTINEL)).all() and (_f32_bits(cm)[~wc] == _bits_of(COL_SENTINEL)).all()
    check_rel(rm[wr].double().sqrt(), want_r[wr], tol, "rowmin")
    check_rel(cm[wc].double().sqrt(), want_c[wc], tol, "colmin")
    krm, _, karg, key = (t.cpu() if t is not None else None
                         for t in _launch(hi, lo, n2, n_old, N, P, precision, _outputs(n_old, N, P, True), window=window))
    assert (_f32_bits(krm)[~wr] == _bits_of(ROW_SENTINEL)).all()
    assert (karg[~wr] == ARG_SENTINEL).all() and (key[~wc] == KEY_SENTINEL).all()
    check_rel(krm[wr].double().sqrt(), want_r[wr], tol, "rowmin (arg form)")
    assert ((karg >= 0) & (karg < P))[wr].all() and (_key_rows(key)[wc] < P).all()
    assert torch.equal(_key_d2_bits(key)[wc], _f32_bits(cm)[wc])


# ----------------------------------------------------------------------------------------------- c. past 4096 query blocks
def test_growth_beyond_unit_table_sampled_pairs_vs_fp64():
    """N = 1025 (8 old + 1017 new), P = 1032, D = 64: 1,049,544 new rows = 4,100 query blocks of 256, past the 4,096 whose image
    ranges the unit builder tabulates; a new image's candidates are all 1025 images (KU = nb_img).  Every owned entry is
    written (row minima start as NaN), every unowned column entry still holds the init value, and sampled (new, old) and
    (new, new) pairs of the first and last raster groups (16 blocks, about 4 images) match float64 in both orientations."""
    n_old, M, P, D = 8, 1017, 1032, 64
    N, Mq = n_old + M, M * P
    assert (Mq + 255) // 256 == 4100 and M % 2 == 1                            # M odd: no tie among the new images
    gen = torch.Generator().manual_seed(4100)
    base = torch.randn(P, D, generator=gen)
    cgen = torch.Generator(device="cuda").manual_seed(4102)
    Z = base.cuda().repeat(N, 1)
    Z.add_(torch.randn(N * P, D, generator=cgen, device="cuda"), alpha=0.5)
    hi, _ = ops.split_operand(Z, "f16", want_lo=False)
    del Z
    n2 = ops.row_norms(hi)
    row = torch.full((N, Mq), float("nan"), dtype=torch.float32, device="cuda")
    col = torch.full((M, N * P), COL_SENTINEL, dtype=torch.float32, device="cuda")
    _launch(hi, None, n2, n_old, N, P, "f16", (row, col, None, None), init=1)
    own = grow_owned(n_old, N, device="cuda")                                  # [N, M]
    step = 64
    for k0 in range(0, M, step):
        k1 = min(M, k0 + step)
        o = own[:, k0:k1].repeat_interleave(P, dim=1)
        r_ = row[:, k0 * P:k1 * P]
        assert torch.isfinite(r_[o]).all() and (r_[o] >= 0).all()              # every owned (new row, image) unit ran
        assert torch.isnan(r_[~o]).all()                                        # ... and no other
        c_ = _f32_bits(col[k0:k1])
        co = own.T[k0:k1].repeat_interleave(P, dim=1)
        assert (c_[co] != COLMIN_INIT).all() and (c_[~co] == COLMIN_INIT).all()
        del o, r_, c_, co
    # images 8..11 fill the first raster group, image 1023 ends the tabulated blocks, image 1024 is the last group
    for i in (8, 9, 11, 1023, 1024):
        k = i - n_old
        partners = [0, n_old - 1] + [n_old + (k + off) % M for off in (1, 508, 509, 1016)]
        for j in partners:
            o_, t_ = (i, j) if pair_owned_grow(n_old, i, j, N) else (j, i)       # owner (a new image), other
            ro = hi[o_ * P:(o_ + 1) * P].double().cpu()
            rt = hi[t_ * P:(t_ + 1) * P].double().cpu()
            d = cdist64(ro, rt)
            got_row = row[t_, (o_ - n_old) * P:(o_ - n_old + 1) * P].cpu().double().sqrt()
            got_col = col[o_ - n_old, t_ * P:(t_ + 1) * P].cpu().double().sqrt()
            check_rel(got_row, d.min(dim=1)[0], 5e-4, "rowmin %d->%d" % (o_, t_))   # one pass
            check_rel(got_col, d.min(dim=0)[0], 5e-4, "colmin %d->%d" % (o_, t_))
    del row, col


# ----------------------------------------------------------------------------------------------- d. refine, growth form
def _refine_grow_case(dtype: str, bank: str, n_old: int, M: int, P: int, D: int, seed: int):
    N, Mn = n_old + M, M * P
    gen = torch.Generator().manual_seed(seed)
    Z = torch.randn(N * P, D, generator=gen)
    hi, lo, n2, op = operands(Z, dtype + ("x3" if bank == "lo" else ""))
    rm, cm = grow_masks(n_old, N, P)
    rowarg = torch.randint(0, P, (N, Mn), generator=gen, dtype=torch.int32)
    colrow = torch.randint(0, P, (M, N * P), generator=gen, dtype=torch.int64)
    # a pair of two new images has an entry in both tables: the one the rule does not read names another row
    A, C, read_a = rowarg[n_old:], colrow[:, n_old * P:], rm[n_old:]           # both [M, Mn], the same (partner, row) pairs
    C[read_a] = (A[read_a].long() + 1) % P
    A[~read_a] = ((C[~read_a] + 1) % P).int()
    d2_bits = torch.randint(0x3F800000, 0x42C80000, (M, N * P), generator=gen, dtype=torch.int64)   # arbitrary floats 1 .. 100
    colkey = (d2_bits << 32) | colrow
    drow = torch.full((N, Mn), ROW_SENTINEL, dtype=torch.float32, device="cuda")
    dcol = torch.full((M, N * P), ROW_SENTINEL, dtype=torch.float32, device="cuda")
    lib = _lib.load()
    Zd, rowarg_d, colkey_d = Z.cuda(), rowarg.cuda(), colkey.cuda()
    rc = lib.ac_refine_min_dist_grow(ops._ptr(Zd), ops._ptr(hi), ops._ptr(lo), ops._TORCH_TO_AC[hi.dtype], n_old, N, P, D,
                                     ops._ptr(rowarg_d), ops._ptr(colkey_d), ops._ptr(n2 if bank != "plain" else None),
                                     ops._ptr(drow), ops._ptr(dcol), ops._stream())
    _lib.check(rc, "ac_refine_min_dist_grow")
    torch.cuda.synchronize()
    want_r, want_c = refine_grow_expect(Z.double(), op, P, n_old, rowarg, colrow)
    dr, dc = drow.cpu(), dcol.cpu()
    assert (_f32_bits(dr)[~rm] == _bits_of(ROW_SENTINEL)).all()               # other pairs untouched
    assert (_f32_bits(dc)[~cm] == _bits_of(ROW_SENTINEL)).all()
    rel, ab = (2e-5, 1e-5) if bank == "norms" else (2e-6, 1e-6)                # dot form / plain form
    for got, want, m, what in ((dr, want_r, rm, "drow"), (dc, want_c, cm, "dcol")):
        err = (got.double()[m] - want[m]).abs()
        assert (err <= rel * want[m] + ab).all(), "%s: max error %.3g" % (what, err.max().item())


@pytest.mark.parametrize("D", [4096, 1024, 200])
@pytest.mark.parametrize("bank", ["lo", "norms", "plain"])
@pytest.mark.parametrize("dtype", ["f16", "bf16"])
def test_refine_grow_instantiations_vs_fp64(dtype, bank, D):
    """All twelve growth refine kernels: element type x (bank as hi + lo | squared norms -> dot form with 16 / 4 / generic
    iterations | neither -> plain form with 16 / generic iterations).  P = 37 with 3 old and 5 new images: neither launch's
    row count (111, 185) is a multiple of the kernel's 4-row block.  rowarg and colkey hold arbitrary rows, and where a pair
    of new images has an entry in both, the one the rule does not read names another row; outside the rule drow / dcol keep
    their sentinel."""
    _refine_grow_case(dtype, bank, 3, 5, 37, D, seed=D + 10 * len(bank) + len(dtype))


@pytest.mark.parametrize("dtype,bank,n_old,M,P,D", [
    ("f16", "norms", 3, 18, 784, 4096),     # Jb = 16: 21 and 18 partner images take 2 groups in both launches
    ("bf16", "lo", 3, 18, 784, 4096),       # Jb = 8: 3 groups in both launches
    ("f16", "plain", 0, 5, 37, 200),        # no old image: the second launch is empty
    ("bf16", "norms", 30, 1, 37, 200),      # one new image against 30 old ones
])
def test_refine_grow_partner_groups_and_edge_counts(dtype, bank, n_old, M, P, D):
    """The partner images of each launch are split into groups of Jb (refine_jb, the formula of run_refine); the shapes at
    config-2 width run several groups in both launches, so the second launch's jbase + blockIdx.y * Jb offset is used."""
    N = n_old + M
    if P == 784:
        jb = refine_jb(P, D, bank == "lo")
        assert jb == (8 if bank == "lo" else 16)
        assert math.ceil(N / jb) > 1 and math.ceil(M / jb) > 1
    _refine_grow_case(dtype, bank, n_old, M, P, D, seed=N * 100 + P)


# ----------------------------------------------------------------------------------------------- e. accumulate, replayed
def grow_tables(n_old: int, N: int, P: int, rng: np.random.Generator):
    """Synthetic positive fp32 (rowv [N, M*P], colv [M, N*P]) with NaN in every entry the rule says is not read."""
    rm, cm = grow_masks(n_old, N, P)
    rowv = rng.uniform(0.25, 60.0, rm.shape).astype(np.float32)
    colv = rng.uniform(0.25, 60.0, cm.shape).astype(np.float32)
    rowv[~rm.numpy()] = np.nan
    colv[~cm.numpy()] = np.nan
    return rowv, colv


def _accumulate(rowv, colv, squared, n_old, N, P, S):
    w = torch.full((N * P,), float("inf"), dtype=torch.float32, device="cuda")
    lib = _lib.load()
    r, c = torch.from_numpy(rowv).cuda(), torch.from_numpy(colv).cuda()
    _lib.check(lib.ac_accumulate_weights_grow(ops._ptr(r), ops._ptr(c), int(squared), n_old, N, P, ops._ptr(S), ops._ptr(w),
                                              ops._stream()), "ac_accumulate_weights_grow")
    torch.cuda.synchronize()
    return w


@pytest.mark.parametrize("P", [37, 784])
@pytest.mark.parametrize("squared", [0, 1])
def test_accumulate_grow_replayed_exactly(squared, P):
    """Six growth steps (2, +1, +3, +1, +5, +2) on one S buffer that starts as NaN: after each, S and w equal the CPU replay of
    the documented order bit for bit; S is within 1e-12 relative of a plain float64 sum over every pair so far (each pair
    added once, none dropped across steps); w is the fp32 rounding of S / (N - 1)."""
    seq = [2, 1, 3, 1, 5, 2]
    nf = sum(seq)
    rng = np.random.default_rng(P * 10 + squared)
    S = torch.full((nf * P,), float("nan"), dtype=torch.float64, device="cuda")
    every = np.full((nf, nf * P), np.nan)                 # value of (partner image j, row R) for every pair so far
    S_prev = np.zeros(0)
    n_old = 0
    for m in seq:
        N = n_old + m
        rowv, colv = grow_tables(n_old, N, P, rng)
        w = _accumulate(rowv, colv, squared, n_old, N, P, S)
        S_want, w_want = accumulate_replay(rowv, colv, squared, n_old, N, P, S_prev)
        got_S = S[:N * P].cpu()
        assert torch.equal(got_S, torch.from_numpy(S_want))                   # bit for bit
        assert torch.equal(w.cpu(), torch.from_numpy(w_want))
        assert torch.equal(w.cpu(), (got_S / (N - 1)).float())
        V = new_pair_values(rowv, colv, squared, n_old, N, P)
        new = ~np.isnan(V)
        blk = every[:N, :N * P]
        assert np.isnan(blk[new]).all()                   # no pair arrives twice
        blk[new] = V[new]
        own = np.repeat(np.eye(N, dtype=bool), P, axis=1)
        assert not np.isnan(blk[~own]).any() and np.isnan(blk[own]).all()
        straight = np.nansum(blk[::-1], axis=0)           # any order
        assert (np.abs(got_S.numpy() - straight) <= 1e-12 * straight).all()
        S_prev, n_old = S_want, N


def test_accumulate_grow_single_image():
    """nb_img = 1, n_old = 0 (one image, no partner): S = 0 and w = NaN, as the header states."""
    P = 40
    S = torch.full((P,), float("nan"), dtype=torch.float64, device="cuda")
    nan = np.full((1, P), np.nan, dtype=np.float32)
    w = _accumulate(nan, nan, 1, 0, 1, P, S)
    assert (S.cpu() == 0).all() and torch.isnan(w).all()


# ----------------------------------------------------------------------------------------------- f. GrowingCategory
SMALL = dict(layers=[(96, 12, 12, True), (96, 12, 12, True)], Dp=256, D=512)      # P = 144
CONFIG2 = dict(layers=[(768, 28, 28, True), (768, 28, 28, True)], Dp=2048, D=4096)  # P = 784 (bench config 2)


def _features(cfg, n, seed):
    feats, _ = synth.planted_features(n, cfg["layers"], n_classes=3, seed=seed)
    return [f.cuda() for f in feats]


def _mean_other_images(dmin: torch.Tensor, n: int, P: int) -> torch.Tensor:
    """w64[R] = mean over j != i(R), j < n of dmin[j, R] for the rows of the first n images."""
    d = dmin[:n, :n * P].clone()
    own = torch.eye(n, dtype=torch.bool).repeat_interleave(P, dim=1)
    d[own] = 0.0
    return d.sum(dim=0) / (n - 1)


@pytest.mark.parametrize("precision", ["f16r", "bf16r"])
def test_growing_category_refined_config2_width_vs_fp64(precision):
    """f16r and bf16r at P = 784, D = 4096 over 6, +1, +5 images: tau = 0 arg-max positions equal run_path's, and every w lies in
    [w64 (1 - 2e-5) - 1e-5, w64 (1 + 2e-3) + 1e-5], w64[R] = mean over j != i(R) of min_c |Z[R] - hi[j, c]| in float64: the
    dot-form refine tolerance below, the arg-min acceptance above."""
    seq, taus, cfg = [6, 1, 5], [0.0, 1.0], CONFIG2
    feats = _features(cfg, sum(seq), seed=11)
    g = pipeline.GrowingCategory(3, 1, cfg["Dp"], cfg["D"], taus, precision=precision)
    n, ws = 0, []
    for m in seq:
        res = g.add([f[n:n + m] for f in feats])
        n += m
        ref = pipeline.run_path([f[:n] for f in feats], 3, 1, cfg["Dp"], cfg["D"], "unsupervised", taus, precision=precision)
        torch.cuda.synchronize()
        assert torch.equal(res.alpha64[0].argmax(dim=-1), ref.alpha64[0].argmax(dim=-1))
        ws.append(res.w.reshape(-1).double().cpu())
        del ref
    P = g.P
    Z = g._images.Z[:n * P].cpu()
    hi = g._images.hi[:n * P].double().cpu()
    dmin, _ = image_min(Z, hi, P)                         # [n, n*P]: rows of the earlier images are unchanged by later adds
    k = 0
    for m, w in zip(seq, ws):
        k += m
        w64 = _mean_other_images(dmin, k, P)
        assert (w >= w64 * (1 - 2e-5) - 1e-5).all(), (w64 - w).max().item()   # dot-form refine
        assert (w <= w64 * (1 + 2e-3) + 1e-5).all(), (w - w64).max().item()   # + a near-tie arg-min


def test_growing_category_long_f16_sequence_vs_fp64():
    """2, then +1 eleven times (12 growth steps, old rows carried across all of them): after every step w is within 5e-4
    relative of the float64 mean over the other images of the per-image minima of the stored hi rows."""
    cfg = SMALL
    feats = _features(cfg, 13, seed=12)
    g = pipeline.GrowingCategory(3, 1, cfg["Dp"], cfg["D"], [1.0], precision="f16")
    n = 0
    for m in [2] + [1] * 11:
        res = g.add([f[n:n + m] for f in feats])
        n += m
        P = g.P
        op = g._images.hi[:n * P].double().cpu()
        dmin, _ = image_min(op, op, P)
        check_rel(res.w.reshape(-1).cpu(), _mean_other_images(dmin, n, P), 5e-4, "w after %d images" % n)   # one pass
