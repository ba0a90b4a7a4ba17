"""Feature maps -> (Z, w, alpha, X, Dmat) on one B200, and its query-sharded multi-GPU form.

This is the device-resident replacement of the body of make_category_data
(reference: Anomaly-Clustering/examples/main.py:266-296) from the hooked backbone features on:

    Z      = AnomalyClusteringCore.embed(...)                      main.py:266-267
    alpha  = Matrix_Alpha_Unsupervised / _Supervised / average     main.py:281-291
    X      = bmm(alpha, Z)                                         main.py:294-296
    Dmat   = pairwise Euclid on X (Ward's input)                   test.py:193-195

Nothing bounces through the host (the reference copies every patch row to numpy and back,
patchcore.py:358-361 + main.py:267) and one min-distance pass serves every tau.
"""
from __future__ import annotations

import functools
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import ops

# Unsupervised self-bank runs multiply every unordered image pair once (ac_min_dist_sym); set to
# False to force the straightforward all-pairs kernel (bench.py --no-symmetry, A/B tests).
SYMMETRIC = True

# bench.py sets this to a list to collect (tag, cuda event) marks at stage boundaries
PROFILE = None


def _mark(tag: str) -> None:
    if PROFILE is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        PROFILE.append((tag, ev))


# taus below this go to the refined mode under precision="auto" (DESIGN.md section 5: one fp16 pass keeps alpha inside
# 1e-3 with a 2x margin from tau = 1 on, also at real-data patch norms; tau = 0 is the arg-max and needs exact w too)
AUTO_REFINE_BELOW_TAU = 1.0


def resolve_precision(precision: str, taus: Sequence[float]) -> str:
    """'auto' -> the cheapest mode that keeps alpha inside the 1e-3 max-abs tolerance with a 2x margin (measured table in
    DESIGN.md section 5): one fp16 tensor-core pass when every tau >= 1; otherwise 'f16r' = the same pass recording the
    arg-min + an exact fp32 re-evaluation of the selected pairs (ac_refine_min_dist, ~1.4x the one-pass cost)."""
    if precision != "auto":
        return precision
    small = [t for t in taus if abs(float(t)) < AUTO_REFINE_BELOW_TAU]
    return "f16r" if small else "f16"


@functools.lru_cache(maxsize=64)
def _fusable(n_layers: int, pretrain_dim: int, target_dim: int) -> bool:
    return ops.aggregator_fusable(n_layers, pretrain_dim, target_dim)


_OPERAND_OF = {"f16": ("f16", False), "bf16": ("bf16", False), "f16x3": ("f16", True), "bf16x3": ("bf16", True), "f32": (None, False),
               "f16r": ("f16", False), "bf16r": ("bf16", False)}
REFINED = ("f16r", "bf16r")


@dataclass
class PatchSet:
    """Embedded images: fp32 Z plus the tensor-core operands and their squared norms."""

    n_img: int
    P: int
    D: int
    grid: Tuple[int, int]
    Z: Optional[torch.Tensor] = None      # [n_img*P, D] fp32
    hi: Optional[torch.Tensor] = None     # [n_img*P, D] f16 | bf16
    lo: Optional[torch.Tensor] = None
    n2: Optional[torch.Tensor] = None     # [n_img*P] fp32 squared norms of the operand (hi [+ lo])


@dataclass
class PathResult:
    Z: Optional[torch.Tensor]             # [N, P, D] fp32 (None when run with keep_z=False)
    w: Optional[torch.Tensor]             # [N, P] fp32 (None in 'average' mode)
    alpha64: torch.Tensor                 # [T, N, P] float64  (reference dtype, utils.py:246)
    alpha32: torch.Tensor                 # [T, N, P] float32  (main.py:294 `.float()`)
    X: torch.Tensor                       # [T, N, D] fp32
    Dmat: torch.Tensor                    # [T, N, N] fp32
    taus: List[float] = field(default_factory=list)
    grid: Tuple[int, int] = (0, 0)


def embed_images(
    features: Sequence[torch.Tensor],
    patchsize: int,
    stride: int,
    pretrain_dim: int,
    target_dim: int,
    precision: str = "f16",
    want_z: bool = True,
    layernorm: bool = True,
    batch: Optional[int] = None,
    out=None,
) -> PatchSet:
    """Stage 1 for a set of images in one C-ABI call (ac_embed_ex: Z and / or the tensor-core operands, and the operands'
    squared norms); `batch` only caps the images per call.  `out` = (hi, lo | None, n2) preallocated operand buffers (the
    sharded path hands in its slice of the symmetric bank so that no staging copy is needed)."""
    operand, want_lo = _OPERAND_OF[precision]
    views = [ops.feature_view(f) for f in features]
    N = views[0].shape[0]
    _mark("embed_begin")
    h, w = ops.patch_grid(views[0].shape[2], views[0].shape[3], patchsize, stride)
    P = h * w
    dev = views[0].device
    # operand-only output needs Aggregator windows that stay inside one layer; otherwise Z is produced (and dropped below)
    need_z = want_z or operand is None or not _fusable(len(views), pretrain_dim, target_dim)
    Z = torch.empty(N * P, target_dim, dtype=torch.float32, device=dev) if need_z else None
    hi = lo = n2 = None
    if operand is not None:
        tdt = torch.float16 if operand == "f16" else torch.bfloat16
        if out is not None:
            hi, lo, n2 = out
            assert hi.shape == (N * P, target_dim) and hi.dtype == tdt and hi.is_contiguous() and n2.shape == (N * P,)
            assert (lo is not None) == want_lo
        else:
            hi = torch.empty(N * P, target_dim, dtype=tdt, device=dev)
            lo = torch.empty(N * P, target_dim, dtype=tdt, device=dev) if want_lo else None
            n2 = torch.empty(N * P, dtype=torch.float32, device=dev)
    step = N if not batch else batch
    for b0 in range(0, N, step):
        b1 = min(N, b0 + step)
        sl = slice(b0 * P, b1 * P)
        ops.embed(
            [v[b0:b1] for v in views], patchsize, stride, pretrain_dim, target_dim, layernorm=layernorm,
            want_z=need_z, operand=operand, want_lo=want_lo,
            out_z=None if Z is None else Z[sl], out_hi=None if hi is None else hi[sl], out_lo=None if lo is None else lo[sl],
            out_n2=None if n2 is None else n2[sl],
        )
    _mark("embed_end")
    if not (want_z or operand is None):
        Z = None
    return PatchSet(n_img=N, P=P, D=target_dim, grid=(h, w), Z=Z, hi=hi, lo=lo, n2=n2)


# element range inside which an arbitrary fp32 embedding may be rounded to fp16 operands: fp16 overflows at 65 504 and
# loses relative precision below its normal range (6e-5); LayerNorm'd embeddings of this path are O(1)
F16_OPERAND_RANGE = (2.0 ** -7, 2.0 ** 14)


def guard_operand_range(precision: str, *tensors: torch.Tensor) -> str:
    """Precision mode that is safe for embeddings that did NOT come out of this package's embed stage (the mirror
    Matrix_Alpha_* / Weight_Distance_* accept any fp32 Z, like the reference's torch.cdist, utils.py:226).  Non-finite
    values are refused; if the largest magnitude lies outside F16_OPERAND_RANGE the fp16 modes are replaced by the exact
    fp32 kernel (slow, correct) with a warning instead of silently overflowing / flushing the operands."""
    if precision == "f32":
        return precision
    fp16_mode = precision.startswith("f16")
    lo, hi = F16_OPERAND_RANGE
    for t in tensors:
        if t is None or not t.numel():
            continue
        amax = float(t.detach().abs().amax())
        if amax != amax or amax == float("inf"):
            raise ValueError("embedding contains non-finite values")
        if fp16_mode and amax > 0 and not (lo <= amax <= hi):
            import warnings

            warnings.warn("embedding magnitude %.3g is outside the fp16 operand range [%.3g, %.3g]: using the exact fp32 distance kernel "
                          "(precision='f32'); rescale Z to O(1) for the tensor-core path" % (amax, lo, hi), RuntimeWarning, stacklevel=3)
            return "f32"
    return precision


def patchset_from_Z(Z: torch.Tensor, precision: str = "f16") -> PatchSet:
    """Wrap an existing [N,P,D] fp32 embedding (e.g. the reference's `Z`) for the distance stage."""
    N, P, D = Z.shape
    Zf = Z.reshape(N * P, D).contiguous().float()
    operand, want_lo = _OPERAND_OF[precision]
    ps = PatchSet(n_img=N, P=P, D=D, grid=(0, 0), Z=Zf)
    if operand is not None:
        ps.hi, ps.lo = ops.split_operand(Zf, operand, want_lo)
        ps.n2 = ops.row_norms(ps.hi, ps.lo)
    return ps


def min_distance_weights(
    q: PatchSet,
    bank: PatchSet,
    mode: str,
    precision: str = "f16",
    q_self: Optional[torch.Tensor] = None,
    return_dmin: bool = False,
    groups: Optional[torch.Tensor] = None,
    bank_ready: Optional[torch.Tensor] = None,
    bank_first: int = 0,
    bank_landed=None,
):
    """Stage 2: w [Nq, P].  mode 'unsupervised' = mean over bank images != self (utils.py:222-227),
    'supervised' = min over bank images (utils.py:230-237).  q_self[i] = bank index of query image i.
    groups (ops.make_groups): the images are several categories back to back, each its own bank (symmetric form only).
    bank_ready / bank_first / bank_landed (sharded supervised runs): arrival flags of a bank whose remote shards are still being
    pulled, the first resident bank image, and a callable that orders the current stream after all pulls (called before the
    refine pass, which gathers from the whole bank)."""
    refined = precision in REFINED
    if (mode == "unsupervised" and SYMMETRIC and q is bank and precision != "f32" and q.P >= 32 and not return_dmin
            and q_self is None):
        _mark("mindist_begin")
        if refined:
            rowmin, rowarg, colkey = ops.min_dist_sym_arg(q.hi, q.lo, q.n2, 0, q.hi, q.lo, q.n2, q.n_img, q.P, precision, groups=groups)
        else:
            rowmin, colmin = ops.min_dist_sym(q.hi, q.lo, q.n2, 0, q.hi, q.lo, q.n2, q.n_img, q.P, precision, groups=groups)
        _mark("mindist_end")
        if not refined:
            return ops.reduce_weights_sym(rowmin, colmin, q.P, 0, groups=groups).reshape(q.n_img, q.P)
        _mark("refine_begin")
        dex = ops.refine_min_dist(q.Z, q.hi, q.lo, q.hi, q.lo, q.n_img, q.P, rowarg, colkey=colkey, q_img0=0, groups=groups, Bn2=q.n2)
        _mark("refine_end")
        own = torch.arange(q.n_img, dtype=torch.int32, device=dex.device)
        return ops.reduce_weights(dex, q.P, own, "mean", groups=groups).reshape(q.n_img, q.P)
    if groups is not None:
        raise ValueError("per-category groups need the symmetric unsupervised form (P >= 32, tensor-core precision)")
    _mark("mindist_begin")
    if precision == "f32":
        dmin = ops.min_dist(q.Z, None, None, bank.Z, None, None, bank.n_img, bank.P, "f32")
    elif refined:
        dmin, arg = ops.min_dist_arg(q.hi, q.lo, q.n2, bank.hi, bank.lo, bank.n2, bank.n_img, bank.P, precision, ready=bank_ready,
                                     first_image=bank_first)
    else:
        dmin = ops.min_dist(q.hi, q.lo, q.n2, bank.hi, bank.lo, bank.n2, bank.n_img, bank.P, precision, ready=bank_ready,
                            first_image=bank_first)
    _mark("mindist_end")
    if bank_landed is not None:
        bank_landed()
    if refined:
        if mode == "unsupervised" and q_self is None:
            q_self = torch.arange(q.n_img, dtype=torch.int32, device=dmin.device)
        _mark("refine_begin")
        dmin = ops.refine_min_dist(q.Z, q.hi, q.lo, bank.hi, bank.lo, bank.n_img, bank.P, arg,
                                   q_self=q_self if mode == "unsupervised" else None, Pq=q.P, Bn2=bank.n2)
        _mark("refine_end")
    if mode == "unsupervised":
        if q_self is None:
            q_self = torch.arange(q.n_img, dtype=torch.int32, device=dmin.device)
        w = ops.reduce_weights(dmin, q.P, q_self, "mean")
    elif mode == "supervised":
        w = ops.reduce_weights(dmin, q.P, None, "min")
    else:
        raise ValueError(mode)
    w = w.reshape(q.n_img, q.P)
    return (w, dmin) if return_dmin else w


def alpha_X_dist(ps: PatchSet, w: Optional[torch.Tensor], taus: Sequence[float], features=None, embed_args=None, want_dmat=True):
    """Stage 3 for every tau from one w.  w=None -> 'average' mode (main.py:290-291).
    When the PatchSet carries no fp32 Z, X is computed straight from `features` (ac_weighted_embed_from_features)."""
    N, P, D = ps.n_img, ps.P, ps.D
    dev = (ps.Z if ps.Z is not None else ps.hi).device
    if w is None:
        a32 = torch.full((1, N, P), 1.0 / P, dtype=torch.float32, device=dev)
        a64 = a32.double()
        taus = [float("nan")]
    else:
        a64, a32 = ops.alpha(w, taus)
    if ps.Z is not None:
        Z3 = ps.Z.reshape(N, P, D)
        X = ops.weighted_embed_multi(a32, Z3)                    # [T, N, D], Z read once for all taus
    else:
        patchsize, stride, Dp, layernorm = embed_args
        X = torch.stack([ops.weighted_embed_from_features(features, a32[t], patchsize, stride, Dp, D, layernorm=layernorm)
                         for t in range(a32.shape[0])])
    Dm = torch.stack([ops.pairwise_l2(X[t]) for t in range(a32.shape[0])]) if want_dmat else None
    return a64, a32, X, Dm


def z_free_supported(features, patchsize, stride, pretrain_dim, target_dim, precision) -> bool:
    """Shapes covered by ac_weighted_embed_from_features (see include/ac_b200.h)."""
    if precision == "f32" or patchsize != 3 or stride != 1:
        return False
    views = [ops.feature_view(f) for f in features]
    if any(v.shape[2:] != views[0].shape[2:] for v in views):
        return False
    L = len(views)
    if (L * pretrain_dim) % target_dim != 0 or pretrain_dim % ((L * pretrain_dim) // target_dim) != 0:
        return False
    # the alpha map of an image with its one-position zero halo is staged in shared memory: at most 200 KB of fp32
    h, w = ops.patch_grid(views[0].shape[2], views[0].shape[3], patchsize, stride)
    return (h + 2) * (w + 2) * 4 <= 200 * 1024


def run_path(
    features: Sequence[torch.Tensor],
    patchsize: int = 3,
    stride: int = 1,
    pretrain_dim: int = 1024,
    target_dim: int = 1024,
    mode: str = "unsupervised",
    taus: Sequence[float] = (1.0,),
    bank_features: Optional[Sequence[torch.Tensor]] = None,
    precision: str = "auto",
    layernorm: bool = True,
    keep_z: bool = True,
) -> PathResult:
    """Single-GPU hot path: hooked features (device tensors) -> PathResult (device tensors).
    keep_z=False never materialises the fp32 Z (1.3 GB at config 2): the embed kernel writes only the
    tensor-core operands and X comes straight from the feature maps; falls back to keep_z=True for shapes the
    Z-free form does not cover (resampled layers, patch size != 3, fp32 precision)."""
    precision = resolve_precision(precision, taus)
    if not keep_z and not z_free_supported(features, patchsize, stride, pretrain_dim, target_dim, precision):
        keep_z = True
    if precision in REFINED and mode != "average":
        keep_z = True      # the exact re-evaluation takes the QUERY rows from fp32 Z (their rounding would not average out)
    q = embed_images(features, patchsize, stride, pretrain_dim, target_dim, precision, want_z=keep_z, layernorm=layernorm)
    w = None
    if mode == "unsupervised":
        w = min_distance_weights(q, q, "unsupervised", precision)
    elif mode == "supervised":
        if bank_features is None:
            raise ValueError("supervised mode needs bank_features (the normal training images)")
        bank = embed_images(bank_features, patchsize, stride, pretrain_dim, target_dim, precision, want_z=False,
                            layernorm=layernorm)
        w = min_distance_weights(q, bank, "supervised", precision)
    elif mode != "average":
        raise ValueError("mode must be unsupervised | supervised | average")
    a64, a32, X, Dm = alpha_X_dist(q, w, list(taus), features, (patchsize, stride, pretrain_dim, layernorm))
    return PathResult(Z=None if q.Z is None else q.Z.reshape(q.n_img, q.P, q.D), w=w, alpha64=a64, alpha32=a32, X=X, Dmat=Dm,
                      taus=list(taus), grid=q.grid)


def run_categories(
    features: Sequence[torch.Tensor],
    sizes: Sequence[int],
    patchsize: int = 3,
    stride: int = 1,
    pretrain_dim: int = 1024,
    target_dim: int = 1024,
    taus: Sequence[float] = (1.0,),
    precision: str = "auto",
    keep_z: bool = True,
    layernorm: bool = True,
) -> List[PathResult]:
    """Several independent categories (the reference's own semantics: one make_category_data per category, each with
    its own bank -- examples/main.py:353) from ONE batch of hooked features and ONE launch sequence: `features` hold the
    images of all categories back to back, `sizes[c]` images each.  The embed, the tensor-core pass (image pairs only
    inside a category: ac_min_dist_sym_ex with a category table), the reductions, alpha and X run once for all
    categories; only the small per-category distance matrices are separate launches.  Returns one PathResult per category
    (views into the shared tensors).  Shapes the batched form does not cover run category by category."""
    precision = resolve_precision(precision, taus)
    sizes = [int(n) for n in sizes]
    views = [ops.feature_view(f) for f in features]
    N = views[0].shape[0]
    if sum(sizes) != N:
        raise ValueError("sizes sum to %d but the features hold %d images" % (sum(sizes), N))
    h, w_ = ops.patch_grid(views[0].shape[2], views[0].shape[3], patchsize, stride)
    batched = SYMMETRIC and precision != "f32" and h * w_ >= 32 and min(sizes) >= 2
    if not batched:
        out, start = [], 0
        for n in sizes:
            out.append(run_path([f[start:start + n] for f in features], patchsize, stride, pretrain_dim, target_dim, "unsupervised",
                                taus, precision=precision, keep_z=keep_z, layernorm=layernorm))
            start += n
        return out
    if not keep_z and not z_free_supported(features, patchsize, stride, pretrain_dim, target_dim, precision):
        keep_z = True
    if precision in REFINED:
        keep_z = True
    q = embed_images(features, patchsize, stride, pretrain_dim, target_dim, precision, want_z=keep_z, layernorm=layernorm)
    groups = ops.make_groups(sizes, q.hi.device)
    w = min_distance_weights(q, q, "unsupervised", precision, groups=groups)
    a64, a32, X, _ = alpha_X_dist(q, w, list(taus), features, (patchsize, stride, pretrain_dim, layernorm), want_dmat=False)
    out, start = [], 0
    Z3 = None if q.Z is None else q.Z.reshape(q.n_img, q.P, q.D)
    for n in sizes:
        sl = slice(start, start + n)
        Dm = torch.stack([ops.pairwise_l2(X[t][sl]) for t in range(len(taus))])
        out.append(PathResult(Z=None if Z3 is None else Z3[sl], w=w[sl], alpha64=a64[:, sl], alpha32=a32[:, sl], X=X[:, sl], Dmat=Dm,
                              taus=list(taus), grid=q.grid))
        start += n
    return out


def _growth_precision(precision: str, taus: Sequence[float]) -> str:
    """The precision of a growing category, resolved once from its taus; growth multiplies on the tensor cores only."""
    precision = resolve_precision(precision, taus)
    if precision not in _OPERAND_OF or precision == "f32":
        raise ValueError("growth needs a tensor-core precision (f16, bf16, f16x3, bf16x3, f16r, bf16r), got %r" % precision)
    return precision


def _feature_signature(features, first: Optional[tuple]) -> tuple:
    """(layer count, per-layer shape without the image axis, dtype) of one call's hooked features; every later call of a
    growing category must repeat the first call's."""
    sig = (len(features), tuple(tuple(f.shape[1:]) for f in features), features[0].dtype)
    if first is not None and sig != first:
        raise ValueError("features of shape / dtype %s differ from the first add's %s" % (sig, first))
    return sig


def _image_count(features) -> int:
    M = features[0].shape[0]
    if M < 1 or any(f.shape[0] != M for f in features):
        raise ValueError("every layer must hold the same, non-zero number of images")
    return M


def _regrow(old: Optional[torch.Tensor], n_keep: int, shape, dtype, dev, dim: int = 0) -> torch.Tensor:
    """A new buffer of `shape` holding the first n_keep entries of `old` along `dim`, copied on the current stream."""
    t = torch.empty(tuple(shape), dtype=dtype, device=dev)
    if old is not None and n_keep:
        t.narrow(dim, 0, n_keep).copy_(old.narrow(dim, 0, n_keep))
    return t


class _GrowingImages:
    """Embedded images that gain more over time: the tensor-core operands and their squared norms, plus the fp32 Z (keep_z)
    or the hooked feature maps as they came in (keep_maps: the source of the Z-free X).  Buffers hold `capacity` images
    (0: the first addition) and double when full; the rows of the images so far are copied over on the current stream."""

    def __init__(self, precision: str, P: int, D: int, keep_z: bool, keep_maps: bool, capacity: int):
        self.precision, self.P, self.D, self.keep_z, self.keep_maps = precision, P, D, keep_z, keep_maps
        self.capacity = capacity
        self.n_img = 0
        self.hi = self.lo = self.n2 = self.Z = None
        self.maps: List[torch.Tensor] = []

    def _reserve(self, n: int, features) -> None:
        if self.hi is not None and n <= self.capacity:
            return
        cap = max(n, 2 * self.capacity) if self.hi is not None else max(n, self.capacity)
        P, D, rows, dev = self.P, self.D, self.n_img * self.P, features[0].device
        operand, want_lo = _OPERAND_OF[self.precision]
        tdt = torch.float16 if operand == "f16" else torch.bfloat16
        self.hi = _regrow(self.hi, rows, (cap * P, D), tdt, dev)
        self.lo = _regrow(self.lo, rows, (cap * P, D), tdt, dev) if want_lo else None
        self.n2 = _regrow(self.n2, rows, (cap * P,), torch.float32, dev)
        if self.keep_z:
            self.Z = _regrow(self.Z, rows, (cap * P, D), torch.float32, dev)
        if self.keep_maps:
            olds = self.maps or [None] * len(features)
            self.maps = [_regrow(old, self.n_img, (cap,) + tuple(f.shape[1:]), f.dtype, dev) for old, f in zip(olds, features)]
        self.capacity = cap

    def append(self, features, patchsize: int, stride: int, pretrain_dim: int, layernorm: bool) -> None:
        """Embeds the new images (one ac_embed_dt call) into the rows after the images so far."""
        n_old, N, P = self.n_img, self.n_img + features[0].shape[0], self.P
        self._reserve(N, features)
        rows = slice(n_old * P, N * P)
        operand, want_lo = _OPERAND_OF[self.precision]
        need_z = self.keep_z or not _fusable(len(features), pretrain_dim, self.D)
        _mark("embed_begin")
        ops.embed(features, patchsize, stride, pretrain_dim, self.D, layernorm=layernorm, want_z=need_z, operand=operand,
                  want_lo=want_lo, out_z=self.Z[rows] if self.keep_z else None, out_hi=self.hi[rows],
                  out_lo=None if self.lo is None else self.lo[rows], out_n2=self.n2[rows])
        for buf, f in zip(self.maps, features):
            buf[n_old:N].copy_(f)
        _mark("embed_end")
        self.n_img = N

    def patchset(self, i0: int, i1: int, grid) -> PatchSet:
        """Images [i0, i1) as views into the buffers."""
        rows = slice(i0 * self.P, i1 * self.P)
        return PatchSet(n_img=i1 - i0, P=self.P, D=self.D, grid=grid, Z=self.Z[rows] if self.keep_z else None, hi=self.hi[rows],
                        lo=None if self.lo is None else self.lo[rows], n2=self.n2[rows])


class GrowingCategory:
    """One unsupervised category that gains images over time (an inspection line collecting defective images), clustered
    after every addition without recomputing the image pairs it already has.

    w[i, p] is a mean over the other images of one per-image minimum each (utils.py:222-227), so when M images join N_old
    the old pairs keep their minima: `add` runs the distance pass over the M*N_old + M*(M-1)/2 new pairs only
    (ac_min_dist_sym_grow), adds them to fp64 running sums kept per patch row (ac_accumulate_weights_grow) and runs stage 3 for
    every image so far, which does change everywhere because every w does.  The result of each `add` is what `run_path`
    returns for all images so far, up to the order of the sums (DESIGN.md section 5c).

    Device state: the tensor-core operands and their norms, the running sums, and the source of X: the fp32 Z when keep_z or
    a refined precision (whose exact re-evaluation reads it) is in use, else the hooked feature maps as they came in (fp32,
    bf16 or fp16), from which ac_weighted_embed_from_features computes X exactly as `run_path` does.  Buffers hold `capacity`
    images (default: the first addition) and double when full."""

    def __init__(self, patchsize: int, stride: int, pretrain_dim: int, target_dim: int, taus: Sequence[float],
                 precision: str = "auto", keep_z: bool = False, layernorm: bool = True, capacity: Optional[int] = None):
        self.patchsize, self.stride, self.pretrain_dim, self.target_dim = patchsize, stride, pretrain_dim, target_dim
        self.taus = [float(t) for t in taus]
        self.precision = _growth_precision(precision, self.taus)
        self.refined = self.precision in REFINED
        self.keep_z = keep_z or self.refined
        self.layernorm = layernorm
        self._capacity = int(capacity) if capacity else 0
        self._sig = None
        self.P = 0
        self.grid = (0, 0)
        self._images: Optional[_GrowingImages] = None
        self._S = None

    @property
    def n_img(self) -> int:
        return self._images.n_img if self._images is not None else 0

    @property
    def capacity(self) -> int:
        return self._images.capacity if self._images is not None else self._capacity

    def add(self, features: Sequence[torch.Tensor]) -> PathResult:
        """Embeds the new images (hooked features, device tensors of the layout run_path takes), multiplies only the pairs they
        bring and returns the PathResult of all images so far."""
        features = list(features)
        sig = _feature_signature(features, self._sig)
        if self._sig is None:
            if features[0].shape[0] < 2:
                raise ValueError("the first add needs at least 2 images")
            if not self.keep_z and not z_free_supported(features, self.patchsize, self.stride, self.pretrain_dim, self.target_dim,
                                                        self.precision):
                self.keep_z = True
            v0 = ops.feature_view(features[0])
            self.grid = ops.patch_grid(v0.shape[2], v0.shape[3], self.patchsize, self.stride)
            self.P = self.grid[0] * self.grid[1]
            if self.P < 32:
                raise ValueError("growth runs the symmetric distance form, which needs at least 32 patches per image")
            self._sig = sig
        M = _image_count(features)
        n_old, N, P, D = self.n_img, self.n_img + M, self.P, self.target_dim
        if self._images is None:
            self._images = _GrowingImages(self.precision, P, D, self.keep_z, not self.keep_z, self._capacity)
        images = self._images
        images.append(features, self.patchsize, self.stride, self.pretrain_dim, self.layernorm)
        if self._S is None or self._S.numel() < images.capacity * P:
            self._S = _regrow(self._S, n_old * P, (images.capacity * P,), torch.float64, features[0].device)
        ps = images.patchset(0, N, self.grid)
        hi, lo, n2, Z = ps.hi, ps.lo, ps.n2, ps.Z
        _mark("mindist_begin")
        if self.refined:
            _, rowarg, colkey = ops.min_dist_sym_grow(hi, lo, n2, n_old, N, P, self.precision, arg=True)
            _mark("mindist_end")
            _mark("refine_begin")
            rowv, colv = ops.refine_min_dist_grow(Z, hi, lo, n2, n_old, N, P, rowarg, colkey)
            _mark("refine_end")
        else:
            rowv, colv = ops.min_dist_sym_grow(hi, lo, n2, n_old, N, P, self.precision)
            _mark("mindist_end")
        w = ops.accumulate_weights_grow(rowv, colv, not self.refined, n_old, N, P, self._S).reshape(N, P)
        feats = None if self.keep_z else [buf[:N] for buf in images.maps]
        a64, a32, X, Dm = alpha_X_dist(ps, w, self.taus, feats, (self.patchsize, self.stride, self.pretrain_dim, self.layernorm))
        return PathResult(Z=None if Z is None else Z.reshape(N, P, D), w=w, alpha64=a64, alpha32=a32, X=X, Dmat=Dm,
                          taus=list(self.taus), grid=self.grid)


# query rows per block of the refine kernel (kRQ in csrc/refine.cu).  Unless D is a multiple of 256, the lanes that sum a query
# row's |q|^2 there depend on the row's place in its block, so a refine launch over new query rows starts on a multiple of it,
# as run_path's launch from row 0 does.
_REFINE_QUERY_ROWS = 4


class GrowingSupervisedCategory:
    """One supervised category whose query images and normal bank both grow over time (an inspection line clustering its
    defects against known-good images), clustered after every call without recomputing the image pairs it already has.

    w[r] of Weight_Distance_Supervised (utils.py:230-237) is a minimum over bank images of one per-(row, bank image) minimum
    each, and a min of fp32 values does not depend on the order it is taken in.  So `add` runs the new query rows against the
    whole bank and leaves the old queries' w, alpha and X alone; `add_normal` runs every query row against the new bank images
    only and lowers w in place (ac_reduce_weights, AC_REDUCE_MIN_UPDATE), then runs stage 3 for every query.  Each result is
    bit-identical to `run_path(queries so far, mode="supervised", bank_features=normals so far)` (DESIGN.md section 5d).

    Device state: for the queries the tensor-core operands and their norms, w, alpha64 / alpha32 / X per tau and the source of X
    (the fp32 Z when keep_z or a refined precision is in use, else the hooked feature maps as they came in); for the bank the
    operands and norms only.  Buffers hold `capacity` query / `bank_capacity` bank images (default: the first addition) and
    double when full.  Both sides must give the features of the first call's layer count, shapes and dtype."""

    def __init__(self, patchsize: int, stride: int, pretrain_dim: int, target_dim: int, taus: Sequence[float],
                 precision: str = "auto", keep_z: bool = False, layernorm: bool = True, capacity: Optional[int] = None,
                 bank_capacity: Optional[int] = None):
        self.patchsize, self.stride, self.pretrain_dim, self.target_dim = patchsize, stride, pretrain_dim, target_dim
        self.taus = [float(t) for t in taus]
        self.precision = _growth_precision(precision, self.taus)
        self.refined = self.precision in REFINED
        self.keep_z = keep_z or self.refined
        self.layernorm = layernorm
        self._capacity = (int(capacity) if capacity else 0, int(bank_capacity) if bank_capacity else 0)
        self._sig = None
        self.P = 0
        self.grid = (0, 0)
        self._q: Optional[_GrowingImages] = None
        self._bank: Optional[_GrowingImages] = None
        self._w = self._a64 = self._a32 = self._X = None

    @property
    def n_img(self) -> int:
        """Query images so far."""
        return self._q.n_img if self._q is not None else 0

    @property
    def n_normal(self) -> int:
        """Normal (bank) images so far."""
        return self._bank.n_img if self._bank is not None else 0

    def _check(self, features) -> int:
        """Refuses features unlike the first call's (on either side); the first call fixes the patch grid and whether Z is
        kept, as run_path would decide them.  Returns the image count."""
        sig = _feature_signature(features, self._sig)
        M = _image_count(features)
        if self._sig is None:
            if not self.keep_z and not z_free_supported(features, self.patchsize, self.stride, self.pretrain_dim, self.target_dim,
                                                        self.precision):
                self.keep_z = True
            v0 = ops.feature_view(features[0])
            self.grid = ops.patch_grid(v0.shape[2], v0.shape[3], self.patchsize, self.stride)
            self.P = self.grid[0] * self.grid[1]
            self._q = _GrowingImages(self.precision, self.P, self.target_dim, self.keep_z, not self.keep_z, self._capacity[0])
            self._bank = _GrowingImages(self.precision, self.P, self.target_dim, False, False, self._capacity[1])
            self._sig = sig
        return M

    def _nearest(self, r0: int, r1: int, b0: int, b1: int) -> torch.Tensor:
        """dmin [b1 - b0, r1 - r0]: distance of query rows [r0, r1) to their nearest row of each bank image [b0, b1), from one
        all-pairs tensor-core launch and, in f16r / bf16r, the exact fp32 re-evaluation of the selected pairs."""
        q, bank, P = self._q, self._bank, self.P
        rows, brows = slice(r0, r1), slice(b0 * P, b1 * P)
        qhi, qlo, qn2 = q.hi[rows], None if q.lo is None else q.lo[rows], q.n2[rows]
        bhi, blo, bn2 = bank.hi[brows], None if bank.lo is None else bank.lo[brows], bank.n2[brows]
        _mark("mindist_begin")
        if not self.refined:
            dmin = ops.min_dist(qhi, qlo, qn2, bhi, blo, bn2, b1 - b0, P, self.precision)
            _mark("mindist_end")
            return dmin
        dmin, arg = ops.min_dist_arg(qhi, qlo, qn2, bhi, blo, bn2, b1 - b0, P, self.precision)
        _mark("mindist_end")
        _mark("refine_begin")
        dmin = ops.refine_min_dist(q.Z[rows], qhi, qlo, bhi, blo, b1 - b0, P, arg, Pq=P, Bn2=bn2)
        _mark("refine_end")
        return dmin

    def _stage3(self, i0: int, i1: int, features) -> None:
        """alpha and X of query images [i0, i1) from their w, into the state buffers."""
        P = self.P
        w = self._w[i0 * P:i1 * P].reshape(i1 - i0, P)
        a64, a32, X, _ = alpha_X_dist(self._q.patchset(i0, i1, self.grid), w, self.taus, features,
                                      (self.patchsize, self.stride, self.pretrain_dim, self.layernorm), want_dmat=False)
        self._a64[:, i0:i1].copy_(a64)
        self._a32[:, i0:i1].copy_(a32)
        self._X[:, i0:i1].copy_(X)

    def _result(self) -> PathResult:
        """The PathResult of all queries so far, in tensors of its own (later calls do not change it)."""
        N, P, D = self.n_img, self.P, self.target_dim
        own = lambda t: t.clone(memory_format=torch.contiguous_format)
        X = own(self._X[:, :N])
        Dm = torch.stack([ops.pairwise_l2(X[t]) for t in range(len(self.taus))])
        return PathResult(Z=self._q.Z[:N * P].reshape(N, P, D) if self.keep_z else None, w=own(self._w[:N * P]).reshape(N, P),
                          alpha64=own(self._a64[:, :N]), alpha32=own(self._a32[:, :N]), X=X, Dmat=Dm, taus=list(self.taus),
                          grid=self.grid)

    def add_normal(self, features: Sequence[torch.Tensor]) -> Optional[PathResult]:
        """Normal images join the bank: every query row runs against the new bank images only, w is lowered in place and stage 3
        runs for every query.  Returns the PathResult of all queries so far (None while there are none)."""
        features = list(features)
        K = self._check(features)
        k_old, N, P = self.n_normal, self.n_img, self.P
        self._bank.append(features, self.patchsize, self.stride, self.pretrain_dim, self.layernorm)
        if N == 0:
            return None
        dmin = self._nearest(0, N * P, k_old, k_old + K)
        ops.reduce_weights(dmin, P, None, "min_update", out=self._w[:N * P])
        self._stage3(0, N, None if self.keep_z else [buf[:N] for buf in self._q.maps])
        return self._result()

    def add(self, features: Sequence[torch.Tensor]) -> PathResult:
        """Query images join: only their rows run against the bank, and only their alpha and X are computed.  Returns the
        PathResult of all queries so far."""
        features = list(features)
        if self.n_normal == 0:
            raise ValueError("add needs a normal bank: call add_normal first")
        M = self._check(features)
        n_old, N, P, T, D = self.n_img, self.n_img + M, self.P, len(self.taus), self.target_dim
        q = self._q
        q.append(features, self.patchsize, self.stride, self.pretrain_dim, self.layernorm)
        if self._w is None or self._w.numel() < q.capacity * P:
            dev, cap = q.hi.device, q.capacity
            self._w = _regrow(self._w, n_old * P, (cap * P,), torch.float32, dev)
            self._a64 = _regrow(self._a64, n_old, (T, cap, P), torch.float64, dev, dim=1)
            self._a32 = _regrow(self._a32, n_old, (T, cap, P), torch.float32, dev, dim=1)
            self._X = _regrow(self._X, n_old, (T, cap, D), torch.float32, dev, dim=1)
        r0 = n_old * P
        if self.refined:
            r0 -= r0 % _REFINE_QUERY_ROWS     # the rows before n_old * P get the w they already hold
        dmin = self._nearest(r0, N * P, 0, self.n_normal)
        ops.reduce_weights(dmin, P, None, "min", out=self._w[r0:N * P])
        self._stage3(n_old, N, features)
        return self._result()


