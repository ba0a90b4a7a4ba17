"""Torch-tensor wrappers over the C ABI (include/ac_b200.h).  PyTorch is plumbing here: it owns
device memory and streams; every computation happens in libac_b200.so."""
from __future__ import annotations

import ctypes
import math
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import AcLayer, check

_OP_DTYPES = {"f16": (torch.float16, _lib.AC_DT_F16), "bf16": (torch.bfloat16, _lib.AC_DT_BF16)}
_TORCH_TO_AC = {torch.float32: _lib.AC_DT_F32, torch.float16: _lib.AC_DT_F16, torch.bfloat16: _lib.AC_DT_BF16}


def launches() -> int:
    """Kernels launched by libac_b200 so far, counted inside the library (bench.py: gpu_launches)."""
    return int(_lib.load().ac_debug_launches())


def watchdog_code() -> int:
    """Which mbarrier wait of the tensor-core kernel timed out (0 = none); readable after the launch has trapped, i.e. after
    torch reports the sticky CUDA error at the next synchronisation (ac_last_watchdog)."""
    return int(_lib.load().ac_last_watchdog())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise ValueError("libac_b200 operates on CUDA tensors only (no CPU fallback)")


def device_ok(dev: Optional[int] = None) -> bool:
    lib = _lib.load()
    if dev is None:
        dev = torch.cuda.current_device()
    return lib.ac_device_ok(int(dev)) == 0


def feature_view(f: torch.Tensor) -> torch.Tensor:
    """[B,C,H,W] stays; ViT block output [B,1+P,C] becomes a strided [B,C,s,s] VIEW with the CLS
    token skipped (reference: models/patchcore/patchcore.py:377-383) -- no copy is made."""
    if f.dim() == 3:
        B, T, C = f.shape
        s = int(math.sqrt(T - 1))
        if s * s != T - 1:
            raise ValueError("token count minus CLS is not a square: %d" % (T - 1))
        return f[:, 1:, :].unflatten(1, (s, s)).permute(0, 3, 1, 2)
    if f.dim() != 4:
        raise ValueError("feature must be [B,C,H,W] or [B,1+P,C]")
    return f


def patch_grid(H: int, W: int, patchsize: int, stride: int) -> Tuple[int, int]:
    pad = int((patchsize - 1) / 2)
    return ((H + 2 * pad - (patchsize - 1) - 1) // stride + 1, (W + 2 * pad - (patchsize - 1) - 1) // stride + 1)


def aggregator_fusable(n_layers: int, pretrain_dim: int, target_dim: int) -> bool:
    """True when no Aggregator window (adaptive_avg_pool1d of the L*Dp concat to D, common.py:181-183) straddles two layers:
    only then can ac_embed write the tensor-core operands without the fp32 Z (same rule as csrc/embed.cu)."""
    agg_in = n_layers * pretrain_dim
    for t in range(target_dim):
        g0 = (t * agg_in) // target_dim
        g1 = ((t + 1) * agg_in + target_dim - 1) // target_dim
        if g0 // pretrain_dim != (g1 - 1) // pretrain_dim:
            return False
    return True


def make_groups(sizes: Sequence[int], device) -> torch.Tensor:
    """Category table of the _ex entry points: int32 [sum(sizes), 2] = (first image, image count) of the category of every
    image, for categories stored back to back (per-category banks, examples/main.py:353)."""
    key = (tuple(int(n) for n in sizes), str(torch.device(device)))
    t = _GROUPS_CACHE.get(key)
    if t is None:                          # built once per layout: no host-to-device copy inside a step
        rows, start = [], 0
        for n in key[0]:
            rows += [[start, n]] * n
            start += n
        t = torch.tensor(rows, dtype=torch.int32).reshape(-1, 2).contiguous().to(device)
        if len(_GROUPS_CACHE) > 64:
            _GROUPS_CACHE.clear()
        _GROUPS_CACHE[key] = t
    return t


_GROUPS_CACHE = {}


def _groups_ok(groups, nb_img):
    if groups is not None:
        assert groups.dtype == torch.int32 and groups.shape == (nb_img, 2) and groups.is_contiguous() and groups.is_cuda


def embed(
    features: Sequence[torch.Tensor],
    patchsize: int,
    stride: int,
    pretrain_dim: int,
    target_dim: int,
    layernorm: bool = True,
    eps: float = 1e-5,
    want_z: bool = True,
    operand: Optional[str] = None,
    want_lo: bool = False,
    out_z: Optional[torch.Tensor] = None,
    out_hi: Optional[torch.Tensor] = None,
    out_lo: Optional[torch.Tensor] = None,
    out_n2: Optional[torch.Tensor] = None,
):
    """Fused stage 1.  Returns (Z [B*P, D] fp32 | None, Zhi | None, Zlo | None, (h, w)).  out_n2 [B*P] fp32 (needs an
    operand) receives the squared norms of the operand rows (ac_embed_dt).  The maps are float32, float16 or bfloat16, one
    dtype for all layers; 16-bit maps give the same bits as their float32 upcast."""
    view0 = feature_view(features[0])
    B = view0.shape[0]
    h, w = patch_grid(view0.shape[2], view0.shape[3], patchsize, stride)
    rows = B * h * w
    dev = view0.device
    tdt, op_code = _OP_DTYPES[operand] if operand is not None else (None, 0)
    # caller buffers are written as dense [rows, target_dim] arrays: anything else would be written out of bounds
    _out_ok(out_z if want_z else None, "out_z", (rows, target_dim), torch.float32, dev)
    _out_ok(out_hi if operand is not None else None, "out_hi", (rows, target_dim), tdt, dev)
    _out_ok(out_lo if operand is not None and want_lo else None, "out_lo", (rows, target_dim), tdt, dev)
    lib = _lib.load()
    views, arr, feat_dt = _layer_array(features)
    L = len(views)
    Z = hi = lo = None
    if want_z:
        Z = out_z if out_z is not None else torch.empty(rows, target_dim, dtype=torch.float32, device=dev)
    if operand is not None:
        hi = out_hi if out_hi is not None else torch.empty(rows, target_dim, dtype=tdt, device=dev)
        if want_lo:
            lo = out_lo if out_lo is not None else torch.empty(rows, target_dim, dtype=tdt, device=dev)
    ws_bytes = lib.ac_embed_workspace_bytes_dt(arr, L, feat_dt, B, patchsize, stride, pretrain_dim, target_dim)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    if out_n2 is not None:
        assert hi is not None and out_n2.dtype == torch.float32 and out_n2.numel() == rows and out_n2.is_contiguous()
    rc = lib.ac_embed_dt(arr, L, feat_dt, B, patchsize, stride, pretrain_dim, target_dim, int(layernorm), float(eps), _ptr(Z),
                         _ptr(hi), _ptr(lo), op_code, _ptr(out_n2), _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_embed")
    return Z, hi, lo, (h, w)


def _out_ok(t: Optional[torch.Tensor], name: str, shape, dtype, dev) -> None:
    """A caller-provided output buffer of ops.embed: exactly `shape`, `dtype`, on `dev`, contiguous (any storage offset)."""
    if t is None:
        return
    if tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != dev or not t.is_contiguous():
        raise ValueError("%s must be a contiguous %s tensor of shape %s on %s, got %s %s on %s (contiguous: %s)"
                         % (name, dtype, tuple(shape), dev, t.dtype, tuple(t.shape), t.device, t.is_contiguous()))


def patchify(x: torch.Tensor, patchsize: int, stride: int):
    lib = _lib.load()
    _need_cuda(x)
    x = x.contiguous().float()
    B, C, H, W = x.shape
    h, w = patch_grid(H, W, patchsize, stride)
    out = torch.empty(B, h * w, C, patchsize, patchsize, dtype=torch.float32, device=x.device)
    grid = (ctypes.c_int * 2)()
    check(lib.ac_patchify(_ptr(x), B, C, H, W, patchsize, stride, _ptr(out), grid, _stream()), "ac_patchify")
    return out, [int(grid[0]), int(grid[1])]


def adaptive_pool1d(x: torch.Tensor, out_dim: int) -> torch.Tensor:
    lib = _lib.load()
    _need_cuda(x)
    x2 = x.reshape(len(x), -1).contiguous().float()
    out = torch.empty(x2.shape[0], out_dim, dtype=torch.float32, device=x.device)
    check(lib.ac_adaptive_pool1d(_ptr(x2), x2.shape[0], x2.shape[1], out_dim, _ptr(out), _stream()), "ac_adaptive_pool1d")
    return out


def split_operand(x: torch.Tensor, operand: str, want_lo: bool):
    lib = _lib.load()
    _need_cuda(x)
    x = x.contiguous()
    tdt, code = _OP_DTYPES[operand]
    hi = torch.empty(x.shape, dtype=tdt, device=x.device)
    lo = torch.empty(x.shape, dtype=tdt, device=x.device) if want_lo else None
    check(lib.ac_split_operand(_ptr(x), x.numel(), _ptr(hi), _ptr(lo), code, _stream()), "ac_split_operand")
    return hi, lo


def row_norms(A: torch.Tensor, A2: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _need_cuda(A, A2)
    assert A.dim() == 2 and A.is_contiguous()
    out = torch.empty(A.shape[0], dtype=torch.float32, device=A.device)
    check(lib.ac_row_norms(_ptr(A), _ptr(A2), _TORCH_TO_AC[A.dtype], A.shape[0], A.shape[1], _ptr(out), _stream()), "ac_row_norms")
    return out


def min_dist(Qhi, Qlo, Qn2, Bhi, Blo, Bn2, nb_img: int, P: int, precision: str, out: Optional[torch.Tensor] = None,
             ready: Optional[torch.Tensor] = None, first_image: int = 0) -> torch.Tensor:
    """dmin [nb_img, Mq]: per bank image, distance of each query row to its nearest bank row.
    ready / first_image: arrival flags of a bank that is still landing and the bank image the walk starts at (ac_min_dist_ready)."""
    lib = _lib.load()
    _need_cuda(Qhi, Bhi)
    prec = _lib.PRECISIONS[precision]
    Mq, D = Qhi.shape
    assert Bhi.shape == (nb_img * P, D), (Bhi.shape, nb_img, P, D)
    assert Qhi.is_contiguous() and Bhi.is_contiguous()
    dmin = out if out is not None else torch.empty(nb_img, Mq, dtype=torch.float32, device=Qhi.device)
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, nb_img, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=Qhi.device)
    if ready is not None or first_image:
        _ready_ok(ready, nb_img)
        rc = lib.ac_min_dist_ready(_ptr(Qhi), _ptr(Qlo), _ptr(Qn2), Mq, _ptr(Bhi), _ptr(Blo), _ptr(Bn2), nb_img, P, D, prec, _ptr(dmin),
                                   None, _ptr(ready), int(first_image), _ptr(ws), ws_bytes, _stream())
    else:
        rc = lib.ac_min_dist(_ptr(Qhi), _ptr(Qlo), _ptr(Qn2), Mq, _ptr(Bhi), _ptr(Blo), _ptr(Bn2), nb_img, P, D, prec, _ptr(dmin),
                             _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_min_dist")
    return dmin


def _ready_ok(ready: Optional[torch.Tensor], nb_img: int) -> None:
    """bank_ready flags of ac_min_dist_sym_ready: one int32 per bank image on the device, or None (whole bank resident)."""
    if ready is not None:
        assert ready.is_cuda and ready.dtype == torch.int32 and ready.is_contiguous() and ready.numel() == nb_img


def min_dist_sym(Qhi, Qlo, Qn2, q_img0: int, Bhi, Blo, Bn2, nb_img: int, P: int, precision: str,
                 bank_window: Optional[Tuple[int, int]] = None, init: bool = True, out=None, groups: Optional[torch.Tensor] = None,
                 ready: Optional[torch.Tensor] = None):
    """Symmetric self-bank form: (rowmin_d2 [nb_img, Mq], colmin_d2 [Mq/P, nb_img*P]) squared distances.
    bank_window=(begin, count) restricts the launch to a circular range of bank images; pass the previous
    call's result as `out` with init=False to accumulate a second window into the same buffers."""
    lib = _lib.load()
    _need_cuda(Qhi, Bhi)
    prec = _lib.PRECISIONS[precision]
    Mq, D = Qhi.shape
    assert Bhi.shape == (nb_img * P, D) and Qhi.is_contiguous() and Bhi.is_contiguous()
    if out is None:
        rowmin = torch.empty(nb_img, Mq, dtype=torch.float32, device=Qhi.device)
        colmin = torch.empty(Mq // P, nb_img * P, dtype=torch.float32, device=Qhi.device)
    else:
        rowmin, colmin = out
    begin, count = bank_window if bank_window is not None else (0, nb_img)
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, nb_img, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=Qhi.device)
    _groups_ok(groups, nb_img)
    _ready_ok(ready, nb_img)
    rc = lib.ac_min_dist_sym_ready(_ptr(Qhi), _ptr(Qlo), _ptr(Qn2), Mq, q_img0, _ptr(Bhi), _ptr(Blo), _ptr(Bn2), nb_img, P, D, prec,
                                   int(begin), int(count), int(bool(init)), _ptr(rowmin), _ptr(colmin), None, None, _ptr(groups),
                                   _ptr(ready), _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_min_dist_sym")
    return rowmin, colmin


def min_dist_arg(Qhi, Qlo, Qn2, Bhi, Blo, Bn2, nb_img: int, P: int, precision: str, ready: Optional[torch.Tensor] = None,
                 first_image: int = 0):
    """ac_min_dist_arg: (dmin [nb_img, Mq], argmin [nb_img, Mq] int32 = row inside bank image j nearest to query row r)."""
    lib = _lib.load()
    _need_cuda(Qhi, Bhi)
    prec = _lib.PRECISIONS[precision]
    Mq, D = Qhi.shape
    assert Bhi.shape == (nb_img * P, D) and Qhi.is_contiguous() and Bhi.is_contiguous()
    dmin = torch.empty(nb_img, Mq, dtype=torch.float32, device=Qhi.device)
    arg = torch.empty(nb_img, Mq, dtype=torch.int32, device=Qhi.device)
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, nb_img, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=Qhi.device)
    _ready_ok(ready, nb_img)
    rc = lib.ac_min_dist_ready(_ptr(Qhi), _ptr(Qlo), _ptr(Qn2), Mq, _ptr(Bhi), _ptr(Blo), _ptr(Bn2), nb_img, P, D, prec, _ptr(dmin),
                               _ptr(arg), _ptr(ready), int(first_image), _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_min_dist_arg")
    return dmin, arg


def min_dist_sym_arg(Qhi, Qlo, Qn2, q_img0: int, Bhi, Blo, Bn2, nb_img: int, P: int, precision: str,
                     bank_window: Optional[Tuple[int, int]] = None, init: bool = True, out=None, groups: Optional[torch.Tensor] = None,
                     ready: Optional[torch.Tensor] = None):
    """ac_min_dist_sym_arg: (rowmin_d2 [nb_img, Mq], rowarg [nb_img, Mq] int32, colkey [Mq/P, nb_img*P] int64 =
    (fp32 bits of the column minimum << 32) | row inside the query image).  Windows / accumulation as min_dist_sym."""
    lib = _lib.load()
    _need_cuda(Qhi, Bhi)
    prec = _lib.PRECISIONS[precision]
    Mq, D = Qhi.shape
    assert Bhi.shape == (nb_img * P, D) and Qhi.is_contiguous() and Bhi.is_contiguous()
    if out is None:
        rowmin = torch.empty(nb_img, Mq, dtype=torch.float32, device=Qhi.device)
        rowarg = torch.zeros(nb_img, Mq, dtype=torch.int32, device=Qhi.device)
        colkey = torch.empty(Mq // P, nb_img * P, dtype=torch.int64, device=Qhi.device)
    else:
        rowmin, rowarg, colkey = out
    begin, count = bank_window if bank_window is not None else (0, nb_img)
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, nb_img, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=Qhi.device)
    _groups_ok(groups, nb_img)
    _ready_ok(ready, nb_img)
    rc = lib.ac_min_dist_sym_ready(_ptr(Qhi), _ptr(Qlo), _ptr(Qn2), Mq, q_img0, _ptr(Bhi), _ptr(Blo), _ptr(Bn2), nb_img, P, D, prec,
                                   int(begin), int(count), int(bool(init)), _ptr(rowmin), None, _ptr(rowarg), _ptr(colkey),
                                   _ptr(groups), _ptr(ready), _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_min_dist_sym_arg")
    return rowmin, rowarg, colkey


def min_dist_sym_grow(hi, lo, n2, n_old: int, nb_img: int, P: int, precision: str, arg: bool = False):
    """ac_min_dist_sym_grow: the new pairs of a category whose images [n_old, nb_img) have just joined images [0, n_old).
    hi / lo / n2 are the operands and norms of all nb_img images (new ones last); the query window is the new images.
    Returns (rowmin_d2 [nb_img, M*P], colmin_d2 [M, nb_img*P]) or, arg=True, (rowmin_d2, rowarg, colkey [M, nb_img*P] int64)."""
    lib = _lib.load()
    _need_cuda(hi, n2)
    prec = _lib.PRECISIONS[precision]
    D = hi.shape[1]
    assert hi.shape == (nb_img * P, D) and hi.is_contiguous() and n2.shape == (nb_img * P,)
    assert lo is None or (lo.shape == hi.shape and lo.is_contiguous())
    q0 = n_old * P
    Mq = nb_img * P - q0
    dev = hi.device
    rowmin = torch.empty(nb_img, Mq, dtype=torch.float32, device=dev)
    rowarg = colmin = colkey = None
    if arg:
        rowarg = torch.zeros(nb_img, Mq, dtype=torch.int32, device=dev)
        colkey = torch.empty(Mq // P, nb_img * P, dtype=torch.int64, device=dev)
    else:
        colmin = torch.empty(Mq // P, nb_img * P, dtype=torch.float32, device=dev)
    ws_bytes = lib.ac_min_dist_workspace_bytes(Mq, nb_img, P, D, prec)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    rc = lib.ac_min_dist_sym_grow(_ptr(hi[q0:]), _ptr(None if lo is None else lo[q0:]), _ptr(n2[q0:]), Mq, n_old, _ptr(hi), _ptr(lo),
                                  _ptr(n2), nb_img, P, D, prec, 0, nb_img, 1, _ptr(rowmin), _ptr(colmin), _ptr(rowarg), _ptr(colkey),
                                  None, int(n_old), _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_min_dist_sym_grow")
    return (rowmin, rowarg, colkey) if arg else (rowmin, colmin)


def refine_min_dist_grow(Z: torch.Tensor, hi, lo, n2, n_old: int, nb_img: int, P: int, rowarg: torch.Tensor, colkey: torch.Tensor):
    """ac_refine_min_dist_grow: exact fp32 distances of the new pairs of one growth launch, (drow [nb_img, M*P],
    dcol [M, nb_img*P]) in the layouts of its minima.  Z [nb_img*P, D] fp32 of every image of the category."""
    lib = _lib.load()
    _need_cuda(Z, hi, rowarg, colkey)
    D = hi.shape[1]
    Mq = (nb_img - n_old) * P
    assert Z.shape == (nb_img * P, D) and Z.dtype == torch.float32 and Z.is_contiguous()
    assert hi.shape == (nb_img * P, D) and hi.is_contiguous()
    assert rowarg.shape == (nb_img, Mq) and rowarg.dtype == torch.int32 and rowarg.is_contiguous()
    assert colkey.shape == (nb_img - n_old, nb_img * P) and colkey.dtype == torch.int64 and colkey.is_contiguous()
    drow = torch.empty(nb_img, Mq, dtype=torch.float32, device=hi.device)
    dcol = torch.empty(nb_img - n_old, nb_img * P, dtype=torch.float32, device=hi.device)
    rc = lib.ac_refine_min_dist_grow(_ptr(Z), _ptr(hi), _ptr(lo), _TORCH_TO_AC[hi.dtype], int(n_old), nb_img, P, D, _ptr(rowarg),
                                     _ptr(colkey), _ptr(n2), _ptr(drow), _ptr(dcol), _stream())
    check(rc, "ac_refine_min_dist_grow")
    return drow, dcol


def accumulate_weights_grow(rowv: torch.Tensor, colv: torch.Tensor, squared: bool, n_old: int, nb_img: int, P: int,
                            S: torch.Tensor) -> torch.Tensor:
    """ac_accumulate_weights_grow: adds the new pairs of one growth launch to the fp64 running sums S [>= nb_img*P] (in place)
    and returns w [nb_img*P] fp32 for every row of the category."""
    lib = _lib.load()
    _need_cuda(rowv, colv, S)
    Mq = (nb_img - n_old) * P
    assert rowv.shape == (nb_img, Mq) and colv.shape == (nb_img - n_old, nb_img * P)
    assert rowv.dtype == colv.dtype == torch.float32 and rowv.is_contiguous() and colv.is_contiguous()
    assert S.dtype == torch.float64 and S.is_contiguous() and S.numel() >= nb_img * P
    w = torch.empty(nb_img * P, dtype=torch.float32, device=rowv.device)
    check(lib.ac_accumulate_weights_grow(_ptr(rowv), _ptr(colv), int(bool(squared)), int(n_old), nb_img, P, _ptr(S), _ptr(w), _stream()),
          "ac_accumulate_weights_grow")
    return w


def refine_min_dist(Zq: Optional[torch.Tensor], Qhi, Qlo, Bhi, Blo, nb_img: int, P: int, rowarg: torch.Tensor,
                    colkey: Optional[torch.Tensor] = None, q_img0: int = 0, q_self: Optional[torch.Tensor] = None,
                    Pq: Optional[int] = None, groups: Optional[torch.Tensor] = None, Bn2: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ac_refine_min_dist: exact fp32 distances [nb_img, Mq] of the (query row, selected bank row) pairs.
    colkey given -> symmetric form (layout [nb_img, Mq], i.e. after the column-block exchange)."""
    lib = _lib.load()
    _need_cuda(Bhi, rowarg)
    Mq = rowarg.shape[1]
    D = Bhi.shape[1]
    assert rowarg.shape == (nb_img, Mq) and rowarg.dtype == torch.int32 and rowarg.is_contiguous()
    assert Bhi.shape == (nb_img * P, D) and Bhi.is_contiguous()
    if Zq is not None:
        assert Zq.shape == (Mq, D) and Zq.dtype == torch.float32 and Zq.is_contiguous()
    else:
        assert Qhi is not None and Qhi.shape == (Mq, D) and Qhi.is_contiguous() and Qhi.dtype == Bhi.dtype
    sym = colkey is not None
    if sym:
        assert colkey.shape == (nb_img, Mq) and colkey.dtype == torch.int64 and colkey.is_contiguous()
    if q_self is not None:
        assert q_self.dtype == torch.int32
    _groups_ok(groups, nb_img)
    out = torch.empty(nb_img, Mq, dtype=torch.float32, device=Bhi.device)
    rc = lib.ac_refine_min_dist(_ptr(Zq), _ptr(Qhi), _ptr(Qlo), Mq, _ptr(Bhi), _ptr(Blo), _TORCH_TO_AC[Bhi.dtype], nb_img, P, D,
                                _ptr(rowarg), _ptr(colkey), int(sym), int(q_img0), _ptr(q_self), int(Pq or P), _ptr(groups),
                                _ptr(Bn2), _ptr(out), _stream())
    check(rc, "ac_refine_min_dist")
    return out


def reduce_weights_sym(rowmin: torch.Tensor, colfull: torch.Tensor, Pq: int, q_img0: int,
                       groups: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    _need_cuda(rowmin, colfull)
    nb_img, Mq = rowmin.shape
    assert colfull.shape == rowmin.shape and colfull.is_contiguous() and rowmin.is_contiguous()
    _groups_ok(groups, nb_img)
    w = torch.empty(Mq, dtype=torch.float32, device=rowmin.device)
    check(lib.ac_reduce_weights_sym_ex(_ptr(rowmin), _ptr(colfull), Mq, nb_img, Pq, q_img0, _ptr(groups), _ptr(w), _stream()),
          "ac_reduce_weights_sym")
    return w


_REDUCE_MODES = {"mean": _lib.AC_REDUCE_MEAN, "min": _lib.AC_REDUCE_MIN, "min_update": _lib.AC_REDUCE_MIN_UPDATE}


def reduce_weights(dmin: torch.Tensor, Pq: int, q_self: Optional[torch.Tensor], mode: str,
                   groups: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ac_reduce_weights_ex: w [Mq] from dmin [nb_img, Mq].  mode 'mean' | 'min' | 'min_update'; 'min_update' lowers the running
    minimum held in `out` in place.  `out` (contiguous fp32 [Mq] on dmin's device) receives w, else a new tensor does."""
    if mode not in _REDUCE_MODES:
        raise ValueError("reduce mode must be one of %s, got %r" % (sorted(_REDUCE_MODES), mode))
    if out is None and mode == "min_update":
        raise ValueError("mode 'min_update' updates the running minimum passed as out=")
    lib = _lib.load()
    _need_cuda(dmin, q_self, out)
    nb_img, Mq = dmin.shape
    _groups_ok(groups, nb_img)
    _out_ok(out, "out", (Mq,), torch.float32, dmin.device)
    w = out if out is not None else torch.empty(Mq, dtype=torch.float32, device=dmin.device)
    m = _REDUCE_MODES[mode]
    if q_self is not None:
        assert q_self.dtype == torch.int32 and q_self.numel() * Pq >= Mq
    check(lib.ac_reduce_weights_ex(_ptr(dmin), Mq, nb_img, Pq, _ptr(q_self), _ptr(groups), m, _ptr(w), _stream()), "ac_reduce_weights")
    return w


def alpha(w: torch.Tensor, taus: Sequence[float], want64: bool = True, want32: bool = True):
    """w [N,P] fp32 -> (alpha64 [T,N,P] | None, alpha32 [T,N,P] | None)."""
    lib = _lib.load()
    _need_cuda(w)
    w = w.contiguous()
    N, P = w.shape
    T = len(taus)
    a64 = torch.empty(T, N, P, dtype=torch.float64, device=w.device) if want64 else None
    a32 = torch.empty(T, N, P, dtype=torch.float32, device=w.device) if want32 else None
    tarr = (ctypes.c_double * T)(*[float(t) for t in taus])
    check(lib.ac_alpha(_ptr(w), N, P, tarr, T, _ptr(a64), _ptr(a32), _stream()), "ac_alpha")
    return a64, a32


def weighted_embed(alpha32: torch.Tensor, Z: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _need_cuda(alpha32, Z)
    N, P, D = Z.shape
    a = alpha32.reshape(N, P).contiguous().float()
    assert Z.is_contiguous() and Z.dtype == torch.float32
    X = torch.empty(N, D, dtype=torch.float32, device=Z.device)
    check(lib.ac_weighted_embed(_ptr(a), _ptr(Z), N, P, D, _ptr(X), _stream()), "ac_weighted_embed")
    return X


def weighted_embed_multi(alpha32: torch.Tensor, Z: torch.Tensor) -> torch.Tensor:
    """X [T, N, D] for alpha [T, N, P] from ONE pass over Z [N, P, D] (ac_weighted_embed_multi): a tau sweep re-read Z per tau."""
    lib = _lib.load()
    _need_cuda(alpha32, Z)
    N, P, D = Z.shape
    T = alpha32.shape[0]
    a = alpha32.reshape(T, N, P).contiguous().float()
    assert Z.is_contiguous() and Z.dtype == torch.float32
    X = torch.empty(T, N, D, dtype=torch.float32, device=Z.device)
    check(lib.ac_weighted_embed_multi(_ptr(a), _ptr(Z), T, N, P, D, _ptr(X), _stream()), "ac_weighted_embed_multi")
    return X


def _layer_array(features):
    """(views, AcLayer array, AC_DT_* code of the maps).  float32, float16 and bfloat16 maps, one dtype for all layers."""
    views = [feature_view(f) for f in features]
    _need_cuda(*views)
    dt = views[0].dtype
    if dt not in _TORCH_TO_AC:
        raise ValueError("features must be float32, float16 or bfloat16, got %s" % dt)
    if any(v.dtype != dt for v in views):
        raise ValueError("all feature maps must share one dtype, got %s" % sorted({str(v.dtype) for v in views}))
    arr = (AcLayer * len(views))()
    for i, v in enumerate(views):
        _, C, H, W = v.shape
        sb, sc, sh, sw = v.stride()
        arr[i] = AcLayer(v.data_ptr(), C, H, W, sb, sc, sh, sw)
    return views, arr, _TORCH_TO_AC[dt]


def weighted_embed_from_features(features: Sequence[torch.Tensor], alpha32: torch.Tensor, patchsize: int, stride: int,
                                 pretrain_dim: int, target_dim: int, layernorm: bool = True, eps: float = 1e-5) -> torch.Tensor:
    """X [B, D] = sum_p alpha[b,p] Z[b,p] computed from the feature maps (no Z).  Raises AcError(AC_ERR_UNSUPPORTED)
    for shapes outside the fast form (callers fall back to embed + weighted_embed)."""
    lib = _lib.load()
    views, arr, feat_dt = _layer_array(features)
    B, L = views[0].shape[0], len(views)
    a = alpha32.reshape(B, -1).contiguous().float()
    X = torch.empty(B, target_dim, dtype=torch.float32, device=views[0].device)
    ws_bytes = lib.ac_weighted_embed_from_features_workspace_bytes_dt(arr, L, feat_dt, B, patchsize)
    ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=views[0].device)
    rc = lib.ac_weighted_embed_from_features_dt(arr, L, feat_dt, B, patchsize, stride, pretrain_dim, target_dim, int(layernorm),
                                                float(eps), _ptr(a), _ptr(X), _ptr(ws), ws_bytes, _stream())
    check(rc, "ac_weighted_embed_from_features")
    return X


def pairwise_l2(X: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    _need_cuda(X)
    X = X.contiguous().float()
    N, D = X.shape
    out = torch.empty(N, N, dtype=torch.float32, device=X.device)
    check(lib.ac_pairwise_l2(_ptr(X), N, D, _ptr(out), _stream()), "ac_pairwise_l2")
    return out


def copy_blocks(dsts: Sequence[torch.Tensor], srcs: Sequence[torch.Tensor]) -> None:
    """dsts[k].copy_(srcs[k]) for up to 16 two-dimensional blocks (unit stride along the last axis, any row stride) in ONE
    launch -- ac_copy_blocks.  The sources may be peer mappings of symmetric memory."""
    import ctypes

    lib = _lib.load()
    n = len(dsts)
    assert n == len(srcs) and n <= 16
    if n == 0:
        return
    _need_cuda(*dsts)
    _need_cuda(*srcs)
    for d, s_ in zip(dsts, srcs):
        assert d.dim() == 2 and d.shape == s_.shape and d.dtype == s_.dtype and d.stride(1) == 1 and s_.stride(1) == 1
    es = dsts[0].element_size()
    src = (ctypes.c_void_p * n)(*[s_.data_ptr() for s_ in srcs])
    dst = (ctypes.c_void_p * n)(*[d.data_ptr() for d in dsts])
    sst = (ctypes.c_int64 * n)(*[s_.stride(0) * s_.element_size() for s_ in srcs])
    dstr = (ctypes.c_int64 * n)(*[d.stride(0) * d.element_size() for d in dsts])
    rows = (ctypes.c_int32 * n)(*[d.shape[0] for d in dsts])
    rb = (ctypes.c_int64 * n)(*[d.shape[1] * es for d in dsts])
    check(lib.ac_copy_blocks(n, src, sst, dst, dstr, rows, rb, _stream()), "ac_copy_blocks")
