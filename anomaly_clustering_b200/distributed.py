"""Query-sharded multi-GPU form of the path (one process per GPU, torch.distributed / NCCL).

w_i, alpha_i and X_i depend only on query image i and the read-only bank
(reference: models/patchcore/utils.py:245-246, 265-266 -- the loop over i is independent), so:
  rank r embeds its slice of images  ->  the tensor-core operands (+ norms) of the bank images whose pairs it owns travel to
  it  ->  rank r runs stages 2/3 for its query slice (symmetric form: every unordered image pair once, the column minima of
  other ranks' query rows are exchanged)  ->  all-gather of the X rows  ->  Dmat.  fp32 Z never leaves its rank.
On CPU (gloo) the same sharding / gather logic is exercised by tests with a stand-in compute.

The operand shards travel over one of two transports (DESIGN.md section 6):
  symmetric memory  the embed kernel writes into this rank's slice of a symmetric-memory bank, every rank pulls the shards it
                    needs with copy-engine copies (symm_transport.SymmetricBank), ONE distance launch waits for per-bank-image
                    arrival flags (ac_min_dist_sym_ready), and the column minima are exchanged through symmetric memory too.
                    Chosen by _symmetric_bank: the CUDA back-end on an NCCL group of more than one rank, a tensor-core
                    precision, and a set-up that succeeds; run_path_sharded also needs the symmetric form with P >= 32.
  NCCL collectives  everywhere else (gloo groups, precision 'f32', P < 32, symmetric memory that cannot be set up): the bank
                    shards are all-gathered or sent point to point, the local shard is multiplied while they travel, and the
                    column minima go through an all_to_all (exchange_colmin)."""
from __future__ import annotations

import functools
from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import ops, pipeline
from .symm_transport import SymmetricBank


def pair_owned(i: int, j: int, n: int) -> bool:
    """Host mirror of the kernel's pair-ownership rule (csrc/mindist_tc.cu: pair_owned)."""
    d = (j - i) % n
    if d == 0:
        return False
    if 2 * d < n:
        return True
    if 2 * d == n:
        return i < j
    return False


def pair_owned_grow(n_old: int, i: int, j: int, n: int) -> bool:
    """Host mirror of the growth ownership rule (csrc/common.cuh: pair_owned_grow): images [n_old, n) join images [0, n_old); a
    new image owns its pairs with the old ones, two new images follow pair_owned among the new, two old images have no owner."""
    if i < n_old:
        return False
    if j < n_old:
        return True
    return pair_owned(i - n_old, j - n_old, n - n_old)


def shard_bounds(n_items: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous, balanced slices: the first n % world ranks get one extra item."""
    base, extra = divmod(n_items, world)
    out, start = [], 0
    for r in range(world):
        cnt = base + (1 if r < extra else 0)
        out.append((start, start + cnt))
        start += cnt
    return out


def lpt_assign(costs: Sequence[float], world: int) -> List[List[int]]:
    """Greedy longest-processing-time assignment of work items (e.g. categories with cost
    n_c * (n_c - 1)) to ranks; returns item indices per rank (SURVEY.md section 8e)."""
    order = sorted(range(len(costs)), key=lambda i: -costs[i])
    loads = [0.0] * world
    bins: List[List[int]] = [[] for _ in range(world)]
    for i in order:
        r = min(range(world), key=lambda k: loads[k])
        bins[r].append(i)
        loads[r] += costs[i]
    return bins


def all_gather_rows(local: torch.Tensor, counts: Sequence[int], group=None) -> torch.Tensor:
    """All-gather row blocks of unequal length: local [counts[rank], ...] -> [sum(counts), ...].

    NCCL: every rank's block lands directly in its slice of the result (equal counts: one
    all_gather_into_tensor; unequal: torch's grouped-broadcast all_gather on views) -- no padding and no
    compaction copy of the gathered bank.  gloo (CPU tests): padded all_gather_into_tensor + compaction."""
    world = dist.get_world_size(group)
    tail = tuple(local.shape[1:])
    local = local.contiguous()
    if all(c == counts[0] for c in counts):
        buf = torch.empty((sum(counts),) + tail, dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(buf, local, group=group)
        return buf
    if dist.get_backend(group) == "nccl":
        buf = torch.empty((sum(counts),) + tail, dtype=local.dtype, device=local.device)
        views, start = [], 0
        for c in counts:
            views.append(buf[start:start + c])
            start += c
        dist.all_gather(views, local, group=group)
        return buf
    mx = max(counts)
    send = torch.zeros((mx,) + tail, dtype=local.dtype, device=local.device)
    send[: local.shape[0]] = local
    buf = torch.empty((world * mx,) + tail, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(buf, send, group=group)
    return torch.cat([buf[r * mx : r * mx + counts[r]] for r in range(world)], dim=0)


def needed_shards(bounds: Sequence[Tuple[int, int]], n_total: int) -> List[List[int]]:
    return [list(x) for x in _needed_shards(tuple(tuple(b) for b in bounds), n_total)]


@functools.lru_cache(maxsize=64)
def _needed_shards(bounds: Tuple[Tuple[int, int], ...], n_total: int):
    """Symmetric form: need[r] = ranks whose images appear as BANK images of pairs owned by rank r's
    query images (the circular window of the next n_total//2 images) -- about half of the other ranks."""
    world = len(bounds)
    owner = [0] * n_total
    for s, (a, b) in enumerate(bounds):
        for i in range(a, b):
            owner[i] = s
    need = []
    for r, (a, b) in enumerate(bounds):
        ranks = set()
        for i in range(a, b):
            for d in range(1, n_total // 2 + 1):
                j = (i + d) % n_total
                if pair_owned(i, j, n_total):
                    ranks.add(owner[j])
        ranks.discard(r)
        need.append(tuple(sorted(ranks)))
    return tuple(need)


def start_gather_needed_rows(local: torch.Tensor, bounds: Sequence[Tuple[int, int]], rows_per_item: int,
                             need: Sequence[Sequence[int]], group=None):
    """Like all_gather_rows, but a rank only receives the shards listed in need[rank]; the rest of the
    returned [sum rows, ...] buffer stays uninitialised (the symmetric kernel never touches it).
    Point-to-point NCCL sends/receives in one batch (roughly half the all-gather volume), left IN FLIGHT:
    returns (buffer, requests); the caller waits on the requests before touching remote shards."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    total = bounds[-1][1] * rows_per_item
    buf = torch.empty((total,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    a, b = bounds[rank]
    local = local.contiguous()
    buf[a * rows_per_item : b * rows_per_item].copy_(local)
    ops_ = []
    for dst in range(world):
        if dst != rank and rank in need[dst] and local.shape[0] > 0:
            ops_.append(dist.P2POp(dist.isend, local, dst, group=group))
    for src in need[rank]:
        sa, sb = bounds[src]
        if sb > sa:
            ops_.append(dist.P2POp(dist.irecv, buf[sa * rows_per_item : sb * rows_per_item], src, group=group))
    reqs = dist.batch_isend_irecv(ops_) if ops_ else []
    return buf, reqs


def start_all_gather_rows(local: torch.Tensor, counts: Sequence[int], group=None):
    """Asynchronous all-gather of row blocks into one buffer whose local slice is already valid, so work on
    the local shard can overlap the collective.  Returns (buffer, [work])."""
    rank = dist.get_rank(group)
    tail = tuple(local.shape[1:])
    local = local.contiguous()
    buf = torch.empty((sum(counts),) + tail, dtype=local.dtype, device=local.device)
    start = sum(counts[:rank])
    buf[start:start + counts[rank]].copy_(local)
    if all(c == counts[0] for c in counts):
        work = dist.all_gather_into_tensor(buf, local, group=group, async_op=True)
    elif dist.get_backend(group) != "nccl":
        # gloo (CPU tests) rejects all_gather on unequal blocks: point-to-point exchange of the same blocks
        world = dist.get_world_size(group)
        offs = [sum(counts[:r]) for r in range(world)]
        ops_ = []
        for peer in range(world):
            if peer == rank:
                continue
            if counts[rank] > 0:
                ops_.append(dist.P2POp(dist.isend, local, peer, group=group))
            if counts[peer] > 0:
                ops_.append(dist.P2POp(dist.irecv, buf[offs[peer]:offs[peer] + counts[peer]], peer, group=group))
        return buf, (dist.batch_isend_irecv(ops_) if ops_ else [])
    else:
        views, s0 = [], 0
        for c in counts:
            views.append(buf[s0:s0 + c])
            s0 += c
        work = dist.all_gather(views, local, group=group, async_op=True)
    return buf, [work]


def _weighted_embed_all_taus(compute, a32, Z3, T: int) -> torch.Tensor:
    """[n_r, T, D]: one pass over Z for all taus when the compute back-end has the fused form (the CUDA library), else per tau."""
    if hasattr(compute, "weighted_embed_multi"):
        return compute.weighted_embed_multi(a32, Z3).transpose(0, 1).contiguous()
    return torch.stack([compute.weighted_embed(a32[t], Z3) for t in range(T)], dim=1)


def exchange_colmin(colmin: torch.Tensor, bounds: Sequence[Tuple[int, int]], P: int, group=None) -> torch.Tensor:
    """Symmetric mode: rank r holds colmin [n_r, N*P] = (its images as BANK image, every global query
    row); the owner of query rows [a*P, b*P) needs those columns from every rank.  All-to-all of the
    column blocks -> [N, n_r*P] (bank image, local query row)."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    n_r = bounds[rank][1] - bounds[rank][0]
    send = [colmin[:, a * P : b * P].contiguous() for a, b in bounds]
    recv = [torch.empty((b - a, n_r * P), dtype=colmin.dtype, device=colmin.device) for a, b in bounds]
    if dist.get_backend(group) == "nccl":
        dist.all_to_all(recv, send, group=group)
    else:  # gloo (CPU tests) has no all_to_all for uneven splits: point-to-point exchange
        recv[rank].copy_(send[rank])
        reqs = []
        for peer in range(world):
            if peer == rank:
                continue
            reqs.append(dist.isend(send[peer], peer, group=group))
            reqs.append(dist.irecv(recv[peer], peer, group=group))
        for r in reqs:
            r.wait()
    return torch.cat(recv, dim=0)


class _CudaCompute:
    """The default compute back-end of the sharded paths: the CUDA library (tests substitute a CPU stand-in)."""

    embed_images = staticmethod(pipeline.embed_images)
    min_distance_weights = staticmethod(pipeline.min_distance_weights)
    alpha = staticmethod(ops.alpha)
    weighted_embed = staticmethod(ops.weighted_embed)
    weighted_embed_multi = staticmethod(ops.weighted_embed_multi)
    weighted_embed_from_features = staticmethod(ops.weighted_embed_from_features)
    pairwise_l2 = staticmethod(ops.pairwise_l2)
    min_dist_sym = staticmethod(ops.min_dist_sym)
    min_dist_sym_arg = staticmethod(ops.min_dist_sym_arg)
    refine_min_dist = staticmethod(ops.refine_min_dist)
    reduce_weights_sym = staticmethod(ops.reduce_weights_sym)
    reduce_weights = staticmethod(ops.reduce_weights)


def _symmetric_bank(compute, rows: int, D: int, precision: str, device, group) -> Optional[SymmetricBank]:
    """The symmetric-memory bank of `rows` operand rows of width D, or None where the NCCL collectives carry the operands:
    a back-end other than the CUDA library, a group that is not NCCL or has one rank, precision 'f32' (no tensor-core
    operands), or a symmetric-memory set-up that fails (reported once; the transport then stays off in this process)."""
    if not (compute is _CudaCompute and dist.get_world_size(group) > 1 and dist.get_backend(group) == "nccl"
            and precision != "f32" and SymmetricBank.disabled_reason is None):
        return None
    operand, want_lo = pipeline._OPERAND_OF[precision]
    try:
        return SymmetricBank.get(rows, D, torch.float16 if operand == "f16" else torch.bfloat16, want_lo, device, group)
    except Exception as e:  # noqa: BLE001 -- symmetric memory unavailable on this system: say so once, use NCCL
        SymmetricBank.disabled_reason = repr(e)
        import warnings

        warnings.warn("symmetric-memory transport unavailable (%r): the sharded path uses NCCL collectives" % (e,))
        return None


def _sym_minima_symmetric_memory(compute, symm_bank: SymmetricBank, q, bounds, n_total: int, precision: str, rank: int,
                                 world: int):
    """Symmetric form over the symmetric-memory transport.  q's operands already sit in this rank's slice of the bank.
    The needed shards are pulled on the copy engines while ONE distance launch runs over the whole bank: its loader waits
    for a bank image's arrival flag before reading it (measured on one GPU with the launches of an 8-GPU config-2 rank:
    2.40 ms in one launch against 2.59 ms in three windows of landed shards).  The column minima (keys in the refined
    modes) are written straight into symmetric memory and collected by SymmetricBank.exchange_colmin.
    Returns (bank, minima of the launch, column block [N, n_r*P])."""
    P, (lo_i, hi_i) = q.P, bounds[rank]
    refined = precision in pipeline.REFINED
    pipeline._mark("gather_begin")
    # every shard for the refined modes (each rank re-evaluates all of its rows against the whole bank)
    need = [r for r in range(world) if r != rank] if refined else needed_shards(bounds, n_total)[rank]
    ready = torch.zeros(n_total, dtype=torch.int32, device=q.hi.device)
    ready[lo_i:hi_i] = 1
    (hi_buf, lo_buf, n2_buf), pulls = symm_bank.publish_and_pull(bounds, P, need, rank, world, ready)
    bank = pipeline.PatchSet(n_total, P, q.D, q.grid, hi=hi_buf, lo=lo_buf, n2=n2_buf)
    pipeline._mark("gather_end")
    n_max = max(b - a for a, b in bounds)
    Mq = q.n_img * P
    rowmin = torch.empty(n_total, Mq, dtype=torch.float32, device=q.hi.device)
    if refined:
        out = (rowmin, torch.zeros(n_total, Mq, dtype=torch.int32, device=q.hi.device),
               symm_bank.colmin_buffer(q.n_img, n_max, n_total * P, torch.int64))
    else:
        out = (rowmin, symm_bank.colmin_buffer(q.n_img, n_max, n_total * P, torch.float32))
    launch = compute.min_dist_sym_arg if refined else compute.min_dist_sym
    pipeline._mark("mindist_begin")
    out = launch(q.hi, q.lo, q.n2, lo_i, bank.hi, bank.lo, bank.n2, n_total, P, precision, init=True, out=out, ready=ready)
    pipeline._mark("mindist_end")
    # the launch itself does not need the pulls to have completed; refine and the next step's buffer reuse do
    for r in pulls:
        r.wait()
    pipeline._mark("exchange_begin")
    colfull = symm_bank.exchange_colmin(bounds, P, rank, world)
    pipeline._mark("exchange_end")
    return bank, out, colfull


def _sym_minima_nccl(compute, q, bounds, n_total: int, precision: str, group):
    """Symmetric form over NCCL collectives: the bank shards travel asynchronously while the pairs inside the local shard
    are multiplied, the remote bank images follow in a second launch, and the column minima go through exchange_colmin.
    Returns (bank, minima of the launches, column block [N, n_r*P])."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    P, (lo_i, hi_i) = q.P, bounds[rank]
    refined = precision in pipeline.REFINED
    launch = compute.min_dist_sym_arg if refined else compute.min_dist_sym
    pipeline._mark("gather_begin")
    if (3 <= world <= 4 or dist.get_backend(group) != "nccl") and not refined:
        # 3-4 ranks: point-to-point transfers of just the shards that hold bank images of pairs this rank owns (the next
        # n_total//2 images, about 2/3 of the volume).  At 2 ranks the needed shard IS the other rank's shard and NCCL's
        # all-gather moves it faster (0.5 vs 0.9 ms).
        need = needed_shards(bounds, n_total)
        hi_buf, r1 = start_gather_needed_rows(q.hi, bounds, P, need, group)
        lo_buf, r2 = (None, []) if q.lo is None else start_gather_needed_rows(q.lo, bounds, P, need, group)
        n2_buf, r3 = start_gather_needed_rows(q.n2, bounds, P, need, group)
    else:
        # many ranks: NCCL's all-gather moves the whole bank faster than 4+ send/recv pairs per rank
        # move half of it (measured at 8 GPUs: 562 MB in 1.0 ms vs 321 MB in 1.2 ms)
        row_counts = [(b - a) * P for a, b in bounds]
        hi_buf, r1 = start_all_gather_rows(q.hi, row_counts, group)
        lo_buf, r2 = (None, []) if q.lo is None else start_all_gather_rows(q.lo, row_counts, group)
        n2_buf, r3 = start_all_gather_rows(q.n2, row_counts, group)
    pending = list(r1) + list(r2) + list(r3)
    bank = pipeline.PatchSet(n_total, P, q.D, q.grid, hi=hi_buf, lo=lo_buf, n2=n2_buf)
    pipeline._mark("gather_end")
    # NCCL's transfer kernels take a few SMs away from the persistent GEMM; its dynamic unit scheduler absorbs that (with
    # the earlier static round-robin the overlap cost more than it hid at 2 ranks).  A one-rank group transfers nothing.
    if pending and q.n_img > 1 and world > 1:
        # phase 1: bank images of the local shard (no remote data needed) overlaps the NCCL transfers
        pipeline._mark("mindist_begin")
        out = launch(q.hi, q.lo, q.n2, lo_i, bank.hi, bank.lo, bank.n2, n_total, P, precision,
                     bank_window=(lo_i, q.n_img), init=True)
        pipeline._mark("mindist_end")
        for r in pending:
            r.wait()
        pipeline._mark("mindist_begin")
        out = launch(q.hi, q.lo, q.n2, lo_i, bank.hi, bank.lo, bank.n2, n_total, P, precision,
                     bank_window=(hi_i % n_total, n_total - q.n_img), init=False, out=out)
        pipeline._mark("mindist_end")
    else:
        for r in pending:
            r.wait()
        pipeline._mark("mindist_begin")
        out = launch(q.hi, q.lo, q.n2, lo_i, bank.hi, bank.lo, bank.n2, n_total, P, precision)
        pipeline._mark("mindist_end")
    pipeline._mark("exchange_begin")
    colfull = exchange_colmin(out[-1], bounds, P, group)   # float minima, or (distance, row) keys when refined
    pipeline._mark("exchange_end")
    return bank, out, colfull


def run_path_sharded(
    local_features: Sequence[torch.Tensor],
    n_total: int,
    patchsize: int,
    stride: int,
    pretrain_dim: int,
    target_dim: int,
    taus: Sequence[float] = (1.0,),
    precision: str = "auto",
    group=None,
    compute=None,
    symmetric: bool = True,
    keep_z: bool = True,
):
    """Unsupervised path over n_total images sharded by shard_bounds(); `local_features` are this
    rank's images.  Returns (alpha64_local [T,n_r,P], X_all [T,N,D], Dmat [T,N,N], w_local).

    `compute` (tests only) substitutes the compute back-end -- an object with embed_images,
    min_distance_weights, alpha, weighted_embed, pairwise_l2 -- so that the sharding / gather logic
    can be exercised on CPU with gloo; the default is the CUDA library and nothing else."""
    precision = pipeline.resolve_precision(precision, taus)
    if compute is None:
        compute = _CudaCompute
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if n_total < world:
        # an empty shard has no patch grid to agree on; callers with fewer images than ranks pass a sub-group
        raise ValueError("run_path_sharded: %d images over %d ranks leaves empty shards; use a smaller group" % (n_total, world))
    bounds = shard_bounds(n_total, world)
    lo_i, hi_i = bounds[rank]
    z_free = (not keep_z) and hasattr(compute, "weighted_embed_from_features") and pipeline.z_free_supported(
        local_features, patchsize, stride, pretrain_dim, target_dim, precision) and precision not in pipeline.REFINED
    refined = precision in pipeline.REFINED
    symm_bank = outs = None
    if symmetric:
        v0 = ops.feature_view(local_features[0])
        gh, gw = ops.patch_grid(v0.shape[2], v0.shape[3], patchsize, stride)
        if gh * gw >= 32:   # the symmetric kernel's shapes (use_sym below)
            symm_bank = _symmetric_bank(compute, n_total * gh * gw, target_dim, precision, v0.device, group)
        if symm_bank is not None:   # the embed kernel writes straight into this rank's slice of the bank
            outs = symm_bank.local_slices(lo_i * gh * gw, hi_i * gh * gw)
    q = compute.embed_images(local_features, patchsize, stride, pretrain_dim, target_dim, precision, want_z=not z_free, out=outs)
    assert q.n_img == hi_i - lo_i
    P = q.P
    use_sym = symmetric and precision != "f32" and P >= 32 and hasattr(compute, "min_dist_sym")
    # refined modes ('f16r'): the tensor-core pass records arg-mins, ac_refine_min_dist re-evaluates the selected pairs
    # exactly.  Every rank refines ALL (own row, other image) entries, so it needs the whole bank (every shard) and the
    # (distance, row) keys of the column minima travel instead of the float minima.
    if refined and not (use_sym and hasattr(compute, "min_dist_sym_arg")):
        raise ValueError("precision %r needs the symmetric sharded path" % precision)
    if use_sym:
        # every unordered image pair is multiplied once, by the rank that owns the pair's first image;
        # the column minima it produces for other ranks' query rows travel back to their owners
        if symm_bank is not None:
            bank, out, colfull = _sym_minima_symmetric_memory(compute, symm_bank, q, bounds, n_total, precision, rank, world)
        else:
            bank, out, colfull = _sym_minima_nccl(compute, q, bounds, n_total, precision, group)
        if refined:
            pipeline._mark("refine_begin")
            dex = compute.refine_min_dist(q.Z, q.hi, q.lo, bank.hi, bank.lo, n_total, P, out[1], colkey=colfull, q_img0=lo_i,
                                          Bn2=bank.n2)
            pipeline._mark("refine_end")
            own = torch.arange(lo_i, hi_i, dtype=torch.int32, device=dex.device)
            w = compute.reduce_weights(dex, P, own, "mean").reshape(q.n_img, P)
        else:
            w = compute.reduce_weights_sym(out[0], colfull, P, lo_i).reshape(q.n_img, P)
    else:
        row_counts = [(b - a) * P for a, b in bounds]
        pipeline._mark("gather_begin")
        if precision == "f32":
            bank = pipeline.PatchSet(n_total, P, q.D, q.grid, Z=all_gather_rows(q.Z, row_counts, group))
        else:
            bank = pipeline.PatchSet(
                n_total, P, q.D, q.grid,
                hi=all_gather_rows(q.hi, row_counts, group),
                lo=None if q.lo is None else all_gather_rows(q.lo, row_counts, group),
                n2=all_gather_rows(q.n2, row_counts, group),
            )
        pipeline._mark("gather_end")
        q_self = torch.arange(lo_i, hi_i, dtype=torch.int32, device=q.hi.device if q.Z is None else q.Z.device)
        w = compute.min_distance_weights(q, bank, "unsupervised", precision, q_self=q_self)
    a64, a32 = compute.alpha(w, list(taus))
    if z_free:
        X_loc = torch.stack([compute.weighted_embed_from_features(local_features, a32[t], patchsize, stride, pretrain_dim, q.D)
                             for t in range(len(taus))], dim=1)
    else:
        Z3 = q.Z.reshape(q.n_img, P, q.D)
        X_loc = _weighted_embed_all_taus(compute, a32, Z3, len(taus))                               # [n_r, T, D]
    pipeline._mark("xgather_begin")
    X_all = all_gather_rows(X_loc, [b - a for a, b in bounds], group).permute(1, 0, 2).contiguous()  # [T, N, D]
    pipeline._mark("xgather_end")
    Dm = torch.stack([compute.pairwise_l2(X_all[t]) for t in range(len(taus))])
    return a64, X_all, Dm, w


def run_path_sharded_supervised(
    local_features: Sequence[torch.Tensor],
    n_total: int,
    local_bank_features: Sequence[torch.Tensor],
    n_bank_total: int,
    patchsize: int,
    stride: int,
    pretrain_dim: int,
    target_dim: int,
    taus: Sequence[float] = (1.0,),
    precision: str = "auto",
    group=None,
    compute=None,
    overlap: bool = True,
):
    """Supervised path (utils.py:230-237, 260-277) sharded both ways (SURVEY.md section 8e): the n_total query
    images by shard_bounds(n_total), the n_bank_total normal images by shard_bounds(n_bank_total) for the embed
    only; the bank's tensor-core operands (+ norms; fp32 Z for precision 'f32') are all-gathered and every rank
    takes w = min over ALL bank images for its own queries.  The min over bank images splits over bank pieces, so
    the local bank shard is multiplied while the gather is in flight (`overlap`), the remote pieces after it.
    Returns (alpha64_local [T,n_r,P], X_all [T,N,D], Dmat [T,N,N], w_local) like run_path_sharded.
    `compute`: tests only, see run_path_sharded."""
    precision = pipeline.resolve_precision(precision, taus)
    if compute is None:
        compute = _CudaCompute
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if n_total < world or n_bank_total < world:
        raise ValueError("run_path_sharded_supervised: %d query / %d bank images over %d ranks leaves empty shards; "
                         "use a smaller group" % (n_total, n_bank_total, world))
    qb, bb = shard_bounds(n_total, world), shard_bounds(n_bank_total, world)
    q = compute.embed_images(local_features, patchsize, stride, pretrain_dim, target_dim, precision, want_z=True)
    b_loc = compute.embed_images(local_bank_features, patchsize, stride, pretrain_dim, target_dim, precision,
                                 want_z=(precision == "f32"))
    assert q.n_img == qb[rank][1] - qb[rank][0] and b_loc.n_img == bb[rank][1] - bb[rank][0] and b_loc.P == q.P
    P = q.P
    counts = [(b - a) * P for a, b in bb]

    def piece(bufs, a, b):
        """Bank images [a, b) of the gathered buffers as a PatchSet (row slices of contiguous buffers)."""
        Zb, hib, lob, n2b = bufs
        cut = lambda t: None if t is None else t[a * P : b * P]  # noqa: E731
        return pipeline.PatchSet(b - a, P, q.D, q.grid, Z=cut(Zb), hi=cut(hib), lo=cut(lob), n2=cut(n2b))

    # Symmetric-memory transport for the bank (as in run_path_sharded): the bank shard is copied into a symmetric buffer,
    # every rank pulls the other shards with copy-engine copies, and ONE all-pairs launch walks the bank from the local shard
    # on while they land (arrival flags, ac_min_dist_ready).
    symm_bank = _symmetric_bank(compute, n_bank_total * P, target_dim, precision, local_features[0].device, group)
    if symm_bank is not None:
        lo_b, hi_b = bb[rank]
        hi_s, lo_s, n2_s = symm_bank.local_slices(lo_b * P, hi_b * P)
        hi_s.copy_(b_loc.hi)
        if lo_s is not None:
            lo_s.copy_(b_loc.lo)
        n2_s.copy_(b_loc.n2)
        pipeline._mark("gather_begin")
        ready = torch.zeros(n_bank_total, dtype=torch.int32, device=q.hi.device)
        ready[lo_b:hi_b] = 1
        (hib, lob, n2b), pulls = symm_bank.publish_and_pull(bb, P, [r for r in range(world) if r != rank], rank, world, ready)
        pipeline._mark("gather_end")

        def landed():
            for r in pulls:
                r.wait()

        bank_all = pipeline.PatchSet(n_bank_total, P, q.D, q.grid, hi=hib, lo=lob, n2=n2b)
        w = compute.min_distance_weights(q, bank_all, "supervised", precision, bank_ready=ready, bank_first=lo_b, bank_landed=landed)
        return _supervised_tail(compute, q, w, taus, qb, P, group)

    pipeline._mark("gather_begin")
    pending = []
    if precision == "f32":
        Zb, r0 = start_all_gather_rows(b_loc.Z, counts, group)
        bufs, pending = (Zb, None, None, None), list(r0)
    else:
        hib, r1 = start_all_gather_rows(b_loc.hi, counts, group)
        lob, r2 = (None, []) if b_loc.lo is None else start_all_gather_rows(b_loc.lo, counts, group)
        n2b, r3 = start_all_gather_rows(b_loc.n2, counts, group)
        bufs, pending = (None, hib, lob, n2b), list(r1) + list(r2) + list(r3)
    pipeline._mark("gather_end")
    lo_b, hi_b = bb[rank]
    w = None
    if overlap and world > 1:
        w = compute.min_distance_weights(q, piece(bufs, lo_b, hi_b), "supervised", precision)   # local shard: already valid
        rest = [(0, lo_b), (hi_b, n_bank_total)]
    else:
        rest = [(0, n_bank_total)]
    for r in pending:
        r.wait()
    for a, b in rest:
        if b > a:
            wp = compute.min_distance_weights(q, piece(bufs, a, b), "supervised", precision)
            w = wp if w is None else torch.minimum(w, wp)
    return _supervised_tail(compute, q, w, taus, qb, P, group)


def _supervised_tail(compute, q, w, taus, qb, P, group):
    """alpha, X of the local query rows, all-gather of the X rows, Dmat (stage 3 of run_path_sharded_supervised)."""
    a64, a32 = compute.alpha(w, list(taus))
    Z3 = q.Z.reshape(q.n_img, P, q.D)
    X_loc = _weighted_embed_all_taus(compute, a32, Z3, len(taus))                                   # [n_r, T, D]
    pipeline._mark("xgather_begin")
    X_all = all_gather_rows(X_loc, [b - a for a, b in qb], group).permute(1, 0, 2).contiguous()     # [T, N, D]
    pipeline._mark("xgather_end")
    Dm = torch.stack([compute.pairwise_l2(X_all[t]) for t in range(len(taus))])
    return a64, X_all, Dm, w


def run_path_sharded_average(local_features: Sequence[torch.Tensor], n_total: int, patchsize: int, stride: int, pretrain_dim: int,
                             target_dim: int, group=None):
    """'average' mode (examples/main.py:290-291: alpha = 1/P) sharded by query image: every rank reduces its own images,
    the X rows are all-gathered, Dmat on every rank.  Returns (X_all [1,N,D], Dmat [1,N,N])."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    bounds = shard_bounds(n_total, world)
    r = pipeline.run_path(local_features, patchsize, stride, pretrain_dim, target_dim, "average", keep_z=False)
    assert r.X.shape[1] == bounds[rank][1] - bounds[rank][0]
    X_all = all_gather_rows(r.X[0], [b - a for a, b in bounds], group)
    return X_all.unsqueeze(0), ops.pairwise_l2(X_all).unsqueeze(0)


def run_categories_sharded(sizes: Sequence[int], run_category, group=None):
    """Per-category banks (the reference's own semantics: one make_category_data per category, main.py:353):
    whole categories are assigned to ranks by greedy LPT on n_c * (n_c - 1) (the pair count, SURVEY.md section 8e)
    and each rank calls `run_category(c)` for its own; there is no collective on the data path.
    Returns {category index: result} for this rank's categories and the full assignment."""
    rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    bins = lpt_assign([float(n) * (n - 1) for n in sizes], world)
    return {c: run_category(c) for c in bins[rank]}, bins
