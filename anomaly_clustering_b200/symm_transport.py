"""Copy-engine transport of the tensor-core operands for the sharded path (used on NCCL groups with the CUDA back-end;
distributed._symmetric_bank decides, and falls back to NCCL collectives when symmetric memory cannot be set up).

Why (measured at 8 B200, config 2, profiles/r02_timeline_*): NCCL moves a rank's 80 MB operand shard at 120-140 GB/s
through its send/recv kernels and the uneven all-gather (grouped broadcasts, LL protocol) needs 1.2 ms for 562 MB -- both
slower than the 0.6 ms GEMM that consumes a shard, so the min-distance kernel waited for data.  With the bank buffers
allocated as torch symmetric memory (CUDA VMM allocations mapped into every rank of the node over NVLink / NVSwitch)

  * the embed kernel writes its operands and norms STRAIGHT into this rank's slice of the symmetric bank (no staging copy),
  * one device-side barrier publishes the slices,
  * every rank PULLS the shards it needs from the peer mappings with plain device-to-device copies on a side stream:
    they run on the copy engines at NVLink speed and cost no SM while the persistent GEMM is running (ring order
    rank+1, rank+2, ...).

Two buffer sets alternate between steps, so ONE barrier per buffer kind and step is enough: a rank reaches the barrier of step
t+1 only after its stream has consumed every shard it pulled in step t, hence after that barrier the set of step t may be
overwritten (that happens in step t+2).

The same object carries the two later stages of the step:
  * arrival flags -- publish_and_pull(ready=...) sets one int32 per bank image on the side stream right after the shard that holds
    it has landed; the distance kernel (ac_min_dist_sym_ready) is launched ONCE over the whole bank and waits per bank image;
  * the column-minimum exchange -- colmin_buffer() hands the distance kernel a symmetric buffer for its column minima,
    exchange_colmin() is one more barrier plus one batched strided read (ac_copy_blocks) of this rank's columns out of every
    peer's buffer, instead of an NCCL all_to_all."""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch


class _EventRequest:
    """Looks like a torch.distributed Work to run_path_sharded: wait() orders the current stream after the pull."""

    def __init__(self, event: torch.cuda.Event):
        self.event = event

    def wait(self) -> None:
        torch.cuda.current_stream().wait_event(self.event)


class SymmetricBank:
    """Persistent symmetric buffers for (hi, lo, n2) of the WHOLE bank, two sets per (rows, D, dtype, lo?, group)."""

    _cache = {}
    disabled_reason: Optional[str] = None          # set when the symmetric-memory set-up failed once (NCCL transport is used)

    @classmethod
    def get(cls, total_rows: int, D: int, dtype: torch.dtype, want_lo: bool, device, group) -> "SymmetricBank":
        import torch.distributed as dist

        g = group if group is not None else dist.group.WORLD
        key = (total_rows, D, dtype, want_lo, str(device), g.group_name)
        if key not in cls._cache:
            if len(cls._cache) >= 4:               # shapes change rarely; do not hoard VMM mappings
                cls._cache.clear()
            cls._cache[key] = cls(total_rows, D, dtype, want_lo, device, g)
        return cls._cache[key]

    def __init__(self, total_rows: int, D: int, dtype: torch.dtype, want_lo: bool, device, group):
        import torch.distributed._symmetric_memory as symm

        self.group = group
        self.sets = []
        for _ in range(2):
            hi = symm.empty((total_rows, D), dtype=dtype, device=device)
            lo = symm.empty((total_rows, D), dtype=dtype, device=device) if want_lo else None
            n2 = symm.empty((total_rows,), dtype=torch.float32, device=device)
            handles = [None if t is None else symm.rendezvous(t, group) for t in (hi, lo, n2)]   # collective
            self.sets.append({"bufs": (hi, lo, n2), "handles": handles, "peers": {}})
        self.step = 0
        self.side = torch.cuda.Stream(device=device)
        self.device = device
        self.colmin = {}          # (rows, cols, dtype) -> two symmetric buffers for the column-minimum exchange

    def local_slices(self, row_a: int, row_b: int):
        """This step's (hi, lo, n2) slices for rows [row_a, row_b): the embed kernel writes into them."""
        hi, lo, n2 = self.sets[self.step & 1]["bufs"]
        return hi[row_a:row_b], None if lo is None else lo[row_a:row_b], n2[row_a:row_b]

    def _peer(self, cur, which: int, src: int):
        key = (which, src)
        if key not in cur["peers"]:
            buf = cur["bufs"][which]
            cur["peers"][key] = cur["handles"][which].get_buffer(src, tuple(buf.shape), buf.dtype)
        return cur["peers"][key]

    def publish_and_pull(self, bounds: Sequence[Tuple[int, int]], P: int, need_rank: Sequence[int], rank: int, world: int,
                         ready: torch.Tensor):
        """After the local slices were written on the current stream: barrier, then pull the shards of `need_rank`.
        ready [n_total] int32 (zeroed by the caller on the current stream): the flags of a shard's images are set to 1 on the
        side stream right after its copies -- the arrival flags of ac_min_dist_sym_ready.
        Returns ((hi_buf, lo_buf, n2_buf), requests): one request whose wait() orders the current stream after the last
        pull (the side stream runs in order, so after every pull), or none when nothing is pulled."""
        cur = self.sets[self.step & 1]
        self.step += 1
        main = torch.cuda.current_stream()
        cur["handles"][0].barrier(channel=0)              # stream-ordered: every rank's slice of this set is written
        self.side.wait_stream(main)
        pulled = False
        with torch.cuda.stream(self.side):
            for k in range(1, world):
                src = (rank + k) % world
                if src not in need_rank:
                    continue
                sa, sb = bounds[src]
                if sb <= sa:
                    continue
                for which, buf in enumerate(cur["bufs"]):
                    if buf is None:
                        continue
                    peer = self._peer(cur, which, src)
                    buf[sa * P : sb * P].copy_(peer[sa * P : sb * P], non_blocking=True)
                ready[sa:sb].fill_(1)
                pulled = True
        if not pulled:
            return cur["bufs"], []
        ev = torch.cuda.Event()
        ev.record(self.side)
        return cur["bufs"], [_EventRequest(ev)]

    # ---- column minima (symmetric form): every rank writes its [n_r, N*P] block straight into symmetric memory, and after ONE
    # barrier each rank pulls the columns that belong to its query rows from every peer.  Replaces the NCCL all_to_all of
    # distributed.exchange_colmin, which at 8 GPUs spent 48 us packing eight send blocks and 183 us in ncclDevKernel_SendRecv
    # for 0.5 MB per peer (timeline of round 2: 8 % of a config-2 step).
    def colmin_buffer(self, n_local: int, n_max: int, cols: int, dtype: torch.dtype) -> torch.Tensor:
        """This step's [n_local, cols] view of the symmetric column-minimum buffer (float minima, or int64 keys in the refined
        modes).  Call after publish_and_pull of the same step (the two sets alternate with the bank's)."""
        import torch.distributed._symmetric_memory as symm

        key = (n_max, cols, dtype)
        if key not in self.colmin:
            if len(self.colmin) >= 2:
                self.colmin.clear()
            sets = []
            for _ in range(2):
                buf = symm.empty((n_max, cols), dtype=dtype, device=self.device)
                sets.append({"buf": buf, "handle": symm.rendezvous(buf, self.group), "peers": {}})   # collective
            self.colmin[key] = sets
        cur = self.colmin[key][(self.step - 1) & 1]
        self._colmin_cur = cur
        return cur["buf"][:n_local]

    def exchange_colmin(self, bounds: Sequence[Tuple[int, int]], P: int, rank: int, world: int) -> torch.Tensor:
        """After the last distance launch of the step wrote colmin_buffer(): barrier, then [N, n_r*P] = for every bank image
        (owned by some rank) the minima over this rank's query rows, pulled from the peers' buffers."""
        cur = self._colmin_cur
        buf = cur["buf"]
        a_r, b_r = bounds[rank]
        n_total = bounds[-1][1]
        cur["handle"].barrier(channel=1)                  # stream-ordered: every rank's distance launches of this step are done
        out = torch.empty((n_total, (b_r - a_r) * P), dtype=buf.dtype, device=buf.device)
        dsts, srcs = [], []
        for src in range(world):
            sa, sb = bounds[src]
            if sb <= sa:
                continue
            if src == rank:
                peer = buf
            else:
                if src not in cur["peers"]:
                    cur["peers"][src] = cur["handle"].get_buffer(src, tuple(buf.shape), buf.dtype)
                peer = cur["peers"][src]
            dsts.append(out[sa:sb])
            srcs.append(peer[: sb - sa, a_r * P : b_r * P])
        if len(dsts) <= 16 and buf.element_size() % 4 == 0:
            from . import ops

            ops.copy_blocks(dsts, srcs)                   # one launch for all peers
        else:
            for d, s_ in zip(dsts, srcs):
                d.copy_(s_, non_blocking=True)
        return out
