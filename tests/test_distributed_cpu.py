"""CPU: host-side sharding logic of the multi-GPU path, world_size 2 over gloo.  The compute
back-end is replaced by the oracle HERE ONLY (the product default is the CUDA library); what is
tested is shard bounds, uneven all-gather + compaction, self-exclusion with global image ids and
the gather order of X."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from anomaly_clustering_b200 import distributed, pipeline

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pair_ownership_covers_every_pair_once():
    for n in (1, 2, 3, 4, 5, 8, 9, 100):
        for i in range(n):
            assert not distributed.pair_owned(i, i, n)
            for j in range(i + 1, n):
                assert distributed.pair_owned(i, j, n) != distributed.pair_owned(j, i, n)
        if n > 1:
            per_image = [sum(distributed.pair_owned(i, j, n) for j in range(n)) for i in range(n)]
            assert max(per_image) - min(per_image) <= 1     # balanced: each image owns ~(n-1)/2 pairs


def test_needed_shards_cover_owned_pairs_only():
    for n, world in ((100, 8), (13, 2), (21, 4), (5, 3), (1210, 8)):
        bounds = distributed.shard_bounds(n, world)
        need = distributed.needed_shards(bounds, n)
        owner = [r for r, (a, b) in enumerate(bounds) for _ in range(a, b)]
        step = max(1, n // 60)
        for r, (a, b) in enumerate(bounds):
            want = {owner[j] for i in range(a, b, step) for j in range(n) if distributed.pair_owned(i, j, n)} - {r}
            assert want <= set(need[r])
            assert r not in need[r]
        if world == 8 and n == 100:
            assert max(len(x) for x in need) <= 5      # about half of the 7 other ranks


def test_shard_bounds_and_lpt():
    assert distributed.shard_bounds(100, 8) == [(0, 13), (13, 26), (26, 39), (39, 52), (52, 64), (64, 76), (76, 88), (88, 100)]
    assert distributed.shard_bounds(3, 4) == [(0, 1), (1, 2), (2, 3), (3, 3)]
    counts = [83, 150, 132, 110, 115, 167, 160, 42, 100, 151]          # MVTec object test-set sizes (SURVEY 8d)
    costs = [n * (n - 1) for n in counts]
    bins = distributed.lpt_assign(costs, 4)
    assert sorted(i for b in bins for i in b) == list(range(10))
    loads = [sum(costs[i] for i in b) for b in bins]
    assert max(loads) / (sum(loads) / 4) < 1.25                           # imbalance bound quoted in SURVEY 8e


def test_all_tau_weighted_embed_uses_the_fused_form_when_the_backend_has_it():
    """distributed._weighted_embed_all_taus: [n_r, T, D] from one pass over Z when the compute back-end offers
    weighted_embed_multi (the CUDA library), else one weighted_embed per tau -- same numbers either way."""
    gen = torch.Generator().manual_seed(3)
    T, n, P, D = 4, 3, 10, 8
    a32 = torch.softmax(torch.randn(T, n, P, generator=gen), dim=2)
    Z3 = torch.randn(n, P, D, generator=gen)
    calls = []

    class PerTau:
        @staticmethod
        def weighted_embed(a, Z):
            calls.append("one")
            return torch.bmm(a.reshape(n, 1, P), Z).reshape(n, D)

    class Fused(PerTau):
        @staticmethod
        def weighted_embed_multi(a, Z):
            calls.append("multi")
            return torch.einsum("tnp,npd->tnd", a, Z)

    x1 = distributed._weighted_embed_all_taus(PerTau, a32, Z3, T)
    assert calls == ["one"] * T and x1.shape == (n, T, D)
    calls.clear()
    x2 = distributed._weighted_embed_all_taus(Fused, a32, Z3, T)
    assert calls == ["multi"] and x2.shape == (n, T, D) and x2.is_contiguous()
    assert torch.allclose(x1, x2, atol=1e-6)


class _OracleCompute:
    """Stand-in compute for the CPU test (oracle arithmetic on CPU tensors)."""

    @staticmethod
    def embed_images(features, patchsize, stride, Dp, D, precision, want_z=True, out=None):
        """`out` = (hi, lo, n2) slices to write the operands into, as pipeline.embed_images takes them."""
        from oracle import restated

        Z = restated.embed(features, patchsize, stride, Dp, D)
        n = features[0].shape[0]
        P = Z.shape[0] // n
        if out is None:
            return pipeline.PatchSet(n, P, D, (0, 0), Z=Z, hi=Z.clone(), lo=None, n2=(Z * Z).sum(1))
        hi, lo, n2 = out
        assert lo is None
        hi.copy_(Z)
        n2.copy_((Z * Z).sum(1))
        return pipeline.PatchSet(n, P, D, (0, 0), Z=Z, hi=hi, lo=None, n2=n2)

    @staticmethod
    def min_distance_weights(q, bank, mode, precision, q_self=None):
        from oracle import restated

        dm = restated.per_image_min_dist(q.Z.reshape(q.n_img, q.P, q.D), bank.hi.reshape(bank.n_img, bank.P, bank.D))
        w = torch.empty(q.n_img, q.P)
        for i in range(q.n_img):
            if mode == "supervised":                    # utils.py:236: min over the bank images
                w[i] = dm[i].min(dim=1)[0]
                continue
            keep = torch.ones(bank.n_img, dtype=torch.bool)
            keep[int(q_self[i])] = False
            w[i] = dm[i][:, keep].mean(dim=1)
        return w

    launches = []                    # (begin, count, with arrival flags) of the min_dist_sym calls, for the schedule assertions

    @staticmethod
    def min_dist_sym(Qhi, Qlo, Qn2, q_img0, Bhi, Blo, Bn2, nb_img, P, precision, bank_window=None, init=True, out=None,
                     ready=None):
        """What ac_min_dist_sym produces: squared minima only for the pairs the query image owns, restricted
        to the circular bank-image window, written into `out` when it is given.  Only the bank images of owned
        pairs are read, and with `ready` each of them must be flagged; rows of other bank images may still be in
        flight or never arrive (NaN in the symmetric-memory test), and the NaN initialisation of rowmin makes
        an entry the launch should have written but did not fail the comparison."""
        nq = Qhi.shape[0] // P
        begin, count = bank_window if bank_window is not None else (0, nb_img)
        _OracleCompute.launches.append((int(begin), int(count), ready is not None))
        if out is None:
            out = (torch.empty(nb_img, nq * P), torch.empty(nq, nb_img * P))
        rowmin, colmin = out
        if init:
            rowmin.fill_(float("nan"))
            colmin.fill_(3.0e38)
        for j in [(begin + t) % nb_img for t in range(count)]:
            for il in range(nq):
                if distributed.pair_owned(q_img0 + il, j, nb_img):
                    assert ready is None or int(ready[j]) == 1, "bank image %d read before its arrival flag" % j
                    d2 = torch.cdist(Qhi[il * P:(il + 1) * P].double(), Bhi[j * P:(j + 1) * P].double()).pow(2).float()
                    rowmin[j, il * P:(il + 1) * P] = d2.min(dim=1)[0]
                    colmin[il, j * P:(j + 1) * P] = torch.minimum(colmin[il, j * P:(j + 1) * P], d2.min(dim=0)[0])
        return rowmin, colmin

    @staticmethod
    def reduce_weights_sym(rowmin, colfull, P, q_img0):
        nb_img, Mq = rowmin.shape
        w = torch.empty(Mq)
        for r in range(Mq):
            i = q_img0 + r // P
            vals = [(rowmin[j, r] if distributed.pair_owned(i, j, nb_img) else colfull[j, r]).sqrt() for j in range(nb_img) if j != i]
            w[r] = torch.stack(vals).mean()
        return w

    @staticmethod
    def alpha(w, taus):
        from oracle import restated

        a = torch.stack([restated.alpha_from_weights(w, t, stable=True) for t in taus])
        return a, a.float()

    @staticmethod
    def weighted_embed(a32, Z3):
        return torch.bmm(a32.unsqueeze(1), Z3).squeeze(1)

    @staticmethod
    def pairwise_l2(X):
        return torch.cdist(X.double(), X.double()).float()


class _NoWait:
    @staticmethod
    def wait():
        pass


class _FakeSymmetricBank:
    """CPU stand-in for symm_transport.SymmetricBank over gloo.  The whole-bank buffers start as NaN; publish_and_pull
    all-gathers the shards but copies in only those listed in need_rank and flags only their images, so a read of a
    shard the schedule did not ask for fails the comparison."""

    def __init__(self, rows, D, group):
        self.group = group
        self.bufs = (torch.full((rows, D), float("nan")), None, torch.full((rows,), float("nan")))
        self.need_rank = None

    def local_slices(self, row_a, row_b):
        hi, lo, n2 = self.bufs
        return hi[row_a:row_b], None, n2[row_a:row_b]

    def publish_and_pull(self, bounds, P, need_rank, rank, world, ready):
        self.need_rank = list(need_rank)
        a, b = bounds[rank]
        counts = [(sb - sa) * P for sa, sb in bounds]
        for buf in (self.bufs[0], self.bufs[2]):
            full = distributed.all_gather_rows(buf[a * P:b * P], counts, self.group)
            for src in need_rank:
                sa, sb = bounds[src]
                buf[sa * P:sb * P] = full[sa * P:sb * P]
        for src in need_rank:
            ready[bounds[src][0]:bounds[src][1]] = 1
        return self.bufs, [_NoWait()]

    def colmin_buffer(self, n_local, n_max, cols, dtype):
        self.colmin = torch.empty(n_local, cols, dtype=dtype)
        return self.colmin

    def exchange_colmin(self, bounds, P, rank, world):
        return distributed.exchange_colmin(self.colmin, bounds, P, self.group)


def _worker(rank, world, port, n_total, tmp, symm_memory=False):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from anomaly_clustering_b200 import synth

    banks = []
    if symm_memory:     # the symmetric-memory schedule, which the oracle back-end on gloo would otherwise never select
        def fake_symmetric_bank(compute, rows, D, precision, device, group):
            banks.append(_FakeSymmetricBank(rows, D, group))
            return banks[-1]

        distributed._symmetric_bank = fake_symmetric_bank
    feats, _ = synth.planted_features(n_total, [(12, 6, 6, True), (12, 6, 6, True)], seed=3)
    lo, hi = distributed.shard_bounds(n_total, world)[rank]
    if n_total < world:     # empty shards are refused on every rank, before any collective
        with pytest.raises(ValueError, match="empty shards"):
            distributed.run_path_sharded([f[lo:hi] for f in feats], n_total, 3, 1, 32, 64, [1.0], precision="f16", compute=_OracleCompute)
        dist.destroy_process_group()
        return
    # uneven all-gather of row blocks
    local = torch.arange(lo, hi, dtype=torch.float32).reshape(-1, 1).repeat(1, 3)
    allr = distributed.all_gather_rows(local, [b - a for a, b in distributed.shard_bounds(n_total, world)])
    assert torch.equal(allr[:, 0], torch.arange(n_total, dtype=torch.float32))
    a64, X, Dm, w = distributed.run_path_sharded([f[lo:hi] for f in feats], n_total, 3, 1, 32, 64, [1.0, 2.0], precision="f16",
                                                 compute=_OracleCompute, symmetric=True)
    launches = list(_OracleCompute.launches)
    if symm_memory:
        assert len(banks) == 1 and banks[0].need_rank == distributed.needed_shards(distributed.shard_bounds(n_total, world), n_total)[rank]
    _, _, _, w_full = distributed.run_path_sharded([f[lo:hi] for f in feats], n_total, 3, 1, 32, 64, [1.0], precision="f16",
                                                   compute=_OracleCompute, symmetric=False)
    assert (w - w_full).abs().max().item() <= 1e-4      # symmetric exchange == straightforward all-pairs
    np.savez(os.path.join(tmp, "r%d.npz" % rank), a=a64.numpy(), X=X.numpy(), D=Dm.numpy(), w=w.numpy(),
             launches=np.asarray(launches, dtype=np.int64).reshape(-1, 3))
    dist.destroy_process_group()


def _check_against_single_process(tmp, n_total, world, expected_launches):
    """Every rank's w, alpha, X and Dmat against the oracle run on all images in one process; each rank's min_dist_sym
    calls against expected_launches(rank) = [(begin, count, with arrival flags), ...]."""
    from oracle import restated

    from anomaly_clustering_b200 import synth

    feats, _ = synth.planted_features(n_total, [(12, 6, 6, True), (12, 6, 6, True)], seed=3)
    Z = restated.embed(feats, 3, 1, 32, 64).reshape(n_total, -1, 64)
    w = restated.weight_distance_unsupervised(Z)
    bounds = distributed.shard_bounds(n_total, world)
    for r in range(world):
        g = np.load(os.path.join(tmp, "r%d.npz" % r))
        lo, hi = bounds[r]
        assert [tuple(x) for x in g["launches"]] == expected_launches(r)
        assert np.abs(g["w"] - w[lo:hi].numpy()).max() <= 1e-5
        for ti, tau in enumerate([1.0, 2.0]):
            a = restated.alpha_from_weights(w, tau)
            assert np.abs(g["a"][ti] - a[lo:hi].numpy()).max() <= 1e-6
            X = restated.weighted_embedding(a, Z)
            assert np.abs(g["X"][ti] - X).max() <= 1e-5           # every rank holds ALL X rows, in global order
            assert np.abs(g["D"][ti] - restated.pairwise_euclidean(X)).max() <= 1e-4


@pytest.mark.timeout(600)
@pytest.mark.parametrize("n_total,world", [(3, 2), (4, 4), (5, 2), (7, 3), (9, 4), (6, 4), (3, 4)])
def test_sharded_path_matches_single_process(tmp_path, n_total, world):
    """NCCL-collective schedule over gloo, uneven shards (2+1, 3+2, 3+2+2, 3+2+2+2, 2+2+1+1; 1+1+1+0 has an EMPTY rank and
    must be refused).  A rank with more than one image runs the two-phase schedule: the local shard's pairs while the remote
    shards are still in flight, then the remote bank images.  A rank with one image (rank 1 of (3, 2), every rank of (4, 4),
    ranks 2 and 3 of (6, 4)) has no pair inside its shard and runs one launch over the whole bank."""
    port = 29500 + (os.getpid() * 7 + n_total * 13 + world * 101) % 2000
    mp.spawn(_worker, args=(world, port, n_total, str(tmp_path)), nprocs=world, join=True)
    if n_total < world:
        return
    bounds = distributed.shard_bounds(n_total, world)

    def expected(r):
        lo, hi = bounds[r]
        if hi - lo > 1:
            return [(lo, hi - lo, False), (hi % n_total, n_total - (hi - lo), False)]
        return [(0, n_total, False)]

    _check_against_single_process(str(tmp_path), n_total, world, expected)


@pytest.mark.timeout(600)
@pytest.mark.parametrize("n_total,world", [(5, 2), (4, 4), (9, 4)])
def test_symmetric_memory_schedule_matches_single_process(tmp_path, n_total, world):
    """The symmetric-memory schedule (the default on a multi-GPU node) with a stand-in bank over gloo: the operands are
    embedded into the bank's slices, only the needed shards are pulled and flagged, ONE distance launch covers the whole
    bank and reads only flagged bank images, and the column minima come back through the bank's exchange.  The refined
    modes stay uncovered here: the oracle back-end has no arg-min or refine."""
    port = 29500 + (os.getpid() * 11 + n_total * 17 + world * 131 + 1000) % 2000
    mp.spawn(_worker, args=(world, port, n_total, str(tmp_path), True), nprocs=world, join=True)
    _check_against_single_process(str(tmp_path), n_total, world, lambda r: [(0, n_total, True)])


def _worker_supervised(rank, world, port, n_total, n_bank, overlap, tmp):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from anomaly_clustering_b200 import synth

    layers = [(12, 6, 6, True), (12, 6, 6, True)]
    feats, _ = synth.planted_features(n_total, layers, seed=3)
    bank, _ = synth.planted_features(n_bank, layers, seed=11)
    (lo, hi), (blo, bhi) = distributed.shard_bounds(n_total, world)[rank], distributed.shard_bounds(n_bank, world)[rank]
    a64, X, Dm, w = distributed.run_path_sharded_supervised([f[lo:hi] for f in feats], n_total, [f[blo:bhi] for f in bank], n_bank,
                                                            3, 1, 32, 64, [1.0, 2.0], precision="f16", compute=_OracleCompute,
                                                            overlap=overlap)
    np.savez(os.path.join(tmp, "r%d.npz" % rank), a=a64.numpy(), X=X.numpy(), D=Dm.numpy(), w=w.numpy())
    cats, bins = distributed.run_categories_sharded([83, 150, 132, 110, 115], lambda c: c * 10)
    assert cats == {c: c * 10 for c in bins[rank]} and sorted(c for b in bins for c in b) == [0, 1, 2, 3, 4]
    dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("n_total,n_bank,world,overlap", [(5, 7, 2, True), (5, 7, 2, False), (4, 5, 3, True)])
def test_supervised_sharded_matches_single_process(tmp_path, n_total, n_bank, world, overlap):
    """Queries and the normal-image bank both sharded unevenly; w = min over ALL bank images whichever rank
    embedded them, with the local bank shard multiplied before the gather completes."""
    from oracle import restated

    from anomaly_clustering_b200 import synth

    port = 29500 + (os.getpid() * 5 + n_total * 17 + n_bank * 29 + world * 211 + int(overlap)) % 2000
    mp.spawn(_worker_supervised, args=(world, port, n_total, n_bank, overlap, str(tmp_path)), nprocs=world, join=True)
    layers = [(12, 6, 6, True), (12, 6, 6, True)]
    feats, _ = synth.planted_features(n_total, layers, seed=3)
    bank, _ = synth.planted_features(n_bank, layers, seed=11)
    Z = restated.embed(feats, 3, 1, 32, 64).reshape(n_total, -1, 64)
    Zb = restated.embed(bank, 3, 1, 32, 64).reshape(n_bank, -1, 64)
    w = restated.weight_distance_supervised(Z, Zb)
    bounds = distributed.shard_bounds(n_total, world)
    for r in range(world):
        g = np.load(os.path.join(str(tmp_path), "r%d.npz" % r))
        lo, hi = bounds[r]
        assert np.abs(g["w"] - w[lo:hi].numpy()).max() <= 1e-5
        for ti, tau in enumerate([1.0, 2.0]):
            a = restated.alpha_from_weights(w, tau)
            assert np.abs(g["a"][ti] - a[lo:hi].numpy()).max() <= 1e-6
            X = restated.weighted_embedding(a, Z)
            assert np.abs(g["X"][ti] - X).max() <= 1e-5
            assert np.abs(g["D"][ti] - restated.pairwise_euclidean(X)).max() <= 1e-4
