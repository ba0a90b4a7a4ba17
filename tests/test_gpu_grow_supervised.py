"""B200: growing a supervised category (pipeline.GrowingSupervisedCategory and the running-minimum reduction
AC_REDUCE_MIN_UPDATE) against run_path from scratch on the same query and normal images, bit for bit."""
import pytest
import torch

from anomaly_clustering_b200 import ops, pipeline, synth

pytestmark = pytest.mark.gpu

SMALL = dict(layers=[(96, 12, 12, True), (96, 12, 12, True)], Dp=256, D=512)      # P = 144: query blocks cross images
TINY = dict(layers=[(96, 5, 5, True), (96, 5, 5, True)], Dp=160, D=320)          # P = 25, D not a multiple of 256
CONFIG3 = dict(layers=[(768, 28, 28, True), (768, 28, 28, True)], Dp=2048, D=4096)  # P = 784 (bench config 3)
FIELDS = ("Z", "w", "alpha64", "alpha32", "X", "Dmat")


@pytest.mark.parametrize("K", [1, 5])
@pytest.mark.parametrize("Mq", [61, 5 * 61, 1000])
def test_min_update_reduction_is_bit_exact(K, Mq):
    """w = min(w_in, min_j dmin[j]) with w_in holding +inf, values below every dmin and ordinary values; Mq not a multiple of
    the 256-row block.  MEAN and MIN give the bits of their reference reductions."""
    gen = torch.Generator().manual_seed(K * 1000 + Mq)
    dmin = (0.1 + torch.rand(K, Mq, generator=gen)).cuda()
    w_in = (0.1 + torch.rand(Mq, generator=gen))
    w_in[::3] = float("inf")
    w_in[1::5] = 0.01                                         # below every dmin: kept
    w_in = w_in.cuda()
    w = w_in.clone()
    got = ops.reduce_weights(dmin, 61, None, "min_update", out=w)
    torch.cuda.synchronize()
    assert got.data_ptr() == w.data_ptr()
    assert torch.equal(w, torch.minimum(w_in, dmin.min(0).values))
    assert torch.equal(ops.reduce_weights(dmin, 61, None, "min"), dmin.min(0).values)
    s = torch.zeros(Mq, device="cuda")
    for j in range(K):                                        # left-to-right fp32 sum, as the kernel adds
        s = s + dmin[j]
    # divided by a tensor: torch turns a division by a Python scalar into a multiplication by its reciprocal
    assert torch.equal(ops.reduce_weights(dmin, 61, None, "mean"), s / torch.full_like(s, K))


def test_min_update_reduction_keeps_the_meaning_of_q_self():
    """q_self names the bank image a query row skips, exactly as for AC_REDUCE_MIN."""
    nb, Pq = 6, 61
    Mq = 5 * Pq
    gen = torch.Generator().manual_seed(3)
    dmin = (0.1 + torch.rand(nb, Mq, generator=gen)).cuda()
    q_self = torch.tensor([0, -1, 3, 5, -1], dtype=torch.int32, device="cuda")
    w_in = (0.1 + torch.rand(Mq, generator=gen)).cuda()
    w = w_in.clone()
    ops.reduce_weights(dmin, Pq, q_self, "min_update", out=w)
    want = torch.minimum(w_in, ops.reduce_weights(dmin, Pq, q_self, "min"))
    torch.cuda.synchronize()
    assert torch.equal(w, want)


class _Run:
    """A growing category next to the images it has seen, checked against run_path from scratch after every call."""

    def __init__(self, cfg, taus, precision, keep_z, dtype=torch.float32, n=(16, 16), **kw):
        fq, _ = synth.planted_features(n[0], cfg["layers"], n_classes=3, seed=5)
        fb, _ = synth.planted_features(n[1], cfg["layers"], n_classes=1, seed=6)
        self.fq = [f.to(dtype).cuda() for f in fq]
        self.fb = [f.to(dtype).cuda() for f in fb]
        self.cfg, self.taus, self.precision, self.keep_z = cfg, taus, precision, keep_z
        self.g = pipeline.GrowingSupervisedCategory(3, 1, cfg["Dp"], cfg["D"], taus, precision=precision, keep_z=keep_z, **kw)
        self.nq = self.nb = 0

    def query(self, m):
        res = self.g.add([f[self.nq:self.nq + m] for f in self.fq])
        self.nq += m
        return self.check(res)

    def normal(self, k):
        res = self.g.add_normal([f[self.nb:self.nb + k] for f in self.fb])
        self.nb += k
        if self.nq == 0:
            assert res is None
            return None
        return self.check(res)

    def check(self, res):
        ref = pipeline.run_path([f[:self.nq] for f in self.fq], 3, 1, self.cfg["Dp"], self.cfg["D"], "supervised", self.taus,
                                bank_features=[f[:self.nb] for f in self.fb], precision=self.precision, keep_z=self.keep_z)
        torch.cuda.synchronize()
        assert self.g.n_img == self.nq and self.g.n_normal == self.nb
        for k in FIELDS:
            a, b = getattr(res, k), getattr(ref, k)
            assert (a is None) == (b is None), k
            if b is not None:
                assert a.shape == b.shape and a.dtype == b.dtype, k
                assert torch.equal(a, b), (k, self.nq, self.nb)
        return res


def _interleaved(run):
    run.normal(4)
    run.query(3)
    run.query(1)
    run.normal(2)
    run.query(2)
    run.normal(1)


VARIANTS = {
    "f16-zfree": ([1.0, 2.0], "f16", False, torch.float32),
    "f16-keepz": ([1.0, 2.0], "f16", True, torch.float32),
    "bf16": ([1.0], "bf16", False, torch.float32),
    "f16x3": ([0.5, 1.0], "f16x3", False, torch.float32),
    "auto-f16r": ([0.0, 0.1], "auto", False, torch.float32),
    "bf16-maps": ([1.0, 2.0], "f16", False, torch.bfloat16),
}


@pytest.mark.parametrize("cfg", [SMALL, TINY], ids=["P144", "P25"])
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_interleaved_growth_is_bit_identical_to_run_path(variant, cfg):
    """normal 4 -> query 3 -> query +1 -> normal +2 -> query +2 -> normal +1: every result equals run_path from scratch on the
    images so far in every field (Z when it is kept)."""
    taus, precision, keep_z, dtype = VARIANTS[variant]
    run = _Run(cfg, taus, precision, keep_z, dtype)
    if precision == "auto":
        assert run.g.precision == "f16r" and run.g.keep_z
    _interleaved(run)
    assert run.g.keep_z == (keep_z or precision == "auto")       # the Z-free X covers these shapes


def test_growth_at_the_config3_width_is_bit_identical_to_run_path():
    """bank 12, queries 6, query +1, normal +1, normal +5 at P = 784, D = 4096 (Z-free, f16)."""
    run = _Run(CONFIG3, [1.0], "f16", False, n=(7, 18))
    run.normal(12)
    run.query(6)
    run.query(1)
    run.normal(1)
    run.normal(5)


@pytest.mark.parametrize("precision", ["f16", "f16r"])
def test_regrowth_gives_identical_results(precision):
    """capacity = bank_capacity = 2: both sides are regrown twice (2 -> 4 -> 8) and give the bits of ample room."""
    out = []
    for cap in (2, 64):
        run = _Run(SMALL, [0.5, 1.0], precision, False, n=(6, 8), capacity=cap, bank_capacity=cap)
        res = [run.normal(1), run.query(1), run.query(2), run.normal(2), run.query(2), run.normal(3)]
        out.append(((run.g._q.capacity, run.g._bank.capacity), res))
    assert out[0][0] == (8, 8) and out[1][0] == (64, 64)
    for a, b in zip(out[0][1], out[1][1]):
        assert (a is None) == (b is None)
        if a is not None:
            for k in FIELDS:
                assert (getattr(a, k) is None) or torch.equal(getattr(a, k), getattr(b, k)), k


def test_results_are_not_changed_by_later_calls():
    run = _Run(SMALL, [1.0], "f16", False)
    run.normal(3)
    first = run.query(2)
    kept = {k: getattr(first, k).clone() for k in ("w", "alpha64", "X", "Dmat")}
    run.normal(2)
    run.query(1)
    torch.cuda.synchronize()
    for k, v in kept.items():
        assert torch.equal(getattr(first, k), v), k


def test_refusals_leave_the_state_unchanged():
    """Each refusal is a ValueError raised before anything is enqueued; the next valid call still matches run_path."""
    run = _Run(SMALL, [1.0], "f16", False)
    g = run.g
    with pytest.raises(ValueError, match="add_normal first"):
        g.add([f[:2] for f in run.fq])
    with pytest.raises(ValueError, match="non-zero number of images"):
        g.add_normal([f[:0] for f in run.fb])
    run.normal(3)
    run.query(2)
    other_c, _ = synth.planted_features(1, [(64, 12, 12, True), (96, 12, 12, True)], seed=1)
    other_grid, _ = synth.planted_features(1, [(96, 10, 10, True), (96, 10, 10, True)], seed=1)
    bad = [[f[:1] for f in run.fq[:1]], [f.cuda() for f in other_c], [f.cuda() for f in other_grid],
           [f[:1].to(torch.bfloat16) for f in run.fq]]
    for call in (g.add, g.add_normal):
        for b in bad:
            with pytest.raises(ValueError, match="differ from the first add"):
                call(b)
        with pytest.raises(ValueError, match="non-zero number of images"):
            call([run.fq[0][:2], run.fq[1][:3]])
        with pytest.raises(ValueError, match="non-zero number of images"):
            call([f[:0] for f in run.fq])
    assert g.n_img == 2 and g.n_normal == 3
    run.query(1)
    run.normal(1)
