"""Stage 1 (csrc/embed.cu) at its tiling and dispatch edges, against the float64 CPU reference.

Every expected value comes from oracle/restated.embed(..., dtype=torch.float64) on exactly the values the kernel reads (a
16-bit map enters as its exact float64 value), never from another GPU path.  That reference is itself pinned against the
unmodified reference's outputs in tests/test_embed_reference_cpu.py, which runs without a GPU.

Each case also proves which kernel form ran: the call runs once under torch.profiler (CUDA activities only, kernel names
read, nothing timed) and the test asserts the intended kernel and template instantiation.  Forms are forced only through
the library's test hooks (ac_debug_set key 2: kernel variant, key 9: lean fused kernel), reset after every test.

Tolerances (each one is restated beside its assert).  s = (|mean| + max|x - mean|) / sqrt(var + eps) of a map is its input
scale in LayerNorm units (without the LayerNorm: max|x|); s is the largest over the images and layers of a call.
  Z        |Z - Z64| <= 2e-6 + 2^-22 s        (fp32 LayerNorm of values of size s, then fp32 pooling sums)
  hi       |hi - Z64| <= ulp/2 of the operand type at |Z64| + the Z bound, plus the Z bound
  hi, lo   where Z is written as well: hi == round(Z) and lo == round(Z - hi) exactly
  n2       within 2e-6 relative of the float64 sum of squares of the operand rows the kernel wrote
  X        |X - X64| <= 2^-24 (H W / 4 + 64) sum|alpha| max|Z64| + (Z bound) sum|alpha|   per image
"""
import ctypes
import re

import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from anomaly_clustering_b200 import _lib, ops, pipeline
from oracle import restated

pytestmark = pytest.mark.gpu

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
TNAME = {F32: "float", BF16: "__nv_bfloat16", F16: "__half"}
OPDT = {"f16": F16, "bf16": BF16}


def _hooks(variant, lean):
    lib = _lib.load()
    assert lib.ac_debug_set(2, variant) == 0 and lib.ac_debug_set(9, lean) == 0


@pytest.fixture(autouse=True)
def _reset_hooks():
    _hooks(0, 1)
    yield
    _hooks(0, 1)


# ----------------------------------------------------------------------------------------------------------------- helpers
def kernels_of(fn):
    """(fn(), names of the CUDA kernels it launched, spaces removed)."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name.replace(" ", "") for e in prof.events()}


def assert_ran(names, *patterns):
    for pat in patterns:
        assert any(re.search(pat, n) for n in names), (pat, sorted(n for n in names if "kernel" in n))


def make_maps(B, layers, seed, mean=1.5, std=1.0, dtype=F32):
    """layers [(C, H, W, kind)] -> device maps: kind True = ViT tokens [B, 1+H*W, C] (CLS first), False = CNN [B, C, H, W],
    "cl" = channels_last [B, C, H, W] (channel-contiguous like tokens, any H x W).  Values N(mean, std^2): a non-zero mean
    makes the zero padding after the LayerNorm differ from padding the raw map."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for C, H, W, kind in layers:
        x = torch.randn(B, C, H, W, generator=g) * std + mean
        if kind == "cl":
            x = x.contiguous(memory_format=torch.channels_last)
        elif kind:
            x = torch.cat([torch.randn(B, 1, C, generator=g), x.flatten(2).transpose(1, 2)], 1)
        out.append(x.to("cuda", dtype))
    return out


def scale_of(feats, layernorm=True, eps=1e-5):
    s = 0.0
    for f in feats:
        v = ops.feature_view(f).double().cpu().flatten(1)
        if not layernorm:
            s = max(s, v.abs().max().item())
            continue
        m = v.mean(1, keepdim=True)
        sd = (v.var(1, unbiased=False, keepdim=True) + eps).sqrt()
        s = max(s, ((m.abs() + (v - m).abs().max(1, keepdim=True)[0]) / sd).max().item())
    return s


def z_bound(s):
    return 2e-6 + 2.0 ** -22 * s


def ref64(feats, ps, st, Dp, D, layernorm=True, eps=1e-5):
    return restated.embed([ops.feature_view(f).cpu() for f in feats], ps, st, Dp, D, layernorm=layernorm, eps=eps,
                          dtype=torch.float64)


def half_ulp(v, dt):
    """ulp/2 of operand type dt at magnitude v (float64 tensor)."""
    mant, emin = (10, -14) if dt == F16 else (7, -126)
    _, e = torch.frexp(v.clamp_min(2.0 ** emin))
    return torch.pow(2.0, (e - 1).clamp_min(emin).double() - mant) / 2


def run_embed(feats, ps, st, Dp, D, want_z=True, operand="f16", want_lo=False, layernorm=True, eps=1e-5, off=(0, 0, 0)):
    """ops.embed with caller buffers at element offsets off = (Z, hi, lo) of their storage (+ n2 when an operand is asked)."""
    v0 = ops.feature_view(feats[0])
    h, w = ops.patch_grid(v0.shape[2], v0.shape[3], ps, st)
    rows = v0.shape[0] * h * w

    def buf(dt, o):
        return torch.full((rows * D + o,), float("nan"), dtype=dt, device="cuda")[o:].view(rows, D)

    z = buf(F32, off[0]) if want_z else None
    hi = buf(OPDT[operand], off[1]) if operand else None
    lo = buf(OPDT[operand], off[2]) if operand and want_lo else None
    n2 = torch.full((rows,), float("nan"), device="cuda") if operand else None
    Z, Hi, Lo, _ = ops.embed(feats, ps, st, Dp, D, layernorm=layernorm, eps=eps, want_z=want_z, operand=operand,
                             want_lo=want_lo, out_z=z, out_hi=hi, out_lo=lo, out_n2=n2)
    return Z, Hi, Lo, n2


def check_outputs(outs, z64, zb, rows_mask=None):
    """Z, hi, lo, n2 of one call against the float64 reference (tolerances in the module docstring)."""
    Z, hi, lo, n2 = outs
    sel = (lambda t: t) if rows_mask is None else (lambda t: t[rows_mask])
    if Z is not None:
        err = (Z.double().cpu() - z64).abs()
        assert sel(err).max().item() <= zb, ("Z", sel(err).max().item(), zb)        # 2e-6 + 2^-22 s
    if hi is not None:
        dt = hi.dtype
        h = hi.cpu().double()
        lim = half_ulp(z64.abs() + zb, dt) + zb                                       # one operand rounding + the Z bound
        assert bool(sel(((h - z64).abs() <= lim)).all()), ("hi", sel((h - z64).abs() - lim).max().item())
        if Z is not None:
            assert torch.equal(hi, Z.to(dt))                                          # hi == round(Z)
            if lo is not None:
                assert torch.equal(lo, (Z - hi.float()).to(dt))                       # lo == round(Z - hi)
        if n2 is not None and rows_mask is None:
            v = h + lo.cpu().double() if lo is not None else h
            ref = (v * v).sum(1)
            rel = ((n2.cpu().double() - ref).abs() / ref.clamp_min(1e-30)).max().item()
            assert rel <= 2e-6, ("n2", rel)                                           # 2e-6 relative


def border_rows(B, h, w):
    y = torch.arange(h).view(h, 1).expand(h, w)
    x = torch.arange(w).view(1, w).expand(h, w)
    m = (y == 0) | (y == h - 1) | (x == 0) | (x == w - 1)
    return m.reshape(-1).repeat(B)


# -------------------------------------------------------------------------------------------------------------- lean kernel
LEAN_PAT = {8: (768, 2048, 128), 4: (768, 1024, 128), 16: (384, 2048, 64)}     # B of 27/B -> (C, Dp, threads)
LEAN = [  # (period B, Z written, map dtype, grid, batch, layers, extra)
    (8, True, F32, 1, 1, 1, ""), (8, False, BF16, 2, 2, 2, ""), (8, True, F16, 3, 3, 1, ""),
    (8, False, F32, 14, 2, 1, "noln"), (8, True, BF16, 16, 1, 1, ""), (8, False, F16, 17, 2, 1, ""),
    (4, True, F32, 32, 1, 1, ""), (4, False, BF16, 33, 1, 1, ""), (4, True, F16, 37, 1, 1, ""),
    (4, False, F32, 56, 1, 1, ""), (4, True, BF16, 28, 12, 1, ""), (4, False, F16, 14, 3, 1, "slice"),
    (16, True, F32, 14, 2, 2, ""), (16, False, BF16, 20, 2, 1, ""), (16, True, F16, 3, 2, 1, "noln"),
    (16, False, F32, 37, 1, 1, ""), (16, True, BF16, 56, 1, 1, ""), (16, False, F16, 17, 3, 1, ""),
]


@pytest.mark.parametrize("case", range(len(LEAN)), ids=lambda i: "27_%d-z%d-%s-g%d-b%d-l%d-%s" % (
    LEAN[i][0], LEAN[i][1], TNAME[LEAN[i][2]], LEAN[i][3], LEAN[i][4], LEAN[i][5], LEAN[i][6]))
def test_lean_fused_kernel(case):
    """Every instantiation of embed_fused_fast_kernel (3 periods x Z written or not x 3 map types), grids 1-56, B 1-12
    (grid 28, B 12: more work items than resident CTAs), layernorm=0, a batch slice [1:] and the CLS skip.  The rows on the
    map border (closed-form padding correction) are checked on their own as well."""
    pb, wz, dt, g, B, L, extra = LEAN[case]
    C, Dp, ft = LEAN_PAT[pb]
    ln = extra != "noln"
    feats = make_maps(B + (extra == "slice"), [(C, g, g, True)] * L, seed=case, mean=1.5, dtype=dt)
    if extra == "slice":
        feats = [f[1:] for f in feats]
    D = L * Dp
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, Dp, D, want_z=wz, layernorm=ln))
    assert_ran(names, r"embed_fused_fast_kernel<27,%d,1,%d,%s,7,%d,%s>" % (pb, ft, "true" if wz else "false",
                                                                          3 if ft == 128 else 5, TNAME[dt]))
    z64 = ref64(feats, 3, 1, Dp, D, layernorm=ln)
    zb = z_bound(scale_of(feats, ln))
    check_outputs(outs, z64, zb)
    check_outputs(outs, z64, zb, rows_mask=border_rows(B, g, g))


# --------------------------------------------------------------------------------------------------- general fused kernel
GEN_PAT = [(27, 4, 1, 32), (27, 8, 1, 64), (27, 16, 1, 128), (9, 1, 1, 24), (9, 2, 1, 48), (9, 4, 1, 96), (18, 1, 1, 12),
           (9, 2, 2, 48), (18, 2, 2, 24), (9, 4, 2, 96), (27, 8, 2, 64), (27, 16, 2, 128)]     # (A, B, R, Dp) at C = 24
GEN_HW = [(5, 1), (3, 16), (4, 17), (2, 33), (6, 6), (7, 2)]


@pytest.mark.parametrize("case", range(len(GEN_PAT)), ids=lambda i: "%d_%d_r%d" % GEN_PAT[i][:3])
def test_general_fused_kernel(case):
    """All 12 AC_PERIODIC_CASES in embed_fused_kernel: non-square grids with w0 in {1, 16, 17, 33}, B around the look-ahead
    of 2, hi + lo with fp16 and bf16 operands, fp32 and 16-bit maps."""
    A, Bp, R, Dp = GEN_PAT[case]
    dt = [F32, BF16, F16][case % 3]
    H, W = GEN_HW[case % len(GEN_HW)]
    B = 1 + case % 3
    L = 1 + case % 2
    D = L * Dp // R
    operand = ["f16", "bf16"][case % 2]
    feats = make_maps(B, [(24, H, W, "cl")] * L, seed=200 + case, dtype=dt)
    _hooks(0, 0)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, Dp, D, operand=operand, want_lo=True))
    assert_ran(names, r"embed_fused_kernel<%d,%d,%d,%s>" % (A, Bp, R, TNAME[dt]))
    check_outputs(outs, ref64(feats, 3, 1, Dp, D), z_bound(scale_of(feats)))


# ------------------------------------------------------------------------------------------------------- per-layer forms
@pytest.mark.parametrize("form,dt", [("tma", F32), ("tma", BF16), ("ldg", F16), ("ldg", F32)])
def test_periodic_per_layer_forms(form, dt):
    """embed_tma_kernel and embed_periodic_kernel (forced), channels_last maps; 16-bit maps go through the fp32 channel-contiguous copy."""
    feats = make_maps(3, [(24, 9, 11, "cl"), (24, 9, 11, "cl")], seed=11, dtype=dt)
    _hooks(3 if form == "tma" else 1, 1)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, 64, 128, want_lo=True))
    assert_ran(names, r"embed_tma_kernel<27,8,3,1>" if form == "tma" else r"embed_periodic_kernel<27,8,3,1>")
    check_outputs(outs, ref64(feats, 3, 1, 64, 128), z_bound(scale_of(feats)))


@pytest.mark.parametrize("g0,g1,dt", [(28, 14, F32), (28, 7, BF16), (27, 13, F16)])
def test_cnn_resampled_layers(g0, g1, dt):
    """CNN layouts: transpose to channel-contiguous scratch, pool at the layer's own grid, resample (upsample_store_kernel)."""
    feats = make_maps(2, [(24, g0, g0, False), (24, g1, g1, False)], seed=g1, dtype=dt)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, 24, 48, operand="bf16", want_lo=True))
    assert_ran(names, r"nchw_to_nhwc_kernel<", r"embed_tma_kernel<9,1,3,1>", r"upsample_store_kernel")
    check_outputs(outs, ref64(feats, 3, 1, 24, 48), z_bound(scale_of(feats)))


def _maxtaps(C, k, Dp, L, D):
    """Largest tap count of one output column (for_each_tap of csrc/embed.cu, fused Aggregator)."""
    agg_in = L * Dp
    best = 0
    for t in range(D):
        g0, g1 = (t * agg_in) // D, -((-(t + 1) * agg_in) // D)
        n = 0
        for gg in range(g0, g1):
            d = gg % Dp
            n += -((-(d + 1) * C * k * k) // Dp) - (d * C * k * k) // Dp
        best = max(best, n)
    return best


@pytest.mark.parametrize("C,Dp,bucket", [(4, 9, 5), (4, 4, 10), (16, 9, 18), (32, 10, 32), (64, 10, 0)])
def test_tap_kernel_buckets(C, Dp, bucket):
    """embed_kernel<MAXTAPS, RESAMPLE> at every MAXTAPS bucket, the second layer resampled (8 -> 4 grid)."""
    mt = _maxtaps(C, 3, Dp, 2, 2 * Dp)
    assert mt <= bucket if bucket else mt > 32
    feats = make_maps(2, [(C, 8, 8, False), (C, 4, 4, False)], seed=C + Dp, dtype=[F32, BF16][C % 3 == 1])
    _hooks(2, 1)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, Dp, 2 * Dp, want_lo=True))
    assert_ran(names, r"embed_kernel<%d,false>" % bucket, r"embed_kernel<%d,true>" % bucket)
    check_outputs(outs, ref64(feats, 3, 1, Dp, 2 * Dp), z_bound(scale_of(feats)))


GEOM = [  # (layers, B, patchsize, stride, Dp, D, map dtype)
    ([(8, 8, 8, False)], 2, 1, 1, 6, 6, F32),
    ([(6, 11, 9, False), (6, 6, 6, True)], 2, 5, 2, 40, 60, F16),
    ([(3, 1, 2, False)], 3, 7, 3, 20, 20, F32),                    # map smaller than the patch
    ([(5, 1, 1, False)], 2, 5, 3, 12, 12, BF16),
    ([(4, 7, 1, False)], 2, 3, 2, 16, 16, F32),
    ([(2, 9, 9, False)], 2, 3, 1, 40, 40, F32),                    # Dp > C k^2
]


@pytest.mark.parametrize("case", range(len(GEOM)))
def test_patch_geometries(case):
    """Patch sizes 1, 3, 5 and 7, strides 1-3, maps smaller than the patch (H = 1, W = 1 or 2), Dp > C k^2."""
    layers, B, ps, st, Dp, D, dt = GEOM[case]
    feats = make_maps(B, layers, seed=300 + case, dtype=dt)
    outs, names = kernels_of(lambda: run_embed(feats, ps, st, Dp, D, want_lo=True))
    assert_ran(names, r"embed_kernel<")
    check_outputs(outs, ref64(feats, ps, st, Dp, D), z_bound(scale_of(feats)))


@pytest.mark.parametrize("dt", [F32, BF16])
def test_straddling_aggregator_windows(dt):
    """D > L Dp with windows straddling the two layers: concat scratch, pool1d_kernel, split_operand and row_norms."""
    feats = make_maps(2, [(8, 6, 6, False), (8, 6, 6, True)], seed=5, dtype=dt)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, 10, 25, operand="bf16", want_lo=True))
    assert not ops.aggregator_fusable(2, 10, 25)
    assert_ran(names, r"pool1d_kernel", r"split_kernel<__nv_bfloat16>", r"row_norms_kernel<__nv_bfloat16>")
    check_outputs(outs, ref64(feats, 3, 1, 10, 25), z_bound(scale_of(feats)))


def test_plan_halves_chunks_and_segments():
    """C = 4096, Dp = 64: 576 taps per column; the staged tile does not fit until build_plan has halved the column chunk
    (512 -> 32) and then the row segment (16 -> 4): the on-the-fly tap kernel embed_kernel<0, false>."""
    feats = make_maps(1, [(4096, 16, 16, False)], seed=4096)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, 64, 64))
    assert_ran(names, r"embed_kernel<0,false>")
    check_outputs(outs, ref64(feats, 3, 1, 64, 64), z_bound(scale_of(feats)))


# ------------------------------------------------------------------------------------------------------------- statistics
@pytest.mark.parametrize("case", ["vector", "dense_scalar", "odd_offset", "channel_strided", "constant", "eps"])
def test_statistics_prepass_branches(case):
    """ln_stats_kernel: aligned 4-wide loads, the dense scalar loop (n % 128 != 0 or an image offset not a multiple of 4),
    the strided loop (a channel-strided view); a constant map and a non-default eps."""
    g = torch.Generator().manual_seed(17)
    eps = 1e-2 if case == "eps" else 1e-5
    if case == "vector":
        x = (torch.randn(2, 32, 8, 8, generator=g) + 0.7).cuda()                  # n = 2048 = 16 * 128
    elif case == "dense_scalar":
        x = (torch.randn(2, 24, 7, 7, generator=g) + 0.7).cuda()                  # n = 1176
    elif case == "odd_offset":
        x = (torch.randn(2 * 32 * 64 + 1, generator=g) + 0.7).cuda()[1:].view(2, 32, 8, 8)
    elif case == "channel_strided":
        x = (torch.randn(2, 64, 8, 8, generator=g) + 0.7).cuda()[:, ::2]
    elif case == "constant":
        x = torch.full((2, 32, 8, 8), 0.75, device="cuda")
    else:
        x = (torch.randn(2, 32, 8, 8, generator=g) * 0.1 + 0.3).cuda()
    feats = [x]
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, 96, 96, want_lo=True, eps=eps))
    assert_ran(names, r"ln_stats_kernel<float>")
    check_outputs(outs, ref64(feats, 3, 1, 96, 96, eps=eps), z_bound(scale_of(feats, eps=eps)))


PRODUCERS = {"prepass": ([(32, 12, 12, False)], 96, 96, (0, 1), r"ln_stats_kernel<float>"),
             "fused": ([(24, 12, 12, True)], 64, 64, (0, 0), r"embed_fused_kernel<27,8,1,float>"),
             "lean": ([(768, 14, 14, True)], 2048, 2048, (0, 1), r"embed_fused_fast_kernel<27,8,1,128,")}


@pytest.mark.parametrize("ratio", [0, 3, 30, 100])
@pytest.mark.parametrize("producer", sorted(PRODUCERS))
def test_statistics_large_common_offset(producer, ratio):
    """Maps N(ratio, 1): mean/std in {0, 3, 30, 100} through each of the three statistics producers.  The Z bound scales
    with s ~ ratio + 4, the precision a two-pass fp32 LayerNorm keeps."""
    layers, Dp, D, hooks, pat = PRODUCERS[producer]
    feats = make_maps(2, layers, seed=ratio, mean=float(ratio), std=1.0)
    _hooks(*hooks)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, Dp, D))
    assert_ran(names, pat)
    z64 = ref64(feats, 3, 1, Dp, D)
    zb = z_bound(scale_of(feats))
    err = (outs[0].double().cpu() - z64).abs().max().item()
    print("statistics producer=%s mean/std=%d max|Z-Z64|=%.3e bound=%.3e" % (producer, ratio, err, zb))
    check_outputs(outs, z64, zb)


# ------------------------------------------------------------------------------------------------------------ large batch
def test_batch_over_grid_z_limit():
    """B = 65 600 tiny CNN maps (C = 8, 3 x 3): the per-layer path and X from features split the batch at 65 535 images."""
    B = 65600
    feats = make_maps(B, [(8, 3, 3, False)], seed=65600)
    outs, names = kernels_of(lambda: run_embed(feats, 3, 1, 8, 8))
    assert_ran(names, r"ln_stats_kernel<float>", r"nchw_to_nhwc_kernel<float>")
    z64 = ref64(feats, 3, 1, 8, 8)
    check_outputs(outs, z64, z_bound(scale_of(feats)))
    alpha = torch.randn(B, 9, generator=torch.Generator().manual_seed(1))
    X = ops.weighted_embed_from_features(feats, alpha.cuda(), 3, 1, 8, 8)
    _check_x(X, alpha, z64.reshape(B, 9, 8), 3, 3, z_bound(scale_of(feats)))


# ----------------------------------------------------------------------------------------------------- X from the features
def _check_x(X, alpha, z64, H, W, zb):
    a = alpha.double().cpu()
    x64 = restated.weighted_embedding64(a, z64)
    sa = a.abs().sum(1, keepdim=True)
    # fp32 correlation sums over H W / 4 positions per row slice and the pooled taps, plus the Z error carried by alpha
    lim = 2.0 ** -24 * (H * W / 4 + 64) * sa * z64.abs().amax(dim=(1, 2)).unsqueeze(1) + zb * sa
    err = (X.double().cpu() - x64).abs()
    assert bool((err <= lim).all()), ("X", (err - lim).max().item())


XF = [  # (C, grid, L, tokens, Dp, D, B, map dtype, layernorm)
    (255, 1, 1, False, 64, 64, 2, F32, True),
    (257, 2, 2, True, 128, 128, 3, BF16, True),      # R = 2
    (1, 3, 3, False, 9, 27, 2, F32, False),
    (768, 28, 2, True, 2048, 4096, 2, BF16, True),
    (8, 110, 1, False, 16, 16, 2, F16, True),        # alpha tile over 48 KB
    (4, 224, 1, False, 12, 12, 1, F32, True),        # alpha tile just under 200 KB
]


def _alphas(B, h, w, seed):
    """One-hot on each corner and on two edge midpoints (unnormalised weight 2.5), then N(0, 1) (negative, unnormalised)."""
    spots = [(0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (0, w // 2), (h // 2, 0)]
    out = []
    for y, x in spots:
        a = torch.zeros(B, h, w)
        a[:, y, x] = 2.5
        out.append(a.reshape(B, -1))
    out.append(torch.randn(B, h * w, generator=torch.Generator().manual_seed(seed)))
    return out


@pytest.mark.parametrize("case", range(len(XF)))
def test_x_from_features(case):
    """xcorr_kernel + xpool_kernel: grids 1-3 (empty kXSplit row slices), 28, 110 and 224, C in {1, 255, 257, 768},
    L 1-3, R = 2, layernorm=0, 16-bit maps, alpha on corners and edges, negative and unnormalised, B > 1."""
    C, g, L, tok, Dp, D, B, dt, ln = XF[case]
    feats = make_maps(B, [(C, g, g, tok)] * L, seed=400 + case, dtype=dt)
    z64 = ref64(feats, 3, 1, Dp, D, layernorm=ln).reshape(B, g * g, D)
    zb = z_bound(scale_of(feats, ln))
    for i, a in enumerate(_alphas(B, g, g, case)):
        X, names = kernels_of(lambda: ops.weighted_embed_from_features(feats, a.cuda(), 3, 1, Dp, D, layernorm=ln))
        if i == 0:
            assert_ran(names, r"xcorr_kernel<3,%s>" % TNAME[dt], r"xpool_kernel")
        _check_x(X, a, z64, g, g, zb)


def test_z_free_falls_back_at_grid_225():
    """Grid 225: the alpha tile exceeds the 200 KB the X-from-features kernel stages, so keep_z=False must take the Z path
    and give the same bits as keep_z=True."""
    feats = make_maps(2, [(8, 225, 225, False)], seed=225)
    assert not pipeline.z_free_supported(feats, 3, 1, 8, 8, "f16")
    a = pipeline.run_path(feats, 3, 1, 8, 8, "average", keep_z=False)
    b = pipeline.run_path(feats, 3, 1, 8, 8, "average", keep_z=True)
    assert torch.equal(a.X, b.X) and torch.equal(a.alpha32, b.alpha32)


# ------------------------------------------------------------------------------------------------ misaligned output buffers
MISALIGNED = {  # form -> (layers, Dp, D, hooks, operand, want_lo, kernel of the misaligned call)
    "lean": ([(768, 14, 14, True)], 2048, 2048, (0, 1), "f16", False, r"embed_fused_kernel<27,8,1,float>"),
    "fused": ([(24, 5, 7, "cl")], 64, 64, (0, 0), "bf16", True, r"embed_fused_kernel<27,8,1,float>"),
    "tma": ([(24, 9, 9, True)], 64, 64, (3, 1), "f16", True, r"embed_tma_kernel<27,8,3,1>"),
    "ldg": ([(24, 9, 9, True)], 64, 64, (1, 1), "f16", True, r"embed_periodic_kernel<27,8,3,1>"),
    "taps": ([(16, 8, 8, False)], 24, 24, (2, 1), "f16", True, r"embed_kernel<"),
    "upsample": ([(24, 14, 14, False), (24, 7, 7, False)], 24, 48, (0, 1), "bf16", True, r"upsample_store_kernel"),
    "straddle": ([(8, 6, 6, False), (8, 6, 6, False)], 10, 25, (0, 1), "f16", True, r"split_kernel<"),
}


@pytest.mark.parametrize("off", [(1, 1, 1), (0, 0, 3)], ids=["all_odd", "lo_only"])
@pytest.mark.parametrize("form", sorted(MISALIGNED))
def test_misaligned_outputs_bit_identical(form, off):
    """Contiguous out_z / out_hi / out_lo at an odd element offset take scalar stores and write the bits an aligned buffer
    gets.  The lean kernel needs aligned outputs: the misaligned call runs the general fused kernel, compared with that
    kernel on aligned buffers."""
    layers, Dp, D, hooks, operand, want_lo, pat = MISALIGNED[form]
    feats = make_maps(2, layers, seed=99)
    if form == "lean" and off == (0, 0, 3):
        off = (0, 1, 0)                        # the lean kernel writes no lo: misalign hi instead
    _hooks(*((0, 0) if form == "lean" else hooks))
    ref = run_embed(feats, 3, 1, Dp, D, operand=operand, want_lo=want_lo)
    _hooks(*hooks)
    got, names = kernels_of(lambda: run_embed(feats, 3, 1, Dp, D, operand=operand, want_lo=want_lo, off=off))
    assert_ran(names, pat)
    for a, b in zip(ref, got):
        assert (a is None) == (b is None)
        if a is not None:
            assert torch.equal(a, b)


@pytest.mark.parametrize("form", sorted(MISALIGNED))
def test_misaligned_workspace_is_invalid(form):
    layers, Dp, D, hooks, operand, want_lo, _ = MISALIGNED[form]
    feats = make_maps(2, layers, seed=98)
    _hooks(*hooks)
    lib = _lib.load()
    views, arr, fdt = ops._layer_array(feats)
    v0 = views[0]
    rows = 2 * v0.shape[2] * v0.shape[3]
    Z = torch.empty(rows, D, device="cuda")
    hi = torch.empty(rows, D, dtype=OPDT[operand], device="cuda")
    n = lib.ac_embed_workspace_bytes_dt(arr, len(views), fdt, 2, 3, 1, Dp, D)
    ws = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    for o in (1, 8):
        rc = lib.ac_embed_dt(arr, len(views), fdt, 2, 3, 1, Dp, D, 1, 1e-5, ctypes.c_void_p(Z.data_ptr()),
                             ctypes.c_void_p(hi.data_ptr()), None, _lib.AC_DT_F16 if operand == "f16" else _lib.AC_DT_BF16, None,
                             ctypes.c_void_p(ws.data_ptr() + o), n, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == _lib.AC_ERR_INVALID
    torch.cuda.synchronize()
