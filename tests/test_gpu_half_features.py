"""GPU: bf16 / fp16 feature maps read natively by the embed and X-from-features kernels.

A 16-bit value has an exact fp32 value and everything from the LayerNorm on runs in fp32, so every output of the 16-bit
path must be BIT-IDENTICAL (torch.equal) to the fp32 path run on the upcast maps, with the same slicing applied to both.
Each embed form is forced through the test hooks (ac_debug_set 2 / 9) for both inputs."""
import os
import subprocess
import sys

import pytest
import torch

from anomaly_clustering_b200 import _lib, ops, pipeline, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

HALF = [torch.bfloat16, torch.float16]
# form -> (ac_debug_set key 2, key 9)
FORMS = {"lean": (0, 1), "fused": (0, 0), "tma": (3, 1), "ldg": (1, 1), "taps": (2, 1)}


def _hooks(variant, lean):
    lib = _lib.load()
    assert lib.ac_debug_set(2, variant) == 0 and lib.ac_debug_set(9, lean) == 0


@pytest.fixture(autouse=True)
def _reset_hooks():
    yield
    _hooks(0, 1)


def _pair(feats, dt, offset=0.0):
    """(16-bit device maps, their fp32 upcast): the reference is computed from exactly the values the 16-bit run reads."""
    x16 = [(f + offset).to("cuda", dt) for f in feats]
    return x16, [x.float() for x in x16]


def _embed(f, ps, st, Dp, D, want_z, want_lo, layernorm=True):
    rows = f[0].shape[0] * ops.patch_grid(*ops.feature_view(f[0]).shape[2:], ps, st)[0] * ops.patch_grid(
        *ops.feature_view(f[0]).shape[2:], ps, st)[1]
    n2 = torch.empty(rows, dtype=torch.float32, device="cuda")
    Z, hi, lo, _ = ops.embed(f, ps, st, Dp, D, layernorm=layernorm, want_z=want_z, operand="f16", want_lo=want_lo, out_n2=n2)
    return [t for t in (Z, hi, lo, n2) if t is not None]


def _assert_same(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.dtype == y.dtype and x.shape == y.shape, i
        assert torch.equal(x, y), (i, (x.float() - y.float()).abs().max().item())


VIT_SHAPES = {"config2": ([(768, 28, 28, True), (768, 28, 28, True)], 2048, 4096),
              "ragged17": ([(768, 17, 17, True), (768, 17, 17, True)], 2048, 4096),
              "vits_config5": ([(384, 20, 20, True), (384, 20, 20, True)], 2048, 4096),
              "one_layer_27_4": ([(768, 12, 12, True)], 1024, 1024)}


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("shape", sorted(VIT_SHAPES))
@pytest.mark.parametrize("form", sorted(FORMS))
def test_embed_forms_bit_identical(form, shape, dt):
    """Z (with and without), hi, lo and n2 of every embed form on token maps; batch slice [1:] and the CLS skip."""
    layers, Dp, D = VIT_SHAPES[shape]
    feats, _ = synth.planted_features(4, layers, seed=77)
    x16, x32 = _pair(feats, dt, offset=2.5)
    x16, x32 = [x[1:] for x in x16], [x[1:] for x in x32]
    _hooks(*FORMS[form])
    for want_z in (True, False):
        want_lo = form != "lean"          # the lean kernel writes hi + norms only
        _assert_same(_embed(x16, 3, 1, Dp, D, want_z, want_lo), _embed(x32, 3, 1, Dp, D, want_z, want_lo))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("form", ["auto", "tma", "ldg", "taps"])
def test_embed_cnn_pyramid_bit_identical(form, channels_last, dt):
    """Config-1 geometry (WRN50 layer2 + layer3: the second layer is resampled), NCHW and channels_last."""
    feats, _ = synth.planted_features(3, [(512, 28, 28, False), (1024, 14, 14, False)], seed=5)
    x16, x32 = _pair(feats, dt)
    if channels_last:
        x16 = [x.contiguous(memory_format=torch.channels_last) for x in x16]
        x32 = [x.contiguous(memory_format=torch.channels_last) for x in x32]
    _hooks(*({"auto": (0, 1)}.get(form) or FORMS[form]))
    _assert_same(_embed(x16, 3, 1, 1024, 1024, True, True), _embed(x32, 3, 1, 1024, 1024, True, True))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("case", ["straddle", "k5s2", "no_layernorm", "constant"])
def test_embed_other_shapes_bit_identical(case, dt):
    layers = [(32, 10, 10, True), (32, 10, 10, False)]
    feats, _ = synth.planted_features(3, layers, seed=9)
    if case == "constant":
        feats = [torch.full_like(f, 0.75) for f in feats]
    x16, x32 = _pair(feats, dt, offset=1.0)
    ps, st, Dp, D, ln = {"straddle": (3, 1, 96, 128, True), "k5s2": (5, 2, 64, 64, True), "no_layernorm": (3, 1, 96, 96, False),
                         "constant": (3, 1, 96, 96, True)}[case]
    _assert_same(_embed(x16, ps, st, Dp, D, True, True, layernorm=ln), _embed(x32, ps, st, Dp, D, True, True, layernorm=ln))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("elem_offset", [1, 2, 4])
def test_embed_image_base_offsets_bit_identical(elem_offset, dt):
    """An image base whose element offset is not a multiple of 4 takes the scalar branch of the statistics pre-pass for both
    inputs (the branch follows the element offset, not the byte alignment of the 16-bit pointer)."""
    B, C, H, W = 3, 32, 8, 8                       # C*H*W = 2048: a multiple of 4 * 32 statistics slices
    buf = (torch.randn(B * C * H * W + elem_offset, generator=torch.Generator().manual_seed(elem_offset)) + 0.5).to("cuda", dt)
    x16 = buf[elem_offset:].view(B, C, H, W)
    x32 = buf.float()[elem_offset:].view(B, C, H, W)
    _assert_same(_embed([x16], 3, 1, 96, 96, True, True), _embed([x32], 3, 1, 96, 96, True, True))
    # token layout with the same offsets
    t16 = buf[elem_offset:].view(B, H * W, C)
    t32 = buf.float()[elem_offset:].view(B, H * W, C)
    v16 = t16.unflatten(1, (H, W)).permute(0, 3, 1, 2)
    v32 = t32.unflatten(1, (H, W)).permute(0, 3, 1, 2)
    _assert_same(_embed([v16], 3, 1, 96, 96, True, True), _embed([v32], 3, 1, 96, 96, True, True))


@pytest.mark.parametrize("dt", HALF)
def test_embed_c_not_multiple_of_8_token_layer(dt):
    """C = 12: 16-byte rows for fp32 (the fused forms take it) but not for 16-bit elements, so the 16-bit map takes the
    per-layer LDG form; it matches the fp32 path forced into that form."""
    layers, Dp, D = [(12, 10, 10, True), (12, 10, 10, True)], 48, 96
    feats, _ = synth.planted_features(3, layers, seed=12)
    x16, x32 = _pair(feats, dt, offset=1.5)
    got = _embed(x16, 3, 1, Dp, D, True, True)
    _hooks(*FORMS["ldg"])
    _assert_same(got, _embed(x32, 3, 1, Dp, D, True, True))
    _assert_same(got, _embed(x16, 3, 1, Dp, D, True, True))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("layers,Dp,D", [([(768, 28, 28, True), (768, 28, 28, True)], 2048, 4096),
                                         ([(64, 12, 12, False), (64, 12, 12, False)], 128, 128)])
def test_weighted_embed_from_features_bit_identical(layers, Dp, D, dt):
    feats, _ = synth.planted_features(4, layers, seed=21)
    x16, x32 = _pair(feats, dt, offset=0.5)
    P = ops.feature_view(x16[0]).shape[2] * ops.feature_view(x16[0]).shape[3]
    a = torch.rand(4, P, generator=torch.Generator().manual_seed(1)).cuda()
    a = a / a.sum(1, keepdim=True)
    _assert_same([ops.weighted_embed_from_features(x16, a, 3, 1, Dp, D)], [ops.weighted_embed_from_features(x32, a, 3, 1, Dp, D)])


def _path_same(a, b):
    for name in ("w", "alpha64", "alpha32", "X", "Dmat", "Z"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None), name
        if x is not None:
            assert torch.equal(x, y), name


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("precision,taus", [("f16", [1.0]), ("f16r", [0.0, 0.5, 1.0])])
@pytest.mark.parametrize("keep_z", [True, False])
def test_run_path_unsupervised_bit_identical(precision, taus, keep_z, dt):
    feats, _ = synth.planted_features(6, [(768, 28, 28, True), (768, 28, 28, True)], seed=2023)
    x16, x32 = _pair(feats, dt)
    a = pipeline.run_path(x16, 3, 1, 2048, 4096, "unsupervised", taus, precision=precision, keep_z=keep_z)
    b = pipeline.run_path(x32, 3, 1, 2048, 4096, "unsupervised", taus, precision=precision, keep_z=keep_z)
    _path_same(a, b)


@pytest.mark.parametrize("dt", HALF)
def test_run_path_supervised_average_and_categories_bit_identical(dt):
    layers = [(768, 28, 28, True), (768, 28, 28, True)]
    feats, _ = synth.planted_features(5, layers, seed=3)
    bank, _ = synth.planted_features(4, layers, n_classes=1, seed=4)
    x16, x32 = _pair(feats, dt)
    b16, b32 = _pair(bank, dt)
    _path_same(pipeline.run_path(x16, 3, 1, 2048, 4096, "supervised", [2.0], bank_features=b16, precision="f16"),
               pipeline.run_path(x32, 3, 1, 2048, 4096, "supervised", [2.0], bank_features=b32, precision="f16"))
    _path_same(pipeline.run_path(x16, 3, 1, 2048, 4096, "average", keep_z=False),
               pipeline.run_path(x32, 3, 1, 2048, 4096, "average", keep_z=False))
    small = [(96, 12, 12, True), (96, 12, 12, True)]
    sizes = [4, 3, 5]
    cf, _ = synth.planted_features(sum(sizes), small, seed=31)
    c16, c32 = _pair(cf, dt)
    for a, b in zip(pipeline.run_categories(c16, sizes, 3, 1, 256, 512, [1.0, 0.25], precision="f16"),
                    pipeline.run_categories(c32, sizes, 3, 1, 256, 512, [1.0, 0.25], precision="f16")):
        _path_same(a, b)


def test_driver_bf16_backbone_equals_upcast_maps():
    """make_category_data(backbone_dtype=bfloat16) on the random-init ViT equals run_path on that backbone's 16-bit hooked
    maps upcast to fp32."""
    from anomaly_clustering_b200 import backbones, driver
    from anomaly_clustering_b200.patchcore.patchcore import AnomalyClusteringCore

    n = 4
    ims = torch.rand(n, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    layers = ["blocks.10", "blocks.11"]
    net = backbones.load("dino_vitbase8", allow_random_init=True)
    res = driver.make_category_data(None, "synthetic", 2048, 4096, ["dino_vitbase8"], layers, 3, None, tau=1.0, dataset="synthetic",
                                    test_dataloader=[ims], backbone=net, precision="f16", allow_random_init=True,
                                    backbone_dtype=torch.bfloat16)
    core = AnomalyClusteringCore(torch.device("cuda")).load(net, layers, torch.device("cuda"), (3, 224, 224), 2048, 4096)
    feats = core._features(ims.to("cuda", torch.bfloat16))
    assert all(f.dtype == torch.bfloat16 for f in feats)
    ref = pipeline.run_path([f.float() for f in feats], 3, 1, 2048, 4096, "unsupervised", [1.0], precision="f16")
    alpha, X = res
    assert torch.equal(alpha, ref.alpha32[0].unsqueeze(1))
    assert torch.equal(torch.from_numpy(X), ref.X[0].cpu())


def test_dtype_errors():
    feats, _ = synth.planted_features(2, [(32, 8, 8, False), (32, 8, 8, False)], seed=1)
    mixed = [feats[0].to("cuda", torch.bfloat16), feats[1].to("cuda", torch.float16)]
    with pytest.raises(ValueError):
        ops.embed(mixed, 3, 1, 64, 64)
    with pytest.raises(ValueError):
        ops.weighted_embed_from_features(mixed, torch.ones(2, 64, device="cuda") / 64, 3, 1, 64, 64)
    with pytest.raises(ValueError):
        ops.embed([f.to("cuda", torch.float64) for f in feats], 3, 1, 64, 64)


@pytest.mark.timeout(600)
def test_sharded_path_single_rank_bit_identical():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(29300 + os.getpid() % 300))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "check_half_sharded.py")], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if "bit-identical" in ln]
    assert len(lines) == 2 and all(ln.endswith("OK") for ln in lines), r.stdout
