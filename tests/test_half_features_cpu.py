"""CPU: the 16-bit feature-map entry points reject bad arguments before any CUDA call, the Python layer checks map dtypes,
and the CLI's --backbone_dtype flag parses and tags the output directory."""
import ctypes

import pytest
import torch

from anomaly_clustering_b200 import _lib, main


@pytest.fixture(scope="module")
def lib():
    from anomaly_clustering_b200 import build

    build.build()
    return _lib.load()


def _layers():
    arr = (_lib.AcLayer * 2)()
    for i in range(2):
        arr[i] = _lib.AcLayer(4096, 768, 28, 28, 785 * 768, 1, 28 * 768, 768)   # a plausible (never dereferenced) address
    return arr


@pytest.mark.parametrize("bad", [-1, 3, 7])
def test_unknown_feat_dtype_is_invalid(lib, bad):
    arr = _layers()
    buf = ctypes.c_void_p(4096)
    assert lib.ac_embed_workspace_bytes_dt(arr, 2, bad, 2, 3, 1, 2048, 4096) == 0
    assert lib.ac_weighted_embed_from_features_workspace_bytes_dt(arr, 2, bad, 2, 3) == 0
    assert lib.ac_embed_dt(arr, 2, bad, 2, 3, 1, 2048, 4096, 1, 1e-5, buf, None, None, 0, None, buf, 1 << 20, None) == _lib.AC_ERR_INVALID
    assert lib.ac_weighted_embed_from_features_dt(arr, 2, bad, 2, 3, 1, 2048, 4096, 1, 1e-5, buf, buf, buf, 1 << 20,
                                                  None) == _lib.AC_ERR_INVALID


@pytest.mark.parametrize("dt", [_lib.AC_DT_F32, _lib.AC_DT_F16, _lib.AC_DT_BF16])
def test_null_pointers_are_invalid(lib, dt):
    arr = _layers()
    buf = ctypes.c_void_p(4096)
    assert lib.ac_embed_dt(None, 2, dt, 2, 3, 1, 2048, 4096, 1, 1e-5, buf, None, None, 0, None, buf, 1 << 20, None) == _lib.AC_ERR_INVALID
    assert lib.ac_embed_dt(arr, 2, dt, 2, 3, 1, 2048, 4096, 1, 1e-5, buf, None, None, 0, None, None, 1 << 20, None) == _lib.AC_ERR_INVALID
    assert lib.ac_embed_dt(arr, 2, dt, 2, 3, 1, 2048, 4096, 1, 1e-5, None, None, None, 0, None, buf, 1 << 20, None) == _lib.AC_ERR_INVALID
    for args in ((None, buf, buf), (buf, None, buf), (buf, buf, None)):
        assert lib.ac_weighted_embed_from_features_dt(arr, 2, dt, 2, 3, 1, 2048, 4096, 1, 1e-5, *args, 1 << 20,
                                                      None) == _lib.AC_ERR_INVALID
    assert lib.ac_embed_workspace_bytes_dt(None, 2, dt, 2, 3, 1, 2048, 4096) == 0


def test_workspace_f32_wrappers_and_16bit_scratch(lib):
    arr = _layers()
    f32 = lib.ac_embed_workspace_bytes(arr, 2, 4, 3, 1, 2048, 4096)
    assert f32 == lib.ac_embed_workspace_bytes_dt(arr, 2, _lib.AC_DT_F32, 4, 3, 1, 2048, 4096) > 0
    # the per-layer forms read a 16-bit map through an fp32 channel-contiguous copy: at least 4 * C*H*W bytes per image and layer
    for dt in (_lib.AC_DT_F16, _lib.AC_DT_BF16):
        assert lib.ac_embed_workspace_bytes_dt(arr, 2, dt, 4, 3, 1, 2048, 4096) >= f32 + 2 * 4 * 768 * 28 * 28 * 4
        assert (lib.ac_weighted_embed_from_features_workspace_bytes_dt(arr, 2, dt, 4, 3)
                == lib.ac_weighted_embed_from_features_workspace_bytes(arr, 2, 4, 3))


def test_layer_array_dtype_checks():
    from anomaly_clustering_b200 import ops

    # dtype errors are raised before anything touches a device: the CPU maps are rejected for being on the CPU first,
    # so check the dtype rule on the helper's message through a stand-in that skips the device check
    saved = ops._need_cuda
    ops._need_cuda = lambda *ts: None
    try:
        x = torch.zeros(2, 8, 6, 6)
        for bad in ([x.double()], [x.int()], [x.bfloat16(), x.half()], [x, x.bfloat16()]):
            with pytest.raises(ValueError):
                ops._layer_array(bad)
        for good in ([x, x], [x.half(), x.half()], [x.bfloat16()]):
            _, _, code = ops._layer_array(good)
            assert code == ops._TORCH_TO_AC[good[0].dtype]
    finally:
        ops._need_cuda = saved


def test_backbone_dtype_flag_and_directory_tag():
    import argparse

    assert main.backbone_dir_name("dino_vitbase8", False) == "dino_vitbase8"
    assert main.backbone_dir_name("dino_vitbase8", False, "bfloat16") == "dino_vitbase8-bf16"
    assert main.backbone_dir_name("dino_vitbase8", True, "float16") == "dino_vitbase8-randinit-fp16"
    assert main.BACKBONE_DTYPES == {"float32": None, "bfloat16": torch.bfloat16, "float16": torch.float16}
    # the flag parses with its choices and rejects anything else (the parser is built inside main(); parse only)
    captured = {}

    def fake_parse(self, argv=None, namespace=None):
        captured["args"] = _orig(self, argv, namespace)
        raise SystemExit(0)

    _orig = argparse.ArgumentParser.parse_args
    argparse.ArgumentParser.parse_args = fake_parse
    try:
        for val in ("float32", "bfloat16", "float16"):
            with pytest.raises(SystemExit):
                main.main(["--backbone_dtype", val])
            assert captured["args"].backbone_dtype == val
        with pytest.raises(SystemExit):
            main.main([])
        assert captured["args"].backbone_dtype == "float32"
    finally:
        argparse.ArgumentParser.parse_args = _orig
    with pytest.raises(SystemExit):
        main.main(["--backbone_dtype", "float64"])


def test_driver_rejects_other_backbone_dtypes():
    from anomaly_clustering_b200 import driver

    with pytest.raises(ValueError):
        driver.make_category_data(None, "c", 64, 64, ["x"], ["a"], 3, None, test_dataloader=[], backbone_dtype=torch.float64)
