"""CPU: the refusals of pipeline.GrowingSupervisedCategory and of the running-minimum reduction (AC_REDUCE_MIN_UPDATE) that
need no GPU."""
import ctypes

import pytest
import torch

from anomaly_clustering_b200 import _lib, build, ops, pipeline

LAYERS = [(96, 12, 12), (96, 12, 12)]


def _maps(n, layers=LAYERS, dtype=torch.float32):
    return [torch.zeros(n, C, H, W, dtype=dtype) for C, H, W in layers]


def test_growing_supervised_category_refuses_the_exact_fp32_mode():
    with pytest.raises(ValueError, match="tensor-core precision"):
        pipeline.GrowingSupervisedCategory(3, 1, 256, 512, [1.0], precision="f32")
    g = pipeline.GrowingSupervisedCategory(3, 1, 256, 512, [0.0, 1.0])
    assert g.precision == "f16r" and g.keep_z                     # resolved once, from the taus; refined modes keep Z
    assert pipeline.GrowingSupervisedCategory(3, 1, 256, 512, [1.0, 2.0]).precision == "f16"
    assert pipeline.GrowingSupervisedCategory(3, 1, 256, 512, [0.1], precision="bf16x3").precision == "bf16x3"


def test_refusals_before_any_device_work():
    """Host tensors reach no kernel: every refusal below is raised before the first embed, and none of them changes the state."""
    g = pipeline.GrowingSupervisedCategory(3, 1, 256, 512, [1.0])
    with pytest.raises(ValueError, match="add_normal first"):
        g.add(_maps(2))
    with pytest.raises(ValueError, match="non-zero number of images"):
        g.add_normal(_maps(0))
    with pytest.raises(ValueError, match="non-zero number of images"):
        g.add_normal([torch.zeros(2, 96, 12, 12), torch.zeros(3, 96, 12, 12)])
    assert g.n_img == 0 and g.n_normal == 0 and g.P == 0


def test_features_must_repeat_the_first_calls_signature():
    sig = pipeline._feature_signature(_maps(2), None)
    pipeline._feature_signature(_maps(5), sig)                     # the image count may change
    for bad in (_maps(1, LAYERS[:1]), _maps(1, [(64, 12, 12), (96, 12, 12)]), _maps(1, [(96, 10, 10), (96, 10, 10)]),
                _maps(1, dtype=torch.bfloat16)):
        with pytest.raises(ValueError, match="differ from the first add"):
            pipeline._feature_signature(bad, sig)


def test_reduce_mode_strings_map_explicitly():
    d = torch.zeros(2, 8)
    with pytest.raises(ValueError, match="reduce mode"):
        ops.reduce_weights(d, 4, None, "max")
    with pytest.raises(ValueError, match="reduce mode"):
        ops.reduce_weights(d, 4, None, "supervised")
    with pytest.raises(ValueError, match="out="):
        ops.reduce_weights(d, 4, None, "min_update")
    assert (_lib.AC_REDUCE_MEAN, _lib.AC_REDUCE_MIN, _lib.AC_REDUCE_MIN_UPDATE) == (0, 1, 2)


def test_reduce_entry_point_refuses_bad_arguments_without_a_gpu():
    build.build()
    lib = _lib.load()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    for mode in (-1, 3, 7):
        assert lib.ac_reduce_weights_ex(p, 8, 2, 4, None, None, mode, p, None) == _lib.AC_ERR_INVALID
        assert lib.ac_reduce_weights(p, 8, 2, 4, None, mode, p, None) == _lib.AC_ERR_INVALID
    for mode in (_lib.AC_REDUCE_MIN, _lib.AC_REDUCE_MIN_UPDATE):
        assert lib.ac_reduce_weights_ex(None, 8, 2, 4, None, None, mode, p, None) == _lib.AC_ERR_INVALID
        assert lib.ac_reduce_weights_ex(p, 8, 2, 4, None, None, mode, None, None) == _lib.AC_ERR_INVALID
        assert lib.ac_reduce_weights_ex(p, 8, 2, 4, None, p, mode, p, None) == _lib.AC_ERR_INVALID     # groups need q_self
    if not torch.cuda.is_available():
        # a valid running-minimum call passes the argument checks and fails only for want of a device
        rc = lib.ac_reduce_weights_ex(p, 8, 2, 4, None, None, _lib.AC_REDUCE_MIN_UPDATE, p, None)
        assert rc in (_lib.AC_ERR_CUDA, _lib.AC_ERR_DEVICE)
