"""Import the UNMODIFIED reference modules from a checkout of the original project.

TEST INFRASTRUCTURE.  The original project (KevinWangHP/Anomaly-Clustering, with
its shipped `outputs/`) is not part of this repository: AC_REFERENCE_DIR names a
checkout of it.  Nothing the suite needs may call this module unconditionally
(`-m gpu` tests, smoke(), bench.py never do); it is used by
`oracle/make_golden.py` (fixture generation) and by the CPU-side tests that are
skipped when AC_REFERENCE_DIR is not set.

The reference imports faiss / timm / matplotlib / munkres at module top level
(Anomaly-Clustering/models/patchcore/common.py:7, backbones.py:1, utils.py:7);
none of them is used by the hot-path arithmetic, so they are stubbed.
"""
from __future__ import annotations

import os
import sys
import types
from unittest import mock

REFERENCE_DIR = os.environ.get("AC_REFERENCE_DIR", "")
_MODELS = os.path.join(REFERENCE_DIR, "models")
OUTPUTS = os.path.join(REFERENCE_DIR, "outputs")


def available() -> bool:
    return bool(REFERENCE_DIR) and os.path.isdir(_MODELS)


def outputs_available() -> bool:
    return bool(REFERENCE_DIR) and os.path.isdir(OUTPUTS)


_cached = None


def load():
    """Returns a namespace with the reference's patchcore.{patchcore,common,utils} modules."""
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise RuntimeError("set AC_REFERENCE_DIR to a checkout of the original Anomaly-Clustering project (got %r)" % REFERENCE_DIR)
    for name in ("faiss", "timm", "matplotlib", "matplotlib.pyplot", "munkres"):
        if name not in sys.modules:
            sys.modules[name] = mock.MagicMock()
    if _MODELS not in sys.path:
        sys.path.insert(0, _MODELS)
    import patchcore.common as common  # noqa: E402  (reference module)
    import patchcore.patchcore as pc  # noqa: E402
    import patchcore.utils as utils  # noqa: E402

    ns = types.SimpleNamespace(common=common, patchcore=pc, utils=utils)
    _cached = ns
    return ns


class _FeatureStub:
    """Stands in for NetworkFeatureAggregator (common.py:211): returns canned features.

    The backbone forward is out of scope (stays in torch); the hot path starts at
    the hooked feature maps, so the oracle feeds them directly.
    """

    def __init__(self, features_by_layer):
        self.features_by_layer = features_by_layer

    def eval(self):
        return self

    def __call__(self, images):
        return self.features_by_layer


def reference_embed(features, patchsize, stride, pretrain_dim, target_dim):
    """Runs the reference's AnomalyClusteringCore._embed (patchcore.py:355-431) on given
    per-layer features (list of [B,C,H,W] or [B,1+P,C] CPU tensors).  Returns Z [B*P, D]."""
    import torch

    ref = load()
    core = ref.patchcore.AnomalyClusteringCore(torch.device("cpu"))
    names = ["l%d" % i for i in range(len(features))]
    core.layers_to_extract_from = names
    core.device = torch.device("cpu")
    core.patch_maker = ref.patchcore.PatchMaker(patchsize, stride=stride)
    core.forward_modules = {
        "feature_aggregator": _FeatureStub(dict(zip(names, features))),
        "preprocessing": ref.common.Preprocessing([0] * len(features), pretrain_dim),
        "preadapt_aggregator": ref.common.Aggregator(target_dim=target_dim),
    }
    with torch.no_grad():
        out = core._embed(None, "unsupervised", detach=False)
    return out


def reference_alpha_unsupervised(tau, Z):
    import torch

    ref = load()
    return ref.utils.Matrix_Alpha_Unsupervised(tau, 1, Z, torch.device("cpu"))


def reference_alpha_supervised(tau, Z, Z_train):
    import torch

    ref = load()
    return ref.utils.Matrix_Alpha_Supervised(tau, 1, Z, Z_train, torch.device("cpu"))
