"""Mirror of the hot-path classes of models/patchcore/common.py (reference lines cited per class).
Same names, constructor arguments and tensor shapes; the arithmetic runs in libac_b200.so."""
from __future__ import annotations

from typing import Dict, List, Sequence

import torch

from .. import ops


class MeanMapper(torch.nn.Module):
    """common.py:163-170 -- adaptive_avg_pool1d of the flattened feature to `preprocessing_dim`."""

    def __init__(self, preprocessing_dim):
        super().__init__()
        self.preprocessing_dim = preprocessing_dim

    def forward(self, features):
        return ops.adaptive_pool1d(features.reshape(len(features), -1), self.preprocessing_dim)


class Preprocessing(torch.nn.Module):
    """common.py:145-160 -- one MeanMapper per layer, outputs stacked to [N, L, Dp]."""

    def __init__(self, input_dims, output_dim):
        super().__init__()
        self.input_dims = input_dims
        self.output_dim = output_dim
        self.preprocessing_modules = torch.nn.ModuleList([MeanMapper(output_dim) for _ in input_dims])

    def forward(self, features):
        return torch.stack([m(f) for m, f in zip(self.preprocessing_modules, features)], dim=1)


class Aggregator(torch.nn.Module):
    """common.py:173-183 -- [N, L, Dp] -> adaptive_avg_pool1d over the L*Dp concat -> [N, D]."""

    def __init__(self, target_dim):
        super().__init__()
        self.target_dim = target_dim

    def forward(self, features):
        return ops.adaptive_pool1d(features.reshape(len(features), -1), self.target_dim)


class LastLayerToExtractReachedException(Exception):
    """common.py:292 -- control flow: stop the backbone once the deepest requested layer fired."""


class ForwardHook:
    """common.py:277-289 -- forward hook that files the module output under `layer_name` and, on the
    deepest requested layer, aborts the rest of the backbone forward."""

    def __init__(self, hook_dict, layer_name: str, last_layer_to_extract: str):
        self.hook_dict = hook_dict
        self.layer_name = layer_name
        self.is_last = layer_name == last_layer_to_extract

    def __call__(self, module, inputs, output):
        self.hook_dict[self.layer_name] = output
        if self.is_last:
            raise LastLayerToExtractReachedException()


class NetworkFeatureAggregator(torch.nn.Module):
    """common.py:211-275 -- runs the (torch) backbone and returns the outputs of the named layers.
    The backbone forward is NOT part of the accelerated path; it stays in PyTorch."""

    def __init__(self, backbone, layers_to_extract_from: Sequence[str], device):
        super().__init__()
        self.layers_to_extract_from = list(layers_to_extract_from)
        self.backbone = backbone
        self.device = device
        if not hasattr(backbone, "hook_handles"):
            self.backbone.hook_handles = []
        for handle in self.backbone.hook_handles:
            handle.remove()
        self.outputs: Dict[str, torch.Tensor] = {}
        modules = dict(backbone.named_modules())
        for name in self.layers_to_extract_from:
            if name not in modules:
                raise KeyError("backbone has no layer named %r" % name)
            hook = ForwardHook(self.outputs, name, self.layers_to_extract_from[-1])
            self.backbone.hook_handles.append(modules[name].register_forward_hook(hook))
        self.to(self.device)

    def forward(self, images):
        self.outputs.clear()
        with torch.no_grad():
            try:
                self.backbone(images)
            except LastLayerToExtractReachedException:
                pass
        return self.outputs

    def feature_dimensions(self, input_shape) -> List[int]:
        """common.py:270-275 (shape[1] of every hooked output for a dummy input)."""
        p = next(self.backbone.parameters(), None)
        _input = torch.ones([1] + list(input_shape), dtype=p.dtype if p is not None else torch.float32).to(self.device)
        _output = self(_input)
        return [_output[layer].shape[1] for layer in self.layers_to_extract_from]
