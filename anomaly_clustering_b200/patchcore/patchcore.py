"""Mirror of PatchMaker / AnomalyClusteringCore (models/patchcore/patchcore.py:276-465).

`_embed` keeps the reference's signature and return convention (list of per-patch numpy rows
when detach=True) but computes LayerNorm + patchify + resize + Preprocessing + Aggregator in ONE
fused CUDA kernel instead of materialising the 9x unfolded tensor; `embed_device` is the
addition that keeps Z on the device (SURVEY.md section 8f row 3)."""
from __future__ import annotations

import numpy as np
import torch
import tqdm

from .. import ops
from . import common


class PatchMaker:
    """patchcore.py:434-482."""

    def __init__(self, patchsize, stride=None):
        self.patchsize = patchsize
        self.stride = stride

    def patchify(self, features, return_spatial_info=False):
        """[B,C,H,W] -> [B, h*w, C, patchsize, patchsize] (+ [h, w]); patchcore.py:439-465."""
        unfolded, grid = ops.patchify(features, self.patchsize, self.stride if self.stride else 1)
        if return_spatial_info:
            return unfolded, grid
        return unfolded

    def unpatch_scores(self, x, batchsize):
        """[B*P, ...] -> [B, P, ...] (patchcore.py:467-468)."""
        return x.reshape(batchsize, -1, *x.shape[1:])

    def score(self, x):
        """Max over all trailing axes, numpy in -> numpy out (patchcore.py:470-481)."""
        t = torch.from_numpy(x) if isinstance(x, np.ndarray) else x
        if t.ndim > 1:
            t = t.reshape(t.shape[0], -1).max(dim=1).values
        return t.numpy() if isinstance(x, np.ndarray) else t


class AnomalyClusteringCore(torch.nn.Module):
    """patchcore.py:276-431.  Detection-only members of the reference (`anomaly_scorer`,
    `anomaly_segmentor`, `featuresampler`) are accepted and ignored: the clustering path never
    calls them (SURVEY.md section 2 rows 9-11)."""

    def __init__(self, device):
        super().__init__()
        self.device = device

    def load(self, backbone, layers_to_extract_from, device, input_shape, pretrain_embed_dimension,
             target_embed_dimension, patchsize=3, patchstride=1, anomaly_score_num_nn=1, featuresampler=None,
             nn_method=None, **kwargs):
        self.backbone = backbone.to(device)
        self.layers_to_extract_from = layers_to_extract_from
        self.input_shape = input_shape
        self.device = device
        self.patch_maker = PatchMaker(patchsize, stride=patchstride)
        self.forward_modules = torch.nn.ModuleDict({})
        feature_aggregator = common.NetworkFeatureAggregator(self.backbone, self.layers_to_extract_from, self.device)
        feature_dimensions = feature_aggregator.feature_dimensions(input_shape)
        self.forward_modules["feature_aggregator"] = feature_aggregator
        self.forward_modules["preprocessing"] = common.Preprocessing(feature_dimensions, pretrain_embed_dimension)
        self.pretrain_embed_dimension = pretrain_embed_dimension
        self.target_embed_dimension = target_embed_dimension
        self.forward_modules["preadapt_aggregator"] = common.Aggregator(target_dim=target_embed_dimension)
        self.featuresampler = featuresampler
        return self

    # -- the hooked backbone features (torch; not the accelerated part)
    def _features(self, images):
        _ = self.forward_modules["feature_aggregator"].eval()
        with torch.no_grad():
            feats = self.forward_modules["feature_aggregator"](images)
        return [feats[layer] for layer in self.layers_to_extract_from]

    def embed_device(self, images, operand=None, want_lo=False):
        """Addition: images [B,3,H,W] -> (Z [B*P, D] device fp32, hi, lo, patch grid); B > 1 allowed.  16-bit hooked maps
        (a backbone run under bf16 / fp16 autocast) go to the kernels as they are: same result as their fp32 upcast."""
        feats = [f if f.dtype in (torch.float16, torch.bfloat16) else f.float()
                 for f in self._features(images.to(torch.float).to(self.device))]
        return ops.embed(feats, self.patch_maker.patchsize, self.patch_maker.stride or 1, self.pretrain_embed_dimension,
                         self.target_embed_dimension, layernorm=True, operand=operand, want_lo=want_lo)

    def embed(self, data, supervised):
        """patchcore.py:337-353 -- a DataLoader yields per-batch embeddings + the `is_anomaly` labels,
        anything else is embedded directly.  (`supervised` is accepted and unused, as in the reference.)"""
        print("{:-^80}".format("embedding"))
        if not isinstance(data, torch.utils.data.DataLoader):
            return self._embed(data, supervised)
        per_batch, flags = [], []
        for batch in tqdm.tqdm(data, total=len(data)):
            flag = batch["is_anomaly"] if isinstance(batch, dict) else None
            pixels = batch["image"] if isinstance(batch, dict) else batch
            with torch.no_grad():
                per_batch.append(self._embed(pixels.to(torch.float).to(self.device), supervised))
            flags.append(flag)
        return per_batch, flags

    def _embed(self, images, supervised, detach=True, provide_patch_shapes=False):
        """patchcore.py:355-431: returns the [B*P, D] embedding (as a list of numpy rows when
        `detach`, like the reference's `_detach`)."""
        Z, _, _, grid = self.embed_device(images)
        patch_shapes = [list(grid)]
        for f in self._last_feature_shapes()[1:]:
            patch_shapes.append(f)
        out = [x for x in Z.detach().cpu().numpy()] if detach else Z
        if provide_patch_shapes:
            return out, patch_shapes
        return out

    def _last_feature_shapes(self):
        outs = self.forward_modules["feature_aggregator"].outputs
        shapes = []
        for layer in self.layers_to_extract_from:
            v = ops.feature_view(outs[layer])
            shapes.append(list(ops.patch_grid(v.shape[2], v.shape[3], self.patch_maker.patchsize, self.patch_maker.stride or 1)))
        return shapes
