"""Drop-in counterpart of `make_category_data` (reference: examples/main.py:183-311).

Same argument names and the same on-disk result; differences (INTEGRATION.md section 4): the data
loaders and the backbone are injected (MVTec and the DINO weights are not available offline and are
out of scope), the supervised bank is explicit, and `tau` may be a list -- every tau is served
from ONE min-distance pass."""
from __future__ import annotations

from typing import Iterable, List, Optional, Sequence, Union

import numpy as np
import torch

from . import io, pipeline
from .patchcore.patchcore import AnomalyClusteringCore

_HALF_MAPS = (torch.float16, torch.bfloat16)   # feature-map dtypes the embed kernels read natively besides float32


def _images(loader: Iterable) -> torch.Tensor:
    """Concatenates the 'image' entries of a reference-style loader (dicts or tensors)."""
    ims = []
    for item in loader:
        im = item["image"] if isinstance(item, dict) else item
        ims.append(im if im.dim() == 4 else im.unsqueeze(0))
    return torch.cat(ims, dim=0)


def collect_info(loader: Iterable) -> list:
    """main.py:253-262: every loader item minus its 'image' and 'mask' entries."""
    return [{k: v for k, v in item.items() if k not in ("image", "mask")} for item in loader if isinstance(item, dict)]


def make_category_data(
    path,
    category,
    pretrain_embed_dimension,
    target_embed_dimension,
    backbone_names,
    layers_to_extract_from,
    patchsize,
    save_path,
    train_ratio=1.0,
    tau: Union[float, Sequence[float]] = 1,
    supervised="unsupervised",
    dataset="mvtec_ad",
    *,
    test_dataloader: Optional[Iterable] = None,
    train_dataloader: Optional[Iterable] = None,
    backbone: Optional[torch.nn.Module] = None,
    device: Optional[torch.device] = None,
    precision: str = "auto",
    batch_size: int = 16,
    input_shape=(3, 224, 224),
    info_root: Optional[str] = None,
    keep_weights: bool = False,
    allow_random_init: bool = False,
    backbone_dtype: Optional[torch.dtype] = None,
):
    """Returns (matrix_alpha [N,1,P] f32 device tensor, X [N,D] f32 ndarray) for a scalar tau, a list of
    such tuples for a list of taus, and writes the reference's pickle(s) when `save_path` is given.
    `info_root` (the reference's `outputs` directory) also writes <info_root>/<dataset>/info/info_<category>.pickle
    from the loader's non-image fields (main.py:253-262, the file test.py:156 reads); `keep_weights` stores the
    tau-independent weights next to the pickles so a later tau sweep can skip the distance pass.
    `backbone` (a torch module with the reference's pretrained weights loaded) is REQUIRED: the offline stand-ins of
    `backbones.load` are random-init and would silently write meaningless results under the reference's file names.
    `allow_random_init=True` permits them for shape / smoke runs (the CLI then tags the backbone directory `-randinit`).
    `backbone_dtype` torch.bfloat16 / torch.float16 casts the backbone module (in place) and the images to that dtype; its
    16-bit feature maps go to the embed kernels as they are (the result equals the fp32 embedding of those maps upcast).
    None keeps the backbone in float32."""
    if backbone_dtype not in (None, torch.float32, torch.bfloat16, torch.float16):
        raise ValueError("backbone_dtype must be None, torch.float32, torch.bfloat16 or torch.float16, got %s" % (backbone_dtype,))
    if test_dataloader is None:
        raise ValueError("inject test_dataloader: the MVTec walker (datasets/mvtec.py) is out of scope and `path` is not read")
    device = device or torch.device("cuda", torch.cuda.current_device())
    if backbone is None:
        if not allow_random_init:
            raise ValueError("make_category_data needs `backbone=` (a pretrained torch module; the reference downloads DINO / ImageNet "
                             "weights, backbones.py:56-79).  For a shape / smoke run with a RANDOM-INIT network pass allow_random_init=True.")
        from . import backbones

        backbone = backbones.load(backbone_names[0], allow_random_init=True)
    elif getattr(backbone, "random_init", False) and not allow_random_init:
        raise ValueError("the injected backbone is a RANDOM-INIT stand-in (backbones.load); pass allow_random_init=True for a shape / "
                         "smoke run, or a module with the pretrained weights loaded")
    image_dtype = torch.float if backbone_dtype is None else backbone_dtype
    if backbone_dtype is not None:
        backbone = backbone.to(backbone_dtype)
    core = AnomalyClusteringCore(device).load(
        backbone=backbone, layers_to_extract_from=layers_to_extract_from, device=device, input_shape=input_shape,
        pretrain_embed_dimension=pretrain_embed_dimension, target_embed_dimension=target_embed_dimension, patchsize=patchsize,
    )

    taus_early = [float(t) for t in (tau if isinstance(tau, (list, tuple)) else [tau])]
    precision = pipeline.resolve_precision(precision, taus_early)

    def embed_all(loader, want_z):
        """Backbone (torch) + fused embed, `batch_size` images at a time; everything stays on the device."""
        ims = _images(loader)
        sets = []
        for b0 in range(0, len(ims), batch_size):
            feats = [f if f.dtype in _HALF_MAPS else f.float()
                     for f in core._features(ims[b0:b0 + batch_size].to(image_dtype).to(device))]
            sets.append(pipeline.embed_images(feats, patchsize, 1, pretrain_embed_dimension, target_embed_dimension, precision,
                                              want_z=want_z))
        cat = lambda xs: None if xs[0] is None else torch.cat(xs, dim=0)  # noqa: E731
        first = sets[0]
        return pipeline.PatchSet(sum(s.n_img for s in sets), first.P, first.D, first.grid, cat([s.Z for s in sets]),
                                 cat([s.hi for s in sets]), cat([s.lo for s in sets]), cat([s.n2 for s in sets]))

    if info_root:
        io.save_info(info_root, dataset, category, collect_info(test_dataloader))
    taus: List[float] = taus_early
    q = embed_all(test_dataloader, want_z=True)
    if supervised == "supervised":
        if train_dataloader is None:
            raise ValueError("supervised mode needs train_dataloader (the normal training images)")
        bank = embed_all(train_dataloader, want_z=(precision == "f32"))
        n_keep = int(train_ratio * q.n_img)          # main.py:281: Z_train[:int(train_ratio * len(Z))]
        rows = n_keep * bank.P
        pick = lambda t: None if t is None else t[:rows]  # noqa: E731
        bank = pipeline.PatchSet(min(n_keep, bank.n_img), bank.P, bank.D, bank.grid, pick(bank.Z), pick(bank.hi), pick(bank.lo),
                                 pick(bank.n2))
        w = pipeline.min_distance_weights(q, bank, "supervised", precision)
    elif supervised == "unsupervised":
        w = pipeline.min_distance_weights(q, q, "unsupervised", precision)
    else:
        w = None                                      # main.py:290-291 'average'
    a64, a32, X, _ = pipeline.alpha_X_dist(q, w, taus)
    if keep_weights and save_path and w is not None:
        io.save_weights(save_path, category, supervised, w)
    results = []
    for t, tau_t in enumerate(taus if w is not None else taus[:1]):
        matrix_alpha = a32[t].unsqueeze(1)            # main.py:294
        Xn = X[t].cpu().numpy()                       # main.py:296
        if save_path:
            io.save_matrix_alpha_X(save_path, layers_to_extract_from, pretrain_embed_dimension, target_embed_dimension, tau_t,
                                   train_ratio, category, supervised, matrix_alpha, Xn)
        results.append((matrix_alpha, Xn))
    return results[0] if not isinstance(tau, (list, tuple)) else results
