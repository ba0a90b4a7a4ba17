"""CPU restatement of the reference's embedding-to-distance path.  TEST INFRASTRUCTURE ONLY.

Every function cites the reference lines it follows (paths relative to the
root of the Anomaly-Clustering project).  Written from the algorithm's closed form
(SURVEY.md section 8c), vectorised so that it finishes in seconds at test sizes.
Pinned against the reference's own code by tests/golden (see oracle/__init__.py).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------- stage 1
def tokens_to_map(feature: torch.Tensor) -> torch.Tensor:
    """models/patchcore/patchcore.py:377-383 -- ViT block output [B,1+P,C] -> [B,C,sqrt(P),sqrt(P)]
    (CLS token dropped).  4-D inputs pass through."""
    if feature.dim() == 3:
        feature = feature[:, 1:, :]
        s = int(math.sqrt(feature.shape[1]))
        feature = feature.reshape(feature.shape[0], s, s, feature.shape[2]).permute(0, 3, 1, 2)
    return feature


def whole_map_layernorm(feature: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """models/patchcore/patchcore.py:384-385 -- fresh nn.LayerNorm([C,H,W]) (gamma=1, beta=0,
    biased variance) applied per image over all C*H*W elements."""
    return F.layer_norm(feature, list(feature.shape[1:]), eps=eps)


def unfold_patches(feature: torch.Tensor, patchsize: int, stride: int) -> Tuple[torch.Tensor, List[int]]:
    """models/patchcore/patchcore.py:439-465 (PatchMaker.patchify) -- returns the unfolded
    tensor viewed as [B, C*k*k, h, w] (flat index f = c*k*k + ki*k + kj; zero outside the map)
    and the patch grid [h, w]."""
    pad = int((patchsize - 1) / 2)
    B, C, H, W = feature.shape
    u = F.unfold(feature, kernel_size=patchsize, stride=stride, padding=pad, dilation=1)
    h = int((H + 2 * pad - (patchsize - 1) - 1) / stride + 1)
    w = int((W + 2 * pad - (patchsize - 1) - 1) / stride + 1)
    return u.reshape(B, C * patchsize * patchsize, h, w), [h, w]


def patchify(feature: torch.Tensor, patchsize: int, stride: int) -> Tuple[torch.Tensor, List[int]]:
    """PatchMaker.patchify with return_spatial_info=True: [B, P, C, k, k], [h, w]
    (models/patchcore/patchcore.py:439-465)."""
    u, grid = unfold_patches(feature, patchsize, stride)
    B, C = feature.shape[:2]
    u = u.reshape(B, C, patchsize, patchsize, -1).permute(0, 4, 1, 2, 3)
    return u, grid


def embed(
    features: Sequence[torch.Tensor],
    patchsize: int,
    stride: int,
    pretrain_dim: int,
    target_dim: int,
    layernorm: bool = True,
    eps: float = 1e-5,
    dtype: torch.dtype = torch.float32,
) -> torch.Tensor:
    """AnomalyClusteringCore._embed after the backbone (models/patchcore/patchcore.py:368-431)
    + Preprocessing/MeanMapper (models/patchcore/common.py:145-170) + Aggregator (:173-183).

    features: per-layer [B,C,H,W] maps or [B,1+P,C] token tensors.  Returns Z [B*P0, D] in `dtype`,
    P0 = patch count of layer 0.  `layernorm=False` gives PatchCore._embed (patchcore.py:92-146).
    Every op is computed in `dtype`: float32 is the reference's own arithmetic, float64 the high-precision
    reference the CUDA kernels are tested against.
    """
    planes = []
    grids = []
    for f in features:
        f = tokens_to_map(f.to(dtype))
        if layernorm:
            f = whole_map_layernorm(f, eps)
        u, g = unfold_patches(f, patchsize, stride)
        planes.append(u)
        grids.append(g)
    h0, w0 = grids[0]
    pooled = []
    for u, g in zip(planes, grids):
        B, CK = u.shape[:2]
        if g != [h0, w0]:
            # patchcore.py:398-421: plane-wise bilinear resize of the UNFOLDED tensor
            u = F.interpolate(
                u.reshape(B * CK, 1, g[0], g[1]), size=(h0, w0), mode="bilinear", align_corners=False
            ).reshape(B, CK, h0, w0)
        # [B, CK, h0, w0] -> [B*P0, 1, CK]; common.py:168-170
        v = u.permute(0, 2, 3, 1).reshape(B * h0 * w0, 1, CK)
        pooled.append(F.adaptive_avg_pool1d(v, pretrain_dim).squeeze(1))
    stacked = torch.stack(pooled, dim=1)  # common.py:160  [B*P0, L, Dp]
    z = F.adaptive_avg_pool1d(stacked.reshape(len(stacked), 1, -1), target_dim)  # common.py:181-183
    return z.reshape(len(z), -1)


def preprocessing_forward(features: Sequence[torch.Tensor], output_dim: int) -> torch.Tensor:
    """Preprocessing.forward (common.py:156-160): list of [N,C,k,k] -> [N,L,Dp]."""
    out = []
    for f in features:
        out.append(F.adaptive_avg_pool1d(f.reshape(len(f), 1, -1), output_dim).squeeze(1))
    return torch.stack(out, dim=1)


def aggregator_forward(features: torch.Tensor, target_dim: int) -> torch.Tensor:
    """Aggregator.forward (common.py:178-183): [N,L,Dp] -> [N,D]."""
    f = features.reshape(len(features), 1, -1)
    return F.adaptive_avg_pool1d(f, target_dim).reshape(len(features), -1)


# --------------------------------------------------------------------------- stage 2
def per_image_min_dist(Zq: torch.Tensor, Zb: torch.Tensor, chunk: int = 8) -> torch.Tensor:
    """min_q ||Zq[i,p] - Zb[j,q]||  for every (i, p, j)  ->  [Nq, P, Nb]  (fp32).

    models/patchcore/utils.py:226 / :233-234: torch.cdist(Z[i], Z[j]) followed by min(dim=1);
    the cdist is evaluated against several bank images at once (same arithmetic path:
    euclidean_dist via matmul for P > 25)."""
    Nq, P, D = Zq.shape
    Nb, Pb, _ = Zb.shape
    out = torch.empty(Nq, P, Nb, dtype=torch.float32)
    for i in range(Nq):
        for j0 in range(0, Nb, chunk):
            j1 = min(Nb, j0 + chunk)
            d = torch.cdist(Zq[i], Zb[j0:j1].reshape(-1, D))  # [P, (j1-j0)*Pb]
            out[i, :, j0:j1] = d.reshape(P, j1 - j0, Pb).min(dim=2)[0]
    return out


def weight_distance_unsupervised(Z: torch.Tensor) -> torch.Tensor:
    """Weight_Distance_Unsupervised for all i (utils.py:222-227): mean over j != i of the
    per-image min distance.  Z [N,P,D] -> w [N,P] fp32."""
    N = Z.shape[0]
    dm = per_image_min_dist(Z, Z)  # [N,P,N]
    mask = ~torch.eye(N, dtype=torch.bool)
    w = torch.empty(N, Z.shape[1], dtype=torch.float32)
    for i in range(N):
        w[i] = dm[i][:, mask[i]].mean(dim=1)
    return w


def weight_distance_supervised(Z: torch.Tensor, Z_train: torch.Tensor) -> torch.Tensor:
    """Weight_Distance_Supervised for all i (utils.py:230-237): min over bank images of the
    per-image min distance.  -> w [N,P] fp32."""
    return per_image_min_dist(Z, Z_train).min(dim=2)[0]


# --------------------------------------------------------------------------- stage 3
def alpha_from_weights(w: torch.Tensor, tau: float, stable: bool = False) -> torch.Tensor:
    """Matrix_Alpha_* tail (utils.py:246-255 / 266-275): float64, tau ~ 0 -> one-hot on the
    max (ties split equally), else exp(w/tau) / sum.  The reference does NOT subtract the max
    (overflows to NaN for w/tau > 709); `stable=True` gives the mathematically identical
    max-subtracted form used by the CUDA path."""
    wd = w.double()
    if math.isclose(tau, 0):
        a = (wd == wd.max(dim=1, keepdim=True)[0]).to(torch.float64)
    else:
        if stable:
            wd = wd - wd.max(dim=1, keepdim=True)[0]
        a = torch.exp((1 / tau) * wd)
    return a / a.sum(dim=1, keepdim=True)


def matrix_alpha_unsupervised(tau: float, Z: torch.Tensor) -> torch.Tensor:
    """Matrix_Alpha_Unsupervised (utils.py:240-257) -> [N,P] float64."""
    return alpha_from_weights(weight_distance_unsupervised(Z), tau)


def matrix_alpha_supervised(tau: float, Z: torch.Tensor, Z_train: torch.Tensor) -> torch.Tensor:
    """Matrix_Alpha_Supervised (utils.py:260-277) -> [N,P] float64."""
    return alpha_from_weights(weight_distance_supervised(Z, Z_train), tau)


def matrix_alpha_average(N: int, P: int) -> torch.Tensor:
    """'average' mode (examples/main.py:290-291)."""
    return torch.ones(N, P) / P


def weighted_embedding64(alpha: torch.Tensor, Z: torch.Tensor) -> torch.Tensor:
    """X[i] = sum_p alpha[i,p] Z[i,p] summed in float64 (the reference for the X kernels).  alpha [N,P], Z [N,P,D] -> [N,D]."""
    return torch.einsum("np,npd->nd", alpha.double(), Z.double())


def weighted_embedding(alpha: torch.Tensor, Z: torch.Tensor) -> np.ndarray:
    """examples/main.py:294-296: X = bmm(alpha.unsqueeze(1).float(), Z).squeeze(1) -> ndarray [N,D]."""
    a = alpha.unsqueeze(1).float()
    return torch.bmm(a, Z).squeeze(1).cpu().numpy().copy()


def pairwise_euclidean(X: np.ndarray) -> np.ndarray:
    """The image-to-image Euclidean matrix Ward consumes (examples/test.py:193-195 ->
    sklearn ward_tree -> scipy.cluster.hierarchy.ward(X) -> pdist(X), float64)."""
    from scipy.spatial.distance import pdist, squareform

    return squareform(pdist(np.asarray(X, dtype=np.float64)))


def full_path(
    features: Sequence[torch.Tensor],
    patchsize: int,
    stride: int,
    pretrain_dim: int,
    target_dim: int,
    tau: float,
    mode: str = "unsupervised",
    bank_features: Optional[Sequence[torch.Tensor]] = None,
):
    """features -> (Z [N,P,D], w [N,P] | None, alpha [N,P] f64, X [N,D] ndarray, Dmat [N,N] f64).
    Mirrors make_category_data (examples/main.py:266-296) from the hooked features on."""
    B = features[0].shape[0]
    Z = embed(features, patchsize, stride, pretrain_dim, target_dim)
    Z = Z.reshape(B, -1, Z.shape[-1])
    w = None
    if mode == "unsupervised":
        w = weight_distance_unsupervised(Z)
        alpha = alpha_from_weights(w, tau)
    elif mode == "supervised":
        Zb = embed(bank_features, patchsize, stride, pretrain_dim, target_dim)
        Zb = Zb.reshape(bank_features[0].shape[0], -1, Zb.shape[-1])
        w = weight_distance_supervised(Z, Zb)
        alpha = alpha_from_weights(w, tau)
    else:
        alpha = matrix_alpha_average(Z.shape[0], Z.shape[1])
    X = weighted_embedding(alpha, Z)
    return Z, w, alpha, X, pairwise_euclidean(X)
