"""ORACLE (test infrastructure, not product): DISTS as ``DISTS_pytorch.DISTS()`` computes it (DISTS_pytorch 0.1,
``DISTS_pt.py``), the metric evaluate_Unet_diffusion/evaluate_model.py:46-71 reports.

Trunk convolutions — PINNED to torchvision: ``torchvision.models.vgg16(weights=None).features[:30]`` is the module
DISTS wraps (stage1 = features[0:4], stage2 = [4:9], stage3 = [9:16], stage4 = [16:23], stage5 = [23:30]), loaded here
from the ``stage*`` keys and run in the dtype asked for (fp64 for the parity tests).

L2 pooling, normalisation, head and state-dict keys — PARITY UNPINNED.  The DISTS_pytorch package is not installed
here; the following is restated from DISTS_pytorch 0.1 (DISTS_pt.py):
  * the four MaxPool2d (features 4, 9, 16, 23) are replaced by L2pooling(channels=C):
    ``sqrt(conv2d(x^2, filter, stride=2, padding=1, groups=C) + 1e-12)``, filter = the outer product of
    ``np.hanning(5)[1:-1]`` normalised to sum 1, a [C, 1, 3, 3] buffer (key ``stage{k}.{idx}.filter``);
  * ``h = (x - mean) / std`` with mean = [0.485, 0.456, 0.406], std = [0.229, 0.224, 0.225] ([1, 3, 1, 1] buffers);
    the features are ``[x, relu1_2, relu2_2, relu3_3, relu4_3, relu5_3]``, the first the raw input;
  * alpha, beta: [1, 1475, 1, 1] parameters, divided by ``alpha.sum() + beta.sum()`` and split by
    chns = [3, 64, 128, 256, 512, 512]; c1 = c2 = 1e-6; per stage and channel, with means over H x W,
    ``S1 = (2 mx my + c1) / (mx^2 + my^2 + c1)``, ``S2 = (2 cov + c2) / (vx + vy + c2)``, vx = mean((x - mx)^2),
    cov = mean(xy) - mx my; ``score = 1 - sum(alpha S1) - sum(beta S2)``, then ``.squeeze()``.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

CHNS = (3, 64, 128, 256, 512, 512)
STAGES = ((0, 4), (4, 9), (9, 16), (16, 23), (23, 30))      # features[a:b] of stage1..stage5
CONV_INDICES = (0, 2, 5, 7, 10, 12, 14, 17, 19, 21, 24, 26, 28)
POOL_INDICES = (4, 9, 16, 23)
C1 = C2 = 1e-6


def stage_of(idx: int) -> int:
    return next(s for s, (a, b) in enumerate(STAGES) if a <= idx < b) + 1


def key(idx: int) -> str:
    """State-dict prefix of features[idx]: ``stage{k}.{idx}``."""
    return f"stage{stage_of(idx)}.{idx}"


def hanning_filter(channels: int) -> torch.Tensor:
    a = np.hanning(5)[1:-1]
    g = torch.Tensor(a[:, None] * a[None, :])
    g = g / torch.sum(g)
    return g[None, None, :, :].repeat((channels, 1, 1, 1))


class L2pooling(nn.Module):
    def __init__(self, filt: torch.Tensor):
        super().__init__()
        self.register_buffer("filter", filt.detach().clone())

    def forward(self, x):
        out = F.conv2d(x ** 2, self.filter.to(x), stride=2, padding=1, groups=x.shape[1])
        return (out + 1e-12).sqrt()


def vgg_features(sd, dtype=torch.float64, device="cpu", pool="l2"):
    """torchvision VGG16 features[:30] holding the ``stage*`` weights of a DISTS state dict, the four max-pools
    replaced by L2pooling (``pool="max"`` keeps torchvision's max-pools: a near-miss reference)."""
    import torchvision
    feats = torchvision.models.vgg16(weights=None).features[:30]
    with torch.no_grad():
        for idx in CONV_INDICES:
            feats[idx].weight.copy_(sd[key(idx) + ".weight"])
            feats[idx].bias.copy_(sd[key(idx) + ".bias"])
    if pool == "l2":
        for idx in POOL_INDICES:
            feats[idx] = L2pooling(sd[key(idx) + ".filter"])
    return feats.to(device=device, dtype=dtype).eval()


def normalise(x, sd):
    return (x - sd["mean"].to(x)) / sd["std"].to(x)


def features(feats, x, sd, normalise_input=True):
    """The six feature sets DISTS compares: the raw input, then the output of each stage."""
    out, h = [x], normalise(x, sd) if normalise_input else x
    with torch.no_grad():
        for a, b in STAGES:
            h = feats[a:b](h)
            out.append(h)
    return out


def head(f0, f1, alpha, beta, unbiased=False, divide=True):
    """1 - sum_k sum_c (alpha S1 + beta S2) -> [N] (before the reference's squeeze); alpha, beta [1, 1475, 1, 1].
    ``unbiased`` (vx, vy as torch.var's default) and ``divide=False`` (alpha, beta not divided by their sum) are
    near-miss references."""
    w_sum = alpha.sum() + beta.sum() if divide else 1.0
    al = torch.split(alpha / w_sum, list(CHNS), dim=1)
    be = torch.split(beta / w_sum, list(CHNS), dim=1)
    d1 = d2 = 0
    for k in range(len(CHNS)):
        x, y = f0[k], f1[k]
        mx, my = x.mean([2, 3], keepdim=True), y.mean([2, 3], keepdim=True)
        s1 = (2 * mx * my + C1) / (mx ** 2 + my ** 2 + C1)
        d1 = d1 + (al[k].to(x) * s1).sum(1, keepdim=True)
        n = x.shape[2] * x.shape[3]
        corr = n / (n - 1) if unbiased else 1.0
        vx = ((x - mx) ** 2).mean([2, 3], keepdim=True) * corr
        vy = ((y - my) ** 2).mean([2, 3], keepdim=True) * corr
        cov = (x * y).mean([2, 3], keepdim=True) - mx * my
        s2 = (2 * cov + C2) / (vx + vy + C2)
        d2 = d2 + (be[k].to(x) * s2).sum(1, keepdim=True)
    return (1 - (d1 + d2)).flatten()


def dists(sd, x, y, dtype=torch.float64):
    """DISTS_pytorch.DISTS()(x, y) on x's device in `dtype`, as [N] (no squeeze)."""
    feats = vgg_features(sd, dtype, x.device)
    f0, f1 = features(feats, x.to(dtype), sd), features(feats, y.to(dtype), sd)
    return head(f0, f1, sd["alpha"].to(dtype), sd["beta"].to(dtype))
