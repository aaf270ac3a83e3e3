"""ORACLE (test infrastructure, not product): LPIPS as ``lpips.LPIPS(net='alex')`` computes it (lpips 0.1,
``lpips=True``, ``spatial=False``), the metric evaluate_Unet_diffusion/evaluate_model.py:46-71 reports.

Trunk — PINNED to torchvision: ``torchvision.models.alexnet(weights=None).features[0:12]`` is the module lpips wraps
(lpips/pretrained_networks.py, class alexnet: slice1 = features[0:2], slice2 = [2:5], slice3 = [5:8], slice4 = [8:10],
slice5 = [10:12], one tap after each slice), loaded here from the ``net.slice*`` keys and run in the dtype asked for
(fp64 for the parity tests).

Scaling layer, head and state-dict keys — PARITY UNPINNED.  The lpips package is not installed here; the following is
restated from lpips 0.1.4 (lpips/lpips.py):
  * ScalingLayer: ``(x - shift) / scale``, shift = [-.030, -.088, -.188], scale = [.458, .448, .450] ([1, 3, 1, 1]
    buffers); ``normalize=True`` maps [0, 1] inputs with ``2 x - 1`` first;
  * normalize_tensor: ``x / (sqrt(sum_c x^2) + 1e-10)``;
  * NetLinLayer: ``Sequential(Dropout(), Conv2d(C, 1, 1, bias=False))`` -> key ``lin{l}.model.1.weight``;
  * spatial_average: mean over H, W (keepdim); the five layers are summed in order.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

# state-dict prefix of conv1..conv5 and its index in AlexNet.features
CONV_KEYS = (("net.slice1.0", 0), ("net.slice2.3", 3), ("net.slice3.6", 6), ("net.slice4.8", 8),
             ("net.slice5.10", 10))
TAP_INDICES = (1, 4, 7, 9, 11)        # the ReLU after which each tap is taken
EPS = 1e-10


def alexnet_features(sd, dtype=torch.float64, device="cpu"):
    """torchvision AlexNet features[0:12] holding the ``net.slice*`` weights of an LPIPS state dict."""
    import torchvision
    feats = torchvision.models.alexnet(weights=None).features[:12]
    with torch.no_grad():
        for key, idx in CONV_KEYS:
            feats[idx].weight.copy_(sd[key + ".weight"])
            feats[idx].bias.copy_(sd[key + ".bias"])
    return feats.to(device=device, dtype=dtype).eval()


def scale(x, sd, normalize=False):
    """ScalingLayer in the dtype of x."""
    if normalize:
        x = 2 * x - 1
    return (x - sd["scaling_layer.shift"].to(x)) / sd["scaling_layer.scale"].to(x)


def taps(features, x):
    """The five feature maps lpips compares, in order."""
    out = []
    with torch.no_grad():
        for i, mod in enumerate(features):
            x = mod(x)
            if i in TAP_INDICES:
                out.append(x)
    return out


def head(taps0, taps1, lin_weights):
    """Per image: sum over taps of the spatial mean of sum_c w_c (f0_hat - f1_hat)^2 -> [N, 1, 1, 1]."""
    val = 0
    for f0, f1, w in zip(taps0, taps1, lin_weights):
        n0 = f0 / (torch.sqrt(torch.sum(f0 ** 2, dim=1, keepdim=True)) + EPS)
        n1 = f1 / (torch.sqrt(torch.sum(f1 ** 2, dim=1, keepdim=True)) + EPS)
        d = F.conv2d((n0 - n1) ** 2, w.to(f0))
        val = val + d.mean(dim=(2, 3), keepdim=True)
    return val


def lin_weights(sd):
    return [sd[f"lin{i}.model.1.weight"] for i in range(5)]


def lpips(sd, in0, in1, normalize=False, dtype=torch.float64):
    """lpips.LPIPS(net='alex')(in0, in1, normalize=normalize) on in0's device, computed in `dtype`."""
    feats = alexnet_features(sd, dtype, in0.device)
    t0 = taps(feats, scale(in0.to(dtype), sd, normalize))
    t1 = taps(feats, scale(in1.to(dtype), sd, normalize))
    return head(t0, t1, lin_weights(sd))
