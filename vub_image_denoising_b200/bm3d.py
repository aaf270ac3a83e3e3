"""BM3D / CBM3D on the device, under the names of the ``bm3d`` package: ``bm3d``, ``bm3d_rgb`` and ``BM3DStages``.

The algorithm is Dabov et al. 2007 (grey) and 2007b (colour, opponent space) with the 'np' profile's parameters and an
8 x 8 DCT in both stages; include/b200dn.h states it in full.  A numpy image in gives a numpy image out (one host round
trip, as the package makes); a CUDA fp32 ``[B, C, H, W]`` batch in gives a fresh fp32 tensor out, enqueued on the
current stream without a host synchronisation.  The result is bit-reproducible and an image's result does not depend
on the batch it is in.
"""
from __future__ import annotations

import enum
from typing import Union

import numpy as np
import torch

from . import _lib, ops

__all__ = ["BM3DStages", "bm3d", "bm3d_rgb"]


class BM3DStages(enum.Enum):
    HARD_THRESHOLDING = _lib.BM3D_HARD_THRESHOLDING
    ALL_STAGES = _lib.BM3D_ALL_STAGES


Image = Union[np.ndarray, torch.Tensor]


def bm3d(z: Image, sigma_psd, profile: str = "np", stage_arg=BM3DStages.ALL_STAGES,
         blockmatches=(False, False)) -> Image:
    """Grey BM3D of an ``H x W`` numpy image or a CUDA fp32 ``[B, 1, H, W]`` batch.  ``sigma_psd`` is the noise
    standard deviation in the image's units: one value, or one per image.  ``stage_arg`` is a :class:`BM3DStages` or
    a basic estimate shaped like ``z`` (then only the Wiener stage runs)."""
    return _run(z, sigma_psd, profile, "opp", stage_arg, blockmatches, channels=1)


def bm3d_rgb(z: Image, sigma_psd, profile: str = "np", colorspace: str = "opp", stage_arg=BM3DStages.ALL_STAGES,
             blockmatches=(False, False)) -> Image:
    """CBM3D of an ``H x W x 3`` numpy image or a CUDA fp32 ``[B, 3, H, W]`` batch, in the opponent colour space; the
    groups are matched on its luminance and shared by the three channels.  Arguments as :func:`bm3d`."""
    return _run(z, sigma_psd, profile, colorspace, stage_arg, blockmatches, channels=3)


def _run(z, sigma_psd, profile, colorspace, stage_arg, blockmatches, channels: int):
    if profile != "np":
        raise NotImplementedError(f"bm3d: only the 'np' profile is implemented, got {profile!r}")
    if colorspace != "opp":
        raise NotImplementedError(f"bm3d: only the opponent colour space is implemented, got {colorspace!r}")
    if tuple(bool(b) for b in blockmatches) != (False, False):
        raise NotImplementedError("bm3d: reusing or returning block matches is not implemented")
    if isinstance(sigma_psd, (np.ndarray, torch.Tensor)) and sigma_psd.ndim >= 2:
        raise NotImplementedError("bm3d: coloured noise (a PSD array) is not implemented; give the noise sigma")
    host = isinstance(z, np.ndarray)
    x = _as_batch(z, channels, "z")
    basic = None
    if isinstance(stage_arg, BM3DStages):
        stages = stage_arg.value
    elif isinstance(stage_arg, (np.ndarray, torch.Tensor)):
        basic, stages = _as_batch(stage_arg, channels, "basic estimate"), _lib.BM3D_ALL_STAGES
        if basic.shape != x.shape:
            raise RuntimeError(f"bm3d: basic estimate {tuple(basic.shape)} does not match z {tuple(x.shape)}")
    else:
        raise RuntimeError(f"bm3d: stage_arg must be a BM3DStages or a basic estimate, got {type(stage_arg).__name__}")
    sigma = _sigma(sigma_psd, x.shape[0])
    if host:
        x, basic = _to_device(x), _to_device(basic)
    for t in (x, basic):
        if t is not None and not t.is_cuda:
            raise RuntimeError("bm3d: CUDA (sm_100) tensors only; there is no CPU fallback")
    if isinstance(sigma, torch.Tensor):
        sigma = sigma.to(device=x.device, dtype=torch.float32).expand(x.shape[0])
    else:
        sigma = torch.tensor(sigma * (x.shape[0] // len(sigma)), dtype=torch.float32, device=x.device)
    out = ops.bm3d(x, sigma, basic, stages, False)[0]
    if host:
        out = out[0].cpu().numpy()
        return out[0] if channels == 1 and z.ndim == 2 else out.transpose(1, 2, 0)
    return out


def _as_batch(z, channels: int, what: str):
    """numpy H x W (grey) / H x W x C -> a CPU fp32 [1, C, H, W] tensor; a tensor is checked and passed through."""
    if isinstance(z, np.ndarray):
        if z.ndim == 2 and channels == 1:
            z = z[:, :, None]
        if z.ndim != 3 or z.shape[2] != channels:
            raise RuntimeError(f"bm3d: {what} must be an H x W{' x 3' if channels == 3 else ''} array, got {z.shape}")
        t = torch.from_numpy(np.ascontiguousarray(z.transpose(2, 0, 1), dtype=np.float32))[None]
    elif isinstance(z, torch.Tensor):
        if z.requires_grad and torch.is_grad_enabled():
            raise RuntimeError("bm3d: inference only; call it under torch.no_grad() or on a tensor without grad")
        if z.dim() != 4 or z.shape[1] != channels or z.dtype != torch.float32:
            raise RuntimeError(f"bm3d: {what} must be an fp32 [B, {channels}, H, W] tensor, got {z.dtype} "
                               f"{tuple(z.shape)}")
        t = z
    else:
        raise RuntimeError(f"bm3d: {what} must be a numpy array or a CUDA tensor, got {type(z).__name__}")
    if t.shape[2] < 8 or t.shape[3] < 8:
        raise RuntimeError(f"bm3d: images must be at least 8 x 8, got {t.shape[2]} x {t.shape[3]}")
    return t


def _sigma(sigma_psd, B: int):
    """One value or one per image, as noise.add_gaussian_noise takes sigma: a list of floats, or a CUDA tensor.  Host
    values must be positive; a device tensor is taken as it is (checking it would synchronise)."""
    if isinstance(sigma_psd, torch.Tensor) and sigma_psd.is_cuda:
        s = sigma_psd.detach().reshape(-1)
        n = s.numel()
    else:
        s = np.asarray(sigma_psd.cpu() if isinstance(sigma_psd, torch.Tensor) else sigma_psd, dtype=np.float64)
        s = s.reshape(-1).tolist()
        if not all(v > 0 for v in s):
            raise RuntimeError(f"bm3d: sigma must be positive, got {s}")
        n = len(s)
    if n not in (1, B):
        raise RuntimeError(f"bm3d: sigma must have 1 or B = {B} entries, got {n}")
    return s


def _to_device(t):
    if t is None:
        return None
    if not torch.cuda.is_available():
        raise RuntimeError("bm3d: a CUDA (sm_100) device is required; there is no CPU fallback")
    return t.cuda()
