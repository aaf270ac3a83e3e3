"""On-device PSNR / SSIM with the call signatures the reference's evaluation scripts use.

  * ``calculate_psnr(X, Y, data_range=1.0)``                 evaluate_Unet_diffusion/evaluate_model.py:36-41
  * ``calculate_ssim(X, Y, data_range=1.0, use_rgb=False)``  evaluate_Unet_diffusion/evaluate_model.py:30-34
  * ``peak_signal_noise_ratio(gt, out, data_range=...)``     skimage call at evaluate_SIDD/evaluate_SIDD.py:63
  * ``structural_similarity(gt, out, data_range=..., channel_axis=...)``   evaluate_SIDD/evaluate_SIDD.py:64,
    with every option of skimage 0.22's call (Gaussian window, win_size, covariance, K1/K2, the full SSIM map)
  * ``psnr_torch(pred, target)``                             diffusion_denoising/hyperparams_search.py:11-16
  * ``welch(x, nperseg=256)``                                scipy.signal.welch call at evaluate_Unet_diffusion/plot.py:155-157

The batch entry points (``batch_sse`` / ``batch_ssim`` / ``batch_metrics``) keep everything on the GPU and
return fp64 device tensors, so a sharded evaluation can all-reduce sums without a per-image host sync
(the reference pays a ``.cpu()`` round trip per image, evaluate_model.py:47-48).
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib

__all__ = ["batch_sse", "batch_ssim_planes", "batch_metrics", "calculate_psnr", "calculate_ssim",
           "peak_signal_noise_ratio", "structural_similarity", "psnr_torch", "welch", "high_frequency_psd_mae"]


_SSIM_TRUNCATE = 3.5        # skimage's gaussian_filter truncate
_WIN_EXTENT_MSG = (
    "win_size exceeds image extent. Either ensure that your images are at least 7x7; or pass win_size explicitly in "
    "the function call, with an odd value less than or equal to the smaller side of your images. If your images are "
    "multichannel (with color channels), set channel_axis to the axis number corresponding to the channels.")


def _as_dev_f32(x, like: Optional[torch.Tensor] = None) -> torch.Tensor:
    if isinstance(x, np.ndarray):
        if like is None:
            if not torch.cuda.is_available():
                raise RuntimeError("vub_image_denoising_b200 metrics need a CUDA (sm_100) device; no CPU fallback")
            dev = torch.device("cuda", torch.cuda.current_device())
        else:
            dev = like.device
        x = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    if not isinstance(x, torch.Tensor):
        raise RuntimeError("expected a torch.Tensor or numpy array")
    if not x.is_cuda:
        raise RuntimeError("vub_image_denoising_b200 metrics run on CUDA (sm_100) tensors only; no CPU fallback")
    return x.detach().to(torch.float32)


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Per-call partial-sum workspace (fp64 words) of the two-pass, fixed-order reductions.  Allocated through
    torch's caching allocator on the current stream, so consecutive calls reuse the same block without a sync."""
    return torch.empty(max(1, (int(nbytes) + 7) // 8), dtype=torch.float64, device=device)


def batch_sse(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Per-image sum of squared differences; a, b: [N, ...] fp32 CUDA.  Returns fp64 [N] (device)."""
    a = _as_dev_f32(a).contiguous()
    b = _as_dev_f32(b, a).contiguous()
    if a.shape != b.shape:
        raise RuntimeError(f"shape mismatch {tuple(a.shape)} vs {tuple(b.shape)}")
    n = a.shape[0]
    per = a.numel() // max(n, 1)
    out = torch.empty(n, dtype=torch.float64, device=a.device)
    L = _lib.lib()
    with torch.cuda.device(a.device):
        for i0 in range(0, n, 65535):
            i1 = min(n, i0 + 65535)
            ws = _workspace(L.b200dn_psnr_sse_workspace_bytes(i1 - i0, per), a.device)
            rc = L.b200dn_psnr_sse(a[i0:i1].data_ptr(), b[i0:i1].data_ptr(), i1 - i0, per, out[i0:i1].data_ptr(),
                                   ws.data_ptr(), ws.numel() * 8, torch.cuda.current_stream(a.device).cuda_stream)
            _lib.check(rc, "psnr_sse")
    return out


def _gaussian_taps(sigma: float, radius: int) -> np.ndarray:
    """The taps of scipy.ndimage.gaussian_filter(sigma) at this radius (``_gaussian_kernel1d``): exp(-x^2 / (2 sigma^2)),
    x = -radius .. radius, normalised in fp64.  gaussian_filter leaves an axis with sigma <= 1e-15 unfiltered."""
    if sigma <= 1e-15:
        return np.ones(1)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return phi / phi.sum()


def _ssim_window_opts(H: int, W: int, data_range: float, win_size, gaussian_weights: bool, sigma: float,
                      use_sample_covariance: bool, K1: float, K2: float) -> _lib.SsimWindowOpts:
    """skimage 0.22 structural_similarity's argument checks, in its order and with its messages, and the window they
    define: the filter is gaussian_filter(sigma, truncate=3.5) or uniform_filter(win_size), both mode='reflect'; win_size
    (default 2*radius + 1 with Gaussian weights, else 7) sets the crop and the covariance normaliser."""
    if K1 < 0:
        raise ValueError("K1 must be positive")
    if K2 < 0:
        raise ValueError("K2 must be positive")
    if sigma < 0:
        raise ValueError("sigma must be positive")
    radius = int(_SSIM_TRUNCATE * sigma + 0.5) if gaussian_weights else None
    if win_size is None:
        win_size = 2 * radius + 1 if gaussian_weights else 7
    if min(H, W) < win_size:
        raise ValueError(_WIN_EXTENT_MSG)
    if not (win_size % 2 == 1):
        raise ValueError("Window size must be odd.")
    if not gaussian_weights:
        radius = (win_size - 1) // 2
    if radius > _lib.SSIM_MAX_RADIUS:
        raise NotImplementedError(f"the device SSIM filters with a radius of at most {_lib.SSIM_MAX_RADIUS}; "
                                  f"this call needs {radius}")
    taps = _gaussian_taps(sigma, radius) if gaussian_weights else np.full(2 * radius + 1, 1.0 / win_size)
    NP = win_size ** 2
    R = float(data_range)
    o = _lib.SsimWindowOpts()
    o.radius, o.win_size = radius, win_size
    o.cov_norm = NP / (NP - 1) if use_sample_covariance else 1.0
    o.C1, o.C2 = (K1 * R) ** 2, (K2 * R) ** 2          # in double, used as float32 (as skimage does)
    o.weights[:len(taps)] = taps.astype(np.float32).tolist()
    return o


def batch_ssim_planes(a: torch.Tensor, b: torch.Tensor, data_range: float, *, win_size: Optional[int] = None,
                      gaussian_weights: bool = False, sigma: float = 1.5, use_sample_covariance: bool = True,
                      K1: float = 0.01, K2: float = 0.03, full: bool = False):
    """Mean SSIM of every 2-D plane; a, b: [P, H, W] fp32 CUDA.  Returns fp64 [P] (device), or with ``full=True``
    ``(means, maps)``, the maps of S fp32 [P, H, W].  No host sync.

    The keywords are skimage 0.22 structural_similarity's (``gaussian_weights=True, sigma=1.5,
    use_sample_covariance=False`` is Wang et al. 2004's SSIM).  The default call (7x7 uniform window, sample covariance,
    K1 = 0.01, K2 = 0.03, no map) runs ``ssim_kernel``; every other runs ``ssim_window_kernel``."""
    a = _as_dev_f32(a).contiguous()
    b = _as_dev_f32(b, a).contiguous()
    if a.shape != b.shape or a.dim() != 3:
        raise RuntimeError("expected two [P, H, W] tensors of equal shape")
    P, H, W = a.shape
    opts = _ssim_window_opts(H, W, data_range, win_size, gaussian_weights, sigma, use_sample_covariance, K1, K2)
    out = torch.empty(P, dtype=torch.float64, device=a.device)
    L = _lib.lib()
    if not (full or gaussian_weights) and opts.win_size == 7 and use_sample_covariance and K1 == 0.01 and K2 == 0.03:
        with torch.cuda.device(a.device):
            for i0 in range(0, P, 65535):
                i1 = min(P, i0 + 65535)
                ws = _workspace(L.b200dn_ssim_workspace_bytes(i1 - i0, H, W), a.device)
                rc = L.b200dn_ssim(a[i0:i1].data_ptr(), b[i0:i1].data_ptr(), i1 - i0, H, W, float(data_range),
                                   out[i0:i1].data_ptr(), ws.data_ptr(), ws.numel() * 8,
                                   torch.cuda.current_stream(a.device).cuda_stream)
                _lib.check(rc, "ssim")
        return out / float((H - 6) * (W - 6))
    maps = torch.empty((P, H, W), dtype=torch.float32, device=a.device) if full else None
    with torch.cuda.device(a.device):
        for i0 in range(0, P, 65535):
            i1 = min(P, i0 + 65535)
            ws = _workspace(L.b200dn_ssim_window_workspace_bytes(i1 - i0, H, W), a.device)
            rc = L.b200dn_ssim_window(a[i0:i1].data_ptr(), b[i0:i1].data_ptr(), i1 - i0, H, W, ctypes.byref(opts),
                                      out[i0:i1].data_ptr(), maps[i0:i1].data_ptr() if full else None,
                                      ws.data_ptr(), ws.numel() * 8, torch.cuda.current_stream(a.device).cuda_stream)
            _lib.check(rc, "ssim_window")
    pad = (opts.win_size - 1) // 2
    means = out / float((H - 2 * pad) * (W - 2 * pad))
    return (means, maps) if full else means


def batch_metrics(ref: torch.Tensor, img: torch.Tensor, data_range: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """PSNR [N] and channel-mean SSIM [N] for NCHW batches, all on device (fp64)."""
    ref = _as_dev_f32(ref).contiguous()
    img = _as_dev_f32(img, ref).contiguous()
    N, Cn, H, W = ref.shape
    mse = batch_sse(ref, img) / float(Cn * H * W)
    psnr = 10.0 * torch.log10((float(data_range) ** 2) / mse)
    planes = batch_ssim_planes(ref.view(N * Cn, H, W), img.view(N * Cn, H, W), data_range)
    # skimage stores each channel's mean in a float32 array and averages that array
    ssim = planes.to(torch.float32).view(N, Cn).mean(dim=1).to(torch.float64)
    return psnr, ssim


# ----------------------------------------------------------------------------- reference-shaped calls
def calculate_psnr(X, Y, data_range: float = 1.0) -> float:
    a = _as_dev_f32(X)
    b = _as_dev_f32(Y, a)
    sse = batch_sse(a.reshape(1, -1), b.reshape(1, -1))
    mse = float(sse.item()) / a.numel()
    if mse == 0:
        return float("inf")
    return 10 * math.log10((data_range ** 2) / mse)


def peak_signal_noise_ratio(image_true, image_test, *, data_range=None) -> float:
    if data_range is None:
        raise ValueError("data_range must be given for floating point images")
    return calculate_psnr(image_true, image_test, data_range)


def structural_similarity(im1, im2, *, win_size: Optional[int] = None, gradient: bool = False, data_range: float,
                          channel_axis: Optional[int] = None, multichannel: Optional[bool] = None,
                          gaussian_weights: bool = False, full: bool = False, **kwargs):
    """skimage 0.22's structural_similarity on the device.  kwargs: ``K1=0.01, K2=0.03, sigma=1.5,
    use_sample_covariance=True``.  Returns the mean SSIM as a float, or with ``full=True`` ``(mean, S)``, S the fp32
    CUDA map in the input's layout.  ``gradient=True`` is not implemented."""
    unknown = sorted(set(kwargs) - {"K1", "K2", "sigma", "use_sample_covariance"})
    if unknown:
        raise TypeError(f"structural_similarity() got unexpected keyword arguments {unknown}")
    if gradient:
        raise NotImplementedError("gradient=True is not implemented on device")
    a = _as_dev_f32(im1)
    b = _as_dev_f32(im2, a)
    if a.shape != b.shape:
        raise ValueError("Input images must have the same dimensions.")
    opts = dict(win_size=win_size, gaussian_weights=gaussian_weights, full=full, **kwargs)
    if channel_axis is None:
        if a.dim() != 2:
            raise NotImplementedError("without channel_axis only 2-D images are supported")
        res = batch_ssim_planes(a[None], b[None], data_range, **opts)
        return (float(res[0].item()), res[1][0]) if full else float(res.item())
    a = a.movedim(channel_axis, 0).contiguous()
    b = b.movedim(channel_axis, 0).contiguous()
    res = batch_ssim_planes(a, b, data_range, **opts)
    # skimage stores each channel's mean in a float32 array and averages that array
    mssim = float((res[0] if full else res).to(torch.float32).mean().item())
    return (mssim, res[1].movedim(0, channel_axis).contiguous()) if full else mssim


def calculate_ssim(X, Y, data_range: float = 1.0, use_rgb: bool = False) -> float:
    if use_rgb:
        return structural_similarity(X, Y, data_range=data_range, channel_axis=0)
    return structural_similarity(X, Y, data_range=data_range)


def psnr_torch(pred: torch.Tensor, target: torch.Tensor) -> float:
    """20*log10(1/sqrt(mse)) on [0,1] tensors (diffusion_denoising/hyperparams_search.py:11-16)."""
    a = _as_dev_f32(pred)
    sse = batch_sse(a.reshape(1, -1), _as_dev_f32(target, a).reshape(1, -1))
    mse = float(sse.item()) / a.numel()
    if mse == 0:
        return float("inf")
    return 20 * math.log10(1.0 / math.sqrt(mse))


# ----------------------------------------------------------------------------- frequency-domain analysis (plot.py)
def welch(x, nperseg: int = 256) -> Tuple[np.ndarray, torch.Tensor]:
    """``scipy.signal.welch(x, nperseg=256)`` on the device (plot.py:155-157 calls it on ``image.flatten()``).

    x: CUDA tensor (or numpy array) whose LAST axis is the signal — scipy's ``axis=-1`` — e.g. ``img.flatten()`` or a
    batch ``imgs.flatten(1)``.  Returns ``(f, Pxx)``: ``f`` the 129 sample frequencies k/256 as a float64 numpy array
    (as scipy returns them) and ``Pxx`` a float32 CUDA tensor ``[..., 129]``.  Only scipy's defaults at nperseg = 256
    are implemented (fs = 1, Hann, noverlap = 128, constant detrend, one-sided density, mean)."""
    if nperseg != 256:
        raise NotImplementedError("only nperseg=256 (the reference's call) is implemented on device")
    t = _as_dev_f32(x).contiguous()
    n = t.shape[-1]
    if n < 256:
        raise ValueError("nperseg = 256 is greater than the input length")   # scipy warns and shrinks; not supported here
    flat = t.reshape(-1, n)
    S = flat.shape[0]
    out = torch.empty((S, 129), dtype=torch.float32, device=t.device)
    L = _lib.lib()
    with torch.cuda.device(t.device):
        for i0 in range(0, S, 65535):
            i1 = min(S, i0 + 65535)
            nbytes = L.b200dn_welch_psd_workspace_bytes(i1 - i0, n)
            ws = torch.empty(max(1, (nbytes + 3) // 4), dtype=torch.float32, device=t.device)
            rc = L.b200dn_welch_psd(flat[i0:i1].data_ptr(), i1 - i0, n, out[i0:i1].data_ptr(), ws.data_ptr(), ws.numel() * 4,
                                    torch.cuda.current_stream(t.device).cuda_stream)
            _lib.check(rc, "welch_psd")
    f = np.arange(129, dtype=np.float64) / 256.0
    return f, out.reshape(t.shape[:-1] + (129,))


def high_frequency_psd_mae(gt, pred, high_freq_threshold: float = 0.5) -> torch.Tensor:
    """``mean(|Pxx_gt[f >= thr * max f] - Pxx_pred[...]|)`` per image — the statistic plot.py:159-165 derives from the
    three Welch calls.  gt, pred: [B, ...] CUDA batches; returns a float32 CUDA tensor [B] (no host sync)."""
    g = _as_dev_f32(gt)
    p = _as_dev_f32(pred, g)
    f, pg = welch(g.flatten(1))
    _, pp = welch(p.flatten(1))
    idx = torch.from_numpy(np.nonzero(f >= high_freq_threshold * f.max())[0]).to(g.device)
    return (pg.index_select(1, idx) - pp.index_select(1, idx)).abs().mean(dim=1)
