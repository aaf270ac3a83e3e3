"""ORACLE (test infrastructure, not product): skimage 0.22 ``structural_similarity`` with all of its options.

PARITY UNPINNED, as for ``metrics_oracle``'s SSIM: scikit-image==0.22.0 is not installed here and no reference test
holds a value.  This module restates the published algorithm for every option the device implements:

  * the filter is ``scipy.ndimage.gaussian_filter(sigma, truncate=3.5, mode='reflect')`` with ``gaussian_weights``,
    else ``uniform_filter(size=win_size)`` (mode 'reflect');
  * ``win_size`` defaults to ``2 * int(3.5 * sigma + 0.5) + 1`` with Gaussian weights and to 7 otherwise; it sets the
    covariance normaliser (``NP / (NP - 1)``, ``NP = win_size ** 2``, with ``use_sample_covariance``, else 1) and the
    crop ``(win_size - 1) // 2``;
  * ``C1 = (K1 * R) ** 2``, ``C2 = (K2 * R) ** 2``; float32 arithmetic for float32 input; the map S over the whole
    plane, its fp64 mean over the cropped interior; per-channel means stored as float32 and averaged.

With their defaults ``_ssim_plane`` and ``structural_similarity`` are ``metrics_oracle``'s functions (a CPU test holds
them equal bit for bit).  ``ssim_window_bruteforce`` is an independent fp64 evaluation of the same definition with
explicit windows, weights and border index maps.
"""
from __future__ import annotations

import numpy as np
from scipy.ndimage import gaussian_filter, uniform_filter

TRUNCATE = 3.5


def _check(K1: float, K2: float, sigma: float) -> None:
    if K1 < 0:
        raise ValueError("K1 must be positive")
    if K2 < 0:
        raise ValueError("K2 must be positive")
    if sigma < 0:
        raise ValueError("sigma must be positive")


def _ssim_plane(im1: np.ndarray, im2: np.ndarray, data_range: float, win_size=None, *, gaussian_weights=False,
                sigma=1.5, use_sample_covariance=True, K1=0.01, K2=0.03, full=False):
    _check(K1, K2, sigma)
    if win_size is None:
        win_size = 2 * int(TRUNCATE * sigma + 0.5) + 1 if gaussian_weights else 7
    if min(im1.shape) < win_size:
        raise ValueError("win_size exceeds image extent.")
    if not (win_size % 2 == 1):
        raise ValueError("Window size must be odd.")
    ftype = np.float32 if im1.dtype in (np.float16, np.float32) else np.float64
    im1 = im1.astype(ftype, copy=False)
    im2 = im2.astype(ftype, copy=False)
    NP = win_size ** im1.ndim
    cov_norm = NP / (NP - 1) if use_sample_covariance else 1.0
    if gaussian_weights:
        def filt(x):
            return gaussian_filter(x, sigma=sigma, truncate=TRUNCATE, mode="reflect")
    else:
        def filt(x):
            return uniform_filter(x, size=win_size)
    ux = filt(im1)
    uy = filt(im2)
    uxx = filt(im1 * im1)
    uyy = filt(im2 * im2)
    uxy = filt(im1 * im2)
    vx = cov_norm * (uxx - ux * ux)
    vy = cov_norm * (uyy - uy * uy)
    vxy = cov_norm * (uxy - ux * uy)
    R = data_range
    C1 = (K1 * R) ** 2
    C2 = (K2 * R) ** 2
    A1, A2, B1, B2 = (2 * ux * uy + C1, 2 * vxy + C2, ux ** 2 + uy ** 2 + C1, vx + vy + C2)
    S = (A1 * A2) / (B1 * B2)
    pad = (win_size - 1) // 2
    mssim = S[pad:S.shape[0] - pad, pad:S.shape[1] - pad].mean(dtype=np.float64)
    return (mssim, S) if full else mssim


def structural_similarity(im1: np.ndarray, im2: np.ndarray, data_range: float, channel_axis=None, *, full=False,
                          **kwargs):
    """kwargs: win_size, gaussian_weights, sigma, use_sample_covariance, K1, K2 (as ``_ssim_plane``).  With
    ``full=True`` returns ``(mean, S)``, S in the input's layout."""
    if im1.shape != im2.shape:
        raise ValueError("Input images must have the same dimensions.")
    if channel_axis is None:
        res = _ssim_plane(im1, im2, data_range, full=full, **kwargs)
        return (float(res[0]), res[1]) if full else float(res)
    a = np.moveaxis(im1, channel_axis, 0)
    b = np.moveaxis(im2, channel_axis, 0)
    ftype = np.float32 if im1.dtype in (np.float16, np.float32) else np.float64
    per = np.empty(a.shape[0], dtype=ftype)
    S = np.empty(a.shape, dtype=ftype)
    for c in range(a.shape[0]):
        res = _ssim_plane(a[c], b[c], data_range, full=True, **kwargs)
        per[c], S[c] = res
    return (float(per.mean()), np.moveaxis(S, 0, channel_axis)) if full else float(per.mean())


def _border_index(i: int, n: int, mode: str) -> int:
    """scipy.ndimage's extension of a line of n samples to index i; -1 stands for the constant 0."""
    if mode == "constant":
        return i if 0 <= i < n else -1
    if mode == "nearest":
        return min(max(i, 0), n - 1)
    while not 0 <= i < n:          # bounce off the ends as often as it takes
        if mode == "reflect":      # d c b a | a b c d | d c b a
            i = -i - 1 if i < 0 else 2 * n - 1 - i
        elif mode == "mirror":     # d c b | a b c d | c b a
            if n == 1:
                return 0
            i = -i if i < 0 else 2 * n - 2 - i
        else:
            raise ValueError(mode)
    return i


def ssim_window_bruteforce(im1: np.ndarray, im2: np.ndarray, data_range: float, *, win_size=None,
                           gaussian_weights=False, sigma=1.5, use_sample_covariance=True, K1=0.01, K2=0.03,
                           truncate=TRUNCATE, mode="reflect", crop=None) -> dict:
    """Independent fp64 evaluation of one plane: each pixel's (2r+1) x (2r+1) window of weighted samples, the border
    samples picked by an explicit index map, centred moments.  Returns the mean and the maps S, ux, uy, uxx, uyy
    (raw second moments), vx, vy.  ``truncate``, ``mode`` and ``crop`` build near-miss references for tests."""
    x = im1.astype(np.float64)
    y = im2.astype(np.float64)
    H, W = x.shape
    if gaussian_weights:
        r = int(truncate * sigma + 0.5)
        t = np.arange(-r, r + 1, dtype=np.float64)
        w = np.exp(-t * t / (2.0 * sigma * sigma)) if sigma > 1e-15 else np.ones(1)
        w = w / w.sum()
        if win_size is None:
            win_size = 2 * int(TRUNCATE * sigma + 0.5) + 1
    else:
        win_size = 7 if win_size is None else win_size
        r = (win_size - 1) // 2
        w = np.full(win_size, 1.0 / win_size)
    w2 = np.outer(w, w)
    iy = [_border_index(i, H, mode) for i in range(-r, H + r)]
    ix = [_border_index(i, W, mode) for i in range(-r, W + r)]

    def extend(z):
        iya, ixa = np.array(iy), np.array(ix)
        e = z[np.ix_(np.maximum(iya, 0), np.maximum(ixa, 0))]
        e[iya < 0, :] = 0.0
        e[:, ixa < 0] = 0.0
        return e

    xe, ye = extend(x), extend(y)
    windows = [(w2[ky, kx], xe[ky:ky + H, kx:kx + W], ye[ky:ky + H, kx:kx + W])
               for ky in range(2 * r + 1) for kx in range(2 * r + 1)]
    ux = sum(wk * xs for wk, xs, _ in windows)
    uy = sum(wk * ys for wk, _, ys in windows)
    uxx = sum(wk * xs * xs for wk, xs, _ in windows)
    uyy = sum(wk * ys * ys for wk, _, ys in windows)
    NP = win_size ** 2
    cov = NP / (NP - 1) if use_sample_covariance else 1.0
    vx = cov * sum(wk * (xs - ux) ** 2 for wk, xs, _ in windows)
    vy = cov * sum(wk * (ys - uy) ** 2 for wk, _, ys in windows)
    vxy = cov * sum(wk * (xs - ux) * (ys - uy) for wk, xs, ys in windows)
    C1, C2 = (K1 * data_range) ** 2, (K2 * data_range) ** 2
    S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))
    p = (win_size - 1) // 2 if crop is None else crop
    return dict(mean=float(S[p:H - p, p:W - p].mean()), S=S, ux=ux, uy=uy, uxx=uxx, uyy=uyy, vx=vx, vy=vy)
