"""GPU: structural_similarity with every option (ssim_window_kernel) against the SSIM oracle, the fp64 definition of
the map, near-miss references the bounds must reject, identities with the default kernel, and reproducibility."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.ndimage import zoom

import vub_image_denoising_b200 as b2
from oracle import ssim_oracle as so
from test_ssim_window_oracle import CONFIG_IDS, CONFIGS, WANG
from vub_image_denoising_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = "cuda"
SHAPES = [(4, 3, 256, 256), (3, 3, 40, 72), (2, 1, 11, 11), (1, 3, 33, 45), (2, 1, 7, 7)]
# Per-pixel bound of the map: KAPPA * 2^-24 * ((ux^2 + uy^2 + |uxx| + |uyy|) / (vx + vy + C2) + 1), fp64 moments: the
# fp32 window sums of x^2 + y^2 and of the means cancel in vx + vy down to that size.  The largest kappa needed by
# test_map_matches_fp64_definition on a B200 (1000 W power limit) was 4.24 (uniform 15x15, population covariance,
# R = 1); scipy's fp32 map (the oracle) needs 3.4 on such inputs (CPU).
KAPPA = 64.0


def _images(n, c, h, w, seed, data_range, noise=0.1):
    g = torch.Generator().manual_seed(seed)
    a = torch.rand(n, c, h, w, generator=g)
    b = (a + torch.randn(n, c, h, w, generator=g) * noise).clamp(0, 1)
    return a * data_range, b * data_range


def _smooth_pair(data_range, noise=2 / 255, seed=1):
    """A smooth 256 x 256 plane (bicubic zoom of 8 x 8 noise) and a noisy copy, in [0, R]."""
    rng = np.random.default_rng(seed)
    clean = np.clip(zoom(rng.random((8, 8)), 32, order=3), 0, 1).astype(np.float32)
    noisy = np.clip(clean + rng.normal(0, noise, clean.shape), 0, 1).astype(np.float32)
    return clean * np.float32(data_range), noisy * np.float32(data_range)


def _map_bound(ref, data_range, K2=0.03):
    scale = (ref["ux"] ** 2 + ref["uy"] ** 2 + np.abs(ref["uxx"]) + np.abs(ref["uyy"])) / \
        (ref["vx"] + ref["vy"] + (K2 * data_range) ** 2)
    return KAPPA * 2.0 ** -24 * (scale + 1.0), scale + 1.0


@pytest.mark.parametrize("name,kw,min_side", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("data_range", [1.0, 2.0, 255.0])
def test_mean_matches_oracle(name, kw, min_side, data_range, built_lib):
    for shape in SHAPES:
        if min(shape[-2:]) < min_side:
            continue
        a, b = _images(*shape, seed=sum(shape), data_range=data_range)
        P = shape[0] * shape[1]
        got = b2.metrics.batch_ssim_planes(a.to(DEV).view(P, *shape[2:]), b.to(DEV).view(P, *shape[2:]), data_range,
                                           **kw).cpu().numpy()
        pa, pb = a.view(P, *shape[2:]).numpy(), b.view(P, *shape[2:]).numpy()
        for p in range(P):
            want = so._ssim_plane(pa[p], pb[p], data_range, **kw)
            assert abs(got[p] - want) <= 1e-5, (shape, p, got[p], want)
        want = so.structural_similarity(a[0].numpy(), b[0].numpy(), data_range, channel_axis=0, **kw)
        assert b2.metrics.structural_similarity(a[0].to(DEV), b[0].to(DEV), data_range=data_range, channel_axis=0,
                                                **kw) == pytest.approx(want, abs=1e-5)


@pytest.mark.parametrize("name,kw,min_side", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("data_range", [1.0, 255.0])
def test_map_matches_fp64_definition(name, kw, min_side, data_range, built_lib):
    """The map, borders included, against the fp64 brute force, on a smooth pair (where vx + vy cancels most) and a
    noisy one, under the per-pixel bound above; the mean is the map's over the crop.  (On the 7 x 7 plane the crop is
    one pixel of the smooth pair, where fp32 cancellation moves S by 1e-4: the 1e-5 mean bound does not apply.)"""
    size = 7 if name == "gauss_sigma3_win7" else 96
    pairs = [_smooth_pair(data_range), _smooth_pair(data_range, noise=0.1, seed=2)]
    for clean, noisy in pairs:
        c, n = clean[:size, :size], noisy[:size, :size]
        mean, S = b2.metrics.structural_similarity(torch.from_numpy(c).to(DEV), torch.from_numpy(n).to(DEV),
                                                   data_range=data_range, full=True, **kw)
        assert S.shape == c.shape and S.dtype == torch.float32 and S.is_cuda
        ref = so.ssim_window_bruteforce(c, n, data_range, **kw)
        err = np.abs(S.cpu().numpy().astype(np.float64) - ref["S"])
        bound, unit = _map_bound(ref, data_range, kw.get("K2", 0.03))
        kappa = float((err / (2.0 ** -24 * unit)).max())
        print(f"{name} R={data_range}: kappa needed {kappa:.2f}")
        assert np.all(err <= bound), kappa
        pad = kw.get("win_size", 11 if kw.get("gaussian_weights") else 7) // 2
        assert mean == pytest.approx(float(S[pad:size - pad, pad:size - pad].double().mean()), abs=1e-6)


def test_bounds_reject_near_miss_references(built_lib):
    for R in (1.0, 255.0):
        clean, noisy = _smooth_pair(R)
        got, S = b2.metrics.batch_ssim_planes(torch.from_numpy(clean)[None].to(DEV),
                                              torch.from_numpy(noisy)[None].to(DEV), R, full=True, **WANG)
        got, S = float(got[0]), S[0].cpu().numpy().astype(np.float64)
        ref = so.ssim_window_bruteforce(clean, noisy, R, **WANG)
        assert abs(got - ref["mean"]) <= 1e-5 and np.all(np.abs(S - ref["S"]) <= _map_bound(ref, R)[0])
        for miss_kw in (dict(truncate=4.0), dict(use_sample_covariance=True), dict(crop=3)):
            miss = so.ssim_window_bruteforce(clean, noisy, R, **{**WANG, **miss_kw})["mean"]
            print(f"R={R} {miss_kw}: |got - miss| = {abs(got - miss):.3g}")
            assert abs(got - miss) > 1e-5, miss_kw
        for mode in ("nearest", "constant", "mirror"):
            miss = so.ssim_window_bruteforce(clean, noisy, R, mode=mode, **WANG)
            ratio = float((np.abs(S - miss["S"]) / _map_bound(miss, R)[0]).max())
            print(f"R={R} border {mode}: max |S - miss| / bound = {ratio:.3g}")
            assert ratio > 1, mode


def _pre_existing_ssim_planes(a, b, data_range):
    """The default call exactly as it was before the window options: b200dn_ssim over the planes."""
    P, H, W = a.shape
    L = _lib.lib()
    out = torch.empty(P, dtype=torch.float64, device=a.device)
    ws = torch.empty(max(1, (L.b200dn_ssim_workspace_bytes(P, H, W) + 7) // 8), dtype=torch.float64, device=a.device)
    rc = L.b200dn_ssim(a.data_ptr(), b.data_ptr(), P, H, W, float(data_range), out.data_ptr(), ws.data_ptr(),
                       ws.numel() * 8, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ssim")
    return out / float((H - 6) * (W - 6))


def test_identities(built_lib):
    a, b = _images(4, 3, 256, 256, seed=3, data_range=1.0)
    A, B = a.to(DEV).view(12, 256, 256), b.to(DEV).view(12, 256, 256)
    old = _pre_existing_ssim_planes(A, B, 1.0)
    assert torch.equal(b2.metrics.batch_ssim_planes(A, B, 1.0), old)
    assert torch.equal(b2.metrics.batch_ssim_planes(A, B, 1.0, win_size=7, use_sample_covariance=True, K1=0.01,
                                                    K2=0.03, sigma=3.0), old)
    forced, maps = b2.metrics.batch_ssim_planes(A, B, 1.0, full=True)      # ssim_window_kernel on the default window
    assert float((forced - old).abs().max()) <= 1e-6
    assert maps.shape == (12, 256, 256)
    for kw in (WANG, dict(win_size=11)):
        same, smap = b2.metrics.batch_ssim_planes(A, A, 1.0, full=True, **kw)
        assert float((same - 1).abs().max()) <= 1e-6 and float((smap - 1).abs().max()) <= 1e-5
        ab = b2.metrics.batch_ssim_planes(A, B, 1.0, **kw)
        ba = b2.metrics.batch_ssim_planes(B, A, 1.0, **kw)
        assert float((ab - ba).abs().max()) <= 1e-6
        chw = b2.metrics.structural_similarity(A[:3], B[:3], data_range=1.0, channel_axis=0, full=True, **kw)
        hwc = b2.metrics.structural_similarity(A[:3].permute(1, 2, 0), B[:3].permute(1, 2, 0), data_range=1.0,
                                               channel_axis=-1, full=True, **kw)
        assert chw[0] == hwc[0] and hwc[1].shape == (256, 256, 3) and torch.equal(hwc[1], chw[1].permute(1, 2, 0))


def test_reproducible_and_batch_independent(built_lib):
    a, b = _images(64, 3, 256, 256, seed=5, data_range=1.0)
    A, B = a.to(DEV).view(-1, 256, 256), b.to(DEV).view(-1, 256, 256)
    for full in (False, True):
        r0 = b2.metrics.batch_ssim_planes(A, B, 1.0, full=full, **WANG)
        m0, s0 = r0 if full else (r0, None)
        for _ in range(3):
            r1 = b2.metrics.batch_ssim_planes(A, B, 1.0, full=full, **WANG)
            m1, s1 = r1 if full else (r1, None)
            assert torch.equal(m0, m1) and (not full or torch.equal(s0, s1))
        for i in range(64):
            r1 = b2.metrics.batch_ssim_planes(A[3 * i:3 * i + 3], B[3 * i:3 * i + 3], 1.0, full=full, **WANG)
            m1, s1 = r1 if full else (r1, None)
            assert torch.equal(m1, m0[3 * i:3 * i + 3]) and (not full or torch.equal(s1, s0[3 * i:3 * i + 3]))


def test_device_error_paths(built_lib):
    a, b = _images(1, 1, 32, 32, seed=7, data_range=1.0)
    A, B = a[0, 0].to(DEV), b[0, 0].to(DEV)
    ss = b2.metrics.structural_similarity
    with pytest.raises(ValueError, match="Window size must be odd"):
        ss(A, B, data_range=1.0, win_size=8)
    with pytest.raises(ValueError, match="win_size exceeds image extent"):
        ss(A[:10], B[:10], data_range=1.0, gaussian_weights=True)
    with pytest.raises(ValueError, match="K1 must be positive"):
        ss(A, B, data_range=1.0, K1=-1.0)
    with pytest.raises(ValueError, match="K2 must be positive"):
        ss(A, B, data_range=1.0, K2=-1.0)
    with pytest.raises(ValueError, match="sigma must be positive"):
        ss(A, B, data_range=1.0, gaussian_weights=True, sigma=-1.0)
    with pytest.raises(NotImplementedError):
        ss(A, B, data_range=1.0, gradient=True)
    with pytest.raises(NotImplementedError):
        ss(torch.zeros(40, 40, device=DEV), torch.zeros(40, 40, device=DEV), data_range=1.0, win_size=33)
    with pytest.raises(TypeError):
        ss(A, B, data_range=1.0, truncate=4.0)
    # the C ABI checks its own arguments
    L = _lib.lib()
    o = b2.metrics._ssim_window_opts(32, 32, 1.0, None, True, 1.5, False, 0.01, 0.03)
    o.radius = 16
    out = torch.empty(1, dtype=torch.float64, device=DEV)
    ws = torch.empty(64, dtype=torch.float64, device=DEV)
    rc = L.b200dn_ssim_window(A.data_ptr(), B.data_ptr(), 1, 32, 32, ctypes.byref(o), out.data_ptr(), None,
                              ws.data_ptr(), ws.numel() * 8, None)
    assert rc == _lib.E_ARG and b"radius" in L.b200dn_last_error()
