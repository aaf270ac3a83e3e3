"""CPU: the SSIM oracle with every structural_similarity option (Gaussian or uniform windows of any odd size, sample or
population covariance, K1/K2, the map) against an independent fp64 brute force, the host-side Gaussian taps against
scipy, and the argument checks of the device entry points."""
import numpy as np
import pytest
from scipy.ndimage import gaussian_filter1d

from oracle import metrics_oracle as mo
from oracle import ssim_oracle as so
from vub_image_denoising_b200 import metrics

WANG = dict(gaussian_weights=True, sigma=1.5, use_sample_covariance=False)
# (name, keywords, smallest plane side the window needs)
CONFIGS = [
    ("wang", WANG, 11),
    ("gauss_sample_cov", dict(gaussian_weights=True, sigma=1.5), 11),
    ("uniform3", dict(win_size=3), 3),
    ("uniform11", dict(win_size=11), 11),
    ("uniform15_population", dict(win_size=15, use_sample_covariance=False), 15),
    ("uniform7_K", dict(K1=0.02, K2=0.05), 7),
    ("gauss_win7", dict(gaussian_weights=True, win_size=7), 7),
    ("gauss_sigma3_win7", dict(gaussian_weights=True, sigma=3.0, win_size=7), 7),   # radius 11
]
CONFIG_IDS = [c[0] for c in CONFIGS]


def _pair(shape, seed, noise=0.1):
    rng = np.random.default_rng(seed)
    a = rng.random(shape, dtype=np.float32) * 2 - 1
    b = np.clip(a + rng.normal(0, noise, shape).astype(np.float32), -1, 1)
    return a, b


@pytest.mark.parametrize("name,kw,min_side", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("data_range", [1.0, 2.0])
def test_oracle_matches_bruteforce(name, kw, min_side, data_range):
    shape = (7, 7) if name == "gauss_sigma3_win7" else (24, 20)   # a filter wider than the plane bounces twice
    a, b = _pair(shape, 1)
    mean, S = so.structural_similarity(a, b, data_range, full=True, **kw)
    ref = so.ssim_window_bruteforce(a, b, data_range, **kw)
    assert S.shape == shape and S.dtype == np.float32
    assert mean == pytest.approx(ref["mean"], abs=2e-5)
    assert np.max(np.abs(S - ref["S"])) <= 2e-5          # borders included
    assert so.structural_similarity(a, b, data_range, **kw) == mean


def test_defaults_are_the_existing_oracle():
    a, b = _pair((3, 32, 40), 2)
    for R in (1.0, 2.0, 255.0):
        assert so.structural_similarity(a, b, R, channel_axis=0) == mo.structural_similarity(a, b, R, channel_axis=0)
        assert so._ssim_plane(a[0], b[0], R) == mo._ssim_plane(a[0], b[0], R)
    assert so.ssim_window_bruteforce(a[0, :24, :20], b[0, :24, :20], 1.0)["mean"] == \
        pytest.approx(mo.ssim_bruteforce(a[0, :24, :20], b[0, :24, :20], 1.0), abs=1e-12)


def test_channel_axis_map_layout():
    a, b = _pair((3, 24, 20), 3)
    m0, S0 = so.structural_similarity(a, b, 2.0, channel_axis=0, full=True, **WANG)
    m1, S1 = so.structural_similarity(a.transpose(1, 2, 0), b.transpose(1, 2, 0), 2.0, channel_axis=-1, full=True,
                                      **WANG)
    assert m0 == m1 and S1.shape == (24, 20, 3) and np.array_equal(S1, S0.transpose(1, 2, 0))


@pytest.mark.parametrize("sigma", [0.3, 1.0, 1.5, 2.5, 3.0, 4.4])
def test_gaussian_taps_are_scipys(sigma):
    """The weights the host hands the kernel are gaussian_filter1d's impulse response (truncate 3.5)."""
    r = int(3.5 * sigma + 0.5)
    impulse = np.zeros(4 * r + 1)
    impulse[2 * r] = 1.0
    response = gaussian_filter1d(impulse, sigma, truncate=3.5, mode="constant")
    assert np.count_nonzero(response) == 2 * r + 1
    np.testing.assert_allclose(metrics._gaussian_taps(sigma, r), response[r:3 * r + 1], rtol=1e-15, atol=0)


def test_window_options():
    o = metrics._ssim_window_opts(256, 256, 255.0, None, True, 1.5, False, 0.01, 0.03)    # Wang et al.
    assert (o.radius, o.win_size, o.cov_norm) == (5, 11, 1.0)
    assert o.C1 == np.float32((0.01 * 255.0) ** 2) and o.C2 == np.float32((0.03 * 255.0) ** 2)
    taps = np.array(o.weights[:11])
    assert np.array_equal(taps, metrics._gaussian_taps(1.5, 5).astype(np.float32)) and not np.any(o.weights[11:])
    o = metrics._ssim_window_opts(40, 40, 1.0, 7, True, 3.0, True, 0.01, 0.03)     # explicit win_size: radius from sigma
    assert (o.radius, o.win_size) == (11, 7) and o.cov_norm == np.float32(49 / 48)
    o = metrics._ssim_window_opts(40, 40, 1.0, 31, False, 1.5, True, 0.01, 0.03)
    assert (o.radius, o.win_size) == (15, 31) and np.all(np.array(o.weights) == np.float32(1 / 31))


def test_error_paths():
    def opts(H=32, W=32, win_size=None, gaussian_weights=False, sigma=1.5, K1=0.01, K2=0.03):
        return metrics._ssim_window_opts(H, W, 1.0, win_size, gaussian_weights, sigma, True, K1, K2)

    with pytest.raises(ValueError, match="Window size must be odd"):
        opts(win_size=8)
    with pytest.raises(ValueError, match="win_size exceeds image extent"):
        opts(H=6)
    with pytest.raises(ValueError, match="win_size exceeds image extent"):
        opts(W=10, gaussian_weights=True)
    with pytest.raises(ValueError, match="win_size exceeds image extent"):
        opts(H=9, win_size=10)                 # skimage checks the extent before the parity
    for kw, msg in ((dict(K1=-0.1), "K1 must be positive"), (dict(K2=-0.1), "K2 must be positive"),
                    (dict(sigma=-1.0, gaussian_weights=True), "sigma must be positive")):
        with pytest.raises(ValueError, match=msg):
            opts(**kw)
    with pytest.raises(NotImplementedError):
        opts(H=64, W=64, win_size=33)
    with pytest.raises(NotImplementedError):
        opts(H=64, W=64, gaussian_weights=True, sigma=4.5)      # radius 16
    opts(H=64, W=64, gaussian_weights=True, sigma=4.4)          # radius 15
    a, b = _pair((32, 32), 4)
    with pytest.raises(TypeError):
        metrics.structural_similarity(a, b, data_range=1.0, K3=0.1)
    with pytest.raises(NotImplementedError):
        metrics.structural_similarity(a, b, data_range=1.0, gradient=True)
    # the oracle raises the same way
    with pytest.raises(ValueError, match="Window size must be odd"):
        so.structural_similarity(a, b, 1.0, win_size=8)
    with pytest.raises(ValueError, match="sigma must be positive"):
        so.structural_similarity(a, b, 1.0, gaussian_weights=True, sigma=-1.0)
