"""GPU: LPIPS (lpips 0.1, net='alex') on the B200 against the fp64 oracle — each trunk tap per layer under the
convolution bound of tests/helpers.py, the head alone, and the whole metric end to end; reproducibility, batch
independence, symmetry, CUDA-graph capture and the error paths."""
import copy

import pytest
import torch
import torch.nn.functional as F

from oracle import lpips_oracle
from helpers import bound_tol, from_planes, kernel_conv, tol_excess
from vub_image_denoising_b200 import _lib, perceptual
from vub_image_denoising_b200.perceptual import LPIPS

pytestmark = pytest.mark.gpu
DEV = "cuda"
PREC = perceptual.PREC
SHAPES = [(1, 256, 256), (16, 256, 256), (64, 256, 256), (2, 96, 160), (2, 250, 200), (2, 31, 47)]


def _state_dict(seed=0, trunk_scale=1.0):
    """torchvision's default AlexNet init (seeded) for the trunk, nonnegative uniform lin weights."""
    import torchvision
    torch.manual_seed(seed)
    tv = torchvision.models.alexnet(weights=None)
    sd = LPIPS().state_dict()
    for key, idx in lpips_oracle.CONV_KEYS:
        s = trunk_scale if idx == 0 else 1.0
        sd[key + ".weight"] = tv.features[idx].weight.detach() * s
        sd[key + ".bias"] = tv.features[idx].bias.detach() * s
    for i, c in enumerate(perceptual.CHNS):
        sd[f"lin{i}.model.1.weight"] = sd[f"lins.{i}.model.1.weight"] = torch.rand(1, c, 1, 1)
    return sd


def _model(sd):
    m = LPIPS()
    m.load_state_dict(sd)
    return m.to(DEV)


def _images(N, H, W, seed):
    """Smooth images in [-1, 1] and two partners: sigma = 25/255 noise and 2/255 noise (in [0, 1] units)."""
    g = torch.Generator().manual_seed(seed)
    low = torch.rand(N, 3, max(2, H // 32), max(2, W // 32), generator=g)
    clean = F.interpolate(low, size=(H, W), mode="bicubic", align_corners=False).clamp(0, 1)
    noisy = (clean + torch.randn(clean.shape, generator=g) * 25 / 255).clamp(0, 1)
    near = (clean + torch.randn(clean.shape, generator=g) * 2 / 255).clamp(0, 1)
    return [(2 * t - 1).to(DEV) for t in (clean, noisy, near)]


def _bound(ref):
    """The end-to-end target.  Measured on a B200 (148 SMs, 1000 W power limit): the largest |err| / bound over
    SHAPES and both pairs was 0.020 (31 x 47, clean vs sigma = 25); the weakest near-miss rejection was padding the raw
    image, at 2.7 x the bound."""
    return 1e-4 * ref.abs().clamp_min(1e-2)


@pytest.fixture(scope="module")
def sd():
    return _state_dict()


@pytest.fixture(scope="module")
def model(sd):
    return _model(sd)


@pytest.mark.parametrize("N,H,W", SHAPES)
def test_end_to_end_matches_fp64_oracle(model, sd, N, H, W):
    clean, noisy, near = _images(N, H, W, seed=H * 1000 + W + N)
    sd64 = {k: v.to(DEV) for k, v in sd.items()}
    for other in (noisy, near):
        with torch.no_grad():
            got = model(clean, other)
        assert got.shape == (N, 1, 1, 1) and got.dtype == torch.float32 and got.is_cuda
        ref = lpips_oracle.lpips(sd64, clean, other)
        err = (got.double() - ref).abs()
        print(f"N={N} {H}x{W}: LPIPS {float(ref.min()):.4g}..{float(ref.max()):.4g}, "
              f"max |err| / bound {float((err / _bound(ref)).max()):.3f}")
        assert bool((err <= _bound(ref)).all())


@pytest.mark.parametrize("N,H,W", [(1, 256, 256), (2, 96, 160), (2, 31, 47)])
def test_each_tap_matches_fp64_under_the_conv_bound(model, sd, N, H, W):
    """Every tap from the kernel's own input (the previous tap, pooled) under helpers.bound_tol with the existing kappa:
    conv1 / conv2 are MODE_CONV1X1 GEMMs over gathered patches (K = 384 / N = 64, K = 1600 / N = 192), conv3..conv5 the
    3x3 path; the pools must equal max_pool2d of the kernel's own taps exactly.  Largest kappa needed on a B200
    (148 SMs, 1000 W): 4.5 (conv5 at 96 x 160)."""
    clean, noisy, _ = _images(N, H, W, seed=7)
    with torch.no_grad():
        model(clean, noisy)
    plan = model.plan(N, H, W)
    torch.cuda.synchronize()
    feats = [from_planes(f.hi, f.lo, PREC, 0, f.ctot).cpu() for f in plan.features]
    pools = [from_planes(p.hi, p.lo, PREC, 0, p.ctot).cpu() for p in (plan.pool1, plan.pool2)]
    assert torch.equal(pools[0], F.max_pool2d(feats[0], 3, 2))
    assert torch.equal(pools[1], F.max_pool2d(feats[1], 3, 2))
    x = lpips_oracle.scale(torch.cat([clean, noisy]).cpu(), sd)          # in fp32, the operations the gather fuses
    inputs = [x, pools[0], pools[1], feats[2], feats[3]]
    for i, (key, idx) in enumerate(lpips_oracle.CONV_KEYS):
        w, b = sd[key + ".weight"], sd[key + ".bias"].double()
        stride, pad = (4, 2) if i == 0 else (1, 2) if i == 1 else (1, 1)
        val, S = kernel_conv(lambda a, ww: F.conv2d(a, ww, stride=stride, padding=pad), inputs[i], w, PREC)
        ref = torch.relu(val + b.view(1, -1, 1, 1))
        S = S + b.abs().view(1, -1, 1, 1)
        err = (feats[i].double() - ref).abs()
        print(f"{H}x{W} conv{i + 1}: kappa needed {tol_excess(err, ref, S, PREC):.2f}")
        assert bool((err <= bound_tol(ref, S, PREC)).all()), f"conv{i + 1}"


@pytest.mark.parametrize("N,H,W", [(16, 256, 256), (2, 250, 200)])
def test_head_alone_matches_fp64_head(model, sd, N, H, W):
    clean, noisy, near = _images(N, H, W, seed=3)
    lins = [w.to(DEV) for w in lpips_oracle.lin_weights(sd)]
    for other in (noisy, near):
        with torch.no_grad():
            got = model(clean, other)
        plan = model.plan(N, H, W)
        f = [from_planes(a.hi, a.lo, PREC, 0, a.ctot).double() for a in plan.features]
        ref = lpips_oracle.head([t[:N] for t in f], [t[N:] for t in f], lins)
        rel = float(((got.double() - ref).abs() / ref).max())
        print(f"head alone {H}x{W}: max relative error {rel:.3g}")
        assert rel <= 1e-6      # measured on a B200 (1000 W): 6.6e-8 at most


def _near_miss_refs(sd64, a, b):
    """References that each get one detail of LPIPS wrong; the end-to-end bound must reject every one."""
    feats = lpips_oracle.alexnet_features(sd64, torch.float64, DEV)
    lins = lpips_oracle.lin_weights(sd64)
    sc = lambda x: lpips_oracle.scale(x.double(), sd64)                    # noqa: E731
    out = {"no scaling layer": lpips_oracle.head(lpips_oracle.taps(feats, a.double()),
                                                 lpips_oracle.taps(feats, b.double()), lins)}
    raw = copy.deepcopy(feats)
    raw[0].padding = (0, 0)
    out["padding the raw image"] = lpips_oracle.head(lpips_oracle.taps(raw, sc(F.pad(a, (2, 2, 2, 2)))),
                                                     lpips_oracle.taps(raw, sc(F.pad(b, (2, 2, 2, 2)))), lins)
    ceil = copy.deepcopy(feats)
    ceil[2].ceil_mode = ceil[5].ceil_mode = True
    out["ceil_mode pooling"] = lpips_oracle.head(lpips_oracle.taps(ceil, sc(a)), lpips_oracle.taps(ceil, sc(b)), lins)
    t0, t1 = lpips_oracle.taps(feats, sc(a)), lpips_oracle.taps(feats, sc(b))
    val = 0
    for f0, f1, w in zip(t0, t1, lins):
        n0 = f0 / torch.sqrt(torch.sum(f0 ** 2, dim=1, keepdim=True) + lpips_oracle.EPS)
        n1 = f1 / torch.sqrt(torch.sum(f1 ** 2, dim=1, keepdim=True) + lpips_oracle.EPS)
        val = val + F.conv2d((n0 - n1) ** 2, w.to(f0)).mean(dim=(2, 3), keepdim=True)
    out["eps inside the square root"] = val
    return out


def test_bound_rejects_near_miss_references():
    """At 250 x 200 the second pool's input is 30 x 24 (even), where ceil_mode adds a row and a column.  eps only
    matters where a feature vector's norm is near sqrt(1e-10): the second model scales conv1 by 2e-5 so that tap 0's
    norms are ~1e-4 and eps inside the root moves the result by ~1 % of tap 0's share."""
    N, H, W = 2, 250, 200
    clean, noisy, _ = _images(N, H, W, seed=17)
    for trunk_scale, must_reject in ((1.0, ("no scaling layer", "padding the raw image", "ceil_mode pooling")),
                                     (2e-5, ("eps inside the square root",))):
        sd = _state_dict(seed=1, trunk_scale=trunk_scale)
        sd64 = {k: v.to(DEV) for k, v in sd.items()}
        with torch.no_grad():
            got = _model(sd)(clean, noisy).double()
        ref = lpips_oracle.lpips(sd64, clean, noisy)
        assert bool(((got - ref).abs() <= _bound(ref)).all())
        misses = _near_miss_refs(sd64, clean, noisy)
        for name in must_reject:
            miss = misses[name]
            print(f"{name}: |got - miss| / bound = {float(((got - miss).abs() / _bound(miss)).min()):.3g}")
            assert bool(((got - miss).abs() > _bound(miss)).any()), name


def test_identities_and_reproducibility(model):
    clean, noisy, near = _images(64, 256, 256, seed=29)
    with torch.no_grad():
        zero = model(clean, clean)
        ab, ba = model(clean, noisy), model(noisy, clean)
        ab2 = model(clean, noisy)
        singles = torch.cat([model(clean[i:i + 1], noisy[i:i + 1]) for i in range(64)])
    assert torch.equal(zero, torch.zeros_like(zero))
    assert torch.equal(ab, ba)
    assert torch.equal(ab, ab2)
    assert torch.equal(ab, singles)
    assert bool((ab > 0).all())


def test_normalize_flag(model):
    clean, noisy, _ = _images(2, 64, 96, seed=31)
    with torch.no_grad():
        a = model((clean + 1) / 2, (noisy + 1) / 2, normalize=True)
        b = model(clean, noisy)
    assert torch.allclose(a, b, rtol=1e-5, atol=0)


def test_cuda_graph_replay_equals_eager(model):
    clean, noisy, _ = _images(4, 128, 128, seed=37)
    with torch.no_grad():
        eager = model(clean, noisy)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            model(clean, noisy)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = model(clean, noisy)
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


def test_error_paths(model):
    x = torch.zeros(2, 3, 64, 64, device=DEV)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            model(x.cpu(), x.cpu())
        with pytest.raises(RuntimeError, match="shape mismatch"):
            model(x, torch.zeros(2, 3, 64, 72, device=DEV))
        with pytest.raises(RuntimeError, match="below 31"):
            model(torch.zeros(1, 3, 30, 64, device=DEV), torch.zeros(1, 3, 30, 64, device=DEV))
        with pytest.raises(NotImplementedError):
            model(x, x, retPerLayer=True)
    with pytest.raises(RuntimeError, match="inference-only"):
        model(x.clone().requires_grad_(), x)
    L = _lib.lib()
    assert L.b200dn_maxpool3x3s2(x.data_ptr(), x.data_ptr(), 1, 2, 8, 8, PREC, x.data_ptr(), x.data_ptr(), None) == _lib.E_ARG
    assert L.b200dn_patch_gather(x.data_ptr(), None, 1, 8, 8, 8, 3, 3, 1, 1, 72, PREC, x.data_ptr(), None, None) == _lib.E_ARG
