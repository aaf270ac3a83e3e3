"""GPU: DISTS (DISTS_pytorch 0.1) on the B200 against the fp64 oracle — each convolution under the convolution bound of
tests/helpers.py, each L2 pooling and the head alone from the kernels' own inputs, and the whole metric end to end;
near-miss references the end-to-end bound must reject; reproducibility, batch independence, symmetry, return shapes,
CUDA-graph capture and the error paths."""
import pytest
import torch
import torch.nn.functional as F

from oracle import dists_oracle
from helpers import bound_tol, kernel_conv, tol_excess
from vub_image_denoising_b200 import _lib, perceptual
from vub_image_denoising_b200.perceptual import DISTS

pytestmark = pytest.mark.gpu
DEV = "cuda"
PREC = perceptual.PREC
SHAPES = [(1, 256, 256), (16, 256, 256), (64, 256, 256), (2, 250, 200), (2, 97, 131), (2, 16, 16)]


def _state_dict(seed=0):
    """torchvision's default VGG16 init (seeded) for the trunk, nonnegative uniform alpha / beta."""
    import torchvision
    torch.manual_seed(seed)
    tv = torchvision.models.vgg16(weights=None).features
    sd = DISTS().state_dict()
    for idx in dists_oracle.CONV_INDICES:
        sd[dists_oracle.key(idx) + ".weight"] = tv[idx].weight.detach().clone()
        sd[dists_oracle.key(idx) + ".bias"] = tv[idx].bias.detach().clone()
    sd["alpha"], sd["beta"] = torch.rand(1, 1475, 1, 1), torch.rand(1, 1475, 1, 1)
    return sd


def _model(sd):
    m = DISTS()
    m.load_state_dict(sd)
    return m.to(DEV)


def _images(N, H, W, seed):
    """Smooth images in [0, 1] and two partners: sigma = 25/255 noise and 2/255 noise."""
    g = torch.Generator().manual_seed(seed)
    low = torch.rand(N, 3, max(2, H // 32), max(2, W // 32), generator=g)
    clean = F.interpolate(low, size=(H, W), mode="bicubic", align_corners=False).clamp(0, 1)
    noisy = (clean + torch.randn(clean.shape, generator=g) * 25 / 255).clamp(0, 1)
    near = (clean + torch.randn(clean.shape, generator=g) * 2 / 255).clamp(0, 1)
    return [t.to(DEV) for t in (clean, noisy, near)]


def _bound(ref):
    """The end-to-end target, LPIPS's: |err| <= 1e-4 max(|ref|, 1e-2).  Measured on a B200 (148 SMs, 1000 W power
    limit): the largest |err| / bound over SHAPES and both partners was 0.229 (16 x 16, sigma = 2/255 partner); the
    weakest near-miss rejection was stage 0 omitted, at 3.3 x the bound (250 x 200)."""
    return 1e-4 * ref.abs().clamp_min(1e-2)


def _planes(a):
    """An NHWC hi + lo activation as the exact fp64 NCHW value the kernels read."""
    v = a.hi.view(torch.bfloat16).double() + a.lo.view(torch.bfloat16).double()
    return v.permute(0, 3, 1, 2).contiguous()


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
        assert got.shape == ((N,) if N > 1 else ()) and got.dtype == torch.float32 and got.is_cuda
        ref = dists_oracle.dists(sd64, clean, other)
        err = (got.double().reshape(-1) - ref).abs()
        print(f"N={N} {H}x{W}: DISTS {float(ref.min()):.4g}..{float(ref.max()):.4g}, "
              f"max |err| / bound {float((err / _bound(ref)).max()):.3f}")
        assert bool((err <= _bound(ref)).all())


@pytest.mark.parametrize("N,H,W", [(1, 256, 256), (2, 97, 131)])
def test_each_stage_from_its_own_input(model, sd, N, H, W):
    """Every convolution from the kernel's own stored input under helpers.bound_tol with the existing kappa (conv1_1 is
    the MODE_CONV1X1 GEMM over K = 27 gathered columns, the rest the 3x3 path); every L2 pooling against fp64 conv2d of
    its own stored input, within the storage bound.  Measured on a B200 (148 SMs, 1000 W): largest kappa 20.8
    (conv1_2 at 97 x 131; the existing KAPPA = 48 holds it), the L2 poolings need none beyond the storage rounding."""
    clean, noisy, _ = _images(N, H, W, seed=7)
    with torch.no_grad():
        model(clean, noisy)
    plan = model.plan(N, H, W)
    torch.cuda.synchronize()
    x = dists_oracle.normalise(torch.cat([clean, noisy]).cpu(), sd)        # in fp32, the operations the gather fuses
    feats = [_planes(f).cpu() for f in plan.features]
    pools = [_planes(p).cpu() for p in plan.pools]
    for k, (f, p) in enumerate(zip(feats[:4], pools)):
        filt = sd[dists_oracle.key(dists_oracle.POOL_INDICES[k]) + ".filter"].double()
        ref = (F.conv2d(f ** 2, filt, stride=2, padding=1, groups=f.shape[1]) + 1e-12).sqrt()
        err = (p - ref).abs()
        print(f"{H}x{W} L2 pool {k + 1}: kappa needed {tol_excess(err, ref, ref, PREC):.2f}")
        assert bool((err <= bound_tol(ref, ref, PREC)).all()), f"pool {k + 1}"
    convs = iter(dists_oracle.CONV_INDICES)
    for s, outs in enumerate(plan.conv_outs):
        inp = x if s == 0 else pools[s - 1]
        for i, out in enumerate(outs):
            idx = next(convs)
            key = dists_oracle.key(idx)
            w, b = sd[key + ".weight"], sd[key + ".bias"].double()
            val, S = kernel_conv(lambda a, ww: F.conv2d(a, ww, padding=1), inp.float(), w, PREC)
            ref = torch.relu(val + b.view(1, -1, 1, 1))
            S = S + b.abs().view(1, -1, 1, 1)
            got = _planes(out).cpu()
            err = (got - ref).abs()
            print(f"{H}x{W} conv{s + 1}_{i + 1}: kappa needed {tol_excess(err, ref, S, PREC):.2f}")
            assert bool((err <= bound_tol(ref, S, PREC)).all()), f"conv{s + 1}_{i + 1}"
            inp = got


@pytest.mark.parametrize("N,H,W", [(16, 256, 256), (2, 97, 131)])
def test_head_alone_matches_fp64_head(model, sd, N, H, W):
    clean, noisy, near = _images(N, H, W, seed=3)
    for other in (noisy, near):
        with torch.no_grad():
            got = model(clean, other).reshape(-1)
        plan = model.plan(N, H, W)
        f = [_planes(a) for a in plan.features]
        ref = dists_oracle.head([clean.double()] + [t[:N] for t in f], [other.double()] + [t[N:] for t in f],
                                sd["alpha"].double().to(DEV), sd["beta"].double().to(DEV))
        err = float((got.double() - ref).abs().max())
        print(f"head alone {H}x{W}: max |err| {err:.3g}")       # on a B200 (1000 W): 1.3e-9 at most
        assert bool(((got.double() - ref).abs() <= 2.0 ** -24 * ref.abs().clamp_min(2 ** -7)).all())


def _near_miss_refs(sd64, a, b):
    """References that each get one detail of DISTS wrong."""
    al, be = sd64["alpha"].double(), sd64["beta"].double()
    feats = dists_oracle.vgg_features(sd64, torch.float64, DEV)
    f = lambda x: dists_oracle.features(feats, x.double(), sd64)                   # noqa: E731
    fa, fb = f(a), f(b)
    out = {}
    mx = dists_oracle.vgg_features(sd64, torch.float64, DEV, pool="max")
    out["max-pool instead of L2 pool"] = dists_oracle.head(dists_oracle.features(mx, a.double(), sd64),
                                                           dists_oracle.features(mx, b.double(), sd64), al, be)
    out["no ImageNet normalisation"] = dists_oracle.head(
        dists_oracle.features(feats, a.double(), sd64, normalise_input=False),
        dists_oracle.features(feats, b.double(), sd64, normalise_input=False), al, be)

    def raw_pad(x):
        x = x.double()
        h = dists_oracle.normalise(F.pad(x, (1, 1, 1, 1)), sd64)
        h = torch.relu(F.conv2d(h, feats[0].weight, feats[0].bias))
        out_, h = [x], feats[1:4](h)
        out_.append(h)
        for s, e in dists_oracle.STAGES[1:]:
            h = feats[s:e](h)
            out_.append(h)
        return out_
    with torch.no_grad():
        out["padding the raw image"] = dists_oracle.head(raw_pad(a), raw_pad(b), al, be)
    keep = torch.ones_like(al)
    keep[:, :3] = 0
    out["stage 0 omitted"] = dists_oracle.head(fa, fb, al * keep, be * keep)
    out["unbiased variance"] = dists_oracle.head(fa, fb, al, be, unbiased=True)
    out["alpha / beta not divided by their sum"] = dists_oracle.head(fa, fb, al, be, divide=False)
    return out


# near misses the bound cannot tell apart at any of the shapes below (measured on a B200); reported, not dropped
INDISTINGUISHABLE = ()


def test_bound_rejects_near_miss_references(model, sd):
    """Each near miss is printed with max over pairs of |got - miss| / bound at each shape; every one must exceed 1 at
    one shape at least, except those listed in INDISTINGUISHABLE."""
    N = 2
    worst = {}
    for H, W in ((250, 200), (97, 131)):
        clean, noisy, _ = _images(N, H, W, seed=17)
        sd64 = {k: v.to(DEV) for k, v in sd.items()}
        with torch.no_grad():
            got = model(clean, noisy).double()
            ref = dists_oracle.dists(sd64, clean, noisy)
            assert bool(((got - ref).abs() <= _bound(ref)).all())
            for name, miss in _near_miss_refs(sd64, clean, noisy).items():
                r = float(((got - miss).abs() / _bound(miss)).max())
                print(f"{H}x{W} {name}: max |got - miss| / bound = {r:.3g}")
                worst[name] = max(worst.get(name, 0.0), r)
    not_rejected = sorted(n for n, r in worst.items() if r <= 1)
    print("not rejected at any shape:", not_rejected)
    assert not_rejected == sorted(INDISTINGUISHABLE)


def test_identities_and_reproducibility(model):
    clean, noisy, _ = _images(64, 256, 256, seed=29)
    with torch.no_grad():
        same = model(clean, clean)
        ab, ba = model(clean, noisy), model(noisy, clean)
        ab2 = model(clean, noisy)
        singles = torch.stack([model(clean[i:i + 1], noisy[i:i + 1]) for i in range(64)])
    assert bool((same.abs() <= _bound(same)).all())
    assert torch.equal(ab, ba)
    assert torch.equal(ab, ab2)
    assert torch.equal(ab, singles)
    assert bool((ab > 0).all())


def test_return_shapes(model):
    clean, noisy, _ = _images(3, 64, 48, seed=31)
    with torch.no_grad():
        many = model(clean, noisy)
        one = model(clean[:1], noisy[:1])
        avg = model(clean, noisy, batch_average=True)
        avg1 = model(clean[:1], noisy[:1], batch_average=True)
    assert many.shape == (3,) and one.shape == () and avg.shape == () and avg1.shape == ()
    assert torch.equal(one, many[0])
    assert torch.equal(avg, many.mean())


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
        with pytest.raises(RuntimeError, match=r"\[N, 3, H, W\]"):
            model(torch.zeros(2, 1, 64, 64, device=DEV), torch.zeros(2, 1, 64, 64, device=DEV))
        with pytest.raises(RuntimeError, match="below 16"):
            model(torch.zeros(1, 3, 15, 64, device=DEV), torch.zeros(1, 3, 15, 64, device=DEV))
        with pytest.raises(RuntimeError, match="inference-only"):
            model(x, x, require_grad=True)
    with pytest.raises(RuntimeError, match="inference-only"):
        model(x.clone().requires_grad_(), x)
    L = _lib.lib()
    f = torch.zeros(64 * 9, device=DEV)
    p = x.data_ptr()
    assert L.b200dn_l2pool3x3s2(p, p, 1, 8, 8, 12, f.data_ptr(), PREC, p, p, None) == _lib.E_ARG      # C % 8
    assert L.b200dn_l2pool3x3s2(p, p, 1, 0, 8, 8, f.data_ptr(), PREC, p, p, None) == _lib.E_ARG       # H = 0
    assert L.b200dn_l2pool3x3s2(p, p, 1, 8, 8, 8, None, PREC, p, p, None) == _lib.E_ARG              # no filter
    assert L.b200dn_l2pool3x3s2(p, None, 1, 8, 8, 8, f.data_ptr(), PREC, p, None, None) == _lib.E_ARG  # lo plane
