"""GPU: the x8 geometric self-ensemble.  The two kernels against the torch restatement (oracle/ensemble_oracle.py) bit
for bit; self_ensemble around RDUNet and the sampler against the composition of 8 calls at batch B (bit for bit: an
image's output does not depend on its batch) and against the fp32 CPU oracle under the per-forward bar; equivariance;
reproducibility, CUDA-graph capture and the error paths."""
import numpy as np
import pytest
import torch

from helpers import check_bar
import vub_image_denoising_b200 as b2
from oracle import ensemble_oracle as eo
from oracle import rdunet_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda"
GUARD = 1024                      # floats of sentinel around every output buffer
SENTINEL = -12345.5


def _guarded(n: int) -> torch.Tensor:
    return torch.full((n + 2 * GUARD,), SENTINEL, device=DEV)


def _inner(buf: torch.Tensor, shape, offset: int = 0) -> torch.Tensor:
    n = int(np.prod(shape))
    return buf[GUARD + offset:GUARD + offset + n].view(shape)


def _guards_intact(buf: torch.Tensor, n: int, offset: int = 0) -> bool:
    return bool((buf[:GUARD + offset] == SENTINEL).all() and (buf[GUARD + offset + n:] == SENTINEL).all())


@pytest.mark.parametrize("H,W,offset", [(256, 256, 0), (96, 160, 0), (37, 53, 0), (36, 52, 0), (96, 160, 1)])
@pytest.mark.parametrize("B,C", [(1, 1), (1, 3), (3, 1), (3, 3)])
def test_kernels_match_the_oracle(B, C, H, W, offset, built_lib):
    """Square, non-square, odd sizes (partial transpose tiles, 32-bit path), multiples of 4 off the tile grid and
    pointers 4 bytes off the 16-byte grid (128-bit path not taken).  Only the output ranges are written."""
    L = built_lib
    g = torch.Generator().manual_seed(B * 1000 + C * 100 + H + W)
    x_cpu = torch.randn(B, C, H, W, generator=g)
    xbuf = _guarded(x_cpu.numel())
    x = _inner(xbuf, x_cpu.shape, offset)
    x.copy_(x_cpu.to(DEV))
    n = 4 * x.numel()
    ebuf, obuf = _guarded(n), _guarded(n)
    even, odd = _inner(ebuf, (4 * B, C, H, W), offset), _inner(obuf, (4 * B, C, W, H), offset)
    stream = torch.cuda.current_stream().cuda_stream
    assert L.b200dn_dihedral_expand(x.data_ptr(), B, C, H, W, even.data_ptr(), odd.data_ptr(), stream) == 0
    want_e, want_o = eo.expand(x_cpu)
    assert torch.equal(even.cpu(), want_e) and torch.equal(odd.cpu(), want_o)
    assert _guards_intact(ebuf, n, offset) and _guards_intact(obuf, n, offset)
    assert torch.equal(x.cpu(), x_cpu) and _guards_intact(xbuf, x.numel(), offset)
    # reduce of 8 independent images per output: a position read from the wrong transform or an add out of order shows
    ye_cpu, yo_cpu = torch.randn(4 * B, C, H, W, generator=g), torch.randn(4 * B, C, W, H, generator=g)
    even.copy_(ye_cpu.to(DEV))
    odd.copy_(yo_cpu.to(DEV))
    outbuf = _guarded(x.numel())
    out = _inner(outbuf, x.shape, offset)
    assert L.b200dn_dihedral_reduce(even.data_ptr(), odd.data_ptr(), B, C, H, W, out.data_ptr(), stream) == 0
    assert torch.equal(out.cpu(), eo.reduce(ye_cpu, yo_cpu))
    assert _guards_intact(outbuf, x.numel(), offset)
    # the custom ops give the same bits (flat [even | odd] buffer)
    buf = b2.ops.dihedral_expand(x)
    assert torch.equal(buf[:n].view(4 * B, C, H, W).cpu(), want_e)
    assert torch.equal(buf[n:].view(4 * B, C, W, H).cpu(), want_o)
    assert torch.equal(b2.ops.dihedral_reduce(even, odd), out)


def _noisy(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    clean = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    return (clean + torch.randn(B, 3, H, W, generator=g) * (25 / 127.5)).clamp(-1, 1), clean


@pytest.mark.parametrize("H,W", [(256, 256), (96, 160)])
@pytest.mark.parametrize("F,B", [(32, 2), (128, 1)])
def test_rdunet_self_ensemble(F, B, H, W, built_lib):
    """Against the composition of 8 forwards at batch B (bit for bit) and against the fp32 CPU oracle through the
    same composition (the per-forward bar of test_gpu_network.py)."""
    torch.manual_seed(F + H)
    net = b2.RDUNet(base_filters=F).eval()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.to(DEV)
    noisy, clean = _noisy(B, H, W, F * 7 + W)
    x = noisy.to(DEV)
    keep = x.clone()
    with torch.no_grad():
        got = b2.self_ensemble(net, x)
        comp = eo.self_ensemble(net, x)
        ref = eo.self_ensemble(lambda t: orc.rdunet_forward(sd, t), noisy)
    assert torch.equal(x, keep), "self_ensemble wrote its input"
    assert got.shape == (B, 3, H, W) and got.dtype == torch.float32
    d = float((got - comp).abs().max())
    assert torch.equal(got, comp), f"self_ensemble differs from 8 forwards at batch {B}: max |diff| {d:.3e}"
    frac, mx = check_bar(got.cpu(), ref, clean, what=f"self_ensemble(RDUNet({F})) {H}x{W}")
    print(f"RDUNet({F}) B={B} {H}x{W}: {frac * 100:.3f} % within 1/255 of the oracle, max err {mx:.2e}")


def test_sampler_self_ensemble_full_size(built_lib):
    """B = 2 at 256 x 256, T = 20, the sampler's own precision: one improved_sampling call over 16 images equals the
    8 calls over 2 images bit for bit."""
    torch.manual_seed(3)
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=32), timesteps=20).to(DEV).eval()
    y = _noisy(2, 256, 256, 31)[0].to(DEV)
    keep = y.clone()
    got = b2.self_ensemble(dm, y)
    comp = eo.self_ensemble(dm.improved_sampling, y)
    assert torch.equal(y, keep)
    d = float((got - comp).abs().max())
    assert torch.equal(got, comp), f"sampler ensemble differs from 8 calls at batch 2: max |diff| {d:.3e}"
    assert not dm.last_saturated


@pytest.mark.parametrize("H,W", [(64, 64), (32, 48)])
def test_sampler_self_ensemble_vs_oracle(H, W, built_lib):
    torch.manual_seed(5)
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=32), timesteps=3).eval()
    sd = {k: v.clone() for k, v in dm.state_dict().items()}
    dm = dm.to(DEV)
    noisy, clean = _noisy(2, H, W, 41 + W)
    got = b2.self_ensemble(dm, noisy.to(DEV))
    with torch.no_grad():
        ref = eo.self_ensemble(lambda t: orc.improved_sampling(sd, t, 3), noisy)
        comp = eo.self_ensemble(dm.improved_sampling, noisy.to(DEV))
    assert torch.equal(got, comp)
    frac, mx = check_bar(got.cpu(), ref, clean, what=f"sampler self_ensemble T=3 {H}x{W}")
    print(f"sampler T=3 {H}x{W}: {frac * 100:.3f} % within 1/255 of the oracle, max err {mx:.2e}")


@pytest.mark.parametrize("H,W", [(96, 160), (64, 64)])
def test_equivariance(H, W, built_lib):
    """self_ensemble(T_m(x)) == T_m(self_ensemble(x)) up to the add order: the same 8 network outputs, summed in a
    permuted order.  Two orders of an 8-term fp32 sum differ by at most 2 * 7u * sum|y_k| (u = 2^-24), times 0.125."""
    torch.manual_seed(9)
    net = b2.RDUNet(base_filters=32).to(DEV).eval()
    x = _noisy(2, H, W, 77)[0].to(DEV)
    with torch.no_grad():
        base = b2.self_ensemble(net, x)
        mean_abs = eo.self_ensemble(lambda t: net(t).abs(), x)     # sum_k |y_k| * 0.125, y_k = T_k^-1 net(T_k x)
        worst, equal = 0.0, 0
        for m in range(8):
            a = b2.self_ensemble(net, eo.transform(x, m).contiguous())
            b = eo.transform(base, m)
            bound = 14 * 2.0 ** -24 * eo.transform(mean_abs, m) * (1 + 1e-6)
            err = (a - b).abs()
            assert bool((err <= bound).all()), f"m = {m}: {float((err / bound).max()):.2f} of the bound"
            worst = max(worst, float((err / bound).max()))
            equal += int(torch.equal(a, b))
    print(f"equivariance {H}x{W}: at most {worst:.3f} of the bound; {equal} of 8 transforms bit-equal")


def test_reproducible_capturable_and_input_untouched(built_lib):
    torch.manual_seed(13)
    net = b2.RDUNet(base_filters=32).to(DEV).eval()
    xs = [_noisy(2, 96, 160, s)[0].to(DEV) for s in (1, 2)]
    with torch.no_grad():
        keep = xs[0].clone()
        a, b = b2.self_ensemble(net, xs[0]), b2.self_ensemble(net, xs[0])
        assert torch.equal(a, b) and a.data_ptr() != b.data_ptr()
        assert torch.equal(xs[0], keep)
        want = b2.self_ensemble(net, xs[1])
        static_x = xs[0].clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            b2.self_ensemble(net, static_x)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y = b2.self_ensemble(net, static_x)
        static_x.copy_(xs[1])
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(y, want)
    # the sampler inside a caller's capture (its own graph is not used then)
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=16), timesteps=3).to(DEV).eval()
    ys = [_noisy(1, 32, 32, s)[0].to(DEV) for s in (3, 4)]
    want = b2.self_ensemble(dm, ys[1])
    static_y = ys[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        b2.self_ensemble(dm, static_y)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y = b2.self_ensemble(dm, static_y)
    static_y.copy_(ys[1])
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y, want)


def test_error_paths(built_lib):
    net = b2.RDUNet(base_filters=16).to(DEV).eval()
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=16), timesteps=2).to(DEV).eval()
    with torch.no_grad():
        for model in (net, dm):
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                b2.self_ensemble(model, torch.zeros(1, 3, 16, 16))
            with pytest.raises(RuntimeError, match="divisible by 8"):
                b2.self_ensemble(model, torch.zeros(1, 3, 20, 32, device=DEV))
            with pytest.raises(RuntimeError, match="channels"):
                b2.self_ensemble(model, torch.zeros(1, 4, 16, 16, device=DEV))
    with pytest.raises(RuntimeError, match="inference-only"):
        b2.self_ensemble(net.train(), torch.zeros(1, 3, 16, 16, device=DEV))
    with pytest.raises(RuntimeError, match="inference-only"):
        b2.self_ensemble(net.eval(), torch.zeros(1, 3, 16, 16, device=DEV, requires_grad=True))
    with pytest.raises(RuntimeError, match="not .4B, C, H, W."):
        b2.ops.dihedral_reduce(torch.zeros(4, 3, 8, 16, device=DEV), torch.zeros(4, 3, 8, 16, device=DEV))
