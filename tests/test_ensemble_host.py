"""CPU: the x8 self-ensemble's transforms and batch layout (oracle/ensemble_oracle.py against include/b200dn.h), the
oracle's composition, and the errors of the product entry points without a GPU."""
import itertools
import subprocess
from pathlib import Path

import pytest
import torch

import vub_image_denoising_b200 as b2
from vub_image_denoising_b200 import _lib
from oracle import ensemble_oracle as eo

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("H,W", [(6, 6), (5, 7)])
def test_transforms_are_distinct_and_invert_exactly(H, W):
    x = torch.randn(2, 3, H, W, generator=torch.Generator().manual_seed(H * W))
    ts = [eo.transform(x, k) for k in range(8)]
    for k, t in enumerate(ts):
        assert t.shape == ((2, 3, H, W) if k % 2 == 0 else (2, 3, W, H))
        assert torch.equal(eo.inverse(t, k), x)
    for a, b in itertools.combinations(range(8), 2):
        assert not (ts[a].shape == ts[b].shape and torch.equal(ts[a], ts[b])), f"T_{a} == T_{b}"


def test_transforms_are_the_dihedral_group():
    """Closed under composition, and T_k for k >= 4 are the reflections (order 2); k = 1, 3 the quarter turns."""
    x = torch.arange(30.).view(1, 1, 5, 6)
    ts = [eo.transform(x, k) for k in range(8)]
    for a, b in itertools.product(range(8), repeat=2):
        ab = eo.transform(eo.transform(x, b), a)
        assert any(t.shape == ab.shape and torch.equal(t, ab) for t in ts)
    for k in range(4, 8):
        assert torch.equal(eo.transform(ts[k], k), x)
    assert torch.equal(ts[1], torch.rot90(x, 1, dims=[2, 3])) and torch.equal(ts[4], torch.flip(x, dims=[3]))


def _header_layout(B: int):
    """(group, index) of every (k, b) as the C compiler evaluates b200dn.h's macros"""
    body = "".join(f'printf("%d %d ", B200DN_DIHEDRAL_GROUP({k}), B200DN_DIHEDRAL_INDEX({k}, {b}, {B}));'
                   for k in range(8) for b in range(B))
    src = f'#include "b200dn.h"\n#include <stdio.h>\nint main(){{{body}return 0;}}'
    exe = ROOT / "vub_image_denoising_b200" / "build" / "dihedral_layout"
    exe.parent.mkdir(exist_ok=True)
    subprocess.run(["gcc", "-x", "c", "-", "-I", str(ROOT / "include"), "-o", str(exe)], input=src, text=True, check=True)
    v = [int(s) for s in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    return {(k, b): (v[2 * (k * B + b)], v[2 * (k * B + b) + 1]) for k in range(8) for b in range(B)}


def test_group_layout_matches_the_header():
    B = 3
    x = torch.randn(B, 2, 4, 7, generator=torch.Generator().manual_seed(1))
    groups = eo.expand(x)
    assert groups[0].shape == (4 * B, 2, 4, 7) and groups[1].shape == (4 * B, 2, 7, 4)
    layout = _header_layout(B)
    assert sorted(layout.values()) == [(g, i) for g in (0, 1) for i in range(4 * B)]     # a bijection onto both groups
    for (k, b), (g, i) in layout.items():
        assert (g, i) == (eo.group(k), eo.index(k, b, B))
        assert torch.equal(groups[g][i], eo.transform(x, k)[b])
    # the oracle's reduce reads the images where the layout puts them: T_k^-1 of group image i is x[b] for every k
    even, odd = groups
    assert torch.equal(eo.reduce(even, odd), eo.self_ensemble(lambda t: t, x))


def test_self_ensemble_of_the_identity_is_the_input():
    """The 8 partial sums k*x are exact in fp32 when x has at most 21 significant bits (here k/2^12, |k| < 2^12), so the
    mean of 8 copies of x is x bit for bit; on arbitrary fp32 data 3x and later partial sums round."""
    g = torch.Generator().manual_seed(5)
    x = torch.randint(-4095, 4096, (2, 3, 8, 16), generator=g).float() / 4096
    assert torch.equal(eo.self_ensemble(lambda t: t, x), x)
    assert torch.equal(eo.reduce(*eo.expand(x)), x)
    xs = torch.randint(-4095, 4096, (1, 1, 8, 8), generator=g).float() / 4096
    assert torch.equal(eo.self_ensemble(lambda t: t, xs), xs)


def test_reduce_adds_in_k_order():
    """The 8 values 1, 2^-24 x 7 round differently in other orders: (((1 + e) + e) ...) stays 1, a sum that starts
    with the small values does not."""
    B, e = 1, 2.0 ** -24
    ys = [torch.full((B, 1, 2, 2), 1.0 if k == 0 else e) for k in range(8)]
    even = torch.cat([eo.transform(ys[k], k) for k in (0, 2, 4, 6)])
    odd = torch.cat([eo.transform(ys[k], k) for k in (1, 3, 5, 7)])
    assert torch.equal(eo.reduce(even, odd), torch.full((B, 1, 2, 2), 0.125))
    rev = ys[7]
    for y in reversed(ys[:7]):
        rev = rev + y
    assert not torch.equal(rev * 0.125, torch.full((B, 1, 2, 2), 0.125))


def test_cpu_tensors_raise_no_cpu_fallback():
    net = b2.RDUNet(base_filters=16).eval()
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=16), timesteps=2).eval()
    with torch.no_grad():
        for model in (net, dm):
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                b2.self_ensemble(model, torch.zeros(1, 3, 16, 16))
        with pytest.raises(TypeError, match="RDUNet"):
            b2.self_ensemble(b2.RDUNet_T(base_filters=16).eval(), torch.zeros(1, 3, 16, 16))
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            b2.ops.dihedral_expand(torch.zeros(1, 3, 16, 16))


def test_entry_points_reject_bad_arguments(built_lib):
    L, p = built_lib, 0x1000
    calls = (lambda a, b, c, shape: L.b200dn_dihedral_expand(a, *shape, b, c, None),      # x, even, odd
             lambda a, b, c, shape: L.b200dn_dihedral_reduce(a, b, *shape, c, None))      # even, odd, out
    for call in calls:
        for ptrs in ((None, p, p), (p, None, p), (p, p, None)):
            assert call(*ptrs, (1, 3, 8, 8)) == _lib.E_ARG
            assert b"null pointer" in L.b200dn_last_error()
        for shape in ((0, 3, 8, 8), (1, 0, 8, 8), (1, 3, 0, 8), (1, 3, 8, -1)):
            assert call(p, p, p, shape) == _lib.E_ARG
            assert b"bad shape" in L.b200dn_last_error()
        assert call(p, p, p, (1, 1, 32 * 65535 + 1, 8)) == _lib.E_ARG


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_gpu_means_error_not_fallback(built_lib):
    p = 0x1000
    assert built_lib.b200dn_dihedral_expand(p, 1, 3, 37, 53, p, p, None) == _lib.E_CUDA
    assert built_lib.b200dn_dihedral_reduce(p, p, 1, 3, 37, 53, p, None) == _lib.E_CUDA
