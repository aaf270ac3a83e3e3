"""CPU: the pieces of the BM3D contract (transforms, opponent space, Kaiser taps, reference grid, group rules,
thresholds), the oracle's behaviour on easy inputs and its PSNR on a synthetic image, the ctypes mirror of
b200dn_bm3d_args and the API's error paths."""
import ctypes
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import bm3d_oracle as bo
from vub_image_denoising_b200 import _lib
import vub_image_denoising_b200 as b2

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "vub_image_denoising_b200" / "csrc" / "bm3d.cu"


def test_dct_and_haar_are_orthonormal():
    D = bo.dct_matrix()
    assert np.abs(D @ D.T - np.eye(8)).max() < 1e-14
    x = np.random.default_rng(0).standard_normal((8, 8))
    assert np.abs(D.T @ (D @ x @ D.T) @ D - x).max() < 1e-14
    for n in (1, 2, 4, 8, 16, 32):
        Hn = bo.haar_matrix(n)
        assert np.abs(Hn @ Hn.T - np.eye(n)).max() < 1e-14
        v = np.random.default_rng(n).standard_normal(n)
        assert np.abs(Hn.T @ (Hn @ v) - v).max() < 1e-14
    assert np.allclose(bo.haar_matrix(2), np.array([[1, 1], [1, -1]]) / np.sqrt(2))


def test_opponent_matrix_and_channel_sigmas():
    assert np.abs(bo.A @ bo.A_INV - np.eye(3)).max() < 1e-15
    assert np.abs(bo.A_INV @ bo.A - np.eye(3)).max() < 1e-15
    assert np.allclose(bo.CHANNEL_NORM, [0.5774, 0.7071, 0.6124], atol=5e-5)


def test_kernel_kaiser_taps_equal_np_kaiser():
    """The kernel's constant taps, read from its source, are np.kaiser(8, 2.0) to the bit."""
    body = re.search(r"c_kaiser\[BS\] = \{(.*?)\};", CSRC.read_text(), flags=re.S).group(1)
    taps = [float.fromhex(t.strip()) for t in body.split(",")]
    assert taps == np.kaiser(8, 2.0).tolist()
    assert np.array_equal(bo.kaiser2d(), np.outer(np.kaiser(8, 2.0), np.kaiser(8, 2.0)))


@pytest.mark.parametrize("n", range(8, 41))
def test_reference_positions_cover_every_pixel(n):
    p = bo.ref_positions(n)
    assert len(p) == bo.n_ref(n) == _lib.bm3d_nref(n)
    assert p[0] == 0 and p[-1] == n - 8 and (np.diff(p) > 0).all() and (np.diff(p) <= 3).all()
    covered = np.zeros(n, dtype=bool)
    for r in p:
        covered[r:r + 8] = True
    assert covered.all()
    assert bo.n_ref(256) == 84 and bo.n_ref(97) == 31


def test_tau_int_equals_the_integer_formula():
    assert bo.tau_int(3000) == 3000 * 64 * 2 ** 20 // 255 ** 2 == 3096141
    assert bo.tau_int(400) == 400 * 64 * 2 ** 20 // 255 ** 2 == 412818
    src = CSRC.read_text()
    assert "TAU_HT = 3096141" in src and "TAU_WIE = 412818" in src


def _plane(H, W, seed=0):
    return np.random.default_rng(seed).integers(0, 4096, size=(H, W)).astype(np.int64)


def test_ties_at_d_zero_put_the_reference_first_then_d_r_c():
    """A periodic plane (period 3 in both directions): many candidates at d = 0, before and after the reference."""
    tile = _plane(3, 3)
    q = np.tile(tile, (10, 10))[:30, :30]
    pos, size = bo.block_match(q, 16, bo.tau_int(3000))
    W = 30
    g = pos[3, 3]                                   # reference (9, 9): d = 0 candidates at (9 +- 3k, 9 +- 3l)
    assert g[0] == 9 * W + 9 and size[3, 3] == 16
    rc = [(p // W, p % W) for p in g[1:]]
    assert rc == sorted(rc) and all((r - 9) % 3 == 0 and (c - 9) % 3 == 0 for r, c in rc)
    assert rc[0] == (0, 0)                          # (0, 0) precedes the reference in (r, c) but comes after it
    wrong, _ = bo.block_match(q, 16, bo.tau_int(3000), ref_first=False)
    assert wrong[3, 3, 0] == 0


def test_power_of_two_cut_and_inclusive_tau():
    """A flat plane with one candidate made to sit exactly at tau, and the rest far away."""
    H = W = 8 + 2                                   # references at 0, 2 along each edge: 3 candidates per axis
    q = np.zeros((H, W), dtype=np.int64)
    q[:, 9] = 5000                                  # every block touching column 9 is far (d >= 8 * 5000^2)
    pos, size = bo.block_match(q, 16, 0)            # reference (0, 0): candidates (r, c) with c <= 1 have d = 0
    assert size[0, 0] == 4                          # 1 + 5 kept -> cut to 4
    assert list(pos[0, 0, :4]) == [0, 1, W, W + 1] and (pos[0, 0, 4:] == -1).all()
    q2 = np.zeros((8, 9), dtype=np.int64)
    q2[0, 8] = 7                                    # the candidate at (0, 1) differs from the reference by d = 49
    assert bo.block_match(q2, 16, 49)[1][0, 0] == 2
    assert bo.block_match(q2, 16, 48)[1][0, 0] == 1


def test_search_window_is_clipped_not_shifted():
    q = np.zeros((8, 60), dtype=np.int64)
    pos, size = bo.block_match(q, 32, 0)
    # reference at column 0: candidates at columns 1..19 only (not shifted to 0..38)
    g = pos[0, 0]
    assert size[0, 0] == 16 and g[0] == 0 and list(g[1:16]) == list(range(1, 16))
    full, fsize = bo.block_match(q, 64, 0)
    assert fsize[0, 0] == 16                        # 20 blocks in the clipped window -> 16
    pos, size = bo.block_match(q, 32, 0)
    assert list(pos[0, -1, :4]) == [52, 33, 34, 35]      # last reference at column 52: window 33..52


def test_oracle_is_the_identity_at_tiny_sigma_and_keeps_a_constant_image():
    z = bo.synthetic(3, 32, 40, seed=3)
    out = bo.bm3d(z, 1e-6)
    assert np.abs(out - z).max() < 1e-5
    const = np.full((1, 24, 24), 0.375, dtype=np.float32)
    assert np.abs(bo.stage1(const, 25 / 255)["out"] - 0.375).max() < 1e-12
    # stage 2 keeps the one nonzero coefficient, DC = 0.375 * 8 * sqrt(32), at its Wiener gain DC^2 / (DC^2 + sigma^2)
    dc2 = (0.375 * 8) ** 2 * 32
    assert np.abs(bo.bm3d(const, 25 / 255) - 0.375 * dc2 / (dc2 + (25 / 255) ** 2)).max() < 1e-12


@pytest.mark.parametrize("C", [1, 3])
def test_oracle_lifts_psnr_and_stage2_beats_stage1(C):
    """Low-passed synthetic image at sigma = 25/255 (DESIGN.md records the figures)."""
    clean = bo.synthetic(C, 64, 64, seed=1)
    z = bo.noisy(clean, 25 / 255, seed=2)
    s1 = bo.stage1(z, 25 / 255)["out"]
    s2 = bo.stage2(z, s1.astype(np.float32), 25 / 255)["out"]
    psnr = [10 * np.log10(1 / np.mean((x - clean) ** 2)) for x in (z, s1, s2)]
    print(f"C={C}: PSNR noisy {psnr[0]:.2f} dB, stage 1 {psnr[1]:.2f} dB, stage 2 {psnr[2]:.2f} dB")
    assert psnr[1] > psnr[0] + 8 and psnr[2] > psnr[1]


def test_bm3d_args_layout_matches_the_header(built_lib):
    c_names = ["z", "basic", "sigma", "B", "C", "H", "W", "stages", "out", "match1", "size1", "match2", "size2"]
    body = "".join(f'printf("%zu ", offsetof(b200dn_bm3d_args, {n}));' for n in c_names)
    body += 'printf("%zu %d %d %d %d ", sizeof(b200dn_bm3d_args), B200DN_BM3D_HARD_THRESHOLDING, B200DN_BM3D_ALL_STAGES,'
    body += ' B200DN_BM3D_N2_HT, B200DN_BM3D_N2_WIE);'
    body += "".join(f'printf("%d ", B200DN_BM3D_NREF({n}));' for n in range(8, 41))
    src = f'#include "b200dn.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(){{{body}return 0;}}'
    exe = ROOT / "vub_image_denoising_b200" / "build" / "offsets_bm3d"
    exe.parent.mkdir(exist_ok=True)
    subprocess.run(["gcc", "-x", "c", "-", "-I", str(ROOT / "include"), "-o", str(exe)], input=src, text=True, check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    py_names = [n for n, _ in _lib.Bm3dArgs._fields_]
    assert py_names == c_names
    assert [getattr(_lib.Bm3dArgs, n).offset for n in py_names] == vals[:13]
    assert ctypes.sizeof(_lib.Bm3dArgs) == vals[13]
    assert vals[14:18] == [_lib.BM3D_HARD_THRESHOLDING, _lib.BM3D_ALL_STAGES, _lib.BM3D_N2_HT, _lib.BM3D_N2_WIE]
    assert vals[18:] == [bo.n_ref(n) for n in range(8, 41)]


def test_c_abi_rejects_bad_arguments(built_lib):
    a = _lib.Bm3dArgs(z=8, sigma=8, out=8, B=1, C=3, H=16, W=16, stages=3)
    assert built_lib.b200dn_bm3d_workspace_bytes(ctypes.byref(a)) > 16 * 16 * 3 * 8 * 4
    for field, value in (("C", 2), ("H", 7), ("W", 7), ("B", 0), ("stages", 2), ("out", None)):
        bad = _lib.Bm3dArgs.from_buffer_copy(a)
        setattr(bad, field, value)
        assert built_lib.b200dn_bm3d_workspace_bytes(ctypes.byref(bad)) == _lib.E_ARG, field
        assert built_lib.b200dn_bm3d(ctypes.byref(bad), 8, 1 << 30, None) == _lib.E_ARG, field
    bad = _lib.Bm3dArgs.from_buffer_copy(a)
    bad.basic, bad.stages = 8, 1
    assert built_lib.b200dn_bm3d(ctypes.byref(bad), 8, 1 << 30, None) == _lib.E_ARG
    assert built_lib.b200dn_bm3d(ctypes.byref(a), 8, 16, None) == _lib.E_ARG          # workspace too small
    assert built_lib.b200dn_bm3d(None, 8, 1 << 30, None) == _lib.E_ARG


def test_api_errors():
    img = np.full((16, 16, 3), 0.5, dtype=np.float32)
    with pytest.raises(NotImplementedError):
        b2.bm3d.bm3d_rgb(img, 0.1, profile="refilter")
    with pytest.raises(NotImplementedError):
        b2.bm3d.bm3d_rgb(img, 0.1, colorspace="YCbCr")
    with pytest.raises(NotImplementedError):
        b2.bm3d.bm3d_rgb(img, np.ones((16, 16)))
    with pytest.raises(NotImplementedError):
        b2.bm3d.bm3d(img[..., 0], 0.1, blockmatches=(True, False))
    with pytest.raises(RuntimeError, match="positive"):
        b2.bm3d.bm3d_rgb(img, 0.0)
    with pytest.raises(RuntimeError, match="positive"):
        b2.bm3d.bm3d(img[..., 0], [-0.1])
    with pytest.raises(RuntimeError, match="at least 8"):
        b2.bm3d.bm3d_rgb(img[:7], 0.1)
    with pytest.raises(RuntimeError, match="at least 8"):
        b2.bm3d.bm3d(torch.zeros(1, 1, 16, 5), 0.1)
    with pytest.raises(RuntimeError, match="x 3"):
        b2.bm3d.bm3d_rgb(img[..., :2], 0.1)
    with pytest.raises(RuntimeError, match=r"\[B, 3, H, W\]"):
        b2.bm3d.bm3d_rgb(torch.zeros(1, 2, 16, 16), 0.1)
    with pytest.raises(RuntimeError, match=r"\[B, 1, H, W\]"):
        b2.bm3d.bm3d(torch.zeros(1, 3, 16, 16), 0.1)
    with pytest.raises(RuntimeError, match="inference only"):
        b2.bm3d.bm3d(torch.zeros(1, 1, 16, 16, requires_grad=True), 0.1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        b2.bm3d.bm3d(torch.zeros(1, 1, 16, 16), 0.1)
    with pytest.raises(RuntimeError, match="1 or B = 2"):
        b2.bm3d.bm3d(torch.zeros(2, 1, 16, 16), [0.1, 0.1, 0.1])
    with pytest.raises(RuntimeError, match="does not match"):
        b2.bm3d.bm3d_rgb(img, 0.1, stage_arg=img[:12])
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            b2.bm3d.bm3d_rgb(img, 0.1)


def test_custom_op_fake_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        z, s = torch.empty(2, 3, 20, 30), torch.empty(2)
        shapes = [tuple(t.shape) for t in torch.ops.b200dn.bm3d(z, s, None, _lib.BM3D_ALL_STAGES, True)]
        assert shapes == [(2, 3, 20, 30), (2, 5, 9, 16), (2, 5, 9), (2, 5, 9, 32), (2, 5, 9)]
        shapes = [tuple(t.shape) for t in torch.ops.b200dn.bm3d(z, s, z, _lib.BM3D_ALL_STAGES, False)]
        assert shapes == [(2, 3, 20, 30), (0,), (0,), (0,), (0,)]
