"""GPU parity of every fused layer kernel, called through the C ABI (torch.ops.b200dn.* -> libb200dn.so),
against the oracle's arithmetic (plain fp64 conv / PReLU / add on the operands the kernel actually sees).

Reference semantics checked: Conv2d(3x3, pad 1)+PReLU with dense-block slice writes and `+ x` residual
(UNet/RDUNet_model.py:95-115), Conv2d(2x2, stride 2)+PReLU (:49-56), ConvTranspose2d(2x2, stride 2)+PReLU
scattered into the cat buffer (:58-69), OutputBlock.conv_2 + `+ inputs` (:83-93,186), InputBlock.conv_1 with
the RDUNet_T timestep plane (diffusion_denoising/Unet/Unet_model.py:133-136).
"""
import pytest
import torch
import torch.nn.functional as F

from helpers import (bound_tol, dense_block_ref, effective_input, effective_weight, kernel_conv, to_planes, two_planes,
                     dt16)
from vub_image_denoising_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda"
PRECS = [_lib.PREC_BF16, _lib.PREC_FP16, _lib.PREC_BF16X2, _lib.PREC_BF16X3, _lib.PREC_FP16X2]
PREC_IDS = ["bf16", "fp16", "bf16x2", "bf16x3", "fp16x2"]


def _rand(*shape, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


NAN16 = 0x7FFF          # a NaN in both fp16 and bf16: the poison of channels a kernel must not read or write


def _mk_out(B, H, W, ctot, prec):
    hi = torch.full((B, H, W, ctot), NAN16, dtype=torch.int16, device=DEV)
    lo = hi.clone() if two_planes(prec) else None
    return hi, lo


def _poison(x_hi, x_lo, c0):
    """NaN in channels [c0, ctot) of both input planes (0 x NaN is NaN: a read of them cannot go unnoticed)."""
    x_hi[..., c0:] = NAN16
    if x_lo is not None:
        x_lo[..., c0:] = NAN16


def _check_slice(hi, lo, prec, coff, cout, ref, S, what):
    """Channels [coff, coff + cout) of the output planes against the fp64 reference within helpers.bound_tol (S: the
    fp64 sum of |terms| of each output); every other byte keeps its NaN poison."""
    d = dt16(prec)
    got = hi.view(d)[..., coff:coff + cout].double()
    if lo is not None:
        got = got + lo.view(d)[..., coff:coff + cout].double()
    got = got.permute(0, 3, 1, 2).cpu()
    err = (got - ref).abs()
    bad = ~(err <= bound_tol(ref, S, prec))
    assert not bad.any(), f"{what}: {int(bad.sum())} / {bad.numel()} outside the bound, max err {float(err.max()):.3e}"
    # everything outside the slice must be untouched (the kernels write channel slices of shared buffers)
    mask = torch.ones(hi.shape[-1], dtype=torch.bool, device=hi.device)
    mask[coff:coff + cout] = False
    for p in (hi, lo):
        if p is not None:
            assert torch.all(p[..., mask] == NAN16), f"{what}: wrote outside its channel slice"


CONV_CASES = [
    # B, H, W, cin, cout, extra_in, ctot_out, coff, residual
    (1, 8, 16, 16, 16, 0, 16, 0, False),        # one full tile, one k16 step per tap
    (2, 24, 40, 80, 16, 16, 96, 80, False),     # dense-block growth slice, partial K block, partial tiles
    (1, 16, 16, 64, 64, 0, 64, 0, True),        # residual
    (1, 32, 32, 160, 64, 0, 160, 96, False),    # 3 K blocks (last partial)
    (1, 16, 32, 128, 256, 0, 256, 0, False),    # N = 256
    (1, 16, 16, 64, 512, 0, 512, 0, True),      # two N tiles + residual
    (1, 8, 8, 24, 8, 16, 40, 24, False),        # base_filters 16 level 0: cin 24, cout 8 (N padded to 16)
    (3, 40, 24, 48, 48, 0, 48, 0, True),        # N = 48
]


IMPLS = [1, 2, 3]
IMPL_IDS = ["tap", "slab", "slab-cta-pair"]   # 3 = cta_group::2 (falls back to the one-CTA slab kernel for N < 32)


@pytest.mark.parametrize("impl", IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize("prec", PRECS, ids=PREC_IDS)
@pytest.mark.parametrize("case", CONV_CASES, ids=[f"c{i}" for i in range(len(CONV_CASES))])
def test_conv3x3_bias_prelu(case, prec, impl, built_lib):
    B, H, W, cin, cout, extra, ctot_out, coff, residual = case
    x = _rand(B, cin, H, W, seed=1)
    w = _rand(cout, cin, 3, 3, seed=2, scale=(2.0 / (9 * cin)) ** 0.5)
    bias = _rand(cout, seed=3, scale=0.1)
    slope = torch.rand(cout, device=DEV) * 0.5
    x_hi, x_lo = to_planes(x, prec, ctot=cin + extra)
    _poison(x_hi, x_lo, cin)
    wp = torch.ops.b200dn.pack_weight(w, prec, False)
    out_hi, out_lo = _mk_out(B, H, W, ctot_out, prec)
    res = _rand(B, cout, H, W, seed=4) if residual else None
    r_hi, r_lo = to_planes(res, prec) if residual else (None, None)
    torch.ops.b200dn.conv_igemm(x_hi, x_lo, wp, bias, slope, _lib.MODE_CONV3X3, prec, cin, cout,
                                out_hi, out_lo, coff, r_hi, r_lo, 0, 0, 0, impl)
    torch.cuda.synchronize()
    b64 = bias.double().cpu().view(1, -1, 1, 1)
    pre, S = kernel_conv(lambda a, wt: F.conv2d(a, wt, padding=1), x, w, prec)
    ref, S = F.prelu(pre + b64, slope.double().cpu()), S + b64.abs()
    if residual:
        r = effective_input(res, prec).double().cpu()
        ref, S = ref + r, S + r.abs()
    _check_slice(out_hi, out_lo, prec, coff, cout, ref, S, "conv3x3")


@pytest.mark.parametrize("impl", IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize("block_n,max_ctas,m_tiles", [(16, 0, 1), (32, 3, 2), (64, 1, 2), (128, 0, 1), (128, 5, 2), (64, 0, 1)])
def test_conv3x3_tilings_agree(block_n, max_ctas, m_tiles, impl, built_lib):
    """Different N tilings / CTA counts (multi-tile persistence, TMEM double buffering) give the same bits."""
    prec = _lib.PREC_BF16
    B, H, W, cin, cout = 2, 32, 48, 96, 128
    x = _rand(B, cin, H, W, seed=5)
    w = _rand(cout, cin, 3, 3, seed=6, scale=0.05)
    bias = _rand(cout, seed=7, scale=0.1)
    slope = torch.full((cout,), 0.25, device=DEV)
    x_hi, _ = to_planes(x, prec)
    wp = torch.ops.b200dn.pack_weight(w, prec, False)
    base_hi, _ = _mk_out(B, H, W, cout, prec)
    torch.ops.b200dn.conv_igemm(x_hi, None, wp, bias, slope, _lib.MODE_CONV3X3, prec, cin, cout, base_hi, None, 0,
                                None, None, 0, 0, 0, impl)
    out_hi, _ = _mk_out(B, H, W, cout, prec)
    torch.ops.b200dn.conv_igemm(x_hi, None, wp, bias, slope, _lib.MODE_CONV3X3, prec, cin, cout, out_hi, None, 0,
                                None, None, block_n, max_ctas, m_tiles, impl)
    torch.cuda.synchronize()
    assert torch.equal(base_hi, out_hi)


CTA_PAIR_CASES = [
    # B, H, W, cin, cout, prec — shapes the default dispatch would NOT send to the pair kernel as well as ones it does
    (3, 40, 24, 48, 48, _lib.PREC_BF16),        # 27 spatial tiles (odd): the last pair's second CTA computes a masked tile
    (1, 16, 8, 64, 64, _lib.PREC_FP16),         # ONE spatial tile: a whole CTA of the only pair is masked
    (2, 32, 48, 96, 128, _lib.PREC_BF16),       # partial last K block
    (1, 16, 16, 64, 512, _lib.PREC_BF16),       # two N tiles of 256
    (2, 24, 40, 160, 64, _lib.PREC_BF16X2),     # two (W, A) plane pairs, filter-row W stages
    (1, 8, 8, 128, 256, _lib.PREC_BF16X3),      # three plane pairs
    (5, 64, 64, 128, 64, _lib.PREC_BF16),       # enough tiles for several rounds per cluster, MT = 2
]


@pytest.mark.parametrize("max_ctas", [0, 2, 6])
@pytest.mark.parametrize("case", CTA_PAIR_CASES, ids=[f"p{i}" for i in range(len(CTA_PAIR_CASES))])
def test_conv3x3_cta_pair_bits_equal_single_cta(case, max_ctas, built_lib):
    """The cta_group::2 kernel (each SM holds half of every W tile, M = 256 per UMMA) accumulates in the same order
    as the one-CTA slab kernel: same bits, for any cluster count and for odd tile counts."""
    B, H, W, cin, cout, prec = case
    x = _rand(B, cin, H, W, seed=51)
    w = _rand(cout, cin, 3, 3, seed=52, scale=(2.0 / (9 * cin)) ** 0.5)
    bias = _rand(cout, seed=53, scale=0.1)
    slope = torch.rand(cout, device=DEV) * 0.5
    x_hi, x_lo = to_planes(x, prec)
    wp = torch.ops.b200dn.pack_weight(w, prec, False)
    res = _rand(B, cout, H, W, seed=54)
    r_hi, r_lo = to_planes(res, prec)
    outs = []
    for impl, ctas in ((2, 0), (3, max_ctas)):
        o_hi, o_lo = _mk_out(B, H, W, cout, prec)
        torch.ops.b200dn.conv_igemm(x_hi, x_lo, wp, bias, slope, _lib.MODE_CONV3X3, prec, cin, cout, o_hi, o_lo, 0,
                                    r_hi, r_lo, 0, ctas, 0, impl)
        outs.append((o_hi, o_lo))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0])
    if outs[0][1] is not None:
        assert torch.equal(outs[0][1], outs[1][1])


DOWN_CASES = [(1, 16, 32, 16, 32), (2, 24, 40, 64, 128), (1, 64, 64, 128, 256), (1, 8, 8, 32, 64)]


@pytest.mark.parametrize("prec", PRECS, ids=PREC_IDS)
@pytest.mark.parametrize("case", DOWN_CASES, ids=[f"d{i}" for i in range(len(DOWN_CASES))])
def test_down2x2(case, prec, built_lib):
    B, H, W, cin, cout = case
    x = _rand(B, cin, H, W, seed=11)
    w = _rand(cout, cin, 2, 2, seed=12, scale=(2.0 / (4 * cin)) ** 0.5)
    bias = _rand(cout, seed=13, scale=0.1)
    slope = torch.rand(cout, device=DEV) * 0.5
    x_hi, x_lo = to_planes(x, prec, ctot=cin * 3)          # reads the skip slice of a 3C cat buffer
    _poison(x_hi, x_lo, cin)
    wp = torch.ops.b200dn.pack_weight(w, prec, False)
    ctot_out = cout * 5 // 2
    out_hi, out_lo = _mk_out(B, H // 2, W // 2, ctot_out, prec)
    torch.ops.b200dn.conv_igemm(x_hi, x_lo, wp, bias, slope, _lib.MODE_DOWN2X2, prec, cin, cout,
                                out_hi, out_lo, 0, None, None)
    torch.cuda.synchronize()
    b64 = bias.double().cpu().view(1, -1, 1, 1)
    pre, S = kernel_conv(lambda a, wt: F.conv2d(a, wt, stride=2), x, w, prec)
    ref, S = F.prelu(pre + b64, slope.double().cpu()), S + b64.abs()
    _check_slice(out_hi, out_lo, prec, 0, cout, ref, S, "down2x2")


# c <= 64: the four output phases are one N = 4c accumulator (folded); wider: one tile per phase
UP_CASES = [(1, 8, 16, 32), (2, 12, 20, 64), (1, 32, 32, 256), (1, 4, 4, 128), (3, 24, 40, 48), (1, 16, 16, 16)]


@pytest.mark.parametrize("prec", PRECS, ids=PREC_IDS)
@pytest.mark.parametrize("case", UP_CASES, ids=[f"u{i}" for i in range(len(UP_CASES))])
def test_up2x2_scatter(case, prec, built_lib):
    B, H, W, c = case                      # ConvTranspose2d(c, c, 2, stride=2)
    x = _rand(B, c, H, W, seed=21)
    w = _rand(c, c, 2, 2, seed=22, scale=(1.0 / c) ** 0.5)   # IOHW
    bias = _rand(c, seed=23, scale=0.1)
    slope = torch.rand(c, device=DEV) * 0.5
    x_hi, x_lo = to_planes(x, prec, ctot=c * 5 // 2)
    _poison(x_hi, x_lo, c)
    wp = torch.ops.b200dn.pack_weight(w, prec, True)
    cskip = c // 2
    ctot_out = cskip + c                   # [skip | upsampled]
    out_hi, out_lo = _mk_out(B, 2 * H, 2 * W, ctot_out, prec)
    torch.ops.b200dn.conv_igemm(x_hi, x_lo, wp, bias, slope, _lib.MODE_UP2X2, prec, c, c,
                                out_hi, out_lo, cskip, None, None)
    torch.cuda.synchronize()
    b64 = bias.double().cpu().view(1, -1, 1, 1)
    pre, S = kernel_conv(lambda a, wt: F.conv_transpose2d(a, wt, stride=2), x, w, prec)
    ref, S = F.prelu(pre + b64, slope.double().cpu()), S + b64.abs()
    _check_slice(out_hi, out_lo, prec, cskip, c, ref, S, "up2x2")


@pytest.mark.parametrize("impl", IMPLS, ids=IMPL_IDS)
@pytest.mark.parametrize("prec", PRECS, ids=PREC_IDS)
@pytest.mark.parametrize("B,bx,H,W,cin", [(1, 1, 16, 16, 16), (4, 2, 24, 40, 32), (2, 2, 8, 8, 128)])
def test_output_conv_nchw_residual(B, bx, H, W, cin, prec, impl, built_lib):
    x = _rand(B, cin, H, W, seed=31)
    w = _rand(3, cin, 3, 3, seed=32, scale=(2.0 / (9 * cin)) ** 0.5)
    bias = _rand(3, seed=33, scale=0.1)
    slope = torch.rand(3, device=DEV) * 0.5
    inputs = _rand(bx, 3, H, W, seed=34)
    x_hi, x_lo = to_planes(x, prec)
    wp = torch.ops.b200dn.pack_weight(w, prec, False)
    out = torch.full((B, 3, H, W), 9.0, device=DEV)
    torch.ops.b200dn.conv_out_nchw(x_hi, x_lo, wp, bias, slope, prec, cin, 3, inputs, out, bx, impl)
    torch.cuda.synchronize()
    ref = F.conv2d(effective_input(x, prec).double().cpu(), effective_weight(w, prec).double().cpu(),
                   bias.double().cpu(), padding=1)
    ref = F.prelu(ref, slope.double().cpu()) + inputs.double().cpu().repeat(B // bx, 1, 1, 1)
    err = (out.double().cpu() - ref).abs().max()
    assert float(err) < 5e-5, f"output conv (fp32 NCHW) max err {float(err):.3e}"


@pytest.mark.parametrize("prec", PRECS, ids=PREC_IDS)
@pytest.mark.parametrize("with_t", [False, True])
@pytest.mark.parametrize("B,bx,H,W,cout", [(1, 1, 8, 8, 16), (4, 2, 24, 40, 32), (2, 2, 16, 72, 128)])
def test_conv_in(B, bx, H, W, cout, with_t, prec, built_lib):
    cin = 4 if with_t else 3
    x = _rand(bx, 3, H, W, seed=41)
    w = _rand(cout, cin, 3, 3, seed=42, scale=(2.0 / (9 * cin)) ** 0.5)
    bias = _rand(cout, seed=43, scale=0.1)
    slope = torch.rand(cout, device=DEV) * 0.5
    t = torch.rand(B, device=DEV) if with_t else None
    ctot = cout + 16
    out_hi, out_lo = _mk_out(B, H, W, ctot, prec)
    torch.ops.b200dn.conv_in(x, t, w, bias, slope, prec, B, out_hi, out_lo)
    torch.cuda.synchronize()
    # single-plane modes run the tensor-core ingest: weights rounded to the 16-bit type like every other layer's, the fp32
    # image (and, unless the sampler's twin batch adds t * sum(w_t) in the epilogue, the t plane) gathered as hi + lo planes
    # of that type (bf16: 16 of the fp32 input's 24 bits); the two-plane (validation) modes keep the fp32 CUDA-core kernel
    def planes(v):
        if two_planes(prec):
            return v.double().cpu()
        hi = v.to(dt16(prec))
        return (hi.double() + (v - hi.float()).to(dt16(prec)).double()).cpu()
    xin = planes(x).repeat(B // bx, 1, 1, 1)
    if with_t:
        twin = B == 2 * bx
        tv = t.double().cpu() if twin else planes(t)
        xin = torch.cat([xin, tv.view(B, 1, 1, 1).expand(B, 1, H, W)], 1)
    we = w if two_planes(prec) else effective_weight(w, prec)
    ref = F.prelu(F.conv2d(xin, we.double().cpu(), bias.double().cpu(), padding=1), slope.double().cpu())
    S = F.conv2d(xin.abs(), we.double().cpu().abs(), bias.double().cpu().abs(), padding=1)
    _check_slice(out_hi, out_lo, prec, 0, cout, ref, S, "conv_in")


def test_igemm_argument_errors(built_lib):
    """Bad arguments come back as RuntimeError carrying the C-side message, as the reference's shape errors do."""
    prec = _lib.PREC_BF16
    x_hi = torch.zeros((1, 8, 8, 20), dtype=torch.int16, device=DEV)      # ctot not a multiple of 8
    out = torch.zeros((1, 8, 8, 16), dtype=torch.int16, device=DEV)
    w = torch.zeros((16, 16, 3, 3), device=DEV)
    wp = torch.ops.b200dn.pack_weight(w, prec, False)
    b = torch.zeros(16, device=DEV)
    with pytest.raises(RuntimeError, match="in_ctot"):
        torch.ops.b200dn.conv_igemm(x_hi, None, wp, b, b, _lib.MODE_CONV3X3, prec, 16, 16, out, None, 0, None, None)
    x_ok = torch.zeros((1, 8, 8, 16), dtype=torch.int16, device=DEV)
    with pytest.raises(RuntimeError, match="lo activation plane"):
        torch.ops.b200dn.conv_igemm(x_ok, None, wp, b, b, _lib.MODE_CONV3X3, _lib.PREC_BF16X2, 16, 16, out, None, 0,
                                    None, None)


# ----------------------------------------------------------------------------------------------- fused dense block
@pytest.mark.parametrize("prec", [_lib.PREC_FP16, _lib.PREC_BF16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("shape", [(1, 26, 18), (1, 8, 8), (2, 64, 64), (3, 40, 72), (1, 27, 19), (2, 136, 56)])
def test_fused_dense_block(shape, prec, built_lib):
    """b200dn_dense_block (one launch: input-stationary passes, partial sums in TMEM) against the fp64 block and
    against the four per-layer launches it replaces.  Shapes: exactly one 18 x 26 region, an image smaller than a
    region, several regions with partial ones at the right / bottom borders, odd batch."""
    import ctypes as C
    B, H, W = shape
    L = _lib.lib()
    dt = dt16(prec)
    st = torch.cuda.current_stream().cuda_stream
    x = (_rand(B, H, W, 48, seed=B + H, scale=0.5)).to(dt)                       # block input = channels [0, 32) of a 48-ch buffer
    ws = [_rand(co, ci, 3, 3, seed=10 + j, scale=(2.0 / (9 * ci)) ** 0.5) for j, (co, ci) in enumerate(((16, 32), (16, 48), (16, 64), (32, 80)))]
    bs = [_rand(co, seed=20 + j, scale=0.1) for j, co in enumerate((16, 16, 16, 32))]
    ss = [torch.full((co,), 0.25, device=DEV) + _rand(co, seed=30 + j, scale=0.05) for j, co in enumerate((16, 16, 16, 32))]
    wf = torch.empty(L.b200dn_dense_block_weight_bytes(32) // 2, dtype=torch.int16, device=DEV)
    _lib.check(L.b200dn_pack_dense_block_weights(ws[0].data_ptr(), ws[1].data_ptr(), ws[2].data_ptr(), ws[3].data_ptr(), 32, prec,
                                                 wf.data_ptr(), st))
    out = torch.full((B, H, W, 72), 7.0, device=DEV, dtype=dt)                   # writes the slice [40, 72)
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    a = _lib.DenseBlockArgs()
    a.prec, a.B, a.H, a.W, a.channels = prec, B, H, W, 32
    a.in_, a.in_ctot = x.data_ptr(), 48
    a.out, a.out_ctot, a.out_coff = out.data_ptr(), 72, 40
    a.wfused = wf.data_ptr()
    for j in range(4):
        a.bias[j], a.slope[j] = bs[j].data_ptr(), ss[j].data_ptr()
    a.sat_flag = flag.data_ptr()
    h = C.c_void_p()
    _lib.check(L.b200dn_dense_block_prepare(C.byref(a), C.byref(h)), "dense_block_prepare")
    _lib.check(L.b200dn_igemm_launch(h, st), "launch")
    _lib.check(L.b200dn_igemm_launch(h, st), "launch")          # relaunching a prepared block is idempotent
    torch.cuda.synchronize()
    staged = out.clone()
    # the same block with bias / slopes as host values in the launch parameters (constant bank): identical bits
    out.fill_(7.0)
    fp = C.POINTER(C.c_float)
    hb, hs = [t.cpu() for t in bs], [t.cpu() for t in ss]
    _lib.check(L.b200dn_dense_block_set_epilogue_constants(h, (fp * 4)(*[C.cast(t.data_ptr(), fp) for t in hb]),
                                                           (fp * 4)(*[C.cast(t.data_ptr(), fp) for t in hs])), "set constants")
    _lib.check(L.b200dn_igemm_launch(h, st), "launch")
    torch.cuda.synchronize()
    assert torch.equal(out, staged)
    assert L.b200dn_dense_block_set_epilogue_constants(h, None, None) == -1
    L.b200dn_igemm_release(h)
    ref = dense_block_ref(x[..., :32].permute(0, 3, 1, 2), ws, bs, ss, dt).cpu()
    got = out[..., 40:72].permute(0, 3, 1, 2).double().cpu()
    ulp = 2.0 ** -10 if prec == _lib.PREC_FP16 else 2.0 ** -7
    err = (got - ref).abs()
    # one storage ulp of the result + a rounding flip of an intermediate o_k (a 16-bit ulp times a weight) per stage
    tol = ref.abs() * ulp * 2 + 6 * ulp
    assert not (err > tol).any(), f"{int((err > tol).sum())} / {err.numel()} outside tolerance, max err {float(err.max()):.3e}"
    assert torch.all(out[..., :40].float() == 7.0), "wrote outside its channel slice"
    assert int(flag.item()) == 0
    with pytest.raises(RuntimeError, match="overlaps"):
        a.out, a.out_ctot, a.out_coff = x.data_ptr(), 48, 0
        _lib.check(L.b200dn_dense_block_prepare(C.byref(a), C.byref(h)), "dense_block_prepare")


@pytest.mark.parametrize("B,H,W,prec", [(2, 64, 64, "fp16"), (3, 40, 72, "bf16"), (1, 136, 56, "fp16"), (2, 256, 256, "fp16"),
                                        (3, 56, 40, "bf16")])
def test_fused_dense_block_cta_pairs_bit_equal(built_lib, monkeypatch, B, H, W, prec):
    """CTA pairs (the default; B200DN_DENSE_PAIR=0 turns them off): two regions per pair, cta_group::2 MMAs, half of
    every weight tile per SM.  Same tiles, same MMA order per accumulator row -> the network output is bit-identical to
    one CTA per region.  The level-0 blocks see 24, 24, 24, 300 and 27 regions of 18 x 26 pixels: the odd count runs
    the phantom region of the last pair."""
    import vub_image_denoising_b200 as b2
    torch.manual_seed(3)
    net = b2.RDUNet(base_filters=32).to(DEV).eval()
    net.precision = prec
    x = torch.rand(B, 3, H, W, device=DEV) * 2 - 1
    with torch.no_grad():
        monkeypatch.setenv("B200DN_DENSE_PAIR", "1")
        net.invalidate_plans()
        paired = [net(x).clone() for _ in range(3)]           # eager, graph capture, replay
        monkeypatch.setenv("B200DN_DENSE_PAIR", "0")
        net.invalidate_plans()
        single = net(x)
    for y in paired:
        assert torch.equal(y, single)


def test_fused_and_per_layer_networks_agree(built_lib, monkeypatch):
    """RDUNet_T(32) with the level-0 blocks fused vs launched layer by layer: same 16-bit rounding points, different
    fp32 summation order -> the two forwards agree to a few 16-bit ulps of the activations."""
    import vub_image_denoising_b200 as b2
    from vub_image_denoising_b200 import rdunet
    monkeypatch.setattr(rdunet, "_CHAIN_DENSE", 0)
    torch.manual_seed(5)
    net = b2.RDUNet(base_filters=32).to(DEV).eval()
    net.precision = "fp16"
    x = torch.rand(2, 3, 64, 80, device=DEV) * 2 - 1
    with torch.no_grad():
        fused = net(x)
        plan = net.plan(2, 64, 80)
        assert sum(isinstance(a, _lib.DenseBlockArgs) for a in plan.launches) == 4 and len(plan.launches) == 68 - 12
        monkeypatch.setattr(rdunet, "_FUSE_DENSE", False)
        net.invalidate_plans()
        layered = net(x)
        assert len(net.plan(2, 64, 80).launches) == 68
    assert float((fused - layered).abs().max()) < 5e-3


@pytest.mark.parametrize("F,B,H,W,prec", [
    (32, 1, 256, 256, "fp16"),      # batch 1: under-filled grids, N split to 64 at the deep levels (forced chains)
    (32, 3, 128, 136, "fp16"),      # ragged tiles, odd batch (odd CTA of the last pair idles)
    (32, 8, 256, 256, "bf16"),      # full grids, MT = 2 at levels 1-2
    (64, 2, 64, 72, "bf16"),        # every level chained (no fused 32-channel block)
    (16, 2, 128, 128, "fp16"),      # narrow levels fall back to the per-layer launches where the pair kernel does not apply
])
def test_chained_and_per_layer_dense_blocks_are_bit_equal(built_lib, monkeypatch, F, B, H, W, prec):
    """conv_0..conv_3 of a DenoisingBlock as ONE persistent launch with per-tile dependencies
    (conv3x3_chain_kernel, csrc/conv3x3_slab_sm100.cu) vs the four launches it replaces: same tiles, same MMA order -> identical bits,
    on the first call and on CUDA-graph replays (the dependency counters are monotonic across launches)."""
    import vub_image_denoising_b200 as b2
    from vub_image_denoising_b200 import rdunet
    torch.manual_seed(11)
    net = b2.RDUNet(base_filters=F).to(DEV).eval()
    net.precision = prec
    x = torch.rand(B, 3, H, W, device=DEV) * 2 - 1
    with torch.no_grad():
        monkeypatch.setattr(rdunet, "_CHAIN_DENSE", 2)       # also where the dispatch would launch layer by layer
        net.invalidate_plans()
        chained = [net(x).clone() for _ in range(4)]          # eager, graph capture, two replays
        plan = net.plan(B, H, W)
        n_chain = sum(isinstance(a, rdunet._Chain) for a in plan.launches)
        monkeypatch.setattr(rdunet, "_CHAIN_DENSE", 0)
        net.invalidate_plans()
        layered = net(x)
        assert not any(isinstance(a, rdunet._Chain) for a in net.plan(B, H, W).launches)
    if F >= 32:
        assert n_chain >= 6, n_chain
    for y in chained:
        assert torch.equal(y, layered)
