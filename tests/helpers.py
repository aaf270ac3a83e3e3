"""Shared helpers of the parity tests (layout conversion between the reference's NCHW fp32 world and the
kernels' NHWC 16-bit planes, digests, tolerances), exact-arithmetic DenoisingBlock data with their fp64 reference, and
the host-side enumeration of the network's launches and of the kernel configurations the planner picks for them."""
from __future__ import annotations

import ctypes as C
import hashlib
import math
from typing import NamedTuple

import torch
import torch.nn.functional as F

from vub_image_denoising_b200 import _lib

PIX_TOL = 2.0 / 255.0          # 1/255 in [0,1] space == 2/255 in the networks' [-1,1] space


def sd_digest(sd) -> str:
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(str(tuple(v.shape)).encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def dt16(prec: int):
    return torch.float16 if prec in _lib.FP16_PRECS else torch.bfloat16


def two_planes(prec: int) -> bool:
    return prec in _lib.TWO_PLANE_PRECS


def to_planes(x_nchw: torch.Tensor, prec: int, ctot: int | None = None, coff: int = 0):
    """fp32 NCHW -> (hi, lo|None) NHWC int16-storage planes with `ctot` channels (x placed at [coff, coff+C))."""
    B, Cn, H, W = x_nchw.shape
    ctot = ctot or Cn
    d = dt16(prec)
    nhwc = x_nchw.permute(0, 2, 3, 1).contiguous()
    hi = nhwc.to(d)
    full_hi = torch.zeros((B, H, W, ctot), dtype=d, device=x_nchw.device)
    full_hi[..., coff:coff + Cn] = hi
    lo_t = None
    if two_planes(prec):
        lo = (nhwc - hi.float()).to(d)
        lo_t = torch.zeros((B, H, W, ctot), dtype=d, device=x_nchw.device)
        lo_t[..., coff:coff + Cn] = lo
        lo_t = lo_t.view(torch.int16)
    return full_hi.view(torch.int16), lo_t


def from_planes(hi: torch.Tensor, lo, prec: int, coff: int, c: int) -> torch.Tensor:
    """(hi, lo) NHWC planes -> fp32 NCHW of channels [coff, coff+c)."""
    d = dt16(prec)
    v = hi.view(d)[..., coff:coff + c].float()
    if lo is not None:
        v = v + lo.view(d)[..., coff:coff + c].float()
    return v.permute(0, 3, 1, 2).contiguous()


def effective_input(x_nchw: torch.Tensor, prec: int) -> torch.Tensor:
    """The value the kernel actually sees for an fp32 activation under `prec` (hi [+ lo])."""
    d = dt16(prec)
    hi = x_nchw.to(d).float()
    if two_planes(prec):
        return hi + (x_nchw - hi).to(d).float()
    return hi


def effective_weight(w: torch.Tensor, prec: int) -> torch.Tensor:
    d = dt16(prec)
    hi = w.to(d).float()
    if prec == _lib.PREC_BF16X3:
        return hi + (w - hi).to(d).float()
    return hi


def kernel_conv(conv, x: torch.Tensor, w: torch.Tensor, prec: int):
    """(conv(a, w), conv(|a|, |w|)) in fp64 on the CPU over the products the tensor cores form under `prec`: the 16-bit
    input planes hi (+ lo) times the 16-bit weights; bf16x3 adds a_hi * w_lo and, by design, leaves out the lo x lo
    term (b200dn.h).  `conv(a, w)` is the fp64 convolution of the layer (padding / stride / transposed)."""
    d = dt16(prec)
    xh = x.to(d)
    a_hi = xh.double().cpu()
    a_lo = (x - xh.float()).to(d).double().cpu() if two_planes(prec) else torch.zeros_like(a_hi)
    w_hi = w.to(d).double().cpu()
    val, S = conv(a_hi + a_lo, w_hi), conv(a_hi.abs() + a_lo.abs(), w_hi.abs())
    if prec == _lib.PREC_BF16X3:
        w_lo = (w - w.to(d).float()).to(d).double().cpu()
        val, S = val + conv(a_hi, w_lo), S + conv(a_hi.abs(), w_lo.abs())
    return val, S


# ------------------------------------------------------------------------------------------ bound-based tolerance
# Every tensor-core layer computes v = prelu(sum_k a_k w_k + bias) (+ res) in fp32 (exact products, fp32 sums in some
# order) and rounds v to nearest in the storage format: two planes store hi = rn(v), lo = rn(v - hi), the NCHW output
# stores v itself.  With S = conv(|a|, |w|) + |bias| + |res| (PReLU slopes <= 1), the fp32 part is off by at most
# kappa * 2^-24 * S and the stored value by another half ulp of the last plane written.
KAPPA = 48.0
# Calibrated on a B200 (148 SMs, 1000 W power limit) over the 141 rows of tests/dispatch_configs.py: the largest
# (err - half ulp_store) / (2^-24 S) seen per kernel family (test_gpu_dispatch_parity.py prints it per row), one / two
# activation planes:
#   conv3x3 on CTA pairs       9.3 / 11.6     conv3x3 slab, one CTA   2.7 / 4.6    (NCHW fp32 output 2.8 / 3.2)
#   2x2 down, per-tap kernel   1.5 / 3.0      transposed 2x2          1.7 / 2.3
# KAPPA = 48 keeps 4x margin over the largest (11.6; CTA pairs sum the longest K, up to 9 * 640 terms per plane).

_MANT = {torch.bfloat16: (7, -126), torch.float16: (10, -14), torch.float32: (23, -126)}


def ulp(x: torch.Tensor, dt: torch.dtype) -> torch.Tensor:
    """ulp of `dt` at magnitude |x| (fp64), subnormal range included."""
    mant, emin = _MANT[dt]
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** (emin - mant - 1))))
    return torch.exp2(e.clamp_min(emin) - mant)


def bound_tol(ref: torch.Tensor, S: torch.Tensor, prec: int, nchw: bool = False, kappa: float = KAPPA) -> torch.Tensor:
    """|got - ref| allowed for a layer output: half an ulp of the last stored plane + kappa * 2^-24 * S.

    ref, S: fp64.  The ulp is taken at |ref| + kappa 2^-24 S, the largest |v| the fp32 part can produce.  Two planes:
    |lo| <= half an ulp of hi, so the lo plane's ulp is taken at that magnitude."""
    acc = kappa * 2.0 ** -24 * S
    m = ref.abs() + acc
    if nchw:
        u = ulp(m, torch.float32)
    else:
        d = dt16(prec)
        u = ulp(m, d)
        if two_planes(prec):
            u = ulp(u / 2, d)
    return u / 2 + acc


def tol_excess(err: torch.Tensor, ref: torch.Tensor, S: torch.Tensor, prec: int, nchw: bool = False) -> float:
    """Largest (err - half ulp_store(ref)) / (2^-24 S): the kappa this output needs (the calibration figure)."""
    half = bound_tol(ref, S, prec, nchw, kappa=0.0)
    return float(((err - half).clamp_min(0) / (2.0 ** -24 * S.clamp_min(1e-300))).max())


def store16(v: torch.Tensor, dt: torch.dtype) -> torch.Tensor:
    """v rounded to the 16-bit storage type as the kernels store it: round to nearest even, and fp16 saturates to
    +-65504 instead of overflowing to inf (cvt.rn.satfinite)."""
    return (v.clamp(-65504.0, 65504.0) if dt == torch.float16 else v).to(dt)


def dense_block_ref(x16, ws, bs, ss, dt, premise=None):
    """fp64 evaluation of a DenoisingBlock (UNet/RDUNet_model.py:95-115) of any width and depth with the kernels'
    rounding points: 16-bit weights and inputs, each growth output o_k rounded to the 16-bit storage type before it
    feeds the next conv (helpers.store16), fp64 accumulation.  ws / bs / ss: the growth convs then the last conv (+ x).

    premise: a list, to also check the exact-arithmetic premise of dyadic_block data on the way (dyadic_premise); it
    receives log2 of the largest S_k 2^G_k of every conv."""
    cat, n = x16.double(), len(ws)
    for j in range(n):
        w = ws[j].to(dt).double()
        pre = F.conv2d(cat, w, bs[j].double(), padding=1)
        res = x16.double() if j == n - 1 else None
        if premise is not None:
            premise.append(dyadic_premise(j, cat, w, bs[j], pre, res))
        v = F.prelu(pre, ss[j].double())
        if res is not None:
            return v + res
        cat = torch.cat([cat, store16(v, dt).double()], 1)


# --------------------------------------------------------------------------- exact-arithmetic DenoisingBlock data
# Operands on coarse dyadic grids make a block's arithmetic exact: every product and every partial sum of conv k is a
# multiple of 2^-G_k below 2^DYADIC_BITS * 2^-G_k, so fp32 holds it exactly and any summation order (tensor-core order,
# TMEM partial sums across the passes of the fused block, the fp32 epilogue) gives the same value.  The only roundings
# left are the 16-bit stores of o_0 .. o_{n-2} and of the output, each a round to nearest even of an exact value, the
# same on the GPU and in torch's .to(dtype).  So a kernel must reproduce store16(dense_block_ref(...)) bit for bit.
DYADIC_X, DYADIC_W, DYADIC_B, DYADIC_SLOPE = 3, 2, 5, 2      # fraction bits of x, weights, biases, PReLU slopes
DYADIC_BITS = 21                                             # 3 bits of headroom below fp32's 24-bit significand


def dyadic_grid(k: int) -> int:
    """G_k: fraction bits of every product and bias of conv k (o_j adds a slope and a weight per conv)."""
    return max(DYADIC_X + DYADIC_W, DYADIC_B) + k * (DYADIC_SLOPE + DYADIC_W)


def dyadic_block(C: int, B: int, H: int, W: int, seed: int, n: int = 4):
    """Data of an n-conv DenoisingBlock of C channels (growth C / 2), CPU fp32, all exact in bf16 and fp16:
    x = k/8 (|k| <= 8, NCHW); weights in {0, +-1/4}, nonzero with the probability that gives He variance 2 / (9 cin);
    biases k/32 (|k| <= 6) and PReLU slopes from {1/4, 1/2, 3/4}, both per channel, so that a channel mix-up shows.
    Pre-activations are about half negative, almost never zero, and keep an RMS near 1 through the block."""
    g = torch.Generator().manual_seed(seed)
    gr = C // 2
    shapes = [(gr, C + k * gr) for k in range(n - 1)] + [(C, C + (n - 1) * gr)]
    x = torch.randint(-8, 9, (B, C, H, W), generator=g, dtype=torch.int8).float() / 2 ** DYADIC_X
    ws, bs, ss = [], [], []
    for co, ci in shapes:
        p = min(1.0, (2.0 / (9 * ci)) / 0.25 ** 2)
        nz = torch.rand(co, ci, 3, 3, generator=g) < p
        sign = torch.randint(0, 2, (co, ci, 3, 3), generator=g) * 2 - 1
        ws.append((nz * sign).float() / 2 ** DYADIC_W)
        bs.append(torch.randint(-6, 7, (co,), generator=g).float() / 2 ** DYADIC_B)
        ss.append(torch.randint(1, 4, (co,), generator=g).float() / 2 ** DYADIC_SLOPE)
    return x, ws, bs, ss


def dyadic_premise(k, cat, w, b, pre, x=None) -> float:
    """Assert that conv k of a block (fp64 operands: input channels `cat`, 16-bit weights `w`, bias `b`, `pre` =
    conv(cat, w) + b; `x`: the residual of the last conv) is exact in fp32 in any summation order: every product and
    the bias lie on 2^-G_k, and S_k 2^G_k <= 2^DYADIC_BITS with S_k = conv(|cat|, |w|) + |b| (+ |x|), which bounds every
    partial sum.  A failure means the data generator is wrong, not a kernel.  Returns log2 max S_k 2^G_k.

    An output channel whose bias lies beyond the 16-bit range (the saturation tests drive one to 1e5) is left out: its
    value only has to saturate, not to be exact."""
    G = dyadic_grid(k)
    on_grid = lambda t, f: torch.equal(t * 2.0 ** f, torch.round(t * 2.0 ** f))     # noqa: E731
    assert on_grid(cat, G - DYADIC_W) and on_grid(w, DYADIC_W), f"conv {k}: operands off the 2^-{G} product grid"
    b = b.double().to(cat.device)
    S = F.conv2d(cat.abs(), w.abs(), b.abs(), padding=1)
    if x is not None:
        S = S + x.double().abs()
    keep = b.abs() <= 65504.0
    assert on_grid(b[keep], G) and on_grid(pre[:, keep], G), f"conv {k}: pre-activation off the 2^-{G} grid"
    bits = float(torch.log2(S[:, keep].max() * 2.0 ** G))
    assert bits <= DYADIC_BITS, f"conv {k}: a partial sum needs 2^{bits:.2f} > 2^{DYADIC_BITS} steps of 2^-{G}"
    return bits


# -------------------------------------------------------------------- a DenoisingBlock as per-layer launches (GPU)
NAN16 = 0x7FFF          # a NaN in both fp16 and bf16: the poison of channels a kernel must not read or write


def block_launches(x16, ws, bs, ss, prec):
    """The n convs of a DenoisingBlock as n b200dn_igemm launches in the network's per-layer layout
    (rdunet.ForwardPlan._dense): x16 (NHWC 16-bit, C channels, on the GPU) fills channels [0, C) of a 2.5 C-channel
    buffer `src`; conv_k (k < n - 1) writes [C + k g, C + (k + 1) g) of `src`, the last conv reads [0, C + (n - 1) g)
    and writes its C channels + x to [0, C) of a second 2.5 C-channel buffer `dst`.  Every other channel holds NaN.
    ws / bs / ss: fp32 on the GPU.  Returns dict(src, dst, args (an IgemmArgs array), keep, shapes)."""
    B, H, W, Cn = x16.shape
    g, ctot, n = Cn // 2, Cn * 5 // 2, len(ws)
    src = torch.full((B, H, W, ctot), NAN16, dtype=torch.int16, device=x16.device)
    src[..., :Cn] = x16.view(torch.int16)
    dst = torch.full_like(src, NAN16)
    shapes = [(g, Cn + k * g) for k in range(n - 1)] + [(Cn, Cn + (n - 1) * g)]
    keep = [torch.ops.b200dn.pack_weight(wj, prec, False) for wj in ws]
    args = (_lib.IgemmArgs * n)()
    for k, (co, ci) in enumerate(shapes):
        a = args[k]
        a.mode, a.prec, a.B, a.H, a.W, a.cin, a.cout = _lib.MODE_CONV3X3, prec, B, H, W, ci, co
        a.in_[0], a.in_ctot = src.data_ptr(), ctot
        a.wpacked, a.bias, a.slope = keep[k].data_ptr(), bs[k].data_ptr(), ss[k].data_ptr()
        a.out_kind = _lib.OUT_NHWC16
        if k < n - 1:
            a.out[0], a.out_ctot, a.out_coff = src.data_ptr(), ctot, ci
        else:
            a.out[0], a.out_ctot, a.out_coff = dst.data_ptr(), ctot, 0
            a.res[0], a.res_ctot = src.data_ptr(), ctot
    return dict(src=src, dst=dst, args=args, keep=keep, shapes=shapes)


def run_block_launches(blk, stream) -> None:
    L = _lib.lib()
    for k in range(len(blk["shapes"])):
        _lib.check(L.b200dn_igemm(C.byref(blk["args"][k]), stream), "igemm")


def frac_within(a: torch.Tensor, b: torch.Tensor) -> float:
    return float(((a - b).abs() <= PIX_TOL).double().mean())


def psnr_db(ref: torch.Tensor, x: torch.Tensor, data_range=2.0) -> float:
    mse = float(((ref.double() - x.double()) ** 2).mean())
    return 10 * math.log10(data_range ** 2 / mse)


def check_bar(got, ref, clean=None, what=""):
    """North-star bar: >= 99.9 % of output values within 1/255 (and PSNR within 0.02 dB when `clean` is given).
    The golden micro-cases have ~1.5k values, where 0.1 % is 1.5 values: there the bar reads 'at most 2 values
    outside'; the BASELINE-size tests (196k values per patch) apply the percentage as written."""
    frac = frac_within(got, ref)
    mx = float((got - ref).abs().max())
    n_bad = int(((got - ref).abs() > PIX_TOL).sum())
    ok = frac >= 0.999 or (got.numel() < 4000 and n_bad <= 2)
    assert ok, f"{what}: only {frac * 100:.3f}% of pixels within 1/255 ({n_bad} outside, max err {mx:.3e})"
    if clean is not None:
        d = abs(psnr_db(clean, got) - psnr_db(clean, ref))
        assert d <= 0.02, f"{what}: PSNR differs by {d:.4f} dB"
    return frac, mx


# ------------------------------------------------------------------------ launch planning (host only, no GPU touched)
SMS = 148
DUMMY = 0x1000   # plan-only calls check pointers for NULL, nothing more
PRECS = (_lib.PREC_BF16, _lib.PREC_FP16, _lib.PREC_BF16X2, _lib.PREC_BF16X3, _lib.PREC_FP16X2)
PREC_IDS = {_lib.PREC_BF16: "bf16", _lib.PREC_FP16: "fp16", _lib.PREC_BF16X2: "bf16x2", _lib.PREC_BF16X3: "bf16x3",
            _lib.PREC_FP16X2: "fp16x2"}


def plan(mode, B, H, W, cin, cout, prec=_lib.PREC_BF16, in_ctot=None, out_ctot=None, coff=0, nchw=False, impl=0,
         block_n=0, m_tiles=0, max_ctas=0, sms=SMS):
    a = _lib.IgemmArgs()
    a.mode, a.prec, a.B, a.H, a.W, a.cin, a.cout = mode, prec, B, H, W, cin, cout
    a.in_[0] = DUMMY
    a.in_[1] = DUMMY if prec in _lib.TWO_PLANE_PRECS else None
    a.in_ctot = in_ctot or ((cin + 7) // 8 * 8)
    a.wpacked, a.bias, a.slope = DUMMY, DUMMY, DUMMY
    if nchw:
        a.out_kind = _lib.OUT_NCHW32
        a.out_nchw, a.res_nchw, a.res_bmod = DUMMY, DUMMY, B
    else:
        a.out_kind = _lib.OUT_NHWC16
        a.out[0] = DUMMY
        a.out[1] = DUMMY if prec in _lib.TWO_PLANE_PRECS else None
        a.out_ctot, a.out_coff = out_ctot or (coff + cout + 7) // 8 * 8, coff
    a.impl, a.block_n, a.m_tiles, a.max_ctas = impl, block_n, m_tiles, max_ctas
    info = _lib.IgemmPlanInfo()
    rc = _lib.lib().b200dn_igemm_plan(C.byref(a), sms, C.byref(info))
    _lib.check(rc, "igemm_plan")
    return info


class Layer(NamedTuple):
    """One tensor-core launch of the network (rdunet.ForwardPlan), in the buffers the network gives it."""
    mode: int           # MODE_CONV3X3 / MODE_DOWN2X2 / MODE_UP2X2
    B: int
    H: int              # input height / width
    W: int
    cin: int            # reads channels [0, cin) of an in_ctot-channel NHWC buffer
    cout: int
    in_ctot: int
    out_ctot: int       # writes channels [coff, coff + cout) of an out_ctot-channel NHWC buffer (0: NCHW output)
    coff: int
    nchw: bool          # fp32 NCHW output + fp32 NCHW residual (the output block's last conv)
    residual: bool      # + channels [0, cout) of the input buffer (conv_3 of a DenoisingBlock), or the NCHW residual
    same_buffer: bool   # the output slice lies in the input buffer itself (conv_0..2 of a DenoisingBlock)

    @property
    def macs(self) -> int:
        taps = 9 if self.mode == _lib.MODE_CONV3X3 else 4
        pix = self.B * self.H * self.W // (4 if self.mode == _lib.MODE_DOWN2X2 else 1)
        return pix * taps * self.cin * self.cout


def network_layers(F, B, S=256):
    """The 68 tensor-core launches of an RDUNet of width F on B images of S x S (rdunet.ForwardPlan, per-layer)."""
    L = []
    ch = [F << l for l in range(4)]
    hs = [S >> l for l in range(4)]

    def dense(l, dst_ctot):
        Cc, g = ch[l], ch[l] // 2
        for k in range(3):
            L.append(Layer(0, B, hs[l], hs[l], Cc + k * g, g, Cc * 5 // 2, Cc * 5 // 2, Cc + k * g, False, False, True))
        L.append(Layer(0, B, hs[l], hs[l], Cc + 3 * g, Cc, Cc * 5 // 2, dst_ctot, 0, False, True, False))

    L.append(Layer(0, B, S, S, F, F, F, F * 5 // 2, 0, False, False, False))
    for l in range(4):
        dense(l, ch[l] * 5 // 2)
        dense(l, ch[l] * 3 if l < 3 else ch[l] * 5 // 2)
        if l < 3:
            L.append(Layer(1, B, hs[l], hs[l], ch[l], 2 * ch[l], 3 * ch[l], ch[l + 1] * 5 // 2, 0, False, False, False))
    for l in (2, 1, 0):
        L.append(Layer(2, B, hs[l + 1], hs[l + 1], ch[l + 1], ch[l + 1], ch[l + 1] * 5 // 2, 3 * ch[l], ch[l], False,
                       False, False))
        L.append(Layer(0, B, hs[l], hs[l], 3 * ch[l], ch[l], 3 * ch[l], ch[l] * 5 // 2, 0, False, False, False))
        dense(l, ch[l] * 5 // 2)
        dense(l, ch[l] * 5 // 2)
    L.append(Layer(0, B, S, S, F, F, F * 5 // 2, F, 0, False, False, False))
    L.append(Layer(0, B, S, S, F, 3, F, 0, 0, True, True, False))
    return L


def plan_layer(layer: Layer, prec: int, sms: int = SMS):
    return plan(layer.mode, layer.B, layer.H, layer.W, layer.cin, layer.cout, prec=prec, in_ctot=layer.in_ctot,
                out_ctot=layer.out_ctot, coff=layer.coff, nchw=layer.nchw, sms=sms)


class Signature(NamedTuple):
    """The kernel configuration one launch runs (what b200dn_igemm_plan decides, plus what the layer adds)."""
    mode: int           # 0 conv3x3, 1 down 2x2, 2 transposed 2x2
    kernel: int         # 0 per-tap kernel, 1 slab kernel on one CTA, 2 slab kernel on a CTA pair
    mt: int             # accumulator sub-tiles per W tile (2: M = 256 per CTA, two epilogue warp groups)
    wres: int           # 1: the whole weight set resident in shared memory, 0: streamed through a W ring
    w_taps: int         # taps per W ring stage (3: a filter row)
    multi_n: bool       # more than one N tile per output (per phase group of a transposed conv)
    staged: int         # 1: epilogue transposed through shared memory (128-byte pixel rows), 0: direct stores
    up_fold: bool       # transposed conv with its four phases in one N = 4 * cout accumulator
    nchw: bool          # fp32 NCHW output
    residual: bool      # residual added in the epilogue
    planes: int         # activation / output planes (2: hi + lo)
    w_planes: int       # weight planes (2: bf16x3 hi + lo)
    fp16: bool          # fp16 storage (saturating conversion, sat_flag watch) rather than bf16


def signature(info, layer: Layer, prec: int) -> Signature:
    groups = 4 if layer.mode == _lib.MODE_UP2X2 else 1
    up_fold = layer.mode == _lib.MODE_UP2X2 and info.block_n == 4 * layer.cout
    n_per_group = 1 if up_fold else info.num_n_tiles // groups
    return Signature(layer.mode, info.kernel, info.mt, info.wres, info.w_taps, n_per_group > 1, info.epi_staged,
                     up_fold, layer.nchw, layer.residual, 2 if two_planes(prec) else 1,
                     2 if prec == _lib.PREC_BF16X3 else 1, prec in _lib.FP16_PRECS)


# the production grid the configuration table covers: network widths x the batches of
# test_launch_plans.test_every_network_layer_fits x every precision
GRID_WIDTHS = (16, 32, 48, 64, 128)
GRID_BATCHES = (1, 2, 3, 4, 5, 32, 64)


def dispatch_rows(sms: int = SMS):
    """Rows of tests/dispatch_configs.py: (*signature, F, B, prec, launch index into network_layers(F, B)), one per
    signature the grid produces.  The representative is the layer with the fewest MACs, ties to the first in
    enumeration order (width, batch, precision, launch order)."""
    best = {}
    for F in GRID_WIDTHS:
        for B in GRID_BATCHES:
            for prec in PRECS:
                for idx, layer in enumerate(network_layers(F, B)):
                    sig = signature(plan_layer(layer, prec, sms), layer, prec)
                    if sig not in best or layer.macs < best[sig][1]:
                        best[sig] = ((F, B, prec, idx), layer.macs)
    return sorted(tuple(int(v) for v in sig) + rep for sig, (rep, _) in best.items())


def row_signature(row) -> Signature:
    return Signature(*row[:len(Signature._fields)])


def row_layer(row) -> tuple[Layer, int]:
    F, B, prec, idx = row[len(Signature._fields):]
    return network_layers(F, B)[idx], prec


def render_dispatch_configs(rows) -> str:
    head = ('"""Every kernel configuration the launch planner picks for the network: one row per distinct helpers.Signature\n'
            'over RDUNet widths %s x batches %s x the five precisions (148 SMs), with the cheapest\n'
            'layer that runs it.  tests/test_launch_plans.py checks this table against the planner;\n'
            'tests/test_gpu_dispatch_parity.py runs every row against an fp64 reference.  Regenerate with\n'
            '`python tests/dispatch_configs.py --write` after a dispatch change."""\n'
            % (GRID_WIDTHS, GRID_BATCHES))
    fields = ", ".join(Signature._fields)
    lines = [head, f"# ({fields}, F, B, prec, launch index into helpers.network_layers(F, B))", "ROWS = ["]
    for r in rows:
        layer, prec = row_layer(r)
        lines.append(f"    {r!r},   # {PREC_IDS[prec]} {'conv3x3 down2x2 up2x2'.split()[layer.mode]} "
                     f"B={layer.B} {layer.H}x{layer.W} {layer.cin}->{layer.cout}")
    lines.append("]")
    lines.append("")
    lines.append("if __name__ == \"__main__\":")
    lines.append("    import sys")
    lines.append("    from pathlib import Path")
    lines.append("    sys.path[:0] = [str(Path(__file__).resolve().parent), str(Path(__file__).resolve().parent.parent)]")
    lines.append("    import helpers")
    lines.append("    text = helpers.render_dispatch_configs(helpers.dispatch_rows())")
    lines.append("    if \"--write\" in sys.argv:")
    lines.append("        Path(__file__).write_text(text)")
    lines.append("    else:")
    lines.append("        print(text, end=\"\")")
    return "\n".join(lines) + "\n"
