"""Shared helpers of the parity tests (layout conversion between the reference's NCHW fp32 world and the
kernels' NHWC 16-bit planes, digests, tolerances) and the host-side enumeration of the network's launches and of the
kernel configurations the planner picks for them."""
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


def dense_block_ref(x16, ws, bs, ss, dt):
    """fp64 evaluation of a DenoisingBlock (UNet/RDUNet_model.py:95-115) of any width and depth with the kernels'
    rounding points: 16-bit weights and inputs, each growth output o_k rounded to the 16-bit storage type before it
    feeds the next conv, fp64 accumulation.  ws / bs / ss: the growth convs then the last conv (+ x)."""
    cat = x16.double()
    for j in range(len(ws) - 1):
        o = F.prelu(F.conv2d(cat, ws[j].to(dt).double(), bs[j].double(), padding=1), ss[j].double())
        cat = torch.cat([cat, o.to(dt).double()], 1)
    return F.prelu(F.conv2d(cat, ws[-1].to(dt).double(), bs[-1].double(), padding=1), ss[-1].double()) + x16.double()


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
