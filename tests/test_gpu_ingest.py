"""The ingest conv b200dn_conv_in (InputBlock.conv_1 + PReLU fused with the fp32 NCHW -> NHWC 16-bit ingest and the
RDUNet_T timestep plane, csrc/conv_in.cu) in every path it dispatches, called through the C ABI:
- conv_in_tc_kernel (tcgen05) in the single-plane modes bf16 / fp16, RGB or grayscale, with or without a t plane,
  and its twin mode (B = 2 Bx images with one scalar t each: the image is multiplied once, t * S added per border class);
- conv_in_kernel (fp32 CUDA cores) in the two-plane modes and, for cout > 256, in the single-plane modes.

Every output buffer holds the 16-bit NaN poison and one image more than the call writes; every run checks that only
channels [0, cout) of images [0, B) change and that the image and the timesteps are left alone.

- test_ingest_exact: helpers.dyadic_ingest data, on which every path's arithmetic is exact, bit for bit against the
  stored fp64 value (helpers.INGEST_ROWS names what each row reaches).
- test_ingest_random: the network's and the sampler's calls on real-valued data within helpers.bound_tol.
- the fp16 saturation watch, argument errors, and RDUNet_T with timestep planes that vary in space.
"""
import ctypes as C
import time

import pytest
import torch

from helpers import (INGEST_ROWS, NAN16, PREC_IDS, PRECS, bound_tol, check_bar, dt16, ingest_planes, ingest_premise,
                     ingest_ref, ingest_row_data, ingest_row_id, t_view, tol_excess, two_planes)
from vub_image_denoising_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _call(x, cimg, t, strides, B, cout, w, b, s, prec, out0, out1, out_ctot, flag=None):
    """b200dn_conv_in on GPU tensors; returns its error code."""
    Bx, _, H, W = x.shape
    ptr = lambda u: None if u is None else u.data_ptr()      # noqa: E731
    return _lib.lib().b200dn_conv_in(ptr(x), Bx, cimg, ptr(t), strides[0], strides[1], strides[2], B, H, W, cout,
                                     ptr(w), ptr(b), ptr(s), prec, ptr(out0), ptr(out1), out_ctot, ptr(flag),
                                     torch.cuda.current_stream().cuda_stream)


def _run(x, t, strides, B, cout, out_ctot, w, b, s, prec, flag=None):
    """One call into poisoned [B + 1, H, W, out_ctot] planes.  Checks that nothing outside channels [0, cout) of
    images [0, B) is written and that x and t are unchanged; returns the (hi, lo | None) planes."""
    Bx, cimg, H, W = x.shape
    hi = torch.full((B + 1, H, W, out_ctot), NAN16, dtype=torch.int16, device=DEV)
    lo = hi.clone() if two_planes(prec) else None
    x0, t0 = x.clone(), (t.clone() if t is not None else None)
    _lib.check(_call(x, cimg, t, strides, B, cout, w, b, s, prec, hi, lo, out_ctot, flag), "conv_in")
    torch.cuda.synchronize()
    for p in (hi, lo):
        if p is not None:
            assert bool((p[B] == NAN16).all()), "wrote past image B - 1"
            assert bool((p[..., cout:] == NAN16).all()), "wrote outside channels [0, cout)"
    assert torch.equal(x, x0) and (t is None or torch.equal(t, t0)), "changed its inputs"
    return hi, lo


def _nchw(p, idx, cout, dt):
    return p[idx][..., :cout].view(dt).permute(0, 3, 1, 2).cpu()


def _ids(rows):
    return [ingest_row_id(r) for r in rows]


# --------------------------------------------------------------------------------------------- exact, bit for bit
@pytest.mark.parametrize("row", INGEST_ROWS, ids=_ids(INGEST_ROWS))
def test_ingest_exact(row, monkeypatch, built_lib):
    """Every precision on exact data: the hi plane is store16 of the fp64 value, the lo plane of the two-plane modes
    store16(v - hi).  The reference covers images 0, Bx - 1, Bx and B - 1: the first tile, the tail tiles of the
    persistent loop and both outputs of a twin input.  A twin row also runs with B200DN_CONV_IN_TWIN=0 (the general
    path, which gathers t with the image): the same bytes."""
    t0 = time.time()
    cimg, tk, Bx, B, H, W, cout, out_ctot = row
    x, t_src, strides, w, b, s = ingest_row_data(row, seed=sum(row[2:]))
    idx = sorted({0, Bx - 1, min(Bx, B - 1), B - 1})
    t = t_view(t_src, strides, B, H, W)[idx] if t_src is not None else None
    v, S = ingest_ref(x[[i % Bx for i in idx]], t, w, b, s)
    bits = ingest_premise(x, t_src, w, b, v, S)
    twin = tk == "scalar" and B == 2 * Bx and H >= 2 and W >= 2
    xd, wd, bd, sd = (u.to(DEV) for u in (x, w, b, s))
    td = t_src.to(DEV) if t_src is not None else None
    for prec in PRECS:
        d, two, fp16 = dt16(prec), two_planes(prec), prec in _lib.FP16_PRECS
        flag = torch.zeros(1, dtype=torch.int32, device=DEV)
        hi, lo = _run(xd, td, strides, B, cout, out_ctot, wd, bd, sd, prec, flag)
        want_hi, want_lo = ingest_planes(v, d, two)
        for what, p, want in (("hi", hi, want_hi), ("lo", lo, want_lo)):
            if p is None:
                continue
            diff = _nchw(p, idx, cout, d).view(torch.int16) != want.view(torch.int16)
            assert not diff.any(), f"{PREC_IDS[prec]} {what}: {int(diff.sum())} / {diff.numel()} values differ"
        assert int(flag.item()) == 0, f"{PREC_IDS[prec]}: sat_flag raised without saturation"
        if twin and not two:
            monkeypatch.setenv("B200DN_CONV_IN_TWIN", "0")
            general, _ = _run(xd, td, strides, B, cout, out_ctot, wd, bd, sd, prec, flag)
            monkeypatch.delenv("B200DN_CONV_IN_TWIN")
            assert torch.equal(general, hi), f"{PREC_IDS[prec]}: twin and general path differ"
    print(f"\n[ingest exact] {ingest_row_id(row)}: partial sums need 2^{bits:.2f} steps, {time.time() - t0:.2f} s")


# ------------------------------------------------------------------------------------------ random data, bounded
def _random_cases():
    """(Bx, B, H, W, cout, out_ctot, with_t): RDUNet's calls (cout = out_ctot = the padded width ForwardPlan gives the
    ingest), the sampler's twin calls, and the three shapes of the layer test this file replaced."""
    cases = [(B, B, 64, 64, F, F, False) for F in (16, 32, 48, 64, 128) for B in (1, 2, 64)]
    cases.append((64, 64, 256, 256, 128, 128, False))                      # the bench's call
    cases += [(bx, 2 * bx, 64, 64, F, F, True) for F in (16, 32, 48, 64, 128) for bx in (1, 16)]
    cases += [(bx, B, H, W, c, c + 16, wt) for (B, bx, H, W, c) in ((1, 1, 8, 8, 16), (4, 2, 24, 40, 32),
                                                                     (2, 2, 16, 72, 128)) for wt in (False, True)]
    return cases


RANDOM_CASES = _random_cases()


def _random_id(c):
    bx, B, H, W, cout, ctot, wt = c
    return f"{bx}to{B}-{H}x{W}-c{cout}" + (f"of{ctot}" if ctot != cout else "") + ("-t" if wt else "")


def _hilo(v, dt):
    hi = v.to(dt)
    return hi.double() + (v - hi.float()).to(dt).double()


@pytest.mark.parametrize("case", RANDOM_CASES, ids=[_random_id(c) for c in RANDOM_CASES])
def test_ingest_random(case, built_lib):
    """u8-normalised images plus N(0, 1) noise, real schedule timesteps k / 20 (the sampler's pair k / 20,
    (k - 1) / 20 in twin mode), N(0, He) weights.  The reference takes the operands as each path reads them: on tensor
    cores the image as hi + lo 16-bit planes and 16-bit weights, t exact in twin mode (t * S in fp32) and as hi + lo
    otherwise; on CUDA cores everything in fp32.  Each case prints the kappa it needs and must reject replicate
    padding and, with t, the inner border class's t term at the border."""
    Bx, B, H, W, cout, out_ctot, with_t = case
    g = torch.Generator().manual_seed(sum(case))
    cin = 4 if with_t else 3
    u8 = torch.randint(0, 256, (Bx, 3, H, W), generator=g).float()
    x = (u8 / 255 - 0.5) / 0.5 + torch.randn(Bx, 3, H, W, generator=g)
    w = torch.randn(cout, cin, 3, 3, generator=g) * (2.0 / (9 * cin)) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    s = torch.rand(cout, generator=g) * 0.5
    twin = with_t and B == 2 * Bx
    t = None
    if with_t:
        k = torch.randint(2, 21, (Bx if twin else B,), generator=g)
        t = (torch.cat([k, k - 1]) if twin else k).double().div(20).float()
    xd, wd, bd, sd = (u.to(DEV) for u in (x, w, b, s))
    td = t.to(DEV) if t is not None else None
    idx = sorted({0, Bx - 1, min(Bx, B - 1), B - 1})
    refs = {}
    for prec in PRECS:
        d = dt16(prec)
        tc = not two_planes(prec) and cout <= 256
        key = d if tc else "fp32"
        if key not in refs:
            xe = _hilo(x, d) if tc else x.double()
            we = w.to(d).double() if tc else w.double()
            te = None
            if t is not None:
                te = (t.double() if twin or not tc else _hilo(t, d)).view(B, 1, 1, 1).expand(B, 1, H, W)[idx]
            xs = xe[[i % Bx for i in idx]]
            refs[key] = (ingest_ref(xs, te, we, b, s), ingest_ref(xs, te, we, b, s, pad="replicate")[0],
                         ingest_ref(xs, te, we, b, s, t_pad="replicate")[0] if t is not None else None)
        (ref, S), ref_rep, ref_inner = refs[key]
        hi, lo = _run(xd, td, (1, 0, 0), B, cout, out_ctot, wd, bd, sd, prec)
        got = _nchw(hi, idx, cout, d).double()
        if lo is not None:
            got = got + _nchw(lo, idx, cout, d).double()
        err = (got - ref).abs()
        path = ("tensor cores, twin" if twin else "tensor cores") if tc else "CUDA cores"
        print(f"\n[ingest] {_random_id(case)} {PREC_IDS[prec]} ({path}): max err {float(err.max()):.3e}, "
              f"kappa needed {tol_excess(err, ref, S, prec):.3f}")
        outside = lambda r: ~((got - r).abs() <= bound_tol(r, S, prec))     # noqa: E731
        bad = outside(ref)
        assert not bad.any(), f"{PREC_IDS[prec]}: {int(bad.sum())} / {bad.numel()} outside the bound"
        assert outside(ref_rep).any(), "the bound accepts replicate padding"
        if ref_inner is not None:
            assert outside(ref_inner).any(), "the bound accepts the inner class's t term at the border"


# ------------------------------------------------------------------------------------------- fp16 saturation watch
SAT_ROWS = [
    (3, "scalar", 2, 6, 40, 24, 64, 80),       # fp16: the general tensor-core path
    (3, "scalar", 1, 2, 3, 9, 24, 32),         # fp16: the twin path
    (1, "scalar", 2, 4, 64, 64, 16, 16),       # fp16: the grayscale twin path
    (3, "scalar", 1, 1, 32, 32, 264, 264),     # fp16: the single-plane CUDA-core path
]


@pytest.mark.parametrize("row", SAT_ROWS, ids=_ids(SAT_ROWS))
def test_ingest_saturation_watch(row, built_lib):
    """One channel's bias at 1e5: in fp16 and fp16x2 (two-plane CUDA-core path) the flag is raised and that channel's
    hi plane holds 65504 everywhere; in the bf16 modes the flag stays 0.  Every other channel keeps its bytes."""
    cimg, tk, Bx, B, H, W, cout, out_ctot = row
    x, t_src, strides, w, b, s = ingest_row_data(row, seed=sum(row[2:]))
    xd, wd, bd, sd = (u.to(DEV) for u in (x, w, b, s))
    td = t_src.to(DEV) if t_src is not None else None
    hot = cout - 3
    hb = bd.clone()
    hb[hot] = 1e5
    keep = torch.ones(out_ctot, dtype=torch.bool, device=DEV)
    keep[hot] = False
    for prec in PRECS:
        base = _run(xd, td, strides, B, cout, out_ctot, wd, bd, sd, prec)
        flag = torch.zeros(1, dtype=torch.int32, device=DEV)
        got = _run(xd, td, strides, B, cout, out_ctot, wd, hb, sd, prec, flag)
        for p, p0 in zip(got, base):
            if p is not None:
                assert torch.equal(p[..., keep], p0[..., keep]), f"{PREC_IDS[prec]}: the hot bias moved other channels"
        if prec in _lib.FP16_PRECS:
            assert int(flag.item()) == 1, f"{PREC_IDS[prec]}: saturated without raising sat_flag"
            ch = got[0][:B, ..., hot].view(torch.float16).float()
            assert bool((ch == 65504.0).all()), f"{PREC_IDS[prec]}: saturated channel stores {ch.unique()[:8].tolist()}"
        else:
            assert int(flag.item()) == 0, f"{PREC_IDS[prec]}: sat_flag raised in a bf16 mode"


# ------------------------------------------------------------------------------------------------ argument errors
def test_ingest_argument_errors(built_lib):
    """Each bad argument returns B200DN_E_ARG and launches nothing (the poisoned output keeps its bytes)."""
    B, H, W, cout = 2, 16, 16, 16
    x = torch.zeros(B, 3, H, W, device=DEV)
    w = torch.zeros(cout, 3, 3, 3, device=DEV)
    b = torch.zeros(cout, device=DEV)
    hi = torch.full((B, H, W, cout), NAN16, dtype=torch.int16, device=DEV)
    lo = hi.clone()
    ok = dict(x=x, cimg=3, t=None, strides=(0, 0, 0), B=B, cout=cout, w=w, b=b, s=b, prec=_lib.PREC_BF16X2,
              out0=hi, out1=lo, out_ctot=cout)
    assert _call(**ok) == 0
    torch.cuda.synchronize()
    hi.fill_(NAN16)
    lo.fill_(NAN16)
    bad = [dict(cout=12), dict(out_ctot=8), dict(cimg=2), dict(prec=5), dict(out1=None), dict(B=0), dict(B=-1),
           dict(x=x[:0]), dict(x=x[:, :, :0]), dict(x=x[..., :0])]       # Bx = 0, H = 0, W = 0
    for kw in bad:
        rc = _call(**{**ok, **kw})
        assert rc == _lib.E_ARG, f"{list(kw)} {kw.get('x', x).shape}: returned {rc}"
    torch.cuda.synchronize()
    assert bool((hi == NAN16).all()) and bool((lo == NAN16).all()), "a refused call wrote its output"


# ------------------------------------------------------------------------------- network: timestep planes in space
@pytest.mark.parametrize("precision,max_abs", [("bf16", None), ("fp16", None), ("bf16x2", None), ("bf16x3", 1e-4)])
@pytest.mark.parametrize("H,W", [(16, 24), (32, 32)])
def test_rdunet_t_timestep_planes(H, W, precision, max_abs, built_lib):
    """RDUNet_T(16) with timesteps of shape [B, 1, H, W], [1, 1, H, W] and [1, 1, 1, W] (the reference's
    t.expand(B, 1, H, W) allows them; the forward runs eagerly and passes the view's strides to the ingest) against
    the fp64 oracle on the CPU."""
    import vub_image_denoising_b200 as b2
    from oracle import rdunet_oracle as orc
    torch.manual_seed(11)
    net = b2.RDUNet_T(base_filters=16)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.to(DEV).eval()
    net.precision = precision
    B = 2
    g = torch.Generator().manual_seed(H * W)
    x = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    with torch.no_grad():
        for shape in ((B, 1, H, W), (1, 1, H, W), (1, 1, 1, W)):
            t = torch.rand(*shape, generator=g)
            got = net(x.to(DEV), t.to(DEV)).cpu()
            ref = orc.rdunet_forward(sd, x.double(), t.double()).float()
            check_bar(got, ref, what=f"RDUNet_T(16) {precision} t {list(shape)}")
            if max_abs is not None:
                assert float((got - ref).abs().max()) <= max_abs, f"t {list(shape)}"
