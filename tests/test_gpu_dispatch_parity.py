"""Every kernel configuration the planner dispatches for the network (tests/dispatch_configs.py), run once on the layer
that represents it, in the network's own buffer layout, against an fp64 reference of the same operation.

Each row's launch goes through the C ABI (b200dn_igemm) the way rdunet.ForwardPlan issues it:
- the input is the channel prefix [0, cin) of an in_ctot-channel buffer; conv_0..2 of a DenoisingBlock write their
  slice into that same buffer, conv_3 adds channels [0, cout) of it as the residual (res_ctot = in_ctot);
- every channel the launch must not read, and every byte it must not write, holds a 16-bit NaN (both planes): the
  network's buffers are torch.empty, so a stray read would be as wrong as it can be;
- the reference covers every pixel and channel of the first and the last image (the last one holds the tail tiles of
  the persistent loop and the odd CTA of the last pair); every other byte of the output buffer must be unchanged.

The tolerance is helpers.bound_tol: half an ulp of the stored plane + KAPPA * 2^-24 * S, S = conv(|a|, |w|) + |bias| +
|res|.  Each row also checks that it rejects two near-miss references (a K16 slice of one tap dropped; replicate
instead of zero padding, or for the unpadded 2x2 convs the taps mirrored along x), so the bound stays tight enough
to see an error of that size.

The chain kernel (conv_0..conv_3 of a DenoisingBlock as one persistent launch) is checked at the layer level below.
"""
import ctypes as C
import time

import pytest
import torch
import torch.nn.functional as F

import dispatch_configs
from helpers import (NAN16, PREC_IDS, block_launches, bound_tol, dense_block_ref, dt16, dyadic_block, plan, plan_layer,
                     row_layer, row_signature, run_block_launches, signature, store16, tol_excess, two_planes)
from vub_image_denoising_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda"
ROWS = dispatch_configs.ROWS


def _row_id(row):
    s = row_signature(row)
    layer, prec = row_layer(row)
    parts = ["conv3x3 down up".split()[s.mode], ["tap", "slab", "pair"][s.kernel], f"mt{s.mt}"]
    parts += [name for on, name in ((s.wres, "wres"), (s.w_taps == 3, "wrow"), (s.multi_n, "nN"), (s.staged, "staged"),
                                    (s.up_fold, "fold"), (s.nchw, "nchw"), (s.residual, "res")) if on]
    return "-".join(parts + [PREC_IDS[prec]])


def _rand(*shape, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _uniform(n, seed, scale):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.rand(n, generator=g) * scale).to(DEV)


def _poisoned(shape, two):
    hi = torch.full(shape, NAN16, dtype=torch.int16, device=DEV)
    return hi, (hi.clone() if two else None)


def _conv(mode, a, w):
    if mode == _lib.MODE_CONV3X3:
        return F.conv2d(a, w, padding=1)
    if mode == _lib.MODE_DOWN2X2:
        return F.conv2d(a, w, stride=2)
    return F.conv_transpose2d(a, w, stride=2)


def _pre(mode, a_eff, a_hi, w_hi, w_lo, conv=None):
    """conv(a, w) as the kernel forms it: bf16x3 multiplies (a_hi + a_lo) w_hi + a_hi w_lo (no lo x lo term)."""
    conv = conv or (lambda a, w: _conv(mode, a, w))
    y = conv(a_eff, w_hi)
    return y if w_lo is None else y + conv(a_hi, w_lo)


def _planes_nchw(hi, lo, prec, c0, c1, idx):
    """fp64 NCHW value hi (+ lo) of channels [c0, c1) of images idx."""
    d = dt16(prec)
    v = hi[idx].view(d)[..., c0:c1].double()
    if lo is not None:
        v = v + lo[idx].view(d)[..., c0:c1].double()
    return v.permute(0, 3, 1, 2).cpu()


def _outside(got, ref, S, prec, nchw):
    return ~((got - ref).abs() <= bound_tol(ref, S, prec, nchw))


@pytest.mark.parametrize("row", ROWS, ids=[_row_id(r) for r in ROWS])
def test_dispatch_parity(row, built_lib):
    t0 = time.time()
    L = _lib.lib()
    layer, prec = row_layer(row)
    mode, B, H, W, cin, cout = layer.mode, layer.B, layer.H, layer.W, layer.cin, layer.cout
    two, d = two_planes(prec), dt16(prec)
    fp16 = prec in _lib.FP16_PRECS
    # the planner still sends this layer to the row's configuration on this device
    sig = signature(plan_layer(layer, prec, L.b200dn_sm_count()), layer, prec)
    assert sig == row_signature(row), f"planner now picks {sig} on {L.b200dn_sm_count()} SMs"

    taps = 9 if mode == _lib.MODE_CONV3X3 else 4
    up = mode == _lib.MODE_UP2X2
    Ho, Wo = (H // 2, W // 2) if mode == _lib.MODE_DOWN2X2 else (2 * H, 2 * W) if up else (H, W)
    seed = sum(row)
    x = _rand(B, H, W, cin, seed=seed)
    w = (_rand(cin, cout, 2, 2, seed=seed + 1, scale=cin ** -0.5) if up else
         _rand(cout, cin, 3 if taps == 9 else 2, 3 if taps == 9 else 2, seed=seed + 1, scale=(2.0 / (taps * cin)) ** 0.5))
    bias = _rand(cout, seed=seed + 2, scale=0.1)
    slope = _uniform(cout, seed + 3, 0.5)               # PReLU slopes <= 1 (the bound assumes it)
    wp = torch.ops.b200dn.pack_weight(w, prec, up)

    in_hi, in_lo = _poisoned((B, H, W, layer.in_ctot), two)
    xh = x.to(d)
    in_hi.view(d)[..., :cin] = xh
    if two:
        in_lo.view(d)[..., :cin] = (x - xh.float()).to(d)
    a = _lib.IgemmArgs()
    a.mode, a.prec, a.B, a.H, a.W, a.cin, a.cout = mode, prec, B, H, W, cin, cout
    a.in_[0], a.in_[1] = in_hi.data_ptr(), (in_lo.data_ptr() if two else None)
    a.in_ctot = layer.in_ctot
    a.wpacked, a.bias, a.slope = wp.data_ptr(), bias.data_ptr(), slope.data_ptr()
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    if fp16:
        a.sat_flag = flag.data_ptr()
    bx = max(1, B // 2)
    if layer.nchw:
        out = torch.full((B, cout, H, W), float("nan"), device=DEV)
        image = _rand(bx, cout, H, W, seed=seed + 4)
        a.out_kind = _lib.OUT_NCHW32
        a.out_nchw, a.res_nchw, a.res_bmod = out.data_ptr(), image.data_ptr(), bx
        bufs = ()
    else:
        if layer.same_buffer:
            out_hi, out_lo = in_hi, in_lo
        else:
            out_hi, out_lo = _poisoned((B, Ho, Wo, layer.out_ctot), two)
        a.out_kind = _lib.OUT_NHWC16
        a.out[0], a.out[1] = out_hi.data_ptr(), (out_lo.data_ptr() if two else None)
        a.out_ctot, a.out_coff = layer.out_ctot, layer.coff
        if layer.residual:           # conv_3: + x, the channels [0, cout) of its own input buffer
            a.res[0], a.res[1] = a.in_[0], a.in_[1]
            a.res_ctot = layer.in_ctot
        bufs = tuple(p for p in (out_hi, out_lo) if p is not None)
    before = [p.clone() for p in bufs]
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(L.b200dn_igemm(C.byref(a), stream), "igemm")
    torch.cuda.synchronize()

    # every byte outside the output slice is unchanged (the input prefix, the other slices, the NaN poison)
    for p, p0 in zip(bufs, before):
        keep = torch.ones(p.shape[-1], dtype=torch.bool, device=DEV)
        keep[layer.coff:layer.coff + cout] = False
        assert torch.equal(p[..., keep], p0[..., keep]), "wrote outside its channel slice"

    idx = sorted({0, B - 1})
    a_hi = _planes_nchw(in_hi, None, prec, 0, cin, idx)        # the input prefix is unchanged (checked above)
    a_eff = _planes_nchw(in_hi, in_lo, prec, 0, cin, idx)
    a_abs = a_hi.abs() + (a_eff - a_hi).abs()
    w_hi = w.to(d).double().cpu()
    w_lo = (w - w.to(d).float()).to(d).double().cpu() if prec == _lib.PREC_BF16X3 else None
    b64, s64 = bias.double().cpu().view(1, -1, 1, 1), slope.double().cpu()
    pre = _pre(mode, a_eff, a_hi, w_hi, w_lo) + b64
    S = _pre(mode, a_abs, a_hi.abs(), w_hi.abs(), None if w_lo is None else w_lo.abs()) + b64.abs()
    if layer.nchw:
        res = image.double().cpu()[[i % bx for i in idx]]
        got = out.double().cpu()[idx]
    else:
        res = a_eff[:, :cout] if layer.residual else torch.zeros(())
        got = _planes_nchw(out_hi, out_lo, prec, layer.coff, layer.coff + cout, idx)
    S = S + res.abs()
    ref = F.prelu(pre, s64) + res
    err = (got - ref).abs()
    need = tol_excess(err, ref, S, prec, layer.nchw)
    print(f"\n[parity] {_row_id(row)} B={B} {H}x{W} {cin}->{cout}: max err {float(err.max()):.3e}, "
          f"kappa needed {need:.3f}")
    bad = _outside(got, ref, S, prec, layer.nchw)
    assert not bad.any(), (f"{int(bad.sum())} / {bad.numel()} outside the bound (kappa needed {need:.2f}), "
                           f"max err {float(err.max()):.3e}")

    # near miss (a): the K16 slice [cin - 16, cin) of one tap (the centre tap of a 3x3) left out
    k0 = max(cin - 16, 0)
    tap = (slice(None), slice(k0, cin), 1, 1) if not up else (slice(k0, cin), slice(None), 1, 1)

    def only_slice(wt):
        if wt is None:
            return None
        z = torch.zeros_like(wt)
        z[tap] = wt[tap]
        return z[:, k0:cin] if not up else z[k0:cin]
    drop = _pre(mode, a_eff[:, k0:cin], a_hi[:, k0:cin], only_slice(w_hi), only_slice(w_lo))
    assert _outside(got, F.prelu(pre - drop, s64) + res, S, prec, layer.nchw).any(), \
        "the bound accepts a reference with one K16 slice of a tap missing"
    # near miss (b), on the first output row(s): replicate padding (3x3), or the taps mirrored along x (2x2)
    if mode == _lib.MODE_CONV3X3:
        rows_out, rows_in = 1, 2
        conv_b = lambda t, wt: F.conv2d(F.pad(t, (1, 1, 1, 1), mode="replicate"), wt)[:, :, :1]   # noqa: E731
    else:
        rows_out, rows_in = (1, 2) if not up else (2, 1)
        conv_b = lambda t, wt: _conv(mode, t, wt.flip(-1))                                         # noqa: E731
    pre_b = _pre(mode, a_eff[:, :, :rows_in], a_hi[:, :, :rows_in], w_hi, w_lo, conv_b) + b64
    res_b = res[:, :, :rows_out] if res.dim() else res
    ref_b = F.prelu(pre_b, s64) + res_b
    assert _outside(got[:, :, :rows_out], ref_b, S[:, :, :rows_out], prec, layer.nchw).any(), \
        "the bound accepts a reference with the wrong border handling"

    if fp16:
        # the saturation watch: nothing saturates with the real weights; one channel's bias at 1e5 stores +65504 there
        # (fp16 storage) and raises the flag.  The fp32 NCHW output does not saturate and leaves the flag alone.
        assert int(flag.item()) == 0
        hot = bias.clone()
        hot[cout - 1] = 1e5
        a.bias = hot.data_ptr()
        _lib.check(L.b200dn_igemm(C.byref(a), stream), "igemm")
        torch.cuda.synchronize()
        if layer.nchw:
            assert int(flag.item()) == 0
            assert bool((out[:, cout - 1] > 65504).all())
        else:
            assert int(flag.item()) == 1, "an fp16 output saturated without raising sat_flag"
            ch = out_hi.view(d)[..., layer.coff + cout - 1].float()
            assert bool((ch == 65504.0).all()), f"saturated channel stores {ch.unique()[:8].tolist()}"
    print(f"[parity] {_row_id(row)}: {time.time() - t0:.2f} s")


# ------------------------------------------------------------------------------------------- chain kernel, per layer
CHAIN_SHAPES = [
    # C, B, H, W, prec, expected (mt, N tiles of the last layer) on 148 SMs
    (64, 5, 128, 128, _lib.PREC_FP16, (2, 1)),       # MT = 2, growth layers on N = 32 pairs
    (256, 1, 32, 32, _lib.PREC_BF16, (1, 4)),        # MT = 1, N split to 64: 2 tiles per growth conv, 4 for the last
]


def _block(C, B, H, W, prec, n, seed, exact=False):
    """n layers of a DenoisingBlock of C channels in the network's layout (helpers.block_launches), on random data or,
    with `exact`, on helpers.dyadic_block data."""
    d, g = dt16(prec), C // 2
    if not exact:
        shapes = [(g, C + k * g) for k in range(n - 1)] + [(C, C + (n - 1) * g)]
        x = _rand(B, H, W, C, seed=seed, scale=0.5)
        ws = [_rand(co, ci, 3, 3, seed=seed + 1 + j, scale=(2.0 / (9 * ci)) ** 0.5) for j, (co, ci) in enumerate(shapes)]
        bs = [_rand(co, seed=seed + 10 + j, scale=0.1) for j, (co, _) in enumerate(shapes)]
        ss = [_uniform(co, seed + 20 + j, 0.5) for j, (co, _) in enumerate(shapes)]
    else:
        x, ws, bs, ss = dyadic_block(C, B, H, W, seed, n)
        x = x.permute(0, 2, 3, 1).to(DEV)
        ws, bs, ss = ([t.to(DEV) for t in ts] for ts in (ws, bs, ss))
    blk = block_launches(x.to(d), ws, bs, ss, prec)
    blk.update(ws=ws, bs=bs, ss=ss)
    return blk


def _chain(blk, flags):
    L = _lib.lib()
    n = len(blk["shapes"])
    nbytes = L.b200dn_conv_chain_workspace_bytes(blk["args"], n)
    ws = torch.zeros(max(int(nbytes), 64) // 4, dtype=torch.int32, device=DEV)
    h = C.c_void_p()
    rc = L.b200dn_conv_chain_prepare(blk["args"], n, ws.data_ptr(), flags, C.byref(h))
    return rc, h, ws


@pytest.mark.parametrize("n", [2, 3, 4])
@pytest.mark.parametrize("shape", CHAIN_SHAPES, ids=["mt2", "mt1-split-n"])
def test_chain_layers(shape, n, built_lib):
    C_, B, H, W, prec, (mt, n_last) = shape
    L = _lib.lib()
    d, g = dt16(prec), C_ // 2
    stream = torch.cuda.current_stream().cuda_stream
    sms = L.b200dn_sm_count()
    blk = _block(C_, B, H, W, prec, n, seed=100 * n + C_)
    for k, (co, ci) in enumerate(blk["shapes"]):
        i = plan(0, B, H, W, ci, co, prec=prec, in_ctot=C_ * 5 // 2, out_ctot=C_ * 5 // 2, coff=ci if k < n - 1 else 0,
                 sms=sms)
        assert i.kernel == 2 and i.mt == mt, (k, i.kernel, i.mt)
    assert i.num_n_tiles == n_last

    # per-layer launches
    src0 = blk["src"].clone()
    run_block_launches(blk, stream)
    torch.cuda.synchronize()
    per_src, per_dst = blk["src"].clone(), blk["dst"].clone()
    # the chain: three launches on one workspace zero-filled once (monotonic epoch counters)
    blk["src"].copy_(src0)
    blk["dst"].fill_(NAN16)
    rc, h, ws = _chain(blk, 1)                        # B200DN_CHAIN_FORCE
    _lib.check(rc, "conv_chain_prepare")
    outs = []
    for _ in range(3):
        _lib.check(L.b200dn_igemm_launch(h, stream), "chain launch")
        torch.cuda.synchronize()
        outs.append((blk["src"].clone(), blk["dst"].clone()))
    L.b200dn_igemm_release(h)
    for s, o in outs:
        assert torch.equal(s, per_src) and torch.equal(o, per_dst), "chain differs from the per-layer launches"

    # each layer against fp64 on the operands it read (the stored 16-bit o_k of the layers before it), first and last image
    idx = sorted({0, B - 1})
    cat = per_src[idx].view(d).double().permute(0, 3, 1, 2).cpu()
    x = cat[:, :C_]
    for k, (co, ci) in enumerate(blk["shapes"]):
        wk = blk["ws"][k].to(d).double().cpu()
        bk = blk["bs"][k].double().cpu().view(1, -1, 1, 1)
        res = x if k == n - 1 else torch.zeros(())
        ref = F.prelu(F.conv2d(cat[:, :ci], wk, padding=1) + bk, blk["ss"][k].double().cpu()) + res
        S = F.conv2d(cat[:, :ci].abs(), wk.abs(), padding=1) + bk.abs() + res.abs()
        got = cat[:, ci:ci + co] if k < n - 1 else per_dst[idx].view(d)[..., :C_].double().permute(0, 3, 1, 2).cpu()
        bad = _outside(got, ref, S, prec, False)
        assert not bad.any(), f"layer {k}: {int(bad.sum())} outside the bound"
    # untouched: the unread tail of the input buffer and the rest of the output buffer keep their NaN poison
    top = C_ + (n - 1) * g
    assert bool((per_src[..., top:] == NAN16).all()) and bool((per_dst[..., C_:] == NAN16).all())
    assert torch.equal(per_src[..., :C_], src0[..., :C_])
    # the whole block, per layer and chained, bit for bit against fp64 on data whose arithmetic is exact
    # (helpers.dyadic_block; the reference asserts that premise for every conv)
    ex = _block(C_, B, H, W, prec, n, seed=100 * n + C_, exact=True)
    run_block_launches(ex, stream)
    torch.cuda.synchronize()
    per_dst = ex["dst"].clone()
    ex["dst"].fill_(NAN16)
    rc, h, ws = _chain(ex, 1)
    _lib.check(rc, "conv_chain_prepare")
    _lib.check(L.b200dn_igemm_launch(h, stream), "chain launch")
    torch.cuda.synchronize()
    L.b200dn_igemm_release(h)
    assert torch.equal(ex["dst"], per_dst), "chain differs from the per-layer launches on exact data"
    x16 = ex["src"][idx][..., :C_].view(d).permute(0, 3, 1, 2).cpu()
    bits = []
    ref = store16(dense_block_ref(x16, [t.cpu() for t in ex["ws"]], [t.cpu() for t in ex["bs"]],
                                  [t.cpu() for t in ex["ss"]], d, premise=bits), d)
    got = per_dst[idx][..., :C_].view(d).permute(0, 3, 1, 2).cpu()
    print(f"\n[chain] C={C_} n={n}: exact-data partial sums need 2^{max(bits):.2f} steps of their grid")
    diff = got.view(torch.int16) != ref.view(torch.int16)
    assert not diff.any(), f"{int(diff.sum())} / {diff.numel()} output values differ from the exact block"


def test_chain_needs_two_pair_tiles_per_cluster(built_lib):
    """Without B200DN_CHAIN_FORCE a chain whose layers give fewer than two pair tiles per cluster is refused (E_UNSUP):
    the layers would not overlap, four launches are as fast."""
    blk = _block(256, 1, 32, 32, _lib.PREC_BF16, 4, seed=7)
    rc, h, _ = _chain(blk, 0)
    assert rc == _lib.E_UNSUP and not h.value
