"""The fused DenoisingBlock kernel (dense_block_kernel, csrc/dense_block_sm100.cu) bit for bit against an exact fp64
reference, in the network's buffer layouts and up to the sampler's batch.

The data come from helpers.dyadic_block: operands on coarse dyadic grids, so that every product and partial sum of
every pass is exact in fp32 whatever the summation order, and the only roundings are the 16-bit stores of o0..o2 and
of the output (round to nearest even of an exact value, the same on the GPU and in torch).  The kernel must therefore
store exactly store16(dense_block_ref(...)); there is no tolerance.  The reference asserts that premise for every conv.

Each case also runs the block as its four per-layer b200dn_igemm launches (helpers.block_launches), which are exact by
the same argument.  Fused, per-layer and fp64 must all agree: if fused and per-layer agree with each other but not with
fp64, the premise (the tensor cores accumulate exactly while every partial sum fits 24 bits) is what failed.

Per case: both epilogue variants (bias / slopes staged in shared memory, and as launch constants as the network runs
them) give the same bits; the first, the last and a middle image equal fp64; every image equals the per-layer launches;
every byte outside the output slice is unchanged; a second launch of the same handle stores the same bits; the fp16
saturation flag stays 0.  Regions are 18 x 26 output pixels; CTA pairs take two regions per item.
"""
import ctypes as C
import functools
import re
import time

import pytest
import torch

from helpers import NAN16, block_launches, dense_block_ref, dyadic_block, run_block_launches, store16
from vub_image_denoising_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda"
PRECS = {"fp16": _lib.PREC_FP16, "bf16": _lib.PREC_BF16}
DTS = {"fp16": torch.float16, "bf16": torch.bfloat16}

# (B, H, W, prec, max_ctas, CTA pairs): cases that share (B, H, W, prec) share data and reference, so they stay adjacent
_SHAPES = [
    (1, 1, 1),          # 1 region: a 1-pixel image, one live tile column, the TMA box larger than the tensor
    (1, 26, 18),        # exactly one region
    (3, 26, 18),        # 3 regions: the phantom region of the last pair
    (1, 200, 3),        # 8 regions in one region column 3 pixels wide
    (3, 53, 37),        # 27 regions: seams in x and y, cheap last column numbered last, one live tile column there
    (1, 130, 90),       # 25 regions: no cheap column, three live tile columns
    (2, 64, 64),        # 24 regions: two live tile columns in the last region column
    (1, 512, 512),      # 580 regions: 4 rounds per cluster
]
CASES = []
for _B, _H, _W in _SHAPES:
    for _p in ("fp16", "bf16"):
        CASES.append((_B, _H, _W, _p, 0, True))
        if (_B, _H, _W) == (3, 53, 37):
            # 27 items on one CTA (max_ctas = 1 leaves the pair kernel), 14 items on one cluster, 5 rounds on three
            CASES += [(_B, _H, _W, _p, m, True) for m in (1, 2, 6)]
        if (_B, _H, _W) in ((3, 53, 37), (1, 512, 512)):
            CASES.append((_B, _H, _W, _p, 0, False))          # B200DN_DENSE_PAIR=0: one CTA per region
CASES += [(32, 256, 256, "fp16", 0, True),     # the sampler's level-0 launch: 4,800 regions, 33 rounds per cluster
          (16, 256, 256, "bf16", 0, True)]


def _case_id(c):
    B, H, W, p, m, pair = c
    return f"{B}x{H}x{W}-{p}" + (f"-max{m}" if m else "") + ("" if pair else "-single")


# (name, in_ctot, out_ctot, out_coff, output in the input buffer)
LAYOUTS = [
    ("net", 32, 32, 0, False),        # a fused level's 32-channel dense buffer -> the next one
    ("skip", 32, 96, 0, False),       # -> channels [0, 32) of the 96-channel skip buffer
    ("wide", 64, 32, 0, False),       # a wider input: channels [32, 64) hold NaN and must not be read
    ("inplace", 64, 64, 32, True),    # the output slice [32, 64) of the input buffer itself
]


class Block:
    """One block's data on the GPU (x NHWC 16-bit, fp32 weights packed for the fused kernel, bias / slopes on the device
    and on the host), the per-layer launches' output and the fp64 reference of a few images."""

    def __init__(self, B, H, W, prec, seed, hot=None):
        self.B, self.H, self.W, self.prec, self.dt = B, H, W, PRECS[prec], DTS[prec]
        x, ws, bs, ss = dyadic_block(32, B, H, W, seed)
        if hot is not None:          # (conv, channel): saturate it; later convs do not read an o_k channel driven so
            k, c = hot
            bs[k][c] = 1e5
            for j in range(k + 1, 4):
                ws[j][:, 32 + 16 * k + c] = 0
        self.x16 = x.permute(0, 2, 3, 1).to(self.dt).to(DEV).contiguous()
        self.ws, self.bs, self.ss = ([t.to(DEV) for t in ts] for ts in (ws, bs, ss))
        self.hb, self.hs = bs, ss
        L = _lib.lib()
        stream = torch.cuda.current_stream().cuda_stream
        self.wf = torch.empty(L.b200dn_dense_block_weight_bytes(32) // 2, dtype=torch.int16, device=DEV)
        _lib.check(L.b200dn_pack_dense_block_weights(*[w.data_ptr() for w in self.ws], 32, self.prec,
                                                     self.wf.data_ptr(), stream), "pack_dense_block_weights")
        lay = block_launches(self.x16, self.ws, self.bs, self.ss, self.prec)
        run_block_launches(lay, stream)
        torch.cuda.synchronize()
        self.per_layer = lay["dst"][..., :32].clone()
        del lay
        self.idx = sorted({0, B // 2, B - 1} if B >= 3 else {0, B - 1})
        t0 = time.time()
        self.bits = []
        ref = dense_block_ref(x[self.idx].to(self.dt), ws, bs, ss, self.dt, premise=self.bits)
        self.ref = store16(ref, self.dt).permute(0, 2, 3, 1).contiguous().view(torch.int16)
        self.ref_s = time.time() - t0

    def args(self, inp, in_ctot, out, out_ctot, out_coff, flag, max_ctas=0, timeline=None):
        a = _lib.DenseBlockArgs()
        a.prec, a.B, a.H, a.W, a.channels = self.prec, self.B, self.H, self.W, 32
        a.in_, a.in_ctot = inp.data_ptr(), in_ctot
        a.out, a.out_ctot, a.out_coff = out.data_ptr(), out_ctot, out_coff
        a.wfused = self.wf.data_ptr()
        for j in range(4):
            a.bias[j], a.slope[j] = self.bs[j].data_ptr(), self.ss[j].data_ptr()
        a.max_ctas = max_ctas
        a.sat_flag = flag.data_ptr()
        if timeline is not None:
            a.timeline = timeline.data_ptr()
        return a

    def set_constants(self, h):
        fp = C.POINTER(C.c_float)
        bias = (fp * 4)(*[C.cast(t.data_ptr(), fp) for t in self.hb])
        slope = (fp * 4)(*[C.cast(t.data_ptr(), fp) for t in self.hs])
        _lib.check(_lib.lib().b200dn_dense_block_set_epilogue_constants(h, bias, slope), "set_epilogue_constants")

    def run(self, layout, max_ctas=0, timeline=None):
        """The block in `layout`, staged then with launch constants, each launch on freshly poisoned output channels.
        Returns (output slice, sat_flag) after checking the launches against each other and the bytes outside the slice."""
        name, in_ctot, out_ctot, coff, same = layout
        B, H, W = self.B, self.H, self.W
        inp = torch.full((B, H, W, in_ctot), NAN16, dtype=torch.int16, device=DEV)
        inp[..., :32] = self.x16.view(torch.int16)
        out = inp if same else torch.full((B, H, W, out_ctot), NAN16, dtype=torch.int16, device=DEV)
        before = out.clone()
        flag = torch.zeros(1, dtype=torch.int32, device=DEV)
        L = _lib.lib()
        stream = torch.cuda.current_stream().cuda_stream
        h = C.c_void_p()
        _lib.check(L.b200dn_dense_block_prepare(C.byref(self.args(inp, in_ctot, out, out_ctot, coff, flag, max_ctas,
                                                                   timeline)), C.byref(h)), "dense_block_prepare")
        got = []
        try:
            for step in range(3):          # staged; launch constants (the network's path); the same handle again
                if step == 1:
                    self.set_constants(h)
                out[..., coff:coff + 32] = NAN16
                _lib.check(L.b200dn_igemm_launch(h, stream), "dense block launch")
                torch.cuda.synchronize()
                got.append(out.clone())
        finally:
            L.b200dn_igemm_release(h)
        keep = torch.ones(out_ctot, dtype=torch.bool, device=DEV)
        keep[coff:coff + 32] = False
        for step, o in enumerate(got):
            assert torch.equal(o[..., keep], before[..., keep]), f"{name}: launch {step} wrote outside its channel slice"
        assert torch.equal(got[1], got[0]), f"{name}: launch constants and staged bias / slopes store different bits"
        assert torch.equal(got[2], got[1]), f"{name}: a second launch of the same handle stores different bits"
        return got[1][..., coff:coff + 32], int(flag.item())

    def check(self, got, what):
        """got (B, H, W, 32 int16) against fp64 on self.idx and against the per-layer launches on every image."""
        fused_ref, layer_ref = _diff(got[self.idx].cpu(), self.ref), _diff(self.per_layer[self.idx].cpu(), self.ref)
        fused_layer = _diff(got, self.per_layer)
        if fused_ref and layer_ref:
            pytest.fail(f"{what}: fused and per-layer kernels both differ from the exact fp64 value: the premise that "
                        f"the tensor cores accumulate exactly within 24 bits fails (fused: {fused_ref}; per-layer: "
                        f"{layer_ref}; fused vs per-layer: {fused_layer or 'equal'})")
        assert not fused_ref, f"{what}: the fused kernel differs from fp64 (per-layer matches it): {fused_ref}"
        assert not layer_ref, f"{what}: the per-layer launches differ from fp64 (fused matches it): {layer_ref}"
        assert not fused_layer, f"{what}: the fused kernel differs from the per-layer launches: {fused_layer}"


def _diff(got, want):
    """'' when the 16-bit patterns are equal, else how many differ and the first one (NHWC position)."""
    bad = got != want
    if not bool(bad.any()):
        return ""
    pos = [int(v) for v in bad.nonzero()[0]]
    g, w = int(got[tuple(pos)]) & 0xFFFF, int(want[tuple(pos)]) & 0xFFFF
    return f"{int(bad.sum())} of {bad.numel()} values differ, first at (b, y, x, c) = {tuple(pos)}: {g:#06x} vs {w:#06x}"


@functools.lru_cache(maxsize=1)
def _block(B, H, W, prec):
    return Block(B, H, W, prec, seed=B * 1000003 + H * 1009 + W)


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_dense_block_exact(case, built_lib, monkeypatch):
    B, H, W, prec, max_ctas, pair = case
    t0 = time.time()
    blk = _block(B, H, W, prec)
    if not pair:
        monkeypatch.setenv("B200DN_DENSE_PAIR", "0")        # read at prepare
    for layout in LAYOUTS:
        got, flag = blk.run(layout, max_ctas)
        blk.check(got, f"{_case_id(case)} {layout[0]}")
        assert flag == 0, f"{layout[0]}: sat_flag raised without a saturated value"
    print(f"\n[dense] {_case_id(case)}: exact-data partial sums need 2^{max(blk.bits):.2f} steps of their grid; "
          f"fp64 reference {blk.ref_s:.1f} s, case {time.time() - t0:.1f} s")


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_dense_block_timeline_variant(prec, built_lib):
    """With a timeline buffer the block runs on the one-CTA diagnostics kernel; it stores the same bits."""
    blk = _block(3, 53, 37, prec)
    tl = torch.zeros(3 * 2730, dtype=torch.int64, device=DEV)
    got, flag = blk.run(LAYOUTS[0], timeline=tl)
    blk.check(got, "timeline")
    assert flag == 0
    assert bool((tl != 0).any()), "the timeline buffer was not written: the diagnostics kernel did not run"


# (conv, channel) driven to saturation by a bias of 1e5: an o_k that stays in shared memory, or an output channel
HOT = [(0, 3), (1, 9), (2, 14), (3, 21)]


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("hot", HOT, ids=[f"conv{k}" for k, _ in HOT])
def test_dense_block_saturation(hot, prec, built_lib):
    """fp16 stores saturate to 65504 and raise sat_flag, from the intermediate watch on o0..o2 (the later convs do not
    read the saturated channel, so the output stays exact) and from the output watch.  bf16 has the range: no flag."""
    k, c = hot
    blk = Block(3, 53, 37, prec, seed=77, hot=hot)
    got, flag = blk.run(LAYOUTS[0])
    blk.check(got, f"conv_{k} channel {c} at 1e5")
    if prec == "fp16":
        assert flag == 1, f"an fp16 value of conv_{k} saturated without raising sat_flag"
        if k == 3:
            assert bool((got[..., c] == 0x7BFF).all()), "the saturated output channel does not store 65504 everywhere"
    else:
        assert flag == 0


def test_dense_block_argument_errors(built_lib):
    """Arguments the fused kernel does not support come back as B200DN_E_ARG with a message and no handle."""
    L = _lib.lib()
    blk = _block(1, 26, 18, "bf16")
    inp = torch.zeros((1, 26, 18, 64), dtype=torch.int16, device=DEV)
    out = torch.zeros((1, 26, 18, 64), dtype=torch.int16, device=DEV)
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)

    def prepare(**kw):
        a = blk.args(inp, 64, out, 64, 0, flag)
        for k, v in kw.items():
            if k == "bias2":
                a.bias[2] = None
            else:
                setattr(a, k, v)
        h = C.c_void_p()
        rc = L.b200dn_dense_block_prepare(C.byref(a), C.byref(h))
        msg = L.b200dn_last_error().decode()
        if rc == 0:
            L.b200dn_igemm_release(h)
        else:
            assert not h.value
        return rc, msg

    assert prepare()[0] == 0
    bad = [
        (dict(channels=64), "only 32-channel blocks"),
        (dict(prec=_lib.PREC_BF16X2), "single-plane"),
        (dict(in_ctot=36), "bad in_ctot 36"),
        (dict(in_ctot=24), "bad in_ctot 24"),
        (dict(out_coff=4), "must be 8-channel aligned"),
        (dict(out_coff=40), r"output slice \[40,72\) of 64"),
        (dict(out=inp.data_ptr(), out_coff=16), "overlaps the block input"),
        (dict(bias2=None), "null bias / slope 2"),
    ]
    for kw, pattern in bad:
        rc, msg = prepare(**kw)
        assert rc == _lib.E_ARG, (kw, rc, msg)
        assert re.search(pattern, msg), (kw, msg)
