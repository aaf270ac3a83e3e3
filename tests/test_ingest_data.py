"""The exact-arithmetic ingest conv data (helpers.dyadic_ingest) on the CPU: the image splits exactly into 16-bit hi +
lo planes and the lo plane is not empty, the premise the bit-exact GPU test rests on holds at every row it runs, an fp32
evaluation in another order (another channel order, another hi / lo split, the twin epilogue's t * sum(w_t))
reproduces the fp64 reference bit for bit, and the reference sees the near misses the GPU test is there to catch."""
import pytest
import torch
import torch.nn.functional as F

from helpers import (INGEST_BITS, INGEST_ROWS, INGEST_X, dyadic_ingest, dyadic_timesteps, ingest_planes, ingest_premise,
                     ingest_ref, ingest_row_data, ingest_row_id, store16, t_view)

DTS = [torch.float16, torch.bfloat16]
DT_IDS = ["fp16", "bf16"]


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
def test_image_split_is_exact(dt):
    """Every x = k / 2^12, |k| <= 2^12, is hi + lo exactly, with the kernels' split (hi = rn(x), lo = rn(x - hi) in
    fp32); the lo plane is nonzero for ~80 % of the values in bf16 and ~25 % in fp16."""
    x = torch.arange(-2 ** INGEST_X, 2 ** INGEST_X + 1).float() / 2 ** INGEST_X
    hi = x.to(dt)
    lo = (x - hi.float()).to(dt)
    assert torch.equal(hi.double() + lo.double(), x.double())
    frac = float((lo != 0).double().mean())
    assert frac > (0.7 if dt == torch.bfloat16 else 0.2), frac


@pytest.mark.parametrize("row", INGEST_ROWS, ids=[ingest_row_id(r) for r in INGEST_ROWS])
def test_ingest_premise_holds(row):
    """On the images the GPU test checks (0, Bx - 1, Bx, B - 1), with the same seed."""
    cimg, tk, Bx, B, H, W, cout, _ = row
    x, t_src, strides, w, b, s = ingest_row_data(row, seed=sum(row[2:]))
    idx = sorted({0, Bx - 1, min(Bx, B - 1), B - 1})
    t = t_view(t_src, strides, B, H, W)[idx] if t_src is not None else None
    v, S = ingest_ref(x[[i % Bx for i in idx]], t, w, b, s)
    assert ingest_premise(x, t_src, w, b, v, S) <= INGEST_BITS


def _fp32_ingest(x, t, w, b, s, split_dt, twin, seed):
    """The ingest in fp32, summed in another order: the image as hi + lo of split_dt, each plane convolved
    separately with the channels in a random order; the t plane as its own channel or, in twin form, as
    t * (sum of the t-plane weights over the in-image taps) added after the bias."""
    g = torch.Generator().manual_seed(seed)
    hi = x.to(split_dt).float()
    lo = x - hi
    p = torch.randperm(x.shape[1], generator=g)
    wx = w[:, :x.shape[1]]
    acc = F.conv2d(lo[:, p], wx[:, p], padding=1) + F.conv2d(hi[:, p], wx[:, p], padding=1)
    if t is not None and not twin:
        acc = F.conv2d(t, w[:, -1:], padding=1) + acc
    acc = acc + b.view(1, -1, 1, 1)
    if twin:
        ones = torch.ones_like(t[:1])
        acc = acc + t[:, :, :1, :1] * F.conv2d(ones, w[:, -1:], padding=1)
    return F.prelu(acc, s)


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
@pytest.mark.parametrize("cimg,kind", [(3, "twin"), (3, "plane"), (1, "twin"), (3, None), (1, None)])
def test_fp32_reproduces_the_reference(dt, cimg, kind):
    B, H, W, cout = 2, 19, 27, 64
    x, w, b, s = dyadic_ingest(B, cimg, H, W, cout, kind is not None, seed=3 + cimg)
    t = None
    if kind == "twin":
        t = dyadic_timesteps(B, seed=4).view(B, 1, 1, 1).expand(B, 1, H, W)
    elif kind == "plane":
        t = dyadic_timesteps(B * H * W, seed=4).view(B, 1, H, W)
    v, S = ingest_ref(x, t, w, b, s)
    ingest_premise(x, t, w, b, v, S)
    other = torch.bfloat16 if dt == torch.float16 else torch.float16
    for seed in range(3):
        for split in (dt, other):
            got = _fp32_ingest(x, t, w, b, s, split, kind == "twin", seed)
            assert torch.equal(got.double(), v), (seed, split)
            for p, q in zip(ingest_planes(got.double(), dt, True), ingest_planes(v, dt, True)):
                assert torch.equal(p.view(torch.int16), q.view(torch.int16))


@pytest.mark.parametrize("dt", DTS, ids=DT_IDS)
def test_reference_sees_the_near_misses(dt):
    """A gather that drops the image's lo plane moves the stored hi plane somewhere and the lo plane of the two-plane
    modes almost everywhere; a twin epilogue that adds the inner class's t term at the border moves most border
    outputs."""
    B, H, W, cout = 2, 32, 40, 32
    x, w, b, s = dyadic_ingest(B, 3, H, W, cout, True, seed=11)
    t = dyadic_timesteps(B, seed=12).view(B, 1, 1, 1).expand(B, 1, H, W)
    v, _ = ingest_ref(x, t, w, b, s)
    hi, lo = ingest_planes(v, dt, True)
    no_lo, _ = ingest_ref(x.to(dt).float(), t, w, b, s)
    hi_b, lo_b = ingest_planes(no_lo, dt, True)
    assert int((hi_b != hi).sum()) > v.numel() // 1000
    assert float((lo_b != lo).double().mean()) > 0.5
    inner, _ = ingest_ref(x, t, w, b, s, t_pad="replicate")
    border = torch.ones(H, W, dtype=torch.bool)
    border[1:-1, 1:-1] = False
    changed = store16(inner, dt) != store16(v, dt)
    assert not changed[..., ~border].any()
    assert float(changed[..., border].double().mean()) > 0.3
