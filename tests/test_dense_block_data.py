"""The exact-arithmetic DenoisingBlock data (helpers.dyadic_block) on the CPU: the premise the bit-exact GPU tests rest
on holds at the widths they use, an fp32 evaluation in another summation order reproduces the fp64 reference bit for
bit, and the data are sensitive to a channel mix-up of the slopes or biases."""
import pytest
import torch
import torch.nn.functional as F

from helpers import DYADIC_BITS, dense_block_ref, dyadic_block, store16

DTS = [torch.float16, torch.bfloat16]


@pytest.mark.parametrize("C,B,H,W,n", [(32, 1, 256, 256, 4), (64, 1, 128, 128, 2), (64, 1, 128, 128, 3),
                                       (64, 1, 128, 128, 4), (256, 1, 32, 32, 4)])
def test_dyadic_premise_holds(C, B, H, W, n):
    x, ws, bs, ss = dyadic_block(C, B, H, W, seed=C + n, n=n)
    for dt in DTS:
        bits = []
        dense_block_ref(x.to(dt), ws, bs, ss, dt, premise=bits)       # asserts the premise conv by conv
        assert len(bits) == n and max(bits) <= DYADIC_BITS


def _fp32_block(x16, ws, bs, ss, dt, seed):
    """The block in fp32 with the input channels of every conv summed in a random order, in two partial sums."""
    g = torch.Generator().manual_seed(seed)
    cat = x16.float()
    for j in range(len(ws)):
        p = torch.randperm(cat.shape[1], generator=g)
        h = cat.shape[1] // 3
        w = ws[j].to(dt).float()
        pre = F.conv2d(cat[:, p[h:]], w[:, p[h:]], padding=1) + F.conv2d(cat[:, p[:h]], w[:, p[:h]], padding=1)
        v = F.prelu(pre + bs[j].view(1, -1, 1, 1), ss[j])
        if j == len(ws) - 1:
            return store16(v + x16.float(), dt)
        cat = torch.cat([cat, store16(v, dt).float()], 1)


@pytest.mark.parametrize("dt", DTS, ids=["fp16", "bf16"])
def test_dyadic_block_is_exact_in_fp32(dt):
    x, ws, bs, ss = dyadic_block(32, 2, 53, 37, seed=5)
    ref = store16(dense_block_ref(x.to(dt), ws, bs, ss, dt), dt)
    for seed in range(3):
        assert torch.equal(_fp32_block(x.to(dt), ws, bs, ss, dt, seed).view(torch.int16), ref.view(torch.int16))


@pytest.mark.parametrize("dt", DTS, ids=["fp16", "bf16"])
def test_dyadic_block_sees_channel_mixups(dt):
    """A kernel that reads the slopes of conv_3's channels 16..31 from 0..15, or swaps two biases of conv_2, stores
    different bits in many places."""
    x, ws, bs, ss = dyadic_block(32, 1, 53, 37, seed=9)
    x16 = x.to(dt)
    ref = store16(dense_block_ref(x16, ws, bs, ss, dt), dt)
    s3 = ss[3].clone()
    s3[16:] = s3[:16]
    b2 = bs[2].clone()
    b2[[4, 11]] = b2[[11, 4]]
    for what, bad in (("slopes", dense_block_ref(x16, ws, bs, ss[:3] + [s3], dt)),
                      ("biases", dense_block_ref(x16, ws, bs[:2] + [b2, bs[3]], ss, dt))):
        changed = int((store16(bad, dt) != ref).sum())
        assert changed > ref.numel() // 100, f"{what}: only {changed} of {ref.numel()} outputs change"
