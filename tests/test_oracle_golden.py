"""CPU: the oracle reproduces the reference's own outputs (golden vectors generated from the real reference
modules by oracle/pin_against_reference.py), and the drop-in modules reproduce the reference constructor's
seeded initialisation and state_dict layout."""
import numpy as np
import pytest
import torch

from helpers import sd_digest
import vub_image_denoising_b200 as b2
from oracle import rdunet_oracle as orc


def _t(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(autouse=True)
def golden_thread_count():
    """The CPU forward matches the stored reference outputs bit for bit only at the thread count they were made with."""
    before = torch.get_num_threads()
    torch.set_num_threads(orc.GOLDEN_THREADS)
    yield
    torch.set_num_threads(before)


def test_state_dict_layout_matches_reference():
    torch.manual_seed(7)
    net = b2.RDUNet(base_filters=16)
    sd = net.state_dict()
    assert len(sd) == 207
    assert sum(k.endswith(".bias") for k in sd) == 69
    assert sum(k.endswith(".weight") for k in sd) == 138
    assert sd["down_0.conv.weight"].shape == (32, 16, 2, 2)
    assert sd["up_2.conv_t.weight"].shape == (128, 128, 2, 2)       # ConvTranspose2d is [Cin, Cout, 2, 2]
    assert sd["up_2.conv.weight"].shape == (64, 192, 3, 3)
    assert sd["block_3_1.conv_3.weight"].shape == (128, 320, 3, 3)
    assert sd["output_block.actv_2.weight"].shape == (3,)
    assert all(v.dtype == torch.float32 for v in sd.values())
    t = b2.RDUNet_T(base_filters=16)
    assert t.state_dict()["input_block.conv_1.weight"].shape == (16, 4, 3, 3)
    assert t.state_dict()["output_block.conv_2.weight"].shape == (3, 16, 3, 3)
    d = b2.DiffusionModel(t)
    assert all(k.startswith("unet.") for k in d.state_dict())
    assert d.timesteps == 20
    d.timesteps = 7                                                   # mutable attribute (evaluate_model.py:105)
    assert d.timesteps == 7


def test_seeded_init_equals_reference(golden):
    torch.manual_seed(7)
    assert sd_digest(b2.RDUNet(base_filters=16).state_dict()) == bytes(golden["A_digest"]).hex()
    torch.manual_seed(11)
    assert sd_digest(b2.RDUNet_T(base_filters=16).state_dict()) == bytes(golden["B_digest"]).hex()
    torch.manual_seed(13)
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=16), timesteps=4)
    assert sd_digest(dm.state_dict()) == bytes(golden["C_digest"]).hex()


def test_oracle_rdunet_matches_reference_outputs(golden):
    torch.manual_seed(7)
    sd = b2.RDUNet(base_filters=16).state_dict()
    with torch.no_grad():
        for k in ("0", "1"):
            y = orc.rdunet_forward(sd, _t(golden[f"A_x{k}"]))
            assert torch.equal(y, _t(golden[f"A_y{k}"]))


def test_oracle_grayscale_matches_reference_outputs(golden):
    """RDUNet(channels=1): seeded init == the reference ctor's, oracle == the reference's output."""
    torch.manual_seed(17)
    net = b2.RDUNet(channels=1, base_filters=16)
    sd = net.state_dict()
    assert sd_digest(sd) == bytes(golden["E_digest"]).hex()
    assert sd["input_block.conv_1.weight"].shape == (16, 1, 3, 3) and sd["output_block.conv_2.weight"].shape == (1, 16, 3, 3)
    with torch.no_grad():
        assert torch.equal(orc.rdunet_forward(sd, _t(golden["E_x"])), _t(golden["E_y"]))


def test_oracle_and_zero_padded_embedding_at_widths_off_the_channel_tiling(golden):
    """base_filters = 24 / 10 (growth = F // 2): seeded init == the reference ctor's, oracle == the reference's outputs,
    and the zero-padded network the launch plan is built from (rdunet._zero_padded_network) computes the same
    function — checked with the oracle on the CPU, so the embedding is pinned without a GPU."""
    from vub_image_denoising_b200.rdunet import _zero_padded_network
    with torch.no_grad():
        torch.manual_seed(19)
        n24 = b2.RDUNet(base_filters=24)
        assert sd_digest(n24.state_dict()) == bytes(golden["F_digest24"]).hex()
        x, y = _t(golden["F_x24"]), _t(golden["F_y24"])
        assert torch.equal(orc.rdunet_forward(n24.state_dict(), x), y)
        wide = _zero_padded_network(n24, 32)
        assert wide.base_filters == 32 and wide.block_0_0.conv_1.weight.shape == (16, 48, 3, 3)
        assert float((orc.rdunet_forward(wide.state_dict(), x) - y).abs().max()) < 2e-6
        torch.manual_seed(23)
        n10 = b2.RDUNet_T(base_filters=10)
        assert sd_digest(n10.state_dict()) == bytes(golden["F_digest10"]).hex()
        x, t, y = _t(golden["F_x10"]), _t(golden["F_t10"]), _t(golden["F_y10"])
        assert torch.equal(orc.rdunet_forward(n10.state_dict(), x, t), y)
        wide = _zero_padded_network(n10, 16)
        assert float((orc.rdunet_forward(wide.state_dict(), x, t) - y).abs().max()) < 2e-6
        # the embedding leaves the caller's module alone
        assert n10.base_filters == 10 and n10.block_1_0.conv_0.weight.shape == (10, 20, 3, 3)


def test_oracle_rdunet_t_matches_reference_outputs(golden):
    torch.manual_seed(11)
    sd = b2.RDUNet_T(base_filters=16).state_dict()
    with torch.no_grad():
        for k in ("0", "1"):
            y = orc.rdunet_forward(sd, _t(golden["B_x"]), _t(golden[f"B_t{k}"]))
            assert torch.equal(y, _t(golden[f"B_y{k}"]))


def test_oracle_sampler_matches_reference_outputs(golden):
    torch.manual_seed(13)
    sd = b2.DiffusionModel(b2.RDUNet_T(base_filters=16), timesteps=4).state_dict()
    with torch.no_grad():
        out = orc.improved_sampling(sd, _t(golden["C_noisy"]), 4)
    assert torch.equal(out, _t(golden["C_out"]))
    fd = orc.forward_diffusion(_t(golden["C_clean"]), _t(golden["C_noisy"]), 3, 4)
    assert torch.equal(fd, _t(golden["C_fd3"]))


def test_oracle_sampler_closed_form():
    """x_{t-1} = x_t - (1-a_t) U1 + (1-a_{t-1}) U2 - y/T (SURVEY.md §8 a7) up to fp32 rounding."""
    g = torch.Generator().manual_seed(5)
    x, u1, u2, y = (torch.randn(2, 3, 8, 8, generator=g) for _ in range(4))
    T = 20
    for t in (20, 7, 1):
        got = orc.sampler_step(x, u1, u2, y, t, T)
        want = x - (1 - t / T) * u1 + (1 - (t - 1) / T) * u2 - y / T
        assert torch.allclose(got, want, atol=1e-5)
    # at t = T the first U-Net output has weight exactly 0
    assert torch.equal(orc.sampler_step(x, u1, u2, y, T, T), orc.sampler_step(x, 5 * u1, u2, y, T, T))


def test_flop_formula_matches_survey():
    assert abs(orc.conv_flops(32) / 1e9 - 96.26) < 0.01
    assert abs(orc.conv_flops(64) / 1e9 - 384.58) < 0.01
    assert abs(orc.conv_flops(128) / 1e9 - 1537.43) < 0.01


def test_init_weights_variants():
    conv = torch.nn.Conv2d(4, 4, 3)
    convt = torch.nn.ConvTranspose2d(4, 4, 2)
    before = convt.weight.clone()
    for kind in ("xavier", "he", "orthogonal"):
        fn = b2.init_weights(kind)
        torch.manual_seed(0)
        fn(conv)
        fn(convt)
        assert torch.equal(convt.weight, before)        # 'ConvTranspose2d' does not contain 'Conv2d'
    bn = torch.nn.BatchNorm2d(4)
    b2.init_weights()(bn)
    assert torch.all(bn.bias == 0)
