"""ORACLE (test infrastructure): pin the oracle to the REAL reference and emit golden vectors.

Runs only where /root/reference is mounted (the build container).  It imports the reference's own
``RDUNet`` (UNet/RDUNet_model.py), ``RDUNet_T`` (diffusion_denoising/Unet/Unet_model.py) and
``DiffusionModel`` (diffusion_denoising/diffusion_RDUnet.py) — with empty stub modules for the
plotting / loss packages those files import but the hot path never touches (matplotlib,
pytorch_msssim) — runs them on seeded inputs, checks oracle/rdunet_oracle.py against them, and writes
tests/golden/rdunet_golden.npz (reference outputs + state_dict digests).  The GPU box has no
/root/reference; tests there compare against the committed vectors.

Usage:  python -m oracle.pin_against_reference
"""
from __future__ import annotations

import hashlib
import sys
import types
from pathlib import Path

import numpy as np
import torch

REF = Path("/root/reference")
OUT = Path(__file__).resolve().parent.parent / "tests" / "golden" / "rdunet_golden.npz"


def sd_digest(sd) -> str:
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(str(tuple(v.shape)).encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def import_reference():
    if not REF.exists():
        raise SystemExit("/root/reference is not mounted here; golden vectors are generated in the build container")
    for name in ("matplotlib", "matplotlib.pyplot", "pytorch_msssim"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.path.insert(0, str(REF))
    from diffusion_denoising.Unet.Unet_model import RDUNet_T  # noqa: E402
    from diffusion_denoising.diffusion_RDUnet import DiffusionModel  # noqa: E402
    from UNet.RDUNet_model import RDUNet  # noqa: E402  (slow: builds a bf128 model at import)
    return RDUNet, RDUNet_T, DiffusionModel


def main() -> None:
    from oracle import rdunet_oracle as orc

    RDUNet, RDUNet_T, DiffusionModel = import_reference()
    torch.set_grad_enabled(False)
    torch.set_num_threads(orc.GOLDEN_THREADS)
    gold = {}

    # ---- case A: RDUNet(base_filters=16), 1x3x32x32 and 2x3x16x24
    torch.manual_seed(7)
    net = RDUNet(base_filters=16).eval()
    sd = net.state_dict()
    gold["A_digest"] = np.frombuffer(bytes.fromhex(sd_digest(sd)), dtype=np.uint8)
    g = torch.Generator().manual_seed(1234)
    xa = torch.rand(1, 3, 32, 32, generator=g) * 2 - 1
    xb = torch.rand(2, 3, 16, 24, generator=g) * 2 - 1
    ya, yb = net(xa), net(xb)
    for x, y in ((xa, ya), (xb, yb)):
        mine = orc.rdunet_forward(sd, x)
        assert torch.equal(mine, y), f"oracle != reference RDUNet: max {float((mine - y).abs().max())}"
    gold.update(A_x0=xa.numpy(), A_y0=ya.numpy(), A_x1=xb.numpy(), A_y1=yb.numpy())

    # ---- case B: RDUNet_T(base_filters=16), t scalar-broadcast and per-sample
    torch.manual_seed(11)
    net_t = RDUNet_T(base_filters=16).eval()
    sd_t = net_t.state_dict()
    gold["B_digest"] = np.frombuffer(bytes.fromhex(sd_digest(sd_t)), dtype=np.uint8)
    xt = torch.rand(2, 3, 16, 16, generator=g) * 2 - 1
    t0 = torch.tensor([0.35]).view(1, 1, 1, 1)
    t1 = torch.tensor([0.25, 0.9]).view(2, 1, 1, 1)
    y0, y1 = net_t(xt, t0), net_t(xt, t1)
    assert torch.equal(orc.rdunet_forward(sd_t, xt, t0), y0)
    assert torch.equal(orc.rdunet_forward(sd_t, xt, t1), y1)
    gold.update(B_x=xt.numpy(), B_t0=t0.numpy(), B_y0=y0.numpy(), B_t1=t1.numpy(), B_y1=y1.numpy())

    # ---- case C: DiffusionModel(RDUNet_T(16), timesteps=4).improved_sampling / forward_diffusion
    torch.manual_seed(13)
    dm = DiffusionModel(RDUNet_T(base_filters=16), timesteps=4).eval()
    sd_d = dm.state_dict()
    gold["C_digest"] = np.frombuffer(bytes.fromhex(sd_digest(sd_d)), dtype=np.uint8)
    noisy = torch.rand(2, 3, 16, 16, generator=g) * 2 - 1
    clean = torch.rand(2, 3, 16, 16, generator=g) * 2 - 1
    out = dm.improved_sampling(noisy)
    mine = orc.improved_sampling(sd_d, noisy, 4)
    assert torch.equal(mine, out), f"oracle sampler != reference: {float((mine - out).abs().max())}"
    fd = dm.forward_diffusion(clean, noisy, 3)
    assert torch.equal(orc.forward_diffusion(clean, noisy, 3, 4), fd)
    gold.update(C_noisy=noisy.numpy(), C_clean=clean.numpy(), C_out=out.numpy(), C_fd3=fd.numpy())

    # ---- case D: evaluation widths, digests only (tensors would be too large to commit):
    #      RDUNet(128) seed 7 and DiffusionModel(RDUNet_T(32)) seed 7 on one 256x256... output statistics
    torch.manual_seed(7)
    big_t = DiffusionModel(RDUNet_T(base_filters=32), timesteps=20).eval()
    gold["D_digest_T32"] = np.frombuffer(bytes.fromhex(sd_digest(big_t.state_dict())), dtype=np.uint8)
    x64 = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    y64 = big_t.unet(x64, torch.tensor([0.5]).view(1, 1, 1, 1))
    assert torch.equal(orc.rdunet_forward(big_t.state_dict(), x64, torch.tensor([0.5]).view(1, 1, 1, 1), "unet."), y64)
    gold.update(D_x=x64.numpy(), D_y=y64.numpy())

    # ---- case E: grayscale RDUNet(channels=1, base_filters=16) — the reference ctor takes `channels` for both ends
    #      (UNet/RDUNet_model.py:117-155); evaluate_model.calculate_ssim(use_rgb=False) is its metric path
    torch.manual_seed(17)
    gray = RDUNet(channels=1, base_filters=16).eval()
    sd_g = gray.state_dict()
    gold["E_digest"] = np.frombuffer(bytes.fromhex(sd_digest(sd_g)), dtype=np.uint8)
    xg = torch.rand(2, 1, 16, 24, generator=g) * 2 - 1
    yg = gray(xg)
    assert torch.equal(orc.rdunet_forward(sd_g, xg), yg)
    gold.update(E_x=xg.numpy(), E_y=yg.numpy())

    # ---- case F: widths off the kernels' channel tiling (the reference ctor takes any base_filters, growth = F // 2):
    #      RDUNet(base_filters=24) and RDUNet_T(base_filters=10)
    torch.manual_seed(19)
    n24 = RDUNet(base_filters=24).eval()
    gold["F_digest24"] = np.frombuffer(bytes.fromhex(sd_digest(n24.state_dict())), dtype=np.uint8)
    x24 = torch.rand(1, 3, 16, 24, generator=g) * 2 - 1
    y24 = n24(x24)
    assert torch.equal(orc.rdunet_forward(n24.state_dict(), x24), y24)
    torch.manual_seed(23)
    n10 = RDUNet_T(base_filters=10).eval()
    gold["F_digest10"] = np.frombuffer(bytes.fromhex(sd_digest(n10.state_dict())), dtype=np.uint8)
    x10 = torch.rand(2, 3, 16, 16, generator=g) * 2 - 1
    t10 = torch.tensor([0.15, 0.7]).view(2, 1, 1, 1)
    y10 = n10(x10, t10)
    assert torch.equal(orc.rdunet_forward(n10.state_dict(), x10, t10), y10)
    gold.update(F_x24=x24.numpy(), F_y24=y24.numpy(), F_x10=x10.numpy(), F_t10=t10.numpy(), F_y10=y10.numpy())

    # FLOP count of the oracle's formula vs the survey's hook measurement (SURVEY.md §8 a6)
    assert abs(orc.conv_flops(32) / 1e9 - 96.26) < 0.01, orc.conv_flops(32) / 1e9
    assert abs(orc.conv_flops(128) / 1e9 - 1537.43) < 0.01, orc.conv_flops(128) / 1e9
    assert abs(orc.conv_flops(32, in_channels=4) / 1e9 - 96.30) < 0.01

    OUT.parent.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(OUT, **gold)
    print(f"oracle == reference on all cases (bit-exact); wrote {OUT} ({OUT.stat().st_size / 1024:.1f} KiB)")


if __name__ == "__main__":
    main()
