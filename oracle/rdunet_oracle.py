"""ORACLE (test infrastructure, not product): CPU restatement of the reference's RDUNet / RDUNet_T
forward and of the DiffusionModel sampler, written as pure functions over a ``state_dict``.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs
may import this package; nothing under ``vub_image_denoising_b200/`` does.

Pinned: ``oracle/pin_against_reference.py`` runs THIS file against the reference's own ``nn.Module``s
imported from /root/reference (same seed, same inputs) and stores the reference outputs as golden
vectors under tests/golden/; ``tests/test_oracle_golden.py`` re-checks the oracle against them on every
run (no access to /root/reference needed).

What each function follows (reference file:line):
  dense_block        UNet/RDUNet_model.py:95-115          (twin: diffusion_denoising/Unet/Unet_model.py:69-89)
  down / up          UNet/RDUNet_model.py:49-69
  io_block           UNet/RDUNet_model.py:71-93
  rdunet_forward     UNet/RDUNet_model.py:157-186, diffusion_denoising/Unet/Unet_model.py:133-166
  improved_sampling  diffusion_denoising/diffusion_RDUnet.py:38-50
  forward_diffusion  diffusion_denoising/diffusion_RDUnet.py:33-36
  direct_sampling    diffusion_denoising/diffusion_RDUnet_direct.py:198-201
"""
from __future__ import annotations

from typing import Dict, Mapping, Optional

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
SD = Mapping[str, Tensor]

# Intra-op CPU threads of the run that produced tests/golden/rdunet_golden.npz.  oneDNN splits some convolution
# reductions by thread count, so the stored reference outputs are reproduced bit for bit only at this count.
GOLDEN_THREADS = 8


def _p(sd: SD, name: str, like: Tensor) -> Tensor:
    return sd[name].to(dtype=like.dtype, device=like.device)


def _conv_act(sd: SD, x: Tensor, conv: str, actv: str, **kw) -> Tensor:
    y = F.conv2d(x, _p(sd, conv + ".weight", x), _p(sd, conv + ".bias", x), **kw)
    return F.prelu(y, _p(sd, actv + ".weight", x))


def io_block(sd: SD, pre: str, x: Tensor) -> Tensor:
    x = _conv_act(sd, x, f"{pre}.conv_1", f"{pre}.actv_1", padding=1)
    return _conv_act(sd, x, f"{pre}.conv_2", f"{pre}.actv_2", padding=1)


def dense_block(sd: SD, pre: str, x: Tensor) -> Tensor:
    feats = x
    for k in range(3):
        grown = _conv_act(sd, feats, f"{pre}.conv_{k}", f"{pre}.actv_{k}", padding=1)
        feats = torch.cat([feats, grown], dim=1)          # order [x, o0, o1, o2]
    return _conv_act(sd, feats, f"{pre}.conv_3", f"{pre}.actv_3", padding=1) + x


def down(sd: SD, pre: str, x: Tensor) -> Tensor:
    return _conv_act(sd, x, f"{pre}.conv", f"{pre}.actv", stride=2)


def up(sd: SD, pre: str, deep: Tensor, skip: Tensor) -> Tensor:
    u = F.conv_transpose2d(deep, _p(sd, f"{pre}.conv_t.weight", deep), _p(sd, f"{pre}.conv_t.bias", deep), stride=2)
    u = F.prelu(u, _p(sd, f"{pre}.actv_t.weight", deep))
    return _conv_act(sd, torch.cat([skip, u], dim=1), f"{pre}.conv", f"{pre}.actv", padding=1)


def rdunet_forward(sd: SD, inputs: Tensor, t: Optional[Tensor] = None, prefix: str = "") -> Tensor:
    """RDUNet (t is None) or RDUNet_T (t broadcastable to [B,1,H,W]) forward."""
    x = inputs
    if t is not None:
        x = torch.cat((inputs, t.to(inputs.dtype).expand(inputs.size(0), 1, inputs.size(2), inputs.size(3))), dim=1)
    n = lambda s: prefix + s  # noqa: E731
    skips: Dict[int, Tensor] = {}
    h = io_block(sd, n("input_block"), x)
    for lvl in range(4):
        h = dense_block(sd, n(f"block_{lvl}_0"), h)
        h = dense_block(sd, n(f"block_{lvl}_1"), h)
        if lvl < 3:
            skips[lvl] = h
            h = down(sd, n(f"down_{lvl}"), h)
    for lvl in (2, 1, 0):
        h = up(sd, n(f"up_{lvl}"), h, skips[lvl])
        h = dense_block(sd, n(f"block_{lvl}_2"), h)
        h = dense_block(sd, n(f"block_{lvl}_3"), h)
    return io_block(sd, n("output_block"), h) + inputs


def forward_diffusion(clean: Tensor, noisy: Tensor, t, timesteps: int) -> Tensor:
    alpha = t / timesteps
    return alpha * noisy + (1 - alpha) * clean


def improved_sampling(sd: SD, noisy: Tensor, timesteps: int = 20, prefix: str = "unet.") -> Tensor:
    x_t = noisy
    for step in range(timesteps, 0, -1):
        a_t, a_p = step / timesteps, (step - 1) / timesteps
        # the reference builds float32 [1,1,1,1] tensors from the python quotients
        tt = torch.tensor([a_t], dtype=torch.float32).view(1, 1, 1, 1)
        tp = torch.tensor([a_p], dtype=torch.float32).view(1, 1, 1, 1)
        u_t = rdunet_forward(sd, x_t, tt, prefix)
        x_tilde = (1 - a_t) * u_t + a_t * noisy
        u_p = rdunet_forward(sd, x_t, tp, prefix)
        x_tilde_prev = (1 - a_p) * u_p + a_p * noisy
        x_t = x_t - x_tilde + x_tilde_prev
    return x_t


def direct_sampling(sd: SD, noisy: Tensor, prefix: str = "unet.") -> Tensor:
    return rdunet_forward(sd, noisy, torch.ones(1, 1, 1, 1), prefix)


def sampler_step(x: Tensor, u1: Tensor, u2: Tensor, y: Tensor, t: int, timesteps: int) -> Tensor:
    """One update of the loop above (diffusion_RDUnet.py:45,48,49) on given U-Net outputs."""
    a_t, a_p = t / timesteps, (t - 1) / timesteps
    return x - ((1 - a_t) * u1 + a_t * y) + ((1 - a_p) * u2 + a_p * y)


def conv_flops(base_filters: int, in_channels: int = 3, out_channels: int = 3, hw: int = 256 * 256) -> int:
    """2*MAC of all 69 convolutions for one hw-pixel image (SURVEY.md §8 a6: F=32 -> 96.26 G, F=128 -> 1537.43 G)."""
    f = [base_filters << l for l in range(4)]
    px = [hw >> (2 * l) for l in range(4)]
    total = 9 * px[0] * (in_channels * f[0] + f[0] * f[0])                       # input block
    total += 9 * px[0] * (f[0] * f[0] + f[0] * out_channels)                     # output block

    def block(c, p):
        g = c // 2
        return 9 * p * (c * g + (c + g) * g + (c + 2 * g) * g + (c + 3 * g) * c)

    total += 4 * block(f[0], px[0]) + 4 * block(f[1], px[1]) + 4 * block(f[2], px[2]) + 2 * block(f[3], px[3])
    for l in range(3):
        total += 4 * f[l] * (2 * f[l]) * px[l + 1]                               # down: K = 4C, N = 2C, M = px/4
        total += (2 * f[l]) * (4 * 2 * f[l]) * px[l + 1]                         # convT: K = 2C, N = 4*2C
        total += 9 * px[l] * (3 * f[l]) * f[l]                                   # up conv: K = 9*3C, N = C
    return 2 * total
