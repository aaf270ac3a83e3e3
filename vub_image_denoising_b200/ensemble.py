"""x8 geometric self-ensemble: a better output from a fixed denoising checkpoint without retraining.

The image is denoised in its 8 flips / rotations (the dihedral group of the square), each output is transformed back,
and the 8 results are averaged (include/b200dn.h gives the transforms and the batch layout):

    out = (((y_0 + y_1) + y_2) + ... + y_7) * 0.125    in fp32, adds in k order, y_k = T_k^-1(f(T_k(x)))

The fixed add order makes the result bit-reproducible.  ``b200dn_dihedral_expand`` writes the 8 transforms as two
groups — the even k at H x W, the odd k at W x H — and each group goes through ONE call of the wrapped model at batch
4B (a square image: one call at batch 8B), so the network runs at a batch size where it is cheaper per image than at B.
``b200dn_dihedral_reduce`` transforms the outputs back and averages them.
"""
from __future__ import annotations

import contextlib

import torch

from . import ops
from .diffusion import DiffusionModel
from .rdunet import RDUNet, RDUNet_T

__all__ = ["self_ensemble"]


def self_ensemble(model, x: torch.Tensor) -> torch.Tensor:
    """The x8 self-ensemble of ``model(x)`` for an :class:`RDUNet`, or of ``model.improved_sampling(x)`` for a
    :class:`DiffusionModel` around an :class:`RDUNet_T`.

    Inputs are checked as the wrapped call checks them (CUDA, channel count, H and W divisible by 8, inference only)
    and raise the same ``RuntimeError``.  Returns a fresh fp32 ``[B, C, H, W]`` tensor; ``x`` is never written.  The
    work is enqueued on the current stream without a host synchronisation (so the call can be captured in a CUDA graph),
    except for what the wrapped call itself does: ``improved_sampling``'s fp16 saturation check reads one flag from
    the device.  Plans, sampler states and precision are the model's own."""
    if isinstance(model, RDUNet):
        net, run, checking = model, model, contextlib.nullcontext()
    elif isinstance(model, DiffusionModel) and isinstance(model.unet, RDUNet_T):
        net, run, checking = model.unet, model.improved_sampling, torch.no_grad()   # improved_sampling is no_grad
    else:
        raise TypeError(f"self_ensemble takes an RDUNet or a DiffusionModel around an RDUNet_T, got {type(model).__name__}")
    with checking:
        x = net._check_input(x)
    B, C, H, W = x.shape
    n = 4 * x.numel()
    buf = ops.dihedral_expand(x)
    if H == W:
        y = run(buf.view(8 * B, C, H, W))
        even, odd = y[:4 * B], y[4 * B:]
    else:
        even = run(buf[:n].view(4 * B, C, H, W))
        odd = run(buf[n:].view(4 * B, C, W, H))
    return ops.dihedral_reduce(even, odd)
