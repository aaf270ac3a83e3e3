"""``torch.ops.b200dn.*`` — the torch.library custom-op layer over the C ABI of libb200dn.so.

Two kinds of ops live here:

* **network-level ops** — ``b200dn::rdunet_forward`` and ``b200dn::improved_sampling``.  These are the product call
  path: ``RDUNet.forward`` / ``RDUNet_T.forward`` / ``DiffusionModel.improved_sampling`` dispatch through them, so the
  whole fused forward (1 ingest launch + 68 prepared tcgen05 launches) or the whole sampling loop is ONE opaque node for
  the dispatcher, with a fake (meta) implementation so that ``torch.compile``-d callers trace through it.  The op takes
  the id of a prebuilt launch plan (packed weights, workspaces, encoded tensor maps) registered by the module.
* **layer-level ops** — ``pack_weight``, ``conv_igemm``, ``conv_out_nchw``, ``conv_in``, ``sampler_step``: the
  functional per-layer surface; each forwards raw pointers to the matching ``b200dn_*`` entry point on the current
  CUDA stream (used by the layer-level parity tests and by callers that want a single fused layer).
"""
from __future__ import annotations

import itertools
import weakref
from typing import Optional

import torch

from . import _lib
from ._lib import IgemmArgs

__all__ = ["pack_weight", "conv_igemm", "conv_out_nchw", "conv_in", "sampler_step", "rdunet_forward",
           "improved_sampling", "lpips_forward", "register_plan"]

# ------------------------------------------------------------------------------ plan registry (network-level ops)
# Custom-op schemas carry tensors and scalars only, so the modules register their launch plans / sampler states here and
# pass the integer id.  Weak references: a plan dies with the module cache that owns it.
_PLAN_IDS = itertools.count(1)
_PLANS: "weakref.WeakValueDictionary[int, object]" = weakref.WeakValueDictionary()


def register_plan(obj) -> int:
    pid = next(_PLAN_IDS)
    _PLANS[pid] = obj
    return pid


def _lookup(pid: int):
    obj = _PLANS.get(pid)
    if obj is None:
        raise RuntimeError(f"b200dn: launch plan {pid} no longer exists (its module was moved, reloaded or freed)")
    return obj


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _cuda(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("b200dn ops take CUDA (sm_100) tensors only; there is no CPU fallback")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


@torch.library.custom_op("b200dn::pack_weight", mutates_args=())
def pack_weight(weight: torch.Tensor, prec: int, transposed: bool) -> torch.Tensor:
    """OIHW Conv2d (or IOHW ConvTranspose2d 2x2) fp32 weight -> packed tensor-core operand (int16 storage)."""
    _cuda(weight)
    w = weight.detach().to(torch.float32).contiguous()
    L = _lib.lib()
    if transposed:
        cin, cout, groups = w.shape[0], w.shape[1], 4
    else:
        cout, cin, groups = w.shape[0], w.shape[1], w.shape[2] * w.shape[3]
    packed = torch.empty(L.b200dn_packed_weight_bytes(cout, cin, groups, prec) // 2, dtype=torch.int16, device=w.device)
    with torch.cuda.device(w.device):
        if transposed:
            rc = L.b200dn_pack_convt_weight(w.data_ptr(), cin, cout, prec, packed.data_ptr(), _stream(w))
        else:
            rc = L.b200dn_pack_conv_weight(w.data_ptr(), cout, cin, w.shape[2], w.shape[3], prec, packed.data_ptr(),
                                           _stream(w))
    _lib.check(rc, "pack_weight")
    return packed


@pack_weight.register_fake
def _(weight, prec, transposed):
    L = _lib.lib()
    if transposed:
        cin, cout, groups = weight.shape[0], weight.shape[1], 4
    else:
        cout, cin, groups = weight.shape[0], weight.shape[1], weight.shape[2] * weight.shape[3]
    return weight.new_empty(L.b200dn_packed_weight_bytes(cout, cin, groups, prec) // 2, dtype=torch.int16)


def _fill_common(a: IgemmArgs, mode, prec, x_hi, x_lo, cin, cout, wpacked, bias, slope, block_n, max_ctas, m_tiles=0,
                 impl=0):
    B, H, W, ctot = x_hi.shape
    a.mode, a.prec = mode, prec
    a.B, a.H, a.W = B, H, W
    a.cin, a.cout = cin, cout
    a.in_[0], a.in_[1] = _ptr(x_hi), _ptr(x_lo)
    a.in_ctot = ctot
    a.wpacked, a.bias, a.slope = _ptr(wpacked), _ptr(bias), _ptr(slope)
    a.block_n, a.max_ctas, a.m_tiles, a.impl = block_n, max_ctas, m_tiles, impl


@torch.library.custom_op("b200dn::conv_igemm", mutates_args=("out_hi", "out_lo"))
def conv_igemm(x_hi: torch.Tensor, x_lo: Optional[torch.Tensor], wpacked: torch.Tensor, bias: torch.Tensor,
               slope: Optional[torch.Tensor], mode: int, prec: int, cin: int, cout: int,
               out_hi: torch.Tensor, out_lo: Optional[torch.Tensor], out_coff: int,
               res_hi: Optional[torch.Tensor], res_lo: Optional[torch.Tensor],
               block_n: int = 0, max_ctas: int = 0, m_tiles: int = 0, impl: int = 0) -> None:
    """conv (3x3 / 2x2-s2 / transposed 2x2-s2) + bias + PReLU (+ NHWC residual) into a channel slice of
    ``out_*`` ([B, Ho, Wo, ctot] int16 storage of bf16/fp16)."""
    _cuda(x_hi, x_lo, wpacked, bias, slope, out_hi, out_lo, res_hi, res_lo)
    a = IgemmArgs()
    _fill_common(a, mode, prec, x_hi, x_lo, cin, cout, wpacked, bias, slope, block_n, max_ctas, m_tiles, impl)
    a.out_kind = _lib.OUT_NHWC16
    a.out[0], a.out[1] = _ptr(out_hi), _ptr(out_lo)
    a.out_ctot, a.out_coff = out_hi.shape[-1], out_coff
    if res_hi is not None:
        a.res[0], a.res[1] = _ptr(res_hi), _ptr(res_lo)
        a.res_ctot = res_hi.shape[-1]
    with torch.cuda.device(x_hi.device):
        rc = _lib.lib().b200dn_igemm(a, _stream(x_hi))
    _lib.check(rc, "igemm")


@torch.library.custom_op("b200dn::conv_out_nchw", mutates_args=("out",))
def conv_out_nchw(x_hi: torch.Tensor, x_lo: Optional[torch.Tensor], wpacked: torch.Tensor, bias: torch.Tensor,
                  slope: Optional[torch.Tensor], prec: int, cin: int, cout: int,
                  residual: Optional[torch.Tensor], out: torch.Tensor, res_bmod: int = 0, impl: int = 0) -> None:
    """OutputBlock.conv_2 + PReLU + `+ inputs` with fp32 NCHW output (UNet/RDUNet_model.py:83-93,186)."""
    _cuda(x_hi, x_lo, wpacked, bias, slope, residual, out)
    a = IgemmArgs()
    _fill_common(a, _lib.MODE_CONV3X3, prec, x_hi, x_lo, cin, cout, wpacked, bias, slope, 0, 0, 0, impl)
    a.out_kind = _lib.OUT_NCHW32
    a.out_nchw, a.res_nchw, a.res_bmod = _ptr(out), _ptr(residual), res_bmod
    with torch.cuda.device(x_hi.device):
        rc = _lib.lib().b200dn_igemm(a, _stream(x_hi))
    _lib.check(rc, "igemm")


@torch.library.custom_op("b200dn::conv_in", mutates_args=("out_hi", "out_lo"))
def conv_in(x: torch.Tensor, t: Optional[torch.Tensor], weight: torch.Tensor, bias: torch.Tensor,
            slope: torch.Tensor, prec: int, batch: int, out_hi: torch.Tensor, out_lo: Optional[torch.Tensor]) -> None:
    """InputBlock.conv_1 + PReLU from fp32 NCHW (x[b % Bx]) (+ t plane [batch] per image) to NHWC planes."""
    _cuda(x, t, weight, bias, slope, out_hi, out_lo)
    Bx, _, H, W = x.shape
    with torch.cuda.device(x.device):
        rc = _lib.lib().b200dn_conv_in(x.data_ptr(), Bx, x.shape[1], _ptr(t), 1 if t is not None else 0, 0, 0, batch, H, W,
                                       weight.shape[0], weight.data_ptr(), bias.data_ptr(), slope.data_ptr(), prec,
                                       out_hi.data_ptr(), _ptr(out_lo), out_hi.shape[-1], None, _stream(x))
    _lib.check(rc, "conv_in")


@torch.library.custom_op("b200dn::sampler_step", mutates_args=())
def sampler_step(x: torch.Tensor, u1: torch.Tensor, u2: torch.Tensor, y: torch.Tensor,
                 one_m_at: float, at: float, one_m_ap: float, ap: float) -> torch.Tensor:
    """x - ((1-a_t) u1 + a_t y) + ((1-a_p) u2 + a_p y) in the reference's fp32 op order."""
    _cuda(x, u1, u2, y)
    x, u1, u2, y = (v.detach().to(torch.float32).contiguous() for v in (x, u1, u2, y))
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _lib.lib().b200dn_sampler_step(x.data_ptr(), u1.data_ptr(), u2.data_ptr(), y.data_ptr(), one_m_at, at,
                                            one_m_ap, ap, out.data_ptr(), x.numel(), _stream(x))
    _lib.check(rc, "sampler_step")
    return out


@sampler_step.register_fake
def _(x, u1, u2, y, one_m_at, at, one_m_ap, ap):
    return torch.empty_like(x)


# ------------------------------------------------------------------------------ network-level ops (the product path)
@torch.library.custom_op("b200dn::rdunet_forward", mutates_args=())
def rdunet_forward(x: torch.Tensor, t: Optional[torch.Tensor], plan_id: int) -> torch.Tensor:
    """RDUNet / RDUNet_T forward (UNet/RDUNet_model.py:157-186, diffusion_denoising/Unet/Unet_model.py:133-166) over a
    registered :class:`rdunet.ForwardPlan`: fp32 NCHW in, fresh fp32 NCHW out."""
    _cuda(x, t)
    plan = _lookup(plan_id)
    with torch.cuda.device(x.device):
        return plan.forward(x, t)


@rdunet_forward.register_fake
def _(x, t, plan_id):
    return torch.empty_like(x)


@torch.library.custom_op("b200dn::improved_sampling", mutates_args=())
def improved_sampling(noisy: torch.Tensor, state_id: int) -> torch.Tensor:
    """DiffusionModel.improved_sampling (diffusion_denoising/diffusion_RDUnet.py:38-50) over a registered sampler
    state (2B-batched forwards + fused update step, one CUDA graph)."""
    _cuda(noisy)
    st = _lookup(state_id)
    with torch.cuda.device(noisy.device):
        return st.sample(noisy)


@improved_sampling.register_fake
def _(noisy, state_id):
    return torch.empty_like(noisy)


@torch.library.custom_op("b200dn::lpips_forward", mutates_args=())
def lpips_forward(in0: torch.Tensor, in1: torch.Tensor, normalize: bool, plan_id: int) -> torch.Tensor:
    """lpips.LPIPS(net='alex')(in0, in1, normalize=normalize) (evaluate_Unet_diffusion/evaluate_model.py:46-71) over a
    registered :class:`perceptual.LpipsPlan`: two fp32 NCHW batches in, fresh fp32 [N, 1, 1, 1] out."""
    _cuda(in0, in1)
    plan = _lookup(plan_id)
    with torch.cuda.device(in0.device):
        return plan.forward(in0, in1, normalize)


@lpips_forward.register_fake
def _(in0, in1, normalize, plan_id):
    return in0.new_empty((in0.shape[0], 1, 1, 1))
