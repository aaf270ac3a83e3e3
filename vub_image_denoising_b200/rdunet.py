"""Drop-in RDUNet / RDUNet_T modules whose forward runs on the hand-written sm_100a kernels.

Reference interface mirrored here (pierregab/VUB_Image_denoising):
  * ``RDUNet(channels=3, base_filters=64).forward(inputs)``            UNet/RDUNet_model.py:117-186
  * ``RDUNet_T(channels=4, base_filters=64).forward(inputs, t)``       diffusion_denoising/Unet/Unet_model.py:92-166
  * ``init_weights(init_type='xavier')``                               UNet/RDUNet_model.py:30-47
  * the 207-tensor ``state_dict`` (names, shapes, fp32, registration order) — so reference
    checkpoints load unchanged and ``torch.manual_seed(s); RDUNet(...)`` draws the same init.

The parameter tree is made of real ``nn.Conv2d`` / ``nn.ConvTranspose2d`` / ``nn.PReLU`` holders whose
``forward`` is never called.  ``forward`` builds (and caches) a :class:`ForwardPlan`: NHWC 16-bit
activation buffers laid out so that every ``torch.cat`` of the reference is a channel slice, packed
tensor-core weights, and the list of C-ABI launches (``b200dn_conv_in`` + 68 ``b200dn_igemm``).
Inference only; there is no CPU or PyTorch fallback — a CPU tensor raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict
from typing import Optional

import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import DenseBlockArgs, IgemmArgs

__all__ = ["RDUNet", "RDUNet_T", "init_weights", "ForwardPlan", "DEFAULT_PREC"]

DEFAULT_PREC = os.environ.get("B200DN_PREC", "bf16")
_USE_GRAPH = os.environ.get("B200DN_GRAPH", "1") != "0"   # replay nn.Module forwards as one CUDA graph from the 2nd call on
# 32-channel DenoisingBlocks (level 0 of base_filters = 32) run as ONE fused kernel instead of four launches
_FUSE_DENSE = os.environ.get("B200DN_FUSED_DENSE", "1") != "0"
MODE_DENSE_BLOCK = 4     # layer_info "mode" of a fused block (the per-layer modes are _lib.MODE_*)
# wider DenoisingBlocks (the single-plane modes): conv_0..conv_3 as ONE persistent launch whose tiles wait on the tiles
# they read instead of on a launch boundary (conv3x3_chain_kernel, csrc/conv3x3_slab_sm100.cu); bit-equal to the four launches it replaces
# B200DN_CHAIN: 0 = never, 1 = where a layer has at least two rounds of tiles per SM pair (default), 2 = wherever it applies
_CHAIN_DENSE = int(os.environ.get("B200DN_CHAIN", "1"))
# B200DN_DENSE_CONST=0: fused blocks stage bias / slopes in shared memory instead of taking them as launch parameters
_DENSE_CONST = int(os.environ.get("B200DN_DENSE_CONST", "1"))
MODE_CONV_CHAIN = 5      # layer_info "mode" of such a chain


class _Chain:
    """The four b200dn_igemm_args of a DenoisingBlock, to be prepared as one chain launch (or one by one)."""

    __slots__ = ("layers", "infos")

    def __init__(self, layers, infos):
        self.layers, self.infos = layers, infos


# --------------------------------------------------------------------------- init
@torch.no_grad()
def init_weights(init_type: str = "xavier"):
    """Return an ``nn.Module.apply`` callback (reference: UNet/RDUNet_model.py:30-47).

    Modules whose class name contains ``Conv2d`` get Xavier-normal / Kaiming-normal / orthogonal
    weights; ``ConvTranspose2d`` does not contain that substring, so — as in the reference —
    transposed convolutions and all biases keep PyTorch's defaults.
    """
    fill = {"xavier": nn.init.xavier_normal_, "he": nn.init.kaiming_normal_}.get(init_type, nn.init.orthogonal_)

    def visit(module: nn.Module) -> None:
        kind = type(module).__name__
        if "Conv2d" in kind:
            fill(module.weight)
        elif "BatchNorm" in kind:
            nn.init.normal_(module.weight, 1.0, 0.01)
            nn.init.zeros_(module.bias)

    return visit


# --------------------------------------------------------------------------- parameter tree
class _Params(nn.Module):
    """Ordered bag of parameter-holding submodules (never executed)."""

    def __init__(self, members: "OrderedDict[str, nn.Module]"):
        super().__init__()
        for name, mod in members.items():
            self.add_module(name, mod)

    def forward(self, *_a, **_k):  # pragma: no cover - guard
        raise RuntimeError("parameter holder: the fused B200 forward of the owning network must be used")


def _conv3(cin: int, cout: int) -> nn.Conv2d:
    return nn.Conv2d(cin, cout, 3, padding=1)


def _io_block(cin: int, cmid: int, cout: int) -> _Params:
    # registration order conv_1, conv_2, actv_1, actv_2 (UNet/RDUNet_model.py:71-93)
    return _Params(OrderedDict(conv_1=_conv3(cin, cmid), conv_2=_conv3(cmid, cout),
                               actv_1=nn.PReLU(cmid), actv_2=nn.PReLU(cout)))


def _dense_block(c: int) -> _Params:
    # conv_0..3 then actv_0..3 (UNet/RDUNet_model.py:95-105); growth g = c // 2
    g = c // 2
    members: "OrderedDict[str, nn.Module]" = OrderedDict()
    for k in range(3):
        members[f"conv_{k}"] = _conv3(c + k * g, g)
    members["conv_3"] = _conv3(c + 3 * g, c)
    for k in range(3):
        members[f"actv_{k}"] = nn.PReLU(g)
    members["actv_3"] = nn.PReLU(c)
    return _Params(members)


def _down_block(c: int) -> _Params:
    return _Params(OrderedDict(conv=nn.Conv2d(c, 2 * c, kernel_size=2, stride=2), actv=nn.PReLU(2 * c)))


def _up_block(c_deep: int, c_skip: int, c_out: int) -> _Params:
    # conv, conv_t, actv, actv_t (UNet/RDUNet_model.py:58-64)
    return _Params(OrderedDict(conv=_conv3(c_deep + c_skip, c_out),
                               conv_t=nn.ConvTranspose2d(c_deep, c_deep, 2, stride=2),
                               actv=nn.PReLU(c_out), actv_t=nn.PReLU(c_deep)))


class _RDUNetBase(nn.Module):
    """Shared wiring of RDUNet and RDUNet_T (they differ in the input conv's Cin and the t plane)."""

    _in_channels: int   # channels seen by input_block.conv_1
    _img_channels = 3   # channels of the image tensor handed to forward()

    def _build(self, in_channels: int, out_channels: int, base_filters: int, init: bool = True) -> None:
        f = [base_filters * (1 << l) for l in range(4)]
        self.base_filters = base_filters
        self._in_channels = in_channels
        self._out_channels = out_channels
        self.input_block = _io_block(in_channels, f[0], f[0])
        self.block_0_0 = _dense_block(f[0])
        self.block_0_1 = _dense_block(f[0])
        self.down_0 = _down_block(f[0])
        self.block_1_0 = _dense_block(f[1])
        self.block_1_1 = _dense_block(f[1])
        self.down_1 = _down_block(f[1])
        self.block_2_0 = _dense_block(f[2])
        self.block_2_1 = _dense_block(f[2])
        self.down_2 = _down_block(f[2])
        self.block_3_0 = _dense_block(f[3])
        self.block_3_1 = _dense_block(f[3])
        self.up_2 = _up_block(f[3], f[2], f[2])
        self.block_2_2 = _dense_block(f[2])
        self.block_2_3 = _dense_block(f[2])
        self.up_1 = _up_block(f[2], f[1], f[1])
        self.block_1_2 = _dense_block(f[1])
        self.block_1_3 = _dense_block(f[1])
        self.up_0 = _up_block(f[1], f[0], f[0])
        self.block_0_2 = _dense_block(f[0])
        self.block_0_3 = _dense_block(f[0])
        self.output_block = _io_block(f[0], f[0], out_channels)
        if init:
            self.apply(init_weights())
        # private caches (not parameters / buffers -> invisible to state_dict)
        self._plans: dict = {}
        self.precision = DEFAULT_PREC

    # ---- nn.Module plumbing that must drop caches
    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._plans = {}
        return out

    def __deepcopy__(self, memo):
        import copy
        plans, self._plans = self._plans, {}      # plans hold raw device pointers: never copy them
        try:
            new = self.__class__.__new__(self.__class__)
            memo[id(self)] = new
            for key, val in self.__dict__.items():
                new.__dict__[key] = copy.deepcopy(val, memo)
        finally:
            self._plans = plans
        return new

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_plans"] = {}
        return state

    def invalidate_plans(self) -> None:
        """Drop every cached ForwardPlan (packed weights, bias / slope snapshots, captured graphs).  Needed only after
        in-place parameter writes that bypass autograd's version counter (``p.data.copy_()``, ``p.data.mul_()``);
        ``load_state_dict``, ``.to()`` and ordinary in-place ops are detected automatically."""
        self._plans = {}

    # ---- helpers
    def _param_signature(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def plan(self, batch: int, height: int, width: int, precision: Optional[str] = None) -> "ForwardPlan":
        prec = precision or self.precision
        key = (batch, height, width, prec)
        plan = self._plans.get(key)
        sig = self._param_signature()
        if plan is None or plan.signature != sig:
            # drop stale plans (parameters were moved / reloaded); keep at most a few shapes alive
            if plan is None and len(self._plans) >= 4:
                self._plans.pop(next(iter(self._plans)))
            plan = ForwardPlan(self, batch, height, width, prec)
            plan.signature = sig
            self._plans[key] = plan
        return plan

    def _check_input(self, inputs: torch.Tensor) -> torch.Tensor:
        if not isinstance(inputs, torch.Tensor) or inputs.dim() != 4:
            raise RuntimeError("expected a 4-D [B, C, H, W] tensor")
        if not inputs.is_cuda:
            raise RuntimeError("vub_image_denoising_b200 runs on CUDA (sm_100) tensors only; there is no CPU fallback")
        if inputs.size(1) != self._img_channels:
            raise RuntimeError(f"expected input with {self._img_channels} channels, got {inputs.size(1)}")
        if inputs.size(2) % 8 or inputs.size(3) % 8:
            raise RuntimeError(f"spatial size {tuple(inputs.shape[2:])} must be divisible by 8 "
                               "(three stride-2 levels; the reference fails in torch.cat otherwise)")
        if torch.is_grad_enabled() and (inputs.requires_grad or self.training):
            raise RuntimeError("the B200 path is inference-only: use model.eval() and torch.no_grad() "
                               "(training / autograd through the fused kernels is out of scope)")
        p0 = next(self.parameters())
        if p0.device != inputs.device:
            raise RuntimeError(f"module parameters are on {p0.device}, input is on {inputs.device}")
        return inputs.detach().to(torch.float32).contiguous()


class RDUNet(_RDUNetBase):
    """Residual-dense U-Net, `channels` in and out: 3 (RGB) or 1 (grayscale) (reference: UNet/RDUNet_model.py:117-186)."""

    def __init__(self, channels: int = 3, base_filters: int = 64):
        super().__init__()
        self._img_channels = channels
        self._build(channels, channels, base_filters)

    def forward(self, inputs: torch.Tensor) -> torch.Tensor:
        x = self._check_input(inputs)
        plan = self.plan(x.size(0), x.size(2), x.size(3))
        return torch.ops.b200dn.rdunet_forward(x, None, plan.plan_id)


class RDUNet_T(_RDUNetBase):
    """RDUNet with a broadcast timestep plane as 4th input channel
    (reference: diffusion_denoising/Unet/Unet_model.py:92-166)."""

    def __init__(self, channels: int = 4, base_filters: int = 64):
        super().__init__()
        self._img_channels = channels - 1
        self._build(channels, 3, base_filters)

    def forward(self, inputs: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        x = self._check_input(inputs)
        if not isinstance(t, torch.Tensor):
            t = torch.tensor(float(t), device=x.device)
        t = t.detach().to(device=x.device, dtype=torch.float32)
        # same broadcast as `t.expand(B, 1, H, W)` at Unet_model.py:135 (raises on incompatible shapes)
        t.expand(x.size(0), 1, x.size(2), x.size(3))
        plan = self.plan(x.size(0), x.size(2), x.size(3))
        return torch.ops.b200dn.rdunet_forward(x, t, plan.plan_id)


# --------------------------------------------------------------------------- widths the kernels do not tile
def _copy_blocks(dst: torch.Tensor, src: torch.Tensor, out_segs, in_segs, transposed: bool = False) -> None:
    """dst[physical] = src[logical] block by block; segs are [(logical length, physical length), ...] along the
    output / input channel axes (Conv2d weight [out, in, kh, kw]; ConvTranspose2d weight [in, out, kh, kw])."""
    if transposed:
        out_segs, in_segs = in_segs, out_segs      # dim 0 is the input axis
    o_l = o_p = 0
    for ol, op in out_segs:
        i_l = i_p = 0
        for il, ip in in_segs:
            dst[o_p:o_p + ol, i_p:i_p + il] = src[o_l:o_l + ol, i_l:i_l + il]
            i_l, i_p = i_l + il, i_p + ip
        o_l, o_p = o_l + ol, o_p + op


def _copy_vec(dst: torch.Tensor, src: torch.Tensor, segs) -> None:
    l = p = 0
    for sl, sp in segs:
        dst[p:p + sl] = src[l:l + sl]
        l, p = l + sl, p + sp


@torch.no_grad()
def _zero_padded_network(net: "_RDUNetBase", Fp: int) -> "_RDUNetBase":
    """The same function as `net`, embedded in a network of base_filters Fp > F whose extra channels are exactly zero.

    The reference ctor takes any `base_filters` (UNet/RDUNet_model.py:117-155; growth = filters // 2); the kernels tile
    channels in groups of 8, i.e. want F % 16 == 0.  Every logical channel segment ([x | o0 | o1 | o2] of a
    DenoisingBlock, [skip | upsampled] of an UpsampleBlock) keeps its place at the FRONT of the wider physical segment;
    the padded rows / columns of every weight and the padded biases are 0, so a padded channel is PReLU(0) = 0 in
    every layer, contributes nothing downstream and the residual adds 0 + 0.  Used only while a plan is built."""
    F = net.base_filters
    dev = next(net.parameters()).device
    with torch.device(dev):
        wide = net.__class__.__new__(net.__class__)
        nn.Module.__init__(wide)
        wide._img_channels = net._img_channels
        wide._build(net._in_channels, net._out_channels, Fp, init=False)
    for p in wide.parameters():
        p.zero_()

    def conv(dst, src, out_segs, in_segs, transposed=False):
        _copy_blocks(dst.weight, src.weight.to(torch.float32), out_segs, in_segs, transposed)
        _copy_vec(dst.bias, src.bias.to(torch.float32), out_segs)

    def actv(dst, src, segs):
        _copy_vec(dst.weight, src.weight.to(torch.float32), segs)

    cin, cout = net._in_channels, net._out_channels
    f0 = [(F, Fp)]
    conv(wide.input_block.conv_1, net.input_block.conv_1, f0, [(cin, cin)])
    conv(wide.input_block.conv_2, net.input_block.conv_2, f0, f0)
    actv(wide.input_block.actv_1, net.input_block.actv_1, f0)
    actv(wide.input_block.actv_2, net.input_block.actv_2, f0)
    conv(wide.output_block.conv_1, net.output_block.conv_1, f0, f0)
    conv(wide.output_block.conv_2, net.output_block.conv_2, [(cout, cout)], f0)
    actv(wide.output_block.actv_1, net.output_block.actv_1, f0)
    actv(wide.output_block.actv_2, net.output_block.actv_2, [(cout, cout)])
    for l in range(4):
        c, cp = F << l, Fp << l
        x, o = [(c, cp)], [(c // 2, cp // 2)]
        for j in range(4):
            name = f"block_{l}_{j}"
            if not hasattr(net, name):
                continue
            src, dst = getattr(net, name), getattr(wide, name)
            for k in range(4):
                out = o if k < 3 else x
                conv(getattr(dst, f"conv_{k}"), getattr(src, f"conv_{k}"), out, x + o * k)
                actv(getattr(dst, f"actv_{k}"), getattr(src, f"actv_{k}"), out)
        if l < 3:
            deep = [(2 * c, 2 * cp)]
            conv(getattr(wide, f"down_{l}").conv, getattr(net, f"down_{l}").conv, deep, x)
            actv(getattr(wide, f"down_{l}").actv, getattr(net, f"down_{l}").actv, deep)
            up_s, up_d = getattr(net, f"up_{l}"), getattr(wide, f"up_{l}")
            conv(up_d.conv_t, up_s.conv_t, deep, deep, transposed=True)
            actv(up_d.actv_t, up_s.actv_t, deep)
            conv(up_d.conv, up_s.conv, x, x + deep)        # torch.cat([skip, upsampled]) (RDUNet_model.py:69)
            actv(up_d.actv, up_s.actv, x)
    return wide.eval()


# --------------------------------------------------------------------------- the launch plan
class _Act:
    """An NHWC 16-bit activation buffer: one (hi) or two (hi, lo) planes of [B, H, W, ctot]."""

    __slots__ = ("hi", "lo", "ctot", "H", "W")

    def __init__(self, B, H, W, ctot, two, device):
        self.hi = torch.empty((B, H, W, ctot), dtype=torch.int16, device=device)
        self.lo = torch.empty((B, H, W, ctot), dtype=torch.int16, device=device) if two else None
        self.ctot, self.H, self.W = ctot, H, W

    def ptrs(self):
        return self.hi.data_ptr(), (self.lo.data_ptr() if self.lo is not None else None)


class ForwardPlan:
    """Buffers + packed weights + the ordered C-ABI launch list of one (B, H, W, precision) forward.

    Buffer plan per level l (C = F*2^l channels, g = C/2): two dense buffers ``Da, Db`` of 2.5*C channels
    (``[x | o0 | o1 | o2]`` — the reference's three torch.cat per DenoisingBlock, RDUNet_model.py:107-113)
    that ping-pong between consecutive blocks, and for l < 3 a ``K`` buffer of 3*C channels holding
    ``[skip | upsampled]`` (the torch.cat of UpsampleBlock.forward, RDUNet_model.py:69): the encoder's last
    block writes ``K[0:C)``, the transposed conv scatters into ``K[C:3C)``.
    """

    def __init__(self, net: _RDUNetBase, B: int, H: int, W: int, precision: str):
        if precision not in _lib.PREC_NAMES:
            raise RuntimeError(f"unknown precision {precision!r}; choose from {sorted(_lib.PREC_NAMES)}")
        F = net.base_filters
        if F < 2:
            raise RuntimeError(f"base_filters={F}: a DenoisingBlock needs filters // 2 >= 1 inner channels")
        if net._img_channels not in (1, 3) or net._out_channels != net._img_channels:
            raise RuntimeError("the B200 path implements the reference's RGB (3-channel) and grayscale (1-channel) "
                               f"networks; got channels={net._img_channels} in / {net._out_channels} out")
        self.lib = _lib.lib()
        self.prec = _lib.PREC_NAMES[precision]
        self.precision = precision
        self.device = next(net.parameters()).device
        self.logical_filters = F
        if F % 16:      # widths the kernels do not tile run zero-padded to the next multiple of 16 (exact, see above)
            F = -(-F // 16) * 16
            net = _zero_padded_network(net, F)
        self.B, self.H, self.W, self.F = B, H, W, F
        self.two = self.prec in _lib.TWO_PLANE_PRECS
        self.with_t = net._in_channels == net._img_channels + 1
        self.out_channels = net._out_channels
        self.img_channels = net._img_channels
        self.signature = None
        self._keep = []          # tensors referenced by raw pointer from the arg blocks
        self._handles = None     # b200dn_igemm_prepared* per launch (encoded tensor maps + launch geometry)
        self._ready = None       # event recorded after the weight-pack kernels of _build
        self._ready_streams = set()
        # fp16 storage saturates at +-65504 (cvt.rn.satfinite): every fp16 launch ORs 1 into this device flag when a
        # stored value hit the limit, so a caller (the sampler) can detect it and retry at a wider precision
        self.sat_flag = (torch.zeros(1, dtype=torch.int32, device=next(net.parameters()).device)
                         if self.prec in _lib.FP16_PRECS else None)
        self.launches = []       # list[IgemmArgs]
        self.layer_info = []     # per launch: mode / shape / FLOPs (diagnostics)
        self.flops = 0
        self._graph = None       # captured CUDA graph of one forward over static input / output buffers
        self._gx = self._gout = self._gt = None
        self._calls = 0
        dev = self.device
        with torch.cuda.device(dev):
            self._build(net)
        self.plan_id = ops.register_plan(self)      # handle the torch.ops.b200dn.rdunet_forward custom op takes

    # ---- weights
    def _pack(self, conv: nn.Module, transposed: bool = False) -> torch.Tensor:
        w = conv.weight.detach()
        if w.dtype != torch.float32 or not w.is_contiguous():
            w = w.float().contiguous()
            self._keep.append(w)
        if transposed:
            cin, cout, groups = w.shape[0], w.shape[1], 4
        else:
            cout, cin, groups = w.shape[0], w.shape[1], w.shape[2] * w.shape[3]
        nbytes = self.lib.b200dn_packed_weight_bytes(cout, cin, groups, self.prec)
        packed = torch.empty(nbytes // 2, dtype=torch.int16, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if transposed:
            rc = self.lib.b200dn_pack_convt_weight(w.data_ptr(), cin, cout, self.prec, packed.data_ptr(), stream)
        else:
            rc = self.lib.b200dn_pack_conv_weight(w.data_ptr(), cout, cin, w.shape[2], w.shape[3], self.prec,
                                                  packed.data_ptr(), stream)
        _lib.check(rc, "pack weight")
        self._keep.append(packed)
        return packed

    @staticmethod
    def _f32(p: torch.Tensor, keep: list) -> int:
        """Plan-owned fp32 snapshot of a bias / PReLU-slope / ingest-weight parameter.  The packed conv weights are
        copies too, so a plan is self-consistent even if the caller later writes the parameters in place without
        bumping their version (EMA / weight averaging through ``p.data``); ``invalidate_plans()`` refreshes it."""
        t = p.detach().to(torch.float32).contiguous().clone()
        keep.append(t)
        return t.data_ptr()

    def _igemm(self, mode, conv, actv, src: _Act, cin, dst: Optional[_Act], coff, B, H, W, res: Optional[_Act] = None,
               transposed=False, nchw=False, collect: Optional[list] = None) -> IgemmArgs:
        a = IgemmArgs()
        a.mode, a.prec = mode, self.prec
        a.B, a.H, a.W = B, H, W
        cout = conv.weight.shape[1] if transposed else conv.weight.shape[0]
        a.cin, a.cout = cin, cout
        hi, lo = src.ptrs()
        a.in_[0], a.in_[1] = hi, lo
        a.in_ctot = src.ctot
        if self.sat_flag is not None:
            a.sat_flag = self.sat_flag.data_ptr()
        a.wpacked = self._pack(conv, transposed).data_ptr()
        a.bias = self._f32(conv.bias, self._keep)
        a.slope = self._f32(actv.weight, self._keep)
        if nchw:
            a.out_kind = _lib.OUT_NCHW32
        else:
            a.out_kind = _lib.OUT_NHWC16
            ohi, olo = dst.ptrs()
            a.out[0], a.out[1] = ohi, olo
            a.out_ctot, a.out_coff = dst.ctot, coff
            if res is not None:
                rhi, rlo = res.ptrs()
                a.res[0], a.res[1] = rhi, rlo
                a.res_ctot = res.ctot
        taps = {_lib.MODE_CONV3X3: 9, _lib.MODE_DOWN2X2: 4, _lib.MODE_UP2X2: 4}[mode]
        pix = B * H * W if mode != _lib.MODE_DOWN2X2 else B * (H // 2) * (W // 2)
        self.flops += 2 * pix * taps * cin * cout
        info = dict(mode=mode, H=H, W=W, cin=cin, cout=cout * (4 if transposed else 1),
                    flops=2 * pix * taps * cin * cout, nchw=nchw)
        if collect is not None:        # part of a chain: listed by the caller
            collect.append((a, info))
            return a
        self.launches.append(a)
        self.layer_info.append(info)
        return a

    def _fusable(self, C: int) -> bool:
        return _FUSE_DENSE and C == 32 and self.prec in (_lib.PREC_BF16, _lib.PREC_FP16)

    def _dense_fused(self, blk: _Params, src: _Act, dst: _Act, dst_coff: int, B, H, W, C) -> None:
        """One b200dn_dense_block launch: input-stationary passes, partial sums in TMEM, o0..o2 never leave the SM."""
        convs = [getattr(blk, f"conv_{k}") for k in range(4)]
        ws = []
        for c in convs:
            w = c.weight.detach().to(torch.float32).contiguous()
            self._keep.append(w)
            ws.append(w)
        nbytes = self.lib.b200dn_dense_block_weight_bytes(C)
        packed = torch.empty(nbytes // 2, dtype=torch.int16, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(self.lib.b200dn_pack_dense_block_weights(ws[0].data_ptr(), ws[1].data_ptr(), ws[2].data_ptr(),
                                                            ws[3].data_ptr(), C, self.prec, packed.data_ptr(), stream),
                   "pack_dense_block_weights")
        self._keep.append(packed)
        a = DenseBlockArgs()
        a.prec, a.B, a.H, a.W, a.channels = self.prec, B, H, W, C
        a.in_, a.in_ctot = src.hi.data_ptr(), src.ctot
        a.out, a.out_ctot, a.out_coff = dst.hi.data_ptr(), dst.ctot, dst_coff
        a.wfused = packed.data_ptr()
        a._epi_dev = []
        for k in range(4):
            a.bias[k] = self._f32(convs[k].bias, self._keep)
            a._epi_dev.append(self._keep[-1])
            a.slope[k] = self._f32(getattr(blk, f"actv_{k}").weight, self._keep)
            a._epi_dev.append(self._keep[-1])
        if self.sat_flag is not None:
            a.sat_flag = self.sat_flag.data_ptr()
        g = C // 2
        flops = 2 * B * H * W * 9 * (C * g + (C + g) * g + (C + 2 * g) * g + (C + 3 * g) * C)
        self.flops += flops
        self.launches.append(a)
        self.layer_info.append(dict(mode=MODE_DENSE_BLOCK, H=H, W=W, cin=C, cout=C, flops=flops, nchw=False))

    def _dense_constants(self, a: DenseBlockArgs, handle) -> None:
        """Bias / PReLU slopes of a fused block as host values in the launch parameters (constant bank) instead of
        shared-memory staging: the kernel sits at the shared-memory bandwidth wall (b200dn.h).  Needs one device -> host
        read of 160 floats while the plan is built, so it is skipped when the plan is built inside a stream capture
        (the kernel then stages the device arrays, same bits)."""
        if not _DENSE_CONST or torch.cuda.is_current_stream_capturing():
            return
        host = [t.cpu() for t in a._epi_dev]                    # [b0, s0, b1, s1, ...] fp32 snapshots of this plan
        fp = C.POINTER(C.c_float)
        bias = (fp * 4)(*[C.cast(host[2 * k].data_ptr(), fp) for k in range(4)])
        slope = (fp * 4)(*[C.cast(host[2 * k + 1].data_ptr(), fp) for k in range(4)])
        _lib.check(self.lib.b200dn_dense_block_set_epilogue_constants(handle, bias, slope),
                   "dense_block_set_epilogue_constants")

    def _dense(self, blk: _Params, src: _Act, dst: _Act, dst_coff: int, B, H, W, C) -> None:
        if self._fusable(C):
            self._dense_fused(blk, src, dst, dst_coff, B, H, W, C)
            return
        g = C // 2
        chain = [] if (_CHAIN_DENSE and self.prec in (_lib.PREC_BF16, _lib.PREC_FP16)) else None
        for k in range(3):
            self._igemm(_lib.MODE_CONV3X3, getattr(blk, f"conv_{k}"), getattr(blk, f"actv_{k}"),
                        src, C + k * g, src, C + k * g, B, H, W, collect=chain)
        # conv_3 + PReLU, then `+ x` (RDUNet_model.py:114-115): residual = channels [0, C) of the block input
        self._igemm(_lib.MODE_CONV3X3, blk.conv_3, blk.actv_3, src, C + 3 * g, dst, dst_coff, B, H, W, res=src,
                    collect=chain)
        if chain is not None:
            self.launches.append(_Chain([a for a, _ in chain], [i for _, i in chain]))
            self.layer_info.append(dict(mode=MODE_CONV_CHAIN, H=H, W=W, cin=C, cout=C,
                                        flops=sum(i["flops"] for _, i in chain), nchw=False))

    def _build(self, net: _RDUNetBase) -> None:
        B, H, W, F, dev, two = self.B, self.H, self.W, self.F, self.device, self.two
        ch = [F << l for l in range(4)]
        hs = [H >> l for l in range(4)]
        ws = [W >> l for l in range(4)]
        # dense buffers [x | o0 | o1 | o2] of 2.5 C channels; a level whose blocks run fused keeps o0..o2 on the SM and
        # needs only the C channels of x (no channel-prefix reads of a wider pixel: the TMA frame is dense)
        dch = [ch[l] if self._fusable(ch[l]) else ch[l] * 5 // 2 for l in range(4)]
        Da = [_Act(B, hs[l], ws[l], dch[l], two, dev) for l in range(4)]
        Db = [_Act(B, hs[l], ws[l], dch[l], two, dev) for l in range(4)]
        K = [_Act(B, hs[l], ws[l], ch[l] * 3, two, dev) for l in range(3)]
        I0 = _Act(B, H, W, F, two, dev)
        self.bufs = dict(Da=Da, Db=Db, K=K, I0=I0)
        self.act_bytes = sum(b.hi.numel() * 2 * (2 if two else 1) for b in (*Da, *Db, *K, I0))

        # input block: conv_1 is the CUDA-core ingest kernel (launched separately in run()); conv_2 on tensor cores
        ib = net.input_block
        self.in_w = self._f32(ib.conv_1.weight, self._keep)
        self.in_b = self._f32(ib.conv_1.bias, self._keep)
        self.in_s = self._f32(ib.actv_1.weight, self._keep)
        self.flops += 2 * B * H * W * 9 * net._in_channels * F
        self._igemm(_lib.MODE_CONV3X3, ib.conv_2, ib.actv_2, I0, F, Da[0], 0, B, H, W)

        # encoder
        for l in range(4):
            b0, b1 = getattr(net, f"block_{l}_0"), getattr(net, f"block_{l}_1")
            self._dense(b0, Da[l], Db[l], 0, B, hs[l], ws[l], ch[l])
            if l < 3:
                self._dense(b1, Db[l], K[l], 0, B, hs[l], ws[l], ch[l])
                dn = getattr(net, f"down_{l}")
                self._igemm(_lib.MODE_DOWN2X2, dn.conv, dn.actv, K[l], ch[l], Da[l + 1], 0, B, hs[l], ws[l])
            else:
                self._dense(b1, Db[l], Da[l], 0, B, hs[l], ws[l], ch[l])
        # decoder
        for l in (2, 1, 0):
            up = getattr(net, f"up_{l}")
            # conv_t + actv_t scatter into K[l][C : 3C); input = Da[l+1][0 : 2C) at half resolution
            self._igemm(_lib.MODE_UP2X2, up.conv_t, up.actv_t, Da[l + 1], ch[l + 1], K[l], ch[l],
                        B, hs[l + 1], ws[l + 1], transposed=True)
            self._igemm(_lib.MODE_CONV3X3, up.conv, up.actv, K[l], 3 * ch[l], Da[l], 0, B, hs[l], ws[l])
            b2, b3 = getattr(net, f"block_{l}_2"), getattr(net, f"block_{l}_3")
            self._dense(b2, Da[l], Db[l], 0, B, hs[l], ws[l], ch[l])
            self._dense(b3, Db[l], Da[l], 0, B, hs[l], ws[l], ch[l])
        # output block
        ob = net.output_block
        self._igemm(_lib.MODE_CONV3X3, ob.conv_1, ob.actv_1, Da[0], F, I0, 0, B, H, W)
        self.out_args = self._igemm(_lib.MODE_CONV3X3, ob.conv_2, ob.actv_2, I0, F, None, 0, B, H, W, nchw=True)
        # prepare every launch once: validation, tiling plan and the 2-3 CUtensorMap encodes (~25 us of host time per
        # layer when done per call) happen here; run() then costs one C call that enqueues the 68 kernels
        handles, launches, infos = [], [], []

        def prepare_one(a, info):
            h = C.c_void_p()
            if a.out_kind == _lib.OUT_NCHW32:      # bound per call in run(); prepare wants a non-null placeholder
                a.out_nchw = self._keep[0].data_ptr()
            _lib.check(self.lib.b200dn_igemm_prepare(C.byref(a), C.byref(h)), f"igemm_prepare (launch {len(handles)})")
            handles.append(h), launches.append(a), infos.append(info)

        for a, info in zip(self.launches, self.layer_info):
            h = C.c_void_p()
            if isinstance(a, DenseBlockArgs):
                _lib.check(self.lib.b200dn_dense_block_prepare(C.byref(a), C.byref(h)),
                           f"dense_block_prepare (launch {len(handles)})")
                self._dense_constants(a, h)
                handles.append(h), launches.append(a), infos.append(info)
            elif isinstance(a, _Chain):
                arr = (IgemmArgs * len(a.layers))(*a.layers)
                nbytes = self.lib.b200dn_conv_chain_workspace_bytes(arr, len(a.layers))
                ws = torch.zeros(max(int(nbytes), 64) // 4, dtype=torch.int32, device=self.device)
                rc = self.lib.b200dn_conv_chain_prepare(arr, len(a.layers), ws.data_ptr(), 1 if _CHAIN_DENSE == 2 else 0,
                                                        C.byref(h))
                if rc == _lib.E_UNSUP:             # e.g. resident-weight or single-CTA layers: launch them one by one
                    for la, li in zip(a.layers, a.infos):
                        prepare_one(la, li)
                else:
                    _lib.check(rc, f"conv_chain_prepare (launch {len(handles)})")
                    self._keep.extend((ws, arr))
                    handles.append(h), launches.append(a), infos.append(info)
            else:
                prepare_one(a, info)
        self.launches, self.layer_info = launches, infos
        n = len(launches)
        self._handles = (C.c_void_p * n)(*handles)
        self._out_handle = self._handles[n - 1]
        self._ready = torch.cuda.Event()
        self._ready.record(torch.cuda.current_stream(self.device))

    def __del__(self):
        handles, self._handles = getattr(self, "_handles", None), None
        if handles is not None:
            try:
                for h in handles:
                    if h:
                        self.lib.b200dn_igemm_release(h)
            except Exception:   # interpreter shutdown
                pass

    # ---- execution
    def forward(self, x: torch.Tensor, t: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One forward for the nn.Module call: returns a fresh fp32 [B, 3, H, W] tensor.

        The reference pays ~70 eager kernel launches per call; here the same launch list costs ~25 us of host time
        per launch (tensor-map encodes + ctypes), which dominates a batch-1 forward.  From the second call of a plan
        on, the launch list is replayed as ONE CUDA graph over static input / output buffers (copy in, replay, clone
        out).  ``B200DN_GRAPH=0`` keeps every call eager; a call made while the caller is itself capturing stays eager.
        t: None, or the timestep as a tensor that broadcasts to [B, 1, H, W]; only per-sample timesteps
        (numel 1 or B) go through the graph."""
        B = self.B
        t_exp = None
        per_sample_t = True
        if self.with_t:
            if t is None:
                raise RuntimeError("RDUNet_T forward needs the timestep tensor t")
            t_exp = t.expand(B, 1, self.H, self.W)
            per_sample_t = t.numel() in (1, B) and (t.numel() == 1 or t.shape[0] == B)
        self._calls += 1
        use_graph = (_USE_GRAPH and per_sample_t and self._calls >= 2
                     and not torch.cuda.is_current_stream_capturing())
        if not use_graph:
            out = torch.empty_like(x)
            self.run(x, out, t=t_exp)
            return out
        dev = self.device
        if self._graph is None:
            self._gx = torch.empty_like(x)
            self._gout = torch.empty_like(x)
            self._gt = torch.zeros(B, dtype=torch.float32, device=dev) if self.with_t else None
            kw = dict(t_ptr=self._gt.data_ptr(), t_strides=(1, 0, 0)) if self.with_t else {}
            self._gx.copy_(x)
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s):      # warm-up on a side stream, then capture
                self.run(self._gx, self._gout, **kw)
            torch.cuda.current_stream(dev).wait_stream(s)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.run(self._gx, self._gout, **kw)
            self._graph = g
        self._gx.copy_(x)
        if self.with_t:
            self._gt.copy_(t.reshape(-1).expand(B) if t.numel() == 1 else t.reshape(B))
        self._graph.replay()
        return self._gout.clone()

    def run(self, x: torch.Tensor, out: torch.Tensor, t: Optional[torch.Tensor] = None,
            x_batch: Optional[int] = None, t_strides=None, t_ptr: Optional[int] = None, events=None,
            layer_events=None) -> None:
        """Enqueue one forward on the current stream.

        x: fp32 NCHW [Bx, 3, H, W] with Bx = x_batch or B; image b of the network batch reads x[b % Bx]
        (the sampler evaluates the same x_t at two timesteps as one 2B batch).  out: fp32 [B, 3, H, W].
        t: expanded [B, 1, H, W] view (strides are honoured), or (t_ptr, t_strides) raw.
        events: optional (start, end) torch.cuda.Event pair recorded around the tensor-core launches
        (after the ingest conv, after the last igemm) — bench.py's live per-kernel timing.
        """
        lib = self.lib
        cur = torch.cuda.current_stream(self.device)
        stream = cur.cuda_stream
        if stream not in self._ready_streams and not torch.cuda.is_current_stream_capturing():
            # the pack kernels ran on whichever stream was current when the plan was built: order this stream after them
            cur.wait_event(self._ready)
            self._ready_streams.add(stream)
        bx = x_batch or self.B
        if self.with_t:
            if t is not None:
                sb, _, sh, sw = t.stride()
                t_ptr, t_strides = t.data_ptr(), (sb, sh, sw)
            if t_ptr is None:
                raise RuntimeError("RDUNet_T forward needs the timestep tensor t")
        else:
            t_ptr, t_strides = None, (0, 0, 0)
        I0 = self.bufs["I0"]
        hi, lo = I0.ptrs()
        rc = lib.b200dn_conv_in(x.data_ptr(), bx, self.img_channels, t_ptr, t_strides[0], t_strides[1], t_strides[2],
                                self.B, self.H, self.W, self.F, self.in_w, self.in_b, self.in_s, self.prec,
                                hi, lo, I0.ctot, self.sat_flag.data_ptr() if self.sat_flag is not None else None, stream)
        _lib.check(rc, "conv_in")
        _lib.check(lib.b200dn_igemm_rebind_nchw(self._out_handle, out.data_ptr(), x.data_ptr(), bx), "igemm_rebind_nchw")
        if events is not None:
            events[0].record()
        if layer_events is None:
            rc = lib.b200dn_igemm_launch_list(self._handles, len(self.launches), stream)
            if rc:
                _lib.check(rc, "igemm_launch_list")
        else:   # diagnostic: one event after every tensor-core launch (tools/layer_times.py)
            layer_events[0].record()
            for i in range(len(self.launches)):
                _lib.check(lib.b200dn_igemm_launch(self._handles[i], stream), "igemm_launch")
                layer_events[i + 1].record()
        if events is not None:
            events[1].record()
