"""LPIPS (lpips 0.1, ``net='alex'``) on the device: the perceptual metric evaluate_Unet_diffusion/evaluate_model.py:46-71
scores every image with.

``LPIPS()`` holds the parameters under the names and shapes of ``lpips.LPIPS(net='alex').state_dict()``, so the weights
come from the caller's own lpips install::

    m = LPIPS().cuda()
    m.load_state_dict(lpips.LPIPS(net='alex').state_dict())        # or torch.load('alex.pth'), strict=False

What is computed (restated from lpips 0.1.4, lpips/lpips.py and lpips/pretrained_networks.py; the package is not a
dependency, so this restatement is not pinned against it):

1. ScalingLayer ``x' = (x - shift) / scale`` per channel (``x = 2x - 1`` first with ``normalize=True``);
2. torchvision AlexNet ``features[0:12]``, tapped after each of the five ReLUs;
3. per tap and pixel: both feature vectors divided by ``sqrt(sum_c f^2) + 1e-10``, the squared difference weighted by
   ``lin{l}.model.1.weight`` and summed over channels, then the mean over the tap's H x W; the sum over the taps.

The trunk runs on the tensor-core implicit GEMM at ``B200DN_PREC_BF16X3`` (fp32-class accuracy: the trunk's rounding
goes straight into ``f0 - f1``, which is small for a good denoiser, and the whole metric costs ~0.1 % of an RDUNet(128)
forward).  conv1 (11x11/s4) and conv2 (5x5) are MODE_CONV1X1 GEMMs over gathered patch rows, conv3..conv5 the 3x3 path;
the patch gathers, the max-pools and the head are the kernels of csrc/lpips.cu.  Inference only; no CPU fallback.

``DISTS()`` (DISTS_pytorch 0.1, ``DISTS_pt.py``) holds the parameters under the names and shapes of
``DISTS().state_dict()`` in the same way; the VGG16 trunk runs on the same convolutions and the L2 pooling and the
structure / texture head are the kernels of csrc/dists.cu (see :class:`DISTS`).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from ._lib import DistsStage, IgemmArgs, LpipsTap
from .rdunet import _Act

__all__ = ["LPIPS", "LpipsPlan", "DISTS", "DistsPlan", "gemm_weight", "trunk_shapes", "dists_stage_sizes", "MIN_SIZE",
           "DISTS_MIN_SIZE"]

PREC = _lib.PREC_BF16X3
CHNS = (64, 192, 384, 256, 256)
# (slice, index in AlexNet.features) of conv1..conv5: lpips registers features[0:2], [2:5], [5:8], [8:10], [10:12]
_CONV_KEYS = ((1, 0), (2, 3), (3, 6), (4, 8), (5, 10))
# (in, out, kernel, stride, padding) of torchvision's AlexNet convolutions
_CONVS = ((3, 64, 11, 4, 2), (64, 192, 5, 1, 2), (192, 384, 3, 1, 1), (384, 256, 3, 1, 1), (256, 256, 3, 1, 1))
K1PAD = 384                  # conv1's 11 * 11 * 3 = 363 patch columns, padded to the GEMM's 64-column K blocks
K2 = 25 * 64                 # conv2's 5 * 5 * 64 patch columns
MIN_SIZE = 31                # smallest H, W the second max-pool accepts (torch raises below it)


def gemm_weight(w: torch.Tensor, kpad: int) -> torch.Tensor:
    """OIHW conv weight -> the [Cout, kpad, 1, 1] weight of the 1x1 GEMM over (ky, kx, ci)-ordered patch rows."""
    cout = w.shape[0]
    g = w.permute(0, 2, 3, 1).reshape(cout, -1)
    return F.pad(g, (0, kpad - g.shape[1])).reshape(cout, kpad, 1, 1).contiguous()


def trunk_shapes(H: int, W: int):
    """Spatial sizes (conv1, pool1, pool2) of the trunk: conv2 keeps pool1's size, conv3..conv5 pool2's."""
    c1 = ((H + 4 - 11) // 4 + 1, (W + 4 - 11) // 4 + 1)
    p1 = ((c1[0] - 3) // 2 + 1, (c1[1] - 3) // 2 + 1)
    p2 = ((p1[0] - 3) // 2 + 1, (p1[1] - 3) // 2 + 1)
    return c1, p1, p2


class _DeviceMetric(nn.Module):
    """Module plumbing shared by the device metrics: launch plans per (N, H, W) (``_new_plan``), rebuilt when a parameter
    or buffer changes and dropped whenever the module is moved, copied or pickled (they hold raw device pointers)."""

    min_size = 1
    _min_size_reason = ""
    _metric_name = ""

    def __init__(self):
        super().__init__()
        self._plans = {}

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._plans = {}
        return out

    def __deepcopy__(self, memo):
        import copy
        plans, self._plans = self._plans, {}
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
        """Drop the cached plans; needed only after in-place writes that bypass the version counter (``p.data``)."""
        self._plans = {}

    def _signature(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers()))

    def _new_plan(self, N: int, H: int, W: int):
        raise NotImplementedError

    def plan(self, N: int, H: int, W: int):
        key = (N, H, W)
        plan = self._plans.get(key)
        sig = self._signature()
        if plan is None or plan.signature != sig:
            if plan is None and len(self._plans) >= 4:
                self._plans.pop(next(iter(self._plans)))
            plan = self._new_plan(N, H, W)
            plan.signature = sig
            self._plans[key] = plan
        return plan

    def _check_inputs(self, in0: torch.Tensor, in1: torch.Tensor):
        for t in (in0, in1):
            if not isinstance(t, torch.Tensor) or t.dim() != 4 or t.size(1) != 3:
                raise RuntimeError("expected two [N, 3, H, W] image tensors")
            if not t.is_cuda:
                raise RuntimeError("vub_image_denoising_b200 runs on CUDA (sm_100) tensors only; there is no CPU fallback")
        if in0.shape != in1.shape:
            raise RuntimeError(f"shape mismatch {tuple(in0.shape)} vs {tuple(in1.shape)}")
        if min(in0.shape[2:]) < self.min_size:
            raise RuntimeError(f"spatial size {tuple(in0.shape[2:])} is below {self.min_size} x {self.min_size}: "
                               f"{self._min_size_reason}")
        if torch.is_grad_enabled() and (in0.requires_grad or in1.requires_grad or self.training):
            raise RuntimeError("the B200 path is inference-only: use model.eval() and torch.no_grad() "
                               f"({self._metric_name} as a training loss is out of scope)")
        buf = next(self.buffers())
        if in1.device != in0.device or buf.device != in0.device:
            raise RuntimeError(f"module buffers are on {buf.device}, inputs on {in0.device} and {in1.device}")
        return (in0.detach().to(torch.float32).contiguous(), in1.detach().to(torch.float32).contiguous())


class _DevicePlan:
    """What every metric plan holds: plan-owned fp32 parameter snapshots, packed weights, prepared GEMM handles
    (released with the plan) and the event after which the weight-pack kernels are done."""

    def __init__(self, device: torch.device, N: int, H: int, W: int):
        self.lib = _lib.lib()
        self.device = device
        self.N, self.H, self.W = N, H, W
        self.signature = None
        self._keep = []
        self._prepared = []

    def _f32(self, t: torch.Tensor) -> int:
        """Plan-owned fp32 snapshot of a parameter (see rdunet.ForwardPlan._f32)."""
        c = t.detach().to(torch.float32).contiguous().clone()
        self._keep.append(c)
        return c.data_ptr()

    def _pack(self, w: torch.Tensor) -> torch.Tensor:
        w = w.contiguous()
        cout, cin, kh, kw = w.shape
        packed = torch.empty(self.lib.b200dn_packed_weight_bytes(cout, cin, kh * kw, PREC) // 2, dtype=torch.int16,
                             device=self.device)
        _lib.check(self.lib.b200dn_pack_conv_weight(w.data_ptr(), cout, cin, kh, kw, PREC, packed.data_ptr(),
                                                    torch.cuda.current_stream(self.device).cuda_stream), "pack weight")
        self._keep.extend((w, packed))
        return packed

    def _prepare(self, a: IgemmArgs, what: str) -> C.c_void_p:
        h = C.c_void_p()
        _lib.check(self.lib.b200dn_igemm_prepare(C.byref(a), C.byref(h)), f"igemm_prepare ({what})")
        self._prepared.append(h)
        self._keep.append(a)
        return h

    def _conv_args(self, mode: int, src, cin: int, h: int, w: int, wpacked: torch.Tensor, conv: nn.Conv2d,
                   out) -> IgemmArgs:
        """b200dn_igemm arguments of conv + bias + ReLU (PReLU with slopes 0) from ``src`` into all of ``out``."""
        a = IgemmArgs()
        a.mode = mode
        a.prec = PREC
        a.B, a.H, a.W = 2 * self.N, h, w
        a.cin, a.cout = cin, conv.out_channels
        a.in_[0], a.in_[1] = src.ptrs()
        a.in_ctot = src.ctot
        a.wpacked = wpacked.data_ptr()
        a.bias = self._f32(conv.bias)
        a.slope = self._f32(torch.zeros(conv.out_channels, device=self.device))
        a.out_kind = _lib.OUT_NHWC16
        a.out[0], a.out[1] = out.ptrs()
        a.out_ctot, a.out_coff = conv.out_channels, 0
        return a

    def _register(self) -> None:
        """Record the weight-pack event on the current stream and register the finished plan with the custom ops."""
        self._ready = torch.cuda.Event()
        self._ready.record(torch.cuda.current_stream(self.device))
        self._ready_streams = set()
        self.plan_id = ops.register_plan(self)

    def _stream(self) -> int:
        """The current stream, made to wait (once, outside graph capture) for the weight-pack kernels."""
        cur = torch.cuda.current_stream(self.device)
        stream = cur.cuda_stream
        if stream not in self._ready_streams and not torch.cuda.is_current_stream_capturing():
            cur.wait_event(self._ready)    # the weight-pack kernels ran on the stream current at plan time
            self._ready_streams.add(stream)
        return stream

    def __del__(self):
        handles, self._prepared = getattr(self, "_prepared", None), None
        if handles is not None:
            try:
                for h in handles:
                    if h:
                        self.lib.b200dn_igemm_release(h)
            except Exception:   # interpreter shutdown
                pass


class _ScalingLayer(nn.Module):
    def __init__(self):
        super().__init__()
        self.register_buffer("shift", torch.tensor([-.030, -.088, -.188])[None, :, None, None])
        self.register_buffer("scale", torch.tensor([.458, .448, .450])[None, :, None, None])


class _AlexNetSlices(nn.Module):
    """Parameter holder of lpips.pretrained_networks.alexnet: slice1..slice5 keep AlexNet.features' indices."""

    def __init__(self):
        super().__init__()
        for (s, idx), (cin, cout, k, stride, pad) in zip(_CONV_KEYS, _CONVS):
            sl = nn.Sequential()
            sl.add_module(str(idx), nn.Conv2d(cin, cout, k, stride=stride, padding=pad))
            self.add_module(f"slice{s}", sl)

    def convs(self):
        return [getattr(self, f"slice{s}")[0] for s, _ in _CONV_KEYS]


class _NetLinLayer(nn.Module):
    def __init__(self, chn_in: int):
        super().__init__()
        self.model = nn.Sequential(nn.Dropout(), nn.Conv2d(chn_in, 1, 1, stride=1, padding=0, bias=False))


class LPIPS(_DeviceMetric):
    """``lpips.LPIPS(net='alex')`` for inference on the B200: ``forward(in0, in1)`` -> fp32 ``[N, 1, 1, 1]``."""

    min_size = MIN_SIZE
    _min_size_reason = "AlexNet's second max-pool has no output there"
    _metric_name = "LPIPS"

    def __init__(self, net: str = "alex", version: str = "0.1", lpips: bool = True, spatial: bool = False):
        super().__init__()
        if net != "alex" or version != "0.1" or not lpips or spatial:
            raise NotImplementedError("only lpips.LPIPS(net='alex', version='0.1', lpips=True, spatial=False) is "
                                      "implemented on device")
        self.scaling_layer = _ScalingLayer()
        self.net = _AlexNetSlices()
        for i, c in enumerate(CHNS):
            setattr(self, f"lin{i}", _NetLinLayer(c))
        self.lins = nn.ModuleList([getattr(self, f"lin{i}") for i in range(len(CHNS))])
        for p in self.parameters():
            p.requires_grad_(False)
        self.eval()

    def _new_plan(self, N: int, H: int, W: int) -> "LpipsPlan":
        return LpipsPlan(self, N, H, W)

    def forward(self, in0: torch.Tensor, in1: torch.Tensor, retPerLayer: bool = False,
                normalize: bool = False) -> torch.Tensor:
        """LPIPS distance of each image pair: in0, in1 fp32 CUDA [N, 3, H, W] in [-1, 1] (in [0, 1] with
        ``normalize=True``).  Returns a fresh fp32 CUDA tensor [N, 1, 1, 1]; no host synchronisation."""
        if retPerLayer:
            raise NotImplementedError("retPerLayer=True is not implemented on device")
        x0, x1 = self._check_inputs(in0, in1)
        plan = self.plan(x0.size(0), x0.size(2), x0.size(3))
        return torch.ops.b200dn.lpips_forward(x0, x1, bool(normalize), plan.plan_id)


class LpipsPlan(_DevicePlan):
    """Buffers, packed weights, prepared GEMM handles and the launch list of one (N, H, W) LPIPS call.

    Image pair n is batch entries n (in0) and N + n (in1) of every buffer.  Launches: conv1 patch gather, conv1 GEMM,
    pool, conv2 patch gather, conv2 GEMM, pool, conv3..conv5, head, head sum."""

    def __init__(self, m: LPIPS, N: int, H: int, W: int):
        super().__init__(m.scaling_layer.shift.device, N, H, W)
        B = 2 * N
        (h1, w1), (hp1, wp1), (hp2, wp2) = trunk_shapes(H, W)
        dev = self.device
        with torch.cuda.device(dev):
            self.g1 = _Act(B, h1, w1, K1PAD, True, dev)
            self.g2 = _Act(B, hp1, wp1, K2, True, dev)
            self.pool1 = _Act(B, hp1, wp1, CHNS[0], True, dev)
            self.pool2 = _Act(B, hp2, wp2, CHNS[1], True, dev)
            sizes = ((h1, w1), (hp1, wp1), (hp2, wp2), (hp2, wp2), (hp2, wp2))
            self.features = [_Act(B, h, w, c, True, dev) for (h, w), c in zip(sizes, CHNS)]
            self.shift = self._f32(m.scaling_layer.shift.reshape(-1))
            self.scale = self._f32(m.scaling_layer.scale.reshape(-1))
            convs = m.net.convs()
            gemm_w = [gemm_weight(convs[0].weight.detach().float(), K1PAD), gemm_weight(convs[1].weight.detach().float(), K2)]
            srcs = [(self.g1, K1PAD, h1, w1), (self.g2, K2, hp1, wp1), (self.pool2, CHNS[1], hp2, wp2),
                    (self.features[2], CHNS[2], hp2, wp2), (self.features[3], CHNS[3], hp2, wp2)]
            handles = []
            for i, (conv, (src, cin, h, w)) in enumerate(zip(convs, srcs)):
                wpacked = self._pack(gemm_w[i] if i < 2 else conv.weight.detach().float())
                a = self._conv_args(_lib.MODE_CONV1X1 if i < 2 else _lib.MODE_CONV3X3, src, cin, h, w, wpacked, conv,
                                    self.features[i])
                handles.append(self._prepare(a, f"conv{i + 1}"))
            self._handles = (C.c_void_p * 5)(*handles)
            self._tail = (C.c_void_p * 3)(*handles[2:])      # conv3..conv5, one launch-list call
            taps = []
            for i, f in enumerate(self.features):
                t = LpipsTap()
                t.feat[0], t.feat[1] = f.ptrs()
                t.weight = self._f32(getattr(m, f"lin{i}").model[1].weight.reshape(-1))
                t.H, t.W, t.C = f.H, f.W, f.ctot
                taps.append(t)
            self.taps = (LpipsTap * 5)(*taps)
            nbytes = self.lib.b200dn_lpips_head_workspace_bytes(self.taps, 5, N)
            if nbytes <= 0:
                raise RuntimeError(f"lpips_head_workspace_bytes failed: {self.lib.b200dn_last_error().decode()}")
            self.workspace = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=dev)
            self._register()

    def forward(self, x0: torch.Tensor, x1: torch.Tensor, normalize: bool,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Enqueue one LPIPS call on the current stream; x0, x1 contiguous fp32 [N, 3, H, W]."""
        lib, N = self.lib, self.N
        if out is None:
            out = torch.empty((N, 1, 1, 1), dtype=torch.float32, device=x0.device)
        stream = self._stream()
        g1, g2, p1, p2, f = self.g1, self.g2, self.pool1, self.pool2, self.features
        _lib.check(lib.b200dn_patch_gather_image(x0.data_ptr(), x1.data_ptr(), N, 3, self.H, self.W, self.shift,
                                                 self.scale, int(normalize), 11, 11, 4, 2, K1PAD, PREC, *g1.ptrs(),
                                                 stream), "patch_gather_image")
        _lib.check(lib.b200dn_igemm_launch(self._handles[0], stream), "igemm_launch (conv1)")
        _lib.check(lib.b200dn_maxpool3x3s2(*f[0].ptrs(), 2 * N, f[0].H, f[0].W, CHNS[0], PREC, *p1.ptrs(), stream),
                   "maxpool3x3s2")
        _lib.check(lib.b200dn_patch_gather(*p1.ptrs(), 2 * N, p1.H, p1.W, CHNS[0], 5, 5, 1, 2, K2, PREC, *g2.ptrs(),
                                           stream), "patch_gather")
        _lib.check(lib.b200dn_igemm_launch(self._handles[1], stream), "igemm_launch (conv2)")
        _lib.check(lib.b200dn_maxpool3x3s2(*f[1].ptrs(), 2 * N, f[1].H, f[1].W, CHNS[1], PREC, *p2.ptrs(), stream),
                   "maxpool3x3s2")
        _lib.check(lib.b200dn_igemm_launch_list(self._tail, 3, stream), "igemm_launch_list (conv3..conv5)")
        _lib.check(lib.b200dn_lpips_head(self.taps, 5, N, PREC, out.data_ptr(), self.workspace.data_ptr(),
                                         self.workspace.numel() * 8, stream), "lpips_head")
        return out


# ------------------------------------------------------------------------------------------------------------- DISTS
DISTS_CHNS = (3, 64, 128, 256, 512, 512)      # the six compared feature sets: the input, relu1_2 .. relu5_3
# torchvision vgg16().features indices of each stage's convolutions (in, out channels); a ReLU follows each one
DISTS_CONVS = (((0, 3, 64), (2, 64, 64)),
               ((5, 64, 128), (7, 128, 128)),
               ((10, 128, 256), (12, 256, 256), (14, 256, 256)),
               ((17, 256, 512), (19, 512, 512), (21, 512, 512)),
               ((24, 512, 512), (26, 512, 512), (28, 512, 512)))
DISTS_POOLS = (4, 9, 16, 23)                   # the MaxPool2d indices DISTS replaces with L2pooling
DISTS_K1PAD = 64                               # conv1_1's 3 * 3 * 3 = 27 patch columns, padded to the GEMM's K block
DISTS_MIN_SIZE = 16                            # smallest H, W the device path is tested at (stage 5 is 1 x 1 there)


def dists_stage_sizes(H: int, W: int):
    """Spatial size of stages 1..5: each L2 pooling (3x3, stride 2, padding 1) maps n to (n - 1) // 2 + 1."""
    sizes = [(H, W)]
    for _ in range(4):
        h, w = sizes[-1]
        sizes.append(((h - 1) // 2 + 1, (w - 1) // 2 + 1))
    return sizes


def hanning_filter(channels: int) -> torch.Tensor:
    """DISTS' L2pooling taps: the outer product of np.hanning(5)[1:-1] = [.5, 1, .5], normalised to sum 1, per channel."""
    a = torch.tensor([0.5, 1.0, 0.5], dtype=torch.float64)
    g = a[:, None] * a[None, :]
    return (g / g.sum()).float()[None, None].repeat(channels, 1, 1, 1)


class L2pooling(nn.Module):
    """Parameter holder of DISTS_pt.L2pooling(channels=C): the depthwise 3x3 ``filter`` buffer."""

    def __init__(self, channels: int):
        super().__init__()
        self.channels = channels
        self.register_buffer("filter", hanning_filter(channels))


class DISTS(_DeviceMetric):
    """``DISTS_pytorch.DISTS()`` for inference on the B200: ``forward(x, y)`` -> fp32 ``[N]`` (0-d for N = 1).

    The parameters sit under the names and shapes of ``DISTS().state_dict()`` (``alpha``, ``beta``, ``mean``, ``std``,
    then ``stage1.0.weight`` .. ``stage5.28.bias`` with the ``stage{k}.{idx}.filter`` buffers of the L2 poolings), so
    the weights come from the caller's own DISTS_pytorch install::

        m = DISTS().cuda()
        m.load_state_dict(DISTS_pytorch.DISTS().state_dict())

    What is computed (restated from DISTS_pytorch 0.1, DISTS_pt.py; the package is not a dependency, so this
    restatement is not pinned against it):

    1. ``h = (x - mean) / std`` (ImageNet mean / std, inputs in [0, 1]);
    2. torchvision VGG16 ``features[0:30]`` with the four max-pools replaced by L2pooling
       ``sqrt(conv2d(h^2, filter, stride=2, padding=1, groups=C) + 1e-12)``; the features compared are
       ``[x, relu1_2, relu2_2, relu3_3, relu4_3, relu5_3]`` (the first is the raw input);
    3. per stage and channel, with the population moments over H x W: ``S1 = (2 mx my + c1) / (mx^2 + my^2 + c1)``,
       ``S2 = (2 cov + c2) / (vx + vy + c2)``, c1 = c2 = 1e-6;
       ``score = 1 - sum (alpha S1 + beta S2) / (sum alpha + sum beta)``.

    The trunk runs at bf16x3 like LPIPS's: S2 is a covariance, so the trunk's rounding goes straight into it.  conv1_1
    is a MODE_CONV1X1 GEMM over patch rows gathered from the fp32 images with the normalisation fused in (the padding
    holds zeros of the normalised image, as in the reference), the other twelve the 3x3 path.  Inference only; no CPU
    fallback.  Construction loads nothing; ``alpha`` and ``beta`` start as the package's ``normal_(0.1, 0.01)``."""

    min_size = DISTS_MIN_SIZE
    _min_size_reason = "the smallest size the device path is tested at"
    _metric_name = "DISTS"

    def __init__(self):
        super().__init__()
        for s, convs in enumerate(DISTS_CONVS):
            st = nn.Sequential()
            if s > 0:
                st.add_module(str(DISTS_POOLS[s - 1]), L2pooling(convs[0][1]))
            for idx, cin, cout in convs:
                st.add_module(str(idx), nn.Conv2d(cin, cout, 3, padding=1))
                st.add_module(str(idx + 1), nn.ReLU(inplace=True))
            self.add_module(f"stage{s + 1}", st)
        self.register_buffer("mean", torch.tensor([0.485, 0.456, 0.406]).view(1, -1, 1, 1))
        self.register_buffer("std", torch.tensor([0.229, 0.224, 0.225]).view(1, -1, 1, 1))
        self.chns = list(DISTS_CHNS)
        self.register_parameter("alpha", nn.Parameter(torch.randn(1, sum(self.chns), 1, 1)))
        self.register_parameter("beta", nn.Parameter(torch.randn(1, sum(self.chns), 1, 1)))
        self.alpha.data.normal_(0.1, 0.01)
        self.beta.data.normal_(0.1, 0.01)
        for p in self.parameters():
            p.requires_grad_(False)
        self.eval()

    def convs(self):
        """The 13 convolutions in trunk order."""
        return [getattr(self, f"stage{s + 1}")._modules[str(idx)]
                for s, convs in enumerate(DISTS_CONVS) for idx, _, _ in convs]

    def pools(self):
        """The four L2 poolings in trunk order."""
        return [getattr(self, f"stage{s + 2}")._modules[str(idx)] for s, idx in enumerate(DISTS_POOLS)]

    def _new_plan(self, N: int, H: int, W: int) -> "DistsPlan":
        return DistsPlan(self, N, H, W)

    def forward(self, x: torch.Tensor, y: torch.Tensor, require_grad: bool = False,
                batch_average: bool = False) -> torch.Tensor:
        """DISTS of each image pair: x, y fp32 CUDA [N, 3, H, W] in [0, 1].  Returns a fresh fp32 CUDA tensor [N] (0-d
        for N = 1, as the reference's ``.squeeze()``), or its mean with ``batch_average``; no host synchronisation."""
        if require_grad:
            raise RuntimeError("the B200 path is inference-only: require_grad=True is not supported "
                               "(DISTS as a training loss is out of scope)")
        x0, x1 = self._check_inputs(x, y)
        plan = self.plan(x0.size(0), x0.size(2), x0.size(3))
        score = torch.ops.b200dn.dists_forward(x0, x1, plan.plan_id)
        return score.mean() if batch_average else score.squeeze()


class DistsPlan(_DevicePlan):
    """Buffers, packed weights, prepared GEMM handles and the launch list of one (N, H, W) DISTS call.

    Image pair n is batch entries n (x) and N + n (y) of every buffer.  Launches: conv1_1 patch gather, conv1_1 +
    conv1_2, then per stage 2..5 an L2 pooling and the stage's convolutions (one launch-list call per stage), head,
    head sum: 15 launches."""

    def __init__(self, m: DISTS, N: int, H: int, W: int):
        super().__init__(m.mean.device, N, H, W)
        B = 2 * N
        dev = self.device
        sizes = dists_stage_sizes(H, W)
        convs = iter(m.convs())
        with torch.cuda.device(dev):
            self.g1 = _Act(B, H, W, DISTS_K1PAD, True, dev)
            self.mean = self._f32(m.mean.reshape(-1))
            self.std = self._f32(m.std.reshape(-1))
            self.pools, self.filters, self.conv_outs, self._lists = [], [], [], []
            src, cin = self.g1, DISTS_K1PAD
            for s, ((h, w), layers) in enumerate(zip(sizes, DISTS_CONVS)):
                if s > 0:
                    pool = m.pools()[s - 1]
                    self.filters.append(self._f32(pool.filter.reshape(-1)))
                    src = _Act(B, h, w, cin, True, dev)
                    self.pools.append(src)
                handles, outs = [], []
                for i in range(len(layers)):
                    conv = next(convs)
                    out = _Act(B, h, w, conv.out_channels, True, dev)
                    if s == 0 and i == 0:
                        mode, wpacked = _lib.MODE_CONV1X1, self._pack(gemm_weight(conv.weight.detach().float(),
                                                                                  DISTS_K1PAD))
                    else:
                        mode, wpacked = _lib.MODE_CONV3X3, self._pack(conv.weight.detach().float())
                    a = self._conv_args(mode, src, cin, h, w, wpacked, conv, out)
                    handles.append(self._prepare(a, f"conv{s + 1}_{i + 1}"))
                    outs.append(out)
                    src, cin = out, conv.out_channels
                self.conv_outs.append(outs)
                self._lists.append((C.c_void_p * len(handles))(*handles))
            self.features = [outs[-1] for outs in self.conv_outs]     # relu1_2, relu2_2, relu3_3, relu4_3, relu5_3
            stages = []
            for f in self.features:
                st = DistsStage()
                st.feat[0], st.feat[1] = f.ptrs()
                st.H, st.W, st.C = f.H, f.W, f.ctot
                stages.append(st)
            self.stages = (DistsStage * 5)(*stages)
            self.alpha = self._f32(m.alpha.reshape(-1))
            self.beta = self._f32(m.beta.reshape(-1))
            nbytes = self.lib.b200dn_dists_head_workspace_bytes(H, W, self.stages, 5, N)
            if nbytes <= 0:
                raise RuntimeError(f"dists_head_workspace_bytes failed: {self.lib.b200dn_last_error().decode()}")
            self.workspace = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=dev)
            self._register()

    def forward(self, x0: torch.Tensor, x1: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Enqueue one DISTS call on the current stream; x0, x1 contiguous fp32 [N, 3, H, W]."""
        lib, N = self.lib, self.N
        if out is None:
            out = torch.empty((N,), dtype=torch.float32, device=x0.device)
        stream = self._stream()
        _lib.check(lib.b200dn_patch_gather_image(x0.data_ptr(), x1.data_ptr(), N, 3, self.H, self.W, self.mean,
                                                 self.std, 0, 3, 3, 1, 1, DISTS_K1PAD, PREC, *self.g1.ptrs(), stream),
                   "patch_gather_image")
        for s, handles in enumerate(self._lists):
            if s > 0:
                f, p = self.features[s - 1], self.pools[s - 1]
                _lib.check(lib.b200dn_l2pool3x3s2(*f.ptrs(), 2 * N, f.H, f.W, f.ctot, self.filters[s - 1], PREC,
                                                  *p.ptrs(), stream), "l2pool3x3s2")
            _lib.check(lib.b200dn_igemm_launch_list(handles, len(handles), stream), f"igemm_launch_list (stage {s + 1})")
        _lib.check(lib.b200dn_dists_head(x0.data_ptr(), x1.data_ptr(), self.H, self.W, self.stages, 5, N, self.alpha,
                                         self.beta, PREC, out.data_ptr(), self.workspace.data_ptr(),
                                         self.workspace.numel() * 8, stream), "dists_head")
        return out
