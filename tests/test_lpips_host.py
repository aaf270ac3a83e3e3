"""CPU: the LPIPS module's parameter layout (lpips.LPIPS(net='alex').state_dict()), the host-side weight reshape and
patch order of the two GEMM-lowered convolutions, the trunk shapes, and the oracle's trunk against torchvision."""
import ctypes
import subprocess
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

from oracle import lpips_oracle
from vub_image_denoising_b200 import _lib, perceptual
from vub_image_denoising_b200.perceptual import LPIPS

ROOT = Path(__file__).resolve().parent.parent

# lpips 0.1.4 (not installed here; restated, unpinned): lpips/lpips.py LPIPS.__init__ registers scaling_layer, net,
# lin0..lin4 and then lins = nn.ModuleList([lin0, ..., lin4]), so the lin weights appear under both names;
# lpips/pretrained_networks.py alexnet keeps torchvision's features indices in slice1..slice5; NetLinLayer is
# Sequential(Dropout(), Conv2d(C, 1, 1, bias=False)).
LPIPS_ALEX_KEYS = [
    ("scaling_layer.shift", (1, 3, 1, 1)), ("scaling_layer.scale", (1, 3, 1, 1)),
    ("net.slice1.0.weight", (64, 3, 11, 11)), ("net.slice1.0.bias", (64,)),
    ("net.slice2.3.weight", (192, 64, 5, 5)), ("net.slice2.3.bias", (192,)),
    ("net.slice3.6.weight", (384, 192, 3, 3)), ("net.slice3.6.bias", (384,)),
    ("net.slice4.8.weight", (256, 384, 3, 3)), ("net.slice4.8.bias", (256,)),
    ("net.slice5.10.weight", (256, 256, 3, 3)), ("net.slice5.10.bias", (256,)),
    ("lin0.model.1.weight", (1, 64, 1, 1)), ("lin1.model.1.weight", (1, 192, 1, 1)),
    ("lin2.model.1.weight", (1, 384, 1, 1)), ("lin3.model.1.weight", (1, 256, 1, 1)),
    ("lin4.model.1.weight", (1, 256, 1, 1)),
    ("lins.0.model.1.weight", (1, 64, 1, 1)), ("lins.1.model.1.weight", (1, 192, 1, 1)),
    ("lins.2.model.1.weight", (1, 384, 1, 1)), ("lins.3.model.1.weight", (1, 256, 1, 1)),
    ("lins.4.model.1.weight", (1, 256, 1, 1)),
]


def test_state_dict_matches_lpips_alex():
    sd = LPIPS().state_dict()
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == LPIPS_ALEX_KEYS
    assert torch.equal(sd["scaling_layer.shift"].flatten(), torch.tensor([-.030, -.088, -.188]))
    assert torch.equal(sd["scaling_layer.scale"].flatten(), torch.tensor([.458, .448, .450]))
    assert all(v.dtype == torch.float32 for v in sd.values())


def test_full_and_lin_only_state_dicts_load():
    src = LPIPS()
    torch.manual_seed(3)
    full = {k: torch.rand(v.shape) for k, v in src.state_dict().items()}
    for i in range(5):                       # the two names of a lin weight are one tensor in lpips
        full[f"lins.{i}.model.1.weight"] = full[f"lin{i}.model.1.weight"]
    m = LPIPS()
    m.load_state_dict(full)
    for k, v in m.state_dict().items():
        assert torch.equal(v, full[k]), k
    # weights/v0.1/alex.pth holds the lin layers only and is loaded with strict=False
    lin_only = {f"lin{i}.model.1.weight": torch.rand(1, c, 1, 1) for i, c in enumerate(perceptual.CHNS)}
    m2 = LPIPS()
    res = m2.load_state_dict(lin_only, strict=False)
    assert not res.unexpected_keys
    assert sorted(res.missing_keys) == sorted(k for k, _ in LPIPS_ALEX_KEYS
                                              if not k.startswith("lin") or k.startswith("lins."))
    for i in range(5):
        assert torch.equal(m2.lins[i].model[1].weight, lin_only[f"lin{i}.model.1.weight"])


def test_unsupported_options_raise():
    for kw in (dict(spatial=True), dict(net="vgg"), dict(lpips=False), dict(version="0.0")):
        with pytest.raises(NotImplementedError):
            LPIPS(**kw)
    m = LPIPS()
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 3, 64, 64), torch.zeros(1, 3, 64, 64), retPerLayer=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 64, 64), torch.zeros(1, 3, 64, 64))


def _gemm_conv(x, w, stride, pad, kpad):
    """The GPU lowering emulated: patch rows in (ky, kx, ci) order, zero padded to kpad, times gemm_weight."""
    N, Cin, H, W = x.shape
    cout, _, kh, kw = w.shape
    Ho, Wo = (H + 2 * pad - kh) // stride + 1, (W + 2 * pad - kw) // stride + 1
    cols = F.unfold(x, (kh, kw), padding=pad, stride=stride)              # [N, Cin*kh*kw, L], (ci, ky, kx) order
    cols = cols.view(N, Cin, kh * kw, -1).permute(0, 3, 2, 1).reshape(N, Ho * Wo, kh * kw * Cin)
    rows = F.pad(cols, (0, kpad - cols.shape[-1]))
    out = rows @ perceptual.gemm_weight(w, kpad).view(cout, kpad).t()
    return out.view(N, Ho, Wo, cout).permute(0, 3, 1, 2)


@pytest.mark.parametrize("which", ["conv1", "conv2"])
def test_gemm_lowering_equals_conv2d(which):
    # small integers in fp64: every product and sum is exact, so any order gives the same bits
    g = torch.Generator().manual_seed(5)
    if which == "conv1":
        x = torch.randint(-8, 9, (2, 3, 47, 33), generator=g).double()
        w = torch.randint(-8, 9, (64, 3, 11, 11), generator=g).double()
        got, want = _gemm_conv(x, w, 4, 2, perceptual.K1PAD), F.conv2d(x, w, stride=4, padding=2)
    else:
        x = torch.randint(-8, 9, (2, 64, 11, 7), generator=g).double()
        w = torch.randint(-8, 9, (192, 64, 5, 5), generator=g).double()
        got, want = _gemm_conv(x, w, 1, 2, perceptual.K2), F.conv2d(x, w, padding=2)
    assert torch.equal(got, want)


@pytest.mark.parametrize("hw", [(256, 256), (96, 160), (250, 200), (31, 47)])
def test_trunk_shapes(hw):
    torch.manual_seed(0)
    feats = lpips_oracle.alexnet_features(LPIPS().state_dict(), torch.float32)
    t = lpips_oracle.taps(feats, torch.rand(1, 3, *hw))
    c1, p1, p2 = perceptual.trunk_shapes(*hw)
    assert [tuple(x.shape[2:]) for x in t] == [c1, p1, p2, p2, p2]


def test_min_size_is_where_torch_stops():
    feats = lpips_oracle.alexnet_features(LPIPS().state_dict(), torch.float32)
    lpips_oracle.taps(feats, torch.rand(1, 3, perceptual.MIN_SIZE, perceptual.MIN_SIZE))
    with pytest.raises(RuntimeError):
        lpips_oracle.taps(feats, torch.rand(1, 3, perceptual.MIN_SIZE - 1, 64))


def test_oracle_trunk_is_torchvision_alexnet():
    import torchvision
    torch.manual_seed(11)
    tv = torchvision.models.alexnet(weights=None).eval()
    sd = LPIPS().state_dict()
    for key, idx in lpips_oracle.CONV_KEYS:
        sd[key + ".weight"], sd[key + ".bias"] = tv.features[idx].weight.detach(), tv.features[idx].bias.detach()
    x = torch.rand(2, 3, 96, 80)
    got = lpips_oracle.taps(lpips_oracle.alexnet_features(sd, torch.float32), x)
    want, y = [], x
    with torch.no_grad():                    # lpips' slices: features[0:2], [2:5], [5:8], [8:10], [10:12]
        for a, b in ((0, 2), (2, 5), (5, 8), (8, 10), (10, 12)):
            y = tv.features[a:b](y)
            want.append(y.clone())
    assert len(got) == 5
    for g, w in zip(got, want):
        assert torch.equal(g, w)


def test_oracle_head_identities():
    torch.manual_seed(2)
    sd = {k: torch.rand(v.shape, dtype=torch.float64) for k, v in LPIPS().state_dict().items()}
    a, b = torch.rand(2, 3, 64, 48, dtype=torch.float64) * 2 - 1, torch.rand(2, 3, 64, 48, dtype=torch.float64) * 2 - 1
    sd["scaling_layer.shift"], sd["scaling_layer.scale"] = LPIPS().state_dict()["scaling_layer.shift"].double(), \
        LPIPS().state_dict()["scaling_layer.scale"].double()
    assert torch.equal(lpips_oracle.lpips(sd, a, a), torch.zeros(2, 1, 1, 1, dtype=torch.float64))
    ab, ba = lpips_oracle.lpips(sd, a, b), lpips_oracle.lpips(sd, b, a)
    assert ab.shape == (2, 1, 1, 1) and bool((ab > 0).all())
    assert torch.allclose(ab, ba, rtol=1e-14, atol=0)


def test_lpips_tap_struct_layout(built_lib):
    c_names = ["feat", "weight", "H", "W", "C"]
    body = "".join(f'printf("%zu ", offsetof(b200dn_lpips_tap, {n}));' for n in c_names)
    body += 'printf("%zu", sizeof(b200dn_lpips_tap));'
    src = f'#include "b200dn.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(){{{body}return 0;}}'
    exe = ROOT / "vub_image_denoising_b200" / "build" / "offsets_lpips_tap"
    exe.parent.mkdir(exist_ok=True)
    subprocess.run(["gcc", "-x", "c", "-", "-I", str(ROOT / "include"), "-o", str(exe)], input=src, text=True, check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert [getattr(_lib.LpipsTap, n).offset for n, _ in _lib.LpipsTap._fields_] == vals[:-1]
    assert ctypes.sizeof(_lib.LpipsTap) == vals[-1]
    taps = (_lib.LpipsTap * 5)()
    for t, c, hw in zip(taps, perceptual.CHNS, (63 * 63, 31 * 31, 15 * 15, 15 * 15, 15 * 15)):
        t.feat[0], t.weight, t.H, t.W, t.C = 16, 16, hw, 1, c
    # 64-pixel blocks per tap: 63, 16, 4, 4, 4 -> 91 fp64 partials per image pair
    assert built_lib.b200dn_lpips_head_workspace_bytes(taps, 5, 2) == 2 * 91 * 8
    taps[1].C = 12
    assert built_lib.b200dn_lpips_head_workspace_bytes(taps, 5, 2) == 0
