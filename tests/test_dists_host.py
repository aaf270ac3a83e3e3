"""CPU: the DISTS module's parameter layout (DISTS_pytorch.DISTS().state_dict()), its L2 pooling taps, the oracle's
trunk against torchvision's VGG16, the oracle's head against an explicit fp64 brute force, the C struct layout and the
errors raised before any kernel runs."""
import ctypes
import itertools
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import dists_oracle
from vub_image_denoising_b200 import _lib, perceptual
from vub_image_denoising_b200.perceptual import DISTS

ROOT = Path(__file__).resolve().parent.parent


def _conv(prefix, cin, cout):
    return [(prefix + ".weight", (cout, cin, 3, 3)), (prefix + ".bias", (cout,))]


# DISTS_pytorch 0.1 (not installed here; restated, unpinned): DISTS.__init__ builds stage1..stage5 from
# vgg16().features with L2pooling(channels=C) at indices 4, 9, 16, 23, then registers the mean / std buffers and the
# alpha / beta parameters; state_dict() lists a module's own parameters, then its own buffers, then its children.
DISTS_KEYS = ([("alpha", (1, 1475, 1, 1)), ("beta", (1, 1475, 1, 1)), ("mean", (1, 3, 1, 1)), ("std", (1, 3, 1, 1))]
              + _conv("stage1.0", 3, 64) + _conv("stage1.2", 64, 64)
              + [("stage2.4.filter", (64, 1, 3, 3))] + _conv("stage2.5", 64, 128) + _conv("stage2.7", 128, 128)
              + [("stage3.9.filter", (128, 1, 3, 3))] + _conv("stage3.10", 128, 256) + _conv("stage3.12", 256, 256)
              + _conv("stage3.14", 256, 256)
              + [("stage4.16.filter", (256, 1, 3, 3))] + _conv("stage4.17", 256, 512) + _conv("stage4.19", 512, 512)
              + _conv("stage4.21", 512, 512)
              + [("stage5.23.filter", (512, 1, 3, 3))] + _conv("stage5.24", 512, 512) + _conv("stage5.26", 512, 512)
              + _conv("stage5.28", 512, 512))


def test_state_dict_matches_dists_pytorch():
    m = DISTS()
    sd = m.state_dict()
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == DISTS_KEYS
    assert all(v.dtype == torch.float32 for v in sd.values())
    assert torch.equal(sd["mean"].flatten(), torch.tensor([0.485, 0.456, 0.406]))
    assert torch.equal(sd["std"].flatten(), torch.tensor([0.229, 0.224, 0.225]))
    assert m.chns == [3, 64, 128, 256, 512, 512]
    assert not any(p.requires_grad for p in m.parameters())
    full = {k: torch.rand(v.shape) for k, v in sd.items()}
    m.load_state_dict(full)
    for k, v in m.state_dict().items():
        assert torch.equal(v, full[k]), k


def test_filters_are_the_normalised_hanning_product():
    a = np.hanning(5)[1:-1]
    g = torch.Tensor(a[:, None] * a[None, :])
    g = g / torch.sum(g)
    sd = DISTS().state_dict()
    for k in ("stage2.4.filter", "stage3.9.filter", "stage4.16.filter", "stage5.23.filter"):
        assert torch.equal(sd[k], g[None, None].repeat(sd[k].shape[0], 1, 1, 1)), k
        assert torch.equal(sd[k], dists_oracle.hanning_filter(sd[k].shape[0])), k


def test_oracle_indices_are_torchvision_vgg16():
    import torchvision
    feats = torchvision.models.vgg16(weights=None).features
    assert len(feats) == 31 and isinstance(feats[30], torch.nn.MaxPool2d)
    for i, mod in enumerate(feats[:30]):
        if i in dists_oracle.CONV_INDICES:
            assert isinstance(mod, torch.nn.Conv2d) and mod.kernel_size == (3, 3) and mod.padding == (1, 1), i
        elif i in dists_oracle.POOL_INDICES:
            assert isinstance(mod, torch.nn.MaxPool2d), i
        else:
            assert isinstance(mod, torch.nn.ReLU), i
    convs = [feats[i] for i in dists_oracle.CONV_INDICES]
    want = [(idx, cin, cout) for stage in perceptual.DISTS_CONVS for idx, cin, cout in stage]
    assert [(i, c.in_channels, c.out_channels) for i, c in zip(dists_oracle.CONV_INDICES, convs)] == want
    assert perceptual.DISTS_POOLS == dists_oracle.POOL_INDICES
    # every key the oracle loads is a key of the module
    keys = set(DISTS().state_dict())
    assert {dists_oracle.key(i) + ".weight" for i in dists_oracle.CONV_INDICES} <= keys
    assert {dists_oracle.key(i) + ".filter" for i in dists_oracle.POOL_INDICES} <= keys


@pytest.mark.parametrize("hw", [(256, 256), (250, 200), (97, 131), (16, 16)])
def test_oracle_trunk_shapes(hw):
    torch.manual_seed(0)
    sd = DISTS().state_dict()
    f = dists_oracle.features(dists_oracle.vgg_features(sd, torch.float32), torch.rand(1, 3, *hw), sd)
    assert [tuple(t.shape[1:]) for t in f] == [(c, h, w) for c, (h, w) in
                                               zip(perceptual.DISTS_CHNS, [hw] + perceptual.dists_stage_sizes(*hw))]


def test_oracle_head_equals_brute_force():
    g = torch.Generator().manual_seed(4)
    chns = dists_oracle.CHNS
    sizes = [(3, 4), (3, 3), (2, 2), (2, 1), (1, 2), (1, 1)]
    f0 = [torch.rand(2, c, h, w, generator=g, dtype=torch.float64) for c, (h, w) in zip(chns, sizes)]
    f1 = [a + 0.3 * torch.rand(a.shape, generator=g, dtype=torch.float64) for a in f0]
    alpha = torch.rand(1, sum(chns), 1, 1, generator=g, dtype=torch.float64)
    beta = torch.rand(1, sum(chns), 1, 1, generator=g, dtype=torch.float64)
    got = dists_oracle.head(f0, f1, alpha, beta)
    wsum = float(alpha.sum() + beta.sum())
    for n in range(2):
        total, c0 = 0.0, 0
        for k, (x, y) in enumerate(zip(f0, f1)):
            H, W = x.shape[2:]
            for c in range(x.shape[1]):
                px = [float(x[n, c, i, j]) for i, j in itertools.product(range(H), range(W))]
                py = [float(y[n, c, i, j]) for i, j in itertools.product(range(H), range(W))]
                mx, my = sum(px) / len(px), sum(py) / len(py)
                vx = sum((v - mx) ** 2 for v in px) / len(px)
                vy = sum((v - my) ** 2 for v in py) / len(py)
                cov = sum(a * b for a, b in zip(px, py)) / len(px) - mx * my
                s1 = (2 * mx * my + 1e-6) / (mx * mx + my * my + 1e-6)
                s2 = (2 * cov + 1e-6) / (vx + vy + 1e-6)
                total += float(alpha[0, c0 + c]) / wsum * s1 + float(beta[0, c0 + c]) / wsum * s2
            c0 += x.shape[1]
        assert abs(float(got[n]) - (1 - total)) <= 1e-12
    same = dists_oracle.head(f0, f0, alpha, beta)
    assert float(same.abs().max()) <= 1e-12


def test_errors_before_any_kernel():
    m = DISTS()
    x = torch.zeros(1, 3, 64, 64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(x, x)
    with pytest.raises(RuntimeError, match="inference-only"):
        m(x, x, require_grad=True)
    m.train()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(x, x)


def test_dists_stage_struct_layout(built_lib):
    c_names = ["feat", "H", "W", "C"]
    body = "".join(f'printf("%zu ", offsetof(b200dn_dists_stage, {n}));' for n in c_names)
    body += 'printf("%zu", sizeof(b200dn_dists_stage));'
    src = f'#include "b200dn.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(){{{body}return 0;}}'
    exe = ROOT / "vub_image_denoising_b200" / "build" / "offsets_dists_stage"
    exe.parent.mkdir(exist_ok=True)
    subprocess.run(["gcc", "-x", "c", "-", "-I", str(ROOT / "include"), "-o", str(exe)], input=src, text=True, check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert [getattr(_lib.DistsStage, n).offset for n, _ in _lib.DistsStage._fields_] == vals[:-1]
    assert ctypes.sizeof(_lib.DistsStage) == vals[-1]
    stages = (_lib.DistsStage * 5)()
    for s, c, (h, w) in zip(stages, perceptual.DISTS_CHNS[1:], perceptual.dists_stage_sizes(256, 256)):
        s.feat[0], s.H, s.W, s.C = 16, h, w, c
    # 1024-pixel chunks per channel: 64 for the image and stage 1, 16, 4, 1, 1 -> slots of 5 fp64 moments per pair
    slots = 3 * 64 + 64 * 64 + 128 * 16 + 256 * 4 + 512 + 512
    assert built_lib.b200dn_dists_head_workspace_bytes(256, 256, stages, 5, 2) == 2 * slots * 5 * 8
    stages[1].C = 96
    assert built_lib.b200dn_dists_head_workspace_bytes(256, 256, stages, 5, 2) == 0
