"""LPIPS (net='alex') time per 64 image pairs at 256 x 256: the B200 path (b2.perceptual.LPIPS, bf16x3 trunk) next to
stock PyTorch fp32 (torchvision AlexNet features + the lpips head, cuDNN, default TF32 settings) on the same GPU, with
the card's name and power limit read in the same run.  Random weights: the time does not depend on their values.

python tools/lpips_bench.py [N=64] [H=256] [iters=50]"""
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import vub_image_denoising_b200 as b2  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 64
H = int(sys.argv[2]) if len(sys.argv) > 2 else 256
ITERS = int(sys.argv[3]) if len(sys.argv) > 3 else 50
dev = "cuda"


def stock_lpips(features, lins, shift, scale):
    """lpips.LPIPS(net='alex').forward as the package computes it, in fp32 eager PyTorch."""
    taps = (1, 4, 7, 9, 11)

    def run(x):
        out, x = [], (x - shift) / scale
        for i, mod in enumerate(features):
            x = mod(x)
            if i in taps:
                out.append(x)
        return out

    def fn(a, b):
        val = 0
        for f0, f1, w in zip(run(a), run(b), lins):
            n0 = f0 / (torch.sqrt(torch.sum(f0 ** 2, dim=1, keepdim=True)) + 1e-10)
            n1 = f1 / (torch.sqrt(torch.sum(f1 ** 2, dim=1, keepdim=True)) + 1e-10)
            val = val + F.conv2d((n0 - n1) ** 2, w).mean(dim=(2, 3), keepdim=True)
        return val
    return fn


def time_ms(fn, a, b):
    for _ in range(3):
        fn(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(ITERS):
        fn(a, b)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / ITERS


def main():
    import torchvision
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(f"device: {name}, power limit / max SM clock: {q.stdout.strip() or 'unavailable'}")
    torch.manual_seed(0)
    m = b2.perceptual.LPIPS()
    tv = torchvision.models.alexnet(weights=None).features[:12]
    sd = m.state_dict()
    for key, idx in (("net.slice1.0", 0), ("net.slice2.3", 3), ("net.slice3.6", 6), ("net.slice4.8", 8),
                     ("net.slice5.10", 10)):
        sd[key + ".weight"], sd[key + ".bias"] = tv[idx].weight.detach(), tv[idx].bias.detach()
    for i in range(5):
        sd[f"lin{i}.model.1.weight"] = sd[f"lins.{i}.model.1.weight"] = torch.rand_like(sd[f"lin{i}.model.1.weight"])
    m.load_state_dict(sd)
    m = m.to(dev)
    tv = tv.to(dev).eval()
    lins = [sd[f"lin{i}.model.1.weight"].to(dev) for i in range(5)]
    stock = stock_lpips(tv, lins, sd["scaling_layer.shift"].to(dev), sd["scaling_layer.scale"].to(dev))
    a = torch.rand(N, 3, H, H, device=dev) * 2 - 1
    b = (a + 0.1 * torch.randn_like(a)).clamp(-1, 1)
    gflop = 2 * N * sum(cout * cin * k * k * ho * wo for (cin, cout, k), (ho, wo) in zip(
        ((3, 64, 11), (64, 192, 5), (192, 384, 3), (384, 256, 3), (256, 256, 3)),
        [s for s in (b2.perceptual.trunk_shapes(H, H)[i] for i in (0, 1, 2, 2, 2))])) * 2 / 1e9
    with torch.no_grad():
        t_b2 = time_ms(lambda x, y: m(x, y), a, b)
        t_stock = time_ms(stock, a, b)
        d = (m(a, b).double() - stock(a, b).double()).abs().max()
    print(f"LPIPS alex, {N} pairs at {H}x{H} ({gflop:.1f} GFLOP of convolutions per call), {ITERS} timed calls")
    print(f"  B200 path (bf16x3 trunk):  {t_b2:8.3f} ms   {gflop / t_b2:8.1f} TFLOP/s")
    print(f"  stock PyTorch fp32 eager:  {t_stock:8.3f} ms   {gflop / t_stock:8.1f} TFLOP/s")
    print(f"  max |B200 - stock| = {float(d):.3g}")


if __name__ == "__main__":
    main()
