"""DISTS time per 64 image pairs at 256 x 256: the B200 path (b2.perceptual.DISTS, bf16x3 trunk) next to stock PyTorch
fp32 (torchvision VGG16 features on cuDNN with default TF32 settings, the L2 pooling and the DISTS head as DISTS_pt.py
writes them) on the same GPU, with the card's name and power limit read in the same run.  Random weights: the time does
not depend on their values.

python tools/dists_bench.py [N=64] [H=256] [iters=20]"""
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import vub_image_denoising_b200 as b2  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 64
H = int(sys.argv[2]) if len(sys.argv) > 2 else 256
ITERS = int(sys.argv[3]) if len(sys.argv) > 3 else 20
dev = "cuda"
STAGES = ((0, 4), (4, 9), (9, 16), (16, 23), (23, 30))
POOLS = (4, 9, 16, 23)


def stock_dists(features, filters, mean, std, alpha, beta):
    """DISTS_pytorch.DISTS.forward as the package computes it, in fp32 eager PyTorch."""
    chns = [3, 64, 128, 256, 512, 512]

    def run(x):
        out, h = [x], (x - mean) / std
        for a, b in STAGES:
            for i in range(a, b):
                if i in POOLS:
                    h = (F.conv2d(h ** 2, filters[i], stride=2, padding=1, groups=h.shape[1]) + 1e-12).sqrt()
                else:
                    h = features[i](h)
            out.append(h)
        return out

    def fn(x, y):
        f0, f1 = run(x), run(y)
        w_sum = alpha.sum() + beta.sum()
        al, be = torch.split(alpha / w_sum, chns, dim=1), torch.split(beta / w_sum, chns, dim=1)
        d1 = d2 = 0
        for k in range(len(chns)):
            mx, my = f0[k].mean([2, 3], keepdim=True), f1[k].mean([2, 3], keepdim=True)
            s1 = (2 * mx * my + 1e-6) / (mx ** 2 + my ** 2 + 1e-6)
            d1 = d1 + (al[k] * s1).sum(1, keepdim=True)
            vx = ((f0[k] - mx) ** 2).mean([2, 3], keepdim=True)
            vy = ((f1[k] - my) ** 2).mean([2, 3], keepdim=True)
            cov = (f0[k] * f1[k]).mean([2, 3], keepdim=True) - mx * my
            s2 = (2 * cov + 1e-6) / (vx + vy + 1e-6)
            d2 = d2 + (be[k] * s2).sum(1, keepdim=True)
        return 1 - (d1 + d2).squeeze()
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
    m = b2.perceptual.DISTS()
    tv = torchvision.models.vgg16(weights=None).features[:30]
    sd = m.state_dict()
    convs = [idx for stage in b2.perceptual.DISTS_CONVS for idx, _, _ in stage]
    for s, (a, b) in enumerate(STAGES):
        for idx in convs:
            if a <= idx < b:
                sd[f"stage{s + 1}.{idx}.weight"] = tv[idx].weight.detach()
                sd[f"stage{s + 1}.{idx}.bias"] = tv[idx].bias.detach()
    sd["alpha"], sd["beta"] = torch.rand_like(sd["alpha"]), torch.rand_like(sd["beta"])
    m.load_state_dict(sd)
    m = m.to(dev)
    tv = tv.to(dev).eval()
    filters = {idx: sd[f"stage{s + 2}.{idx}.filter"].to(dev) for s, idx in enumerate(POOLS)}
    stock = stock_dists(tv, filters, sd["mean"].to(dev), sd["std"].to(dev), sd["alpha"].to(dev), sd["beta"].to(dev))
    a = torch.rand(N, 3, H, H, device=dev)
    b = (a + 0.1 * torch.randn_like(a)).clamp(0, 1)
    sizes = [(H, H)] + b2.perceptual.dists_stage_sizes(H, H)[1:]
    gflop = 2 * N * sum(2 * cout * cin * 9 * sizes[s][0] * sizes[s][1]
                        for s, stage in enumerate(b2.perceptual.DISTS_CONVS) for _, cin, cout in stage) / 1e9
    with torch.no_grad():
        t_b2 = time_ms(lambda x, y: m(x, y), a, b)
        t_stock = time_ms(stock, a, b)
        d = (m(a, b).double() - stock(a, b).double()).abs().max()
    print(f"DISTS, {N} pairs at {H}x{H} ({gflop:.1f} GFLOP of convolutions per call), {ITERS} timed calls")
    print(f"  B200 path (bf16x3 trunk):  {t_b2:8.3f} ms   {gflop / t_b2:8.1f} TFLOP/s")
    print(f"  stock PyTorch fp32 eager:  {t_stock:8.3f} ms   {gflop / t_stock:8.1f} TFLOP/s")
    print(f"  max |B200 - stock| = {float(d):.3g}")


if __name__ == "__main__":
    main()
