"""BM3D / CBM3D on the GPU, with the card's name, power limit and max SM clock read in the same run.

RGB 256^2 images, sigma cycling 10, 20, ..., 50 / 255 over the batch, at B = 1 and B = 64: CUDA-event time of stage 1
(hard thresholding), stage 2 (Wiener, on a given basic estimate) and the full call, per call and per image, and the
number of candidate distances each stage evaluates (one per candidate block in the clipped 39 x 39 window of every
reference block, 64 squared differences each).  Random smooth images: the groups, not the values, set the work.

python tools/bm3d_bench.py [iters=10]"""
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import vub_image_denoising_b200 as b2  # noqa: E402
from vub_image_denoising_b200 import _lib, ops  # noqa: E402

ITERS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
dev = "cuda"


def time_ms(fn, iters=ITERS, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def candidates(H, W):
    """candidate blocks over all reference blocks of one image (the reference itself excluded)"""
    def per_axis(n):
        refs = sorted(set(range(0, n - 7, 3)) | {n - 8})
        return [min(n - 8, r + 19) - max(0, r - 19) + 1 for r in refs]
    rows, cols = per_axis(H), per_axis(W)
    return sum(a * b - 1 for a in rows for b in cols)


def main():
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(f"device: {name}, power limit / max SM clock: {q.stdout.strip() or 'unavailable'}")
    H = W = 256
    n_cand = candidates(H, W)
    print(f"{H}x{W}: {n_cand / 1e6:.3f} M candidate distances per image and stage "
          f"({n_cand * 64 / 1e9:.3f} G squared differences)")
    torch.manual_seed(0)
    for B in (1, 64):
        clean = torch.nn.functional.avg_pool2d(torch.rand(B, 3, H + 7, W + 7, device=dev), 8, stride=1)
        sig = torch.tensor([(10 + 10 * (b % 5)) / 255 for b in range(B)], device=dev)
        z = (clean + sig.view(B, 1, 1, 1) * torch.randn(B, 3, H, W, device=dev)).contiguous()
        basic = ops.bm3d(z, sig, None, _lib.BM3D_HARD_THRESHOLDING, False)[0]
        t1 = time_ms(lambda: ops.bm3d(z, sig, None, _lib.BM3D_HARD_THRESHOLDING, False))
        t2 = time_ms(lambda: ops.bm3d(z, sig, basic, _lib.BM3D_ALL_STAGES, False))
        tf = time_ms(lambda: b2.bm3d.bm3d_rgb(z, sig))
        print(f"B = {B:2d} RGB {H}x{W}: stage 1 {t1:9.3f} ms ({t1 / B:7.3f} ms/image), stage 2 {t2:9.3f} ms "
              f"({t2 / B:7.3f} ms/image), full call {tf:9.3f} ms ({tf / B:7.3f} ms/image); "
              f"{B * n_cand * 64 / (t1 * 1e-3) / 1e12:.2f} T squared differences/s through stage 1")


if __name__ == "__main__":
    main()
