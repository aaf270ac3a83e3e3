"""Achieved HBM GB/s of the bandwidth-bound kernels (CUDA events, inputs larger than L2) vs MEASURED_PEAKS.json."""
import json
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import vub_image_denoising_b200 as b2  # noqa: E402

peak = 6451.5
p = ROOT / "MEASURED_PEAKS.json"
if p.exists():
    peak = json.loads(p.read_text()).get("hbm_gbs", peak)
dev = "cuda"


def timeit(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def report(name, ms, nbytes):
    gbs = nbytes / ms / 1e6
    print(f"  {name:44s} {ms * 1e3:9.1f} us  {nbytes / 1e6:9.1f} MB  {gbs:8.1f} GB/s  {gbs / peak * 100:5.1f}% of measured {peak:.0f}", flush=True)


print("device:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                capture_output=True, text=True).stdout.strip(), flush=True)
B = 256   # 256 patches of 256x256x3: 201 MB per fp32 tensor (> 126 MB L2)
n = B * 3 * 256 * 256
x, u1, u2, y = (torch.rand(B, 3, 256, 256, device=dev) for _ in range(4))
y2 = torch.empty_like(y)
report("device copy (1 read + 1 write fp32)", timeit(lambda: y2.copy_(x)), 2 * 4 * n)
report("sampler_step (4 reads + 1 write fp32)", timeit(lambda: torch.ops.b200dn.sampler_step(x, u1, u2, y, 0.3, 0.7, 0.35, 0.65)), 5 * 4 * n)
report("psnr sse (2 reads fp32)", timeit(lambda: b2.metrics.batch_sse(x, y)), 2 * 4 * n)
xs, ys = x.view(-1, 256, 256), y.view(-1, 256, 256)
report("ssim (2 reads fp32)", timeit(lambda: b2.metrics.batch_ssim_planes(xs, ys, 1.0)), 2 * 4 * n)
WANG = dict(gaussian_weights=True, sigma=1.5, use_sample_covariance=False)   # 11x11 Gaussian, population covariance
report("ssim Wang Gaussian, mean (2 reads fp32)", timeit(lambda: b2.metrics.batch_ssim_planes(xs, ys, 1.0, **WANG)), 2 * 4 * n)
report("ssim Wang Gaussian + map (2 reads + 1 write fp32)",
       timeit(lambda: b2.metrics.batch_ssim_planes(xs, ys, 1.0, full=True, **WANG)), 3 * 4 * n)
report("ssim uniform 11x11, mean (2 reads fp32)", timeit(lambda: b2.metrics.batch_ssim_planes(xs, ys, 1.0, win_size=11)), 2 * 4 * n)
# stock PyTorch fp32 (cuDNN, TF32 off) of the Wang mean: separable F.conv2d of the five products on the valid region
torch.backends.cudnn.allow_tf32 = False
g = torch.tensor(b2.metrics._gaussian_taps(1.5, 5), dtype=torch.float32, device=dev)


def torch_wang():
    P = xs.shape[0]
    t = torch.stack([xs, ys, xs * xs, ys * ys, xs * ys], 1).view(5 * P, 1, 256, 256)
    f = F.conv2d(F.conv2d(t, g.view(1, 1, -1, 1)), g.view(1, 1, 1, -1)).view(P, 5, 246, 246)
    ux, uy, uxx, uyy, uxy = f.unbind(1)
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    S = ((2 * ux * uy + C1) * (2 * (uxy - ux * uy) + C2)) / ((ux * ux + uy * uy + C1) * (uxx - ux * ux + uyy - uy * uy + C2))
    return S.mean(dim=(1, 2), dtype=torch.float64)


report("ssim Wang mean, stock PyTorch fp32 F.conv2d (2 reads fp32)", timeit(torch_wang), 2 * 4 * n)
diff = float((torch_wang() - b2.metrics.batch_ssim_planes(xs, ys, 1.0, **WANG)).abs().max())
print(f"  Wang mean: stock PyTorch vs ssim_window_kernel, max |diff| over {xs.shape[0]} planes {diff:.2e}", flush=True)
report("welch psd nperseg=256 (1 read fp32, 129 floats out / image)", timeit(lambda: b2.metrics.welch(x.flatten(1))), 4 * n)
clean_u8 = torch.randint(0, 256, (B, 256, 256, 3), dtype=torch.uint8, device=dev)
sig = torch.full((B,), 25.0, device=dev)
report("gauss_noise_u8 (1 B read, u8 + 2 fp32 written)", timeit(lambda: b2.noise.add_gaussian_noise(clean_u8, sig, seed=1)), n * (1 + 1 + 4 + 4))
report("gauss_noise_u8 (1 B read, 1 fp32 written)", timeit(lambda: b2.noise.add_gaussian_noise(clean_u8, sig, seed=1, return_u8=False, return_clean=False)), n * (1 + 4))
report("u8_to_normalized (1 B read, 4 B written)", timeit(lambda: b2.noise.u8_to_normalized(clean_u8)), n * 5)
report("normalized_to_u8 (4 B read, 1 B written)", timeit(lambda: b2.noise.normalized_to_u8(x)), n * 5)
net = b2.RDUNet(base_filters=128).to(dev).eval()
plan = net.plan(64, 256, 256)
xin = x[:64].contiguous()
out = torch.empty_like(xin)
I0 = plan.bufs["I0"]
L = b2._lib.lib()


def conv_in():
    hi, lo = I0.ptrs()
    L.b200dn_conv_in(xin.data_ptr(), 64, 3, None, 0, 0, 0, 64, 256, 256, 128, plan.in_w, plan.in_b, plan.in_s, plan.prec, hi, lo, I0.ctot,
                     None, torch.cuda.current_stream().cuda_stream)


report("conv_in F=128 B=64 (12 B read, 256 B written /px)", timeit(conv_in), 64 * 65536 * (12 + 256))
