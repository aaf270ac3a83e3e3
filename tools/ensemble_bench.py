"""x8 geometric self-ensemble on the GPU, with the card's name, power limit and max SM clock read in the same run.

1. b200dn_dihedral_expand / _reduce on 256 x 3 x 256^2 fp32 (201 MB in, 1.6 GB of groups: far larger than L2), in
   TB/s of the bytes each kernel must move (9 x the input: one read + eight writes, or eight reads + one write), next
   to a device-to-device copy of the group buffer (1.6 GB read + 1.6 GB written).  The same at 250^2 (W % 4 != 0:
   32-bit accesses).
2. self_ensemble(RDUNet(128)) at B = 8 against one forward at 8B = 64 (256^2, bf16): the difference is expand + reduce.
3. ms per ensembled sample of the sampler (RDUNet_T(32), T = 20, 256^2, fp16) at B = 1 and 2, next to plain
   improved_sampling at the same B.  Random weights: the times do not depend on their values.

python tools/ensemble_bench.py [iters=20]"""
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import vub_image_denoising_b200 as b2  # noqa: E402

ITERS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
dev = "cuda"


def time_ms(fn, iters=ITERS, warmup=3):
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


def kernels(L, B, C, H, W):
    x = torch.randn(B, C, H, W, device=dev)
    n = 4 * x.numel()
    buf = torch.empty(2 * n, device=dev)
    out = torch.empty_like(x)
    dst = torch.empty_like(buf)
    s = torch.cuda.current_stream().cuda_stream
    nbytes = 9 * x.numel() * 4

    def expand():
        L.b200dn_dihedral_expand(x.data_ptr(), B, C, H, W, buf.data_ptr(), buf[n:].data_ptr(), s)

    def reduce():
        L.b200dn_dihedral_reduce(buf.data_ptr(), buf[n:].data_ptr(), B, C, H, W, out.data_ptr(), s)

    t_copy = time_ms(lambda: dst.copy_(buf))
    copy_rate = 2 * buf.numel() * 4 / t_copy / 1e9
    print(f"{B} x {C} x {H} x {W} ({x.numel() * 4 / 1e6:.0f} MB in, {9 * x.numel() * 4 / 1e9:.2f} GB moved per kernel)")
    print(f"  device copy of the groups: {t_copy:8.3f} ms  {copy_rate:6.2f} TB/s")
    for name, fn in (("dihedral_expand", expand), ("dihedral_reduce", reduce)):
        t = time_ms(fn)
        rate = nbytes / t / 1e9
        print(f"  {name}:           {t:8.3f} ms  {rate:6.2f} TB/s = {rate / copy_rate:.2f} of the copy rate")


def main():
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(f"device: {name}, power limit / max SM clock: {q.stdout.strip() or 'unavailable'}")
    L = b2.lib()
    kernels(L, 256, 3, 256, 256)
    kernels(L, 256, 3, 250, 250)

    torch.manual_seed(0)
    net = b2.RDUNet(base_filters=128).to(dev).eval()
    x8 = torch.rand(8, 3, 256, 256, device=dev) * 2 - 1
    x64 = torch.rand(64, 3, 256, 256, device=dev) * 2 - 1
    with torch.no_grad():
        # the power-capped clock drifts by about 1 % between windows: alternate the two arms and compare pair by pair
        pairs = [(time_ms(lambda: b2.self_ensemble(net, x8), iters=10), time_ms(lambda: net(x64), iters=10))
                 for _ in range(4)]
        xk = x8.clone()
        buf = b2.ops.dihedral_expand(xk)
        y = net(buf.view(64, 3, 256, 256))
        t_k = (time_ms(lambda: b2.ops.dihedral_expand(xk), iters=50)
               + time_ms(lambda: b2.ops.dihedral_reduce(y[:32], y[32:]), iters=50))
    print(f"RDUNet(128), 256^2, {net.precision}, alternating windows of 10 calls (ms):")
    for t_ens, t_fwd in pairs:
        print(f"  self_ensemble at B = 8 {t_ens:.2f}, one forward at B = 64 {t_fwd:.2f}, difference {t_ens - t_fwd:+.2f}")
    print(f"  expand + reduce alone {t_k:.3f} ms")

    torch.manual_seed(0)
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=32), timesteps=20).to(dev).eval()
    for B in (1, 2):
        y = torch.rand(B, 3, 256, 256, device=dev) * 2 - 1
        t_plain = time_ms(lambda: dm.improved_sampling(y), iters=10)
        t_ens = time_ms(lambda: b2.self_ensemble(dm, y), iters=10)
        print(f"sampler RDUNet_T(32), T = 20, 256^2, {dm.precision}, B = {B}: improved_sampling {t_plain / B:.2f} ms per "
              f"sample, self_ensemble {t_ens / B:.2f} ms per ensembled sample ({t_ens / t_plain:.2f} x a plain call)")


if __name__ == "__main__":
    main()
