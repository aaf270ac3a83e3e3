#!/usr/bin/env python
"""bench.py — the headline benchmark of the B200-native RDUNet denoising hot path.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    (the reference's CPU path = the oracle port)

Metric (BASELINE.json): denoised MPix/s, RDUNet(base_filters=128) bf16 inference on batches of 64
256x256 RGB patches, sigma cycling over {10,20,30,40,50}, PSNR/SSIM evaluated on device.
One "step" = one batch through the hot path: device noise synthesis from the clean uint8 patches ->
RDUNet forward (1 ingest conv + the plan's tcgen05 launches: 68 convolutions, the four of a DenoisingBlock in one
chained launch where the plan chains them) -> PSNR + SSIM reductions.
`value` is timed with the clean batch resident in HBM; `e2e` runs the same step from pinned HOST buffers
with the H2D copy of the patches and the D2H copy of the denoised batch + metrics inside the timed region
(copies on two side streams, double-buffered, so they overlap the neighbouring steps' compute).
Each rank processes its own batch (weak scaling, NO collective inside the timed region: patches are independent
units); every rank accumulates its metric sums on device and ONE NCCL all-reduce combines them after the timed
region (SURVEY.md §8 e), so the N-GPU curve measures replica independence, not communication.
The `diffusion` key carries the second half of BASELINE.json's metric, ms per diffusion sample
(DiffusionModel(RDUNet_T(32), T=20).improved_sampling, 256x256): device-timed value, roofline, an end-to-end number
from pinned host buffers, batch-1 latencies, and for N > 1 both the weak (16 samples per GPU) and the strong
(16 samples split over the GPUs, BASELINE config 3) reading.
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (denoised batch, per-image PSNR / SSIM, and
the diffusion samples of the last timed sampler call) as DIR/<name>.npy, so that two builds can be compared output for
output: every input is seeded, so the same arguments give the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SIGMAS = (10.0, 20.0, 30.0, 40.0, 50.0)
PATCH = 256
MPIX_PER_PATCH = PATCH * PATCH / 1e6
DUMP_BYTES = 64_000_000          # all files --dump-outputs writes, headers included


def synthetic_clean_u8(batch: int, seed: int = 1234) -> np.ndarray:
    """Image-like synthetic patches: uniform noise low-passed with a 9x9 box (SURVEY.md §8 d), as uint8 HWC."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(batch, 3, PATCH, PATCH, generator=g)
    x = torch.nn.functional.pad(x, (4, 4, 4, 4), mode="reflect")
    x = torch.nn.functional.avg_pool2d(x, 9, stride=1)
    x = (x - x.amin(dim=(1, 2, 3), keepdim=True)) / (x.amax(dim=(1, 2, 3), keepdim=True) - x.amin(dim=(1, 2, 3), keepdim=True))
    return (x * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous().numpy()


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each float32 / float64 array as <out_dir>/<name>.npy.  If everything together would exceed DUMP_BYTES, each
    batch of images (ndim > 1) keeps the same fixed, seeded sample of its images, whose indices go to <name>_images.npy."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    images = {k: a for k, a in arrays.items() if a.ndim > 1}
    fixed = sum(a.nbytes for k, a in arrays.items() if k not in images) + 2 * 128 * len(arrays)   # 128-byte .npy headers
    image_bytes = sum(a.nbytes + 8 * a.shape[0] for a in images.values())                         # + float64 index
    keep = min(1.0, (DUMP_BYTES - fixed) / image_bytes) if images else 1.0
    for name, a in arrays.items():
        if name in images and keep < 1.0:
            idx = np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * keep), replace=False))
            np.save(d / f"{name}_images.npy", idx.astype(np.float64))
            a = a[idx]
        np.save(d / f"{name}.npy", a)


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "hbm_gbs": d.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (sustained bf16: the kernels are timed inside a long step)"}
    return {"bf16_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons through NVML while the timed region runs."""

    def __init__(self, device: torch.device, period: float = 0.1):
        super().__init__(daemon=True)
        self.period = period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(device).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device.index or 0)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------ reference arm
def cpu_reference_pass(base_filters: int, batch: int, threads: int, repeats: int, warmup: int, seed: int = 7):
    """The reference's CPU path for the same step on `batch` patches: numpy/PIL-style noise + RDUNet fp32 forward
    (oracle port of the reference modules) + host PSNR/SSIM.  Returns (seconds of every timed step, MPix/s from their
    MEAN) — the same estimator for `cpu_baseline` and for the `--impl reference` arm."""
    from oracle import metrics_oracle, noise_oracle, rdunet_oracle
    import vub_image_denoising_b200 as b2

    torch.set_num_threads(threads)
    torch.manual_seed(seed)
    sd = b2.RDUNet(base_filters=base_filters).state_dict()       # same seeded random-init weights as the GPU arm
    clean_u8 = synthetic_clean_u8(batch)
    sig = np.array([SIGMAS[i % len(SIGMAS)] for i in range(batch)], dtype=np.float32)
    times = []
    with torch.no_grad():
        for it in range(warmup + repeats):
            t0 = time.perf_counter()
            _, noisy, clean = noise_oracle.degrade(clean_u8, sig, seed=it)
            out = rdunet_oracle.rdunet_forward(sd, torch.from_numpy(noisy)).numpy()
            for i in range(batch):
                metrics_oracle.calculate_psnr(clean[i], out[i], 1.0)
                metrics_oracle.structural_similarity(clean[i], out[i], data_range=1.0, channel_axis=0)
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
    return times, batch * MPIX_PER_PATCH / float(np.mean(times))


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample_batch = 1
    times, _ = cpu_reference_pass(128, sample_batch, cores, repeats=args.steps, warmup=min(args.warmup, 1))
    ms = 1e3 * float(np.mean(times))
    value = sample_batch * MPIX_PER_PATCH / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "denoised_mpix_per_s", "value": value, "unit": "MPix/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "RDUNet(base_filters=128) bf16 inference, batch 64 x 256x256 RGB per GPU, "
                               "sigma cycling {10,20,30,40,50}, noise synthesis + PSNR/SSIM on device",
                   "global_batch": sample_batch, "patch": PATCH, "note": "reference CPU path of that workload (oracle port of the "
                   "reference's PyTorch modules in fp32 + numpy/scipy metrics) on the host cores; each step = 1 patch of the "
                   "64-patch batch (bounded sample)"},
        "cpu_baseline": {"value": value, "unit": "MPix/s", "cores": cores, "kind": "port",
                         "sample": f"{sample_batch} patch per step, mean of {args.steps} steps after "
                                   f"{min(args.warmup, 1)} warm-up"},
        "e2e": {"value": value, "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)



# ------------------------------------------------------------------------------------ diffusion half of the metric
DIFF_T = 20
DIFF_F = 32
# SURVEY.md §8 d: 40 forwards x 96.30 GFLOP, 40 x 425 MB of layer-by-layer 16-bit traffic per sample
DIFF_FLOP_PER_SAMPLE = 40 * 96.30e9
DIFF_BYTES_PER_SAMPLE = 40 * 425e6


def _sampler_traffic_per_sample():
    """DRAM bytes per diffusion sample from the committed ncu launch list of one sampler timestep (None if absent)."""
    summ = ROOT / "profiles" / "r02_sampler_step_launches_summary.json"
    if not summ.exists():
        return None
    d = json.loads(summ.read_text())
    step_bytes = sum((k["dram_read_MB"] + k["dram_write_MB"]) * 1e6 for k in d["by_kernel"].values())
    return step_bytes * DIFF_T / 16


def _time_sampler(dm, noisy, reps, barrier):
    """(ms per call, the samples of the last timed call)."""
    import torch.distributed as dist
    for _ in range(3):
        dm.improved_sampling(noisy)
    barrier()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    for _ in range(reps):
        samples = dm.improved_sampling(noisy)
    d1.record()
    barrier()
    t = torch.tensor([d0.elapsed_time(d1) / reps], dtype=torch.float64, device=noisy.device)
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0]), samples


def diffusion_metrics(b2, dev, world, rank, clean_dev, peaks, barrier):
    """ms per diffusion sample: DiffusionModel(RDUNet_T(32), 20).improved_sampling on 256x256 (the reference's own
    evaluation width, evaluate_model.py:103-105).  Device-timed (inputs resident), MAX over ranks.
    Returns (the result dict, the samples of the last timed call of the 16-sample batch)."""
    torch.manual_seed(7)
    dm = b2.DiffusionModel(b2.RDUNet_T(base_filters=DIFF_F), timesteps=DIFF_T).to(dev).eval()
    dm.check_saturation = True        # the product default: one 4-byte flag read per call is inside the timing

    def noisy_batch(n):
        reps = (n + clean_dev.shape[0] - 1) // clean_dev.shape[0]
        src = clean_dev.repeat(reps, 1, 1, 1)[:n].contiguous()
        return b2.noise.add_gaussian_noise(src, 25.0, seed=5, return_u8=False)[1]

    res = {"metric": "ms_per_diffusion_sample", "unit": "ms", "timesteps": DIFF_T,
           "model": f"RDUNet_T(base_filters={DIFF_F})", "precision": dm.precision, "higher_is_better": False}
    # (1) the BASELINE configuration on one GPU / weak reading on N GPUs: 16 samples per GPU
    per_gpu = 16
    noisy16 = noisy_batch(per_gpu)
    ms16, samples16 = _time_sampler(dm, noisy16, 3, barrier)
    res.update({"value": ms16 / per_gpu, "batch_per_gpu": per_gpu, "ms_per_batch": ms16,
                "samples_per_s_all_gpus": world * per_gpu / (ms16 / 1e3), "scaling": "weak"})
    # roofline: the slower of the tensor and the HBM time of a sample's algorithmic work
    t_tensor = DIFF_FLOP_PER_SAMPLE / (peaks["bf16_tflops"] * 1e12)
    t_hbm = DIFF_BYTES_PER_SAMPLE / (peaks["hbm_gbs"] * 1e9)
    bound = "tensor" if t_tensor >= t_hbm else "hbm"
    t_s = ms16 / per_gpu / 1e3
    if bound == "tensor":
        ach, peak, unit = DIFF_FLOP_PER_SAMPLE / t_s / 1e12, peaks["bf16_tflops"], "TFLOP/s"
    else:
        ach, peak, unit = DIFF_BYTES_PER_SAMPLE / t_s / 1e9, peaks["hbm_gbs"], "GB/s"
    res["roofline"] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                       "roofline_ms_per_sample": max(t_tensor, t_hbm) * 1e3, "tensor_ms_per_sample": t_tensor * 1e3,
                       "hbm_ms_per_sample": t_hbm * 1e3, "hbm_gbs_achieved": DIFF_BYTES_PER_SAMPLE / t_s / 1e9,
                       "algorithmic_flops_per_sample": DIFF_FLOP_PER_SAMPLE,
                       "algorithmic_bytes_per_sample": DIFF_BYTES_PER_SAMPLE, "peak_source": peaks["source"],
                       "traffic": _sampler_traffic_per_sample(), "traffic_note": "dram__bytes_read+write of ONE sampler timestep at "
                       "B = 16 (ncu launch list, profiles/r02_sampler_step_launches_summary.json) x 20 timesteps / 16 samples",
                       "kernels": "40 x (conv_in + 68 tcgen05 convolutions, level 0 as fused blocks, levels 1-2 as chained "
                                                   "launches) + 20 x sampler_step per sample batch, "
                                                   "one CUDA graph; per-layer ncu captures under profiles/"}
    # (2) end to end through the public call with HOST buffers: pinned noisy batch -> H2D -> improved_sampling -> D2H
    host_in = noisy16.cpu().pin_memory()
    host_out = torch.empty_like(host_in).pin_memory()
    for _ in range(2):
        host_out.copy_(dm.improved_sampling(host_in.to(dev, non_blocking=True)), non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        x = host_in.to(dev, non_blocking=True)
        host_out.copy_(dm.improved_sampling(x), non_blocking=True)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["e2e"] = {"value": float(t[0]) / per_gpu, "unit": "ms", "ms_per_batch": float(t[0]),
                  "h2d_bytes_per_step": int(host_in.numel() * 4), "d2h_bytes_per_step": int(host_out.numel() * 4)}
    # (3) strong reading for N > 1 (BASELINE config 3: 16 samples split by batch over the GPUs)
    if world > 1:
        n_loc = max(1, 16 // world)
        ms_s, _ = _time_sampler(dm, noisy_batch(n_loc), 3, barrier)
        res["strong"] = {"scaling": "strong", "samples_total": n_loc * world, "batch_per_gpu": n_loc, "ms_per_batch": ms_s,
                         "ms_per_sample_per_gpu": ms_s / n_loc, "samples_per_s_all_gpus": world * n_loc / (ms_s / 1e3)}
    # (4) batch 1: the reference's own call pattern (evaluate_model.py:318, evaluate_SIDD.py:116, benchmark.py:82-90)
    ms1, _ = _time_sampler(dm, noisy_batch(1), 5, barrier)
    res["batch1"] = {"sampler_ms_per_sample": ms1,
                     "sampler_frac_of_roofline": max(t_tensor, t_hbm) * 1e3 / ms1}
    del dm
    torch.manual_seed(7)
    net = b2.RDUNet(base_filters=128).to(dev).eval()
    x1 = noisy_batch(1)
    with torch.no_grad():
        for _ in range(4):
            net(x1)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(20):
            net(x1)
        f1.record()
        barrier()
    ms_f = f0.elapsed_time(f1) / 20
    res["batch1"].update({"rdunet128_forward_ms": ms_f, "rdunet128_tflops": 1537.43e9 / (ms_f / 1e3) / 1e12,
                          "rdunet128_mpix_per_s": MPIX_PER_PATCH / (ms_f / 1e3)})
    return res, samples16


# ------------------------------------------------------------------------------------ B200 arm
def ensure_library() -> None:
    """libb200dn.so normally travels with the repo snapshot (built by __graft_entry__.build()); on a fresh checkout the
    first local rank compiles it with nvcc and the others wait for it.  There is no fallback if it cannot be built."""
    from vub_image_denoising_b200 import _build, _lib
    if _lib.lib_available():
        return
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        _build.build_lib()
        return
    t0 = time.time()
    while not (_lib.lib_available() and _build.STAMP.exists()):
        if time.time() - t0 > 600:
            raise SystemExit("libb200dn.so was not built by local rank 0 within 10 minutes")
        time.sleep(1.0)


def run_b200(args) -> None:
    import torch.distributed as dist
    ensure_library()
    import vub_image_denoising_b200 as b2
    from vub_image_denoising_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200 GPU: the product has no CPU path (use --impl reference for the CPU arm)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B, F = args.batch, args.base_filters
    peaks = load_peaks()

    torch.manual_seed(7)
    net = b2.RDUNet(base_filters=F).to(dev).eval()
    net.precision = args.precision
    clean_host = torch.from_numpy(synthetic_clean_u8(B, seed=1234 + rank)).pin_memory()
    clean_dev = clean_host.to(dev)
    sigma = torch.tensor([SIGMAS[i % len(SIGMAS)] for i in range(B)], dtype=torch.float32, device=dev)
    plan = net.plan(B, PATCH, PATCH)
    out = torch.empty((B, 3, PATCH, PATCH), dtype=torch.float32, device=dev)
    out_host = torch.empty((B, 3, PATCH, PATCH), dtype=torch.float32).pin_memory()
    met_host = torch.empty(3, dtype=torch.float64).pin_memory()
    acc = sharding.MetricAccumulator(dev)
    ev_pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]

    def step(i: int, src_u8: torch.Tensor, events=None):
        """Denoises into `out`; returns the per-image (psnr, ssim)."""
        _, noisy, clean = b2.noise.add_gaussian_noise(src_u8, sigma, seed=1000 + i, stream_id=rank, return_u8=False)
        plan.run(noisy, out, events=events)
        psnr, ssim = b2.metrics.batch_metrics(clean, out, 1.0)    # evaluate_model.py:50-51 convention
        acc.update(psnr, ssim)
        return psnr, ssim

    def step_public_api(i: int, src_u8: torch.Tensor) -> torch.Tensor:
        """The same step through the calls a user of the reference makes: module __call__ + metric functions."""
        _, noisy, clean = b2.noise.add_gaussian_noise(src_u8, sigma, seed=1000 + i, stream_id=rank, return_u8=False)
        den = net(noisy)                                           # RDUNet.forward (drop-in nn.Module call)
        psnr, ssim = b2.metrics.batch_metrics(clean, den, 1.0)
        acc.update(psnr, ssim)
        return den

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    with torch.no_grad():
        for i in range(args.warmup):
            step(i, clean_dev)
        barrier()
        # ---------------- timed region 1: inputs resident in HBM
        sampler = ClockSampler(dev)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(args.steps):
            psnr, ssim = step(i, clean_dev, events=ev_pairs[i])
        e1.record()
        barrier()
        clocks = sampler.finish()
        dumped = {}
        if args.dump_outputs and rank == 0:                        # copied before region 2 runs more steps
            dumped = {"denoised": out.cpu().numpy(), "psnr": psnr.cpu().numpy(), "ssim": ssim.cpu().numpy()}
        ms_total = e0.elapsed_time(e1)
        # device time of the tensor-core launches of a step, averaged over the timed steps
        igemm_last_ms = float(np.mean([a.elapsed_time(b) for a, b in ev_pairs]))
        red = acc.reduce()                                         # ONE all-reduce of (sum psnr, sum ssim, n)
        # ---------------- timed region 2: end to end from pinned host buffers
        # Every step copies its patches host->device and its denoised batch + metric sums device->host inside the
        # timed region.  The copies run on two side streams (one per direction, double-buffered source) so that the
        # H2D of step i+1 and the D2H of step i-1 overlap the compute of step i, as a serving loop would do.
        h2d_s, d2h_s = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        main_s = torch.cuda.current_stream(dev)
        src_bufs = [torch.empty_like(clean_dev), torch.empty_like(clean_dev)]
        n_e2e = args.steps + 2
        ev_in = [torch.cuda.Event() for _ in range(n_e2e)]
        ev_done = [torch.cuda.Event() for _ in range(n_e2e)]

        def e2e_step(i: int):
            buf = src_bufs[i % 2]
            with torch.cuda.stream(h2d_s):
                if i >= 2:
                    h2d_s.wait_event(ev_done[i - 2])               # the step that last read this buffer is done
                buf.copy_(clean_host, non_blocking=True)           # H2D of this step's patches
                ev_in[i].record(h2d_s)
            main_s.wait_event(ev_in[i])
            den = step_public_api(i, buf)
            met = acc.acc.clone()                                  # snapshot: the next step updates the accumulator
            ev_done[i].record(main_s)
            with torch.cuda.stream(d2h_s):
                d2h_s.wait_event(ev_done[i])
                out_host.copy_(den, non_blocking=True)             # D2H of the denoised batch
                met_host.copy_(met, non_blocking=True)             # D2H of the running metric sums
                den.record_stream(d2h_s)
                met.record_stream(d2h_s)

        for i in range(2):
            e2e_step(i)
        main_s.wait_stream(d2h_s)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(2, n_e2e):
            e2e_step(i)
        main_s.wait_stream(d2h_s)                                  # the last D2H is inside the timed region
        t1.record()
        barrier()
        e2e_ms_total = t0.elapsed_time(t1)

    t_ms = torch.tensor([ms_total, e2e_ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms_total = float(t_ms[0]), float(t_ms[1])
    ms_step = ms_total / args.steps
    value = world * B * MPIX_PER_PATCH / (ms_step / 1e3)
    e2e_value = world * B * MPIX_PER_PATCH / (e2e_ms_total / args.steps / 1e3)

    # roofline of the dominant kernel family: algorithmic FLOPs of the tensor-core launches / their device time
    # 2*MAC of the 68 tensor-core convolutions of one step (SURVEY.md §8 d: F = 128 -> 1537.43 - 0.45 GFLOP per image),
    # summed from the launch plan itself
    igemm_flops = sum(info["flops"] for info in plan.layer_info)
    achieved = igemm_flops / (igemm_last_ms / 1e3) / 1e12
    # DRAM traffic of the same launches from the committed ncu pass over this command (profiles/), per launch
    traffic = None
    summ = ROOT / "profiles" / "r02_bench_launches_summary.json"
    if not summ.exists():
        summ = ROOT / "profiles" / "r01_bench_launches_summary.json"
    if summ.exists() and F == 128 and B == 64:
        traffic = json.loads(summ.read_text())["tensor_core_kernels"]["dram_bytes_per_launch"]
    n_tc = len(plan.launches)
    roofline = {"bound": "tensor", "kernel": "conv3x3_slab2_kernel / conv3x3_chain_kernel (cta_group::2) + conv3x3_slab_kernel + "
                                             f"igemm_kernel ({n_tc} tcgen05 launches per step for 68 convolutions)",
                "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": achieved / peaks["bf16_tflops"], "traffic": traffic,
                "traffic_note": f"dram__bytes_read+write per launch, mean over the tensor-core launches of one step (ncu, "
                                f"profiles/{summ.name}); algorithmic layer-by-layer bytes are 124.6 GB per step = "
                                f"{124.6 / n_tc:.2f} GB per launch, so L2 already absorbs re-reads",
                "peak_source": peaks["source"],
                "algorithmic_flops_per_step": igemm_flops, "kernel_ms_per_step": igemm_last_ms,
                "kernel_share_of_step": igemm_last_ms / ms_step}

    line = {
        "metric": "denoised_mpix_per_s", "value": value, "unit": "MPix/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else args.precision, "data": "synthetic",
        "config": {"workload": f"RDUNet(base_filters={F}) {args.precision} inference, batch {B} x 256x256 RGB per GPU, "
                               "sigma cycling {10,20,30,40,50}, noise synthesis + PSNR/SSIM on device",
                   "global_batch": world * B, "patch": PATCH, "parallelism": f"batch-sharded x{world}, metric all-reduce",
                   "l2": "working set per step (>= 18 GB of activations) far exceeds the 126 MB L2; no flush needed",
                   "weights": "random init, torch.manual_seed(7)"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "MPix/s", "h2d_bytes_per_step": int(clean_host.numel()),
                "d2h_bytes_per_step": int(out_host.numel() * 4 + met_host.numel() * 8),
                "ms_per_step": e2e_ms_total / args.steps},
        "gpu_launches": args.steps * (1 + 1 + len(plan.launches) + 2),
        "roofline": roofline,
        "quality": {"mean_psnr_db": red["psnr"], "mean_ssim": red["ssim"], "images": red["count"]},
    }

    # ---------------- second half of the metric: ms per diffusion sample (RDUNet_T(32), T = 20, 256x256)
    if not args.skip_diffusion:
        del plan, out, net
        line["diffusion"], samples = diffusion_metrics(b2, dev, world, rank, clean_dev, peaks, barrier)
        if dumped:
            dumped["diffusion_samples"] = samples.cpu().numpy()
    if dumped:
        dump_outputs(args.dump_outputs, dumped)

    # ---------------- CPU baseline (rank 0, N = 1 only): the oracle port on the host cores, bounded sample
    if rank == 0 and world == 1 and not args.skip_cpu:
        cores = os.cpu_count() or 1
        times, mpix = cpu_reference_pass(F, 1, cores, repeats=2, warmup=1)
        line["cpu_baseline"] = {"value": mpix, "unit": "MPix/s", "cores": cores, "kind": "port",
                                "sample": f"1 of the {B} patches per step (RDUNet({F}) fp32 forward + noise + PSNR/SSIM), "
                                          f"mean of 2 steps after 1 warm-up, {float(np.mean(times)):.2f} s per step "
                                          "(same estimator as --impl reference)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--base-filters", type=int, default=128)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--skip-diffusion", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 path")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
