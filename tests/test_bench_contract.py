"""bench.py contract checks: the reference arm (the oracle port timed on the host cores) prints ONE JSON line with the
keys a consumer of the benchmark reads, on the B200 arm's metric / unit / workload; --dump-outputs writes a bounded,
reproducible copy of what the timed path computed (on the GPU)."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS=str(min(8, os.cpu_count() or 1)))
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "denoised_mpix_per_s" and d["unit"] == "MPix/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "RDUNet(base_filters=128)" in d["config"]["workload"]


def test_non_zero_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env, cwd=str(ROOT))
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_keep_a_seeded_sample_within_the_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    rng = np.random.default_rng(0)
    arrays = {"denoised": rng.random((40, 3, 16, 16), dtype=np.float32), "psnr": rng.random(40)}   # 122 kB of images
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["denoised.npy", "denoised_images.npy", "psnr.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 100_000
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    idx = np.load(tmp_path / "a" / "denoised_images.npy")
    got = np.load(tmp_path / "a" / "denoised.npy")
    assert idx.dtype == np.float64 and 20 < len(idx) < 40 and np.all(np.diff(idx) > 0)
    assert got.dtype == np.float32 and np.array_equal(got, arrays["denoised"][idx.astype(int)])
    assert np.array_equal(np.load(tmp_path / "a" / "psnr.npy"), arrays["psnr"])
    bench.dump_outputs(str(tmp_path / "c"), {"denoised": arrays["denoised"][:8]})      # within the budget: whole
    assert [p.name for p in (tmp_path / "c").iterdir()] == ["denoised.npy"]
    assert np.array_equal(np.load(tmp_path / "c" / "denoised.npy"), arrays["denoised"][:8])


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(built_lib, tmp_path):
    """--dump-outputs writes the last timed step's denoised batch and metrics; the same arguments give the same bits."""
    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "3",
                            "--base-filters", "32", "--skip-diffusion", "--skip-cpu", "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=600, cwd=str(ROOT))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == 2
        dumps.append({p.stem: np.load(p) for p in (tmp_path / run).iterdir()})
    a, b = dumps
    assert sorted(a) == ["denoised", "psnr", "ssim"]
    assert a["denoised"].shape == (3, 3, 256, 256) and a["denoised"].dtype == np.float32
    assert a["psnr"].shape == a["ssim"].shape == (3,) and a["psnr"].dtype == np.float64
    assert np.isfinite(a["denoised"]).all() and np.isfinite(a["psnr"]).all() and np.all(np.abs(a["ssim"]) <= 1)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_launch_list_summariser(tmp_path):
    """tools/summarize_launches.py: one bench step = the launches between two noise-kernel launches."""
    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"'
    rows = []
    names = ["gauss_noise_kernel<3>(x)", "void b200dn::igemm::<unnamed>::conv3x3_slab2_kernel<(int)1>(b200dn::igemm::KParams)",
             "b200dn::ssim_kernel(const float *)", "gauss_noise_kernel<3>(x)", "void b200dn::igemm_kernel<2, 1>(b200dn::igemm::KParams)",
             "gauss_noise_kernel<3>(x)"]
    for i, n in enumerate(names):
        for m, u, v in (("gpu__time_duration.sum", "ns", 1000 * (i + 1)), ("dram__bytes_read.sum", "byte", 100),
                        ("dram__bytes_write.sum", "byte", 50)):
            rows.append(f'"{i}","1","python","h","{n}","1","7","(256, 1, 1)","(148, 1, 1)","0","10.0","s","{m}","{u}","{v}"')
    src = tmp_path / "l.csv"
    src.write_text("==PROF== x\n" + hdr + "\n" + "\n".join(rows) + "\n")
    out = tmp_path / "o"
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "summarize_launches.py"), str(src), str(out)],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    s = json.loads((tmp_path / "o_summary.json").read_text())
    # last complete step = launches 3 and 4; launch 4 is the tensor-core kernel
    assert s["step_total_us"] == 4.0 + 5.0
    assert s["tensor_core_kernels"]["launches"] == 1 and s["tensor_core_kernels"]["dram_bytes_per_launch"] == 150
    assert "igemm_kernel<2, 1>" in s["by_kernel"]
