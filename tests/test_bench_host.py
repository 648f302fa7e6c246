"""bench.py's host-side logic (CPU): the reference arm runs without the product library, the CPU sample covers the whole frame,
the profile digest is tied to the kernel sources it was captured from, bad arguments are refused.  On the GPU: what --dump-outputs
writes is the film of the last timed step."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402


def test_cpu_sample_is_a_strided_cover_of_the_whole_frame():
    wl = bench.WORKLOADS["scene19_4k"]
    k, spp, n_pix = bench.cpu_sample(wl, 5.0e6)
    assert spp == 64 and k >= 2 and n_pix == ((3840 + k - 1) // k) * ((2160 + k - 1) // k)
    assert 0.4 * 5.0e6 <= n_pix * spp <= 2.5 * 5.0e6
    # a frame too small to fill the budget: every pixel, more samples
    k, spp, n_pix = bench.cpu_sample(bench.WORKLOADS["scene3_test"], 1.0e7)
    assert k == 1 and n_pix == 200 * 150 and 64 < spp <= 512


def test_reference_arm_runs_without_libtcpt(built):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "scene3_test", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "Mrays/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["loaded_native"] == ["liboracle.so"]                       # the product library is never mapped by this arm
    assert line["config"]["reference_arm_paths_per_step"] > 0 and 1.5 < line["rays_per_path"] < 8.0


def test_profile_digest_names_the_kernel_sources_it_came_from():
    doc = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
    assert set(doc["kernels"]) >= {"k_trace_fused", "k_shade", "k_generate", "k_film"}
    assert len(doc["kernel_source_sha"]) == 16 and doc["workload"] == "scene19_4k"
    t, s = doc["kernels"]["k_trace_fused"], doc["kernels"]["k_shade"]
    rays = doc["closest_rays"] + doc["shadow_rays"]
    assert 48.0 <= t["dram_bytes"] / rays <= 120.0                          # measured bytes per ray can only exceed the algorithmic 48
    assert 150.0 <= s["dram_bytes"] / doc["closest_rays"] <= 400.0
    assert t["launches"] == 17 and t["fadd"] > 0 and t["fmul"] > 0
    assert len(bench.kernel_source_sha()) == 16


def test_argument_checks():
    for argv, msg in ((["--steps", "0"], "--steps must be at least 1"), (["--impl", "reference", "--dump-outputs", "out"], "--dump-outputs")):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *argv], capture_output=True, text=True, timeout=120, cwd=str(ROOT))
        assert r.returncode == 2 and msg in r.stderr, r.stderr[-2000:]


def test_dump_sample_is_fixed():
    a = bench.sample_rows(3840 * 2160, 1 << 20)
    assert np.array_equal(a, bench.sample_rows(3840 * 2160, 1 << 20))
    assert len(a) == 1 << 20 and np.all(np.diff(a) > 0) and a[-1] < 3840 * 2160
    assert np.array_equal(bench.sample_rows(30000, 1 << 20), np.arange(30000))      # a small output is written whole


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(bundle_factory, tmp_path):
    """--steps 3 --warmup 1 at 4 sample indices per step: the timed steps are 1..3, the last one renders sample indices [12, 16)."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "scene3_test", "--steps", "3", "--warmup", "1", "--spp-per-step", "4",
                        "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["counts_rank0"]["paths"] == 3 * 200 * 150 * 4
    assert sorted(p.name for p in tmp_path.iterdir()) == ["accumulators.npy"]
    got = np.load(tmp_path / "accumulators.npy")
    assert got.dtype == np.float32 and got.shape == (200 * 150, 3)
    want = bundle_factory(3, 200, 150).image("mis", 512).render("sobol", spp_begin=12, spp_end=16).accumulators.reshape(-1, 3)
    assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max())
