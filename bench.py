#!/usr/bin/env python3
"""bench.py — throughput of the path-integration hot path on B200 (Mrays/s, with Mpaths/s beside it).

Default workload (BASELINE.json configs[3], the configuration the metric's 1/2/4/8-GPU numbers are quoted on): scene 19 (floor +
three dragon instances: textured SimplePbr, smooth clearcoat, plastic; environment light) at 3840x2160, MIS integrator, Z-Sobol
sampler, max_depth 16, as a 4096-spp frame.  One STEP = one pass of the hot path over one batch = `--spp-per-step` sample indices
of every pixel of the frame per GPU (default 16 -> 132.7 M paths per GPU per step, 35 GB of wavefront state in HBM), film kernel
included, and at N > 1 the ONE ncclReduce of the film accumulators that libtcpt issues itself (tcpt_render_sharded_device).
Ranks render disjoint sample-index ranges of the same frame (spp-pass sharding), per-GPU work fixed as N grows: "scaling": "weak".
The fixed-total-work curve is reported next to it in `scaling_strong`; the full 4096-spp frame at N = 8 in `time_to_image`.

  value      whole-job Mrays/s, film accumulators resident in HBM, CUDA events on the launching stream, max over ranks
  e2e        the same metric through the reference-facing call RendererImage.render_sharded() -> tcpt_render_sharded() with HOST
             buffers: per step the job parameters go in and ONE complete tone-mapped frame comes back to rank 0's host memory
  roofline   dominant kernel k_trace_fused; roofline_shade, roofline_step, roofline_fp32 beside it (DESIGN.md "Measurement")
  cpu_baseline / --impl reference: the CPU restatement of the reference algorithm (oracle, kind "port": the Rust reference cannot be
             compiled in this image) on all host threads, on a strided subsample of the SAME frame (every k-th pixel in x and y)
  parity_probe  outside the timed region: N-rank film vs the 1-rank film of the same job (tile: bitwise, spp: rounding), and at
             N = 1 GPU paths of the bench frame against the oracle's

`--workload soup_1M | soup_10M | soup_100M` (BASELINE.json configs[4]) times the traversal kernels alone on synthetic triangle
soups: 16.8 M coherent primary rays and the incoherent cosine-weighted bounce rays from their hits, closest-hit and any-hit.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

WORKLOADS = {
    "scene19_4k": dict(scene=19, width=3840, height=2160, frame_spp=4096, integrator="mis", sampler="sobol"),
    "scene17_1080p": dict(scene=17, width=1920, height=1080, frame_spp=1024, integrator="mis", sampler="sobol"),
    "scene17_1080p_nocoat": dict(scene=17, width=1920, height=1080, frame_spp=1024, integrator="mis", sampler="sobol", kw={"coat": False}),
    "scene10_test": dict(scene=10, width=200, height=150, frame_spp=512, integrator="mis", sampler="sobol"),
    "scene3_test": dict(scene=3, width=200, height=150, frame_spp=512, integrator="mis", sampler="sobol"),
    "soup_1M": dict(soup=1_000_000), "soup_10M": dict(soup=10_000_000), "soup_100M": dict(soup=100_000_000),
}
KERNEL_SOURCES = ["kernels.cuh", "dtraverse.cuh", "dshade.cuh", "dcommon.cuh"]   # device code only: the host orchestration (tcpt_api.cu) changes for unrelated reasons


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="scene19_4k", choices=sorted(WORKLOADS))
    ap.add_argument("--spp-per-step", type=int, default=16)
    ap.add_argument("--max-slots", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip scaling_strong / time_to_image / parity_probe (profiling runs)")
    ap.add_argument("--strong-spp", type=int, default=128, help="total sample indices per pixel of the strong-scaling job")
    ap.add_argument("--time-to-image", action="store_true", help="render the whole frame once (default: only at N >= 8)")
    ap.add_argument("--clock-period", type=float, default=0.05, help="seconds between NVML clock samples during the timed region")
    ap.add_argument("--opt", action="append", default=[], help="developer knob: libtcpt option as name=value (tcpt_set_option), repeatable")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--max-depth", type=int, default=16, help="developer knob (what the deep bounces cost); the benchmarked configuration is 16, the reference's default")
    ap.add_argument("--soup-rays", type=int, default=4096, help="soup workloads: the primary-ray grid is N x N (4096 -> 16.8 M rays)")
    ap.add_argument("--soup-builder", default="device", choices=["device", "host"], help="soup workloads: LBVH built on the device (csrc/lbvh.cuh) or the host binned-SAH builder")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (a fixed sample of rows when the "
                         "output is large), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    return args


def sample_rows(n, k):
    """Indices of a fixed, seeded sample of k of n rows (all of them when n <= k), in ascending order."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def dump_outputs(out_dir, arrays):
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def kernel_source_sha():
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        h.update((ROOT / "toy_cpu_pathtracing_b200" / "csrc" / name).read_bytes())
    return h.hexdigest()[:16]


# ---------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML from a thread every 50 ms
    (ctypes calls into libtcpt release the GIL), nvidia-smi polling as a fallback when pynvml is unavailable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int, period: float = 0.05):
        self.index, self.rows, self.proc, self.thread, self.stop, self.period = index, [], None, None, False, period
        self.sm, self.sm_max, self.reasons = [], None, set()

    def _nvml_loop(self, nv, h):
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        while not self.stop:
            try:
                self.sm.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.reasons |= {k for k, b in bits.items() if r & b}
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it holds plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = int(vis.split(",")[self.index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        self.stop = True
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        elif self.thread:
            self.thread.join(timeout=1)

    def summary(self):
        if self.sm:
            return {"sm_mhz": int(np.median(self.sm)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        sm = [int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm), "source": "nvidia-smi"}


# ---------------------------------------------------------------- shared setup
def describe_scene(wl, **scene_kw):
    """The scene of the workload through the host mirror of the reference's construction API.  scene_kw: device=..., or
    describe_only=True (no libtcpt context: the reference arm)."""
    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import scenes
    scene = tp.Scene(**scene_kw)
    if "soup" in wl:
        cam = tp.Camera(45.0, 1024, 1024)
        scenes.load_soup(scene, cam, wl["soup"])
    else:
        cam = tp.Camera(45.0, wl["width"], wl["height"])
        scenes.load_scene(wl["scene"], scene, cam, **wl.get("kw", {}))
    return tp, scene, cam


def cpu_sample(wl, want_paths):
    """A strided subsample of the WHOLE frame: pixels (i*k, j*k), 64 consecutive sample indices each (more when the whole frame is too
    small to fill the time), so that the CPU sees the same mix of floor / dragon / sky pixels -- the same rays per path -- as the GPU arm,
    and the pixel-major order of the reference's loop (every sample of a pixel back to back, renderer.rs:120-134 -> base_renderer.rs:160):
    its cache locality is part of the CPU's speed (measured on one box: 10.6 / 11.1 / 12.5 / 12.9 Mrays/s at 4 / 6 / 9 / 11 samples per pixel)."""
    W, H = wl["width"], wl["height"]
    spp = int(min(64, wl["frame_spp"]))
    k = int(max(1, np.floor(np.sqrt(W * H * spp / max(1.0, want_paths)))))
    n_pix = ((W + k - 1) // k) * ((H + k - 1) // k)
    if k == 1 and n_pix * spp < 0.7 * want_paths:
        spp = int(min(wl["frame_spp"], max(spp, want_paths / n_pix)))
    return k, spp, n_pix


class CpuArm:
    """The reference algorithm on the host cores: the oracle port in reference-faithful mode (exhaustive traversal without t-shrinking,
    per-call instance-matrix inverses).  `optimised=True`: the same port with an ordered, t-shrinking traversal and cached inverses
    (SURVEY 8d), bit-identical film.  The oracle is test infrastructure: it is only ever the thing measured in this CPU leg."""

    def __init__(self, wl, scene_desc, cam, threads=0, optimised=False):
        from toy_cpu_pathtracing_b200 import capi   # load_tables only reads the data files; libtcpt is not loaded here
        from oracle import oracle
        self.wl, self.cam, self.threads = wl, cam, threads
        std, tab = capi.load_tables()
        self.osc = oracle.scene_from_description(scene_desc, cam.position, std, tab, faithful=not optimised, literal_build=False)
        if optimised:
            self.osc.set_optimised(True)
        self.rate = None

    def sample(self, seconds):
        wl = self.wl
        if self.rate is None:   # calibrate on a small sample first
            self.rate = 2.0e5
            st, _, _ = self._render(0.5 * self.rate)
            self.rate = st["paths"] / max(st["seconds"], 1e-6)
        st, k, spp = self._render(seconds * self.rate)
        self.rate = st["paths"] / max(st["seconds"], 1e-6)
        rays = st["closest_rays"] + st["shadow_rays"]
        ncores = self.threads if self.threads > 0 else (os.cpu_count() or 1)
        return {"mrays": rays / st["seconds"] / 1e6, "mpaths": st["paths"] / st["seconds"] / 1e6, "cores": ncores, "seconds": st["seconds"], "paths": st["paths"], "rays": rays,
                "rays_per_path": rays / max(1, st["paths"]),
                "sample": f"every {k}-th pixel in x and y of the whole {wl['width']}x{wl['height']} frame, sample indices 0..{spp - 1}: {st['paths']} paths, "
                          f"{rays / max(1, st['paths']):.3f} rays/path, {st['seconds']:.2f} s"}

    def _render(self, want_paths):
        wl = self.wl
        k, spp, _ = cpu_sample(wl, max(2000.0, want_paths))
        # the oracle's frame loop runs p.spp samples per pixel with the sampler sized for p.spp; throughput does not depend on which
        # low-discrepancy points are drawn, so the sample renders `spp` samples with the sampler sized for them
        p = self.osc.params(wl["width"], wl["height"], spp, wl["integrator"], wl["sampler"], self.cam, threads=self.threads, stride=k, max_depth=wl.get("max_depth", 16))
        _, _, st = self.osc.render(p)
        return st, k, spp


def workload_config(args, wl, world, cpu_info=None):
    W, H = wl["width"], wl["height"]
    cfg = {"workload": f"scene{wl['scene']} {W}x{H} {wl['integrator']}+{wl['sampler']} max_depth {args.max_depth}, {wl['frame_spp']}-spp frame, "
                       f"{args.spp_per_step} sample indices of every pixel per GPU per step" + (" (BASELINE.json configs[3])" if wl["scene"] == 19 else "") + (" no-coat" if wl.get("kw") else ""),
           "paths_per_gpu_per_step": W * H * args.spp_per_step, "sharding": "spp-pass", "collective": "one ncclReduce of the film accumulators per step, issued inside libtcpt",
           "cache": (f"working set (path state + ray queues, {W * H * args.spp_per_step * 304 / 1e9:.1f} GB per GPU) exceeds the 126 MB L2; no explicit flush"
                     if W * H * args.spp_per_step * 304 > 4 * 126e6 else
                     f"working set {W * H * args.spp_per_step * 304 / 1e6:.0f} MB per GPU does not exceed the 126 MB L2 by a wide margin and nothing is flushed: a test-size workload, not a bench line"),
           "assets": "procedural stand-ins (reference assets are LFS stubs)"}
    if cpu_info is not None:   # the reference arm: what one of ITS steps really covers
        cfg["reference_arm_paths_per_step"] = cpu_info["paths"]
        cfg["reference_arm_sample"] = cpu_info["sample"]
    return cfg


# ---------------------------------------------------------------- reference arm
def main_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if "soup" in wl:
        return soup_reference(args, wl)
    _, scene, cam = describe_scene(wl, describe_only=True)     # no tcpt_ctx: this arm never loads the product library
    arm = CpuArm(wl, scene.desc, cam)
    per_step = max(2.0, min(args.cpu_seconds, 120.0 / max(1, args.steps + args.warmup)))
    tot_r = tot_p = tot_s = 0.0
    info = None
    for i in range(args.warmup + args.steps):
        info = arm.sample(per_step)
        if i >= args.warmup:
            tot_r += info["rays"]; tot_p += info["paths"]; tot_s += info["seconds"]
    value = tot_r / tot_s / 1e6
    line = {"impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * tot_s / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, wl, 1, info), "mpaths_per_s": tot_p / tot_s / 1e6, "rays_per_path": tot_r / max(1.0, tot_p),
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": info["cores"], "kind": "port", "sample": info["sample"]},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "loaded_native": sorted({Path(l.split()[-1]).name for l in open("/proc/self/maps") if "libtcpt" in l or "liboracle" in l} if os.path.exists("/proc/self/maps") else [])}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------- GPU arm (scenes)
def main_gpu(args, wl):
    import ctypes as C

    import torch
    import torch.distributed as dist
    from toy_cpu_pathtracing_b200 import capi
    from toy_cpu_pathtracing_b200.multi_gpu import init_comm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))   # plumbing: barriers, max-over-ranks of the timings, the NCCL id of libtcpt's own communicator
    if "soup" in wl:
        return soup_gpu(args, wl, world, rank, local)
    tp, scene, cam = describe_scene(wl, device=local)
    ctx = scene.ctx
    for kv in args.opt:                  # before the build: some options are decided when the scene is uploaded
        name, _, val = kv.partition("=")
        ctx.set_option(name, int(val))
    t0 = time.time(); scene.build(cam); build_s = time.time() - t0
    init_comm(ctx, rank, world)          # tcpt_comm_init: the film reduce is libtcpt's own ncclReduce from here on
    W, H, S = wl["width"], wl["height"], args.spp_per_step
    SPP, TILE = capi.SHARD_MODES["spp"], capi.SHARD_MODES["tile"]
    renderer = tp.RENDERERS[wl["integrator"]](tp.RendererArgs((W, H), wl["frame_spp"], scene, cam, seed=0), max_depth=args.max_depth)
    image = tp.RendererImage(W, H, renderer)
    acc = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
    frame = torch.zeros_like(acc) if rank == 0 else None
    # a real (non-default) stream: libtcpt launches on the handle it is given, its ncclReduce and the torch events use the same
    # stream, so the CUDA events bracket exactly the kernels of the timed steps
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)

    def window(k):
        lo = (k * world * S) % wl["frame_spp"]
        return lo, min(lo + world * S, wl["frame_spp"])

    def sharded_device(mode, lo, hi, target):
        p = renderer.params(wl["sampler"], max_slots=args.max_slots, spp_begin=lo, spp_end=hi)
        ctx.check(ctx.lib.tcpt_render_sharded_device(ctx.handle, C.byref(p), mode, C.c_void_p(target.data_ptr()), C.c_void_p(stream.cuda_stream)))
        return ctx.stats()

    def step(k):
        # step k of the job: `world * S` fresh sample indices of the frame, rank r renders its S of them; one ncclReduce onto rank 0
        lo, hi = window(k)
        acc.zero_()
        st = sharded_device(SPP, lo, hi, acc)
        if rank == 0:
            frame.add_(acc)
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def over_ranks(vals):
        """(max, sum) over ranks of a list of floats."""
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world == 1:
            return list(vals), list(vals)
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        return tm.tolist(), ts.tolist()

    for k in range(args.warmup):
        step(k)
    ctx.set_option("stage_timing", 1)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    keys = ("paths", "closest_rays", "shadow_rays", "kernel_launches", "trace_launches", "shade_launches", "passes",
            "trace_closest_ms", "trace_shadow_ms", "shade_ms", "generate_ms", "film_ms", "reduce_ms")
    tot = {k: 0.0 for k in keys}
    with ClockSampler(local, args.clock_period) as clk:
        e0.record(stream)
        for k in range(args.steps):
            st = step(args.warmup + k)
            for key in keys:
                tot[key] += st[key]
        e1.record(stream)
        barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs is not None and rank == 0:
        # the film accumulators of the last timed step, reduced onto rank 0; acc is reused by everything below
        idx = torch.from_numpy(sample_rows(W * H, 1 << 20)).to(dev)
        dump_outputs(args.dump_outputs, {"accumulators": acc.view(-1, 3)[idx].cpu().numpy()})
    ctx.set_option("stage_timing", 0)
    rays_mine = tot["closest_rays"] + tot["shadow_rays"]
    mx, sm = over_ranks([ms, rays_mine, tot["paths"], tot["kernel_launches"]])   # libtcpt's own kernels only: the ncclReduce kernel of a step is NCCL's
    ms_max, rays_all, paths_all, launches_all = mx[0], sm[1], sm[2], sm[3]
    value = rays_all / (ms_max * 1e-3) / 1e6

    # ---- e2e through the reference-facing API with host buffers: ONE complete frame per step lands in rank 0's host memory
    def e2e_step(k):
        lo, hi = window(k)
        image.render_sharded(wl["sampler"], mode="spp", want_accumulators=False, spp_window=(lo, hi), max_slots=args.max_slots)
        return image.stats["closest_rays"] + image.stats["shadow_rays"]
    e2e_step(0)
    barrier()
    n_e2e = max(2, min(args.steps, 4))
    t0 = time.perf_counter(); e2e_rays = 0
    for k in range(n_e2e):
        e2e_rays += e2e_step(args.warmup + k)
    barrier()
    e2e_s = time.perf_counter() - t0
    mx, sm = over_ranks([e2e_s, float(e2e_rays)])
    e2e_value = sm[1] / mx[0] / 1e6

    extras = {}
    if not args.no_extras:
        # ---- strong scaling: a FIXED job (args.strong_spp sample indices of every pixel) split over the N ranks, both shard modes
        T = min(args.strong_spp, wl["frame_spp"])
        strong = {"total_sample_indices_per_pixel": T, "total_paths": W * H * T,
                  "what": "one fixed job split over N ranks, one ncclReduce per job; efficiency(N) = ms(1) / (N * ms(N)) against the N=1 line"}
        for mode_name, mode in (("spp", SPP), ("tile", TILE)):
            best = None
            for rep in range(2):
                acc.zero_()
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                st = sharded_device(mode, 0, T, acc)
                b.record(stream)
                barrier()
                mx, sm = over_ranks([a.elapsed_time(b), float(st["closest_rays"] + st["shadow_rays"]), float(st["paths"]), float(st["passes"])])
                if best is None or mx[0] < best["ms"]:
                    best = {"ms": mx[0], "mrays_per_s": sm[1] / mx[0] / 1e3, "mpaths_per_s": sm[2] / mx[0] / 1e3, "passes_per_rank_max": int(mx[3])}
            strong[mode_name] = best
        extras["scaling_strong"] = strong

        # ---- time to image: the whole frame through the reference-facing call, once (N >= 8 by default: 34 G paths)
        if args.time_to_image or world >= 8:
            barrier()
            t0 = time.perf_counter()
            image.render_sharded(wl["sampler"], mode="spp", want_accumulators=False, max_slots=args.max_slots)
            barrier()
            wall = time.perf_counter() - t0
            mx, sm = over_ranks([wall, float(image.stats["closest_rays"] + image.stats["shadow_rays"]), float(image.stats["paths"]), float(image.stats["render_ms"]), float(image.stats["reduce_ms"])])
            extras["time_to_image"] = {"seconds": mx[0], "frame": f"{W}x{H}, {wl['frame_spp']} spp, {wl['integrator']}+{wl['sampler']}", "paths": sm[2], "mrays_per_s": sm[1] / mx[0] / 1e6,
                                       "device_ms_max": mx[3], "reduce_ms_max": mx[4], "collectives": 1 if world > 1 else 0,
                                       "call": "RendererImage.render_sharded(mode='spp') -> tcpt_render_sharded: one host frame on rank 0"}

        # ---- parity probe (outside every timed region): the N-rank film against the 1-rank film of the same job
        probe = {}
        lo, hi = 0, min(wl["frame_spp"], max(2, world))
        shards = {}
        for mode_name, mode in (("tile", TILE), ("spp", SPP)):
            acc.zero_()
            sharded_device(mode, lo, hi, acc)
            shards[mode_name] = acc.clone() if rank == 0 else None
        barrier()
        if rank == 0:
            alone = torch.zeros_like(acc)
            p = renderer.params(wl["sampler"], max_slots=args.max_slots, spp_begin=lo, spp_end=hi)
            ctx.check(ctx.lib.tcpt_render_device(ctx.handle, C.byref(p), C.c_void_p(alone.data_ptr()), C.c_void_p(stream.cuda_stream)))
            torch.cuda.synchronize()
            scale = max(1.0, float(alone.abs().max()))
            probe = {"job": f"sample indices [{lo}, {hi}) of the bench frame, {world} rank(s) vs rank 0 alone (tcpt_render_device)",
                     "tile_bitwise_equal": bool(torch.equal(shards["tile"].view(torch.int32), alone.view(torch.int32))),
                     "spp_max_rel_err": float((shards["spp"] - alone).abs().max()) / scale, "finite": bool(torch.isfinite(alone).all())}
            del alone
        barrier()
        extras["parity_probe"] = probe

    if rank != 0:
        ctx.comm_destroy()
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- rooflines.  One extra counted step OUTSIDE the timed region gives box / triangle tests per ray.
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback (B200_PROFILING.md)"
    ctx.set_option("count_tests", 1)
    p = renderer.params(wl["sampler"], max_slots=args.max_slots, spp_begin=0, spp_end=1)
    acc.zero_()
    ctx.check(ctx.lib.tcpt_render_device(ctx.handle, C.byref(p), C.c_void_p(acc.data_ptr()), C.c_void_p(stream.cuda_stream)))
    cs = ctx.stats()
    ctx.set_option("count_tests", 0)
    rays_c = max(1, cs["closest_rays"] + cs["shadow_rays"])
    box_per_ray, tri_per_ray = cs["box_tests"] / rays_c, cs["tri_tests"] / rays_c
    clk_s = clk.summary()
    sm_mhz = clk_s["sm_mhz"] or 1965
    n_trace = max(1.0, tot["trace_launches"]); n_shade = max(1.0, tot["shade_launches"])
    trace_s = (tot["trace_closest_ms"] + tot["trace_shadow_ms"]) * 1e-3
    shade_s = tot["shade_ms"] * 1e-3
    step_s = ms * 1e-3
    stage_sum = tot["trace_closest_ms"] + tot["trace_shadow_ms"] + tot["shade_ms"] + tot["generate_ms"] + tot["film_ms"]
    # measured DRAM bytes and FP32 instruction counts per ray / per vertex / per path from the committed ncu capture of ONE step of
    # this workload (tools/ncu_digest.py -> profiles/ncu_traffic.json), valid only for the kernel sources it was captured from
    prof, prof_note = None, None
    try:
        prof = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
        if prof.get("kernel_source_sha") != kernel_source_sha():
            prof_note = f"STALE: profiles/ncu_traffic.json was captured from kernel sources {prof.get('kernel_source_sha')}, this run is {kernel_source_sha()}; re-run tools/prof.sh <tag> traffic"
            print("bench.py: " + prof_note, file=sys.stderr)
            prof = None
        elif prof.get("workload") != args.workload:
            prof_note = f"profiles/ncu_traffic.json is for workload {prof.get('workload')}"
            prof = None
    except Exception as e:  # noqa: BLE001
        prof_note = f"profiles/ncu_traffic.json unreadable: {e}"
    vertices = tot["closest_rays"]      # every extension ray ends in exactly one shading work item (hit bucket or miss bucket)
    bytes_per_ray = 48.0    # SURVEY.md 8(d): 32 B ray read + 16 B hit write (compulsory wavefront traffic; the BVH is L2 resident)
    bytes_per_vertex = 192.0
    achieved = bytes_per_ray * rays_mine / trace_s / 1e9 if trace_s > 0 else 0.0
    sh_achieved = bytes_per_vertex * vertices / shade_s / 1e9 if shade_s > 0 else 0.0
    flops_per_ray = 18.0 * box_per_ray + 64.0 * tri_per_ray + 60.0
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    fp32_model = flops_per_ray * rays_mine / trace_s / 1e12 if trace_s > 0 else 0.0
    traffic = sh_traffic = step_traffic = None
    fp32_measured = {}
    if prof:
        kt, ks = prof["kernels"].get("k_trace_fused"), prof["kernels"].get("k_shade")
        pr = max(1, prof["closest_rays"] + prof["shadow_rays"])
        if kt:
            traffic = kt["dram_bytes"] / pr * (rays_mine / n_trace)
            fl = (kt["fadd"] + kt["fmul"] + 2 * kt["ffma"]) / pr
            fp32_measured["k_trace_fused"] = {"flops_per_ray": fl, "achieved": fl * rays_mine / trace_s / 1e12, "frac": fl * rays_mine / trace_s / 1e12 / fp32_peak,
                                              "fadd_fmul_ffma_per_ray": [kt["fadd"] / pr, kt["fmul"] / pr, kt["ffma"] / pr]}
        if ks:
            pv = max(1, prof["closest_rays"])
            sh_traffic = ks["dram_bytes"] / pv * (vertices / n_shade)
            fl = (ks["fadd"] + ks["fmul"] + 2 * ks["ffma"]) / pv
            fp32_measured["k_shade"] = {"flops_per_vertex": fl, "achieved": fl * vertices / shade_s / 1e12, "frac": fl * vertices / shade_s / 1e12 / fp32_peak,
                                        "fadd_fmul_ffma_per_vertex": [ks["fadd"] / pv, ks["fmul"] / pv, ks["ffma"] / pv]}
        step_traffic = prof["total_dram_bytes"] / max(1, prof["paths"]) * (tot["paths"] / args.steps)
    line = {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, wl, world),
        "mpaths_per_s": paths_all / (ms_max * 1e-3) / 1e6, "rays_per_path": rays_all / max(1.0, paths_all),
        "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": C.sizeof(capi.RenderParams), "d2h_bytes_per_step": int(image.pixels.nbytes), "steps": n_e2e,
                "call": "RendererImage.render_sharded -> tcpt_render_sharded(job, host sRGB frame out on rank 0): shard render, one ncclReduce, Sensor::to_rgb, one D2H"},
        "gpu_launches": int(launches_all),
        "clocks": clk_s,
        "roofline": {"kernel": "k_trace_fused", "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                     "peak_source": peak_src, "bytes_per_ray": bytes_per_ray, "rays_per_launch": rays_mine / n_trace, "launches": int(n_trace),
                     "avg_launch_ms": 1e3 * trace_s / n_trace, "share_of_step": 1e3 * trace_s / stage_sum if stage_sum else None,
                     "traffic_source": (f"profiles/ncu_traffic.json ({prof.get('captured')}): measured dram bytes per ray of every k_trace_fused launch of one step, scaled to this run's rays per launch" if prof else prof_note),
                     "note": "BVH + textures are L2 resident: the kernel is instruction-issue / latency bound, see roofline_fp32"},
        "roofline_shade": {"kernel": "k_shade<B> + k_shade_all", "bound": "hbm", "achieved": sh_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": sh_achieved / hbm_peak, "traffic": sh_traffic,
                           "bytes_per_vertex": bytes_per_vertex, "vertices_per_launch": vertices / n_shade, "launches": int(n_shade), "avg_launch_ms": 1e3 * shade_s / n_shade,
                           "share_of_step": tot["shade_ms"] / stage_sum if stage_sum else None},
        "roofline_step": {"bound": "hbm", "unit": "GB/s", "peak": hbm_peak, "traffic_per_step": step_traffic, "achieved": (step_traffic / (step_s / args.steps) / 1e9) if step_traffic else None,
                          "frac": (step_traffic / (step_s / args.steps) / 1e9 / hbm_peak) if step_traffic else None, "what": "measured DRAM bytes of every kernel of one step (ncu) / live step time"},
        "roofline_fp32": {"kernels": "k_trace_fused", "achieved": fp32_model, "peak": fp32_peak, "unit": "TFLOP/s", "frac": fp32_model / fp32_peak if fp32_peak else None,
                          "flops_per_ray": flops_per_ray, "box_tests_per_ray": box_per_ray, "tri_tests_per_ray": tri_per_ray, "sm_mhz": sm_mhz,
                          "definition": "model: 18*B + 64*T + 60 flops per ray (SURVEY.md 8d); peak = 148 SM x 128 lanes x 2 x f_SM",
                          "measured": fp32_measured or None,
                          "measured_definition": "ncu smsp__sass_thread_inst_executed_op_{fadd,fmul,ffma}_pred_on.sum per ray / vertex (fadd + fmul + 2 ffma; --fmad=false, so nearly no ffma) x this run's rate"},
        # SURVEY.md 8(d): 4-wide node records (128 B = 32 B per box test) and triangle records (48 B per test) are served by L1 / L2
        "bvh_traffic": {"kernel": "k_trace_fused", "bytes_per_ray": 32.0 * box_per_ray + 48.0 * tri_per_ray,
                        "achieved": (32.0 * box_per_ray + 48.0 * tri_per_ray) * rays_mine / trace_s / 1e9 if trace_s > 0 else 0.0, "unit": "GB/s",
                        "served_by": "L1/L2", "trace_only_mrays_per_s": rays_mine / trace_s / 1e6 if trace_s > 0 else 0.0},
        "stage_ms_per_step": {"gen_ms": tot["generate_ms"] / args.steps, "closest_ms": tot["trace_closest_ms"] / args.steps, "shade_ms": tot["shade_ms"] / args.steps,
                              "shadow_ms": tot["trace_shadow_ms"] / args.steps, "film_ms": tot["film_ms"] / args.steps, "reduce_ms": tot["reduce_ms"] / args.steps},
        "counts_rank0": {"paths": int(tot["paths"]), "closest_rays": int(tot["closest_rays"]), "shadow_rays": int(tot["shadow_rays"]), "trace_launches": int(tot["trace_launches"]),
                         "shade_launches": int(tot["shade_launches"]), "passes": int(tot["passes"])},
        "kernel_source_sha": kernel_source_sha(),
        "scene_build_s": build_s,
    }
    line.update(extras)
    if not args.no_cpu_baseline and world == 1:   # rank 0 at N = 1 only
        try:
            arm = CpuArm(wl, scene.desc, cam)
            arm.sample(max(2.0, args.cpu_seconds / 4.0))      # warm-up: settles the paths-per-second estimate the real sample is sized with (the reference arm has warm-up steps too)
            info = arm.sample(args.cpu_seconds)
            line["cpu_baseline"] = {"value": info["mrays"], "unit": "Mrays/s", "cores": info["cores"], "kind": "port", "sample": info["sample"], "mpaths_per_s": info["mpaths"],
                                    "rays_per_path": info["rays_per_path"]}
            # GPU paths of the bench frame against the oracle's, sampler tables live (the prefix table exists from the timed steps)
            try:
                rng = np.random.default_rng(7)
                n = 2000
                xy = np.stack([rng.integers(0, W, n), rng.integers(0, H, n)], 1).astype(np.uint32)
                si = rng.integers(0, wl["frame_spp"], n).astype(np.uint32)
                g = image.path_samples(wl["sampler"], xy, si)
                o = arm.osc.path_samples(arm.osc.params(W, H, wl["frame_spp"], wl["integrator"], wl["sampler"], cam), xy, si)
                err = np.abs(g - o).max(1)
                line.setdefault("parity_probe", {})["vs_oracle"] = {"paths": n, "bit_identical_frac": float((err == 0).mean()),
                                                                    "mean_rel_err": float(np.abs(g - o).mean() / max(1e-12, np.abs(o).mean())),
                                                                    "what": "tcpt_path_samples vs the oracle on random (pixel, sample) pairs of the bench frame"}
            except Exception as e:  # noqa: BLE001
                line.setdefault("parity_probe", {})["vs_oracle"] = {"failed": str(e)}
            try:
                arm2 = CpuArm(wl, scene.desc, cam, optimised=True)
                info2 = arm2.sample(max(2.0, args.cpu_seconds / 3.0))
                line["cpu_baseline"]["optimised"] = {"value": info2["mrays"], "unit": "Mrays/s", "mpaths_per_s": info2["mpaths"], "sample": info2["sample"],
                                                     "what": "same port, ordered t-shrinking traversal + cached instance inverses (not the reference's algorithmic cost)"}
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"]["optimised"] = {"value": None, "what": f"failed: {e}"}
        except Exception as e:  # the oracle is test infrastructure; its absence must not hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line))
    ctx.comm_destroy()
    if world > 1:
        dist.destroy_process_group()
    return 0


# ---------------------------------------------------------------- triangle-soup traversal workloads (BASELINE.json configs[4])
def soup_rays_numpy(n_side, hits_t=None):
    """Pinhole primaries from the render-space origin (the camera sits at (0,0,3) looking down -z, fov 45), n_side x n_side."""
    y, x = np.mgrid[0:n_side, 0:n_side].astype(np.float32)
    s = np.float32(np.tan(np.deg2rad(45.0) / 2))
    d = np.stack([(2 * (x + 0.5) / n_side - 1) * s, (1 - 2 * (y + 0.5) / n_side) * s, -np.ones_like(x)], -1).reshape(-1, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.zeros_like(d), d.astype(np.float32)


def soup_bounce_numpy(o, d, t, hit, seed=1):
    """Cosine-weighted directions about a random axis at each primary hit (incoherent: neighbouring rays share an origin region, not a direction)."""
    n = len(o)
    rng = np.random.default_rng(seed)
    u1, u2 = rng.random(n, dtype=np.float32), rng.random(n, dtype=np.float32)
    r, ph = np.sqrt(u1), 2 * np.pi * u2
    loc = np.stack([r * np.cos(ph), r * np.sin(ph), np.sqrt(1 - u1)], -1)
    axis = rng.normal(size=(n, 3)).astype(np.float32); axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    tng = np.cross(axis, np.roll(axis, 1, axis=1)); tng /= np.linalg.norm(tng, axis=1, keepdims=True)
    btn = np.cross(axis, tng)
    d2 = (tng * loc[:, :1] + btn * loc[:, 1:2] + axis * loc[:, 2:3]).astype(np.float32)
    o2 = (o + d * np.where(hit, t, 1.0)[:, None] + d2 * 1e-4).astype(np.float32)
    sel = np.nonzero(hit)[0]
    return o2[sel], d2[sel]


def soup_gpu(args, wl, world, rank, local):
    import ctypes as C

    import torch
    import torch.distributed as dist
    dev = f"cuda:{local}"
    tp, scene, cam = describe_scene(wl, device=local)
    ctx = scene.ctx
    ctx.set_option("binned_builder", 1)      # soups are outside topology parity: the reference's builder is O(N^2)
    for kv in args.opt:
        name, _, val = kv.partition("=")
        ctx.set_option(name, int(val))
    device_builder = args.soup_builder == "device"
    t0 = time.time()
    if device_builder:
        # the BVH is built where the triangles are (csrc/lbvh.cuh); the scene is the soup alone, in world space (camera at (0, 0, 3))
        mesh = scene.desc.meshes[0]
        scene.build_soup(mesh.positions[mesh.indices.reshape(-1)].reshape(-1, 3, 3))
        build_info = scene.soup_build_info()
    else:
        scene.build(cam)
        build_info = {}
    build_s = time.time() - t0
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    FMAX = np.finfo(np.float32).max
    shift = np.asarray(cam.position, dtype=np.float32) if device_builder else np.zeros(3, np.float32)    # Render space -> the space the scene was built in

    def pack(o, d):
        n = len(o)
        r = np.zeros((2 * n, 4), dtype=np.float32)
        r[:n, :3], r[:n, 3], r[n:, :3] = o + shift, FMAX, d
        return torch.from_numpy(r).to(dev)

    def trace_dev(rays, n, any_hit, hits):
        ctx.check(ctx.lib.tcpt_trace_device(ctx.handle, C.c_void_p(rays.data_ptr()), n, int(any_hit), C.c_void_p(hits.data_ptr()), C.c_void_p(stream.cuda_stream)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(rays, n, any_hit, steps, warmup, hits):
        for _ in range(warmup):
            trace_dev(rays, n, any_hit, hits)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(steps):
            trace_dev(rays, n, any_hit, hits)
        b.record(stream)
        barrier()
        return a.elapsed_time(b) / steps

    def hit_records(nn, any_hit):
        """What tcpt_trace hands its caller for a fixed sample of the nn rays last traced into `hits`: {prim, tri, t, b0, b1, b2} per
        closest hit (prim -1, the rest 0 for a miss), or the 0|1 flag of an any-hit ray (k_unpack_hits)."""
        idx = torch.from_numpy(sample_rows(nn, 1 << 18)).to(dev)
        tb = hits[: nn * 16].view(torch.float32).view(nn, 4)[idx].cpu().numpy().astype(np.float64)
        pt = hits[nn * 16: nn * 24].view(torch.int32).view(nn, 2)[idx].cpu().numpy().astype(np.float64)
        if any_hit:
            return (pt[:, :1] >= 0).astype(np.float64)
        rec = np.concatenate([pt, tb], 1)
        rec[pt[:, 0] < 0, 1:] = 0.0
        return rec

    dump = args.dump_outputs is not None and rank == 0
    outputs = {}
    o, d = soup_rays_numpy(args.soup_rays)
    n = len(o)
    rays_c = pack(o, d)
    hits = torch.empty(n * 24, dtype=torch.uint8, device=dev)
    trace_dev(rays_c, n, False, hits); torch.cuda.synchronize()
    h = hits.cpu().numpy()
    t = h[: n * 16].view(np.float32).reshape(n, 4)[:, 0]
    hit = h[n * 16:].view(np.int32).reshape(n, 2)[:, 0] >= 0
    o2, d2 = soup_bounce_numpy(o, d, t, hit, seed=1 + rank)
    m = len(o2)
    rays_i = pack(o2, d2)
    with ClockSampler(local, args.clock_period) as clk:
        ms_i = timed(rays_i, m, False, args.steps, args.warmup, hits)
    if dump:
        outputs["incoherent_closest"] = hit_records(m, False)
    ms_c = timed(rays_c, n, False, args.steps, args.warmup, hits)
    if dump:
        outputs["coherent_closest"] = hit_records(n, False)
    ms_s = timed(rays_i, m, True, args.steps, args.warmup, hits)
    if dump:
        outputs["incoherent_anyhit"] = hit_records(m, True)
        dump_outputs(args.dump_outputs, outputs)
    counts = {}
    ctx.set_option("count_tests", 1)
    for name, (rr, nn, ah) in {"incoherent": (rays_i, m, False), "coherent": (rays_c, n, False), "anyhit": (rays_i, m, True)}.items():
        trace_dev(rr, nn, ah, hits); torch.cuda.synchronize()
        st = ctx.stats()
        counts[name] = (st["box_tests"] / nn, st["tri_tests"] / nn)
    ctx.set_option("count_tests", 0)
    depth = ctx.stats()["max_bvh_depth"]
    # e2e: the host-buffer entry point (rays in, hit records out)
    host_rays = np.concatenate([o2, d2, np.full((m, 1), FMAX, np.float32)], 1)
    e2e_n = min(m, 4_000_000)
    e2e_rays = host_rays[:e2e_n].copy(); e2e_rays[:, :3] += shift
    scene.trace(e2e_rays)
    barrier(); t0 = time.perf_counter()
    scene.trace(e2e_rays)
    barrier(); e2e_s = time.perf_counter() - t0
    tt = torch.tensor([ms_i, float(m), e2e_s, float(e2e_n)], dtype=torch.float64, device=dev)
    if world > 1:
        tm = tt.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = tt.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        ms_max, rays_all, e2e_max, e2e_all = tm[0].item(), ts[1].item(), tm[2].item(), ts[3].item()
    else:
        ms_max, rays_all, e2e_max, e2e_all = ms_i, float(m), e2e_s, float(e2e_n)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))

    def roof(name, ms, nn):
        B, T = counts[name]
        bpr = 48.0 + 32.0 * B + 48.0 * T
        ach = bpr * nn / (ms * 1e-3) / 1e9
        return {"mrays_per_s": nn / ms / 1e3, "ms_per_launch": ms, "rays": nn, "box_tests_per_ray": B, "tri_tests_per_ray": T, "bytes_per_ray": bpr, "achieved": ach, "frac": ach / hbm_peak}
    ri, rc, rs = roof("incoherent", ms_i, m), roof("coherent", ms_c, n), roof("anyhit", ms_s, m)
    traffic, note = None, None
    try:
        prof = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text()).get("soups", {}).get(args.workload)
        if prof and prof.get("kernel_source_sha") == kernel_source_sha():
            traffic = prof["incoherent_dram_bytes_per_ray"] * m
        elif prof:
            note = "STALE soup capture in profiles/ncu_traffic.json"
    except Exception:
        pass
    line = {"metric": "Mrays/s", "value": rays_all / ms_max / 1e3, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {wl['soup']} random triangles (centres uniform in [-1,1]^3, edge 0.5 N^(-1/3)), incoherent cosine-weighted bounce rays from the "
                                   f"hits of {args.soup_rays}x{args.soup_rays} pinhole primaries, closest hit (BASELINE.json configs[4])", "rays_per_gpu_per_step": m,
                       "sharding": "replicas (every rank traces its own ray batch against its own copy of the soup)", "cache": "BVH + triangles exceed the 126 MB L2 from 10 M triangles on; ray batch 800 MB"},
            "e2e": {"value": e2e_all / e2e_max / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(e2e_n * 28), "d2h_bytes_per_step": int(e2e_n * 24), "call": "Scene.trace -> tcpt_trace(host rays, host hit records)"},
            "gpu_launches": args.steps, "clocks": clk.summary(),
            "roofline": {"kernel": "k_trace_closest (soup, incoherent)", "bound": "hbm", "achieved": ri["achieved"], "peak": hbm_peak, "unit": "GB/s", "frac": ri["frac"], "traffic": traffic,
                         "traffic_note": note, "definition": "48 + 32*B + 48*T bytes per ray (SURVEY.md 8d), B and T counted by the kernel"},
            "incoherent_closest": ri, "coherent_closest": rc, "incoherent_anyhit": rs, "bvh_depth": depth, "scene_build_s": build_s, "builder": args.soup_builder, "device_build": build_info,
            "kernel_source_sha": kernel_source_sha()}
    if not args.no_cpu_baseline and world == 1 and wl["soup"] <= 10_000_000:
        try:
            line["cpu_baseline"] = soup_cpu(args, wl, scene.desc, cam, host_rays, np.concatenate([o, d, np.full((n, 1), FMAX, np.float32)], 1))
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def soup_cpu(args, wl, desc, cam, rays_inc, rays_coh, seconds=None):
    """The oracle's ORDERED, t-shrinking traversal (the reference's exhaustive walk is quadratic-ish on a soup) over all host threads,
    on a bounded sample of the same ray batches."""
    from toy_cpu_pathtracing_b200 import capi
    from oracle import oracle
    seconds = seconds or args.cpu_seconds
    std, tab = capi.load_tables()
    osc = oracle.OracleScene(std, tab, faithful=False, literal_build=False)
    t0 = time.time(); desc.replay(osc); osc.build(cam.position); build_s = time.time() - t0
    osc.set_optimised(True)
    rng = np.random.default_rng(3)
    out = {}
    for name, rays in (("incoherent", rays_inc), ("coherent", rays_coh)):
        probe = rays[rng.integers(0, len(rays), 20000)]
        _, sec, _, _ = osc.trace_mt(probe)
        n = int(min(len(rays), max(20000, 0.5 * seconds / max(sec, 1e-6) * 20000)))
        sample = rays[rng.integers(0, len(rays), n)]
        _, sec, nb, nt = osc.trace_mt(sample)
        out[name] = {"mrays_per_s": n / sec / 1e6, "rays": n, "seconds": sec, "box_tests_per_ray": nb / n, "tri_tests_per_ray": nt / n}
    return {"value": out["incoherent"]["mrays_per_s"], "unit": "Mrays/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"{out['incoherent']['rays']} random rays of the incoherent batch in {out['incoherent']['seconds']:.2f} s (ordered t-shrinking traversal of the oracle; BVH built in {build_s:.1f} s)",
            "coherent": out["coherent"], "incoherent": out["incoherent"]}


def soup_reference(args, wl):
    """--impl reference for a soup: primaries and bounce rays are produced by the oracle itself (no GPU, no libtcpt)."""
    from toy_cpu_pathtracing_b200 import capi
    from oracle import oracle
    _, scene, cam = describe_scene(wl, describe_only=True)
    std, tab = capi.load_tables()
    osc = oracle.OracleScene(std, tab, faithful=False, literal_build=False)
    scene.desc.replay(osc); osc.build(cam.position)
    osc.set_optimised(True)
    FMAX = np.finfo(np.float32).max
    side = 1024
    o, d = soup_rays_numpy(side)
    prim = np.concatenate([o, d, np.full((len(o), 1), FMAX, np.float32)], 1)
    hits, _, _, _ = osc.trace_mt(prim)
    hit = hits[:, 0] >= 0
    t = hits[:, 2].view(np.float32)
    o2, d2 = soup_bounce_numpy(o, d, t, hit)
    rays = np.concatenate([o2, d2, np.full((len(o2), 1), FMAX, np.float32)], 1)
    per_step = max(1.0, min(args.cpu_seconds, 120.0 / max(1, args.steps + args.warmup)))
    _, sec, _, _ = osc.trace_mt(rays[:20000])
    n = int(min(len(rays), max(20000, per_step / max(sec, 1e-6) * 20000)))
    tot_n = tot_s = 0.0
    for i in range(args.warmup + args.steps):
        _, sec, _, _ = osc.trace_mt(rays[:n])
        if i >= args.warmup:
            tot_n += n; tot_s += sec
    value = tot_n / tot_s / 1e6
    print(json.dumps({"impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1e3 * tot_s / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": f"{args.workload}: incoherent bounce rays from {side}x{side} primaries, closest hit, oracle ordered traversal", "rays_per_step": n},
                      "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": f"{n} rays per step"},
                      "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    return 0


def main():
    args = parse()
    wl = dict(WORKLOADS[args.workload], max_depth=args.max_depth)
    if args.impl == "reference":
        return main_reference(args, wl)
    return main_gpu(args, wl)


if __name__ == "__main__":
    sys.exit(main())
