#!/usr/bin/env python3
"""Adaptive vs uniform sampling: time and error against a high-spp reference (DESIGN.md "Adaptive sampling").

Per scene (19 and 17 by default, 1920x1080, MIS + Z-Sobol, job spp N = 4096):
  reference  uniform N spp, seed 1 (noise independent of the compared renders)
  uniform    256 / 512 / 1024 spp, seed 0
  adaptive   thresholds 0.02 / 0.01 / 0.005, seed 0, min_spp 64, step 64, N = 4096
Each run reports the device time of the call (stats render_ms), the paths traced, the rounds (adaptive) and passes, and the RMSE of the
tone-mapped sRGB pixels against the reference.  One JSON line per run goes to OUT/adaptive_quality.jsonl, headed by a line with the
GPU's name and power limit.

usage: adaptive_quality.py OUT [--scenes 19 17] [--width 1920 --height 1080] [--spp 4096]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:   # the numbers are still the GPU's; say that the card could not be named
        return {"gpu": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", type=Path)
    ap.add_argument("--scenes", type=int, nargs="+", default=[19, 17])
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=4096)
    ap.add_argument("--uniform", type=int, nargs="+", default=[256, 512, 1024])
    ap.add_argument("--thresholds", type=float, nargs="+", default=[0.02, 0.01, 0.005])
    ap.add_argument("--min-spp", type=int, default=64)
    ap.add_argument("--step", type=int, default=64)
    a = ap.parse_args()

    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import scenes

    a.out.mkdir(parents=True, exist_ok=True)
    path = a.out / "adaptive_quality.jsonl"
    w, h, N = a.width, a.height, a.spp
    with open(path, "w") as f:
        def emit(rec):
            line = json.dumps(rec)
            print(line, flush=True)
            f.write(line + "\n"); f.flush()

        emit({"kind": "machine", **gpu_info(), "width": w, "height": h, "spp": N, "integrator": "mis", "sampler": "sobol",
              "min_spp": a.min_spp, "step": a.step})
        for sid in a.scenes:
            scene = tp.Scene(device=0)
            cam = tp.Camera(45.0, w, h)
            scenes.load_scene(sid, scene, cam)
            scene.build(cam)

            def image(spp, seed):
                return tp.RendererImage(w, h, tp.SrgbRendererMis(tp.RendererArgs((w, h), spp, scene, cam, seed=seed)))

            image(16, 0).render("sobol", want_accumulators=False)   # warm-up: module load, wavefront state, slot budget
            ref = image(N, 1).render("sobol", want_accumulators=False)
            ref_px = ref.pixels.astype(np.float64)
            emit({"kind": "reference", "scene": sid, "spp": N, "seed": 1, "render_ms": ref.stats["render_ms"], "paths": ref.stats["paths"],
                  "passes": ref.stats["passes"]})

            def rmse(img):
                return float(np.sqrt(np.mean((img.pixels.astype(np.float64) - ref_px) ** 2)))

            for spp in a.uniform:
                img = image(spp, 0).render("sobol", want_accumulators=False)
                emit({"kind": "uniform", "scene": sid, "spp": spp, "seed": 0, "render_ms": img.stats["render_ms"], "paths": img.stats["paths"],
                      "rounds": 1, "passes": img.stats["passes"], "rmse": rmse(img)})
            for thr in a.thresholds:
                img = image(N, 0).render_adaptive("sobol", threshold=thr, min_spp=a.min_spp, step=a.step, want_accumulators=False)
                c = img.sample_counts
                emit({"kind": "adaptive", "scene": sid, "threshold": thr, "seed": 0, "render_ms": img.stats["render_ms"], "paths": img.stats["paths"],
                      "rounds": img.stats["rounds"], "passes": img.stats["passes"], "rmse": rmse(img), "mean_spp": float(c.mean()),
                      "frac_at_min": float((c == a.min_spp).mean()), "frac_at_max": float((c == N).mean())})


if __name__ == "__main__":
    main()
