#!/usr/bin/env python3
"""How adaptive frames split over GPUs (DESIGN.md section 10, "Several GPUs").

One process (no torchrun): the whole adaptive frame (tcpt_render_adaptive) and the whole uniform frame (tcpt_render_device) on GPU 0, then
for each world size W every one of the W tile shards of the adaptive job rendered ALONE through tcpt_render_adaptive_device, next to the
same shard of the uniform job through tcpt_render_device.  Every shard is rendered twice in a row: render_ms is the device time of the
second call (first_ms that of the first, which also pays for whatever the new shard shape makes the context grow), with the rounds it ran
and the paths it traced.  The maximum over the shards is a PROJECTION of the W-GPU frame time without the reduce (each GPU would run its
shard alone), not a W-GPU measurement; projected_speedup = the one-GPU frame's render_ms / that maximum.  Defaults: scenes 19 and 17
at 1920x1080, MIS + Z-Sobol, N = 4096, threshold 0.02, min_spp = step = 64.

Under torchrun with W processes (one GPU each): tcpt_render_adaptive_sharded is timed on every rank (render_ms, reduce_ms), and rank 0 checks
its frame bitwise against the same job rendered alone with tcpt_render_adaptive.

Every run starts with a line naming the GPU and its power limit; one JSON line per record, also written to OUT/adaptive_scaling.jsonl.

usage: adaptive_scaling.py OUT [--scenes 19 17] [--worlds 2 4 8] [--width 1920 --height 1080] [--spp 4096] [--threshold 0.02]
       torchrun --nproc-per-node W adaptive_scaling.py OUT ...
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import numpy as np  # noqa: E402
from adaptive_quality import gpu_info  # noqa: E402


def rounds_of(counts, min_spp, step):
    return 1 + -(-(int(counts.max()) - min_spp) // step) if counts.size else 0


def single_process(a, emit, tp, scenes, capi):
    import torch
    w, h, N = a.width, a.height, a.spp
    ap = capi.AdaptiveParams(a.threshold, a.min_spp, a.step)
    for sid in a.scenes:
        scene = tp.Scene(device=0)
        cam = tp.Camera(45.0, w, h)
        scenes.load_scene(sid, scene, cam)
        scene.build(cam)
        ctx = scene.ctx
        img = tp.RendererImage(w, h, tp.SrgbRendererMis(tp.RendererArgs((w, h), N, scene, cam)))
        img.render("sobol", want_accumulators=False, spp_begin=0, spp_end=16)   # warm-up: module load, wavefront state, slot budget
        full = tp.RendererImage(w, h, img.renderer).render_adaptive("sobol", threshold=a.threshold, min_spp=a.min_spp, step=a.step,
                                                                    want_accumulators=False)
        job = img.renderer.params("sobol")
        acc = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda:0")
        cnt = torch.zeros((h, w), dtype=torch.int32, device="cuda:0")
        stream = torch.cuda.Stream(device=0)

        def uniform(p):
            acc.zero_(); torch.cuda.synchronize()
            ctx.check(ctx.lib.tcpt_render_device(ctx.handle, C.byref(p), C.c_void_p(acc.data_ptr()), C.c_void_p(stream.cuda_stream)))
            return ctx.stats()

        def adaptive(p):
            acc.zero_(); cnt.zero_(); torch.cuda.synchronize()
            ctx.check(ctx.lib.tcpt_render_adaptive_device(ctx.handle, C.byref(p), C.byref(ap), C.c_void_p(acc.data_ptr()),
                                                          C.c_void_p(cnt.data_ptr()), C.c_void_p(stream.cuda_stream)))
            return ctx.stats()

        u = uniform(job)
        one_gpu = {"adaptive": full.stats["render_ms"], "uniform": u["render_ms"]}
        emit({"kind": "adaptive_one_gpu", "scene": sid, "render_ms": one_gpu["adaptive"], "rounds": full.stats["rounds"],
              "paths": full.stats["paths"]})
        emit({"kind": "uniform_one_gpu", "scene": sid, "render_ms": one_gpu["uniform"], "paths": u["paths"]})
        for world in a.worlds:
            shards = {"adaptive": [], "uniform": []}
            for r in range(world):
                mine = capi.RenderParams()
                ctx.check(ctx.lib.tcpt_shard_params(C.byref(job), capi.SHARD_MODES["tile"], r, world, C.byref(mine)))
                first, st = uniform(mine)["render_ms"], uniform(mine)
                shards["uniform"].append({"rank": r, "render_ms": st["render_ms"], "first_ms": first, "rounds": 1, "paths": st["paths"]})
                mine.spp_begin = mine.spp_end = 0
                first, st = adaptive(mine)["render_ms"], adaptive(mine)
                owned = cnt.cpu().numpy().view(np.uint32)[r::world]
                shards["adaptive"].append({"rank": r, "render_ms": st["render_ms"], "first_ms": first, "rounds": rounds_of(owned, a.min_spp, a.step),
                                           "paths": st["paths"]})
            for kind, recs in shards.items():
                ms = [s["render_ms"] for s in recs]
                emit({"kind": f"{kind}_shards", "scene": sid, "world": world, "shards": recs,
                      "projected_frame_ms_without_reduce": max(ms), "sum_of_shards_ms": sum(ms),
                      "projected_speedup": one_gpu[kind] / max(ms)})


def multi_process(a, emit, tp, scenes, capi):
    import torch
    import torch.distributed as dist
    from toy_cpu_pathtracing_b200.multi_gpu import init_comm
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    w, h, N = a.width, a.height, a.spp
    kw = dict(threshold=a.threshold, min_spp=a.min_spp, step=a.step)
    for sid in a.scenes:
        scene = tp.Scene(device=local)
        cam = tp.Camera(45.0, w, h)
        scenes.load_scene(sid, scene, cam)
        scene.build(cam)
        init_comm(scene.ctx, rank, world)
        mk = lambda: tp.RendererImage(w, h, tp.SrgbRendererMis(tp.RendererArgs((w, h), N, scene, cam)))  # noqa: E731
        mk().render_sharded("sobol", want_accumulators=False, spp_window=(0, 16))   # warm-up
        img = mk().render_adaptive_sharded("sobol", **kw)
        mine = torch.tensor([img.stats["render_ms"], img.stats["reduce_ms"], float(img.stats["paths"])], dtype=torch.float64)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        dist.barrier()
        if rank == 0:
            alone = mk().render_adaptive("sobol", **kw)   # this GPU alone: tcpt_render_adaptive never uses the communicator
            same = (np.array_equal(img.sample_counts, alone.sample_counts)
                    and np.array_equal(img.accumulators.view(np.uint32), alone.accumulators.view(np.uint32))
                    and np.array_equal(img.pixels.view(np.uint32), alone.pixels.view(np.uint32)))
            emit({"kind": "adaptive_sharded", "scene": sid, "world": world, "rounds": img.stats["rounds"],
                  "ranks": [{"rank": i, "render_ms": float(t[0]), "reduce_ms": float(t[1]), "paths": int(t[2])} for i, t in enumerate(every)],
                  "frame_ms": max(float(t[0]) for t in every), "one_gpu_ms": alone.stats["render_ms"], "bitwise_equal_to_one_gpu": bool(same)})
            if not same:
                raise SystemExit("the sharded adaptive frame differs from the one-GPU frame")
        dist.barrier()
        scene.ctx.comm_destroy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", type=Path)
    ap.add_argument("--scenes", type=int, nargs="+", default=[19, 17])
    ap.add_argument("--worlds", type=int, nargs="+", default=[2, 4, 8])
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=4096)
    ap.add_argument("--threshold", type=float, default=0.02)
    ap.add_argument("--min-spp", type=int, default=64)
    ap.add_argument("--step", type=int, default=64)
    a = ap.parse_args()

    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import capi, scenes

    torchrun = int(os.environ.get("WORLD_SIZE", "1")) > 1
    if torchrun:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("gloo")    # carries the NCCL unique id only; the reduce is libtcpt's own
    root = not torchrun or int(os.environ["RANK"]) == 0
    a.out.mkdir(parents=True, exist_ok=True)
    with open(a.out / "adaptive_scaling.jsonl", "w") if root else open(os.devnull, "w") as f:
        def emit(rec):
            line = json.dumps(rec)
            print(line, flush=True)
            f.write(line + "\n"); f.flush()

        if root:
            emit({"kind": "machine", **gpu_info(), "width": a.width, "height": a.height, "spp": a.spp, "integrator": "mis", "sampler": "sobol",
                  "threshold": a.threshold, "min_spp": a.min_spp, "step": a.step, "mode": "torchrun" if torchrun else "one GPU, shards in turn"})
        (multi_process if torchrun else single_process)(a, emit, tp, scenes, capi)
    if torchrun:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
