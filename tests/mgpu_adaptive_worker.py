"""Worker of tests/test_adaptive_sharded.py::test_two_ranks_reproduce_the_one_gpu_adaptive_frame, launched by torchrun with one rank per GPU.
Every rank: scene 19 at 200x150, its own libtcpt context on its GPU, tcpt_comm_init (the NCCL unique id travels through a gloo process
group), then tcpt_render_adaptive_sharded; the other ranks check that their host buffers were left alone.  Then every rank, with its
communicator still in place, renders the adaptive frame alone (tcpt_render_adaptive, which must not reduce); rank 0 compares its sharded
frame with that one bitwise, and every rank's alone frame must equal rank 0's."""
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def main():
    import torch
    import torch.distributed as dist
    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import scenes
    from toy_cpu_pathtracing_b200.multi_gpu import init_comm

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")            # plumbing only: carries the NCCL unique id; the reduce is libtcpt's own
    w, h, spp = 200, 150, 256
    kw = dict(threshold=0.02, min_spp=32, step=32)
    scene = tp.Scene(device=local)
    cam = tp.Camera(45.0, w, h)
    scenes.load_scene(19, scene, cam)
    scene.build(cam)
    init_comm(scene.ctx, rank, world)
    mk = lambda: tp.RendererImage(w, h, tp.SrgbRendererMis(tp.RendererArgs((w, h), spp, scene, cam)))  # noqa: E731
    img = mk()
    img.accumulators[:] = 7.0; img.pixels[:] = 7.0; img.sample_counts[:] = 7
    img.render_adaptive_sharded("sobol", **kw)
    paths = torch.tensor([img.stats["paths"]], dtype=torch.int64)
    dist.all_reduce(paths)
    if world > 1:
        assert img.stats["reduce_ms"] > 0.0, img.stats
    dist.barrier()
    # tcpt_render_adaptive on a context that holds a communicator renders the whole frame on this GPU alone, on every rank: no collective,
    # every rank's own buffers written.  All ranks must get the same frame (rank 0's is broadcast for the comparison).
    alone = mk().render_adaptive("sobol", **kw)
    assert alone.stats["reduce_ms"] == 0.0 and alone.stats["paths"] == int(alone.sample_counts.sum())
    mine = torch.from_numpy(np.concatenate([alone.accumulators.view(np.int32).ravel(), alone.sample_counts.view(np.int32).ravel()]))
    theirs = mine.clone()
    dist.broadcast(theirs, src=0)
    assert torch.equal(mine, theirs), f"rank {rank}: tcpt_render_adaptive differs from rank 0's"
    if rank == 0:
        assert np.array_equal(img.sample_counts, alone.sample_counts), "counts differ from the one-GPU adaptive frame"
        assert np.array_equal(img.accumulators.view(np.uint32), alone.accumulators.view(np.uint32)), "accumulators differ"
        assert np.array_equal(img.pixels.view(np.uint32), alone.pixels.view(np.uint32)), "sRGB differs"
        assert int(paths) == int(alone.sample_counts.sum()), (int(paths), int(alone.sample_counts.sum()))
        assert img.stats["rounds"] == alone.stats["rounds"]
        print(f"MGPU_ADAPTIVE_OK rounds {alone.stats['rounds']} paths {int(paths)}", flush=True)
    else:
        assert (img.accumulators == 7.0).all() and (img.pixels == 7.0).all() and (img.sample_counts == 7).all()
    dist.barrier()
    scene.ctx.comm_destroy()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
