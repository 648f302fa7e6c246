"""The N > 1 path on CPU: two gloo ranks shard a frame (rows or sample ranges), render their shard (here with the ORACLE as
the per-rank renderer, which tests may use), reduce the film with the product's reduce_film(), and must reproduce the
single-process frame: bitwise for row shards, within rounding for sample-range shards."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_shard_plan_partitions_everything():
    from toy_cpu_pathtracing_b200.multi_gpu import shard_plan
    for world in (1, 2, 3, 8):
        rows = set()
        for r in range(world):
            s = shard_plan(r, world, "tile", 512)
            rows |= set(range(s.row_offset, 150, s.row_stride))
            assert (s.spp_begin, s.spp_end) == (0, 512)
        assert rows == set(range(150))
        got = []
        for r in range(world):
            s = shard_plan(r, world, "spp", 512, 8, 8 + 5 * 3)
            got += list(range(s.spp_begin, s.spp_end))
        assert got == list(range(8, 23))
    with pytest.raises(ValueError):
        shard_plan(2, 2, "tile", 16)
    with pytest.raises(ValueError):
        shard_plan(0, 2, "cube", 16)


def test_python_plan_is_the_c_abi_plan(built):
    """multi_gpu.shard_plan restates tcpt_shard_params (the rule the product applies inside tcpt_render_sharded): same slices for
    every rank, mode and sample window; bad jobs are refused by both."""
    import ctypes as C
    from toy_cpu_pathtracing_b200 import capi
    from toy_cpu_pathtracing_b200.multi_gpu import shard_plan
    lib = capi.load_library()
    job, out = capi.RenderParams(), capi.RenderParams()
    job.width, job.height, job.spp = 200, 150, 512
    for world in (1, 2, 3, 5, 8):
        for mode in ("tile", "spp"):
            for b, e in ((0, 0), (0, 512), (8, 23), (100, 101), (7, 7 + 3)):
                job.spp_begin, job.spp_end = b, e
                for r in range(world):
                    assert lib.tcpt_shard_params(C.byref(job), capi.SHARD_MODES[mode], r, world, C.byref(out)) == 0
                    s = shard_plan(r, world, mode, 512, *((b, e) if (b, e) != (0, 0) else (0, 512)))
                    want = (s.row_offset, s.row_stride, s.spp_begin, s.spp_end) if mode == "tile" else (0, 0, s.spp_begin, s.spp_end)
                    assert (out.row_offset, out.row_stride, out.spp_begin, out.spp_end) == want
                    assert (out.width, out.height, out.spp) == (200, 150, 512)
    job.spp_begin, job.spp_end = 0, 0
    assert lib.tcpt_shard_params(C.byref(job), 0, 2, 2, C.byref(out)) == capi.TCPT_ERR_INVALID      # rank out of range
    assert lib.tcpt_shard_params(C.byref(job), 7, 0, 2, C.byref(out)) == capi.TCPT_ERR_INVALID      # unknown mode
    job.row_stride = 2
    assert lib.tcpt_shard_params(C.byref(job), 0, 0, 2, C.byref(out)) == capi.TCPT_ERR_INVALID      # the job must describe the whole frame
    job.row_stride, job.spp_begin, job.spp_end = 0, 10, 600
    assert lib.tcpt_shard_params(C.byref(job), 1, 0, 2, C.byref(out)) == capi.TCPT_ERR_INVALID      # sample window beyond spp


def _c_abi_shard(rank, world, mode, w, h, spp):
    import ctypes as C
    from toy_cpu_pathtracing_b200 import capi
    job, out = capi.RenderParams(), capi.RenderParams()
    job.width, job.height, job.spp = w, h, spp
    assert capi.load_library().tcpt_shard_params(C.byref(job), capi.SHARD_MODES[mode], rank, world, C.byref(out)) == 0
    return out


def _worker(rank, world, port, mode, out_dir):
    os.environ["CUDA_VISIBLE_DEVICES"] = ""      # a host-only rank on any machine: set before libtcpt initialises CUDA in this process
    sys.path.insert(0, str(ROOT))
    import torch
    import torch.distributed as dist
    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import capi, scenes
    from toy_cpu_pathtracing_b200.multi_gpu import init_comm, reduce_film
    from oracle import oracle
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    w, h, spp = 32, 24, 8
    scene = tp.Scene(require_gpu=False)
    cam = tp.Camera(45.0, w, h)
    scenes.load_scene(10, scene, cam)
    std, tab = capi.load_tables()
    osc = oracle.scene_from_description(scene.desc, cam.position, std, tab)
    # the plumbing of init_comm: the NCCL unique id made on rank 0 reaches every rank through the process group; making the
    # communicator itself then needs a GPU, and a host-only context must refuse with a status code
    try:
        init_comm(scene.ctx, rank, world)
        raise AssertionError("tcpt_comm_init succeeded without a GPU")
    except capi.TcptError as e:
        assert e.code == capi.TCPT_ERR_CUDA
    sh = _c_abi_shard(rank, world, mode, w, h, spp)                                 # the slice the product would render on this rank
    acc = np.zeros((h, w, 3), dtype=np.float32)
    p = osc.params(w, h, spp, "mis", "sobol", cam, threads=2)
    rows = range(sh.row_offset, h, sh.row_stride) if sh.row_stride else range(h)
    xy = np.array([[x, y] for y in rows for x in range(w)], dtype=np.uint32)
    part = np.zeros((len(xy), 3), dtype=np.float32)
    for s in range(sh.spp_begin, sh.spp_end):                                       # ONLY this rank's pixels and sample indices, in sample order
        part += osc.path_samples(p, xy, np.full(len(xy), s, np.uint32))
    acc[list(rows)] = part.reshape(len(rows), w, 3)
    t = torch.from_numpy(acc)
    reduce_film(t, dst=0)
    if rank == 0:
        np.save(Path(out_dir) / f"{mode}.npy", t.numpy())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["tile", "spp"])
def test_two_rank_film_reduce_matches_single_process(built, tables, tmp_path, mode):
    import torch.multiprocessing as mp
    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import scenes
    from oracle import oracle
    port = 29500 + (os.getpid() % 2000) + (0 if mode == "tile" else 1)
    mp.spawn(_worker, args=(2, port, mode, str(tmp_path)), nprocs=2, join=True)
    got = np.load(tmp_path / f"{mode}.npy")
    w, h, spp = 32, 24, 8
    scene = tp.Scene(require_gpu=False)
    cam = tp.Camera(45.0, w, h)
    scenes.load_scene(10, scene, cam)
    osc = oracle.scene_from_description(scene.desc, cam.position, tables[0], tables[1])
    ref, _, _ = osc.render(osc.params(w, h, spp, "mis", "sobol", cam, threads=2))
    if mode == "tile":
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    else:
        assert np.abs(got - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
