"""Adaptive sampling on several GPUs (tcpt_render_adaptive_device / tcpt_render_adaptive_sharded / tcpt_group_render_adaptive): argument
checks on any box; on one GPU the tile shards of a job rendered rank by rank, which must sum bitwise to the one-GPU adaptive frame
(accumulators and counts), touch only their own rows, and keep the edge cases and the determinism of tcpt_render_adaptive.  The two-GPU
cases need two visible GPUs and are skipped otherwise."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

f32 = np.float32
ROOT = Path(__file__).resolve().parent.parent


def _params(**kw):
    from toy_cpu_pathtracing_b200 import capi
    p = capi.RenderParams()
    p.width, p.height, p.spp, p.max_depth = 4, 4, 16, 16
    p.integrator, p.sampler = capi.INTEGRATORS["mis"], capi.SAMPLERS["sobol"]
    p.exposure, p.fov_deg = 1.0, 45.0
    p.cam_dir[2], p.cam_up[1] = -1.0, 1.0
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _ref(x):
    return C.byref(x) if x is not None else None


def _host(a, ctype):
    from toy_cpu_pathtracing_b200 import capi
    return capi.as_ptr(a, ctype) if a is not None else None


def _dev(a):
    """A host array's address where the entry point takes a device pointer: only for calls that must refuse before touching it."""
    return C.c_void_p(a.ctypes.data) if a is not None else None


def _device_call(ctx, p, ap, acc, spp):
    return ctx.lib.tcpt_render_adaptive_device(ctx.handle, _ref(p), _ref(ap), _dev(acc), _dev(spp), None)


def _sharded_call(ctx, p, ap, acc, srgb, spp):
    return ctx.lib.tcpt_render_adaptive_sharded(ctx.handle, _ref(p), _ref(ap), _host(acc, C.c_float), _host(srgb, C.c_float), _host(spp, C.c_uint32))


def _one_context_group(lib):
    """A group over device 0: with a GPU a working one-GPU group, without one a group whose context only does host work."""
    g = C.c_void_p()
    rc = lib.tcpt_group_create((C.c_int32 * 1)(0), 1, C.byref(g))
    assert g, rc
    return g


def test_adaptive_sharded_refusals_are_invalid(built):
    """Every malformed request is refused with TCPT_ERR_INVALID before the device is looked at and writes nothing, with or without a GPU."""
    from toy_cpu_pathtracing_b200 import capi
    ctx = capi.Context(0, require_gpu=False)
    lib = ctx.lib
    acc = np.full(48, 7.0, dtype=f32); srgb = np.full(48, 7.0, dtype=f32); spp = np.full(16, 7, dtype=np.uint32)
    good, AP = capi.AdaptiveParams(0.01, 4, 4), capi.AdaptiveParams
    bad_ap = [AP(-0.01, 4, 4), AP(float("nan"), 4, 4), AP(float("inf"), 4, 4), AP(0.01, 1, 4), AP(0.01, 0, 4), AP(0.01, 17, 4), AP(0.01, 4, 0)]
    aov = [_params(integrator=capi.INTEGRATORS["albedo"]), _params(integrator=capi.INTEGRATORS["normal"])]

    assert lib.tcpt_render_adaptive_device(None, _ref(_params()), _ref(good), _dev(acc), _dev(spp), None) == capi.TCPT_ERR_INVALID
    device_cases = [
        (_params(), None, acc, spp), (None, good, acc, spp),                     # null ap / params
        (_params(), good, None, spp), (_params(), good, acc, None), (_params(), good, None, None),
        (_params(row_offset=2, row_stride=2), good, acc, spp),                   # row_offset >= row_stride
        (_params(row_offset=3, row_stride=2), good, acc, spp),
        (_params(row_offset=1), good, acc, spp),                                 # row_stride 0 = the whole frame
        (_params(spp_begin=4), good, acc, spp), (_params(spp_end=8), good, acc, spp),
        (_params(row_offset=0, row_stride=2, spp_begin=0, spp_end=16), good, acc, spp),   # tcpt_shard_params' form of "every sample"
    ] + [(_params(), ap, acc, spp) for ap in bad_ap] + [(p, good, acc, spp) for p in aov]
    for i, case in enumerate(device_cases):
        assert _device_call(ctx, *case) == capi.TCPT_ERR_INVALID, f"device case {i}"

    assert lib.tcpt_render_adaptive_sharded(None, _ref(_params()), _ref(good), _host(acc, C.c_float), None, None) == capi.TCPT_ERR_INVALID
    sharded_cases = [
        (_params(), None, acc, None, None), (None, good, acc, None, None),
        (_params(), good, None, None, None),                                     # no output buffer on rank 0
        (_params(row_stride=2), good, acc, srgb, spp),                           # the job must describe the whole frame
        (_params(row_offset=1, row_stride=2), good, acc, srgb, spp),
        (_params(row_offset=1), good, acc, srgb, spp),
        (_params(spp_begin=4), good, acc, srgb, spp), (_params(spp_end=8), good, acc, srgb, spp),
    ] + [(_params(), ap, acc, srgb, spp) for ap in bad_ap] + [(p, good, acc, srgb, spp) for p in aov]
    for i, case in enumerate(sharded_cases):
        assert _sharded_call(ctx, *case) == capi.TCPT_ERR_INVALID, f"sharded case {i}"

    g = _one_context_group(lib)
    try:
        group_cases = [(_params(), good, None, None, None), (_params(), None, acc, srgb, spp), (None, good, acc, srgb, spp)] + \
                      [(p, good, acc, srgb, spp) for p in aov] + [(_params(), ap, acc, srgb, spp) for ap in bad_ap]
        for i, (p, ap, a, s, n) in enumerate(group_cases):
            rc = lib.tcpt_group_render_adaptive(g, _ref(p), _ref(ap), _host(a, C.c_float), _host(s, C.c_float), _host(n, C.c_uint32))
            assert rc == capi.TCPT_ERR_INVALID, f"group case {i}"
        assert lib.tcpt_group_render_adaptive(None, _ref(_params()), _ref(good), _host(acc, C.c_float), None, None) == capi.TCPT_ERR_INVALID
    finally:
        lib.tcpt_group_destroy(g)
    assert (acc == 7.0).all() and (srgb == 7.0).all() and (spp == 7).all()


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="GPU present")
def test_adaptive_sharded_without_gpu_writes_nothing(built):
    from toy_cpu_pathtracing_b200 import capi
    ctx = capi.Context(0, require_gpu=False)
    assert not ctx.has_gpu
    acc = np.full(48, 7.0, dtype=f32); srgb = np.full(48, 7.0, dtype=f32); spp = np.full(16, 7, dtype=np.uint32)
    ap = capi.AdaptiveParams(0.01, 4, 4)
    assert _device_call(ctx, _params(), ap, acc, spp) == capi.TCPT_ERR_CUDA
    assert _device_call(ctx, _params(row_offset=1, row_stride=2), ap, acc, spp) == capi.TCPT_ERR_CUDA
    assert _sharded_call(ctx, _params(), ap, acc, srgb, spp) == capi.TCPT_ERR_CUDA
    g = _one_context_group(ctx.lib)
    try:
        rc = ctx.lib.tcpt_group_render_adaptive(g, _ref(_params()), _ref(ap), _host(acc, C.c_float), _host(srgb, C.c_float), _host(spp, C.c_uint32))
        assert rc == capi.TCPT_ERR_CUDA
    finally:
        ctx.lib.tcpt_group_destroy(g)
    assert (acc == 7.0).all() and (srgb == 7.0).all() and (spp == 7).all()


# ---------------------------------------------------------------- GPU
W, H, N, MIN_SPP, STEP, THR = 64, 48, 256, 32, 32, 0.02


def _bits(a):
    return np.ascontiguousarray(a, dtype=f32).view(np.uint32)


def _shard(ctx, job, rank, world):
    """Rank `rank` of `world`'s tile shard of `job` (tcpt_shard_params), in the form tcpt_render_adaptive_device takes: every sample = 0, 0."""
    from toy_cpu_pathtracing_b200 import capi
    mine = capi.RenderParams()
    assert ctx.lib.tcpt_shard_params(C.byref(job), capi.SHARD_MODES["tile"], rank, world, C.byref(mine)) == 0
    mine.spp_begin = mine.spp_end = 0
    return mine


def _render_shard(ctx, mine, ap, acc0=None, spp0=None):
    """tcpt_render_adaptive_device of one shard on a caller-owned stream into device buffers that start as acc0 / spp0 (default zeros);
    returns (accumulators H x W x 3, counts H x W, stats)."""
    import torch
    acc = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda:0") if acc0 is None else torch.from_numpy(acc0.copy()).cuda()
    spp = torch.zeros((H, W), dtype=torch.int32, device="cuda:0") if spp0 is None else torch.from_numpy(spp0.view(np.int32).copy()).cuda()
    stream = torch.cuda.Stream(device=0)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.tcpt_render_adaptive_device(ctx.handle, C.byref(mine), C.byref(ap), C.c_void_p(acc.data_ptr()), C.c_void_p(spp.data_ptr()),
                                                  C.c_void_p(stream.cuda_stream)))
    stream.synchronize()
    return acc.cpu().numpy(), spp.cpu().numpy().view(np.uint32), ctx.stats()


def _rank_by_rank(b, integrator, sampler, world, ap, max_slots=0):
    """Every rank's shard in turn, summed as the reduce would sum them; also the summed paths."""
    ctx = b.scene.ctx
    job = b.image(integrator, N).renderer.params(sampler, max_slots=max_slots)
    acc = np.zeros((H, W, 3), dtype=f32); cnt = np.zeros((H, W), dtype=np.uint32); paths = 0
    for r in range(world):
        a, c, st = _render_shard(ctx, _shard(ctx, job, r, world), ap)
        acc += a; cnt += c; paths += st["paths"]
    return acc, cnt, paths


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,integrator,sampler", [(3, "mis", "sobol"), (19, "mis", "sobol"), (3, "pt", "random")])
def test_adaptive_shards_rendered_rank_by_rank_sum_to_the_one_gpu_frame(bundle_factory, scene_id, integrator, sampler):
    from toy_cpu_pathtracing_b200 import capi
    b = bundle_factory(scene_id, W, H)
    ref = b.image(integrator, N).render_adaptive(sampler, threshold=THR, min_spp=MIN_SPP, step=STEP)
    ref_acc, ref_cnt = ref.accumulators.copy(), ref.sample_counts.copy()
    assert len(np.unique(ref_cnt)) >= 2            # some pixels stop, some go on
    ap = capi.AdaptiveParams(THR, MIN_SPP, STEP)
    for world in (2, 3, 5, 8, H + 2):              # H + 2: two ranks own no row
        acc, cnt, paths = _rank_by_rank(b, integrator, sampler, world, ap)
        assert np.array_equal(cnt, ref_cnt), f"world {world}: {(cnt != ref_cnt).sum()} counts differ"
        assert np.array_equal(_bits(acc), _bits(ref_acc)), f"world {world}: accumulators differ"
        assert paths == int(ref_cnt.sum()), world


@pytest.mark.gpu
def test_adaptive_shard_writes_only_its_own_rows(bundle_factory):
    from toy_cpu_pathtracing_b200 import capi
    b = bundle_factory(3, W, H)
    ctx = b.scene.ctx
    ref = b.image("mis", N).render_adaptive("sobol", threshold=THR, min_spp=MIN_SPP, step=STEP)
    job = b.image("mis", N).renderer.params("sobol")
    ap = capi.AdaptiveParams(THR, MIN_SPP, STEP)
    world = 3
    rng = np.random.default_rng(5)
    acc0 = rng.standard_normal((H, W, 3)).astype(f32)
    spp0 = np.full((H, W), 0xDEADBEEF, dtype=np.uint32)
    for r in range(world):
        acc, cnt, st = _render_shard(ctx, _shard(ctx, job, r, world), ap, acc0, spp0)
        mine = np.arange(H) % world == r
        assert np.array_equal(_bits(acc[~mine]), _bits(acc0[~mine])), r
        assert (cnt[~mine] == 0xDEADBEEF).all(), r
        assert np.array_equal(cnt[mine], ref.sample_counts[mine]), r
        assert st["paths"] == int(ref.sample_counts[mine].sum()), r


@pytest.mark.gpu
def test_adaptive_shard_edges(bundle_factory):
    from toy_cpu_pathtracing_b200 import capi
    world = 3
    b = bundle_factory(3, W, H)
    # threshold 0: no pixel ever stops, the frame is tcpt_render's tile film
    full = b.image("mis", N).render("sobol").accumulators.copy()
    acc, cnt, paths = _rank_by_rank(b, "mis", "sobol", world, capi.AdaptiveParams(0.0, MIN_SPP, STEP))
    assert (cnt == N).all() and paths == W * H * N
    assert np.array_equal(_bits(acc), _bits(full))
    # threshold 1e30: every finite pixel stops at min_spp
    acc, cnt, paths = _rank_by_rank(b, "mis", "sobol", world, capi.AdaptiveParams(1e30, MIN_SPP, STEP))
    assert np.isfinite(acc).all() and (cnt == MIN_SPP).all() and paths == W * H * MIN_SPP
    # scene 11 under MIS has NaN pixels (DESIGN.md section 5): they run to N in every shard
    b11 = bundle_factory(11, W, H)
    ctx = b11.scene.ctx
    job = b11.image("mis", N).renderer.params("sobol")
    seen_bad = 0
    for r in range(world):
        a, c, _ = _render_shard(ctx, _shard(ctx, job, r, world), capi.AdaptiveParams(1e30, MIN_SPP, STEP))
        mine = np.arange(H) % world == r
        bad = ~np.isfinite(a[mine]).all(axis=2)
        seen_bad += int(bad.sum())
        assert (c[mine][bad] == N).all() and (c[mine][~bad] == MIN_SPP).all(), r
    assert seen_bad > 0


@pytest.mark.gpu
def test_adaptive_shard_is_deterministic_across_pass_tilings(bundle_factory):
    from toy_cpu_pathtracing_b200 import capi
    b = bundle_factory(19, W, H)
    ctx = b.scene.ctx
    ap = capi.AdaptiveParams(THR, MIN_SPP, STEP)
    mine = _shard(ctx, b.image("mis", N).renderer.params("sobol"), 1, 3)
    a0, c0, st0 = _render_shard(ctx, mine, ap)
    mine.max_slots = 2000
    a1, c1, st1 = _render_shard(ctx, mine, ap)
    assert st1["passes"] > st0["passes"]          # the slot budget cut rounds into several passes
    assert len(np.unique(c0[1::3])) >= 2
    assert np.array_equal(c1, c0) and np.array_equal(_bits(a1), _bits(a0))


@pytest.mark.gpu
def test_render_adaptive_sharded_without_a_communicator_is_render_adaptive(bundle_factory):
    b = bundle_factory(19, W, H)
    a = b.image("mis", N).render_adaptive("sobol", threshold=THR, min_spp=MIN_SPP, step=STEP)
    s = b.image("mis", N).render_adaptive_sharded("sobol", threshold=THR, min_spp=MIN_SPP, step=STEP)
    assert np.array_equal(s.sample_counts, a.sample_counts)
    assert np.array_equal(_bits(s.accumulators), _bits(a.accumulators))
    assert np.array_equal(_bits(s.pixels), _bits(a.pixels))
    assert s.stats["reduce_ms"] == 0.0
    assert s.stats["paths"] == a.stats["paths"] == int(a.sample_counts.sum())
    assert s.stats["rounds"] == a.stats["rounds"]


def n_gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
@pytest.mark.skipif(n_gpus() < 2, reason="needs two GPUs")
def test_two_ranks_reproduce_the_one_gpu_adaptive_frame(tmp_path):
    """Two processes, one GPU each (torchrun): tcpt_comm_init + tcpt_render_adaptive_sharded; rank 0 compares with its own one-GPU frame."""
    port = 29600 + (os.getpid() + 150) % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(port),
           str(ROOT / "tests" / "mgpu_adaptive_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "MGPU_ADAPTIVE_OK" in r.stdout, r.stdout[-2000:]


@pytest.mark.gpu
@pytest.mark.skipif(n_gpus() < 2, reason="needs two GPUs")
def test_group_render_adaptive_two_gpus(tables):
    """tcpt_group_render_adaptive: one host process, one context and one host thread per GPU, the one-GPU adaptive frame out."""
    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import capi, scenes
    lib = capi.load_library()
    w, h = 200, 150
    scene = tp.Scene(device=0)
    cam = tp.Camera(45.0, w, h)
    scenes.load_scene(19, scene, cam)
    scene.build(cam)
    ref = tp.RendererImage(w, h, tp.SrgbRendererMis(tp.RendererArgs((w, h), N, scene, cam))).render_adaptive(
        "sobol", threshold=THR, min_spp=MIN_SPP, step=STEP)
    g = C.c_void_p()
    assert lib.tcpt_group_create((C.c_int32 * 2)(0, 1), 2, C.byref(g)) == 0, lib.tcpt_group_last_error(g)
    try:
        std, tab = tables
        assert lib.tcpt_group_set_tables(g, std, len(std), capi.as_ptr(tab, C.c_float), tab.size) == 0
        ctx0 = capi.Context.__new__(capi.Context)          # a borrowed handle: the group owns the context
        ctx0.lib, ctx0.handle, ctx0.has_gpu, ctx0.comm_rank, ctx0.comm_size = lib, C.c_void_p(lib.tcpt_group_context(g, 0)), True, 0, 2
        gs = tp.Scene(context=ctx0)
        scenes.load_scene(19, gs, tp.Camera(45.0, w, h))
        lib.tcpt_scene_clear(ctx0.handle)
        gs.desc.replay(gs)
        pos = np.asarray(cam.position, dtype=np.float32)
        assert lib.tcpt_group_build(g, capi.as_ptr(pos, C.c_float)) == 0, lib.tcpt_group_last_error(g)
        p = tp.SrgbRendererMis(tp.RendererArgs((w, h), N, gs, cam)).params("sobol")
        ap = capi.AdaptiveParams(THR, MIN_SPP, STEP)
        acc = np.zeros((h, w, 3), f32); srgb = np.zeros((h, w, 3), f32); cnt = np.zeros((h, w), np.uint32)
        assert lib.tcpt_group_render_adaptive(g, C.byref(p), C.byref(ap), capi.as_ptr(acc, C.c_float), capi.as_ptr(srgb, C.c_float),
                                              capi.as_ptr(cnt, C.c_uint32)) == 0, lib.tcpt_group_last_error(g)
        assert np.array_equal(cnt, ref.sample_counts)
        assert np.array_equal(_bits(acc), _bits(ref.accumulators))
        assert np.array_equal(_bits(srgb), _bits(ref.pixels))
        s0, s1 = capi.Stats(), capi.Stats()
        lib.tcpt_get_stats(lib.tcpt_group_context(g, 0), C.byref(s0)); lib.tcpt_get_stats(lib.tcpt_group_context(g, 1), C.byref(s1))
        assert s0.paths + s1.paths == int(ref.sample_counts.sum()) and s0.paths > 0 and s1.paths > 0
        assert s0.reduce_ms > 0.0
        # tcpt_render_adaptive on ONE context of the group (each holds a communicator) is that GPU's own whole frame: no collective
        for i in range(2):
            acc[:] = 7.0; srgb[:] = 7.0; cnt[:] = 7
            assert lib.tcpt_render_adaptive(lib.tcpt_group_context(g, i), C.byref(p), C.byref(ap), capi.as_ptr(acc, C.c_float),
                                            capi.as_ptr(srgb, C.c_float), capi.as_ptr(cnt, C.c_uint32)) == 0, i
            assert np.array_equal(cnt, ref.sample_counts), i
            assert np.array_equal(_bits(acc), _bits(ref.accumulators)), i
            assert np.array_equal(_bits(srgb), _bits(ref.pixels)), i
            st = capi.Stats()
            lib.tcpt_get_stats(lib.tcpt_group_context(g, i), C.byref(st))
            assert st.paths == int(ref.sample_counts.sum()) and st.reduce_ms == 0.0, i
        ctx0.handle = C.c_void_p()     # do not destroy the borrowed context
    finally:
        lib.tcpt_group_destroy(g)
