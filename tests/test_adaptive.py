"""Adaptive sampling (tcpt_render_adaptive / RendererImage.render_adaptive): argument checks on any box, and on the GPU the prefix
property (a pixel that stopped after k samples holds bitwise the film of the sample window [0, k) of the same job), the stopping rule
restated in numpy, the edge cases and determinism."""
import ctypes as C

import numpy as np
import pytest

f32 = np.float32


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


def _call(ctx, p, ap, acc, srgb, spp):
    from toy_cpu_pathtracing_b200 import capi
    return ctx.lib.tcpt_render_adaptive(ctx.handle if ctx is not None else None, C.byref(p) if p is not None else None,
                                        C.byref(ap) if ap is not None else None,
                                        capi.as_ptr(acc, C.c_float) if acc is not None else None,
                                        capi.as_ptr(srgb, C.c_float) if srgb is not None else None,
                                        capi.as_ptr(spp, C.c_uint32) if spp is not None else None)


def test_adaptive_params_layout(built):
    from toy_cpu_pathtracing_b200 import capi
    assert C.sizeof(capi.AdaptiveParams) == 12
    assert [f for f, _ in capi.AdaptiveParams._fields_] == ["threshold", "min_spp", "step"]


def test_adaptive_refusals_are_invalid(built):
    """Every malformed request is refused with TCPT_ERR_INVALID before the device is looked at, so this holds with or without a GPU."""
    from toy_cpu_pathtracing_b200 import capi
    ctx = capi.Context(0, require_gpu=False)
    lib = ctx.lib
    acc = np.zeros(48, dtype=f32); srgb = np.zeros(48, dtype=f32); spp = np.zeros(16, dtype=np.uint32)
    good = capi.AdaptiveParams(0.01, 4, 4)
    AP = capi.AdaptiveParams
    assert lib.tcpt_render_adaptive(None, C.byref(_params()), C.byref(good), capi.as_ptr(acc, C.c_float), None, None) == capi.TCPT_ERR_INVALID
    cases = [
        (_params(), None, (acc, srgb, spp)),                                   # null ap
        (None, good, (acc, srgb, spp)),                                        # null params
        (_params(), good, (None, None, None)),                                 # no output
        (_params(), AP(-0.01, 4, 4), (acc, None, None)),                       # negative threshold
        (_params(), AP(float("nan"), 4, 4), (acc, None, None)),                # not finite
        (_params(), AP(float("inf"), 4, 4), (None, srgb, None)),
        (_params(), AP(0.01, 1, 4), (acc, None, None)),                        # min_spp < 2
        (_params(), AP(0.01, 0, 4), (acc, None, None)),
        (_params(), AP(0.01, 17, 4), (None, None, spp)),                       # min_spp > spp
        (_params(), AP(0.01, 4, 0), (acc, None, None)),                        # step 0
        (_params(integrator=capi.INTEGRATORS["albedo"]), good, (acc, None, None)),
        (_params(integrator=capi.INTEGRATORS["normal"]), good, (acc, None, None)),
        (_params(row_stride=2), good, (acc, None, None)),
        (_params(row_offset=1), good, (acc, None, None)),
        (_params(spp_begin=4), good, (acc, None, None)),
        (_params(spp_end=8), good, (acc, None, None)),
    ]
    for i, (p, ap, outs) in enumerate(cases):
        assert _call(ctx, p, ap, *outs) == capi.TCPT_ERR_INVALID, i
    assert not acc.any() and not srgb.any() and not spp.any()


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="GPU present")
def test_adaptive_without_gpu_writes_nothing(built):
    from toy_cpu_pathtracing_b200 import capi
    ctx = capi.Context(0, require_gpu=False)
    assert not ctx.has_gpu
    acc = np.full(48, 7.0, dtype=f32); srgb = np.full(48, 7.0, dtype=f32); spp = np.full(16, 7, dtype=np.uint32)
    rc = _call(ctx, _params(), capi.AdaptiveParams(0.01, 4, 4), acc, srgb, spp)
    assert rc == capi.TCPT_ERR_CUDA
    assert (acc == 7.0).all() and (srgb == 7.0).all() and (spp == 7).all()


# ---------------------------------------------------------------- GPU
def _bits(a):
    return np.ascontiguousarray(a, dtype=f32).view(np.uint32)


def _finalize_device(ctx, acc, spp):
    """tcpt_finalize_device of a host accumulator (H x W x 3) with the given spp."""
    import torch
    d_acc = torch.from_numpy(np.ascontiguousarray(acc, dtype=f32)).cuda()
    d_out = torch.empty_like(d_acc)
    torch.cuda.synchronize()
    h, w = acc.shape[:2]
    ctx.check(ctx.lib.tcpt_finalize_device(ctx.handle, C.c_void_p(d_acc.data_ptr()), w, h, int(spp), C.c_void_p(d_out.data_ptr()), None))
    return d_out.cpu().numpy()


def _rounds(counts, min_spp, step):
    return 1 + -(-(int(counts.max()) - min_spp) // step)


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,integrator,sampler", [(3, "mis", "sobol"), (19, "mis", "sobol"), (3, "pt", "random")])
def test_adaptive_pixels_are_prefixes_of_the_job(bundle_factory, scene_id, integrator, sampler):
    N, min_spp, step, thr = 1024, 64, 64, 0.02
    b = bundle_factory(scene_id, 200, 150)
    ad = b.image(integrator, N).render_adaptive(sampler, threshold=thr, min_spp=min_spp, step=step)
    counts, acc, srgb = ad.sample_counts.copy(), ad.accumulators.copy(), ad.pixels.copy()
    assert ad.stats["paths"] == int(counts.sum())
    ks = np.unique(counts)
    assert len(ks) >= 2, ks                               # some pixels stop, some go on
    assert all(k == N or (k - min_spp) % step == 0 for k in ks.tolist()), ks
    assert ad.stats["rounds"] == _rounds(counts, min_spp, step)
    for k in ks:
        k = int(k)
        sel = counts == k
        win = b.image(integrator, N).render(sampler, spp_begin=0, spp_end=k).accumulators.copy()
        assert np.array_equal(_bits(acc[sel]), _bits(win[sel])), f"count {k}: accumulators differ"
        fin = _finalize_device(b.scene.ctx, win, k)
        assert np.array_equal(_bits(srgb[sel]), _bits(fin[sel])), f"count {k}: sRGB differs"


def _restated_counts(rgb, thresholds, min_spp, step, N):
    """The stopping rule of include/tcpt.h in numpy f32, in sample order: rgb = (pixels, N, 3) per-path sensor contributions."""
    r, g, b = rgb[..., 0], rgb[..., 1], rgb[..., 2]
    y = (f32(0.2126) * r + f32(0.7152) * g) + f32(0.0722) * b
    s1 = np.add.accumulate(y, axis=1, dtype=f32)
    s2 = np.add.accumulate(y * y, axis=1, dtype=f32)
    out = {}
    with np.errstate(all="ignore"):
        for thr in thresholds:
            counts = np.full(rgb.shape[0], N, dtype=np.uint32)
            active = np.ones(rgb.shape[0], dtype=bool)
            k = min_spp
            while k < N:
                kf = f32(k)
                S1, S2 = s1[:, k - 1], s2[:, k - 1]
                m = S1 / kf
                v = S2 / kf - m * m
                v = np.where(v > 0, v, f32(0))
                e = np.sqrt(v / (kf - f32(1)))
                stop = active & np.isfinite(S1) & np.isfinite(S2) & (e < f32(thr) * (np.abs(m) + f32(1e-3)))
                counts[stop] = k
                active &= ~stop
                k = min(k + step, N)
            out[thr] = counts
    return out


@pytest.mark.gpu
def test_adaptive_counts_follow_the_stated_rule(bundle_factory):
    w, h, N, min_spp, step = 64, 48, 256, 32, 32
    b = bundle_factory(19, w, h)
    ys, xs = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    pix = np.stack([xs.ravel(), ys.ravel()], 1).astype(np.uint32)              # frame order
    xy = np.repeat(pix, N, axis=0)
    si = np.tile(np.arange(N, dtype=np.uint32), w * h)
    rgb = b.image("mis", N).path_samples("sobol", xy, si).reshape(w * h, N, 3)
    want = _restated_counts(rgb, (0.02, 0.005), min_spp, step, N)
    seen = set()
    for thr, counts in want.items():
        got = b.image("mis", N).render_adaptive("sobol", threshold=thr, min_spp=min_spp, step=step).sample_counts.ravel()
        assert np.array_equal(got, counts), f"threshold {thr}: {(got != counts).sum()} pixels differ"
        seen.add(len(np.unique(counts)))
    assert max(seen) >= 3        # the rule did decide something at this size


@pytest.mark.gpu
def test_adaptive_edges(bundle_factory):
    N, min_spp, step = 256, 32, 32
    b = bundle_factory(3, 64, 48)
    ref = b.image("mis", N).render("sobol")
    ref_acc, ref_srgb = ref.accumulators.copy(), ref.pixels.copy()
    for kw in (dict(threshold=0.0, min_spp=min_spp, step=step), dict(threshold=0.02, min_spp=N, step=step)):
        ad = b.image("mis", N).render_adaptive("sobol", **kw)
        assert (ad.sample_counts == N).all(), kw
        assert np.array_equal(_bits(ad.accumulators), _bits(ref_acc)), kw
        assert np.array_equal(_bits(ad.pixels), _bits(ref_srgb)), kw
        assert ad.stats["paths"] == int(ad.sample_counts.sum()) == 64 * 48 * N
    ad = b.image("mis", N).render_adaptive("sobol", threshold=1e30, min_spp=min_spp, step=step)
    finite = np.isfinite(ad.accumulators).all(axis=2)
    assert finite.all() and (ad.sample_counts == min_spp).all()
    assert ad.stats["paths"] == int(ad.sample_counts.sum()) and ad.stats["rounds"] == 1
    # scene 11 under MIS has NaN pixels (DESIGN.md section 5): they never stop
    b11 = bundle_factory(11, 64, 48)
    ad = b11.image("mis", N).render_adaptive("sobol", threshold=1e30, min_spp=min_spp, step=step)
    bad = ~np.isfinite(ad.accumulators).all(axis=2)
    assert bad.any()
    assert (ad.sample_counts[bad] == N).all() and (ad.sample_counts[~bad] == min_spp).all()
    assert ad.stats["paths"] == int(ad.sample_counts.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,N,min_spp,step,max_slots", [(200, 150, 1024, 64, 64, 200 * 150 * 16), (64, 48, 256, 32, 32, 2000)])
def test_adaptive_is_deterministic(bundle_factory, w, h, N, min_spp, step, max_slots):
    b = bundle_factory(19, w, h)

    def run(**kw):
        ad = b.image("mis", N).render_adaptive("sobol", threshold=0.02, min_spp=min_spp, step=step, **kw)
        return ad.accumulators.copy(), ad.pixels.copy(), ad.sample_counts.copy(), ad.stats

    a0, s0, c0, st0 = run()
    a1, s1, c1, _ = run()
    a2, s2, c2, st2 = run(max_slots=max_slots)
    assert st2["passes"] > st0["passes"]          # the slot budget cut rounds into several passes
    assert len(np.unique(c0)) >= 2
    for a, s, c in ((a1, s1, c1), (a2, s2, c2)):
        assert np.array_equal(c, c0)
        assert np.array_equal(_bits(a), _bits(a0))
        assert np.array_equal(_bits(s), _bits(s0))
