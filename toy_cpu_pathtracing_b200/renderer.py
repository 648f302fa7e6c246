"""Host-side mirror of the reference's renderer entry point (renderer/src/renderer.rs:84-149, camera.rs, main.rs:142-237).

`RendererImage(width, height, SrgbRendererMis(args, tone_map, exposure, max_depth)).render(ZSobolSampler)` is the call a user
of the reference makes; here it renders the WHOLE frame on the GPU through libtcpt's `tcpt_render` (host buffers in and
out) instead of one rayon task per pixel.  Nothing in this module computes radiance on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .scene import Scene

f32 = np.float32


class BoxFilter:                      # renderer/src/filter.rs:13-30 (only width 1.0 is ever constructed: main.rs:60)
    def __init__(self, width: float = 1.0):
        if width != 1.0:
            raise ValueError("the GPU path implements the reference's only filter configuration, BoxFilter::new(1.0)")
        self.width = width


class Camera:                         # renderer/src/camera.rs:14-86
    def __init__(self, fov: float, width: int, height: int, filter: BoxFilter | None = None):
        self.fov, self.width, self.height = float(fov), int(width), int(height)
        self.filter = filter or BoxFilter(1.0)
        self.position = np.zeros(3, dtype=f32)
        self.direction = np.array([0, 0, -1], dtype=f32)
        self.up = np.array([0, 1, 0], dtype=f32)

    def set_look_to(self, position, direction, up):
        self.position = np.asarray(position, dtype=f32)
        self.direction = np.asarray(direction, dtype=f32)
        self.up = np.asarray(up, dtype=f32)


class RandomSampler:                  # renderer/src/sampler/random_sampler.rs (counter RNG stand-in for ThreadRng)
    name = "random"


class ZSobolSampler:                  # renderer/src/sampler/z_sobol_sampler.rs
    name = "sobol"


class ReinhardToneMap:                # renderer/src/tone_map.rs:20-28 (the only tone map main.rs constructs)
    pass


@dataclass
class RendererArgs:                   # renderer/src/renderer.rs:84-90
    resolution: tuple
    spp: int
    scene: Scene
    camera: Camera
    seed: int = 0


class _SrgbRenderer:
    integrator = "pt"

    def __init__(self, args: RendererArgs, tone_map=None, exposure: float = 1.0, max_depth: int = 16):
        self.args, self.tone_map, self.exposure, self.max_depth = args, tone_map or ReinhardToneMap(), float(exposure), int(max_depth)

    new = classmethod(lambda cls, *a, **k: cls(*a, **k))

    def params(self, sampler, **shard) -> capi.RenderParams:
        a, cam = self.args, self.args.camera
        p = capi.RenderParams()
        p.width, p.height, p.spp, p.seed, p.max_depth = a.resolution[0], a.resolution[1], a.spp, a.seed, self.max_depth
        p.integrator = capi.INTEGRATORS[self.integrator]
        p.sampler = capi.SAMPLERS[sampler if isinstance(sampler, str) else sampler.name]
        p.exposure, p.fov_deg = self.exposure, cam.fov
        for k in range(3):
            p.cam_pos[k], p.cam_dir[k], p.cam_up[k] = float(cam.position[k]), float(cam.direction[k]), float(cam.up[k])
        p.row_offset, p.row_stride = shard.get("row_offset", 0), shard.get("row_stride", 0)
        p.spp_begin, p.spp_end = shard.get("spp_begin", 0), shard.get("spp_end", 0)
        p.max_slots = shard.get("max_slots", 0)
        return p


class SrgbRendererPt(_SrgbRenderer):   # renderer/src/renderer/pt_renderer.rs:85-101
    integrator = "pt"


class SrgbRendererNee(_SrgbRenderer):  # renderer/src/renderer/nee_renderer.rs:166-182
    integrator = "nee"


class SrgbRendererMis(_SrgbRenderer):  # renderer/src/renderer/mis_renderer.rs:233-249
    integrator = "mis"


class AlbedoRenderer(_SrgbRenderer):   # renderer/src/renderer/albedo_renderer.rs (AOV: albedo under D65 at the first hit, no tone map)
    integrator = "albedo"

    def __init__(self, args: RendererArgs, **_):
        super().__init__(args, exposure=1.0, max_depth=0)


class NormalRenderer(_SrgbRenderer):   # renderer/src/renderer/normal_renderer.rs (AOV: shading normal * 0.5 + 0.5 at the first hit)
    integrator = "normal"

    def __init__(self, args: RendererArgs, **_):
        super().__init__(args, exposure=1.0, max_depth=0)


RENDERERS = {"pt": SrgbRendererPt, "nee": SrgbRendererNee, "mis": SrgbRendererMis, "albedo": AlbedoRenderer, "normal": NormalRenderer}


def _rounds(sample_counts, min_spp, step) -> int:
    """Rounds an adaptive frame took.  The last round ends at the largest count: round 0 reaches min_spp, every later one `step` more
    (the last clipped at spp)."""
    return 1 + -(-(int(sample_counts.max()) - int(min_spp)) // int(step))


class RendererImage:                  # renderer/src/renderer.rs:101-149
    def __init__(self, width: int, height: int, renderer: _SrgbRenderer):
        self.width, self.height, self.renderer = int(width), int(height), renderer
        self.pixels = np.zeros((self.height, self.width, 3), dtype=f32)       # tone-mapped sRGB, what `pixels` holds in the reference
        self.accumulators = np.zeros((self.height, self.width, 3), dtype=f32)  # Sensor accumulators (linear sRGB sums)
        self.sample_counts = np.zeros((self.height, self.width), dtype=np.uint32)  # samples per pixel of the last render_adaptive
        self.stats: dict = {}

    @classmethod
    def new(cls, width, height, renderer):
        return cls(width, height, renderer)

    def render(self, sampler=ZSobolSampler, want_accumulators: bool = True, **shard) -> "RendererImage":
        r = self.renderer
        ctx = r.args.scene.ctx
        if not r.args.scene.built:
            r.args.scene.build(r.args.camera)
        p = r.params(sampler, **shard)
        # `pixels` / `accumulators` live as long as this image: let libtcpt page-lock them once for direct DMA
        ctx.set_option("pin_host_buffers", 1)
        self._pinned_ctx = ctx
        ctx.check(ctx.lib.tcpt_render(ctx.handle, C.byref(p), capi.as_ptr(self.accumulators, C.c_float) if want_accumulators else None,
                                      capi.as_ptr(self.pixels, C.c_float)))
        self.stats = ctx.stats()
        return self

    def render_adaptive(self, sampler=ZSobolSampler, threshold: float = 0.01, min_spp: int = 64, step: int = 64,
                        want_accumulators: bool = True, max_slots: int = 0) -> "RendererImage":
        """Adaptive sampling (tcpt_render_adaptive): every pixel renders samples [0, min_spp), then `step` more per round while the
        relative standard error of its mean luminance is at least `threshold` (absolute floor 1e-3), up to the renderer's spp.
        `sample_counts` receives each pixel's count k; its accumulator is bitwise what `render` gives for the sample window [0, k) of the
        same job, and `pixels` holds the output transform of accumulator / k.  stats["rounds"] = rounds the job took."""
        r = self.renderer
        ctx = r.args.scene.ctx
        if not r.args.scene.built:
            r.args.scene.build(r.args.camera)
        p = r.params(sampler, max_slots=max_slots)
        ap = capi.AdaptiveParams(float(threshold), int(min_spp), int(step))
        ctx.set_option("pin_host_buffers", 1)
        self._pinned_ctx = ctx
        ctx.check(ctx.lib.tcpt_render_adaptive(ctx.handle, C.byref(p), C.byref(ap),
                                               capi.as_ptr(self.accumulators, C.c_float) if want_accumulators else None,
                                               capi.as_ptr(self.pixels, C.c_float), capi.as_ptr(self.sample_counts, C.c_uint32)))
        self.stats = ctx.stats()
        self.stats["rounds"] = _rounds(self.sample_counts, min_spp, step)
        return self

    def render_adaptive_sharded(self, sampler=ZSobolSampler, threshold: float = 0.01, min_spp: int = 64, step: int = 64,
                                want_accumulators: bool = True, max_slots: int = 0) -> "RendererImage":
        """`render_adaptive` from every GPU of the communicator (tcpt_render_adaptive_sharded; tcpt_comm_init on each rank's context):
        every rank calls this with the same arguments and runs the rounds over its image rows y % N == rank alone; ONE grouped
        ncclReduce of the accumulators and the counts inside libtcpt hands rank 0 the frame, bitwise the one-GPU `render_adaptive` frame.
        `pixels`, `accumulators` and `sample_counts` are filled on rank 0 only; there stats["rounds"] = rounds of the frame."""
        r = self.renderer
        ctx = r.args.scene.ctx
        if not r.args.scene.built:
            r.args.scene.build(r.args.camera)
        p = r.params(sampler, max_slots=max_slots)
        ap = capi.AdaptiveParams(float(threshold), int(min_spp), int(step))
        root = ctx.comm_rank == 0
        if root:
            ctx.set_option("pin_host_buffers", 1)
            self._pinned_ctx = ctx
        ctx.check(ctx.lib.tcpt_render_adaptive_sharded(ctx.handle, C.byref(p), C.byref(ap),
                                                       capi.as_ptr(self.accumulators, C.c_float) if (root and want_accumulators) else None,
                                                       capi.as_ptr(self.pixels, C.c_float) if root else None,
                                                       capi.as_ptr(self.sample_counts, C.c_uint32) if root else None))
        self.stats = ctx.stats()
        if root:
            self.stats["rounds"] = _rounds(self.sample_counts, min_spp, step)
        return self

    def render_sharded(self, sampler=ZSobolSampler, mode: str = "tile", want_accumulators: bool = True, spp_window=None, max_slots: int = 0) -> "RendererImage":
        """One complete frame from every GPU of the communicator (tcpt_comm_init on each rank's context): every rank calls this with the
        same arguments, renders its shard (mode "tile": image rows y % N == rank, bitwise equal to one GPU; "spp": an equal slice of the
        sample indices), ONE ncclReduce inside libtcpt sums the film onto rank 0, which tone-maps and copies out: `pixels` /
        `accumulators` are filled on rank 0 only.  spp_window = (begin, end) restricts the whole job to a block of sample indices."""
        r = self.renderer
        ctx = r.args.scene.ctx
        if not r.args.scene.built:
            r.args.scene.build(r.args.camera)
        kw = {"spp_begin": spp_window[0], "spp_end": spp_window[1]} if spp_window else {}
        p = r.params(sampler, max_slots=max_slots, **kw)
        root = ctx.comm_rank == 0
        if root:
            ctx.set_option("pin_host_buffers", 1)
            self._pinned_ctx = ctx
        ctx.check(ctx.lib.tcpt_render_sharded(ctx.handle, C.byref(p), capi.SHARD_MODES[mode],
                                              capi.as_ptr(self.accumulators, C.c_float) if (root and want_accumulators) else None,
                                              capi.as_ptr(self.pixels, C.c_float) if root else None))
        self.stats = ctx.stats()
        return self

    def __del__(self):
        ctx = getattr(self, "_pinned_ctx", None)
        if ctx is not None and getattr(ctx, "handle", None):
            try:
                ctx.set_option("pin_host_buffers", 0)   # release the page locks before the arrays are freed
            except Exception:
                pass

    def path_samples(self, sampler, pixels_xy, sample_indices) -> np.ndarray:
        """Sensor contribution of individual (pixel, sample) paths (parity probe)."""
        r = self.renderer
        ctx = r.args.scene.ctx
        p = r.params(sampler)
        xy = np.ascontiguousarray(pixels_xy, dtype=np.uint32)
        si = np.ascontiguousarray(sample_indices, dtype=np.uint32)
        out = np.zeros((len(si), 3), dtype=f32)
        ctx.check(ctx.lib.tcpt_path_samples(ctx.handle, C.byref(p), capi.as_ptr(xy, C.c_uint32), capi.as_ptr(si, C.c_uint32), len(si), capi.as_ptr(out, C.c_float)))
        self.stats = ctx.stats()
        return out

    def to_u8(self) -> np.ndarray:
        # (v * 255.0) as u8: truncating, saturating (renderer.rs:140-144)
        return np.clip(np.nan_to_num(self.pixels * f32(255.0), nan=0.0), 0, 255).astype(np.uint8)

    def save(self, path) -> None:
        import cv2
        cv2.imwrite(str(path), self.to_u8()[..., ::-1])
