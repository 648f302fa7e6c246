"""ctypes binding of libtcpt (include/tcpt.h).  This is the only way the Python host mirror reaches the hot path; the
library is hand-written CUDA for sm_100a and there is no CPU fallback: if it is missing, loading raises."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "lib" / "libtcpt.so"
DATA_DIR = PKG_DIR / "data"

TCPT_OK, TCPT_ERR_INVALID, TCPT_ERR_CUDA, TCPT_ERR_LIMIT, TCPT_ERR_NOMEM = 0, -1, -2, -3, -4
INTEGRATORS = {"pt": 0, "nee": 1, "mis": 2, "albedo": 3, "normal": 4}
SAMPLERS = {"random": 0, "sobol": 1}
MAT_LAMBERT, MAT_EMISSIVE, MAT_PLASTIC, MAT_SIMPLE_PBR, MAT_CLEARCOAT_PBR, MAT_METAL, MAT_GLASS = range(7)
SPEC_CONSTANT, SPEC_RGB_ALBEDO_SRGB, SPEC_RGB_ALBEDO_LINEAR, SPEC_D65, SPEC_TEXTURE_SRGB, SPEC_PRESET = range(6)
LIGHT_POINT, LIGHT_SPOT, LIGHT_DIRECTIONAL = 3, 4, 5
SHARD_MODES = {"tile": 0, "spp": 1}
COMM_ID_BYTES = 128
# TCPT_PRESET_* (include/tcpt.h): presets::au_eta() ... presets::glass_sf11_eta() in the order data/std_tables.bin stores them
PRESETS = ["au_eta", "au_k", "ag_eta", "ag_k", "cu_eta", "cu_k", "al_eta", "al_k", "cu_zn_eta", "cu_zn_k",
           "glass_bk7_eta", "glass_baf10_eta", "glass_fk51a_eta", "glass_lasf9_eta", "glass_sf5_eta", "glass_sf10_eta", "glass_sf11_eta"]


class TcptError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libtcpt error {code}: {message}")
        self.code = code


class SpectrumParam(C.Structure):
    _fields_ = [("kind", C.c_int32), ("value", C.c_float * 3), ("texture", C.c_int32)]


class FloatParam(C.Structure):
    _fields_ = [("kind", C.c_int32), ("value", C.c_float), ("texture", C.c_int32), ("gamma_corrected", C.c_int32)]


class NormalParam(C.Structure):
    _fields_ = [("texture", C.c_int32), ("flip_y", C.c_int32)]


class MaterialDesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("color", SpectrumParam), ("intensity", FloatParam), ("normal", NormalParam),
                ("eta", C.c_float), ("thin_surface", C.c_int32),
                ("roughness", FloatParam), ("metallic", FloatParam), ("ior", FloatParam),
                ("coat_ior", FloatParam), ("coat_roughness", FloatParam), ("coat_thickness", FloatParam),
                ("coat_tint", SpectrumParam)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("seed", C.c_uint32), ("max_depth", C.c_uint32),
                ("integrator", C.c_int32), ("sampler", C.c_int32), ("exposure", C.c_float), ("fov_deg", C.c_float),
                ("cam_pos", C.c_float * 3), ("cam_dir", C.c_float * 3), ("cam_up", C.c_float * 3),
                ("row_offset", C.c_uint32), ("row_stride", C.c_uint32), ("spp_begin", C.c_uint32), ("spp_end", C.c_uint32),
                ("max_slots", C.c_uint32)]


class AdaptiveParams(C.Structure):   # tcpt_adaptive_params
    _fields_ = [("threshold", C.c_float), ("min_spp", C.c_uint32), ("step", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("paths", C.c_uint64), ("closest_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("box_tests", C.c_uint64),
                ("tri_tests", C.c_uint64), ("kernel_launches", C.c_uint64), ("render_ms", C.c_double),
                ("trace_closest_ms", C.c_double), ("trace_shadow_ms", C.c_double), ("shade_ms", C.c_double),
                ("generate_ms", C.c_double), ("film_ms", C.c_double), ("passes", C.c_uint32), ("max_bvh_depth", C.c_uint32),
                ("sobol_prefix_ms", C.c_double), ("sobol_prefix_bytes", C.c_uint64), ("reduce_ms", C.c_double), ("trace_launches", C.c_uint32), ("shade_launches", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/tcpt.h and include/tcpt_flat.h declare (tests check the library exports all of them)
EXPORTED_SYMBOLS = [
    "tcpt_create", "tcpt_destroy", "tcpt_last_error", "tcpt_set_option", "tcpt_set_tables", "tcpt_scene_clear",
    "tcpt_scene_add_mesh", "tcpt_scene_add_single_triangle", "tcpt_scene_add_texture", "tcpt_scene_add_material", "tcpt_scene_add_primitive",
    "tcpt_scene_add_env_light", "tcpt_scene_add_delta_light", "tcpt_scene_build", "tcpt_render", "tcpt_render_device", "tcpt_finalize_device",
    "tcpt_render_adaptive", "tcpt_render_adaptive_device", "tcpt_render_adaptive_sharded", "tcpt_group_render_adaptive",
    "tcpt_get_stats", "tcpt_trace", "tcpt_trace_device", "tcpt_sampler_stream", "tcpt_path_samples", "tcpt_get_bvh",
    "tcpt_get_wide_bvh", "tcpt_build_bvh_boxes", "tcpt_rgb_to_coeffs", "tcpt_get_mesh_tangents", "tcpt_upload_flat_scene",
    "tcpt_comm_get_unique_id", "tcpt_comm_init", "tcpt_comm_destroy", "tcpt_shard_params", "tcpt_render_sharded", "tcpt_render_sharded_device",
    "tcpt_group_create", "tcpt_group_destroy", "tcpt_group_size", "tcpt_group_context", "tcpt_group_last_error", "tcpt_group_set_tables",
    "tcpt_group_build", "tcpt_group_render",
    "tcpt_obj_load", "tcpt_obj_counts", "tcpt_obj_copy", "tcpt_obj_free", "tcpt_scene_load_obj", "tcpt_scene_set_tangent_source", "tcpt_image_convert", "tcpt_cdf_search", "tcpt_scene_build_soup", "tcpt_soup_build_info",
]

_lib = None


def load_library() -> C.CDLL:
    """Load libtcpt.so (built in-tree by __graft_entry__.build()).  Raises if it has not been built: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    lib_path = Path(os.environ.get("TCPT_LIB", LIB_PATH))   # developer knob: benchmark an alternative build of the same sources
    if not lib_path.exists():
        raise FileNotFoundError(f"{lib_path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                                "There is no CPU fallback for the path-integration hot path.")
    lib = C.CDLL(str(lib_path))
    P, I, U, F = C.c_void_p, C.c_int, C.c_uint32, C.c_float
    fp, up, ip, bp = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
    sig = {
        "tcpt_create": (I, [I, C.POINTER(P)]), "tcpt_destroy": (None, [P]), "tcpt_last_error": (C.c_char_p, [P]),
        "tcpt_set_option": (I, [P, C.c_char_p, I]), "tcpt_set_tables": (I, [P, C.c_void_p, C.c_size_t, fp, C.c_size_t]),
        "tcpt_scene_clear": (I, [P]), "tcpt_scene_add_mesh": (I, [P, fp, fp, fp, I, up, I]),
        "tcpt_scene_add_single_triangle": (I, [P, fp, fp, fp]),
        "tcpt_scene_add_texture": (I, [P, bp, U, U, U]), "tcpt_scene_add_material": (I, [P, C.POINTER(MaterialDesc)]),
        "tcpt_scene_add_primitive": (I, [P, I, I, fp]), "tcpt_scene_add_env_light": (I, [P, F, fp, U, U, fp]),
        "tcpt_scene_add_delta_light": (I, [P, I, F, C.POINTER(SpectrumParam), F, F, fp]),
        "tcpt_scene_build": (I, [P, fp]), "tcpt_render": (I, [P, C.POINTER(RenderParams), fp, fp]),
        "tcpt_render_device": (I, [P, C.POINTER(RenderParams), C.c_void_p, C.c_void_p]),
        "tcpt_finalize_device": (I, [P, C.c_void_p, U, U, U, C.c_void_p, C.c_void_p]),
        "tcpt_render_adaptive": (I, [P, C.POINTER(RenderParams), C.POINTER(AdaptiveParams), fp, fp, up]),
        "tcpt_render_adaptive_device": (I, [P, C.POINTER(RenderParams), C.POINTER(AdaptiveParams), C.c_void_p, C.c_void_p, C.c_void_p]),
        "tcpt_render_adaptive_sharded": (I, [P, C.POINTER(RenderParams), C.POINTER(AdaptiveParams), fp, fp, up]),
        "tcpt_group_render_adaptive": (I, [P, C.POINTER(RenderParams), C.POINTER(AdaptiveParams), fp, fp, up]),
        "tcpt_get_stats": (I, [P, C.POINTER(Stats)]), "tcpt_trace": (I, [P, fp, I, I, ip]),
        "tcpt_trace_device": (I, [P, C.c_void_p, I, I, C.c_void_p, C.c_void_p]),
        "tcpt_sampler_stream": (I, [P, I, U, U, U, U, U, U, U, ip, I, fp]),
        "tcpt_path_samples": (I, [P, C.POINTER(RenderParams), up, up, I, fp]),
        "tcpt_get_bvh": (I, [P, I, up, I]), "tcpt_get_wide_bvh": (I, [P, I, up, I, up, up]), "tcpt_build_bvh_boxes": (I, [fp, I, up, I]),
        "tcpt_rgb_to_coeffs": (I, [P, fp, I, fp, ip]), "tcpt_get_mesh_tangents": (I, [P, I, fp, I]),
        "tcpt_comm_get_unique_id": (I, [C.c_void_p]), "tcpt_comm_init": (I, [P, I, I, C.c_void_p]), "tcpt_comm_destroy": (I, [P]),
        "tcpt_shard_params": (I, [C.POINTER(RenderParams), I, I, I, C.POINTER(RenderParams)]),
        "tcpt_render_sharded": (I, [P, C.POINTER(RenderParams), I, fp, fp]),
        "tcpt_render_sharded_device": (I, [P, C.POINTER(RenderParams), I, C.c_void_p, C.c_void_p]),
        "tcpt_group_create": (I, [ip, I, C.POINTER(P)]), "tcpt_group_destroy": (None, [P]), "tcpt_group_size": (I, [P]),
        "tcpt_group_context": (P, [P, I]), "tcpt_group_last_error": (C.c_char_p, [P]),
        "tcpt_group_set_tables": (I, [P, C.c_void_p, C.c_size_t, fp, C.c_size_t]), "tcpt_group_build": (I, [P, fp]),
        "tcpt_group_render": (I, [P, C.POINTER(RenderParams), I, fp, fp]),
        "tcpt_obj_load": (I, [C.c_char_p, C.POINTER(P), C.c_char_p, C.c_size_t]), "tcpt_obj_counts": (I, [P, up]),
        "tcpt_obj_copy": (I, [P, fp, fp, fp, up, up]), "tcpt_obj_free": (None, [P]),
        "tcpt_scene_build_soup": (I, [P, fp, U]), "tcpt_soup_build_info": (I, [P, C.POINTER(C.c_double), C.POINTER(C.c_uint64), up]),
        "tcpt_cdf_search": (I, [P, fp, U, U, fp, I, up]),
        "tcpt_image_convert": (I, [C.c_void_p, U, U, U, I, I, C.c_void_p]),
        "tcpt_scene_load_obj": (I, [P, C.c_char_p]), "tcpt_scene_set_tangent_source": (I, [P, I, up, I]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def as_ptr(a: np.ndarray, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def load_tables():
    """(std_tables bytes, rgb2spec float32 array) from the package data directory."""
    std = (DATA_DIR / "std_tables.bin").read_bytes()
    rgb2spec = np.fromfile(DATA_DIR / "srgb_table.bin", dtype="<f4")
    return std, np.ascontiguousarray(rgb2spec)


class Context:
    """Owns one tcpt_ctx.  `require_gpu=False` keeps a host-only context alive (BVH / table introspection on a CPU box)."""

    def __init__(self, device: int = 0, require_gpu: bool = True, set_tables: bool = True):
        self.lib = load_library()
        self.handle = C.c_void_p()
        rc = self.lib.tcpt_create(device, C.byref(self.handle))
        self.has_gpu = rc == TCPT_OK
        self.comm_rank, self.comm_size = 0, 1
        if rc != TCPT_OK and (require_gpu or not self.handle):
            msg = self.last_error()
            self.close()
            raise TcptError(rc, msg)
        if set_tables:
            std, tab = load_tables()
            self._std, self._tab = std, tab
            rc = self.lib.tcpt_set_tables(self.handle, std, len(std), as_ptr(tab, C.c_float), tab.size)
            if rc != TCPT_OK and not (rc == TCPT_ERR_CUDA and not self.has_gpu):
                raise TcptError(rc, self.last_error())

    def last_error(self) -> str:
        return (self.lib.tcpt_last_error(self.handle) or b"").decode() if self.handle else "no context"

    def check(self, rc: int, allow_no_gpu: bool = False) -> int:
        if rc < 0 and not (allow_no_gpu and rc == TCPT_ERR_CUDA and not self.has_gpu):
            raise TcptError(rc, self.last_error())
        return rc

    def set_option(self, name: str, value: int):
        self.check(self.lib.tcpt_set_option(self.handle, name.encode(), int(value)))

    # ---- multi-GPU: the NCCL communicator lives inside libtcpt (include/tcpt.h "multi-GPU")
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(COMM_ID_BYTES)
        rc = load_library().tcpt_comm_get_unique_id(buf)
        if rc != TCPT_OK:
            raise TcptError(rc, "tcpt_comm_get_unique_id failed (libnccl.so.2 not loadable?)")
        return buf.raw

    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        assert len(unique_id) == COMM_ID_BYTES
        self.check(self.lib.tcpt_comm_init(self.handle, nranks, rank, C.c_char_p(unique_id)))
        self.comm_rank, self.comm_size = rank, nranks

    def comm_destroy(self):
        self.check(self.lib.tcpt_comm_destroy(self.handle))
        self.comm_rank, self.comm_size = 0, 1

    def stats(self) -> dict:
        s = Stats()
        self.check(self.lib.tcpt_get_stats(self.handle, C.byref(s)))
        return s.as_dict()

    def close(self):
        if getattr(self, "handle", None):
            self.lib.tcpt_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
