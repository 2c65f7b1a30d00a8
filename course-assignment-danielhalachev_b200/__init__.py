"""crt-b200: B200-native renderer core for the Chaos course ray tracer's per-pixel hot path.

This package is a thin ctypes binding over two in-tree native libraries:

  csrc/libcrtb200.so   the CUDA (sm_100a) wavefront renderer behind the C ABI of include/crtb200.h
  csrc/libcrtfront.so  the C++ host front end (scene loader, KD build, camera, PPM, RayTracer mirror), include/crtfront.h

There is no Python or CPU rendering path: every render call goes to the CUDA library and raises when it is
missing or no sm_100 GPU is usable.  (The CPU oracle lives under /oracle and is test infrastructure only.)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import NamedTuple, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# CRT_CORE_LIB: load a differently-tuned build of the same CUDA core (tools/ tuning runs only)
CORE_PATH = os.environ.get("CRT_CORE_LIB") or os.path.join(CSRC, "libcrtb200.so")
FRONT_PATH = os.path.join(CSRC, "libcrtfront.so")

INVALID = 0xFFFFFFFF
MAT_DIFFUSE, MAT_REFLECTIVE, MAT_CONSTANT, MAT_REFRACTIVE = 0, 1, 2, 3
RAY_PRIMARY, RAY_SHADOW, RAY_REFLECTION, RAY_REFRACTION, RAY_DIFFUSE = 0, 1, 2, 3, 4
# RenderOptimization (RayTracer.h:12-23) + the new enumerator
MODE_BVH_BUCKETS_THREADPOOL = 8
MODE_B200_WAVEFRONT = 10


class CrtError(RuntimeError):
    pass


# ---- C structs (must match include/crtb200.h) -----------------------------------------------------------------
class KdNode(C.Structure):
    _fields_ = [("box_min", C.c_float * 3), ("box_max", C.c_float * 3), ("child", C.c_uint32 * 2),
                ("leaf_start", C.c_uint32), ("leaf_count", C.c_uint32)]


class Mesh(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("material", "first_triangle", "n_triangles", "first_vertex", "n_vertices",
                                          "first_node", "n_nodes", "first_leaf_ref", "n_leaf_refs")]


class Material(C.Structure):
    _fields_ = [("type", C.c_uint32), ("smooth_shading", C.c_uint32), ("texture", C.c_uint32),
                ("albedo", C.c_float * 3), ("ior", C.c_float)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("color_a", C.c_float * 3), ("color_b", C.c_float * 3), ("scalar", C.c_float),
                ("width", C.c_uint32), ("height", C.c_uint32), ("texel_offset", C.c_uint64)]


class Light(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("intensity", C.c_uint32)]


class Scene(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32), ("background", C.c_float * 3),
        ("n_vertices", C.c_uint32), ("vertex_position", C.POINTER(C.c_float)), ("vertex_normal", C.POINTER(C.c_float)),
        ("vertex_uv", C.POINTER(C.c_float)),
        ("n_triangles", C.c_uint32), ("triangle_vertex", C.POINTER(C.c_uint32)), ("triangle_normal", C.POINTER(C.c_float)),
        ("n_meshes", C.c_uint32), ("meshes", C.POINTER(Mesh)),
        ("n_materials", C.c_uint32), ("materials", C.POINTER(Material)),
        ("n_textures", C.c_uint32), ("textures", C.POINTER(Texture)),
        ("n_texels", C.c_uint64), ("texels", C.POINTER(C.c_float)),
        ("n_lights", C.c_uint32), ("lights", C.POINTER(Light)),
        ("n_mesh_nodes", C.c_uint32), ("mesh_nodes", C.POINTER(KdNode)),
        ("n_mesh_leaf_refs", C.c_uint32), ("mesh_leaf_refs", C.POINTER(C.c_uint32)),
        ("n_top_nodes", C.c_uint32), ("top_nodes", C.POINTER(KdNode)),
        ("n_top_leaf_refs", C.c_uint32), ("top_leaf_refs", C.POINTER(C.c_uint32)),
    ]


class Trees(C.Structure):
    """crtb200_trees: the trees of the last crtb200_upload_geometry (crtb200_scene_trees)."""
    _fields_ = [("n_meshes", C.c_uint32), ("n_mesh_nodes", C.c_uint32), ("n_mesh_leaf_refs", C.c_uint32),
                ("n_top_nodes", C.c_uint32), ("n_top_leaf_refs", C.c_uint32), ("reserved", C.c_uint32),
                ("peak_scratch_bytes", C.c_uint64), ("build_ms", C.c_double),
                ("meshes", C.c_void_p), ("mesh_nodes", C.c_void_p), ("mesh_leaf_refs", C.c_void_p),
                ("top_nodes", C.c_void_p), ("top_leaf_refs", C.c_void_p)]


class SceneLayout(C.Structure):
    """crtb200_scene_layout: one GPU's device scene state (crtb200_debug_scene_layout)."""
    _fields_ = [("n_nodes", C.c_uint32), ("n_leaf_refs", C.c_uint32), ("n_top_refs", C.c_uint32), ("n_meshes", C.c_uint32),
                ("top_begin", C.c_uint32), ("top_end", C.c_uint32), ("nested_ok", C.c_uint32), ("reserved", C.c_uint32),
                ("nodes", C.c_void_p), ("leaf_refs", C.c_void_p), ("top_refs", C.c_void_p), ("meshes", C.c_void_p)]


# numpy views of crtb200_kdnode and crtb200_mesh records
KDNODE_DTYPE = np.dtype([("box_min", np.float32, 3), ("box_max", np.float32, 3), ("child", np.uint32, 2),
                         ("leaf_start", np.uint32), ("leaf_count", np.uint32)])
MESH_DTYPE = np.dtype([(n, np.uint32) for n, _ in Mesh._fields_])


class Camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("rotation", C.c_float * 9)]

    @staticmethod
    def make(position=(0.0, 0.0, 0.0), rotation=(1, 0, 0, 0, 1, 0, 0, 0, 1)) -> "Camera":
        cam = Camera()
        cam.position[:] = [float(v) for v in position]
        cam.rotation[:] = [float(v) for v in rotation]
        return cam


class Rect(C.Structure):
    _fields_ = [("row", C.c_uint32), ("col", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32)]


class Options(C.Structure):
    _fields_ = [("max_depth", C.c_uint32), ("shadow_bias", C.c_float), ("reflection_bias", C.c_float),
                ("refraction_bias", C.c_float), ("n_rects", C.c_uint32), ("rects", C.POINTER(Rect)),
                ("traversal", C.c_uint32), ("count_work", C.c_uint32), ("shard_index", C.c_uint32),
                ("shard_count", C.c_uint32), ("shard_full_frame", C.c_uint32)]


class Hit(C.Structure):
    _fields_ = [("mesh", C.c_int32), ("triangle", C.c_int32), ("t", C.c_float)]


HIT_DTYPE = np.dtype([("mesh", np.int32), ("triangle", np.int32), ("t", np.float32)])


class Stats(C.Structure):
    _fields_ = [("rays_primary", C.c_uint64), ("rays_shadow", C.c_uint64), ("rays_reflection", C.c_uint64),
                ("rays_refraction", C.c_uint64), ("node_tests_closest", C.c_uint64), ("triangle_tests_closest", C.c_uint64),
                ("node_tests_shadow", C.c_uint64), ("triangle_tests_shadow", C.c_uint64),
                ("device_ms", C.c_double), ("closest_ms", C.c_double), ("shadow_ms", C.c_double), ("total_ms", C.c_double),
                ("kernel_launches", C.c_uint32), ("levels", C.c_uint32),
                ("handoff_closest", C.c_uint64), ("handoff_shadow", C.c_uint64),
                ("coop_closest_ms", C.c_double), ("coop_shadow_ms", C.c_double), ("shadow_rays_zero_term", C.c_uint64)]

    def as_dict(self) -> dict:
        d = {n: getattr(self, n) for n, _ in self._fields_}
        d["rays_total"] = d["rays_primary"] + d["rays_shadow"] + d["rays_reflection"] + d["rays_refraction"]
        d["node_tests"] = d["node_tests_closest"] + d["node_tests_shadow"]
        d["triangle_tests"] = d["triangle_tests_closest"] + d["triangle_tests_shadow"]
        return d


class RayBatch(C.Structure):
    """crtb200_ray_batch: a batch of caller-supplied rays in device memory (crtb200_trace_rays_device)."""
    _fields_ = [("n", C.c_uint32), ("ray_type", C.c_uint32), ("traversal", C.c_uint32), ("count_work", C.c_uint32),
                ("rays", C.c_void_p), ("max_distance", C.c_void_p), ("hits", C.c_void_p), ("occluded", C.c_void_p)]


class ShadeBatch(C.Structure):
    """crtb200_shade_batch: caller-supplied rays to shade, in device memory (crtb200_shade_rays_device)."""
    _fields_ = [("n", C.c_uint32), ("ray_type", C.c_uint32), ("traversal", C.c_uint32), ("count_work", C.c_uint32),
                ("max_depth", C.c_uint32), ("shadow_bias", C.c_float), ("reflection_bias", C.c_float),
                ("refraction_bias", C.c_float), ("sample", C.c_uint32), ("first_index", C.c_uint32),
                ("rays", C.c_void_p), ("rgb", C.c_void_p), ("hits", C.c_void_p)]


class Hits(NamedTuple):
    """Closest hits of Context.trace: mesh, triangle and t are views of `records`, one (..., 3) int32 tensor in the
    crtb200_hit layout; t holds float32 bits (t.view(torch.float32))."""
    mesh: "object"
    triangle: "object"
    t: "object"
    records: "object"


class Sampling(C.Structure):
    """crtb200_sampling: GI + jittered supersampling under the project's sampling contract (DESIGN.md 3.10)."""
    _fields_ = [("use_gi", C.c_uint32), ("gi_samples", C.c_uint32), ("rays_per_pixel", C.c_uint32),
                ("monte_carlo_bias", C.c_float), ("seed", C.c_uint32), ("frame_index", C.c_uint32)]

    @staticmethod
    def make(use_gi: bool = True, gi_samples: int = 2, rays_per_pixel: int = 1, monte_carlo_bias: float = 1e-4,
             seed: int = 0, frame_index: int = 0) -> "Sampling":
        return Sampling(1 if use_gi else 0, gi_samples, rays_per_pixel, monte_carlo_bias, seed, frame_index)


class Adaptive(C.Structure):
    """crtb200_adaptive: the stop rule of an adaptive progressive session (DESIGN.md 3.10.2)."""
    _fields_ = [("min_samples", C.c_uint32), ("max_samples", C.c_uint32), ("abs_error", C.c_float), ("rel_error", C.c_float)]

    @staticmethod
    def make(min_samples: int = 8, max_samples: int = 128, abs_error: float = 0.0, rel_error: float = 0.05) -> "Adaptive":
        return Adaptive(min_samples, max_samples, abs_error, rel_error)


class AccumProgress(C.Structure):
    _fields_ = [("passes", C.c_uint32), ("reserved", C.c_uint32), ("covered_pixels", C.c_uint64),
                ("active_pixels", C.c_uint64), ("pixel_samples", C.c_uint64)]


class SamplingStats(C.Structure):
    _fields_ = [("rays_diffuse", C.c_uint64), ("samples", C.c_uint32), ("reserved", C.c_uint32)]


class SceneInfo(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("bucket_size", C.c_uint32), ("n_meshes", C.c_uint32),
                ("n_materials", C.c_uint32), ("n_textures", C.c_uint32), ("n_lights", C.c_uint32),
                ("n_triangles", C.c_uint64), ("n_vertices", C.c_uint64), ("background", C.c_float * 3),
                ("camera", Camera)]


# ---- library loading ---------------------------------------------------------------------------------------------
_core = None
_front = None


def build(force: bool = False, verbose: bool = False) -> None:
    from . import nativebuild as _b
    _b.build_all(force=force, verbose=verbose)


def core() -> C.CDLL:
    """libcrtb200.so; raises (no fallback) when it has not been built."""
    global _core
    if _core is None:
        if not os.path.exists(CORE_PATH):
            raise CrtError(f"{CORE_PATH} is missing: build it with __graft_entry__.build(); there is no CPU fallback")
        lib = C.CDLL(CORE_PATH, mode=C.RTLD_GLOBAL)
        lib.crtb200_last_error.restype = C.c_char_p
        lib.crtb200_abi_version.restype = C.c_uint32
        lib.crtb200_render_device.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crtb200_assemble_shards.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crtb200_render.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Options), C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Stats)]
        lib.crtb200_render_frames.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_uint32, C.POINTER(Options), C.c_void_p, C.c_void_p, C.POINTER(Stats)]
        lib.crtb200_upload_scene.argtypes = [C.c_void_p, C.POINTER(Scene)]
        lib.crtb200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.crtb200_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
        lib.crtb200_device_list.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
        lib.crtb200_last_error_ctx.argtypes = [C.c_void_p]
        lib.crtb200_last_error_ctx.restype = C.c_char_p
        lib.crtb200_destroy.argtypes = [C.c_void_p]
        lib.crtb200_set_queue_budget.argtypes = [C.c_void_p, C.c_uint64]
        lib.crtb200_set_concurrency.argtypes = [C.c_void_p, C.c_uint32]
        lib.crtb200_last_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        lib.crtb200_shard_items.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        lib.crtb200_ipc_alloc.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]
        lib.crtb200_ipc_free.argtypes = [C.c_int, C.c_void_p]
        lib.crtb200_ipc_export.argtypes = [C.c_void_p, C.c_void_p]
        lib.crtb200_ipc_open.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        lib.crtb200_ipc_close.argtypes = [C.c_int, C.c_void_p]
        lib.crtb200_generate_rays.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_void_p]
        lib.crtb200_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.crtb200_trace_rays_device.argtypes = [C.c_void_p, C.POINTER(RayBatch), C.c_void_p]
        lib.crtb200_generate_rays_device.argtypes = [C.c_void_p, C.POINTER(Camera), C.c_void_p, C.c_void_p]
        lib.crtb200_last_query_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        lib.crtb200_shade_rays_device.argtypes = [C.c_void_p, C.POINTER(ShadeBatch), C.c_void_p]
        lib.crtb200_device_count.argtypes = [C.POINTER(C.c_int)]
        lib.crtb200_debug_powf5.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        lib.crtb200_upload_geometry.argtypes = [C.c_void_p, C.POINTER(Scene)]
        lib.crtb200_scene_trees.argtypes = [C.c_void_p, C.POINTER(Trees)]
        lib.crtb200_debug_scene_layout.argtypes = [C.c_void_p, C.c_int, C.POINTER(SceneLayout)]
        lib.crtb200_update_vertices_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        lib.crtb200_debug_scene_geometry.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        lib.crtb200_set_sampling.argtypes = [C.c_void_p, C.POINTER(Sampling)]
        lib.crtb200_last_sampling_stats.argtypes = [C.c_void_p, C.POINTER(SamplingStats)]
        lib.crtb200_accum_begin.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Options), C.POINTER(Sampling)]
        lib.crtb200_accum_step.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(Stats)]
        lib.crtb200_accum_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
        lib.crtb200_accum_save.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]
        lib.crtb200_accum_load.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        lib.crtb200_accum_end.argtypes = [C.c_void_p]
        lib.crtb200_accum_begin_adaptive.argtypes = [C.c_void_p, C.POINTER(Camera), C.POINTER(Options), C.POINTER(Sampling),
                                                     C.POINTER(Adaptive)]
        lib.crtb200_accum_progress.argtypes = [C.c_void_p, C.POINTER(AccumProgress)]
        lib.crtb200_accum_counts.argtypes = [C.c_void_p, C.c_void_p]
        lib.crtb200_accum_load_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        _core = lib
    return _core


def front() -> C.CDLL:
    """libcrtfront.so (depends on libcrtb200.so)."""
    global _front
    if _front is None:
        core()
        if not os.path.exists(FRONT_PATH):
            raise CrtError(f"{FRONT_PATH} is missing: build it with __graft_entry__.build()")
        lib = C.CDLL(FRONT_PATH)
        lib.crtfe_last_error.restype = C.c_char_p
        lib.crtfe_scene_load.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_void_p)]
        lib.crtfe_scene_free.argtypes = [C.c_void_p]
        lib.crtfe_scene_get_info.argtypes = [C.c_void_p, C.POINTER(SceneInfo)]
        lib.crtfe_scene_flatten.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.POINTER(Scene)), C.POINTER(C.c_double)]
        lib.crtfe_scene_flatten_geometry.argtypes = [C.c_void_p, C.POINTER(C.POINTER(Scene)), C.POINTER(C.c_double)]
        lib.crtfe_rectangles.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Rect), C.c_uint32, C.POINTER(C.c_uint32)]
        lib.crtfe_camera_pan.argtypes = [C.POINTER(Camera), C.c_float]
        lib.crtfe_camera_tilt.argtypes = [C.POINTER(Camera), C.c_float]
        lib.crtfe_camera_roll.argtypes = [C.POINTER(Camera), C.c_float]
        lib.crtfe_camera_truck.argtypes = [C.POINTER(Camera), C.POINTER(C.c_float)]
        lib.crtfe_write_ppm.argtypes = [C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]
        lib.crtfe_append_f32.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64]
        lib.crtfe_append_u32.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64]
        lib.crtfe_tracer_create.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        lib.crtfe_tracer_free.argtypes = [C.c_void_p]
        lib.crtfe_tracer_set_camera.argtypes = [C.c_void_p, C.POINTER(Camera)]
        lib.crtfe_tracer_get_camera.argtypes = [C.c_void_p, C.POINTER(Camera)]
        lib.crtfe_tracer_render.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(Stats)]
        lib.crtfe_tracer_render_sampled.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                                    C.c_uint32, C.c_uint32, C.c_float, C.c_uint32, C.c_void_p, C.POINTER(Stats)]
        _front = lib
    return _front


def _check_core(rc: int) -> None:
    if rc != 0:
        raise CrtError(f"crtb200 error {rc}: {core().crtb200_last_error().decode(errors='replace')}")


def _check_front(rc: int) -> None:
    if rc != 0:
        raise CrtError(f"crtfront error {rc}: {front().crtfe_last_error().decode(errors='replace')}")


# ---- front end ---------------------------------------------------------------------------------------------------
def rectangles(width: int, height: int, bucket_size: int, mode: int = MODE_B200_WAVEFRONT, hw_threads: int = 8):
    """The rectangle grid the reference's schedulers hand to renderRectangle (RayTracer.cpp:114-158)."""
    n = C.c_uint32(0)
    _check_front(front().crtfe_rectangles(width, height, mode, bucket_size, hw_threads, None, 0, C.byref(n)))
    arr = (Rect * max(1, n.value))()
    _check_front(front().crtfe_rectangles(width, height, mode, bucket_size, hw_threads, arr, n.value, C.byref(n)))
    return arr, n.value


class SceneFile:
    """SceneParser::parseScene + AccelerationStructure build + flattening (host front end)."""

    def __init__(self, path_to_scene: str, scene_folder: str = ""):
        self._h = C.c_void_p()
        _check_front(front().crtfe_scene_load(path_to_scene.encode(), scene_folder.encode(), C.byref(self._h)))
        self.info = SceneInfo()
        _check_front(front().crtfe_scene_get_info(self._h, C.byref(self.info)))
        self._flat: Optional[C.POINTER(Scene)] = None
        self._geometry: Optional[C.POINTER(Scene)] = None
        self.build_seconds = 0.0
        self.geometry_seconds = 0.0

    @property
    def handle(self):
        return self._h

    def flatten(self, threads: int = 0, trees: bool = True) -> "C.POINTER(Scene)":
        """The scene as crtb200_scene arrays, with the host-built KD trees (crtb200_upload_scene), or with trees=False
        without them (tree counts 0, arrays NULL: Context.upload_geometry builds them on the GPU).  Each is built once."""
        if not trees:
            if self._geometry is None:
                p = C.POINTER(Scene)()
                sec = C.c_double(0)
                _check_front(front().crtfe_scene_flatten_geometry(self._h, C.byref(p), C.byref(sec)))
                self._geometry = p
                self.geometry_seconds = sec.value
            return self._geometry
        if self._flat is None:
            p = C.POINTER(Scene)()
            sec = C.c_double(0)
            _check_front(front().crtfe_scene_flatten(self._h, threads, C.byref(p), C.byref(sec)))
            self._flat = p
            self.build_seconds = sec.value
        return self._flat

    def camera(self) -> Camera:
        cam = Camera()
        C.memmove(C.byref(cam), C.byref(self.info.camera), C.sizeof(Camera))
        return cam

    def rects(self, mode: int = MODE_B200_WAVEFRONT, hw_threads: int = 8):
        return rectangles(self.info.width, self.info.height, self.info.bucket_size, mode, hw_threads)

    def close(self):
        if self._h:
            front().crtfe_scene_free(self._h)
            self._h = C.c_void_p()
            self._flat = None
            self._geometry = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scene_vertex_positions(scene_ptr) -> np.ndarray:
    """A (n_vertices, 3) float32 copy of a flattened scene's vertex positions: the rest pose that Context.update_vertices
    takes deformed."""
    s = scene_ptr.contents
    if s.n_vertices == 0:
        return np.zeros((0, 3), np.float32)
    return np.ctypeslib.as_array(s.vertex_position, shape=(s.n_vertices * 3,)).reshape(-1, 3).copy()


def camera_pan(cam: Camera, degrees: float) -> Camera:
    _check_front(front().crtfe_camera_pan(C.byref(cam), degrees))
    return cam


def write_ppm(path: str, rgb: np.ndarray) -> None:
    rgb = np.ascontiguousarray(rgb, dtype=np.float32)
    h, w, _ = rgb.shape
    _check_front(front().crtfe_write_ppm(path.encode(), rgb.ctypes.data, w, h))


# ---- CUDA core ---------------------------------------------------------------------------------------------------
def make_options(max_depth: int = 5, rects=None, n_rects: int = 0, traversal: int = 0, count_work: int = 0,
                 shard_index: int = 0, shard_count: int = 1, bias: float = 1e-4, shard_full_frame: bool = False) -> Options:
    o = Options()
    o.max_depth = max_depth
    o.shadow_bias = o.reflection_bias = o.refraction_bias = bias
    o.n_rects = n_rects if rects is not None else 0
    o.rects = C.cast(rects, C.POINTER(Rect)) if rects is not None else None
    o.traversal = traversal
    o.count_work = int(count_work)
    o.shard_index = shard_index
    o.shard_count = shard_count
    o.shard_full_frame = 1 if shard_full_frame else 0
    return o


def ipc_alloc(device: int, nbytes: int) -> int:
    """A whole cudaMalloc allocation on `device` (zeroed), exportable with ipc_export."""
    p = C.c_void_p()
    _check_core(core().crtb200_ipc_alloc(device, nbytes, C.byref(p)))
    return p.value


def ipc_free(device: int, d_ptr: int) -> None:
    _check_core(core().crtb200_ipc_free(device, d_ptr))


def ipc_export(d_ptr: int) -> bytes:
    """64-byte CUDA IPC handle of a cudaMalloc allocation of this process (crtb200_ipc_export)."""
    buf = (C.c_uint8 * 64)()
    _check_core(core().crtb200_ipc_export(d_ptr, buf))
    return bytes(buf)


def ipc_open(device: int, handle: bytes) -> int:
    """Maps another process's allocation on `device`; returns the device pointer (crtb200_ipc_open)."""
    buf = (C.c_uint8 * 64)(*handle)
    p = C.c_void_p()
    _check_core(core().crtb200_ipc_open(device, buf, C.byref(p)))
    return p.value


def ipc_close(device: int, d_ptr: int) -> None:
    _check_core(core().crtb200_ipc_close(device, d_ptr))


class Context:
    """One GPU context of libcrtb200 (RayTracer's device-side state)."""

    def __init__(self, device=0):
        """device: one CUDA device index, or a sequence of them (crtb200_create_multi: every frame is split by tiles
        over the GPUs, the scene is replicated, results are identical to a single GPU's)."""
        self._h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*[int(d) for d in device])
            _check_core(core().crtb200_create_multi(ids, len(device), C.byref(self._h)))
        else:
            _check_core(core().crtb200_create(int(device), C.byref(self._h)))
        self.width = self.height = 0
        self.n_vertices = self.n_triangles = 0
        self._scene_keepalive = None
        self._session = None  # the Progressive whose session the context holds

    def devices(self):
        n = C.c_int(0)
        _check_core(core().crtb200_device_list(self._h, None, 0, C.byref(n)))
        ids = (C.c_int * n.value)()
        _check_core(core().crtb200_device_list(self._h, ids, n.value, C.byref(n)))
        return list(ids)

    def last_error(self) -> str:
        return core().crtb200_last_error_ctx(self._h).decode(errors="replace")

    def upload(self, scene_ptr, keepalive=None) -> None:
        _check_core(core().crtb200_upload_scene(self._h, scene_ptr))
        self.width, self.height = scene_ptr.contents.width, scene_ptr.contents.height
        self.n_vertices, self.n_triangles = scene_ptr.contents.n_vertices, scene_ptr.contents.n_triangles
        self._scene_keepalive = keepalive

    def upload_geometry(self, scene_ptr, keepalive=None) -> None:
        """crtb200_upload_geometry: uploads a scene without trees (SceneFile.flatten(trees=False), or a Scene built from
        arrays) and builds its KD trees on every GPU of the context; afterwards the context is as upload() of the
        host-built trees leaves it."""
        _check_core(core().crtb200_upload_geometry(self._h, scene_ptr))
        self.width, self.height = scene_ptr.contents.width, scene_ptr.contents.height
        self.n_vertices, self.n_triangles = scene_ptr.contents.n_vertices, scene_ptr.contents.n_triangles
        self._scene_keepalive = keepalive

    def scene_trees(self) -> dict:
        """The trees the last upload_geometry built, in the reference's numbering (crtb200_scene_trees): 'meshes'
        (MESH_DTYPE, tree fields filled), 'mesh_nodes' / 'top_nodes' (KDNODE_DTYPE), 'mesh_leaf_refs' (mesh-local
        triangle indices), 'top_leaf_refs' (mesh indices), 'peak_scratch_bytes' and 'build_ms'."""
        t = Trees()
        _check_core(core().crtb200_scene_trees(self._h, C.byref(t)))
        out = {"meshes": np.zeros(t.n_meshes, MESH_DTYPE), "mesh_nodes": np.zeros(t.n_mesh_nodes, KDNODE_DTYPE),
               "mesh_leaf_refs": np.zeros(t.n_mesh_leaf_refs, np.uint32), "top_nodes": np.zeros(t.n_top_nodes, KDNODE_DTYPE),
               "top_leaf_refs": np.zeros(t.n_top_leaf_refs, np.uint32)}
        for k, a in out.items():
            setattr(t, k, a.ctypes.data)
        _check_core(core().crtb200_scene_trees(self._h, C.byref(t)))
        out["peak_scratch_bytes"], out["build_ms"] = t.peak_scratch_bytes, t.build_ms
        return out

    def debug_scene_layout(self, device_index: int = 0) -> dict:
        """One GPU's device scene state (crtb200_debug_scene_layout): 'nodes' (n x 8 uint32: min.xyz, a, max.xyz, b of the
        visiting-order array), 'leaf_refs', 'top_refs', 'meshes' (n x 5 uint32: node_begin, node_end, material,
        first_triangle, cull_margin bits), 'top_begin', 'top_end' and 'nested_ok'."""
        l = SceneLayout()
        _check_core(core().crtb200_debug_scene_layout(self._h, device_index, C.byref(l)))
        out = {"nodes": np.zeros((l.n_nodes, 8), np.uint32), "leaf_refs": np.zeros(l.n_leaf_refs, np.uint32),
               "top_refs": np.zeros(l.n_top_refs, np.uint32), "meshes": np.zeros((l.n_meshes, 5), np.uint32)}
        for k, a in out.items():
            setattr(l, k, a.ctypes.data)
        _check_core(core().crtb200_debug_scene_layout(self._h, device_index, C.byref(l)))
        out.update(top_begin=l.top_begin, top_end=l.top_end, nested_ok=bool(l.nested_ok))
        return out

    def update_vertices(self, positions) -> None:
        """Moves the uploaded scene's vertices (crtb200_update_vertices_device): positions is a contiguous float32 CUDA
        tensor of shape (n_vertices, 3) on the context's first device, read after the work already enqueued on
        torch.cuda.current_stream().  Face and vertex normals are recomputed as Mesh::Mesh computes them and the KD trees
        rebuilt on every GPU; afterwards the context is as upload_geometry of the scene with these positions leaves it,
        except that the colour buffer keeps its pixels.  Returns once every GPU holds the new scene; a progressive
        session ends."""
        import torch
        dev = self._first_device()
        if not isinstance(positions, torch.Tensor):
            raise CrtError("positions must be a torch tensor")
        if positions.dtype != torch.float32:
            raise CrtError(f"positions must be torch.float32, not {positions.dtype}")
        if positions.device != dev:
            raise CrtError(f"positions must be on {dev}, not {positions.device}")
        if tuple(positions.shape) != (self.n_vertices, 3):
            raise CrtError(f"positions must have shape {(self.n_vertices, 3)}, not {tuple(positions.shape)}")
        if not positions.is_contiguous():
            raise CrtError("positions must be contiguous")
        stream = torch.cuda.current_stream(dev).cuda_stream
        _check_core(core().crtb200_update_vertices_device(self._h, positions.data_ptr() or None, self.n_vertices, stream or None))

    def debug_scene_geometry(self, device_index: int = 0):
        """One GPU's triangle records and vertex normals (crtb200_debug_scene_geometry): (tri_geom (n_triangles, 3, 4)
        float32 -- per corner the position and face-normal component k in the last column --, vertex_normal
        (n_vertices, 3) float32)."""
        geom = np.zeros((self.n_triangles, 3, 4), np.float32)
        vn = np.zeros((self.n_vertices, 3), np.float32)
        _check_core(core().crtb200_debug_scene_geometry(self._h, device_index, geom.ctypes.data, vn.ctypes.data))
        return geom, vn

    def set_queue_budget(self, nbytes: int) -> None:
        _check_core(core().crtb200_set_queue_budget(self._h, nbytes))

    def set_concurrency(self, chunks_in_flight: int) -> None:
        _check_core(core().crtb200_set_concurrency(self._h, chunks_in_flight))

    def set_sampling(self, sampling: Optional[Sampling] = None, **kw) -> None:
        """crtb200_set_sampling for every later render of this context: a Sampling, or Sampling.make(**kw) keywords;
        set_sampling(None) with no keywords turns GI / supersampling off."""
        if sampling is None and kw:
            sampling = Sampling.make(**kw)
        _check_core(core().crtb200_set_sampling(self._h, C.byref(sampling) if sampling is not None else None))

    def sampling_stats(self) -> dict:
        """{'rays_diffuse', 'samples'} of the last render (crtb200_last_sampling_stats)."""
        st = SamplingStats()
        _check_core(core().crtb200_last_sampling_stats(self._h, C.byref(st)))
        return {"rays_diffuse": st.rays_diffuse, "samples": st.samples}

    def render(self, camera: Camera, options: Options, want_rgb: bool = True, want_rgb8: bool = False,
               want_hits: bool = False, rgb_out: Optional[np.ndarray] = None, rgb8_out: Optional[np.ndarray] = None):
        """crtb200_render with host buffers.  Returns (rgb f32 HxWx3 | None, rgb8 | None, hits | None, stats dict)."""
        h, w = self.height, self.width
        rgb = rgb_out if rgb_out is not None else (np.zeros((h, w, 3), np.float32) if want_rgb else None)
        rgb8 = rgb8_out if rgb8_out is not None else (np.zeros((h, w, 3), np.uint8) if want_rgb8 else None)
        hits = np.zeros((h, w), HIT_DTYPE) if want_hits else None
        st = Stats()
        _check_core(core().crtb200_render(self._h, C.byref(camera), C.byref(options),
                                          rgb.ctypes.data if rgb is not None else None,
                                          rgb8.ctypes.data if rgb8 is not None else None,
                                          hits.ctypes.data if hits is not None else None, C.byref(st)))
        return rgb, rgb8, hits, st.as_dict()

    def progressive(self, camera: Camera, options: Options, sampling: Sampling,
                    adaptive: Optional[Adaptive] = None) -> "Progressive":
        """Begins a progressive GI session on the uploaded scene (crtb200_accum_begin, or with `adaptive`
        crtb200_accum_begin_adaptive); a session in progress ends."""
        return Progressive(self, camera, options, sampling, adaptive)

    def resume(self, path: str, camera: Camera, options: Options, sampling: Sampling,
               adaptive: Optional[Adaptive] = None) -> "Progressive":
        """Continues a session saved with Progressive.save on the scene this context holds.  camera, options,
        sampling and adaptive state what is to be continued: a file saved with another image size, camera, max_depth,
        biases, rects, sampling (everything but rays_per_pixel) or stop rule, or an adaptive file for a plain session
        and the reverse, raises CrtError."""
        with np.load(path, allow_pickle=False) as f:
            data = {k: f[k] for k in f.files}
        for k, v in _session_params(self.width, self.height, camera, options, sampling).items():
            got = data.get(k)
            if got is None or got.dtype != v.dtype or got.shape != v.shape or got.tobytes() != v.tobytes():
                raise CrtError(f"{path}: the saved session's {k} differs from the session to continue")
        if ("adaptive" in data) != (adaptive is not None) or ("counts" in data) != (adaptive is not None):
            raise CrtError(f"{path}: the saved session is {'adaptive' if 'adaptive' in data else 'plain'}, the session "
                           f"to continue is {'adaptive' if adaptive is not None else 'plain'}")
        if adaptive is not None and data["adaptive"].tobytes() != _adaptive_param(adaptive).tobytes():
            raise CrtError(f"{path}: the saved session's adaptive parameters differ from the session to continue")
        h, w = self.height, self.width
        arrays = {"sum": ((h, w, 3), np.float32), "sumsq": ((h, w, 3), np.float32), "hit0": ((h, w), HIT_DTYPE),
                  "samples": ((), np.uint32)}
        if adaptive is not None:
            arrays["counts"] = ((h, w), np.uint32)
        for k, (shape, dtype) in arrays.items():
            if k not in data or data[k].shape != shape or data[k].dtype != dtype:
                raise CrtError(f"{path}: {k} is missing or not {dtype} of shape {shape}")
        p = Progressive(self, camera, options, sampling, adaptive)
        s, q, hit0 = (np.ascontiguousarray(data[k]) for k in ("sum", "sumsq", "hit0"))
        if adaptive is None:
            _check_core(core().crtb200_accum_load(self._h, s.ctypes.data, q.ctypes.data, hit0.ctypes.data, int(data["samples"])))
        else:
            counts = np.ascontiguousarray(data["counts"])
            _check_core(core().crtb200_accum_load_counts(self._h, s.ctypes.data, q.ctypes.data, hit0.ctypes.data,
                                                         counts.ctypes.data, int(data["samples"])))
        p.samples = int(data["samples"])
        return p

    def render_frames(self, cameras: Sequence[Camera], options: Options, want_rgb: bool = True, want_rgb8: bool = False):
        n = len(cameras)
        arr = (Camera * n)(*cameras)
        h, w = self.height, self.width
        rgb = np.zeros((n, h, w, 3), np.float32) if want_rgb else None
        rgb8 = np.zeros((n, h, w, 3), np.uint8) if want_rgb8 else None
        st = Stats()
        _check_core(core().crtb200_render_frames(self._h, arr, n, C.byref(options),
                                                 rgb.ctypes.data if rgb is not None else None,
                                                 rgb8.ctypes.data if rgb8 is not None else None, C.byref(st)))
        return rgb, rgb8, st.as_dict()

    def render_frames_into(self, cameras: Sequence[Camera], options: Options, rgb_out: Optional[np.ndarray] = None,
                           rgb8_out: Optional[np.ndarray] = None) -> dict:
        """crtb200_render_frames into caller-owned (ideally pinned) host arrays of shape (n, H, W, 3)."""
        n = len(cameras)
        arr = (Camera * n)(*cameras)
        st = Stats()
        _check_core(core().crtb200_render_frames(self._h, arr, n, C.byref(options),
                                                 rgb_out.ctypes.data if rgb_out is not None else None,
                                                 rgb8_out.ctypes.data if rgb8_out is not None else None, C.byref(st)))
        return st.as_dict()

    def render_device(self, camera: Camera, options: Options, d_rgb: int = 0, d_rgb8: int = 0, stream: int = 0) -> None:
        """Asynchronous; d_rgb / d_rgb8 are raw device pointers (e.g. torch.Tensor.data_ptr())."""
        _check_core(core().crtb200_render_device(self._h, C.byref(camera), C.byref(options), d_rgb or None, d_rgb8 or None,
                                                 stream or None))

    def assemble_shards(self, d_slabs: int, shard_count: int, d_rgb: int = 0, d_rgb8: int = 0, stream: int = 0) -> None:
        _check_core(core().crtb200_assemble_shards(self._h, d_slabs, shard_count, d_rgb or None, d_rgb8 or None, stream or None))

    def shard_items(self, shard_count: int) -> int:
        n = C.c_uint32(0)
        _check_core(core().crtb200_shard_items(self._h, shard_count, C.byref(n)))
        return n.value

    def last_stats(self) -> dict:
        st = Stats()
        _check_core(core().crtb200_last_stats(self._h, C.byref(st)))
        return st.as_dict()

    def generate_rays(self, camera: Camera) -> np.ndarray:
        rays = np.zeros((self.height, self.width, 6), np.float32)
        _check_core(core().crtb200_generate_rays(self._h, C.byref(camera), rays.ctypes.data))
        return rays

    def trace_rays(self, rays: np.ndarray, ray_type: int, max_distance: Optional[np.ndarray] = None, traversal: int = 0):
        rays = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
        n = rays.shape[0]
        if ray_type == RAY_SHADOW:
            md = np.ascontiguousarray(max_distance, dtype=np.float32)
            occ = np.zeros(n, np.uint8)
            _check_core(core().crtb200_trace_rays(self._h, rays.ctypes.data, n, ray_type, traversal, md.ctypes.data, None, occ.ctypes.data))
            return occ
        hits = np.zeros(n, HIT_DTYPE)
        _check_core(core().crtb200_trace_rays(self._h, rays.ctypes.data, n, ray_type, traversal, None, hits.ctypes.data, None))
        return hits

    def _first_device(self):
        import torch
        return torch.device("cuda", self.devices()[0])

    def generate_rays_device(self, camera: Camera):
        """Camera rays of every pixel as an (H, W, 6) float32 CUDA tensor on the context's first device (origin xyz,
        direction xyz; the layout of generate_rays), written on torch.cuda.current_stream() without a host round trip."""
        import torch
        dev = self._first_device()
        out = torch.empty((self.height, self.width, 6), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _check_core(core().crtb200_generate_rays_device(self._h, C.byref(camera), out.data_ptr() or None, stream or None))
        return out

    def trace(self, rays, ray_type: int, max_distance=None, traversal: int = 0, count_work: int = 0, out=None):
        """Traces a batch of caller-supplied rays on the GPU (crtb200_trace_rays_device), on torch.cuda.current_stream().

        rays: float32 CUDA tensor of shape (..., 6) on the context's first device, contiguous in its last dimension
        (origin xyz, direction xyz; directions of any length).  ray_type RAY_PRIMARY / RAY_REFLECTION / RAY_REFRACTION
        returns the closest hits as Hits(mesh, triangle, t, records): views of records, one (..., 3) int32 tensor (t: float32 bits,
        hits.t.view(torch.float32); a miss is -1, -1, 0); RAY_SHADOW needs max_distance (float32, the leading shape) and
        returns a uint8 tensor of the leading shape, 1 where some candidate lies within max_distance.  out= reuses a
        previous result's storage: the (..., 3) int32 tensor (or a Hits of it), or the uint8 tensor.  Asynchronous like
        any CUDA work on the stream; query_stats() synchronises."""
        import torch
        dev = self._first_device()

        def need(t, what, dtype, shape):
            if not isinstance(t, torch.Tensor):
                raise CrtError(f"{what} must be a torch tensor")
            if t.dtype != dtype:
                raise CrtError(f"{what} must be {dtype}, not {t.dtype}")
            if t.device != dev:
                raise CrtError(f"{what} must be on {dev}, not {t.device}")
            if tuple(t.shape) != tuple(shape):
                raise CrtError(f"{what} must have shape {tuple(shape)}, not {tuple(t.shape)}")

        if not isinstance(rays, torch.Tensor) or rays.dim() < 1 or rays.shape[-1] != 6:
            raise CrtError("rays must be a torch tensor of shape (..., 6)")
        lead = tuple(rays.shape[:-1])
        need(rays, "rays", torch.float32, lead + (6,))
        if ray_type not in (RAY_PRIMARY, RAY_SHADOW, RAY_REFLECTION, RAY_REFRACTION):
            raise CrtError(f"ray_type {ray_type} has no query (primary, shadow, reflection or refraction)")
        if rays.numel() and rays.stride(-1) != 1:
            raise CrtError("rays must be contiguous in its last dimension")
        n = rays.numel() // 6
        if n >= 1 << 31:
            raise CrtError(f"a ray batch holds fewer than 2^31 rays, not {n}")
        flat = rays.reshape(-1, 6).contiguous()  # (a copy on the stream only when the leading dimensions are strided)
        b = RayBatch(n=n, ray_type=ray_type, traversal=traversal, count_work=count_work, rays=flat.data_ptr() or None)
        if ray_type == RAY_SHADOW:
            if max_distance is None:
                raise CrtError("a shadow query needs max_distance")
            need(max_distance, "max_distance", torch.float32, lead)
            md = max_distance.contiguous()
            res = out if out is not None else torch.empty(lead, dtype=torch.uint8, device=dev)
            need(res, "out", torch.uint8, lead)
            if not res.is_contiguous():
                raise CrtError("out must be contiguous")
            b.max_distance, b.occluded = md.data_ptr() or None, res.data_ptr() or None
        else:
            buf = out.records if isinstance(out, Hits) else out
            res = buf if buf is not None else torch.empty(lead + (3,), dtype=torch.int32, device=dev)
            need(res, "out", torch.int32, lead + (3,))
            if not res.is_contiguous():
                raise CrtError("out must be contiguous")
            b.hits = res.data_ptr() or None
        if n:
            stream = torch.cuda.current_stream(dev).cuda_stream
            _check_core(core().crtb200_trace_rays_device(self._h, C.byref(b), stream or None))
        if ray_type == RAY_SHADOW:
            return res
        return Hits(res[..., 0], res[..., 1], res[..., 2], res)

    def shade(self, rays, ray_type: int = RAY_PRIMARY, max_depth: int = 5, bias: float = 1e-4, traversal: int = 0,
              count_work: int = 0, sample: int = 0, first_index: int = 0, want_hits: bool = False, out=None):
        """Shades a batch of caller-supplied rays on the GPU (crtb200_shade_rays_device), on torch.cuda.current_stream():
        colour i is RayTracer::shootRay(ray i, 0) bit for bit, with the context's sampling (GI: ray i is sample `sample`
        of pixel first_index + i).

        rays: float32 CUDA tensor of shape (..., 6) on the context's first device, contiguous in its last dimension
        (origin xyz, direction xyz; directions of any length).  ray_type RAY_PRIMARY / RAY_REFLECTION / RAY_REFRACTION;
        bias is the shadow, reflection and refraction bias.  Returns (rgb, hits): rgb a (..., 3) float32 tensor (out=
        reuses one), hits a Hits as trace() returns it with want_hits, else None.  Asynchronous like any CUDA work on
        the stream; last_stats() synchronises."""
        import torch
        dev = self._first_device()

        def need(t, what, dtype, shape):
            if not isinstance(t, torch.Tensor):
                raise CrtError(f"{what} must be a torch tensor")
            if t.dtype != dtype:
                raise CrtError(f"{what} must be {dtype}, not {t.dtype}")
            if t.device != dev:
                raise CrtError(f"{what} must be on {dev}, not {t.device}")
            if tuple(t.shape) != tuple(shape):
                raise CrtError(f"{what} must have shape {tuple(shape)}, not {tuple(t.shape)}")

        if not isinstance(rays, torch.Tensor) or rays.dim() < 1 or rays.shape[-1] != 6:
            raise CrtError("rays must be a torch tensor of shape (..., 6)")
        lead = tuple(rays.shape[:-1])
        need(rays, "rays", torch.float32, lead + (6,))
        if ray_type not in (RAY_PRIMARY, RAY_REFLECTION, RAY_REFRACTION):
            raise CrtError(f"ray_type {ray_type} cannot be shaded (primary, reflection or refraction)")
        if rays.numel() and rays.stride(-1) != 1:
            raise CrtError("rays must be contiguous in its last dimension")
        n = rays.numel() // 6
        if n >= 1 << 31:
            raise CrtError(f"a ray batch holds fewer than 2^31 rays, not {n}")
        flat = rays.reshape(-1, 6).contiguous()  # (a copy on the stream only when the leading dimensions are strided)
        rgb = out if out is not None else torch.empty(lead + (3,), dtype=torch.float32, device=dev)
        need(rgb, "out", torch.float32, lead + (3,))
        if not rgb.is_contiguous():
            raise CrtError("out must be contiguous")
        hits = torch.empty(lead + (3,), dtype=torch.int32, device=dev) if want_hits else None
        b = ShadeBatch(n=n, ray_type=ray_type, traversal=traversal, count_work=count_work, max_depth=max_depth,
                       shadow_bias=bias, reflection_bias=bias, refraction_bias=bias, sample=sample & 0xFFFFFFFF,
                       first_index=first_index & 0xFFFFFFFF, rays=flat.data_ptr() or None, rgb=rgb.data_ptr() or None,
                       hits=hits.data_ptr() if hits is not None and n else None)
        if n:
            stream = torch.cuda.current_stream(dev).cuda_stream
            _check_core(core().crtb200_shade_rays_device(self._h, C.byref(b), stream or None))
        if hits is None:
            return rgb, None
        return rgb, Hits(hits[..., 0], hits[..., 1], hits[..., 2], hits)

    def query_stats(self) -> dict:
        """Statistics of the last trace() / trace_rays() (crtb200_last_query_stats; waits for the query to finish): rays
        of its type, node / triangle tests under its count_work, handoff_closest / handoff_shadow, device_ms,
        kernel_launches."""
        st = Stats()
        _check_core(core().crtb200_last_query_stats(self._h, C.byref(st)))
        return st.as_dict()

    def debug_powf5(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = np.zeros_like(x)
        _check_core(core().crtb200_debug_powf5(self._h, x.ctypes.data, x.size, out.ctypes.data))
        return out

    def close(self):
        if self._h:
            core().crtb200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _session_params(width: int, height: int, camera: Camera, options: Options, sampling: Sampling) -> dict:
    """What a saved progressive session must agree on with the session that continues it (bit for bit)."""
    rects = [(r.row, r.col, r.width, r.height) for r in options.rects[:options.n_rects]] if options.n_rects else []
    return {
        "size": np.array([height, width], np.uint32),
        "camera": np.array(list(camera.position) + list(camera.rotation), np.float32),
        "max_depth": np.array(options.max_depth, np.uint32),
        "biases": np.array([options.shadow_bias, options.reflection_bias, options.refraction_bias], np.float32),
        "rects": np.array(rects, np.uint32).reshape(-1, 4),
        "sampling": np.array([sampling.use_gi, sampling.gi_samples, sampling.seed, sampling.frame_index], np.uint32),
        "monte_carlo_bias": np.array(sampling.monte_carlo_bias, np.float32),
    }


def _adaptive_param(adaptive: Adaptive) -> np.ndarray:
    """The stop rule as saved with an adaptive session: min, max and the bits of abs_error, rel_error."""
    return np.array([adaptive.min_samples, adaptive.max_samples, np.float32(adaptive.abs_error).view(np.uint32),
                     np.float32(adaptive.rel_error).view(np.uint32)], np.uint32)


class Progressive:
    """A progressive GI session of a Context (crtb200_accum_*, DESIGN.md 3.10.1): samples accumulate in steps, and
    after steps totalling n samples read() returns bit for bit the one-shot frame rendered with rays_per_pixel = n.
    An adaptive session (DESIGN.md 3.10.2) stops each pixel once its noise is below the Adaptive bound: pixel p of a
    read is then the one-shot frame's pixel p with rays_per_pixel = counts()[p].  `samples` counts passes."""

    def __init__(self, ctx: Context, camera: Camera, options: Options, sampling: Sampling,
                 adaptive: Optional[Adaptive] = None):
        self._ctx = ctx
        self._params = _session_params(ctx.width, ctx.height, camera, options, sampling)
        self.adaptive = adaptive
        if adaptive is not None:
            self._params["adaptive"] = _adaptive_param(adaptive)
        self.samples = 0
        if adaptive is None:
            _check_core(core().crtb200_accum_begin(ctx._h, C.byref(camera), C.byref(options), C.byref(sampling)))
        else:
            _check_core(core().crtb200_accum_begin_adaptive(ctx._h, C.byref(camera), C.byref(options), C.byref(sampling),
                                                            C.byref(adaptive)))
        ctx._session = self

    def _live(self):
        if self._ctx._session is not self:
            raise CrtError("this progressive session has ended (closed, or another one began on its context)")
        return self._ctx._h

    def step(self, n: int) -> dict:
        """Renders n more samples per pixel (n passes); returns this step's stats (with rays_diffuse and samples), and
        active_pixels and pixel_samples of the session after it."""
        if n < 0:
            raise CrtError("n must not be negative")
        st = Stats()
        _check_core(core().crtb200_accum_step(self._live(), int(n), C.byref(st)))
        self.samples += int(n)
        d = st.as_dict()
        d.update(self._ctx.sampling_stats())
        pr = self.progress()
        d["active_pixels"], d["pixel_samples"] = pr["active_pixels"], pr["pixel_samples"]
        return d

    def progress(self) -> dict:
        """{'passes', 'covered_pixels', 'active_pixels', 'pixel_samples'} (crtb200_accum_progress)."""
        pr = AccumProgress()
        _check_core(core().crtb200_accum_progress(self._live(), C.byref(pr)))
        return {k: getattr(pr, k) for k in ("passes", "covered_pixels", "active_pixels", "pixel_samples")}

    def counts(self) -> np.ndarray:
        """Per-pixel sample counts n_p (HxW uint32, 0 outside the rects; crtb200_accum_counts)."""
        counts = np.zeros((self._ctx.height, self._ctx.width), np.uint32)
        _check_core(core().crtb200_accum_counts(self._live(), counts.ctypes.data))
        return counts

    def run(self, passes_per_step: int = 8, max_steps: Optional[int] = None) -> list:
        """Steps until no pixel is active (at most max_steps steps); returns the steps' stats."""
        out = []
        while self.progress()["active_pixels"] and (max_steps is None or len(out) < max_steps):
            out.append(self.step(passes_per_step))
        return out

    def read(self, want_rgb: bool = True, want_rgb8: bool = False, want_hits: bool = False):
        """The image so far: (rgb f32 HxWx3 | None, rgb8 | None, sample 0's hits | None), laid out as Context.render's."""
        h, w = self._ctx.height, self._ctx.width
        rgb = np.zeros((h, w, 3), np.float32) if want_rgb else None
        rgb8 = np.zeros((h, w, 3), np.uint8) if want_rgb8 else None
        hits = np.zeros((h, w), HIT_DTYPE) if want_hits else None
        _check_core(core().crtb200_accum_read(self._live(), rgb.ctypes.data if rgb is not None else None,
                                              rgb8.ctypes.data if rgb8 is not None else None,
                                              hits.ctypes.data if hits is not None else None, None))
        return rgb, rgb8, hits

    def arrays(self) -> dict:
        """The accumulator: 'sum' and 'sumsq' (HxWx3 f32, 0 outside the rects), 'hit0' (sample 0's hits), 'samples'
        (passes) and 'counts' (per-pixel n_p, HxW uint32)."""
        h, w = self._ctx.height, self._ctx.width
        s = np.zeros((h, w, 3), np.float32)
        q = np.zeros((h, w, 3), np.float32)
        hit0 = np.zeros((h, w), HIT_DTYPE)
        n = C.c_uint32(0)
        _check_core(core().crtb200_accum_save(self._live(), s.ctypes.data, q.ctypes.data, hit0.ctypes.data, C.byref(n)))
        return {"sum": s, "sumsq": q, "hit0": hit0, "samples": np.uint32(n.value), "counts": self.counts()}

    def std_error(self) -> np.ndarray:
        """Per-pixel, per-channel standard error of the mean, in float64: sqrt(max(0, (Q - S^2 / n) / (n - 1)) / n)
        with the pixel's own count n = n_p (a plain session: its samples, outside the rects too); NaN below 2 samples.
        An estimate of the noise left, not part of the bit-exact contract."""
        a = self.arrays()
        n = (a["counts"] if self.adaptive is not None else np.full(a["counts"].shape, a["samples"])).astype(np.float64)[..., None]
        s, q = a["sum"].astype(np.float64), a["sumsq"].astype(np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            se = np.sqrt(np.maximum(0.0, (q - s * s / n) / (n - 1)) / n)
        return np.where(n < 2, np.nan, se)

    def save(self, path: str) -> None:
        """Writes the accumulator and the session's parameters to an .npz file (Context.resume reads it).  A plain
        session's file has no counts, as before adaptive sessions existed."""
        a = self.arrays()
        if self.adaptive is None:
            del a["counts"]
        np.savez(path, **a, **self._params)

    def close(self) -> None:
        """Ends the session and frees its device memory (crtb200_accum_end)."""
        if self._ctx._session is self:
            _check_core(core().crtb200_accum_end(self._ctx._h))
            self._ctx._session = None


class RayTracer:
    """Python view of the C++ `crt::RayTracer` mirror class (csrc/frontend/crt_raytracer.hpp):
    RayTracer(scene) -> setCamera -> render(pathToImage, mode, maxDepth)."""

    def __init__(self, scene: SceneFile, device: int = -1):
        """device >= 0: that GPU; -1 (default, like the C++ class): every visible GPU, each frame split by tiles."""
        self.scene = scene
        self._h = C.c_void_p()
        _check_front(front().crtfe_tracer_create(scene.handle, device, C.byref(self._h)))

    def set_camera(self, cam: Camera) -> None:
        _check_front(front().crtfe_tracer_set_camera(self._h, C.byref(cam)))

    def get_camera(self) -> Camera:
        cam = Camera()
        _check_front(front().crtfe_tracer_get_camera(self._h, C.byref(cam)))
        return cam

    def render(self, path_to_image: str = "", mode: int = MODE_B200_WAVEFRONT, max_depth: int = 5, literal: bool = False,
               use_gi: bool = False, gi_samples: int = 2, rays_per_pixel: int = 1, seed: int = 0,
               monte_carlo_bias: float = 1e-4):
        """use_gi / gi_samples / rays_per_pixel / monte_carlo_bias = RenderOptions' GI members, seed = RenderOptions::SEED."""
        h, w = self.scene.info.height, self.scene.info.width
        rgb = np.zeros((h, w, 3), np.float32)
        st = Stats()
        if use_gi:
            _check_front(front().crtfe_tracer_render_sampled(self._h, path_to_image.encode(), mode, max_depth, 1 if literal else 0,
                                                             1, gi_samples, rays_per_pixel, monte_carlo_bias, seed,
                                                             rgb.ctypes.data, C.byref(st)))
        else:
            _check_front(front().crtfe_tracer_render(self._h, path_to_image.encode(), mode, max_depth, 1 if literal else 0,
                                                     rgb.ctypes.data, C.byref(st)))
        return rgb, st.as_dict()

    def close(self):
        if self._h:
            front().crtfe_tracer_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
