"""TEST INFRASTRUCTURE ONLY.  ctypes binding of tests/shade_oracle.c: RayTracer::shootRay for caller-supplied rays on
the CPU, unsampled and under the sampling contract (DESIGN.md 3.13), and the camera rays that make a frame such a batch.
The library is compiled on first use into a temporary directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from gi_oracle import CSRC, HERE, HIT_DTYPE, OracleStats

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="shade_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libshade_oracle.so")
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared",
                        "-I", CSRC, "-o", so, os.path.join(HERE, "shade_oracle.c"), "-lm"], check=True)
        l = C.CDLL(so)
        l.crt_oracle_shade_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.POINTER(OracleStats), C.c_int]
        l.crt_oracle_shade_rays_sampled.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                    C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                    C.POINTER(OracleStats), C.POINTER(C.c_uint64), C.c_int]
        l.crt_oracle_camera_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        l.crt_oracle_camera_rays_sampled.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        _lib = l
    return _lib


def _stats(st: OracleStats) -> dict:
    return {n: getattr(st, n) for n, _ in st._fields_ if n != "max_query_tests"}


def shade_rays(scene_ptr, rays, ray_type: int, options, sampling=None, sample: int = 0, first_index: int = 0,
               threads: int = 0):
    """crt_oracle_shade_rays (sampling None or use_gi = 0) or crt_oracle_shade_rays_sampled: returns (rgb n x 3 f32,
    hits n, stats dict; with sampling also rays_diffuse)."""
    rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
    n = rays.shape[0]
    rgb = np.zeros((n, 3), np.float32)
    hits = np.zeros(n, HIT_DTYPE)
    st = OracleStats()
    threads = threads if threads > 0 else (os.cpu_count() or 1)
    scene = C.cast(scene_ptr, C.c_void_p)
    if sampling is not None and sampling.use_gi:
        diffuse = C.c_uint64(0)
        rc = lib().crt_oracle_shade_rays_sampled(scene, rays.ctypes.data, n, ray_type, C.addressof(options),
                                                 C.addressof(sampling), sample & 0xFFFFFFFF, first_index & 0xFFFFFFFF,
                                                 rgb.ctypes.data, hits.ctypes.data, C.byref(st), C.byref(diffuse), threads)
        d = _stats(st)
        d["rays_diffuse"] = diffuse.value
    else:
        rc = lib().crt_oracle_shade_rays(scene, rays.ctypes.data, n, ray_type, C.addressof(options), rgb.ctypes.data,
                                         hits.ctypes.data, C.byref(st), threads)
        d = _stats(st)
    if rc != 0:
        raise RuntimeError("crt_oracle_shade_rays failed")
    return rgb, hits, d


def camera_rays(scene_ptr, camera, sampling=None, sample: int = 0) -> np.ndarray:
    """getRay of every pixel, H x W x 6 (one normalisation); with GI sampling the jittered rays of sample `sample`."""
    s = scene_ptr.contents
    out = np.zeros((s.height, s.width, 6), np.float32)
    scene = C.cast(scene_ptr, C.c_void_p)
    if sampling is not None and sampling.use_gi:
        rc = lib().crt_oracle_camera_rays_sampled(scene, C.addressof(camera), C.addressof(sampling), sample, out.ctypes.data)
    else:
        rc = lib().crt_oracle_camera_rays(scene, C.addressof(camera), out.ctypes.data)
    if rc != 0:
        raise RuntimeError("crt_oracle_camera_rays failed")
    return out
