"""Throughput of caller-supplied ray batches (crtb200_trace_rays_device, DESIGN.md 3.12) on one GPU: hw14_dragon_class at
3840x2160 and synthetic_10M at 1920x1080 (bench.py's scenes and cameras), three workloads each:

  camera   the camera rays of every pixel (Context.generate_rays_device), RAY_PRIMARY, next to the closest_ms of a
           concurrency-1 render of the same camera (both scenes are diffuse-only: closest_ms is the primary launch alone)
  shadow   from the primary hits to every light, unit directions, max_distance = the distance to the light
  ao       one incoherent ray per hit: a random unit direction from the hit point, max_distance = 2 % of the scene box's
           diagonal, as a closest-hit (RAY_REFLECTION) and as a shadow query

Device path: CUDA events around Context.trace on the current stream, warm-up passes first, the L2 flushed (a 256 MiB fill,
as bench.py does) before every timed pass, median of --steps passes, traversal 0 and 1.  Host path (traversal 0): wall
time of crtb200_trace_rays (copies to and from the device included) of this build and, with --parent-lib, of another
build of the library (e.g. the one before the query path existed, whose host call ran k_query, one ray per thread).  One JSON line
per (scene, workload, path), with the card's name and power limit read in the same process.

    python tools/query_measure.py [--steps K] [--warmup W] [--parent-lib PATH] [--out profiles/query_measure.jsonl]
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "course-assignment-danielhalachev_b200"
RUNS = [("hw14_dragon_class", 3840, 2160), ("synthetic_10M", 1920, 1080)]


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = (q.stdout.splitlines()[0].split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name.strip(), "power_limit": power.strip(), "max_sm_clock": clk.strip()}


def workloads(torch, crt, flat, rays, hits):
    """name -> (ray type, rays (n, 6), max_distance or None)"""
    s = flat.contents
    r = rays.reshape(-1, 6)
    hit = hits.mesh.reshape(-1) >= 0
    t = hits.t.reshape(-1).view(torch.float32)[hit]
    d_cam = r[hit, 3:]
    p = r[hit, :3] + d_cam * t[:, None]
    lights = torch.tensor([list(s.lights[i].position) for i in range(s.n_lights)], dtype=torch.float32, device=rays.device)
    to = lights[None, :, :] - p[:, None, :]
    ldist = torch.linalg.norm(to, dim=2)
    ld = to / ldist[..., None]
    sh = torch.cat([p[:, None, :] + ld * 1e-3, ld], dim=2).reshape(-1, 6).contiguous()
    v = torch.from_numpy(np.ctypeslib.as_array(s.vertex_position, shape=(3 * s.n_vertices,)).reshape(-1, 3).copy())
    diag = float(torch.linalg.norm(v.max(dim=0).values - v.min(dim=0).values))
    g = torch.Generator(device=rays.device).manual_seed(7)
    ao_d = torch.randn(p.shape, generator=g, device=rays.device)
    ao_d = ao_d / torch.linalg.norm(ao_d, dim=1, keepdim=True)
    ao = torch.cat([p - d_cam * 1e-3, ao_d], dim=1).contiguous()
    ao_dist = torch.full((ao.shape[0],), 0.02 * diag, dtype=torch.float32, device=rays.device)
    return {"camera": (crt.RAY_PRIMARY, r.contiguous(), None), "shadow": (crt.RAY_SHADOW, sh, ldist.reshape(-1).contiguous()),
            "ao_closest": (crt.RAY_REFLECTION, ao, None), "ao_shadow": (crt.RAY_SHADOW, ao, ao_dist)}


def device_ms(torch, ctx, rt, rays, dist, trav, steps, warmup, flush):
    out = None
    for _ in range(warmup):
        out = ctx.trace(rays, rt, dist, traversal=trav, out=out)
    times = []
    for k in range(steps):
        flush.fill_(k & 0xFF)  # L2 flush, outside the events
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = ctx.trace(rays, rt, dist, traversal=trav, out=out)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2], ctx.query_stats()


def host_ms(torch, lib, h, rt, rays, dist, trav, steps, warmup, flush):
    """Wall time of a synchronous host call crtb200_trace_rays of library `lib` on context h."""
    hr = rays.cpu().numpy()
    n = hr.shape[0]
    hd = dist.cpu().numpy() if dist is not None else None
    out = np.zeros(n, np.uint8) if rt == 1 else np.zeros((n, 3), np.int32)
    args = (hd.ctypes.data if hd is not None else None, None if rt == 1 else out.ctypes.data, out.ctypes.data if rt == 1 else None)
    times = []
    for k in range(warmup + steps):
        flush.fill_(k & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = lib.crtb200_trace_rays(h, hr.ctypes.data, n, rt, trav, *args)
        t1 = time.perf_counter()
        assert rc == 0, rc
        if k >= warmup:
            times.append((t1 - t0) * 1e3)
    return sorted(times)[len(times) // 2], out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--host-steps", type=int, default=2)
    ap.add_argument("--parent-lib", default="", help="another build of libcrtb200.so whose host crtb200_trace_rays is timed too")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    crt = importlib.import_module(PKG)
    bench_mod = importlib.import_module("bench")
    info = gpu_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    parent = None
    if args.parent_lib:
        parent = C.CDLL(os.path.abspath(args.parent_lib))  # RTLD_LOCAL: its symbols stay apart from this build's
        parent.crtb200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        parent.crtb200_upload_scene.argtypes = [C.c_void_p, C.c_void_p]
        parent.crtb200_destroy.argtypes = [C.c_void_p]
        parent.crtb200_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    lines = []

    def emit(rec):
        line = json.dumps({**rec, **info})
        print(line, flush=True)
        lines.append(line)

    for name, w, h in RUNS:
        f, folder, kw, tex, depth = bench_mod.ensure_scene(name, {})
        sf = crt.SceneFile(f, folder)
        flat = sf.flatten()
        assert (sf.info.width, sf.info.height) == (w, h)
        ctx = crt.Context(0)
        ctx.upload(flat, keepalive=sf)
        cam = sf.camera()
        ctx.set_concurrency(1)
        closest = []
        for k in range(args.warmup + args.steps):
            flush.fill_(k & 0xFF)
            torch.cuda.synchronize()
            _, _, _, st = ctx.render(cam, crt.make_options(max_depth=depth), want_rgb=False)
            if k >= args.warmup:
                closest.append(st["closest_ms"])
        render_closest_ms = sorted(closest)[len(closest) // 2]
        rays = ctx.generate_rays_device(cam)
        hits = ctx.trace(rays, crt.RAY_PRIMARY)
        ph = None
        if parent is not None:
            ph = C.c_void_p()
            assert parent.crtb200_create(0, C.byref(ph)) == 0
            assert parent.crtb200_upload_scene(ph, C.cast(flat, C.c_void_p)) == 0
        for wl, (rt, q, dist) in workloads(torch, crt, flat, rays, hits).items():
            n = q.shape[0]
            base = {"scene": name, "width": w, "height": h, "workload": wl, "ray_type": int(rt), "rays": n}
            for trav in (0, 1):
                ms, st = device_ms(torch, ctx, rt, q, dist, trav, args.steps, args.warmup, flush)
                rec = dict(base, path="device", traversal=trav, ms=round(ms, 3), mrays_per_s=round(n / ms / 1e3, 1),
                           handoff=st["handoff_closest"] + st["handoff_shadow"], kernel_launches=st["kernel_launches"])
                if wl == "camera":
                    rec["render_closest_ms"] = round(render_closest_ms, 3)
                    rec["render_primary_mrays_per_s"] = round(n / render_closest_ms / 1e3, 1)
                emit(rec)
            for label, lib, hctx in (("host", crt.core(), ctx._h), ("host_parent_build", parent, ph)):
                if lib is None:
                    continue
                ms, _ = host_ms(torch, lib, hctx, rt, q, dist, 0, args.host_steps, 1, flush)
                emit(dict(base, path=label, traversal=0, ms=round(ms, 3), mrays_per_s=round(n / ms / 1e3, 1)))
        if ph is not None:
            parent.crtb200_destroy(ph)
        ctx.close()
        sf.close()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
