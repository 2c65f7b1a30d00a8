"""Cost of moving a scene's vertices on the GPU (crtb200_update_vertices_device, DESIGN.md 3.14) on one GPU, on bench.py's
hw14_dragon_class (1 M triangles) and synthetic_10M scenes, the scene's largest mesh (its sphere) displaced radially by a
torch kernel:

  update         Context.update_vertices: CUDA events on the current stream and host wall time around the (synchronous)
                 call, median of --steps after --warmup; build_ms and peak_scratch_bytes of the last update from
                 scene_trees(); pre_build_ms = update - build: the triangle records, the stable sort of the corners,
                 the vertex normals, scratch allocation and the host's share
  upload         the baseline: Context.upload_geometry of the same edited positions from host arrays, the normals
                 precomputed (tests/update_oracle.py) and not timed; host wall time, same median
  animation      hw14_dragon_class at 3840x2160: 30 frames of (deformation, update, render_device) against 30
                 render_device calls alone; ms per frame from wall time over the 30 frames, ended by a synchronise

One JSON line per (scene, measurement), with the card's name and power limit read in the same process.

    python tools/update_measure.py [--steps 5] [--warmup 1] [--out profiles/update_measure.jsonl]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
PKG = "course-assignment-danielhalachev_b200"

from query_measure import gpu_info  # noqa: E402


def median(xs):
    return sorted(xs)[len(xs) // 2]


def largest_mesh_vertices(torch, crt, flat):
    """Global vertex ids of the vertices the largest mesh's triangles use (CUDA tensor)."""
    s = flat.contents
    best = max(range(s.n_meshes), key=lambda m: s.meshes[m].n_triangles)
    me = s.meshes[best]
    import numpy as np
    tv = np.ctypeslib.as_array(s.triangle_vertex, shape=(s.n_triangles * 3,)).reshape(-1, 3)
    ids = np.unique(tv[me.first_triangle:me.first_triangle + me.n_triangles])
    return torch.from_numpy(ids.astype(np.int64)).cuda(), best, int(me.n_triangles)


def displaced(torch, base, ids, centre, phase):
    """The largest mesh's vertices pushed along their direction from its centre by a travelling sine wave."""
    out = base.clone()
    p = base[ids]
    d = p - centre
    out[ids] = centre + d * (1.0 + 0.05 * torch.sin(6.0 * d[:, 1:2] + phase))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "update_measure.jsonl"))
    a = ap.parse_args()
    import torch
    crt = importlib.import_module(PKG)
    bench = importlib.import_module("bench")
    uo = importlib.import_module("update_oracle")
    info = gpu_info()
    lines = []

    def emit(d):
        d = dict(info, **d)
        lines.append(d)
        print(json.dumps(d), flush=True)

    for name in ("hw14_dragon_class", "synthetic_10M"):
        f, folder, kw, tex, depth = bench.ensure_scene(name, {})
        sf = crt.SceneFile(f, folder)
        geo = sf.flatten(trees=False)
        ctx = crt.Context(0)
        ctx.upload_geometry(geo, keepalive=sf)
        s = geo.contents
        base = torch.from_numpy(crt.scene_vertex_positions(geo)).cuda()
        ids, mesh, mesh_tris = largest_mesh_vertices(torch, crt, geo)
        centre = base[ids].mean(dim=0)
        pos = displaced(torch, base, ids, centre, 0.5).contiguous()

        ev_ms, wall_ms = [], []
        for i in range(a.warmup + a.steps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            ctx.update_vertices(pos)
            e1.record()
            t1 = time.perf_counter()
            e1.synchronize()
            if i >= a.warmup:
                ev_ms.append(e0.elapsed_time(e1))
                wall_ms.append((t1 - t0) * 1e3)
        t = ctx.scene_trees()
        upd = median(wall_ms)
        emit({"scene": name, "measure": "update", "n_triangles": s.n_triangles, "n_vertices": s.n_vertices,
              "displaced_mesh": mesh, "displaced_mesh_triangles": mesh_tris, "update_ms": round(median(ev_ms), 3),
              "update_wall_ms": round(upd, 3), "build_ms": round(t["build_ms"], 3),
              "pre_build_ms": round(upd - t["build_ms"], 3), "peak_scratch_bytes": int(t["peak_scratch_bytes"]),
              "steps": a.steps, "warmup": a.warmup})

        e = uo.EditedScene(crt, geo, pos.cpu().numpy())  # normals precomputed on the host, outside the timing
        up_ms = []
        for i in range(a.warmup + a.steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.upload_geometry(e.ptr, keepalive=e)
            t1 = time.perf_counter()
            if i >= a.warmup:
                up_ms.append((t1 - t0) * 1e3)
        t = ctx.scene_trees()
        emit({"scene": name, "measure": "upload_geometry", "n_triangles": s.n_triangles, "upload_wall_ms": round(median(up_ms), 3),
              "build_ms": round(t["build_ms"], 3), "peak_scratch_bytes": int(t["peak_scratch_bytes"]),
              "update_over_upload": round(upd / median(up_ms), 3)})

        if name == "hw14_dragon_class":
            ctx.upload_geometry(geo, keepalive=sf)
            cam, opt = sf.camera(), crt.make_options(max_depth=depth)
            frame = torch.empty((sf.info.height, sf.info.width, 3), dtype=torch.float32, device="cuda")
            stream = torch.cuda.current_stream().cuda_stream

            def render():
                ctx.render_device(cam, opt, frame.data_ptr(), 0, stream)

            def animate(k):
                ctx.update_vertices(displaced(torch, base, ids, centre, 0.2 * k).contiguous())
                render()

            res = {}
            for label, step in (("render_only", lambda k: render()), ("deform_update_render", animate),
                                ("render_only_again", lambda k: render())):
                step(0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for k in range(a.frames):
                    step(k + 1)
                torch.cuda.synchronize()
                res[label] = (time.perf_counter() - t0) * 1e3 / a.frames
            emit({"scene": name, "measure": "animation", "width": sf.info.width, "height": sf.info.height, "frames": a.frames,
                  "render_ms_per_frame": round(res["render_only"], 3),
                  "render_ms_per_frame_after": round(res["render_only_again"], 3),
                  "animated_ms_per_frame": round(res["deform_update_render"], 3),
                  "update_share": round(1 - res["render_only"] / res["deform_update_render"], 3)})
        ctx.close()
        del e
        sf.close()
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        for d in lines:
            fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
