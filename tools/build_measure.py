"""Scene set-up on one GPU: the host KD build + crtb200_upload_scene against the geometry-only flatten +
crtb200_upload_geometry (the device KD build, DESIGN.md 3.11), for hw11_room at 1920x1080, hw14_dragon_class
(1 009 202 triangles) and synthetic_10M (10 002 830 triangles) -- bench.py's scene files.

Each path runs twice, alternating (host, device, host, device), each time from a freshly parsed scene file.  Host clocks
around calls that end synchronised; the device build's own CUDA-event time and peak scratch come from
crtb200_scene_trees.  The device state both paths leave (crtb200_debug_scene_layout) is compared in the same run.  One
JSON line per run and one summary line per scene, with the GPU name and power limit read in the same process.

    python tools/build_measure.py [--out profiles/build_measure.jsonl] [--scenes hw11_room,hw14_dragon_class,synthetic_10M]
"""
from __future__ import annotations

import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "course-assignment-danielhalachev_b200"


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.splitlines()[0].split(", ") + ["?", "?"])[:2] if q.returncode == 0 else ("?", "?")
    return {"gpu": name.strip(), "power_limit": power.strip()}


def layout_digest(ctx) -> str:
    lay = ctx.debug_scene_layout()
    h = hashlib.sha256()
    for k in ("nodes", "leaf_refs", "top_refs", "meshes"):
        h.update(lay[k].tobytes())
    h.update(repr((lay["top_begin"], lay["top_end"], lay["nested_ok"])).encode())
    return h.hexdigest()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--scenes", default="hw11_room,hw14_dragon_class,synthetic_10M")
    args = ap.parse_args()
    bench = importlib.import_module("bench")
    crt = importlib.import_module(PKG)
    info = gpu_info()
    ctx = crt.Context(0)
    lines = []

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)

    for name in args.scenes.split(","):
        f, folder, kw, tex, depth = bench.ensure_scene(name, {})
        digests = {}
        runs = []
        for rep in range(2):
            for path in ("host", "device"):
                t0 = time.perf_counter()
                sf = crt.SceneFile(f, folder)
                t1 = time.perf_counter()
                rec = {"scene": name, "triangles": int(sf.info.n_triangles), "meshes": int(sf.info.n_meshes), "path": path,
                       "rep": rep, "parse_s": round(t1 - t0, 4)}
                if path == "host":
                    flat = sf.flatten()
                    t2 = time.perf_counter()
                    ctx.upload(flat, keepalive=sf)
                    t3 = time.perf_counter()
                    rec.update(build_seconds=round(sf.build_seconds, 4), flatten_s=round(t2 - t1, 4), upload_scene_s=round(t3 - t2, 4),
                               setup_s=round(t3 - t1, 4))
                else:
                    geo = sf.flatten(trees=False)
                    t2 = time.perf_counter()
                    ctx.upload_geometry(geo, keepalive=sf)
                    t3 = time.perf_counter()
                    tr = ctx.scene_trees()
                    rec.update(geometry_flatten_s=round(t2 - t1, 4), upload_geometry_s=round(t3 - t2, 4), setup_s=round(t3 - t1, 4),
                               build_kernels_ms=round(tr["build_ms"], 3), peak_scratch_bytes=int(tr["peak_scratch_bytes"]),
                               nodes=int(len(tr["mesh_nodes"]) + len(tr["top_nodes"])), leaf_refs=int(len(tr["mesh_leaf_refs"])))
                digests.setdefault(path, set()).add(layout_digest(ctx))
                rec.update(info)
                emit(rec)
                runs.append(rec)
                sf.close()
        best = lambda p, k: min(r[k] for r in runs if r["path"] == p)
        emit({"scene": name, "summary": True, "identical_device_state": len(digests["host"] | digests["device"]) == 1,
              "host_build_plus_upload_s": best("host", "setup_s"), "device_build_plus_upload_s": best("device", "setup_s"),
              "host_build_seconds": best("host", "build_seconds"), "upload_scene_s": best("host", "upload_scene_s"),
              "upload_geometry_s": best("device", "upload_geometry_s"), "build_kernels_ms": best("device", "build_kernels_ms"),
              "parse_s": min(r["parse_s"] for r in runs), **info})
    ctx.close()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
