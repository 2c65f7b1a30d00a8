"""Throughput of caller-supplied rays shaded through the frame pipeline (crtb200_shade_rays_device, DESIGN.md 3.13) on
one GPU, on bench.py's scenes and cameras:

  hw14_dragon_class 3840x2160   camera rays (Context.generate_rays_device), Context.shade against render_device
  hw11_room 1920x1080 depth 5   the same comparison
  hw11_room GI, G = 2           one shaded sample of the camera rays against a rays_per_pixel = 1 GI render_device
  panorama                      a 4096x2048 equirectangular panorama from each scene's camera position, built in torch:
                                no render counterpart, reported in Mrays/s

generate_rays_device writes shootRay-normalised rays, which shade normalises once more: the same work as the frame's
camera rays, not the same bits (the render-identity tests feed getRay's rays).  CUDA events around each call on the
current stream, the L2 flushed (a 256 MiB fill) before every timed pass, median of --steps passes after --warmup.  One
JSON line per (scene, workload, path), with the card's name and power limit read in the same process.

    python tools/shade_measure.py [--steps 7] [--warmup 2] [--out profiles/shade_measure.jsonl]
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
PKG = "course-assignment-danielhalachev_b200"

from query_measure import gpu_info  # noqa: E402


def panorama(torch, pos, w=4096, h=2048):
    """Equirectangular rays from pos: column -> azimuth, row -> polar angle, unit directions."""
    x = (torch.arange(w, device="cuda", dtype=torch.float32) + 0.5) * (2 * math.pi / w)
    y = (torch.arange(h, device="cuda", dtype=torch.float32) + 0.5) * (math.pi / h)
    th, ph = torch.meshgrid(y, x, indexing="ij")
    d = torch.stack([torch.sin(th) * torch.cos(ph), torch.cos(th), torch.sin(th) * torch.sin(ph)], dim=-1)
    o = torch.tensor(list(pos), dtype=torch.float32, device="cuda").expand(h, w, 3)
    return torch.cat([o, d], dim=-1).contiguous()


def timed(torch, fn, steps, warmup, flush):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return sorted(ms)[len(ms) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shade_measure.jsonl"))
    a = ap.parse_args()
    import torch
    crt = importlib.import_module(PKG)
    bench = importlib.import_module("bench")
    info = gpu_info()
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    ctx = crt.Context(0)
    lines = []
    for name, depth_over, gi in (("hw14_dragon_class", None, 0), ("hw11_room", 5, 0), ("hw11_room", 5, 2)):
        f, folder, kw, tex, depth = bench.ensure_scene(name, {})
        depth = depth_over if depth_over is not None else depth
        sf = crt.SceneFile(f, folder)
        ctx.upload(sf.flatten(), keepalive=sf)
        cam, opt = sf.camera(), crt.make_options(max_depth=depth)
        ctx.set_sampling(crt.Sampling.make(gi_samples=gi, rays_per_pixel=1, seed=1) if gi else None)
        h, w = sf.info.height, sf.info.width
        frame = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        rays = ctx.generate_rays_device(cam)
        out = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream
        render_ms = timed(torch, lambda: ctx.render_device(cam, opt, frame.data_ptr(), 0, stream), a.steps, a.warmup, flush)
        shade_ms = timed(torch, lambda: ctx.shade(rays, max_depth=depth, out=out), a.steps, a.warmup, flush)
        st = ctx.last_stats()
        rec = dict(info, scene=name, width=w, height=h, max_depth=depth, gi_samples=gi, workload="camera",
                   render_ms=round(render_ms, 4), shade_ms=round(shade_ms, 4), shade_over_render=round(shade_ms / render_ms, 4),
                   rays_total=st["rays_total"], shade_mrays_s=round(st["rays_total"] / shade_ms / 1e3, 1))
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        if not gi:
            pano = panorama(torch, cam.position)
            pout = torch.empty(pano.shape[:-1] + (3,), dtype=torch.float32, device="cuda")
            ms = timed(torch, lambda: ctx.shade(pano, max_depth=depth, out=pout), a.steps, a.warmup, flush)
            st = ctx.last_stats()
            rec = dict(info, scene=name, width=4096, height=2048, max_depth=depth, gi_samples=0, workload="panorama",
                       shade_ms=round(ms, 4), rays_total=st["rays_total"], shade_mrays_s=round(st["rays_total"] / ms / 1e3, 1),
                       camera_mrays_s=round(pano.shape[0] * pano.shape[1] / ms / 1e3, 1))
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    ctx.close()
    with open(a.out, "w") as fh:
        for rec in lines:
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
