"""GI / supersampling throughput on one GPU: hw11_room at 1920x1080 and hw14_dragon_class at 3840x2160, each with the
reference app's setting (app/main.cpp: RAYS_PER_PIXEL 128, GI_SAMPLE_SIZE 1, MAX_DEPTH 5) and with spp 1, G 2, plus
the unsampled frame for scale.  Warm-up frames first, then CUDA-event time of whole frames (crtb200_render_device into
device memory).  One JSON line per run: ms per frame, rays by type, Mrays/s, and the GPU name and power limit read in
the same process.

    python tools/gi_measure.py [--frames N] [--warmup W] [--out profiles/gi_measure.jsonl]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "course-assignment-danielhalachev_b200"

RUNS = [
    ("hw11_room", 1920, 1080, dict(sphere_n=32)),
    ("hw14_dragon_class", 3840, 2160, dict()),
]
SETTINGS = [("off", None), ("main_cpp", dict(rays_per_pixel=128, gi_samples=1)), ("spp1_G2", dict(rays_per_pixel=1, gi_samples=2))]


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = (q.stdout.splitlines()[0].split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name.strip(), "power_limit": power.strip(), "max_sm_clock": clk.strip()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    crt = importlib.import_module(PKG)
    scenes = importlib.import_module(PKG + ".scenes")
    info = gpu_info()
    lines = []
    with tempfile.TemporaryDirectory() as d:
        for name, w, h, kw in RUNS:
            scenes.write_crtscene(os.path.join(d, name + ".crtscene"), scenes.CONFIGS[name](width=w, height=h, **kw))
            sf = crt.SceneFile(name + ".crtscene", d)
            flat = sf.flatten()
            ctx = crt.Context(0)
            ctx.upload(flat, keepalive=sf)
            out = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
            opt = crt.make_options(max_depth=5)
            off_ms = None
            for label, smp in SETTINGS:
                ctx.set_sampling(crt.Sampling.make(**smp) if smp else None)
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                for _ in range(args.warmup):
                    ctx.render_device(sf.camera(), opt, d_rgb=out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                start.record()
                for _ in range(args.frames):
                    ctx.render_device(sf.camera(), opt, d_rgb=out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
                end.record()
                torch.cuda.synchronize()
                ms = start.elapsed_time(end) / args.frames
                st, ss = ctx.last_stats(), ctx.sampling_stats()
                rays = {k: st[k] for k in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction")}
                rays["rays_diffuse"] = ss["rays_diffuse"]
                total = sum(rays.values())
                spp = ss["samples"]
                rec = {"scene": name, "width": w, "height": h, "setting": label, "spp": spp,
                       "gi_samples": smp["gi_samples"] if smp else 0, "depth": 5, "ms_per_frame": round(ms, 3),
                       **rays, "mrays_per_s": round(total / ms / 1e3, 1), **info}
                if off_ms is None:
                    off_ms = ms
                else:
                    rec["per_sample_pass_over_unsampled_frame"] = round(ms / spp / off_ms, 3)
                line = json.dumps(rec)
                print(line, flush=True)
                lines.append(line)
            ctx.close()
            sf.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
