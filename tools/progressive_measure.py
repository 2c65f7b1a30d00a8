"""Cost of progressive GI sessions (DESIGN.md 3.10.1) against the one-shot frame, on one GPU: hw11_room at 1920x1080 and
hw14_dragon_class at 3840x2160 with the reference app's setting (app/main.cpp: 128 samples, GI_SAMPLE_SIZE 1, MAX_DEPTH
5).  Cases: the one-shot 128-sample frame (crtb200_render_device into device memory, CUDA events); sessions of steps of
1, 8 and 32 samples without reads, and steps of 8 with a float read after each (host clock around the calls, which
synchronise).  Also: the latency to the first image (begin + a 1-sample step + a read), and the cost of a read and of a
save (device -> host copy of S, Q and the hits).  Each case after a warm-up of the same case at fewer samples.  One
JSON line per case, with the GPU name and power limit read in the same process.

    python tools/progressive_measure.py [--samples 128] [--out profiles/progressive_measure.jsonl]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gi_measure import PKG, RUNS, gpu_info  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=128)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    crt = importlib.import_module(PKG)
    scenes = importlib.import_module(PKG + ".scenes")
    info = gpu_info()
    spp = args.samples
    lines = []

    def emit(rec):
        line = json.dumps({**rec, **info})
        print(line, flush=True)
        lines.append(line)

    with tempfile.TemporaryDirectory() as d:
        for name, w, h, kw in RUNS:
            scenes.write_crtscene(os.path.join(d, name + ".crtscene"), scenes.CONFIGS[name](width=w, height=h, **kw))
            sf = crt.SceneFile(name + ".crtscene", d)
            flat = sf.flatten()
            ctx = crt.Context(0)
            ctx.upload(flat, keepalive=sf)
            cam, opt = sf.camera(), crt.make_options(max_depth=5)
            smp = crt.Sampling.make(gi_samples=1, rays_per_pixel=spp)
            base = {"scene": name, "width": w, "height": h, "samples": spp, "gi_samples": 1, "depth": 5}
            # one-shot
            out = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda")
            stream = torch.cuda.current_stream().cuda_stream
            ctx.set_sampling(smp)
            ctx.render_device(cam, opt, d_rgb=out.data_ptr(), stream=stream)
            torch.cuda.synchronize()
            for rep in range(2):
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                start.record()
                ctx.render_device(cam, opt, d_rgb=out.data_ptr(), stream=stream)
                end.record()
                torch.cuda.synchronize()
                ms = start.elapsed_time(end)
                emit({**base, "case": "one_shot", "rep": rep, "ms": round(ms, 3), "ms_per_sample": round(ms / spp, 4)})
            ctx.set_sampling(None)
            # sessions
            for step, read in ((1, False), (8, False), (32, False), (8, True)):
                for warm in (True, False):
                    total = 2 * step if warm else spp
                    p = ctx.progressive(cam, opt, smp)
                    t0 = time.perf_counter()
                    dev = 0.0
                    for _ in range(total // step):
                        dev += p.step(step)["device_ms"]
                        if read:
                            p.read()
                    ms = (time.perf_counter() - t0) * 1e3
                    p.close()
                if read:
                    emit({**base, "case": f"steps_of_{step}_read_each", "ms": round(ms, 3), "ms_per_sample": round(ms / spp, 4)})
                else:
                    emit({**base, "case": f"steps_of_{step}", "ms": round(ms, 3), "ms_per_sample": round(ms / spp, 4),
                          "device_ms": round(dev, 3), "device_ms_per_sample": round(dev / spp, 4)})
            # first image, read, save
            p = ctx.progressive(cam, opt, smp)
            p.step(1)
            p.read()
            p.close()
            t0 = time.perf_counter()
            p = ctx.progressive(cam, opt, smp)
            p.step(1)
            p.read()
            first = (time.perf_counter() - t0) * 1e3
            reads, saves = [], []
            for _ in range(5):
                t0 = time.perf_counter()
                p.read()
                reads.append((time.perf_counter() - t0) * 1e3)
                t0 = time.perf_counter()
                p.arrays()
                saves.append((time.perf_counter() - t0) * 1e3)
            p.close()
            emit({**base, "case": "first_image", "ms": round(first, 3)})
            emit({**base, "case": "read_rgb_f32", "ms_median": round(sorted(reads)[2], 3)})
            emit({**base, "case": "save_to_host_arrays", "ms_median": round(sorted(saves)[2], 3)})
            ctx.close()
            sf.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
