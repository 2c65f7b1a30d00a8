"""Adaptive progressive sessions (DESIGN.md 3.10.2) on one GPU: hw11_room at 1920x1080 and hw14_dragon_class at
3840x2160, GI_SAMPLE_SIZE 1, MAX_DEPTH 5, max_samples 128 (app/main.cpp's sample count).  Cases:
  run_to_completion   Progressive.run(8) at two error bounds: wall time (host clock around calls that synchronise),
                      pixel-samples, a histogram of n_p, and per step the device time against the active fraction at
                      the step's start (pass time against active fraction)
  degenerate          min == max == 32 against a plain session of 32 samples, both in steps of 8
  rmse_equal_time     (hw11_room) RMSE against a 1024-sample plain reference, of the adaptive run at the looser bound
                      and of a plain session stepped by 8 until it has used at least the adaptive run's wall time,
                      over the colour components finite in all three images
Each case after a warm-up.  One JSON line per case, with the GPU name and power limit read in the same process.

    python tools/adaptive_measure.py [--out profiles/adaptive_measure.jsonl]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gi_measure import PKG, RUNS, gpu_info  # noqa: E402

BOUNDS = [dict(abs_error=0.004, rel_error=0.04), dict(abs_error=0.001, rel_error=0.01)]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--reference-samples", type=int, default=1024)
    args = ap.parse_args()
    crt = importlib.import_module(PKG)
    scenes = importlib.import_module(PKG + ".scenes")
    info = gpu_info()
    lines = []

    def emit(rec):
        line = json.dumps({**rec, **info})
        print(line, flush=True)
        lines.append(line)

    def timed_run(ctx, cam, opt, smp, ad):
        t0 = time.perf_counter()
        p = ctx.progressive(cam, opt, smp, ad)
        steps, active = [], p.progress()["active_pixels"]
        while active:
            st = p.step(8)
            steps.append((active, st["device_ms"]))
            active = st["active_pixels"]
        p.read()
        ms = (time.perf_counter() - t0) * 1e3
        return p, ms, steps

    with tempfile.TemporaryDirectory() as d:
        for name, w, h, kw in RUNS:
            scenes.write_crtscene(os.path.join(d, name + ".crtscene"), scenes.CONFIGS[name](width=w, height=h, **kw))
            sf = crt.SceneFile(name + ".crtscene", d)
            flat = sf.flatten()
            ctx = crt.Context(0)
            ctx.upload(flat, keepalive=sf)
            cam, opt = sf.camera(), crt.make_options(max_depth=5)
            smp = crt.Sampling.make(gi_samples=1)
            base = {"scene": name, "width": w, "height": h, "gi_samples": 1, "depth": 5}
            px = w * h
            ctx.progressive(cam, opt, smp, crt.Adaptive.make(2, 2)).run(2)  # warm-up
            results = []
            for b in BOUNDS:
                ad = crt.Adaptive.make(min_samples=8, max_samples=128, **b)
                p, ms, steps = timed_run(ctx, cam, opt, smp, ad)
                counts = p.counts()
                rgb = p.read()[0]
                pr = p.progress()
                p.close()
                edges = [1, 9, 17, 33, 65, 128, 129]
                hist = np.histogram(counts, bins=edges)[0].tolist()
                emit({**base, "case": "run_to_completion", "min_samples": 8, "max_samples": 128, **b, "ms": round(ms, 1),
                      "passes": pr["passes"], "pixel_samples": pr["pixel_samples"],
                      "mean_samples": round(pr["pixel_samples"] / px, 2), "uniform_128_pixel_samples": 128 * px,
                      "hist_edges": edges, "hist": hist,
                      "steps_active_fraction": [round(a / px, 4) for a, _ in steps],
                      "steps_device_ms": [round(t, 2) for _, t in steps]})
                results.append((b, ms, rgb))
            # min == max against plain
            for kind in ("adaptive_min_eq_max", "plain"):
                for rep in range(2):
                    t0 = time.perf_counter()
                    p = ctx.progressive(cam, opt, smp, crt.Adaptive.make(32, 32) if kind != "plain" else None)
                    dev = sum(p.step(8)["device_ms"] for _ in range(4))
                    p.read()
                    ms = (time.perf_counter() - t0) * 1e3
                    p.close()
                    emit({**base, "case": "degenerate_32", "kind": kind, "rep": rep, "ms": round(ms, 1), "device_ms": round(dev, 1)})
            if name == "hw11_room":
                ref = ctx.progressive(cam, opt, smp)
                for _ in range(args.reference_samples // 64):
                    ref.step(64)
                want = ref.read()[0].astype(np.float64)
                ref.close()
                b, ms_ad, rgb_ad = results[0]
                t0 = time.perf_counter()
                p = ctx.progressive(cam, opt, smp)
                while (time.perf_counter() - t0) * 1e3 < ms_ad:
                    p.step(8)
                rgb_pl = p.read()[0]
                ms_pl = (time.perf_counter() - t0) * 1e3
                n_pl = p.samples
                p.close()

                # over the pixels that are finite in all three images (the room has pixels whose samples are NaN)
                ok = np.isfinite(want) & np.isfinite(rgb_ad) & np.isfinite(rgb_pl)

                def rmse(x):
                    return float(np.sqrt(np.mean((x.astype(np.float64)[ok] - want[ok]) ** 2)))
                emit({**base, "case": "rmse_equal_time", "reference_samples": args.reference_samples, **b,
                      "components_excluded": int(ok.size - ok.sum()),
                      "adaptive_ms": round(ms_ad, 1), "adaptive_rmse": rmse(rgb_ad),
                      "plain_ms": round(ms_pl, 1), "plain_samples": n_pl, "plain_rmse": rmse(rgb_pl)})
            ctx.close()
            sf.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
