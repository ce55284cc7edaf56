"""What the denoiser costs and buys on BASELINE config 2 (data/scene.obj, 1920x1080, 8 bounces, target 1024 spp).

Cost: CUDA-event device time of sqt_denoise (stats.device_ms: prep, levels, tone map; the features once per frame) at levels
1..8 with the default sigmas, warmed up, median of --reps calls, on a 16-spp frame; the first call of a frame also computes
the features, reported as `features_ms` (first call minus a cached call at the same levels).
Quality: MSE of the mean against a one-shot 1024-spp reference with another seed, noisy (the preview) and denoised (default
parameters), after k = 4, 16, 64, 256 samples of one progressive frame; the spp at which the noisy preview first reaches the
denoised 16-spp MSE, with the device time (begin + advances) to get there against the time to 16 spp plus one denoise call.
A sweep of sigma_l, sigma_z and levels at 16 spp settles the defaults (DESIGN.md 7.3).  Prints one JSON line with the card's
name, power limit and maximum SM clock; --out also writes it to a file.

    python tools/bench_denoise.py [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200")]
import pysqt

CHECKPOINTS = (2, 4, 8, 12, 16, 24, 32, 48, 64, 96, 128, 192, 256, 384, 512, 768, 1024)
QUALITY_K = (4, 16, 64, 256)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:          # the numbers are still device times; the card is then unknown
        return dict(error=str(e))


def mse(a, ref):
    return float(((a.astype(np.float64) - ref) ** 2).mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    data = os.path.join(ROOT, "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    ctx = pysqt.Context(0)
    ctx.upload(hs)
    W, H = 1920, 1080
    L, SL, SZ = pysqt.DENOISE_LEVELS, pysqt.DENOISE_SIGMA_L, pysqt.DENOISE_SIGMA_Z
    res = dict(config="config2 scene.obj 1920x1080 bounces 8", card=card(), defaults=dict(levels=L, sigma_l=SL, sigma_z=SZ))
    ref_out = ctx.render(cam, pysqt.make_params(W, H, 1024, max_depth=8, seed=12345), want_rgb8=False)
    ref = ref_out["accum"].astype(np.float64) / 1024.0
    res["reference"] = dict(spp=1024, seed=12345, device_ms=round(ref_out["stats"]["device_ms"], 2))

    p = pysqt.make_params(W, H, a.spp, max_depth=8, seed=0)
    cum = ctx.render_begin(cam, p)["device_ms"]
    k, curve, quality = 0, [], {}
    for kc in CHECKPOINTS:
        cum += ctx.render_advance(kc - k)["stats"]["device_ms"]
        k = kc
        noisy = ctx.denoise(0)["mean"]
        curve.append(dict(k=k, device_ms=round(cum, 2), mse_noisy=mse(noisy, ref)))
        if k in QUALITY_K:
            d = ctx.denoise(L, SL, SZ)
            quality[k] = dict(mse_noisy=curve[-1]["mse_noisy"], mse_denoised=mse(d["mean"], ref), device_ms=round(cum, 2),
                              denoise_ms=round(d["stats"]["device_ms"], 3))
        if k == 16:
            # cost per level count, on this 16-spp frame (features already cached by the calls above)
            timing = {}
            for lv in range(1, 9):
                for _ in range(3):
                    ctx.denoise(lv, SL, SZ)
                ms = [ctx.denoise(lv, SL, SZ)["stats"]["device_ms"] for _ in range(a.reps)]
                timing[lv] = dict(median_ms=round(statistics.median(ms), 4), min_ms=round(min(ms), 4), max_ms=round(max(ms), 4))
            res["denoise_device_ms"] = timing
            sweep = []
            for lv in (3, 4, 5, 6):
                for sl in (1.0, 2.0, 4.0, 8.0, 16.0):
                    for sz in (0.01, 0.05, 0.2):
                        sweep.append(dict(levels=lv, sigma_l=sl, sigma_z=sz, mse=mse(ctx.denoise(lv, sl, sz)["mean"], ref)))
            res["sweep_16spp"] = sweep
            res["sweep_best"] = min(sweep, key=lambda r: r["mse"])
    res["quality"] = quality
    res["noisy_curve"] = curve
    target = quality[16]["mse_denoised"]
    hit = next((c for c in curve if c["mse_noisy"] <= target), None)
    res["noisy_reaches_denoised_16spp"] = (dict(k=hit["k"], device_ms=hit["device_ms"]) if hit else
                                           dict(k=None, note="not within %d spp" % a.spp))
    res["denoised_16spp_device_ms"] = round(quality[16]["device_ms"] + quality[16]["denoise_ms"], 2)
    # the features: a new frame's first call against a cached one
    ctx.render_begin(cam, p)
    ctx.render_advance(2)
    first = ctx.denoise(L, SL, SZ)["stats"]
    cached = [ctx.denoise(L, SL, SZ)["stats"]["device_ms"] for _ in range(a.reps)]
    res["features_ms"] = round(first["device_ms"] - statistics.median(cached), 4)
    ctx.close()
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
