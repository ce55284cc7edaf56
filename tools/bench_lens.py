"""What camera sampling costs on BASELINE config 2 (data/scene.obj, data/camera, 1920x1080, 8 bounces, 256 spp).

Three frames, alternated for --reps repetitions: pinhole (primary reuse), jitter (anti-aliasing) and jitter + a thin lens of
aperture 0.05 focused at the centre pixel's primary-hit t.  Per frame: CUDA-event device time (stats.device_ms), rays traced,
rays per sample, Mrays/s and the SHA-256 of the RGB8 frame.  Prints one JSON line with the card's name, power limit and
maximum SM clock read in the same run; --out also writes it to a file.

    python tools/bench_lens.py [--reps 3] [--out FILE]
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200")]
import numpy as np

import pysqt


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:          # the numbers are still device times; the card is then unknown
        return dict(error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--spp", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    data = os.path.join(ROOT, "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    ctx = pysqt.Context(0)
    ctx.upload(hs)
    W, H = 1920, 1080
    p = pysqt.make_params(W, H, a.spp, max_depth=8, seed=0, literal=False)
    # focus: the primary-hit t of the centre pixel (the camera ray is not normalised, so t is the lens' focus parameter)
    o = np.float32(cam[:3])
    R = np.float32(cam[3:]).reshape(3, 3)
    xo, yo = np.float32((W // 2 - W / 2) / W), np.float32((H / 2 - H // 2) / H)
    d = np.float32(1) * R[0] + xo * R[1] + yo * R[2]
    tri, dist, _ = ctx.intersect_batch(o[None], d[None])
    focus = float(dist[0] / np.linalg.norm(d.astype(np.float64))) if tri[0] >= 0 else 3.0
    frames = {"pinhole": None, "jitter": (True, 0.0, 1.0), "jitter+lens": (True, 0.05, focus)}
    res = dict(config="config2 scene.obj 1920x1080 bounces 8 spp %d" % a.spp, card=card(), focus=focus, frames={})
    ctx.render(cam, p, want_accum=False)                         # warm-up: modules, allocations
    runs = {k: [] for k in frames}
    for _ in range(a.reps):
        for name, lens in frames.items():
            ctx.set_lens(*lens) if lens else ctx.set_lens(None)
            out = ctx.render(cam, p, want_accum=False)
            st = out["stats"]
            runs[name].append(dict(device_ms=st["device_ms"], rays_traced=st["rays_traced"], samples=st["samples"],
                                   mrays_s=st["rays_traced"] / (st["device_ms"] * 1e3),
                                   sha256=hashlib.sha256(out["rgb8"].tobytes()).hexdigest()))
    ctx.set_lens(None)
    for name, rs in runs.items():
        res["frames"][name] = dict(
            device_ms=[r["device_ms"] for r in rs], device_ms_median=statistics.median(r["device_ms"] for r in rs),
            rays_traced=rs[0]["rays_traced"], rays_per_sample=rs[0]["rays_traced"] / rs[0]["samples"],
            mrays_s_median=statistics.median(r["mrays_s"] for r in rs), sha256=sorted({r["sha256"] for r in rs}))
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
