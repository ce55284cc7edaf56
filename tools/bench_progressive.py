"""Cost of rendering a frame progressively: BASELINE config 2 (data/scene.obj, 1920x1080, 1024 spp, 8 bounces) one-shot
(sqt_render_resident) against sqt_render_begin + sqt_render_advance in chunks of 16, 64 and 256 spp, alternating the variants
round by round.  Device time per frame is the sum of the calls' CUDA-event times; wall time includes the host's
synchronisation per chunk.  Prints one JSON line with the card's name and power limit, per-variant medians and the ratio to
one-shot, and the frame hash of every variant (all must be equal).

    python tools/bench_progressive.py [--reps 3] [--chunks 16,64,256] [--spp 1024]
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200")]
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
    ap.add_argument("--chunks", default="16,64,256")
    ap.add_argument("--spp", type=int, default=1024)
    a = ap.parse_args()
    data = os.path.join(ROOT, "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    ctx = pysqt.Context(0)
    ctx.upload(hs)
    W, H = 1920, 1080
    p = pysqt.make_params(W, H, a.spp, max_depth=8, seed=0)
    chunks = [int(c) for c in a.chunks.split(",")]

    def one_shot():
        t0 = time.perf_counter()
        st = ctx.render_resident(cam, p)
        return st["device_ms"], (time.perf_counter() - t0) * 1e3, st["kernel_launches"]

    def progressive(n):
        t0 = time.perf_counter()
        st = ctx.render_begin(cam, p)
        dev, nl = st["device_ms"], st["kernel_launches"]
        done = 0
        while done < a.spp:
            pr = ctx.render_advance(n)
            done = pr["samples_done"]
            dev += pr["stats"]["device_ms"]; nl += pr["stats"]["kernel_launches"]
        return dev, (time.perf_counter() - t0) * 1e3, nl

    variants = [("one_shot", one_shot)] + [("chunk_%d" % n, (lambda n=n: progressive(n))) for n in chunks]
    res = {name: dict(device_ms=[], wall_ms=[]) for name, _ in variants}
    for name, f in variants:                      # warm-up: every launch shape once
        _, _, res[name]["launches"] = f()
        res[name]["sha256"] = hashlib.sha256(ctx.download(H, W, want_accum=False)[0].tobytes()).hexdigest()
    for _ in range(a.reps):
        for name, f in variants:
            d, w, _ = f()
            res[name]["device_ms"].append(round(d, 2)); res[name]["wall_ms"].append(round(w, 2))
    base = statistics.median(res["one_shot"]["device_ms"])
    for name in res:
        r = res[name]
        r["device_ms_median"] = statistics.median(r["device_ms"])
        r["wall_ms_median"] = statistics.median(r["wall_ms"])
        r["device_ratio_to_one_shot"] = round(r["device_ms_median"] / base, 4)
    out = dict(workload=dict(scene="data/scene.obj", width=W, height=H, spp=a.spp, max_depth=8), card=card(),
               device=ctx.info()["name"], reps=a.reps, same_frame=len({r["sha256"] for r in res.values()}) == 1, variants=res)
    print(json.dumps(out), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
