"""What adaptive sampling buys on BASELINE config 2 (data/scene.obj, 1920x1080, target 1024 spp, 8 bounces, chunks of 64): a
uniform progressive frame against adaptive frames (sqt_render_retire after every chunk, min_samples 64) at several relative
tolerances, alternating the variants round by round.

Headline: time until a given share of the hit pixels meets the relative-error target of a tolerance (the pixels the retire
test of include/sqt.h passes with abs_tol = 0).  Adaptive run: the time up to the first chunk after which that share has
retired.  Uniform run: the time up to the first chunk after which that share passes the same test, evaluated with numpy on the
downloaded sums and moments.  Times are the begin's and advances' CUDA-event device times (`*_device_ms`); for the adaptive run
`adaptive_with_retire_wall_ms` also adds the WALL time of every retire call, host launch, copies and the stream synchronise
included (the C ABI reports no device time for retire, so this bounds its device time from above).  Per chunk it also reports
active pixels, samples traced, device ms, the global noise estimate and the retire call's wall ms.  Prints one JSON line with
the card's name, power limit and maximum SM clock.

    python tools/bench_adaptive.py [--reps 3] [--tols 0.3,0.2,0.1] [--spp 1024] [--chunk 64] [--min-samples 64]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "squigly-trace_b200")]
import pysqt

SHARES = (0.25, 0.5, 0.75, 0.9)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:          # the numbers are still device times; the card is then unknown
        return dict(error=str(e))


def meets(s1, s2, n, rel):
    """include/sqt.h's retire test with abs_tol = 0, per pixel, in fp64 (NaN never meets)."""
    a = s1.reshape(-1, 3).astype(np.float64)
    q = s2.reshape(-1, 3).astype(np.float64)
    rel = float(np.float32(rel))
    with np.errstate(all="ignore"):
        mu = a / n
        v = np.maximum(0.0, (q - a * mu) / (n - 1))
        e2 = ((v[:, 0] + v[:, 1]) + v[:, 2]) / n
        t = rel * ((mu[:, 0] + mu[:, 1]) + mu[:, 2])
        return e2 < t * t


def first_time(cum_ms, share, want):
    """Cumulative time at the first chunk whose share reaches `want` (None: never)."""
    for t, s in zip(cum_ms, share):
        if s >= want:
            return round(t, 2)
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tols", default="0.3,0.2,0.1")
    ap.add_argument("--spp", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=64)
    ap.add_argument("--min-samples", type=int, default=64)
    a = ap.parse_args()
    tols = [float(t) for t in a.tols.split(",")]
    data = os.path.join(ROOT, "data")
    hs = pysqt.HostScene.load(os.path.join(data, "scene.obj"), data)
    cam = pysqt.load_camera(os.path.join(data, "camera"))
    ctx = pysqt.Context(0)
    ctx.upload(hs)
    W, H = 1920, 1080
    p = pysqt.make_params(W, H, a.spp, max_depth=8, seed=0)

    def uniform(evaluate):
        st = ctx.render_begin(cam, p)
        rows, share = [], {t: [] for t in tols}
        hits = None
        while True:
            pr = ctx.render_advance(a.chunk)
            k = pr["samples_done"]
            hits = hits or pr["stats"]["samples"] // a.chunk
            rows.append(dict(k=k, active=hits, samples=pr["stats"]["samples"], device_ms=round(pr["stats"]["device_ms"], 3),
                             noise=pr["noise"]))
            if evaluate:
                _, s1 = ctx.download(p.rows, p.cols)
                s2 = ctx.download_moments(p.rows, p.cols)
                for t in tols:
                    share[t].append(float(meets(s1, s2, k, t).sum()) / hits if k >= a.min_samples else 0.0)
            if k == a.spp:
                break
        return st["device_ms"], hits, rows, share

    def adaptive(tol):
        st = ctx.render_begin(cam, p)
        rows, hits = [], None
        while True:
            pr = ctx.render_advance(a.chunk)
            k = pr["samples_done"]
            hits = hits or pr["stats"]["samples"] // a.chunk
            t0 = time.perf_counter()
            act = ctx.render_retire(tol, 0.0, a.min_samples)
            rms = (time.perf_counter() - t0) * 1e3
            rows.append(dict(k=k, samples=pr["stats"]["samples"], device_ms=round(pr["stats"]["device_ms"], 3), noise=pr["noise"],
                             active_after_retire=act, retire_wall_ms=round(rms, 3)))
            if k == a.spp:
                break
        return st["device_ms"], hits, rows

    uniform(False)                                    # warm-up: every launch shape once
    for t in tols:
        adaptive(t)
    u_runs, a_runs = [], {t: [] for t in tols}
    share_u = None
    for rep in range(a.reps):
        b, hits, rows, share = uniform(rep == 0)
        u_runs.append((b, rows))
        share_u = share if rep == 0 else share_u
        for t in tols:
            a_runs[t].append(adaptive(t))

    def cum(begin_ms, rows, retire):
        c, out = begin_ms, []
        for r in rows:
            c += r["device_ms"] + (r["retire_wall_ms"] if retire else 0.0)
            out.append(c)
        return out

    u_cum = [statistics.median(x) for x in zip(*[cum(b, rows, False) for b, rows in u_runs])]
    res = dict(workload=dict(scene="data/scene.obj", width=W, height=H, spp=a.spp, max_depth=8, chunk=a.chunk,
                             min_samples=a.min_samples), card=card(), device=ctx.info()["name"], reps=a.reps, hit_pixels=hits,
               uniform=dict(total_device_ms=round(u_cum[-1], 2), per_chunk=u_runs[0][1]), adaptive={})
    for t in tols:
        runs = a_runs[t]
        a_cum = [statistics.median(x) for x in zip(*[cum(b, rows, True) for b, _, rows in runs])]
        a_dev = [statistics.median(x) for x in zip(*[cum(b, rows, False) for b, _, rows in runs])]
        rows = runs[0][2]
        share_a = [(hits - r["active_after_retire"]) / hits for r in rows]
        headline = {}
        for s in SHARES:
            ta, tw, tu = first_time(a_dev, share_a, s), first_time(a_cum, share_a, s), first_time(u_cum, share_u[t], s)
            headline["%d%%" % round(s * 100)] = dict(adaptive_device_ms=ta, adaptive_with_retire_wall_ms=tw, uniform_device_ms=tu,
                                                    speedup_device=round(tu / ta, 3) if ta and tu else None)
        res["adaptive"]["rel_%g" % t] = dict(
            total_device_ms=round(a_dev[-1], 2), total_with_retire_wall_ms=round(a_cum[-1], 2),
            retire_wall_ms_total=round(sum(r["retire_wall_ms"] for r in rows), 2),
            final_share_met=round(share_a[-1], 4), uniform_share_met_at_spp=round(share_u[t][-1], 4),
            time_to_share=headline, per_chunk=rows, uniform_share_per_chunk=[round(x, 4) for x in share_u[t]])
    print(json.dumps(res), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
