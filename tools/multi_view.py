"""Several views per frame: K cameras rendered one after another (render_camera) against the same K cameras as one batched pass schedule
(render_cameras), on one engine, in interleaved rounds.

    python tools/multi_view.py [--rounds 5] [--frames 12] [--out profiles/multi_view_b200.json]

Cases: K in {1, 4, 16, 64} views of Cornell at 128x128, 320x240 and 640x480 and of demo_level at 640x480, and 4 x 960x540 batched
against 1 x 1920x1080 (the same pixels: what batching itself costs).  Per case and arm: the median and spread (min, max over the rounds)
of device ms per frame (CUDA events around the frames, st_mark_begin / st_mark_end), wall ms per frame (host clock around the same frames,
which end in a synchronise) and launches per frame (pass timing on, six extra frames).  Needs a CUDA device; prints the card's name and
power limit with the numbers.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make(scene_fn, w, h, k):
    import strolle_b200
    from strolle_b200 import scenes
    scene = scene_fn(w, h)
    e = strolle_b200.Engine(blue_noise=scenes.blue_noise())
    first = scenes.apply(e, scene)
    c = scene["camera"]
    cams = [first]
    for j in range(1, k):
        t = np.array(c["transform"], np.float32).reshape(-1).copy()
        t[12] += 0.05 * math.sin(j); t[13] += 0.03 * math.cos(j)
        cams.append(e.create_camera(c["mode"], c["denoise"], c["ref_depth"], w, h, t, c["projection"]))
    return e, cams


def frames(e, cams, batched, n):
    """(device ms, wall ms) per frame over n frames."""
    e.synchronize()
    t0 = time.perf_counter()
    e.mark_begin()
    for _ in range(n):
        e.tick()
        if batched:
            e.render_cameras(cams)
        else:
            for c in cams:
                e.render_camera(c)
    ms = e.mark_end()
    e.synchronize()
    return ms / n, (time.perf_counter() - t0) * 1e3 / n


def launches(e, cams, batched):
    """Launches per frame, averaged over one 6-frame GI cycle (the schedule differs from frame to frame)."""
    e.enable_timing(True)
    e.pass_times(reset=True)
    frames(e, cams, batched, 6)
    n = int(e.pass_times(reset=True)[1].sum())
    e.enable_timing(False)
    return n / 6


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def run_case(arms, rounds, n):
    """arms: {name: (engine, cams, batched)}; rounds alternate the arms."""
    for e, cams, b in arms.values():
        frames(e, cams, b, 3)   # warm-up: module loads, allocations, the first GI cycle
    dev = {a: [] for a in arms}; wall = {a: [] for a in arms}
    for _ in range(rounds):
        for a, (e, cams, b) in arms.items():
            d, w = frames(e, cams, b, n)
            dev[a].append(d); wall[a].append(w)
    return {a: {"device_ms_per_frame": stats(dev[a]), "wall_ms_per_frame": stats(wall[a]), "launches_per_frame": launches(*arms[a])} for a in arms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=12)
    ap.add_argument("--views", default="1,4,16,64")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("multi_view: no CUDA device")
    from strolle_b200 import scenes
    result = {"card": card(), "rounds": args.rounds, "frames_per_round": args.frames, "cases": []}
    print("card:", result["card"], flush=True)
    ks = [int(k) for k in args.views.split(",")]
    for name, fn, w, h in [("cornell", scenes.cornell, 128, 128), ("cornell", scenes.cornell, 320, 240), ("cornell", scenes.cornell, 640, 480),
                           ("demo_level", scenes.demo_level, 640, 480)]:
        for k in ks:
            e, cams = make(fn, w, h, k)
            r = run_case({"sequential": (e, cams, False), "batched": (e, cams, True)}, args.rounds, args.frames)
            case = {"scene": name, "w": w, "h": h, "views": k, **r,
                    "speedup_device": r["sequential"]["device_ms_per_frame"]["median"] / r["batched"]["device_ms_per_frame"]["median"]}
            result["cases"].append(case)
            print(json.dumps(case), flush=True)
            e.close()
    e4, c4 = make(scenes.cornell, 960, 540, 4)
    e1, c1 = make(scenes.cornell, 1920, 1080, 1)
    r = run_case({"4x960x540_batched": (e4, c4, True), "1x1920x1080": (e1, c1, False)}, args.rounds, args.frames)
    case = {"scene": "cornell", "case": "4 x 960x540 batched vs 1 x 1920x1080", **r}
    result["cases"].append(case)
    print(json.dumps(case), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
