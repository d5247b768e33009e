#!/usr/bin/env python
"""Cost of delivering the composed frame, per output target, on Cornell at the product default (fast shading, fused passes).

    python tools/output_targets.py [--width 1920 --height 1080 --frames 300 --rounds 3] [--out FILE]

Modes (every step = update_camera + tick + render, as in bench.py's e2e block):
  none            render only, the frame stays in the engine
  host_rgba8      Rgba8UnormSrgb into two alternating pinned host frames, ST_OPT_ASYNC_OUTPUT (bench.py's e2e line)
  host_rgba16f    the same in Rgba16Float
  device_rgba16f  Rgba16Float into a CUDA tensor (the store kernel writes it directly; no staging, no copy)
  device_rgba16f_view  the same into big[y:y+h, x:x+w] of a larger CUDA surface (viewport offset, padded row pitch)

Per mode: ms_per_frame = device events on the engine stream around `frames` steps that only enqueue (device targets through the raw
st_render_camera_to, so the host never waits inside the loop); fps_e2e = wall clock over `frames` steps through the public
Engine.render_camera (which, for a CUDA tensor, synchronises before returning, and for pinned frames returns once the copy is queued),
ending with a full synchronise; composition_ms = frame_composition pass time per frame (composition + store kernel) from a separate
run with per-pass timing on.  Modes are measured in `rounds` interleaved rounds; the table gives the median and the spread.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

MODES = ["none", "host_rgba8", "host_rgba16f", "device_rgba16f", "device_rgba16f_view"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        return q.strip().splitlines()[0]
    except Exception as exc:   # the measurement still stands; the card line says why it is missing
        return f"nvidia-smi unavailable: {exc}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import strolle_b200
    from strolle_b200 import scenes
    from strolle_b200.engine import FORMAT_RGBA8_SRGB, FORMAT_RGBA16F, OPT_ASYNC_OUTPUT
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures on the GPU only")
    W, H = args.width, args.height
    scene = scenes.cornell(W, H)
    c = scene["camera"]
    e = strolle_b200.Engine()
    cam = scenes.apply(e, scene)
    pinned8 = [torch.zeros((H, W, 4), dtype=torch.uint8, pin_memory=True).numpy() for _ in range(2)]
    pinned16 = [torch.zeros((H, W, 4), dtype=torch.float16, pin_memory=True).numpy() for _ in range(2)]
    dev16 = torch.zeros((H, W, 4), dtype=torch.float16, device="cuda:0")
    big16 = torch.zeros((H + 64, W + 96, 4), dtype=torch.float16, device="cuda:0")
    view16 = big16[32:32 + H, 48:48 + W]
    torch.cuda.synchronize()

    def public(mode, i):   # the public API a caller uses
        if mode == "none":
            e.render_camera(cam)
        elif mode == "host_rgba8":
            e.render_camera(cam, pinned8[i & 1], FORMAT_RGBA8_SRGB)
        elif mode == "host_rgba16f":
            e.render_camera(cam, pinned16[i & 1], FORMAT_RGBA16F)
        elif mode == "device_rgba16f":
            e.render_camera(cam, dev16, FORMAT_RGBA16F)
        else:
            e.render_camera(cam, view16, FORMAT_RGBA16F)

    def enqueue(mode, i):  # the same without a host wait inside the step
        if mode == "device_rgba16f":
            e.render_camera_to(cam, dev16.data_ptr(), 0, FORMAT_RGBA16F)
        elif mode == "device_rgba16f_view":
            e.render_camera_to(cam, view16.data_ptr(), view16.stride(0) * 2, FORMAT_RGBA16F)
        else:
            public(mode, i)

    def steps(mode, n, fn):
        for i in range(n):
            e.update_camera(cam, c["mode"], c["denoise"], c["ref_depth"], W, H, c["transform"], c["projection"])
            e.tick()
            fn(mode, i)

    comp = list(strolle_b200.PASS_NAMES).index("frame_composition")
    results = {m: {"ms_per_frame": [], "fps_e2e": [], "composition_ms": []} for m in MODES}
    e.set_option(OPT_ASYNC_OUTPUT, 1)
    for r in range(args.rounds):
        for mode in MODES:
            steps(mode, args.warmup, public)
            e.synchronize()
            e.mark_begin()
            steps(mode, args.frames, enqueue)
            results[mode]["ms_per_frame"].append(e.mark_end() / args.frames)
            e.synchronize()
            t0 = time.perf_counter()
            steps(mode, args.frames, public)
            e.synchronize()
            results[mode]["fps_e2e"].append(args.frames / (time.perf_counter() - t0))
            e.enable_timing(True); e.pass_times(reset=True)
            steps(mode, 50, enqueue)
            e.synchronize()
            ms, launches = e.pass_times(reset=True)
            e.enable_timing(False)
            results[mode]["composition_ms"].append(float(ms[comp]) / 50)
    mean8 = float(pinned8[0][..., :3].mean())
    summary = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "workload": f"cornell {W}x{H}, product default",
               "frames_per_round": args.frames, "rounds": args.rounds, "frame_mean_rgba8": mean8, "modes": {}}
    lines = [f"# {summary['card']}  ({summary['torch_device']})", f"# {summary['workload']}, {args.frames} frames x {args.rounds} interleaved rounds; median [min, max]",
             f"{'mode':22s} {'ms/frame (events)':>26s} {'frames/s e2e':>26s} {'composition ms/frame':>28s}"]
    for mode in MODES:
        d = {k: (float(np.median(v)), float(min(v)), float(max(v))) for k, v in results[mode].items()}
        summary["modes"][mode] = {k: {"median": a, "min": b, "max": c_} for k, (a, b, c_) in d.items()}
        f = lambda t, p: f"{t[0]:.{p}f} [{t[1]:.{p}f}, {t[2]:.{p}f}]"
        lines.append(f"{mode:22s} {f(d['ms_per_frame'], 4):>26s} {f(d['fps_e2e'], 1):>26s} {f(d['composition_ms'], 4):>28s}")
    text = "\n".join(lines)
    print(text)
    print(json.dumps(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n" + json.dumps(summary) + "\n")


if __name__ == "__main__":
    main()
