"""Many views on several GPUs: three ways to render the same views, in interleaved rounds.

    python tools/view_parallel.py [--rounds 5] [--frames 12] [--devices 1,2,4,8] [--out profiles/r5_view_parallel_b200.json]

Arms, per case and device count D:
  (a) one Engine on device 0, all views through render_cameras (one batched pass schedule; D does not apply);
  (b) a strip group of D devices, the views one after another through render_camera_to (every view cut into D row strips);
  (c) a group of D devices with every view placed "auto" (whole views spread over the devices), all through render_cameras.
Cases: 64 x Cornell 128x128, 16 x Cornell 640x480, 16 x demo_level 640x480, and D x Cornell 1920x1080 (one view per device).  Every view
stores RGBA16F into its own tensor on device 0 (a peer store from the other devices).  A frame is tick + render + a synchronise of every
member; ms per frame is a host clock around `--frames` such frames, median and spread (min, max) over the rounds, the arms alternating
round by round.  D runs over the counts in --devices that the box has.  Needs CUDA devices; records the card's name, power limit and
device count with the numbers.  On a box with one GPU only D = 1 runs, which measures what the group path costs over one Engine.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FMT = 2   # FORMAT_RGBA16F: Bevy's HDR view target


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    lines = q.stdout.strip().splitlines() if q.returncode == 0 else []
    return {"name_power_clock": lines[0] if lines else "unknown", "all": lines}


def poses(scene, k):
    c = scene["camera"]
    out = []
    for j in range(k):
        t = np.array(c["transform"], np.float32).reshape(-1).copy()
        t[12] += 0.05 * math.sin(j); t[13] += 0.03 * math.cos(j)
        out.append(t)
    return out


class Arm:
    """One way of rendering the K views of a case: `frame()` ticks, renders every view into its device-0 tensor and synchronises."""

    def __init__(self, kind, scene, k, devices, targets):
        import strolle_b200
        from strolle_b200 import scenes
        self.kind = kind
        bn = scenes.blue_noise()
        c = scene["camera"]
        w, h = c["w"], c["h"]
        if kind == "a":
            self.e = strolle_b200.Engine(device=0, blue_noise=bn)
        else:
            self.e = strolle_b200.MultiEngine(devices, blue_noise=bn)
        first = scenes.apply(self.e, scene)
        kw = {"rank": "auto"} if kind == "c" else {}
        self.cams = [self.e.create_camera(c["mode"], c["denoise"], c["ref_depth"], w, h, p, c["projection"], **kw) for p in poses(scene, k)]
        if kind == "a":
            self.e._check(self.e.lib.st_delete_camera(self.e._h, first))
        else:
            self.e._check(self.e.lib.st_multi_delete_camera(self.e._h, first))
        n = len(self.cams)
        self.handles = (C.c_int32 * n)(*self.cams)
        self.dsts = (C.c_void_p * n)(*[t.data_ptr() for t in targets])
        self.pitches = (C.c_size_t * n)(*[t.stride(0) * t.element_size() for t in targets])
        self.targets = targets

    def frame(self):
        e, lib = self.e, self.e.lib
        e.tick()
        if self.kind == "a":
            e._check(lib.st_render_cameras(e._h, self.handles, len(self.cams), self.dsts, self.pitches, FMT))
        elif self.kind == "b":
            for i, cam in enumerate(self.cams):
                e._check(lib.st_multi_render_camera_to(e._h, cam, self.dsts[i], self.pitches[i], FMT))
        else:
            e._check(lib.st_multi_render_cameras(e._h, self.handles, len(self.cams), self.dsts, self.pitches, FMT))
        e.synchronize()

    def run(self, n):
        t0 = time.perf_counter()
        for _ in range(n):
            self.frame()
        return (time.perf_counter() - t0) * 1e3 / n

    def close(self):
        self.e.close()


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--devices", default="1,2,4,8")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("view_parallel: no CUDA device")
    from strolle_b200 import scenes
    have = torch.cuda.device_count()
    counts = [d for d in (int(x) for x in args.devices.split(",")) if d <= have]
    result = {"card": card(), "device_count": have, "device_counts_run": counts, "rounds": args.rounds, "frames_per_round": args.frames,
              "format": "RGBA16F into one tensor per view on device 0", "cases": []}
    print(json.dumps(result["card"]), "devices:", have, flush=True)
    cases = [("cornell", scenes.cornell, 128, 128, 64), ("cornell", scenes.cornell, 640, 480, 16), ("demo_level", scenes.demo_level, 640, 480, 16)]
    cases += [("cornell", scenes.cornell, 1920, 1080, None)]   # None: one view per device
    for name, fn, w, h, k in cases:
        for d in counts:
            views = d if k is None else k
            scene = fn(w, h)
            targets = [torch.zeros((h, w, 4), dtype=torch.float16, device="cuda:0") for _ in range(views)]
            devices = list(range(d))
            arms = {"a_one_engine_batched": Arm("a", scene, views, devices, targets),
                    "b_strip_group_sequential": Arm("b", scene, views, devices, targets),
                    "c_view_parallel_auto": Arm("c", scene, views, devices, targets)}
            for arm in arms.values():
                arm.run(args.warmup)
            ms = {a: [] for a in arms}
            for _ in range(args.rounds):
                for a, arm in arms.items():
                    ms[a].append(arm.run(args.frames))
            ranks = [arms["c_view_parallel_auto"].e.camera_rank(c) for c in arms["c_view_parallel_auto"].cams]
            case = {"scene": name, "w": w, "h": h, "views": views, "devices": d, "views_per_device": [ranks.count(r) for r in range(d)],
                    **{a: {"ms_per_frame": stats(v)} for a, v in ms.items()}}
            case["c_over_a"] = case["c_view_parallel_auto"]["ms_per_frame"]["median"] / case["a_one_engine_batched"]["ms_per_frame"]["median"]
            case["c_over_b"] = case["c_view_parallel_auto"]["ms_per_frame"]["median"] / case["b_strip_group_sequential"]["ms_per_frame"]["median"]
            result["cases"].append(case)
            print(json.dumps(case), flush=True)
            for arm in arms.values():
                arm.close()
            del arms, targets
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
