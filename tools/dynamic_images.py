"""Dynamic images: what refreshing caller-owned surfaces into the atlas costs at each tick, against the alternatives.

    python tools/dynamic_images.py [--rounds 5] [--ticks 200] [--frames 20] [--out profiles/dynamic_images_b200.json]

Refresh cases (sources in device memory): one 1920x1080 image, 45 x 64x64 images (demo_level's texture count), and a mix of 256 images of
seeded sizes.  Per case:
  * tick: device ms per st_tick between CUDA events (st_mark_begin / st_mark_end around --ticks ticks; nothing but the refresh is dirty);
  * kernel: k_atlas_refresh's own duration from torch.profiler (a separate pass), per launch and summed per tick, and launches per tick;
  * memcpy2d: the same rectangles copied by one cudaMemcpy2DAsync per image into an 8192^2 RGBA8 buffer, CUDA events around --ticks rounds;
  * bytes moved (read + written) over time, as a share of the data-sheet 7.7 TB/s HBM3e figure.  Every working set here is smaller than
    the 126 MB L2, so the repeated copies are served from L2: the share is a ratio against the HBM figure, not a claim about HBM traffic.
Today's route: demo_level at 1920x1080 with its 45 textures changing every frame, as ms per frame for tick + render + synchronise, either
re-inserting every texture with insert_image (host bytes, one blocking upload each) or refreshing them as dynamic images; interleaved
rounds, median and spread.  Needs a CUDA device; prints the card's name and power limit with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_TBPS = 7.7
ATLAS = 8192


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def sizes(case):
    if case == "1x1920x1080":
        return [(1920, 1080)]
    if case == "45x64x64":
        return [(64, 64)] * 45
    rng = np.random.RandomState(256)
    return [(int(rng.randint(4, 300)), int(rng.randint(4, 300))) for _ in range(256)]


def shelf(whs):
    """The engine's shelf allocator (st_insert_image), for the memcpy arm's rectangles."""
    x = y = row = 0
    out = []
    for w, h in whs:
        if x + w > ATLAS:
            x, y, row = 0, y + row, 0
        out.append((x, y))
        x, row = x + w, max(row, h)
    return out


def refresh_case(case, ticks, rounds):
    import torch
    import strolle_b200
    from strolle_b200 import scenes
    whs = sizes(case)
    e = strolle_b200.Engine(blue_noise=scenes.blue_noise())
    scenes.apply(e, scenes.cornell(64, 64))
    g = torch.Generator(device="cuda").manual_seed(1)
    srcs = [torch.randint(0, 256, (h, w, 4), dtype=torch.uint8, device="cuda", generator=g) for w, h in whs]
    for k, s in enumerate(srcs):
        e.insert_dynamic_image(1000 + k, s)
    tick = lambda: e._check(e.lib.st_tick(e._h))   # no torch stream synchronise per tick: the sources do not change here
    for _ in range(20):
        tick()
    e.synchronize()
    tick_ms = []
    for _ in range(rounds):
        e.mark_begin()
        for _ in range(ticks):
            tick()
        tick_ms.append(e.mark_end() / ticks)
    # bytes check: the refresh really copied the sources
    assert all((torch.from_numpy(e.read_image(1000 + k)) == s.cpu()).all() for k, s in enumerate(srcs[:8]))
    # kernel duration from the profiler, in a pass of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(ticks):
            tick()
        e.synchronize()
    ev = [x for x in prof.events() if "atlas_refresh" in x.name]
    kernel_us = [x.device_time for x in ev] if ev and hasattr(ev[0], "device_time") else [x.cuda_time for x in ev]
    launches_per_tick = len(ev) / ticks
    # per-image cudaMemcpy2DAsync of the same rectangles
    rt = C.CDLL("libcudart.so.12")
    rt.cudaMemcpy2DAsync.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p]
    atlas = torch.empty((ATLAS, ATLAS, 4), dtype=torch.uint8, device="cuda")
    at = shelf(whs)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)

    def memcpy_round():
        for (w, h), (x, y), s in zip(whs, at, srcs):
            rc = rt.cudaMemcpy2DAsync(atlas.data_ptr() + 4 * (y * ATLAS + x), ATLAS * 4, s.data_ptr(), w * 4, w * 4, h, 3, sp)
            assert rc == 0, rc
    for _ in range(20):
        memcpy_round()
    torch.cuda.synchronize()
    memcpy_ms = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(ticks):
            memcpy_round()
        b.record(stream)
        b.synchronize()
        memcpy_ms.append(a.elapsed_time(b) / ticks)
    for (w, h), (x, y), s in zip(whs, at, srcs):
        assert (atlas[y:y + h, x:x + w] == s).all()
    nbytes = 2 * sum(4 * w * h for w, h in whs)
    floor_ms = nbytes / (HBM_TBPS * 1e12) * 1e3

    def stat(v):
        v = sorted(v)
        return {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}
    kernel_ms = [u / 1e3 for u in kernel_us]
    kernel_tick_ms = sum(kernel_ms) / ticks if kernel_ms else None   # all launches of a tick
    out = {"case": case, "images": len(whs), "bytes_moved_per_tick": nbytes, "hbm_floor_ms": floor_ms,
           "tick_ms": stat(tick_ms), "kernel_ms_per_launch": stat(kernel_ms) if kernel_ms else "not measured",
           "kernel_ms_per_tick": kernel_tick_ms if kernel_ms else "not measured", "kernel_launches_per_tick": launches_per_tick,
           "memcpy2d_ms": stat(memcpy_ms), "memcpy2d_calls_per_tick": len(whs)}
    out["share_of_hbm_tick"] = floor_ms / out["tick_ms"]["median"]
    out["share_of_hbm_kernel"] = floor_ms / kernel_tick_ms if kernel_ms else "not measured"
    out["share_of_hbm_memcpy2d"] = floor_ms / out["memcpy2d_ms"]["median"]
    e.close()
    return out


def todays_route(frames, rounds):
    """demo_level at 1920x1080, 45 textures changing every frame: Raw re-insert per texture vs dynamic images."""
    import torch
    import strolle_b200
    from strolle_b200 import scenes
    scene = scenes.demo_level(1920, 1080)
    handles = sorted(scene["images"])
    arms = {}
    for arm in ("raw", "dynamic"):
        e = strolle_b200.Engine(blue_noise=scenes.blue_noise())
        cam = scenes.apply(e, scene)
        src = {h: torch.from_numpy(np.ascontiguousarray(scene["images"][h])).to("cuda") for h in handles}
        host = {h: np.ascontiguousarray(scene["images"][h]) for h in handles}
        if arm == "dynamic":
            for h, t in src.items():
                e.insert_dynamic_image(h, t)
        arms[arm] = (e, cam, src, host)

    def frame(arm, f):
        e, cam, src, host = arms[arm]
        if arm == "raw":
            for h in handles:
                host[h][0, 0, 0] = f & 255   # the texture changed
                e.insert_image(h, host[h])
        else:
            for h in handles:
                src[h][0, 0, 0] = f & 255
        e.tick()
        e.render_camera(cam)
        e.synchronize()

    for arm in arms:
        for f in range(5):
            frame(arm, f)
    wall = {a: [] for a in arms}
    dev = {a: [] for a in arms}
    for _ in range(rounds):
        for arm in arms:
            e = arms[arm][0]
            t0 = time.perf_counter()
            e.mark_begin()
            for f in range(frames):
                frame(arm, f)
            dev[arm].append(e.mark_end() / frames)
            wall[arm].append((time.perf_counter() - t0) * 1e3 / frames)
    res = {}
    for arm in arms:
        w, d = sorted(wall[arm]), sorted(dev[arm])
        res[arm] = {"wall_ms_per_frame": {"median": w[len(w) // 2], "min": w[0], "max": w[-1]},
                    "device_ms_per_frame": {"median": d[len(d) // 2], "min": d[0], "max": d[-1]}}
    for e, *_ in arms.values():
        e.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(), "hbm_tbps_datasheet": HBM_TBPS, "rounds": a.rounds, "ticks": a.ticks, "frames": a.frames,
           "refresh": [refresh_case(c, a.ticks, a.rounds) for c in ("1x1920x1080", "45x64x64", "mix256")],
           "demo_level_1920x1080": todays_route(a.frames, a.rounds), "card_after": card()}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
