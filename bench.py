#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native Strolle hot path.

    python bench.py --gpus N --steps K --warmup W            # CUDA path (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (oracle port, all host threads)

A "step" is one frame of the hot path (primary-visibility G-buffer + ReSTIR DI/GI + SVGF + composition).  The main line is
BASELINE.json's configs[1]: Cornell Box 1920x1080, ReSTIR DI+GI + SVGF, static camera (weak scaling for N > 1: the same 16:9
picture with N x the pixels, one ~1080p row strip per GPU).  ONE JSON line on rank 0:

  value      Mrays/s from device time (CUDA events on the engine's stream, max over ranks) over exactly K frames, inputs resident in
             HBM; rays = executed Ray::trace / Ray::intersect calls counted on the device over the SAME frame ids.
  e2e        the same through the reference-facing C ABI with HOST buffers: every step uploads the camera struct, ticks, renders and
             delivers the composed Rgba8UnormSrgb frame into a pinned host frame (every rank copies its own rows into one shared
             host frame); wall clock over K steps incl. the copies.
  roofline   dominant kernel (SVGF à-trous, K22): algorithmic bytes (80 B/px per launch) / mean launch time from CUDA events in the run.
  cpu_baseline  the CPU restatement of the reference (oracle/, OpenMP) on a bounded sample of the same workload.
  c4 / c3 / c5 / small   BASELINE.json's other configurations at this N: c4 = Cornell 3840x2160 FIXED size (strong scaling: its ms at N=1
             over its ms at N is the strip-parallel speed-up), c3 = the reference's dungeon with atmosphere, c5 = Reference{depth:1}
             1024 spp sample-parallel + reduce, small = 640x480 (the size the reference's demo renders; launch-bound).
  strip_parity_ok  (N > 1) the gathered strip-parallel frame is bit-identical to a single-GPU render of the same frame on rank 0.

--dump-outputs DIR writes the composed RGBA32F frame of the last timed step as DIR/output.npy (above 64 MB a fixed seeded sample of its
pixels, with their indices in DIR/output_pixels.npy), so that two builds run with the same arguments (same scene, seeds and frame ids)
can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # one hardware queue per stream (strolle_b200/__init__.py); must precede CUDA initialisation

CPU_THREADS = 1
METRIC = "Mrays/s (+ frames/s) at 1080p-per-GPU Cornell, ReSTIR DI+GI + SVGF; B200 vs CPU restatement of the reference"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=60)
    p.add_argument("--warmup", type=int, default=12)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--scene", default="cornell", choices=["cornell", "dungeon"])
    p.add_argument("--width", type=int, default=1920)
    p.add_argument("--height", type=int, default=1080)
    p.add_argument("--cpu-sample-frames", type=int, default=12)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-extras", action="store_true", help="skip the c3 / c4 / c5 / small blocks")
    p.add_argument("--c5-spp", type=int, default=1024)
    p.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR/*.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64 << 20


def dump_frame(rows, y0, w, h, dist=None):
    """--dump-outputs: the composed RGBA32F frame (h, w, 4) of the last timed step, assembled on rank 0 from every rank's `rows`
    (its strip, starting at row y0).  Whole when it fits in DUMP_BYTES; otherwise the same seeded sample of pixels in every run:
    "output" (n, 4) and "output_pixels", their row-major pixel indices (float64, exact)."""
    import numpy as np
    idx = None
    part = rows
    if h * w * 16 > DUMP_BYTES:
        idx = np.sort(np.random.RandomState(0).choice(h * w, DUMP_BYTES // 32, replace=False))   # 16 B of colour + 8 B of index per pixel
        lo, hi = y0 * w, (y0 + len(rows)) * w
        part = rows.reshape(-1, 4)[idx[(idx >= lo) & (idx < hi)] - lo]
    if dist:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, part)
        part = np.concatenate(parts)
    out = {"output": part}
    if idx is not None:
        out["output_pixels"] = idx.astype(np.float64)
    return out


def write_dump(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler:
    """Samples SM clocks + throttle reasons with nvidia-smi during the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def frame_size(args):
    """Weak scaling (SURVEY §8e): every GPU owns a row strip of ~1920x1080 pixels of ONE 16:9 frame, so the picture
    (and with it the rays per pixel) is the same at every N: N=1 1920x1080 (configs[1]), N=2 2720x1528,
    N=4 3840x2160 (configs[3]'s 4K frame), N=8 5440x3056.  Other N: the 16:9 frame with N x the pixels, width
    rounded to 16 and height to 8*N."""
    n = max(args.gpus, 1)
    if n == 1:
        return args.width, args.height
    table = {2: (2720, 1528), 4: (3840, 2160), 8: (5440, 3056)}
    if (args.width, args.height) == (1920, 1080) and n in table:
        return table[n]
    scale = n ** 0.5
    w = int(round(args.width * scale / 16.0)) * 16
    h = int(round(args.height * scale / (8.0 * n))) * 8 * n
    return w, h


SCENE_LABEL = {"cornell": "Cornell Box", "dungeon": "dungeon demo level (bevy-strolle/assets/demo.zip: 13,001 triangles, 45 textures, 6 lights + sun / atmosphere)"}


def build_scene(name, w, h, **kw):
    from strolle_b200 import scenes
    return scenes.cornell(w, h, **kw) if name == "cornell" else scenes.demo_level(w, h, **kw)


def workload_name(args):
    w, h = frame_size(args)
    return f"{SCENE_LABEL[args.scene]} {w}x{h}, ReSTIR DI+GI + SVGF (Image{{denoise:true}}), static camera"


def run_cpu(args, frames, warm=0, dump=None):
    """Times the CPU restatement (oracle/) on all host cores: `frames` full frames of the workload; `dump`: --dump-outputs DIR."""
    from oracle import pyoracle
    from strolle_b200 import scenes
    global CPU_THREADS
    CPU_THREADS = pyoracle.set_threads()
    e = pyoracle.OracleEngine(blue_noise=scenes.blue_noise())
    w, h = frame_size(args)
    cam = scenes.apply(e, build_scene(args.scene, w, h))
    for _ in range(warm):
        e.tick(); e.render_camera(cam)
    pyoracle.ray_count(reset=True)
    t0 = time.perf_counter()
    for _ in range(frames):
        e.tick(); e.render_camera(cam)
    dt = time.perf_counter() - t0
    rays = pyoracle.ray_count(reset=True)
    if dump:
        write_dump(dump, dump_frame(e.read_buffer(cam, "output").reshape(h, w, 4), 0, w, h))
    return frames / dt, dt, rays


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Rust/wgpu reference cannot be
    built here (no cargo, no Vulkan ICD), so this arm is the oracle port (kind "port") on all host threads, on the
    SAME configuration as the CUDA arm at this N (whole frames)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fps, dt, rays = run_cpu(args, args.steps, warm=args.warmup, dump=args.dump_outputs)
    mrays = rays / dt / 1e6
    w, h = frame_size(args)
    cores = CPU_THREADS
    line = {
        "impl": "reference", "metric": METRIC, "value": mrays, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args)}, "fps": fps, "rays_per_frame": rays / args.steps,
        "cpu_baseline": {"value": mrays, "unit": "Mrays/s", "cores": cores, "kind": "port",
                         "sample": f"each step = one full {w}x{h} frame of the same scene/pipeline, {args.steps} steps after {args.warmup} warm-up frames; "
                                   f"oracle/ (C++ restatement of the reference; the Rust/wgpu original cannot be built here) with OpenMP over rows on {cores} threads"},
        "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


class Ctx:
    """Rank / world plumbing shared by the measured configurations."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the CUDA path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self._shm = []

    def barrier(self, *engines):
        for e in engines:
            e.synchronize()
        self.torch.cuda.synchronize()
        if self.dist:
            self.dist.barrier()

    def reduce(self, values, op="max"):
        t = self.torch.tensor(values, dtype=self.torch.float64, device="cuda")
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(x) for x in t]

    def host_frame(self, h, w, slots=2):
        """`slots` pinned RGBA8 host frames that every rank of this node can write its rows into (one buffer per slot, shared
        between the processes through POSIX shared memory and page-locked in each of them)."""
        import numpy as np
        torch = self.torch
        nbytes = h * w * 4
        if self.world == 1:
            bufs = [torch.empty((h, w, 4), dtype=torch.uint8, pin_memory=True) for _ in range(slots)]
            self._shm.append(bufs)
            return [b.numpy() for b in bufs]
        from multiprocessing import shared_memory
        names = [None] * slots
        segs = []
        if self.rank == 0:
            segs = [shared_memory.SharedMemory(create=True, size=nbytes) for _ in range(slots)]
            names = [s.name for s in segs]
        self.dist.broadcast_object_list(names, src=0)
        if self.rank != 0:
            segs = [shared_memory.SharedMemory(name=n) for n in names]
        views = []
        for s in segs:
            a = np.ndarray((h, w, 4), dtype=np.uint8, buffer=s.buf)
            rc = torch.cuda.cudart().cudaHostRegister(a.ctypes.data, nbytes, 0)
            views.append(a)
        self._shm.append((segs, views))
        self.dist.barrier()
        return views

    def close(self):
        for item in self._shm:
            if isinstance(item, tuple):
                segs, views = item
                for a in views:
                    try:
                        self.torch.cuda.cudart().cudaHostUnregister(a.ctypes.data)
                    except Exception:
                        pass
                del views
                for s in segs:
                    try:
                        s.close()
                        if self.rank == 0:
                            s.unlink()
                    except Exception:
                        pass
        if self.dist:
            self.dist.destroy_process_group()


def measure(ctx, scene, steps, warmup, detail=False, e2e=False, clocks=None, dump=False):
    """One configuration: `warmup` untimed frames, then `steps` frames timed with CUDA events (max over ranks); optionally the
    instrumented replay (per-pass events + ray counter over the same frame ids), the strict-arithmetic timing and the end-to-end region.
    `dump`: out["dump"] = dump_frame of the last timed frame (complete on rank 0)."""
    import numpy as np
    import strolle_b200
    from strolle_b200 import scenes
    from strolle_b200.engine import OPT_SVGF_FAST_MATH, OPT_SHADING_FAST_MATH, OPT_FUSED_PASSES, OPT_ASYNC_OUTPUT, FORMAT_RGBA8_SRGB
    from strolle_b200.multigpu import StripRunner
    c = scene["camera"]
    W, H = c["w"], c["h"]
    eng = strolle_b200.Engine(device=ctx.local)
    cam = scenes.apply(eng, scene)
    runner = StripRunner(eng, cam, W, H, ctx.rank, ctx.world)
    for _ in range(max(warmup, 3)):
        eng.tick(); runner.render()
    ctx.barrier(eng)
    if clocks is not None and ctx.rank == 0:
        clocks.start()
    ctx.barrier(eng)
    first_frame = eng.frame()
    t0 = time.perf_counter()
    eng.mark_begin()
    for _ in range(steps):
        eng.tick(); runner.render()
    dev_ms = eng.mark_end()
    ctx.barrier(eng)
    wall_ms = (time.perf_counter() - t0) * 1000.0
    # read before the replay below renders over the last timed frame
    dumped = dump_frame(eng.read_buffer(cam, "output").reshape(H, W, 4)[runner.y0:runner.y1], runner.y0, W, H, ctx.dist) if dump else None
    # the ray counter and per-pass events over a replay of exactly the same frame ids
    eng.enable_timing(True); eng.pass_times(reset=True); eng.wavelet_times(reset=True)
    eng.count_rays(True); eng.ray_count(reset=True)
    eng.set_frame(first_frame)
    ctx.barrier(eng)
    for _ in range(steps):
        eng.tick(); runner.render()
    ctx.barrier(eng)
    pass_ms, launches = eng.pass_times(reset=True)
    wav_ms, wav_launches = eng.wavelet_times(reset=True)
    rays = eng.ray_count(reset=True)
    eng.enable_timing(False); eng.count_rays(False)
    per_rank = None
    if ctx.dist:   # every rank's own per-pass times: shows how much of the exchange time is waiting for a slower neighbour (content imbalance between strips)
        mine = {"compute_ms_per_frame": float(pass_ms.sum() - pass_ms[26]) / steps, "halo_exchange_ms_per_frame": float(pass_ms[26]) / steps}
        per_rank = [None] * ctx.world
        ctx.dist.all_gather_object(per_rank, mine)
    dev_ms, wall_ms = ctx.reduce([dev_ms, wall_ms], "max")
    rays, total_launches = ctx.reduce([float(rays), float(launches.sum())], "sum")
    out = {"w": W, "h": H, "rows": runner.y1 - runner.y0, "ms_per_step": dev_ms / steps, "fps": 1000.0 * steps / dev_ms, "wall_ms_per_step": wall_ms / steps,
           "rays_per_frame": rays / steps, "mrays": rays / (dev_ms / 1000.0) / 1e6, "launches": int(total_launches), "pass_ms": pass_ms, "pass_launches": launches,
           "wav_ms": wav_ms, "wav_launches": wav_launches, "halo_bytes": runner.halo_bytes_last_frame, "transport": runner.transport_name(), "per_rank": per_rank, "dump": dumped}
    if detail:   # every kernel strict IEEE, one launch per reference dispatch: the configuration that is bit-identical to the oracle
        for opt in (OPT_SVGF_FAST_MATH, OPT_SHADING_FAST_MATH, OPT_FUSED_PASSES):
            eng.set_option(opt, 0)
        for _ in range(2):
            eng.tick(); runner.render()
        ctx.barrier(eng)
        eng.mark_begin()
        for _ in range(steps):
            eng.tick(); runner.render()
        out["exact_ms_per_step"] = ctx.reduce([eng.mark_end()], "max")[0] / steps
        for opt in (OPT_SVGF_FAST_MATH, OPT_SHADING_FAST_MATH, OPT_FUSED_PASSES):
            eng.set_option(opt, 1)
        for _ in range(2):
            eng.tick(); runner.render()
        ctx.barrier(eng)
    if e2e:
        host = ctx.host_frame(H, W, 2)
        eng.set_option(OPT_ASYNC_OUTPUT, 1)

        def step(i):
            eng.update_camera(cam, c["mode"], c["denoise"], c["ref_depth"], W, H, c["transform"], c["projection"])
            eng.tick(); runner.render(out=host[i & 1], fmt=FORMAT_RGBA8_SRGB)
        for i in range(3):
            step(i)
        ctx.barrier(eng)
        t0 = time.perf_counter()
        for i in range(steps):
            step(i)
        ctx.barrier(eng)
        e2e_ms = ctx.reduce([(time.perf_counter() - t0) * 1000.0], "max")[0]
        eng.set_option(OPT_ASYNC_OUTPUT, 0)
        out["e2e_fps"] = steps * 1000.0 / e2e_ms
        out["e2e_frame_mean"] = float(host[(steps - 1) & 1][..., :3].mean()) if ctx.rank == 0 else None
        if ctx.world > 1:
            out["peer_errors"] = eng.peer_errors(cam) if runner.peer else 0
    out["engine"] = eng
    out["cam"] = cam
    return out


def strip_parity(ctx, scene, frames=8):
    """N > 1: fresh strip engines render `frames` frames and deliver the last one into the shared host frame; rank 0 renders the same
    frames on ONE GPU from the same initial state.  True iff the two Rgba8UnormSrgb frames are identical (outside any timed region)."""
    import numpy as np
    import strolle_b200
    from strolle_b200 import scenes
    from strolle_b200.engine import FORMAT_RGBA8_SRGB
    from strolle_b200.multigpu import StripRunner
    c = scene["camera"]
    W, H = c["w"], c["h"]
    eng = strolle_b200.Engine(device=ctx.local)
    cam = scenes.apply(eng, scene)
    runner = StripRunner(eng, cam, W, H, ctx.rank, ctx.world)
    host = ctx.host_frame(H, W, 1)[0]
    for f in range(frames):
        eng.tick(); runner.render(out=host if f == frames - 1 else None, fmt=FORMAT_RGBA8_SRGB)
    ctx.barrier(eng)
    ok = None
    if ctx.rank == 0:
        solo = strolle_b200.Engine(device=ctx.local)
        scam = scenes.apply(solo, scene)
        want = np.zeros((H, W, 4), np.uint8)
        for f in range(frames):
            solo.tick(); solo.render_camera(scam, want if f == frames - 1 else None, FORMAT_RGBA8_SRGB)
        ok = bool((want == host).all()) and int(want[..., :3].max()) > 0
        solo.close()
    errors = eng.peer_errors(cam) if runner.peer else 0
    ctx.barrier(eng)
    eng.close()
    return ok, errors


def c5_reference_mode(ctx, spp):
    """BASELINE config C5: Reference{depth:1}, `spp` accumulations at 1920x1080, sample-parallel (rank g renders accumulations g, g+N, ...)
    and one NCCL reduce of the accumulation buffer to rank 0."""
    import strolle_b200
    from strolle_b200 import scenes
    from strolle_b200.multigpu import ReferenceAccumulator
    scene = scenes.cornell(1920, 1080, mode=scenes.MODE_REFERENCE, ref_depth=1)
    eng = strolle_b200.Engine(device=ctx.local)
    cam = scenes.apply(eng, scene)
    acc = ReferenceAccumulator(eng, cam, ctx.rank, ctx.world)
    acc.accumulate(2 * ctx.world)   # warm-up
    ctx.barrier(eng)
    eng2 = strolle_b200.Engine(device=ctx.local)
    cam2 = scenes.apply(eng2, scene)
    acc2 = ReferenceAccumulator(eng2, cam2, ctx.rank, ctx.world)
    eng2.count_rays(True); eng2.ray_count(reset=True)
    ctx.barrier(eng2)
    t0 = time.perf_counter()
    acc2.accumulate(spp)
    acc2.reduce_and_compose()
    ctx.barrier(eng2)
    sec = ctx.reduce([time.perf_counter() - t0], "max")[0]
    rays = ctx.reduce([float(eng2.ray_count(reset=True))], "sum")[0]
    mean = float(eng2.read_buffer(cam2, "output").reshape(-1, 4)[:, :3].mean()) if ctx.rank == 0 else None
    eng.close(); eng2.close()
    return {"workload": f"Cornell 1920x1080 Reference{{depth:1}}, {spp} accumulations, sample-parallel over {ctx.world} rank(s) + one NCCL reduce (f32 sum of 33 MB)",
            "seconds": sec, "spp_per_s": spp / sec, "mrays_per_s": rays / sec / 1e6, "image_mean": mean}


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
        return
    import numpy as np
    import strolle_b200
    from strolle_b200 import scenes
    from strolle_b200.multigpu import strip_bounds
    ctx = Ctx()
    rank, world = ctx.rank, ctx.world
    W, H = frame_size(args)
    clocks = ClockSampler(ctx.local)
    main_m = measure(ctx, build_scene(args.scene, W, H), args.steps, args.warmup, detail=True, e2e=True, clocks=clocks, dump=bool(args.dump_outputs))
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, main_m.pop("dump"))
    eng = main_m["engine"]
    if world > 1:
        main_m["strip_parity_ok"], perr = strip_parity(ctx, build_scene(args.scene, W, H))
        main_m["peer_errors"] = (main_m.get("peer_errors") or 0) + perr

    # ---- BVH trace on its own (rank 0 engine; the ray-stream entry point) ------------------------------------------------------
    traversal = None
    if rank == 0:
        lo, hi = ((-1.0, 0.0, -1.0), (1.0, 2.0, 3.2)) if args.scene == "cornell" else ((-27.0, 0.1, -35.0), (16.0, 3.0, 30.0))
        rng = np.random.RandomState(5)
        nr = 1 << 20
        rays8 = np.zeros((nr, 8), dtype=np.float32)
        rays8[:, 0:3] = rng.uniform(lo, hi, size=(nr, 3)); dv = rng.normal(size=(nr, 3)); rays8[:, 4:7] = dv / np.linalg.norm(dv, axis=1, keepdims=True)
        rays8[:, 3] = np.float32(3.4028234663852886e38)
        eng.trace_closest(rays8)
        hits, t_ms = eng.trace_closest(rays8, return_ms=True)
        used = float(hits[:, 11].astype(np.float64).mean())
        traversal = {"rays": nr, "kernel_ms": t_ms, "mrays_per_s": nr / (t_ms / 1000.0) / 1e6, "mean_used_memory_bytes_per_ray": used,
                     "requested_GBps": nr * used / (t_ms / 1000.0) / 1e9, "hit_fraction": float((hits[:, 8] < 3e38).mean()),
                     "note": "k_trace_stream_closest on random rays in the scene's bounds; requested bytes = the reference's used_memory estimate "
                             "(ray.rs:141-214): L1/L2 cache traffic, the BVH and triangles are cache resident — not an HBM figure"}
    eng.close()

    # ---- the other BASELINE configurations at this N -----------------------------------------------------------------------------
    extras = {}
    if not args.no_extras:
        k, wu = args.steps, 6
        m = measure(ctx, scenes.cornell(3840, 2160), k, wu)
        extras["c4"] = {"workload": f"Cornell 3840x2160 (fixed size, strong scaling), {world} row strip(s) of {m['rows']} rows", "ms_per_step": m["ms_per_step"], "fps": m["fps"],
                        "mrays_per_s": m["mrays"], "steps": k, "halo_bytes_per_frame_rank0": m["halo_bytes"]}
        m["engine"].close()
        other = "dungeon" if args.scene == "cornell" else "cornell"
        m = measure(ctx, build_scene(other, W, H), k, wu)
        extras["c3" if other == "dungeon" else "c2"] = {"workload": f"{SCENE_LABEL[other]} {W}x{H}, ReSTIR DI+GI + SVGF", "ms_per_step": m["ms_per_step"], "fps": m["fps"],
                                                         "mrays_per_s": m["mrays"], "steps": k}
        m["engine"].close()
        extras["c5"] = c5_reference_mode(ctx, args.c5_spp)
        if world == 1:
            m = measure(ctx, scenes.cornell(640, 480), k, 12)
            extras["small"] = {"workload": "Cornell 640x480 (bevy-strolle/examples/demo.rs:24-25 viewport)", "ms_per_step": m["ms_per_step"], "wall_ms_per_step": m["wall_ms_per_step"],
                               "fps": m["fps"], "launches_per_frame": m["launches"] / k, "steps": k}
            m["engine"].close()

    if rank != 0:
        ctx.close()
        return

    # ---- roofline of the dominant kernel -----------------------------------------------------------------------------------------
    names = list(strolle_b200.PASS_NAMES)
    pass_ms, launches = main_m["pass_ms"], main_m["pass_launches"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    rows = main_m["rows"]
    # algorithmic bytes per pixel (inputs U outputs of the launch, SURVEY §8d; fused launches recomputed, DESIGN.md §4)
    bytes_per_px = {"frame_denoising_wavelet": 80, "frame_denoising_estimate_variance": 112, "frame_denoising_reproject": 192, "prim_gbuffer": 96,
                    "di_temporal_resampling": 176, "di_spatial_resampling_pick": 128, "di_resolving": 128, "gi_temporal_resampling": 336, "gi_preview_resampling": 176,
                    "frame_reprojection": 64, "frame_composition": 112}

    def roof(name):
        i = names.index(name)
        if not launches[i]:
            return None
        dur_s = pass_ms[i] / launches[i] / 1000.0
        alg = bytes_per_px.get(name, 0) * W * rows
        ach = alg / dur_s / 1e9
        return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                "alg_bytes_per_launch": alg, "avg_launch_us": dur_s * 1e6, "peak_source": peak_kind}
    roofline = roof("frame_denoising_wavelet") or {}
    roofline["dominant_by_time"] = names[int(np.argmax(pass_ms))]
    traffic_file = os.path.join(ROOT, "profiles", "wavelet_dram_bytes.json")
    if os.path.exists(traffic_file):
        try:
            roofline["traffic"] = json.load(open(traffic_file)).get("dram_bytes_per_launch")
            roofline["traffic_source"] = "profiles/wavelet_dram_bytes.json (dram__bytes_read+write per launch, mean of the five K22 launches of the committed ncu --set full capture)"
        except Exception:
            pass
    wav_ms, wav_launches = main_m["wav_ms"], main_m["wav_launches"]
    roofline["per_iteration"] = []
    for it in range(5):
        if wav_launches[it]:
            dur_s = float(wav_ms[it]) / int(wav_launches[it]) / 1000.0
            alg = 80 * W * rows
            roofline["per_iteration"].append({"stride": 1 << it, "avg_launch_us": dur_s * 1e6, "achieved": alg / dur_s / 1e9, "frac": alg / dur_s / 1e9 / peak})
    extra_roof = [r for r in (roof(n) for n in ["prim_gbuffer", "frame_denoising_estimate_variance", "frame_denoising_reproject", "di_temporal_resampling", "gi_preview_resampling"]) if r]
    frame_bytes = 2700.0 * W * rows   # whole post-G-buffer frame, SURVEY §8d (~2.7 KB per pixel)
    whole = {"alg_bytes_per_frame": frame_bytes, "achieved": frame_bytes / (main_m["ms_per_step"] / 1000.0) / 1e9, "frac": frame_bytes / (main_m["ms_per_step"] / 1000.0) / 1e9 / peak}

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cfps, cdt, crays = run_cpu(args, args.cpu_sample_frames)
        cpu = {"value": crays / cdt / 1e6, "unit": "Mrays/s", "fps": cfps, "cores": CPU_THREADS, "kind": "port",
               "sample": f"{args.cpu_sample_frames} full-resolution frames of the same workload (frames 1..{args.cpu_sample_frames}), {cdt:.1f} s, oracle/ with OpenMP over rows"}

    e2e_fps = main_m["e2e_fps"]
    line = {
        "metric": METRIC, "value": main_m["mrays"], "unit": "Mrays/s", "fps": main_m["fps"], "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": main_m["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "partition": f"{world} row strip(s) of {W} px x {[y1 - y0 for y0, y1 in strip_bounds(H, world)]} rows (outer strips, with one neighbour, are taller than inner ones from 3 ranks on)", "transport": main_m["transport"], "ranks": world,
                   "l2": "per-frame working set (~1.8 GB of per-camera buffers per 1080p strip) exceeds the 126 MB L2; no explicit flush", "seed_base": "0xC0FFEE",
                   "timing": "value: CUDA events around K frames on the engine stream, max over ranks; rays and per-pass events from a replay of the same frame ids"},
        "exact_ms_per_step": main_m.get("exact_ms_per_step"),
        "arithmetic": "product default: ReSTIR shading (K5-K19) and SVGF weights with FMA + SFU approximations inside north_star's 1e-3 tolerance, fused launches; traversal / primary pass / "
                      "reprojection strict IEEE.  exact_ms_per_step = every kernel strict IEEE, one launch per reference dispatch, bit-identical to the oracle",
        "rays_per_frame": main_m["rays_per_frame"], "wall_ms_per_step": main_m["wall_ms_per_step"], "halo_bytes_per_frame_rank0": main_m["halo_bytes"],
        "strip_parity_ok": main_m.get("strip_parity_ok"), "peer_errors": main_m.get("peer_errors"), "per_rank": main_m.get("per_rank"),
        "clocks": clk,
        "e2e": {"value": main_m["rays_per_frame"] * e2e_fps / 1e6, "unit": "Mrays/s", "fps": e2e_fps, "h2d_bytes_per_step": 148 * world, "d2h_bytes_per_step": W * H * 4,
                "note": "per step: st_update_camera (148 B host camera struct per rank) + st_tick + st_render_strips(host frame, gather 2): every rank converts its own rows to Rgba8UnormSrgb and "
                        "copies them into ONE pinned host frame (two frames alternate, async D2H on a copy stream); wall clock over K steps incl. all copies, ends with a full sync"},
        "gpu_launches": main_m["launches"],
        "roofline": roofline, "roofline_other": extra_roof, "roofline_frame": whole, "traversal": traversal,
        "cpu_baseline": cpu,
        "pass_ms_per_frame": {names[i]: float(pass_ms[i]) / args.steps for i in range(len(names)) if launches[i]},
    }
    line.update(extras)
    print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
