#!/usr/bin/env python
"""Run under torchrun on N GPUs: checks that the NCCL strip-partitioned run reproduces the single-GPU frame
bit for bit (rank 0 also renders the full frame on its own; gathered as RGBA32F, RGBA16F and RGBA8), and that the sample-parallel reference mode
reduces to the single-GPU accumulation.  Prints one OK/FAIL line per check on rank 0.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/verify_multigpu.py
"""
import os
import sys

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import strolle_b200
from strolle_b200 import scenes
from strolle_b200.multigpu import ReferenceAccumulator, StripRunner

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
W, H, FRAMES = 640, 360 * world, 9

scene = scenes.cornell(W, H)


def check_strips(native, peer=False):
    eng = strolle_b200.Engine(device=local)
    cam = scenes.apply(eng, scene)
    runner = StripRunner(eng, cam, W, H, rank, world, native=native, peer=peer)
    full = None
    if rank == 0:
        full = strolle_b200.Engine(device=local)
        cfull = scenes.apply(full, scene)
    ok = True
    out = np.zeros((H, W, 4), dtype=np.float32)
    out8 = np.zeros((H, W, 4), dtype=np.uint8)
    want8 = np.zeros((H, W, 4), dtype=np.uint8)
    out16 = np.zeros((H, W, 4), dtype=np.float16)
    want16 = np.zeros((H, W, 4), dtype=np.float16)
    shared16, seg = shared_frame16() if native else (None, None)
    for f in range(FRAMES):
        last = f == FRAMES - 1
        half1 = f == FRAMES - 2              # Rgba16Float, strips assembled on rank 0 (gather 1)
        half2 = native and f == FRAMES - 3   # Rgba16Float, every rank stores its own rows into one shared host frame (gather 2)
        eng.tick()
        if last:
            runner.render(out=out8, fmt=strolle_b200.engine.FORMAT_RGBA8_SRGB, gather=1)
        elif half1:
            runner.render(out=out16, fmt=strolle_b200.engine.FORMAT_RGBA16F, gather=1)
        elif half2:
            runner.render(out=shared16, fmt=strolle_b200.engine.FORMAT_RGBA16F, gather=2)
            dist.barrier()
        else:
            runner.render(out=out, fmt=strolle_b200.engine.FORMAT_RGBA32F, gather=1)
        if rank == 0:
            full.tick()
            if last:
                full.render_camera(cfull, want8, strolle_b200.engine.FORMAT_RGBA8_SRGB)
            elif half1 or half2:
                full.render_camera(cfull, want16, strolle_b200.engine.FORMAT_RGBA16F)
            else:
                full.render_camera(cfull)
            if last:
                same = out8 == want8
            elif half1 or half2:
                got = out16 if half1 else shared16
                same = (got.view(np.uint16) == want16.view(np.uint16)) | (np.isnan(got) & np.isnan(want16))
            else:
                want = full.read_buffer(cfull, "output").reshape(H, W, 4)
                same = (out.view(np.uint32) == want.view(np.uint32)) | (np.isnan(out) & np.isnan(want))
            if not same.all():
                ok = False
                print(f"FAIL strips frame {f + 1}: {int((~same).sum())} words differ", flush=True)
    if rank == 0:
        how = ("peer-memory stores + device barrier (st_render_strips)" if peer else "engine-owned NCCL (st_render_strips)") if native else "torch.distributed P2P between st_render_range calls"
        if peer and eng.peer_errors(cam):
            ok = False
            print(f"FAIL peer barrier time-outs: {eng.peer_errors(cam)}", flush=True)
        print(f"{'OK' if ok else 'FAIL'} strips via {how}: {world} ranks x {W}x{H // world} rows, {FRAMES} frames (last gathered as RGBA8, "
              f"the one before as RGBA16F{', and the one before that as RGBA16F by every rank into a shared host frame' if native else ''}), "
              f"gathered frame bit-identical to single GPU; halo bytes/frame rank0 = {runner.halo_bytes_last_frame}", flush=True)
    dist.barrier()
    if seg is not None and rank == 0:
        seg.unlink()   # the mapping itself goes with the process


def shared_frame16():
    """An Rgba16Float host frame every rank of this node writes its own rows into (POSIX shared memory, created by rank 0)."""
    from multiprocessing import shared_memory
    name = [None]
    if rank == 0:
        seg = shared_memory.SharedMemory(create=True, size=H * W * 8)
        name = [seg.name]
    dist.broadcast_object_list(name, src=0)
    if rank != 0:
        seg = shared_memory.SharedMemory(name=name[0])
    return np.ndarray((H, W, 4), dtype=np.float16, buffer=seg.buf), seg


check_strips(True, peer=True)
check_strips(True)
check_strips(False)

# ---- sample-parallel reference mode ------------------------------------------------------------------
W2, H2, TOTAL = 320, 180, 8 * world
scene2 = scenes.cornell(W2, H2, mode=scenes.MODE_REFERENCE, ref_depth=1)
e2 = strolle_b200.Engine(device=local)
c2 = scenes.apply(e2, scene2)
acc = ReferenceAccumulator(e2, c2, rank, world)
acc.accumulate(TOTAL)
acc.reduce_and_compose()
if rank == 0:
    got = e2.read_buffer(c2, "output").reshape(-1, 4)[:, :3]
    e3 = strolle_b200.Engine(device=local)
    c3 = scenes.apply(e3, scene2)
    for _ in range(TOTAL):
        e3.tick(); e3.render_camera(c3)
    want = e3.read_buffer(c3, "output").reshape(-1, 4)[:, :3]
    err = float(np.sqrt(((got - want) ** 2).sum() / (want ** 2).sum()))
    print(f"{'OK' if err < 1e-6 else 'FAIL'} reference mode: {TOTAL} accumulations over {world} ranks + NCCL reduce, rel L2 vs single GPU = {err:.2e}", flush=True)
dist.barrier()
dist.destroy_process_group()
