"""Dynamic images (st_insert_dynamic_image / Engine.insert_dynamic_image): caller-owned surfaces copied into the atlas at every tick.

The reference for the rendering comparisons is a twin engine with the same scene and seeds that re-uploads the same bytes with
`insert_image` before each tick (today's route for a changing texture).  Every comparison is bit for bit (NaN == NaN).
"""
import ctypes as C

import numpy as np
import pytest

from strolle_b200 import scenes
from tests.util import CAMERA_BUFFERS, assert_bits_equal

pytestmark = pytest.mark.gpu

MONITOR_IMAGE, MONITOR_MAT, MONITOR_MESH, MONITOR_INST = 790, 190, 290, 390


@pytest.fixture(scope="module")
def gpu():
    import strolle_b200
    return strolle_b200


def _torch():
    import torch
    return torch


def _rand(shape, seed, **kw):
    torch = _torch()
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, generator=g).to(**kw) if kw else torch.randint(0, 256, shape, dtype=torch.uint8, generator=g)


def _np(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)


def _assert_bytes(got, want, what):
    got, want = np.asarray(got), _np(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    bad = got != want
    assert not bad.any(), f"{what}: {int(bad.sum())} bytes differ"


# ---- 1. the refreshed bytes ----------------------------------------------------------------------------------------------------------

def test_refresh_bytes(gpu, blue_noise):
    """Dynamic images of widths 1, 3, 61, 64 and 257 from device memory, pinned host memory and padded-pitch slices, between static images:
    after a tick the atlas holds each source's bytes, the static neighbours are untouched; mutated sources show up at the next tick, not
    before."""
    torch = _torch()
    e = gpu.Engine(blue_noise=blue_noise)
    scenes.apply(e, scenes.cornell(32, 24))
    wide_dev = _rand((9, 64, 4), 1, device="cuda")                     # first on the shelf: x = 0, 16-byte rows on both sides
    one_dev = _rand((5, 1, 4), 2, device="cuda")
    three_pin = _rand((7, 3, 4), 3).pin_memory()
    big = _rand((40, 300, 4), 4, device="cuda")
    slice61 = big[3:3 + 33, 5:5 + 61]                                     # padded rows that start 4 bytes past a 16-byte boundary
    pin_big = _rand((12, 280, 4), 5).pin_memory()
    statics = {10: _np(_rand((6, 13, 4), 6)), 11: _np(_rand((4, 2, 4), 7)), 12: _np(_rand((11, 5, 4), 8))}
    order = [(20, wide_dev), (10, None), (21, one_dev), (22, three_pin), (11, None), (23, slice61), (12, None)]
    x = sum(t.shape[1] if t is not None else statics[h].shape[1] for h, t in order)
    # the 257-wide pinned slice starts at the same address modulo 16 as its atlas row (c0 = x mod 4) and has a 1120-byte pitch: the
    # 16-byte path with a ragged head and tail.  The 61-wide slice's rows (4 mod 16) and atlas rows (x = 83: 12 mod 16) disagree: 4-byte path
    c0 = 4 + x % 4
    slice257 = pin_big[1:1 + 10, c0:c0 + 257]
    order.append((24, slice257))
    dyn = {}
    for h, t in order:
        if t is None:
            e.insert_image(h, statics[h])
        else:
            e.insert_dynamic_image(h, t)
            dyn[h] = t
    e.tick()
    for h, t in dyn.items():
        _assert_bytes(e.read_image(h), t, f"image {h} after the first tick")
    for h, a in statics.items():
        _assert_bytes(e.read_image(h), a, f"static image {h}")
    old = {h: _np(t).copy() for h, t in dyn.items()}
    for k, (h, t) in enumerate(dyn.items()):
        t.add_(17 + k)   # wraps modulo 256
    torch.cuda.synchronize()
    for h in dyn:
        _assert_bytes(e.read_image(h), old[h], f"image {h} before the next tick")
    e.tick()
    for h, t in dyn.items():
        _assert_bytes(e.read_image(h), t, f"image {h} after the second tick")
        assert (_np(t) != old[h]).any()
    for h, a in statics.items():
        _assert_bytes(e.read_image(h), a, f"static image {h} after the second tick")


# ---- 2. equivalent to re-uploading ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tier", ["default", "exact", "unfused"])
def test_equivalent_to_reupload_demo_level(gpu, blue_noise, tier):
    """demo_level at 256x144 with five of its 64x64 textures dynamic, mutated by torch every frame for 13 frames: composed frames and every
    camera buffer equal those of a twin that calls insert_image with the same bytes before each tick."""
    from strolle_b200.engine import OPT_FUSED_PASSES
    torch = _torch()
    scene = scenes.demo_level(256, 144)
    es = []
    for _ in range(2):
        e = gpu.Engine(blue_noise=blue_noise, exact=tier == "exact")
        if tier == "unfused":
            e.set_option(OPT_FUSED_PASSES, 0)
        es.append(e)
    dyn, twin = es
    cams = [scenes.apply(e, scene) for e in es]
    used = sorted({t["base_color"] for t in scene["material_textures"].values()})
    src = {h: torch.from_numpy(np.ascontiguousarray(scene["images"][h])).to("cuda") for h in used[::max(1, len(used) // 5)][:5]}
    assert len(src) == 5
    for h, t in src.items():
        dyn.insert_dynamic_image(h, t)
    c = scene["camera"]
    for f in range(13):
        for k, (h, t) in enumerate(src.items()):
            t.mul_(3).add_(f + k)   # torch kernels on the current stream, wrapping modulo 256
            twin.insert_image(h, t.cpu().numpy())
        tf = np.array(c["transform"], np.float32).reshape(-1).copy()
        tf[12] += 0.01 * f
        for e, cam in zip(es, cams):
            e.update_camera(cam, c["mode"], c["denoise"], c["ref_depth"], 256, 144, tf, c["projection"])
            e.tick()
        frames = [np.zeros((144, 256, 4), np.float32) for _ in es]
        for e, cam, out in zip(es, cams, frames):
            e.render_camera(cam, out)
        assert_bits_equal(frames[0], frames[1], f"{tier} frame {f + 1}")
        for name in CAMERA_BUFFERS:
            assert_bits_equal(dyn.read_buffer(cams[0], name), twin.read_buffer(cams[1], name), f"{tier} frame {f + 1} {name}")


# ---- 3. render to texture ---------------------------------------------------------------------------------------------------------------

FEED_W, FEED_H = 48, 32


def _monitor_scene(w, h):
    """Cornell with an emissive "monitor" quad on the back wall, its emissive texture the image MONITOR_IMAGE."""
    s = scenes.cornell(w, h)
    s["meshes"][MONITOR_MESH] = np.stack(scenes._quad((-0.6, 0.7, -0.97), (0.6, 0.7, -0.97), (0.6, 1.5, -0.97), (-0.6, 1.5, -0.97), (0, 0, 1)))
    s["materials"][MONITOR_MAT] = (scenes.material((0.05, 0.05, 0.05, 1.0), emissive=(3.0, 3.0, 3.0, 1.0)), False)
    s["material_textures"] = {MONITOR_MAT: dict(emissive=MONITOR_IMAGE)}
    s["instances"].append((MONITOR_INST, MONITOR_MESH, MONITOR_MAT, scenes.IDENTITY_AFFINE))
    return s


class MonitorLoop:
    """Camera A looks at the room from the side and renders RGBA8 sRGB into the monitor's texture; camera B moves in front of the monitor.
    mode: "seq" renders A then B with render_camera, "ab" / "ba" with one render_cameras call in that order, "raw" is the twin that
    re-inserts A's previous frame as a Raw image before each tick.  feed: "device" (CUDA tensor) or "pinned" (pinned host tensor, written
    by the copy stream under ST_OPT_ASYNC_OUTPUT).  `engine`: an Engine or MultiEngine to use instead of a new Engine."""

    def __init__(self, gpu, blue_noise, mode, feed="device", w=96, h=54, a_size=(FEED_W, FEED_H), engine=None):
        from strolle_b200.engine import OPT_ASYNC_OUTPUT
        torch = _torch()
        self.mode, self.feed_kind, self.w, self.h = mode, feed, w, h
        aw, ah = a_size
        self.scene = _monitor_scene(w, h)
        self.e = engine if engine is not None else gpu.Engine(blue_noise=blue_noise)
        self.b = scenes.apply(self.e, self.scene)
        proj_a = scenes.perspective_infinite_reverse_rh(np.pi / 3.0, aw / ah, 0.1)
        self.a = self.e.create_camera(0, True, 1, aw, ah, scenes.look_at_transform((0.8, 1.2, 1.5), (-0.3, 0.8, -0.5)), proj_a)
        if mode == "raw":
            self.feed = np.zeros((ah, aw, 4), np.uint8)
            self.e.insert_image(MONITOR_IMAGE, self.feed)
            self.out = np.zeros((h, w, 4), np.uint8)
        elif feed == "pinned":
            self.e.set_option(OPT_ASYNC_OUTPUT, 1)
            self.feed = torch.zeros((ah, aw, 4), dtype=torch.uint8).pin_memory()
            self.out = torch.zeros((h, w, 4), dtype=torch.uint8).pin_memory()
            self.e.insert_dynamic_image(MONITOR_IMAGE, self.feed)
        else:
            self.feed = torch.zeros((ah, aw, 4), dtype=torch.uint8, device="cuda")
            self.out = np.zeros((h, w, 4), np.uint8)
            self.e.insert_dynamic_image(MONITOR_IMAGE, self.feed)

    def frame(self, f):
        """Frame f: B's RGBA8 frame, B's composed RGBA32F frame and A's RGBA8 frame (what the monitor shows on frame f + 1)."""
        from strolle_b200.engine import FORMAT_RGBA8_SRGB
        c = self.scene["camera"]
        tf = scenes.look_at_transform((0.3 * np.sin(0.4 * f), 1.0 + 0.05 * f, 3.2 - 0.1 * f), (0.0, 1.0, -0.5))
        self.e.update_camera(self.b, c["mode"], c["denoise"], c["ref_depth"], self.w, self.h, tf, c["projection"])
        if self.mode == "raw":
            self.e.insert_image(MONITOR_IMAGE, self.feed)
        self.e.tick()
        if self.mode in ("ab", "ba"):
            pairs = [(self.a, self.feed), (self.b, self.out)]
            if self.mode == "ba":
                pairs.reverse()
            self.e.render_cameras([p[0] for p in pairs], [p[1] for p in pairs], FORMAT_RGBA8_SRGB)
        else:
            self.e.render_camera(self.a, self.feed, FORMAT_RGBA8_SRGB)
            self.e.render_camera(self.b, self.out, FORMAT_RGBA8_SRGB)
        if self.feed_kind == "pinned":
            self.e.synchronize()   # ST_OPT_ASYNC_OUTPUT: the copies of both frames may still be in flight
        return _np(self.out).copy(), self.e.read_buffer(self.b, "output"), _np(self.feed).copy()


def _run_loops(loops, frames, what):
    for f in range(frames):
        got = [l.frame(f) for l in loops]
        for l, g in zip(loops[1:], got[1:]):
            for k, name in enumerate(["B frame", "B output buffer", "A frame"]):
                if k == 1:
                    assert_bits_equal(g[k], got[0][k], f"{what} {l.mode}/{l.feed_kind} frame {f + 1} {name}")
                else:
                    _assert_bytes(g[k], got[0][k], f"{what} {l.mode}/{l.feed_kind} frame {f + 1} {name}")
    # the monitor shows something: A's frames are not black, and B sees them
    assert got[0][2][..., :3].max() > 0


def test_render_to_texture_loop(gpu, blue_noise):
    """Camera A renders into the monitor's texture; over 8 frames of a moving camera B, the engine with a dynamic image gives the frames of
    the twin that re-inserts A's previous frame before each tick, whether A and B render one after another, or in one render_cameras call in
    either order."""
    loops = [MonitorLoop(gpu, blue_noise, m) for m in ("raw", "seq", "ab", "ba")]
    _run_loops(loops, 8, "render to texture")


def test_render_to_texture_async_pinned(gpu, blue_noise):
    """The same loop with ST_OPT_ASYNC_OUTPUT into a pinned host source: the tick's refresh waits for the copy stream's copy of A's frame."""
    loops = [MonitorLoop(gpu, blue_noise, "raw"), MonitorLoop(gpu, blue_noise, "seq", feed="pinned"), MonitorLoop(gpu, blue_noise, "ab", feed="pinned")]
    _run_loops(loops, 8, "async pinned")


def _devices(n):
    torch = _torch()
    have = max(torch.cuda.device_count(), 1)
    return [k % have for k in range(n)]


def test_strip_group_loop(gpu, blue_noise):
    """A two-member strip group renders the monitor loop itself (each member stores its rows of A's frame into the monitor's surface):
    its frames equal the single-engine run's."""
    size = dict(w=96, h=256, a_size=(64, 256))   # strips of at least 128 rows
    one = MonitorLoop(gpu, blue_noise, "seq", **size)
    grp = MonitorLoop(gpu, blue_noise, "seq", engine=gpu.MultiEngine(_devices(2), blue_noise=blue_noise), **size)
    _run_loops([one, grp], 6, "strip group")
    assert grp.e.peer_errors(grp.a) == 0 and grp.e.peer_errors(grp.b) == 0


# ---- 4. lifecycle ----------------------------------------------------------------------------------------------------------------------

def test_lifecycle(gpu, blue_noise):
    """Same-size re-insert keeps the rectangle; a new size moves it and the material follows (frames equal a twin's Raw re-insert); a Raw
    insert ends the refresh; after remove_image the source can be freed and later ticks run clean."""
    torch = _torch()
    scene = _monitor_scene(64, 40)
    dyn, twin = gpu.Engine(blue_noise=blue_noise), gpu.Engine(blue_noise=blue_noise)
    cd, ct = scenes.apply(dyn, scene), scenes.apply(twin, scene)
    first = _rand((FEED_H, FEED_W, 4), 11, device="cuda")
    dyn.insert_dynamic_image(MONITOR_IMAGE, first)
    twin.insert_image(MONITOR_IMAGE, _np(first))

    def step(what):
        dyn.tick(); twin.tick()
        a, b = np.zeros((40, 64, 4), np.float32), np.zeros((40, 64, 4), np.float32)
        dyn.render_camera(cd, a); twin.render_camera(ct, b)
        assert_bits_equal(a, b, what)
        assert_bits_equal(dyn.read_scene("materials"), twin.read_scene("materials"), what + ": material rectangles")

    step("first")
    mats = dyn.read_scene("materials")
    # same size, another surface: the rectangle stays
    second = _rand((FEED_H, FEED_W, 4), 12, device="cuda")
    dyn.insert_dynamic_image(MONITOR_IMAGE, second)
    del first
    torch.cuda.empty_cache()
    twin.insert_image(MONITOR_IMAGE, _np(second))
    step("same size")
    assert_bits_equal(dyn.read_scene("materials"), mats, "same-size re-insert moved the rectangle")
    # a new size: a new rectangle, and the monitor's material points at it
    third = _rand((20, 30, 4), 13, device="cuda")
    dyn.insert_dynamic_image(MONITOR_IMAGE, third)
    twin.insert_image(MONITOR_IMAGE, _np(third))
    step("new size")
    assert not np.array_equal(dyn.read_scene("materials").view(np.uint32), mats.view(np.uint32)), "the rectangle did not move"
    _assert_bytes(dyn.read_image(MONITOR_IMAGE), third, "new size")
    # Raw on the handle: the old source no longer reaches the atlas
    raw = _np(_rand((20, 30, 4), 14))
    dyn.insert_image(MONITOR_IMAGE, raw)
    twin.insert_image(MONITOR_IMAGE, raw)
    third.add_(1)
    step("raw")
    _assert_bytes(dyn.read_image(MONITOR_IMAGE), raw, "after the Raw insert")
    # dynamic again, then removed: the source is freed and the ticks go on
    fourth = _rand((20, 30, 4), 15).pin_memory()
    dyn.insert_dynamic_image(MONITOR_IMAGE, fourth)
    twin.insert_image(MONITOR_IMAGE, _np(fourth))
    step("pinned")
    dyn.remove_image(MONITOR_IMAGE)
    twin.remove_image(MONITOR_IMAGE)
    del fourth, third, second
    torch.cuda.empty_cache()
    for f in range(3):
        step(f"after remove {f + 1}")
    dyn.synchronize()
    n = C.c_size_t()
    assert dyn.lib.st_read_image(dyn._h, MONITOR_IMAGE, None, 0, C.byref(n)) == -3   # ST_ERR_NOT_FOUND


# ---- 6. against the CPU oracle --------------------------------------------------------------------------------------------------------

def test_exact_matches_oracle(gpu, oracle, blue_noise):
    """An exact engine whose emissive texture is dynamic (mutated every frame) against the oracle that inserts the same bytes before each
    tick: every camera buffer equal for 3 frames at 80x44."""
    scene = scenes.textured_room(80, 44)
    eg = gpu.Engine(blue_noise=blue_noise, exact=True)
    eo = oracle.OracleEngine(blue_noise=blue_noise)
    cg, co = scenes.apply(eg, scene), scenes.apply(eo, scene)
    src = _torch().from_numpy(np.ascontiguousarray(scene["images"][702])).to("cuda")
    eg.insert_dynamic_image(702, src)
    for f in range(3):
        src.add_(29 + f)
        eo.insert_image(702, _np(src))
        eg.tick(); eo.tick()
        eg.render_camera(cg); eo.render_camera(co)
    for name in CAMERA_BUFFERS:
        assert_bits_equal(eg.read_buffer(cg, name), eo.read_buffer(co, name), f"oracle {name}")


# ---- 7. validation -------------------------------------------------------------------------------------------------------------------

def test_refusals_change_nothing(gpu, blue_noise):
    """Every malformed call returns its code; the image already on the handle keeps its bytes, its rectangle and its refresh."""
    torch = _torch()
    e = gpu.Engine(blue_noise=blue_noise)
    scenes.apply(e, _monitor_scene(32, 24))
    src = _rand((FEED_H, FEED_W, 4), 21, device="cuda")
    e.insert_dynamic_image(MONITOR_IMAGE, src)
    e.tick()
    mats = e.read_scene("materials")
    huge = torch.zeros((1, 8193, 4), dtype=torch.uint8, device="cuda")
    pageable = np.zeros((FEED_H, FEED_W, 4), np.uint8)
    p, w, h = src.data_ptr(), FEED_W, FEED_H
    cases = [("null", None, 0, w, h, -2), ("zero width", p, 0, 0, h, -2), ("zero height", p, 0, w, 0, -2),
             ("pitch below the row", p, 4 * w - 4, w, h, -2), ("misaligned address", p + 2, 0, w - 1, h, -2),
             ("misaligned pitch", p, 4 * w + 2, w, h - 1, -2), ("pageable", pageable.ctypes.data, 0, w, h, -2),
             ("atlas full", huge.data_ptr(), 0, 8193, 1, -4)]
    for what, ptr, pitch, cw, ch, code in cases:
        rc = e.lib.st_insert_dynamic_image(e._h, MONITOR_IMAGE, ptr, pitch, cw, ch)
        assert rc == code, f"{what}: {rc}"
        _assert_bytes(e.read_image(MONITOR_IMAGE), src, f"{what}: bytes")
    with pytest.raises(TypeError):
        e.insert_dynamic_image(MONITOR_IMAGE, pageable)
    with pytest.raises(ValueError):
        e.insert_dynamic_image(MONITOR_IMAGE, torch.zeros((FEED_H, FEED_W, 4), dtype=torch.uint8))
    # the refresh is still the one registered first
    src.add_(5)
    e.tick()
    _assert_bytes(e.read_image(MONITOR_IMAGE), src, "refresh after the refusals")
    assert_bits_equal(e.read_scene("materials"), mats, "a refusal moved the rectangle")
    n = C.c_size_t()
    assert e.lib.st_read_image(e._h, MONITOR_IMAGE, None, 0, C.byref(n)) == 0 and n.value == FEED_W * FEED_H * 4
    small = np.zeros(16, np.uint8)
    assert e.lib.st_read_image(e._h, MONITOR_IMAGE, small.ctypes.data, small.nbytes, C.byref(n)) == -4


def test_group_refusal_registers_nothing(gpu, blue_noise):
    """A group refuses a surface its members cannot read (pageable memory) with nothing registered on any member: the Raw image already on
    the handle stays in every member's atlas."""
    grp = gpu.MultiEngine(_devices(2), blue_noise=blue_noise)
    scenes.apply(grp, _monitor_scene(32, 256))
    first = np.ascontiguousarray(_np(_rand((FEED_H, FEED_W, 4), 31)))
    grp.insert_image(MONITOR_IMAGE, first)
    pageable = np.zeros((FEED_H, FEED_W, 4), np.uint8) + 9
    assert grp.lib.st_multi_insert_dynamic_image(grp._h, MONITOR_IMAGE, pageable.ctypes.data, 0, FEED_W, FEED_H) == -2
    grp.tick()
    for r in range(2):
        _assert_bytes(grp.read_image(MONITOR_IMAGE, rank=r), first, f"member {r}")


def test_unreachable_device_is_refused(gpu, blue_noise):
    """Memory of a device this engine's device cannot reach by peer access is refused."""
    torch = _torch()
    n = torch.cuda.device_count()
    pair = next(((a, b) for a in range(n) for b in range(n) if a != b and not torch.cuda.can_device_access_peer(a, b)), None)
    if pair is None:
        pytest.skip("no pair of devices without peer access on this machine")
    e = gpu.Engine(device=pair[0], blue_noise=blue_noise)
    src = torch.zeros((4, 4, 4), dtype=torch.uint8, device=f"cuda:{pair[1]}")
    assert e.lib.st_insert_dynamic_image(e._h, 5, src.data_ptr(), 0, 4, 4) == -2
