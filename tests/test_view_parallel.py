"""View-parallel groups: cameras placed whole on one member of a MultiEngine (create_camera(..., rank=)), rendered by every member at once
(MultiEngine.render_cameras / st_multi_render_cameras), moved between members with their temporal state (move_camera).

The reference for every comparison is a single `Engine` with the same scene and seed base that renders the same cameras one by one with
`render_camera`.  Every camera buffer must match bit for bit (NaN == NaN).  Members come from `_devices(n)`: a one-GPU box runs every
member on device 0, a box with several GPUs puts them on different devices, so peer copies and peer stores run for real.
"""
import ctypes as C

import numpy as np
import pytest

from strolle_b200 import scenes
from tests.test_dynamic_images import MONITOR_IMAGE, _monitor_scene
from tests.util import CAMERA_BUFFERS, assert_bits_equal

pytestmark = pytest.mark.gpu

W, H = 83, 47


@pytest.fixture(scope="module")
def gpu():
    import strolle_b200
    return strolle_b200


def _devices(n):
    import torch
    have = max(torch.cuda.device_count(), 1)
    return [k % have for k in range(n)]


def _pose(scene, k, f):
    t = np.array(scene["camera"]["transform"], np.float32).reshape(-1).copy()
    t[12] += 0.07 * (k - 2) + 0.011 * f * (k % 3)
    t[13] += 0.03 * k - 0.004 * f
    t[14] += -0.02 * k + 0.013 * f * ((k + 1) % 2)
    return t


def _gdelete(g, cam):
    g._check(g.lib.st_multi_delete_camera(g._h, cam))


def _delete(e, cam):
    e._check(e.lib.st_delete_camera(e._h, cam))


class Twins:
    """A view-parallel group and a single engine with the same scene and the same cameras (placed on the group's members)."""

    def __init__(self, gpu, blue_noise, scene, n=3, exact=False, options=()):
        self.scene = scene
        self.g = gpu.MultiEngine(_devices(n), blue_noise=blue_noise, exact=exact)
        self.one = gpu.Engine(blue_noise=blue_noise, exact=exact)
        for e in (self.g, self.one):
            for o, v in options:
                e.set_option(o, v)
        self.strip = scenes.apply(self.g, scene)      # the scene's own camera: a strip camera of the group
        self.strip_twin = scenes.apply(self.one, scene)
        self.cams, self.twin, self.desc = [], [], []

    def add(self, k, rank, w=W, h=H, mode=None, frame=0):
        c = self.scene["camera"]
        d = (c["mode"] if mode is None else mode, c["denoise"], c["ref_depth"], w, h)
        proj = scenes.perspective_infinite_reverse_rh(np.pi / 4.0, w / h, 0.1)
        self.cams.append(self.g.create_camera(*d, _pose(self.scene, k, frame), proj, rank=rank))
        self.twin.append(self.one.create_camera(*d, _pose(self.scene, k, frame), proj))
        self.desc.append([k, d, proj])
        return len(self.cams) - 1

    def replace(self, j, frame, rank):
        k, d, proj = self.desc[j]
        _gdelete(self.g, self.cams[j]); _delete(self.one, self.twin[j])
        self.cams[j] = self.g.create_camera(*d, _pose(self.scene, k, frame), proj, rank=rank)
        self.twin[j] = self.one.create_camera(*d, _pose(self.scene, k, frame), proj)

    def move(self, frame):
        for j, desc in enumerate(self.desc):
            if desc is None:   # deleted
                continue
            k, d, proj = desc
            self.g.update_camera(self.cams[j], *d, _pose(self.scene, k, frame), proj)
            self.one.update_camera(self.twin[j], *d, _pose(self.scene, k, frame), proj)

    def tick(self):
        self.g.tick(); self.one.tick()

    def render(self, outs=None, twin_outs=None, fmt=0):
        self.g.render_cameras(self.cams, outs, fmt)
        for j, c in enumerate(self.twin):
            self.one.render_camera(c, None if twin_outs is None else twin_outs[j], fmt)

    def check(self, what, names=CAMERA_BUFFERS, which=None):
        for j in (range(len(self.cams)) if which is None else which):
            for name in names:
                assert_bits_equal(self.g.read_buffer(self.cams[j], name), self.one.read_buffer(self.twin[j], name), f"{what} camera {j} {name}")


def _scene(name, w=W, h=H):
    return scenes.cornell(w, h) if name == "cornell" else scenes.demo_level(w, h)


# ---- 1. equivalence ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tier", ["default", "exact", "unfused"])
@pytest.mark.parametrize("scene_name", ["cornell", "demo_level"])
def test_equivalence_13_frames(gpu, blue_noise, tier, scene_name):
    """A 3-member group with 7 cameras of three sizes and three modes, placed by rank and by "auto", created at different frames, one
    re-created, all moving every frame and an instance moving on some: after each of 13 frames every buffer of every camera equals the
    single engine's."""
    from strolle_b200.engine import OPT_FUSED_PASSES
    scene = _scene(scene_name)
    t = Twins(gpu, blue_noise, scene, exact=tier == "exact", options=[(OPT_FUSED_PASSES, 0)] if tier == "unfused" else [])
    t.add(0, 0); t.add(1, "auto", w=40, h=24); t.add(2, 2, mode=3); t.add(3, "auto", w=64, h=40); t.add(4, "auto", w=40, h=24, mode=1)
    h, mesh, mat, xf = scene["instances"][min(6, len(scene["instances"]) - 1)]
    for f in range(13):
        if f == 2:
            t.add(5, "auto", frame=f)
        if f == 4:
            t.add(6, 1, w=64, h=40, mode=3, frame=f)
        if f == 6:
            t.replace(1, f, "auto")
        if f in (3, 4, 9):
            moved = np.array(xf, np.float32).copy(); moved[9] += 0.03 * f; moved[11] -= 0.01 * f
            for e in (t.g, t.one):
                e.insert_instance(h, mesh, mat, moved)
        t.move(f)
        t.tick()
        t.render()
        t.check(f"{scene_name} {tier} frame {f + 1}")
    assert {t.g.camera_rank(c) for c in t.cams} == {0, 1, 2}


# ---- 2. mosaics ---------------------------------------------------------------------------------------------------------------------------

SENTINEL = 0xA5


def _dtype(fmt):
    return {0: np.float32, 2: np.float16}.get(fmt, np.uint8)


def _surface(kind, shape, dtype):
    import torch
    tdtype = {np.float32: torch.float32, np.float16: torch.float16, np.uint8: torch.uint8}[dtype]
    if kind == "pageable":
        a = np.empty(shape, dtype)
        a.view(np.uint8)[...] = SENTINEL
        return a
    s = torch.empty(shape, dtype=tdtype, pin_memory=True) if kind == "pinned" else torch.empty(shape, dtype=tdtype, device="cuda:0")
    s.view(torch.uint8).fill_(SENTINEL)
    return s


def _host(s):
    return s if isinstance(s, np.ndarray) else s.cpu().numpy()


@pytest.mark.parametrize("kind", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_mosaic_into_one_surface(gpu, blue_noise, kind, fmt):
    """16 views placed "auto" on 3 members composed as a 4x4 mosaic into one surface (on device 0 for "device": the views of members 1 and
    2 store into it from their own devices when the box has them): every rectangle holds the single engine's bytes, every byte between
    them keeps the sentinel."""
    w, h, gap = 40, 24, 3
    t = Twins(gpu, blue_noise, scenes.cornell(w, h))
    for k in range(16):
        t.add(k, "auto", w=w, h=h)
    assert [t.g.camera_rank(c) for c in t.cams] == [k % 3 for k in range(16)]
    big = _surface(kind, (4 * (h + gap) + 1, 4 * (w + gap) + 5, 4), _dtype(fmt))
    at = [(gap + (k // 4) * (h + gap), gap + (k % 4) * (w + gap)) for k in range(16)]
    for f in range(2):
        t.move(f)
        t.tick()
        twin = [np.zeros((h, w, 4), _dtype(fmt)) for _ in range(16)]
        t.render([big[y:y + h, x:x + w] for y, x in at], twin, fmt)
        got = _host(big)
        mask = np.ones(got.shape[:2], bool)
        for k, (y, x) in enumerate(at):
            assert (got[y:y + h, x:x + w].view(np.uint8) == twin[k].view(np.uint8)).all(), f"{kind} format {fmt} frame {f + 1} view {k}"
            mask[y:y + h, x:x + w] = False
        assert (got.view(np.uint8).reshape(got.shape[0], got.shape[1], -1)[mask] == SENTINEL).all(), "bytes outside the views were written"
    t.check(f"{kind} format {fmt}", names=["output", "di_diff_curr_colors", "gi_reservoirs_0"])


# ---- 3. placement -------------------------------------------------------------------------------------------------------------------------

def test_placement(gpu, blue_noise):
    """"auto" picks the member with the fewest pixels of placed cameras (strip cameras do not count, deleted ones no longer do), the
    lowest rank on a tie; camera_rank reports it; a placed camera has a handle on its member only, and no buffers anywhere else."""
    from strolle_b200.engine import PLACE_STRIPS, StrolleError
    scene = scenes.cornell(W, H)
    g = gpu.MultiEngine(_devices(3), blue_noise=blue_noise)
    strip = scenes.apply(g, scene)
    c = scene["camera"]

    def make(w, h, rank="auto"):
        return g.create_camera(c["mode"], c["denoise"], c["ref_depth"], w, h, c["transform"], c["projection"], rank=rank)

    cams = [make(100, 100), make(50, 50), make(50, 50), make(10, 10), make(10, 10), make(100, 100, rank=1)]
    ranks = [g.camera_rank(x) for x in cams]
    assert ranks == [0, 1, 2, 1, 2, 1], ranks     # pixels after each: [1e4,0,0] [1e4,2500,0] [.., 2500] [.., 2600, 2500] [.., 2600] [1e4, 12600, 2600]
    assert make(10, 10) == cams[-1] + 1 and g.camera_rank(cams[-1] + 1) == 2
    _gdelete(g, cams[0])                            # member 0 now holds no pixels
    assert g.camera_rank(make(30, 30)) == 0
    assert g.camera_rank(strip) == PLACE_STRIPS
    for x, r in zip(cams[1:], ranks[1:]):
        for m in range(3):
            mh = g.member_camera(x, m)
            assert (mh >= 0) == (m == r), (x, m, mh)
            if m != r:
                with pytest.raises(StrolleError, match="error -3"):
                    g.member(m).read_buffer(mh, "output")
        assert g.member(r).read_buffer(g.member_camera(x, r), "output").size == g.read_buffer(x, "output").size
    assert all(g.member_camera(strip, m) >= 0 for m in range(3))
    with pytest.raises(StrolleError, match="error -3"):
        g.camera_rank(cams[0])
    # a group of one member: a placed camera is an ordinary camera of member 0 and renders as one engine does
    one, solo = gpu.MultiEngine(_devices(1), blue_noise=blue_noise), gpu.Engine(blue_noise=blue_noise)
    for e in (one, solo):
        e._first = scenes.apply(e, scene)
    a = one.create_camera(c["mode"], c["denoise"], c["ref_depth"], 40, 24, c["transform"], c["projection"], rank="auto")
    b = solo.create_camera(c["mode"], c["denoise"], c["ref_depth"], 40, 24, c["transform"], c["projection"])
    assert one.camera_rank(a) == 0
    for f in range(2):
        one.tick(); solo.tick()
        one.render_cameras([one._first, a]); solo.render_cameras([solo._first, b])
    for name in CAMERA_BUFFERS:
        assert_bits_equal(one.read_buffer(a, name), solo.read_buffer(b, name), f"one-member group {name}")


# ---- 4. moves -----------------------------------------------------------------------------------------------------------------------------

def test_move_keeps_temporal_state(gpu, blue_noise):
    """A camera moved to another member before the tick of frame 6 and moved back after the tick of frame 9 renders, through frame 13, the
    single engine's frames bit for bit (its reservoirs, history and moments travelled with it).  A move to its own member does nothing;
    refused moves leave it rendering where it was."""
    from strolle_b200.engine import StrolleError
    t = Twins(gpu, blue_noise, scenes.cornell(W, H))
    x = t.add(0, 0); y = t.add(1, 1, mode=3); t.add(2, 2, w=40, h=24)
    g = t.g
    for f in range(13):
        if f == 3:
            g.move_camera(t.cams[y], 1)   # to its own member
            assert g.camera_rank(t.cams[y]) == 1
        if f == 6:
            g.move_camera(t.cams[x], 2)
            assert g.camera_rank(t.cams[x]) == 2 and g.member_camera(t.cams[x], 0) == -1 and g.member_camera(t.cams[x], 2) >= 0
        t.move(f)
        t.tick()
        if f == 9:
            g.move_camera(t.cams[x], 0)
            assert g.camera_rank(t.cams[x]) == 0
        if f == 7:
            for rank, code in [(3, "error -2"), (-1, "error -2"), (-2, "error -2")]:   # through the C ABI, past the Python check
                assert g.lib.st_multi_move_camera(g._h, t.cams[y], rank) == int(code.split()[1])
            assert g.lib.st_multi_move_camera(g._h, t.strip, 0) == -2
            assert g.lib.st_multi_move_camera(g._h, 999, 0) == -3
            with pytest.raises(ValueError):
                g.move_camera(t.cams[y], 3)
            with pytest.raises(TypeError):
                g.move_camera(t.cams[y], "elsewhere")
            assert g.camera_rank(t.cams[y]) == 1
        t.render()
        t.check(f"frame {f + 1}")
    with pytest.raises(StrolleError, match="error -2"):
        g.move_camera(t.strip, 1)


# ---- 5. the group verbs on placed cameras --------------------------------------------------------------------------------------------------

def test_verbs_on_placed_cameras(gpu, blue_noise):
    """update (with a resize), delete, render_camera into host memory, render_camera into a CUDA tensor and read_buffer on placed cameras
    give the single engine's frames; a strip camera of the same group (strips of 128 rows) still matches the single-GPU frame."""
    import torch
    from strolle_b200.engine import StrolleError
    scene = scenes.cornell(64, 256)
    t = Twins(gpu, blue_noise, scene, n=2)
    p = t.add(0, 1); q = t.add(1, 0, w=40, h=24)
    g, one = t.g, t.one
    for f in range(5):
        if f == 2:   # resize p: buffers re-created on member 1 only
            t.desc[p][1] = t.desc[p][1][:3] + (60, 40)
            t.desc[p][2] = scenes.perspective_infinite_reverse_rh(np.pi / 4.0, 60 / 40, 0.1)
        t.move(f)
        if f == 3:
            _gdelete(g, t.cams[q]); _delete(one, t.twin[q])
            t.desc[q] = None
            with pytest.raises(StrolleError, match="error -3"):
                g.render_cameras([t.cams[q]])
        t.tick()
        pw, ph = t.desc[p][1][3:]
        host, host_twin = np.zeros((ph, pw, 4), np.float32), np.zeros((ph, pw, 4), np.float32)
        g.render_camera(t.cams[p], host); one.render_camera(t.twin[p], host_twin)
        assert_bits_equal(host, host_twin, f"frame {f + 1} render_camera")
        if f < 3:
            dev = torch.zeros((24, 40, 4), dtype=torch.float16, device="cuda:0")
            twin = np.zeros((24, 40, 4), np.float16)
            g.render_camera(t.cams[q], dev, 2); one.render_camera(t.twin[q], twin, 2)
            assert (dev.cpu().numpy().view(np.uint16) == twin.view(np.uint16)).all(), f"frame {f + 1} render_camera into a CUDA tensor"
        s, s_twin = np.zeros((256, 64, 4), np.float32), np.zeros((256, 64, 4), np.float32)
        g.render_camera(t.strip, s); one.render_camera(t.strip_twin, s_twin)
        assert_bits_equal(s, s_twin, f"frame {f + 1} strip camera")
        t.check(f"frame {f + 1}", which=[p] + ([q] if f < 3 else []))
        assert g.peer_errors(t.cams[p]) == 0
    for name in CAMERA_BUFFERS:
        assert_bits_equal(g.read_buffer(t.strip, name), one.read_buffer(t.strip_twin, name), f"strip camera {name}")


# ---- 6. render to texture across members ----------------------------------------------------------------------------------------------------

def test_render_to_texture_across_members(gpu, blue_noise):
    """A feed camera on member 1 renders RGBA8 into a device-0 tensor that is a dynamic image of the group; a camera on member 0 looks at
    the monitor showing it.  Over 8 frames both frames equal those of a single engine doing the same one camera after the other."""
    import torch
    from strolle_b200.engine import FORMAT_RGBA8_SRGB
    w, h, aw, ah = 96, 54, 48, 32
    scene = _monitor_scene(w, h)
    proj_a = scenes.perspective_infinite_reverse_rh(np.pi / 3.0, aw / ah, 0.1)
    ta = scenes.look_at_transform((0.8, 1.2, 1.5), (-0.3, 0.8, -0.5))
    c = scene["camera"]
    runs = []
    for grp in (True, False):
        e = gpu.MultiEngine(_devices(2), blue_noise=blue_noise) if grp else gpu.Engine(blue_noise=blue_noise)
        first = scenes.apply(e, scene)
        kw = [dict(rank=1), dict(rank=0)] if grp else [{}, {}]
        a = e.create_camera(0, True, 1, aw, ah, ta, proj_a, **kw[0])
        b = e.create_camera(c["mode"], c["denoise"], c["ref_depth"], w, h, c["transform"], c["projection"], **kw[1])
        feed = torch.zeros((ah, aw, 4), dtype=torch.uint8, device="cuda:0")
        e.insert_dynamic_image(MONITOR_IMAGE, feed)
        runs.append((e, first, a, b, feed))
    for f in range(8):
        tf = scenes.look_at_transform((0.3 * np.sin(0.4 * f), 1.0 + 0.05 * f, 3.2 - 0.1 * f), (0.0, 1.0, -0.5))
        got = []
        for grp, (e, first, a, b, feed) in zip((True, False), runs):
            e.update_camera(b, c["mode"], c["denoise"], c["ref_depth"], w, h, tf, c["projection"])
            e.tick()
            out = np.zeros((h, w, 4), np.uint8)
            if grp:
                e.render_cameras([a, b], [feed, out], FORMAT_RGBA8_SRGB)
            else:
                e.render_camera(a, feed, FORMAT_RGBA8_SRGB); e.render_camera(b, out, FORMAT_RGBA8_SRGB)
            got.append((out, feed.cpu().numpy(), e.read_buffer(b, "output")))
        assert (got[0][0] == got[1][0]).all(), f"frame {f + 1}: monitor camera"
        assert (got[0][1] == got[1][1]).all(), f"frame {f + 1}: feed camera"
        assert_bits_equal(got[0][2], got[1][2], f"frame {f + 1}: monitor camera output buffer")
    assert got[0][1][..., :3].max() > 0


# ---- 7. refusals ----------------------------------------------------------------------------------------------------------------------------

def test_refusals_change_nothing(gpu, blue_noise):
    """Every refused st_multi_render_cameras call renders nothing on any member and writes no surface; the next frame still matches."""
    import torch
    from strolle_b200.engine import StrolleError
    t = Twins(gpu, blue_noise, scenes.cornell(W, H))
    for k in range(4):
        t.add(k, k % 3)
    g, cams = t.g, t.cams
    fresh = gpu.MultiEngine(_devices(2), blue_noise=blue_noise)
    scenes.apply(fresh, scenes.cornell(W, H))
    early = fresh.create_camera(*t.desc[0][1], _pose(t.scene, 0, 0), t.desc[0][2], rank=1)
    with pytest.raises(StrolleError, match="error -2"):
        fresh.render_cameras([early])            # before the first tick
    t.tick(); t.render()
    gone = g.create_camera(*t.desc[0][1], _pose(t.scene, 9, 0), t.desc[0][2], rank=2)
    _gdelete(g, gone)
    t.tick()
    before = [g.read_buffer(x, "output") for x in cams]
    surfaces = [torch.full((H, W, 4), 7.0, dtype=torch.float32, device="cuda:0") for _ in cams]
    cases = [("duplicate", [cams[0], cams[1], cams[0]], "error -2"), ("deleted", [cams[0], gone], "error -3"),
             ("unknown", [cams[1], 999], "error -3"), ("strip camera", [cams[0], t.strip], "error -2"), ("empty", [], "error -2")]
    for what, lst, code in cases:
        with pytest.raises(StrolleError, match=code):
            g.render_cameras(lst, [surfaces[cams.index(x)] if x in cams else None for x in lst])
        torch.cuda.synchronize()
        assert all((s == 7.0).all() for s in surfaces), f"{what}: a refused call wrote a surface"
        for x, b in zip(cams, before):
            assert_bits_equal(g.read_buffer(x, "output"), b, f"{what}: output changed")
    # a surface the camera's member refuses (misaligned), after surfaces of cameras on other members
    dsts = (C.c_void_p * 4)(*[s.data_ptr() for s in surfaces[:3]], surfaces[3].data_ptr() + 4)
    rc = g.lib.st_multi_render_cameras(g._h, (C.c_int32 * 4)(*cams), 4, dsts, (C.c_size_t * 4)(0, 0, 0, 0), 0)
    assert rc == -2, rc
    torch.cuda.synchronize()
    assert all((s == 7.0).all() for s in surfaces), "a refused call wrote a surface"
    for x, b in zip(cams, before):
        assert_bits_equal(g.read_buffer(x, "output"), b, "bad surface: output changed")
    t.render()
    t.check("after the refusals")
