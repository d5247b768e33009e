"""Several cameras per frame as one batched pass schedule (st_render_cameras / Engine.render_cameras).

The reference for every comparison is a twin engine: the same scene and seed base, rendering the same cameras one by one through
`render_camera`.  Every camera buffer must match bit for bit (NaN == NaN).
"""
import numpy as np
import pytest

from strolle_b200 import scenes
from tests.util import CAMERA_BUFFERS, assert_bits_equal

pytestmark = pytest.mark.gpu

W, H = 83, 47   # not a multiple of the 16x8 tile; (W + 7) / 8 is odd, so the checkerboard half grid leaves a column over


@pytest.fixture(scope="module")
def gpu():
    import strolle_b200
    return strolle_b200


def _pose(scene, k, f):
    """Camera k's transform on frame f: the scene's camera, shifted by an amount that differs per camera and per frame."""
    t = np.array(scene["camera"]["transform"], np.float32).reshape(-1).copy()
    t[12] += 0.07 * (k - 2) + 0.011 * f * (k % 3)
    t[13] += 0.03 * k - 0.004 * f
    t[14] += -0.02 * k + 0.013 * f * ((k + 1) % 2)
    return t


class Twins:
    """A batched engine and its sequential twin with the same scene and the same cameras."""

    def __init__(self, gpu, blue_noise, scene, exact=False, options=()):
        self.scene = scene
        self.e = [gpu.Engine(blue_noise=blue_noise, exact=exact) for _ in range(2)]
        for e in self.e:
            for o, v in options:
                e.set_option(o, v)
        self.first = [scenes.apply(e, scene) for e in self.e]
        self.cams = [[], []]   # handles per engine, same order
        self.desc = []

    def add(self, k, w=W, h=H, mode=None, denoise=None, frame=0):
        c = self.scene["camera"]
        d = (c["mode"] if mode is None else mode, c["denoise"] if denoise is None else denoise, c["ref_depth"], w, h)
        proj = scenes.perspective_infinite_reverse_rh(np.pi / 4.0, w / h, 0.1)
        for i, e in enumerate(self.e):
            self.cams[i].append(e.create_camera(*d, _pose(self.scene, k, frame), proj))
        self.desc.append((k, d, proj))

    def replace(self, j, frame):
        """Deletes camera j and creates it again (its arena then sits at an unrelated address)."""
        k, d, proj = self.desc[j]
        for i, e in enumerate(self.e):
            _delete(e, self.cams[i][j])
            self.cams[i][j] = e.create_camera(*d, _pose(self.scene, k, frame), proj)

    def move(self, frame):
        for i, e in enumerate(self.e):
            for j, (k, d, proj) in enumerate(self.desc):
                e.update_camera(self.cams[i][j], *d, _pose(self.scene, k, frame), proj)

    def tick(self):
        for e in self.e:
            e.tick()

    def render(self, outs=None, twin_outs=None, fmt=0):
        self.e[0].render_cameras(self.cams[0], outs, fmt)
        for j, c in enumerate(self.cams[1]):
            self.e[1].render_camera(c, None if twin_outs is None else twin_outs[j], fmt)

    def check(self, what, names=CAMERA_BUFFERS):
        for j in range(len(self.cams[0])):
            for name in names:
                assert_bits_equal(self.e[0].read_buffer(self.cams[0][j], name), self.e[1].read_buffer(self.cams[1][j], name), f"{what} camera {j} {name}")


def _delete(e, cam):
    e._check(e.lib.st_delete_camera(e._h, cam))


def _scene(name):
    return scenes.cornell(W, H) if name == "cornell" else scenes.demo_level(W, H)


@pytest.mark.parametrize("tier", ["default", "exact", "unfused"])
@pytest.mark.parametrize("scene_name", ["cornell", "demo_level"])
def test_equivalence_13_frames(gpu, blue_noise, tier, scene_name):
    """Five cameras of one odd size, moving differently every frame, created at different times and one re-created between frames, with
    an instance moving on some frames: after each of 13 frames every buffer of every camera equals the twin's."""
    from strolle_b200.engine import OPT_FUSED_PASSES
    scene = _scene(scene_name)
    t = Twins(gpu, blue_noise, scene, exact=tier == "exact", options=[(OPT_FUSED_PASSES, 0)] if tier == "unfused" else [])
    for i, e in enumerate(t.e):
        _delete(e, t.first[i])
    t.add(0); t.add(1); t.add(2)
    h, mesh, mat, xf = scene["instances"][min(6, len(scene["instances"]) - 1)]
    for f in range(13):
        if f == 2:
            t.add(3, frame=f)
        if f == 4:
            t.add(4, frame=f)
        if f == 6:
            t.replace(1, f)
        if f in (3, 4, 9):
            moved = np.array(xf, np.float32).copy(); moved[9] += 0.03 * f; moved[11] -= 0.01 * f
            for e in t.e:
                e.insert_instance(h, mesh, mat, moved)
        t.move(f)
        t.tick()
        t.render()
        t.check(f"{scene_name} {tier} frame {f + 1}")


@pytest.mark.parametrize("denoise", [True, False])
def test_every_mode(gpu, blue_noise, denoise):
    """A group of three views per camera mode matches the twin for 7 frames (reference mode accumulates over them)."""
    t = Twins(gpu, blue_noise, scenes.cornell(W, H))
    for mode in range(7):
        for k in range(3):
            t.add(k, mode=mode, denoise=denoise)
    for f in range(7):
        t.move(f % 2)   # reference mode accumulates while its camera stands still
        t.tick()
        t.render()
        t.check(f"denoise={denoise} frame {f + 1}")


def test_mixed_list_runs_as_groups(gpu, blue_noise):
    """Two sizes and two modes interleaved in the list run as four groups; with timing on, the launches of a frame are the sum over the
    groups of one camera's launches."""
    t = Twins(gpu, blue_noise, scenes.cornell(W, H))
    kinds = [(W, H, 0), (40, 24, 0), (W, H, 3), (40, 24, 3)]
    for k in range(8):
        w, h, mode = kinds[k % 4]
        t.add(k, w=w, h=h, mode=mode)
    for f in range(3):
        t.move(f)
        t.tick()
        t.e[0].enable_timing(True); t.e[1].enable_timing(True)
        t.e[0].pass_times(reset=True); t.e[1].pass_times(reset=True)
        t.render()
        batched = int(t.e[0].pass_times(reset=True)[1].sum())
        per_camera = t.e[1].pass_times(reset=True)[1]
        t.check(f"mixed frame {f + 1}")
    # one camera per kind: what the twin launched for the first camera of every kind, and nothing more
    single = []
    for j in range(4):
        t.e[1].render_camera(t.cams[1][j])
        single.append(int(t.e[1].pass_times(reset=True)[1].sum()))
    assert batched == sum(single), f"{batched} launches for 4 groups, one camera each takes {single}"
    assert int(per_camera.sum()) == 2 * sum(single)


def test_chunking(gpu, blue_noise):
    """70 views of 24x16 are more than one launch holds: they run as several launches per pass and still match the twin."""
    t = Twins(gpu, blue_noise, scenes.cornell(24, 16))
    for k in range(70):
        t.add(k, w=24, h=16)
    for f in range(3):
        t.move(f)
        t.tick()
        t.render()
        t.check(f"70 views frame {f + 1}", names=["di_reservoirs_2", "gi_reservoirs_0", "di_diff_curr_colors", "gi_diff_curr_colors", "output"])


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
    """16 views composed as a 4x4 mosaic into one surface at offsets, with row padding: every rectangle holds the twin's packed bytes and
    every byte between them keeps the sentinel."""
    w, h, gap = 40, 24, 3
    t = Twins(gpu, blue_noise, scenes.cornell(w, h))
    for k in range(16):
        t.add(k, w=w, h=h)
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


def test_some_views_without_output(gpu, blue_noise):
    """A None surface renders that view without writing anything for it; its `output` buffer is still the twin's."""
    import torch
    t = Twins(gpu, blue_noise, scenes.cornell(W, H))
    for k in range(4):
        t.add(k)
    outs = [torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0") if k % 2 == 0 else None for k in range(4)]
    for f in range(2):
        t.move(f); t.tick(); t.render(outs)
        t.check(f"frame {f + 1}", names=["output"])
    for k in (0, 2):
        assert_bits_equal(outs[k].cpu().numpy(), t.e[1].read_buffer(t.cams[1][k], "output"), f"view {k}")


def test_validation_renders_nothing(gpu, blue_noise):
    """Refused calls render nothing and write no surface; the next frame still matches the twin."""
    import torch
    from strolle_b200.engine import StrolleError
    t = Twins(gpu, blue_noise, scenes.cornell(W, H))
    for k in range(4):
        t.add(k)
    t.tick(); t.render()
    e, cams = t.e[0], t.cams[0]
    strip = e.create_camera(*t.desc[0][1], _pose(t.scene, 9, 0), t.desc[0][2])
    e.set_strip(strip, 0, H // 2)
    gone = e.create_camera(*t.desc[0][1], _pose(t.scene, 9, 0), t.desc[0][2])
    _delete(e, gone)
    t.tick()
    before = [e.read_buffer(c, "output") for c in cams]
    good = torch.full((H, W, 4), 7.0, dtype=torch.float32, device="cuda:0")
    bad = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda:0")
    cases = [("duplicate", [cams[0], cams[1], cams[0]], None, "error -2"),   # ST_ERR_INVALID
             ("deleted", [cams[0], gone], None, "error -3"),               # ST_ERR_NOT_FOUND
             ("strip", [cams[0], strip], None, "error -2"),
             ("empty", [], None, "error -2")]
    import ctypes as C
    for what, lst, outs, code in cases:
        with pytest.raises(StrolleError, match=code):
            e.render_cameras(lst, outs)
        for c, b in zip(cams, before):
            assert_bits_equal(e.read_buffer(c, "output"), b, f"{what}: output changed")
    # one bad surface (misaligned address) in the middle of the list, through the C ABI
    dsts = (C.c_void_p * 4)(good.data_ptr(), good.data_ptr(), bad.data_ptr() + 4, good.data_ptr())
    pitches = (C.c_size_t * 4)(0, 0, 0, 0)
    rc = e.lib.st_render_cameras(e._h, (C.c_int32 * 4)(*cams), 4, dsts, pitches, 0)
    assert rc == -2, rc
    torch.cuda.synchronize()
    assert (good == 7.0).all() and (bad == 0.0).all(), "a refused call wrote a surface"
    for c, b in zip(cams, before):
        assert_bits_equal(e.read_buffer(c, "output"), b, "bad surface: output changed")
    t.render()
    t.check("after the refusals")


def test_strict_batch_matches_oracle(gpu, oracle, blue_noise):
    """One view of a strict-tier batch at 96x54 is bit-identical to the CPU oracle's frame for that camera."""
    scene = scenes.cornell(96, 54)
    eg = gpu.Engine(blue_noise=blue_noise, exact=True)
    eo = oracle.OracleEngine(blue_noise=blue_noise)
    cg, co = scenes.apply(eg, scene), scenes.apply(eo, scene)
    c = scene["camera"]
    others = [eg.create_camera(c["mode"], c["denoise"], c["ref_depth"], 96, 54, _pose(scene, k, 0), c["projection"]) for k in range(3)]
    for f in range(3):
        eg.tick(); eo.tick()
        eg.render_cameras([others[0], cg, others[1], others[2]])
        eo.render_camera(co)
    for name in CAMERA_BUFFERS:
        assert_bits_equal(eg.read_buffer(cg, name), eo.read_buffer(co, name), f"oracle {name}")
