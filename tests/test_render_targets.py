"""Composition into caller-owned surfaces (st_render_camera_to / st_multi_render_camera_to): Rgba16Float output, device-memory targets,
row pitch and viewport offset.

The reference for every comparison is the engine's own composed frame (`read_buffer(cam, "output")`, which the parity tests pin to
the oracle) or the packed host read-back of an identically seeded twin engine (`st_render_camera`, whose bytes those tests pin too).
"""
import numpy as np
import pytest

from strolle_b200 import scenes
from tests.util import assert_bits_equal

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
W_ODD, H_ODD = 161, 91


@pytest.fixture(scope="module")
def gpu():
    import strolle_b200
    return strolle_b200


def _devices(n):
    import torch
    have = max(torch.cuda.device_count(), 1)
    return [k % have for k in range(n)]   # a single-GPU box runs every strip on device 0: same protocol, same kernels


def _dtype(fmt):
    from strolle_b200.engine import FORMAT_RGBA32F, FORMAT_RGBA16F
    return {FORMAT_RGBA32F: np.float32, FORMAT_RGBA16F: np.float16}.get(fmt, np.uint8)


def _formats():
    from strolle_b200.engine import FORMAT_RGBA32F, FORMAT_RGBA8_SRGB, FORMAT_RGBA16F
    return [FORMAT_RGBA32F, FORMAT_RGBA8_SRGB, FORMAT_RGBA16F]


def _half_of_output(e, cam, w, h):
    """What an Rgba16Float store of the composed frame must hold: each channel rounded to nearest-even, alpha 1.0."""
    want = np.empty((h, w, 4), np.float16)
    want[..., :3] = e.read_buffer(cam, "output").reshape(h, w, 4)[..., :3].astype(np.float16)
    want[..., 3] = np.float16(1.0)
    return want


def _assert_same_bits(a, b, what):
    """Byte-for-byte equality, except that a NaN matches any NaN of the same width."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype, what
    same = a.view(np.uint8) == b.view(np.uint8)
    if a.dtype.kind == "f":
        same = (a.view(f"u{a.itemsize}") == b.view(f"u{b.itemsize}")) | (np.isnan(a) & np.isnan(b))
    assert same.all(), f"{what}: {int((~same).sum())} values differ"


def _surface(kind, shape, dtype):
    """A surface of `shape` filled with the sentinel byte: "pageable" numpy, "pinned" torch CPU tensor, "device" CUDA tensor."""
    import torch
    tdtype = {np.float32: torch.float32, np.float16: torch.float16, np.uint8: torch.uint8}[dtype]
    if kind == "pageable":
        a = np.empty(shape, dtype)
        a.view(np.uint8)[...] = SENTINEL
        return a
    t = torch.empty(shape, dtype=tdtype, pin_memory=True) if kind == "pinned" else torch.empty(shape, dtype=tdtype, device="cuda:0")
    t.view(torch.uint8).fill_(SENTINEL)
    return t


def _host(surface):
    if isinstance(surface, np.ndarray):
        return surface
    import torch
    if surface.is_cuda:
        torch.cuda.synchronize()
    return surface.cpu().numpy()


def _frame_and_rest(big, y, x, h, w):
    """(the h x w rectangle at (y, x), every byte of the surface outside it)."""
    rect = big[y:y + h, x:x + w].copy()
    mask = np.ones(big.shape[:2], bool)
    mask[y:y + h, x:x + w] = False
    return rect, big.view(np.uint8).reshape(big.shape[0], big.shape[1], -1)[mask]


# ---- Rgba16Float ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("variant", ["cornell_1080p", "demo_level", "cornell_hot"])
def test_rgba16f_host_bit_exact(gpu, blue_noise, variant):
    """The host Rgba16Float frame is the composed frame rounded to binary16 with round-to-nearest-even, bit for bit (NaN matches NaN),
    alpha 0x3C00; the hot variant's emissive of 1e5 composes pixels above 65504, which must overflow to inf like numpy's conversion."""
    from strolle_b200.engine import FORMAT_RGBA16F
    if variant == "cornell_1080p":
        scene = scenes.cornell(1920, 1080)
    elif variant == "demo_level":
        scene = scenes.demo_level(176, 99)
    else:
        scene = scenes.cornell(W_ODD, H_ODD)
        params, alpha = scene["materials"][100]
        params = params.copy(); params[4:8] = (1e5, 1e5, 1e5, 1.0)
        scene["materials"][100] = (params, alpha)
    w, h = scene["camera"]["w"], scene["camera"]["h"]
    e = gpu.Engine(blue_noise=blue_noise)
    cam = scenes.apply(e, scene)
    out = np.zeros((h, w, 4), np.float16)
    for f in range(4):
        e.tick()
        e.render_camera(cam, out, FORMAT_RGBA16F)
        want = _half_of_output(e, cam, w, h)
        _assert_same_bits(out, want, f"{variant} frame {f + 1}")
        assert (out[..., 3].view(np.uint16) == 0x3C00).all()
    assert np.isfinite(out[..., :3]).any() and out[..., :3].astype(np.float32).max() > 0
    if variant == "cornell_hot":
        assert np.isinf(out[..., :3]).any(), "the hot emitter must overflow binary16"


# ---- device targets ---------------------------------------------------------------------------------------------------------------

def test_device_targets_match_host_bytes(gpu, blue_noise):
    """A CUDA tensor in each format holds the bytes the packed host read-back (st_render_camera) of the same frame holds; an identically
    seeded twin engine renders the host side, so the RGBA8 bytes are the ones st_render_camera has always returned."""
    import torch
    scene = scenes.cornell(W_ODD, H_ODD)
    ed, eh = gpu.Engine(blue_noise=blue_noise), gpu.Engine(blue_noise=blue_noise)
    cd, ch = scenes.apply(ed, scene), scenes.apply(eh, scene)
    for f in range(6):
        fmt = _formats()[f % 3]
        dt = _dtype(fmt)
        dev = torch.zeros((H_ODD, W_ODD, 4), dtype={np.float32: torch.float32, np.float16: torch.float16, np.uint8: torch.uint8}[dt], device="cuda:0")
        host = np.zeros((H_ODD, W_ODD, 4), dt)
        ed.tick(); eh.tick()
        ed.render_camera(cd, dev, fmt)
        eh.render_camera(ch, host, fmt)
        _assert_same_bits(dev.cpu().numpy(), host, f"frame {f + 1} format {fmt}")
        assert_bits_equal(ed.read_buffer(cd, "output"), eh.read_buffer(ch, "output"), f"frame {f + 1}: twin engines")
    assert host.view(np.uint8).any()


# ---- pitch and viewport offset (LoadOp::Load) -------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["pageable", "pinned_async", "device"])
@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_viewport_offset_and_pitch(gpu, blue_noise, kind, fmt):
    """Rendering into big[y:y+h, x:x+w] of a larger surface (extra columns and rows, row pitch well above the frame's row) writes
    exactly that rectangle, equal to the packed frame; every other byte, row padding included, keeps the sentinel."""
    from strolle_b200.engine import OPT_ASYNC_OUTPUT
    scene = scenes.cornell(W_ODD, H_ODD)
    ea, eb = gpu.Engine(blue_noise=blue_noise), gpu.Engine(blue_noise=blue_noise)
    ca, cb = scenes.apply(ea, scene), scenes.apply(eb, scene)
    if kind == "pinned_async":
        ea.set_option(OPT_ASYNC_OUTPUT, 1)
    dt = _dtype(fmt)
    y, x = 5, 3
    for f in range(3):
        big = _surface(kind.split("_")[0], (H_ODD + 13, W_ODD + 22, 4), dt)
        want = np.zeros((H_ODD, W_ODD, 4), dt)
        ea.tick(); eb.tick()
        ea.render_camera(ca, big[y:y + H_ODD, x:x + W_ODD], fmt)
        eb.render_camera(cb, want, fmt)
        if kind == "pinned_async":
            ea.synchronize()
        rect, rest = _frame_and_rest(_host(big), y, x, H_ODD, W_ODD)
        _assert_same_bits(rect, want, f"{kind} format {fmt} frame {f + 1}")
        assert (rest == SENTINEL).all(), f"{kind} format {fmt}: {int((rest != SENTINEL).sum())} bytes outside the viewport were written"


def test_split_screen(gpu, blue_noise):
    """Two cameras of one engine (different sizes, Image and GiDiffuse) composed side by side into one CUDA surface: each rectangle is
    that camera's frame rendered alone by an engine of its own, and the gap between them keeps the sentinel."""
    from strolle_b200.engine import FORMAT_RGBA16F
    left = scenes.cornell(W_ODD, H_ODD)
    right = scenes.cornell(96, 72, mode=scenes.MODE_GI_DIFFUSE)
    rc = right["camera"]
    e = gpu.Engine(blue_noise=blue_noise)
    cl = scenes.apply(e, left)
    cr = e.create_camera(rc["mode"], rc["denoise"], rc["ref_depth"], rc["w"], rc["h"], rc["transform"], rc["projection"])
    alone_l, alone_r = gpu.Engine(blue_noise=blue_noise), gpu.Engine(blue_noise=blue_noise)
    al, ar = scenes.apply(alone_l, left), scenes.apply(alone_r, right)
    gap = 4
    for f in range(4):
        big = _surface("device", (H_ODD + 2, W_ODD + gap + rc["w"] + 1, 4), np.float16)
        e.tick(); alone_l.tick(); alone_r.tick()
        e.render_camera(cl, big[1:1 + H_ODD, 0:W_ODD], FORMAT_RGBA16F)
        e.render_camera(cr, big[2:2 + rc["h"], W_ODD + gap:W_ODD + gap + rc["w"]], FORMAT_RGBA16F)
        wl, wr = np.zeros((H_ODD, W_ODD, 4), np.float16), np.zeros((rc["h"], rc["w"], 4), np.float16)
        alone_l.render_camera(al, wl, FORMAT_RGBA16F); alone_r.render_camera(ar, wr, FORMAT_RGBA16F)
        b = _host(big)
        _assert_same_bits(b[1:1 + H_ODD, 0:W_ODD], wl, f"left camera frame {f + 1}")
        _assert_same_bits(b[2:2 + rc["h"], W_ODD + gap:W_ODD + gap + rc["w"]], wr, f"right camera frame {f + 1}")
        assert (b[:, W_ODD:W_ODD + gap].view(np.uint8) == SENTINEL).all() and (b[0].view(np.uint8) == SENTINEL).all()


# ---- row strips (st_multi) --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [2, 3])
def test_strips_into_targets(gpu, blue_noise, n):
    """st_multi_render_camera_to: every member stores its own rows into one surface with offset and pitch (on a multi-GPU box, peer
    stores into device 0 from the other devices); the rectangle holds the single-GPU frame's bytes and nothing else is written."""
    from strolle_b200.engine import FORMAT_RGBA32F, FORMAT_RGBA8_SRGB, FORMAT_RGBA16F
    w, h = 255, 400
    scene = scenes.cornell(w, h)
    one = gpu.Engine(blue_noise=blue_noise)
    grp = gpu.MultiEngine(_devices(n), blue_noise=blue_noise)
    c1, cn = scenes.apply(one, scene), scenes.apply(grp, scene)
    plan = [("device", FORMAT_RGBA16F), ("pageable", FORMAT_RGBA16F), ("device", FORMAT_RGBA8_SRGB), ("pinned", FORMAT_RGBA8_SRGB),
            ("device", FORMAT_RGBA32F), ("pageable", FORMAT_RGBA32F)]
    y, x = 7, 5
    for f, (kind, fmt) in enumerate(plan):
        dt = _dtype(fmt)
        big = _surface(kind, (h + 11, w + 9, 4), dt)
        want = np.zeros((h, w, 4), dt)
        one.tick(); grp.tick()
        one.render_camera(c1, want, fmt)
        grp.render_camera(cn, big[y:y + h, x:x + w], fmt)
        rect, rest = _frame_and_rest(_host(big), y, x, h, w)
        _assert_same_bits(rect, want, f"{n} strips, {kind} format {fmt} frame {f + 1}")
        assert (rest == SENTINEL).all(), f"{n} strips, {kind} format {fmt}: bytes outside the viewport were written"
    assert grp.peer_errors(cn) == 0


# ---- validation -------------------------------------------------------------------------------------------------------------------

def test_invalid_surfaces_are_refused(gpu, blue_noise):
    """Each malformed surface is refused with ST_ERR_INVALID before any pass runs, with nothing written; the Python wrapper refuses
    wrong dtypes, shapes and inner strides itself."""
    import torch
    from strolle_b200.engine import FORMAT_RGBA32F, FORMAT_RGBA8_SRGB, FORMAT_RGBA16F, StrolleError
    w, h = 64, 48
    scene = scenes.cornell(w, h)
    e = gpu.Engine(blue_noise=blue_noise)
    cam = scenes.apply(e, scene)
    e.tick()
    e.render_camera(cam)
    e.synchronize()
    frame_before = e.read_buffer(cam, "output")
    dev = torch.empty((h + 4, w + 4, 4), dtype=torch.float32, device="cuda:0")
    dev.view(torch.uint8).fill_(SENTINEL)
    torch.cuda.synchronize()
    p = dev.data_ptr()
    cases = [("null surface", 0, 0, FORMAT_RGBA32F), ("unknown format", p, 0, 7), ("pitch below the row", p, w * 16 - 16, FORMAT_RGBA32F),
             ("address off the pixel grid", p + 8, 0, FORMAT_RGBA32F), ("pitch off the pixel grid", p, w * 8 + 4, FORMAT_RGBA16F),
             ("address off the pixel grid (RGBA8)", p + 2, 0, FORMAT_RGBA8_SRGB)]
    for what, ptr, pitch, fmt in cases:
        with pytest.raises(StrolleError, match="error -2"):
            e.render_camera_to(cam, ptr or None, pitch, fmt)
    host = np.empty((h, w, 4), np.float32)
    host.view(np.uint8)[...] = SENTINEL
    with pytest.raises(StrolleError, match="error -2"):
        e.render_camera_to(cam, host.ctypes.data, 4, FORMAT_RGBA32F)
    e.synchronize()
    assert (dev.view(torch.uint8) == SENTINEL).all().item() and (host.view(np.uint8) == SENTINEL).all()
    assert_bits_equal(e.read_buffer(cam, "output"), frame_before, "a refused call ran no pass")
    for bad, fmt in [(np.zeros((h, w, 4), np.float32), FORMAT_RGBA16F), (np.zeros((h, w + 1, 4), np.float16), FORMAT_RGBA16F),
                     (np.zeros((h, 2 * w, 4), np.uint8)[:, ::2], FORMAT_RGBA8_SRGB), (np.zeros((h, w, 8), np.uint8)[..., :4], FORMAT_RGBA8_SRGB),
                     (torch.zeros((h, w, 4), dtype=torch.float32, device="cuda:0"), FORMAT_RGBA8_SRGB)]:
        with pytest.raises(ValueError):
            e.render_camera(cam, bad, fmt)
    assert_bits_equal(e.read_buffer(cam, "output"), frame_before, "a refused call ran no pass")
