"""View-parallel groups without a GPU: MultiEngine's placement and render_cameras argument checks happen in Python before the library is
called, and the Rust binding routes batched rendering of any group through st_multi_render_cameras."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Lib:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append((name, args))
            return 0
        return call


def _group(n=3):
    from strolle_b200.engine import MultiEngine
    g = MultiEngine.__new__(MultiEngine)
    g.lib, g._h, g.n, g._cams = _Lib(), None, n, {0: (8, 4), 1: (8, 4)}
    return g


def _create(g, rank):
    return g.create_camera(0, True, 1, 8, 4, np.eye(4, dtype=np.float32).reshape(-1), np.eye(4, dtype=np.float32).reshape(-1), rank=rank)


@pytest.mark.parametrize("rank,entry,arg", [(None, "st_multi_create_camera", None), (0, "st_multi_create_camera_on", 0),
                                            (2, "st_multi_create_camera_on", 2), (np.int64(1), "st_multi_create_camera_on", 1),
                                            ("auto", "st_multi_create_camera_on", -2)])
def test_create_camera_placement(rank, entry, arg):
    g = _group()
    _create(g, rank)
    (name, args), = g.lib.calls
    assert name == entry
    if arg is not None:
        assert args[2] == arg and type(args[2]) is int


@pytest.mark.parametrize("rank,exc", [(3, ValueError), (-1, ValueError), (-2, ValueError), ("Auto", TypeError), (True, TypeError), (1.0, TypeError)])
def test_bad_ranks_are_refused_before_the_call(rank, exc):
    g = _group()
    with pytest.raises(exc):
        _create(g, rank)
    with pytest.raises(exc):
        g.move_camera(0, rank)
    assert not g.lib.calls


def test_move_camera_reaches_the_call():
    g = _group()
    g.move_camera(1, 2)
    assert g.lib.calls == [("st_multi_move_camera", (None, 1, 2))]


@pytest.mark.parametrize("outs", [
    [np.zeros((4, 8, 4), np.float32)],                                            # one surface for two cameras
    [None, np.zeros((4, 8, 4), np.uint8)],                                        # dtype of another format
    [None, np.zeros((4, 7, 4), np.float32)],                                      # wrong shape
    [None, np.zeros((4, 8, 8), np.float32)[:, :, ::2]],                           # channels not contiguous
])
def test_bad_surfaces_are_refused_before_the_call(outs):
    g = _group()
    with pytest.raises(ValueError):
        g.render_cameras([0, 1], outs)
    assert not g.lib.calls


def test_surfaces_reach_the_call():
    g = _group()
    big = np.zeros((10, 20, 4), np.float16)
    g.render_cameras([1, 0], [big[2:6, 3:11], None], fmt=2)
    (name, (_, handles, n, dsts, pitches, fmt)), = g.lib.calls
    assert name == "st_multi_render_cameras"
    assert n == 2 and list(handles[:2]) == [1, 0] and fmt == 2
    assert dsts[0] == big[2:6, 3:11].ctypes.data and dsts[1] is None
    assert pitches[0] == 20 * 8


def _rust_method(name):
    src = open(os.path.join(ROOT, "rust", "strolle-b200", "src", "lib.rs")).read()
    m = re.search(r"pub (?:unsafe )?fn %s\b.*?\n    }\n" % name, src, flags=re.S)
    assert m, f"Engine::{name} missing"
    return m.group(0)


def test_rust_batched_rendering_takes_any_group():
    body = _rust_method("render_cameras_to_raw")
    assert "st_multi_render_cameras(" in body
    assert "st_multi_size" not in body and "st_render_cameras(" not in body, "render_cameras_to_raw still special-cases one device"


@pytest.mark.parametrize("method,ffi", [("create_camera_on", "st_multi_create_camera_on"), ("move_camera", "st_multi_move_camera")])
def test_rust_placement_methods(method, ffi):
    assert ffi in _rust_method(method)
    sys_src = open(os.path.join(ROOT, "rust", "strolle-b200-sys", "src", "lib.rs")).read()
    assert f"pub fn {ffi}(" in sys_src and "pub const ST_PLACE_AUTO: c_int = -2;" in sys_src
