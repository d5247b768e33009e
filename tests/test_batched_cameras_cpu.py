"""Engine.render_cameras checks its arguments in Python, before the library is called (no GPU needed)."""
import numpy as np
import pytest


def _engine(calls):
    from strolle_b200.engine import Engine

    class Lib:
        def st_render_cameras(self, *args):
            calls.append(args)
            return 0

    e = Engine.__new__(Engine)
    e.lib, e._h, e._cams = Lib(), None, {0: (8, 4), 1: (8, 4)}
    return e


@pytest.mark.parametrize("outs", [
    [np.zeros((4, 8, 4), np.float32)],                                            # one surface for two cameras
    [None, np.zeros((4, 8, 4), np.uint8)],                                        # dtype of another format
    [None, np.zeros((4, 7, 4), np.float32)],                                      # wrong shape
    [None, np.zeros((4, 8, 8), np.float32)[:, :, ::2]],                           # channels not contiguous
])
def test_bad_surfaces_are_refused_before_the_call(outs):
    calls = []
    with pytest.raises(ValueError):
        _engine(calls).render_cameras([0, 1], outs)
    assert not calls


def test_surfaces_reach_the_call():
    calls = []
    big = np.zeros((10, 20, 4), np.float32)
    _engine(calls).render_cameras([0, 1], [None, big[2:6, 3:11]])
    (_, handles, n, dsts, pitches, fmt), = calls
    assert n == 2 and list(handles[:2]) == [0, 1] and fmt == 0
    assert dsts[0] is None and dsts[1] == big[2:6, 3:11].ctypes.data
    assert pitches[1] == 20 * 16
