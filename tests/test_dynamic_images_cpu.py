"""Engine.insert_dynamic_image checks its surface in Python, before the library is called (no GPU needed)."""
import numpy as np
import pytest
import torch


class _Lib:
    def __init__(self, calls):
        self.calls = calls

    def st_insert_dynamic_image(self, *args):
        self.calls.append(("insert", args))
        return 0

    def st_remove_image(self, *args):
        self.calls.append(("remove", args))
        return 0


def _engine(calls):
    from strolle_b200.engine import Engine
    e = Engine.__new__(Engine)
    e.lib, e._h, e._cams, e._images, e._dynamic = _Lib(calls), None, {}, {}, {}
    return e


class _CudaLike:
    """Stands for a CUDA uint8 tensor (what a GPU-less box cannot allocate): a CPU tensor that reports itself on cuda:0."""

    def __init__(self, t):
        self.t, self.dtype, self.shape, self.is_cuda, self.device = t, t.dtype, t.shape, True, torch.device("cuda", 0)

    def data_ptr(self):
        return self.t.data_ptr()

    def element_size(self):
        return self.t.element_size()

    def stride(self):
        return self.t.stride()


@pytest.mark.parametrize("surface, error, match", [
    (np.zeros((4, 8, 4), np.uint8), TypeError, "insert_image"),                                     # numpy: host pixels go to insert_image
    (torch.zeros((4, 8, 4), dtype=torch.uint8), ValueError, "insert_image"),                        # pageable tensor
    (_CudaLike(torch.zeros((4, 8, 4), dtype=torch.float32)), ValueError, "uint8"),                 # another dtype
    (_CudaLike(torch.zeros((4, 8, 3), dtype=torch.uint8)), ValueError, "shape|strides"),           # three channels
    (_CudaLike(torch.zeros((4, 8), dtype=torch.uint8)), ValueError, "shape|strides"),              # not (h, w, 4)
    (_CudaLike(torch.zeros((4, 8, 8), dtype=torch.uint8)[:, :, ::2]), ValueError, "contiguous"),   # channels not contiguous
    (_CudaLike(torch.zeros((4, 16, 4), dtype=torch.uint8)[:, ::2]), ValueError, "contiguous"),     # pixels not contiguous
])
def test_bad_surfaces_are_refused_before_the_call(surface, error, match):
    calls = []
    e = _engine(calls)
    with pytest.raises(error, match=match):
        e.insert_dynamic_image(5, surface)
    assert not calls and not e._dynamic


def test_surface_reaches_the_call_and_is_kept_until_removed():
    calls = []
    e = _engine(calls)
    big = torch.zeros((10, 20, 4), dtype=torch.uint8)
    view = _CudaLike(big[2:6, 3:11])
    e.insert_dynamic_image(5, view)
    (what, (_, handle, ptr, pitch, w, h)), = calls
    assert what == "insert" and handle == 5 and ptr == big[2:6, 3:11].data_ptr() and pitch == 20 * 4 and (w, h) == (8, 4)
    assert e._dynamic[5] is view and e._images[5] == (8, 4)
    e.remove_image(5)
    assert calls[-1][0] == "remove" and 5 not in e._dynamic and 5 not in e._images
