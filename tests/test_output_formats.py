"""Output formats and caller-owned surfaces without a device: the Rust crates agree with the C header's formats, the Bevy node composes
in the view's format through the reference's graph, and the Python wrapper turns a strided view into an address and a row pitch."""
import os
import re

import numpy as np
import pytest

from strolle_b200 import engine as st

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BYTES_PER_PIXEL = {"RGBA32F": 16, "RGBA8_SRGB": 4, "RGBA16F": 8}   # include/strolle_b200.h, next to the format enum


def _read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def _header_formats():
    text = re.sub(r"/\*.*?\*/", "", _read("include", "strolle_b200.h"), flags=re.S)
    return dict(re.findall(r"ST_FORMAT_(\w+)\s*=\s*(\d+)", text))


def _match_arms(src, fn):
    body = re.search(r"fn %s\(self\)[^{]*\{\s*match self \{(.*?)\}" % fn, src, flags=re.S).group(1)
    return dict(re.findall(r"Self::(\w+)\s*=>\s*([\w:]+)", body))


def test_every_header_format_has_a_viewport_format():
    formats = _header_formats()
    assert set(formats) == set(BYTES_PER_PIXEL) and formats["RGBA16F"] == "2"
    src = _read("rust", "strolle-b200", "src", "lib.rs")
    variants = re.search(r"pub enum ViewportFormat \{(.*?)\}", src, flags=re.S).group(1)
    variants = re.findall(r"(\w+),", variants)
    bpp, ffi = _match_arms(src, "bytes_per_pixel"), _match_arms(src, "to_ffi")
    assert set(bpp) == set(ffi) == set(variants)
    for name in formats:
        owners = [v for v in variants if ffi[v] == f"sys::ST_FORMAT_{name}"]
        assert len(owners) == 1, f"ST_FORMAT_{name} needs exactly one ViewportFormat variant"
        assert int(bpp[owners[0]]) == BYTES_PER_PIXEL[name], f"ViewportFormat::{owners[0]}"
    assert ffi["Rgba16Float"] == "sys::ST_FORMAT_RGBA16F" and bpp["Rgba16Float"] == "8"


def test_bevy_graph_follows_the_reference_and_composes_in_the_view_format():
    lib = _read("rust", "bevy-strolle-b200", "src", "lib.rs")
    edges = re.search(r"add_render_graph_edges\(graph::NAME,\s*&\[(.*?)\]\)", lib, flags=re.S).group(1)
    assert re.findall(r"graph::node::(\w+)", edges) == ["RENDERING", "FXAA", "TONEMAPPING", "UPSCALING"]
    for node in ("TonemappingNode", "FxaaNode", "UpscalingNode", "RenderingNode"):
        assert f"ViewNodeRunner<{node}>" in lib, node
    for f in os.listdir(os.path.join(ROOT, "rust", "bevy-strolle-b200", "src")):
        assert "Rgba32Float" not in _read("rust", "bevy-strolle-b200", "src", f), f"{f} hard-codes Rgba32Float"
    assert "main_texture_format()" in _read("rust", "bevy-strolle-b200", "src", "sync.rs")


def test_render_camera_to_raw_forwards_to_the_group_entry_point():
    src = _read("rust", "strolle-b200", "src", "lib.rs")
    m = re.search(r"pub unsafe fn render_camera_to_raw\b.*?\n    }\n", src, flags=re.S)
    assert m and "sys::st_multi_render_camera_to(" in m.group(0)
    assert "pub fn st_multi_render_camera_to(" in _read("rust", "strolle-b200-sys", "src", "lib.rs")


@pytest.mark.parametrize("fmt,dtype", [(st.FORMAT_RGBA32F, np.float32), (st.FORMAT_RGBA8_SRGB, np.uint8), (st.FORMAT_RGBA16F, np.float16)])
def test_viewport_view_gives_address_and_pitch(fmt, dtype):
    w, h, y, x = 13, 7, 3, 5
    big = np.zeros((h + 6, w + 9, 4), dtype)
    s = st._Surface(big[y:y + h, x:x + w], fmt, (w, h))
    bpp = 4 * np.dtype(dtype).itemsize
    assert s.pitch == (w + 9) * bpp and s.ptr == big.ctypes.data + y * s.pitch + x * bpp and not s.cuda and not s.packed
    assert st._Surface(np.zeros((h, w, 4), dtype), fmt, (w, h)).packed


@pytest.mark.parametrize("bad,fmt", [(np.zeros((7, 13, 4), np.float32), st.FORMAT_RGBA16F),          # dtype of another format
                                     (np.zeros((7, 14, 4), np.float16), st.FORMAT_RGBA16F),          # not the camera's size
                                     (np.zeros((7, 13, 3), np.float32), st.FORMAT_RGBA32F),          # not 4 channels
                                     (np.zeros((7, 26, 4), np.uint8)[:, ::2], st.FORMAT_RGBA8_SRGB),  # pixels not contiguous
                                     (np.zeros((7, 13, 8), np.uint8)[..., :4], st.FORMAT_RGBA8_SRGB),  # channels padded
                                     (np.zeros((7, 13, 4), np.uint8)[::-1], st.FORMAT_RGBA8_SRGB)])  # rows backwards
def test_malformed_surfaces_are_refused_in_python(bad, fmt):
    with pytest.raises(ValueError):
        st._Surface(bad, fmt, (13, 7))
