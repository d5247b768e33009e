"""ctypes mirror of strolle::Engine (strolle/src/lib.rs:104-395) over libstrolle_b200.so.

Method names follow the reference's Engine API: insert_mesh / insert_material / insert_instance /
insert_light / update_sun / create_camera / update_camera / tick / render_camera, plus the test
hooks of include/strolle_b200.h (read_buffer, trace_closest, pass_times, ...).
"""
import ctypes as C
import numbers
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
PASS_COUNT = 27
FORMAT_RGBA32F, FORMAT_RGBA8_SRGB, FORMAT_RGBA16F = 0, 1, 2
OPT_SVGF_FAST_MATH = 1
OPT_ASYNC_OUTPUT = 2
OPT_HALO_NCCL = 3
OPT_WAVELET_TILED = 4      # bit i = à-trous iteration i runs the tile-staged (TMA) kernel
OPT_WAVELET_TILE_CFG = 5   # 4 bits per iteration: 0 32x8, 1 32x16, 2 64x4, 3 64x8 output tile
OPT_FUSE_REPROJECT = 6     # K20 for DI and GI in one launch
OPT_BVH_REUSE = 7          # graft unchanged subtrees of the previous BVH (reference behaviour)
OPT_VARIANCE_TILED = 8     # K21 window from a TMA-filled shared-memory tile
OPT_FUSED_PASSES = 11        # K5+K6, K7+K8+K9, K12+K13, K11 in K14, K15+K16+K17, preview#2+K19 as single launches
OPT_WAVELET_PAIRED = 13      # wide-stride a-trous iterations read {DI, GI} as interleaved 32-byte records (0 / 1 / 2)
OPT_STRIP_DMA = 12           # strips: gi_reservoirs[1]/[2] halos by copy engine on side streams instead of in-kernel mirror stores
OPT_STRIP_FUSED = 10         # strips: fused transport (mirror stores, neighbour flags, recompute) instead of push+barrier exchanges
OPT_SHADING_FAST_MATH = 9  # ReSTIR kernels K5-K19 from the fast-shading build (FMA + SFU approximations; traversal unchanged)
WAVELET_TILED_DEFAULT = 15   # include/strolle_b200.h ST_WAVELET_TILED_DEFAULT
STAT_WAVELET_TILED_LAUNCHES = 1
STAT_WAVELET_TILED_ERRORS = 2
STAT_BVH_GRAFTED_SUBTREES = 3
STAT_VARIANCE_TILED_LAUNCHES = 4
STAT_STRIP_PULLED_ROWS = 5
STAT_LAST_FRAME_FUSED_STRIPS = 6
STAT_STRIP_FIRST_TIMEOUT = 7
PLACE_STRIPS, PLACE_AUTO = -1, -2   # st_multi_camera_rank of a strip camera; st_multi_create_camera_on's automatic placement


class StrolleError(RuntimeError):
    pass


def lib_path():
    # STROLLE_B200_LIB: development aid, selects a tuning build of the same library (tools/occupancy_tune.py)
    return os.environ.get("STROLLE_B200_LIB") or os.path.join(_HERE, "_lib", "libstrolle_b200.so")


class _MeshTriangle(C.Structure):
    _fields_ = [("positions", C.c_float * 9), ("normals", C.c_float * 9), ("uvs", C.c_float * 6), ("tangents", C.c_float * 12)]


class _Material(C.Structure):
    _fields_ = [("base_color", C.c_float * 4), ("emissive", C.c_float * 4), ("perceptual_roughness", C.c_float), ("metallic", C.c_float),
                ("reflectance", C.c_float), ("ior", C.c_float), ("alpha_blend", C.c_int32)]


class _MaterialTextures(C.Structure):
    _fields_ = [("base_color", C.c_uint64), ("emissive", C.c_uint64), ("metallic_roughness", C.c_uint64), ("normal_map", C.c_uint64), ("mask", C.c_uint32)]


class _Light(C.Structure):
    _fields_ = [("kind", C.c_int32), ("position", C.c_float * 3), ("radius", C.c_float), ("color", C.c_float * 3), ("range", C.c_float),
                ("direction", C.c_float * 3), ("angle", C.c_float)]


class _Camera(C.Structure):
    _fields_ = [("mode", C.c_int32), ("denoise", C.c_int32), ("ref_depth", C.c_int32), ("width", C.c_uint32), ("height", C.c_uint32),
                ("transform", C.c_float * 16), ("projection", C.c_float * 16)]


_LIB = None


def load_library():
    """Loads the C-ABI library; raises if it has not been built (python -m strolle_b200.build)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise StrolleError(f"{path} is missing: build it with `python -m strolle_b200.build` (no CPU fallback exists)")
    lib = C.CDLL(path)
    P, u64, i32, u32, f32p = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint32, C.POINTER(C.c_float)
    sig = {
        "st_engine_create": [C.c_int, C.POINTER(P)], "st_engine_destroy": [P],
        "st_insert_mesh": [P, u64, C.POINTER(_MeshTriangle), C.c_size_t], "st_remove_mesh": [P, u64],
        "st_insert_material": [P, u64, C.POINTER(_Material)], "st_has_material": [P, u64], "st_remove_material": [P, u64],
        "st_insert_image": [P, u64, C.c_void_p, u32, u32], "st_remove_image": [P, u64], "st_insert_dynamic_image": [P, u64, C.c_void_p, C.c_size_t, u32, u32],
        "st_read_image": [P, u64, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)], "st_set_material_textures": [P, u64, C.POINTER(_MaterialTextures)],
        "st_insert_instance": [P, u64, u64, u64, f32p], "st_remove_instance": [P, u64],
        "st_insert_light": [P, u64, C.POINTER(_Light)], "st_remove_light": [P, u64], "st_update_sun": [P, C.c_float, C.c_float],
        "st_create_camera": [P, C.POINTER(_Camera), C.POINTER(i32)], "st_update_camera": [P, i32, C.POINTER(_Camera)], "st_delete_camera": [P, i32],
        "st_tick": [P], "st_render_camera": [P, i32, P, C.c_int], "st_copy_output": [P, i32, P, C.c_int], "st_synchronize": [P],
        "st_render_camera_to": [P, i32, P, C.c_size_t, C.c_int], "st_multi_render_camera_to": [P, i32, P, C.c_size_t, C.c_int],
        "st_render_cameras": [P, C.POINTER(i32), C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int],
        "st_set_seed_base": [P, u32], "st_set_blue_noise": [P, C.c_void_p],
        "st_read_buffer": [P, i32, C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)],
        "st_read_scene": [P, C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)],
        "st_bvh_depth": [P, C.POINTER(C.c_int)],
        "st_trace_closest": [P, C.c_void_p, C.c_size_t, C.c_void_p, f32p], "st_trace_any": [P, C.c_void_p, C.c_size_t, C.c_void_p, f32p],
        "st_device_math": [P, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t],
        "st_set_stream": [P, C.c_void_p, C.c_int], "st_set_option": [P, C.c_int, C.c_int], "st_get_stat": [P, C.c_int, C.POINTER(C.c_uint64)],
        "st_count_rays": [P, C.c_int], "st_ray_count": [P, C.POINTER(C.c_uint64), C.c_int],
        "st_nccl_unique_id": [C.c_void_p], "st_nccl_init": [P, C.c_void_p, C.c_int, C.c_int],
        "st_plan_frame": [C.POINTER(C.c_int), C.c_int, u32, C.c_int, C.c_char_p, C.c_size_t],
        "st_plan_strip_order": [C.POINTER(C.c_int), C.c_int, C.c_int, C.c_char_p, C.c_size_t],
        "st_strip_bounds": [C.c_int, C.c_int, C.POINTER(C.c_int)],
        "st_render_strips": [P, i32, P, C.c_int, C.c_int, C.c_int], "st_halo_bytes": [P, C.POINTER(C.c_uint64)],
        "st_peer_export": [P, i32, C.c_void_p], "st_peer_import": [P, i32, C.c_void_p, C.c_int, C.c_int],
        "st_peer_errors": [P, i32, C.POINTER(u32)],
        "st_mark_begin": [P], "st_mark_end": [P, f32p],
        "st_enable_timing": [P, C.c_int], "st_pass_times": [P, C.c_void_p, C.c_void_p, C.c_int], "st_wavelet_times": [P, C.c_void_p, C.c_void_p, C.c_int],
        "st_camera_set_strip": [P, i32, C.c_int, C.c_int],
        "st_buffer_device_ptr": [P, i32, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)],
        "st_frame_schedule": [P, i32, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)], "st_render_range": [P, i32, C.c_int, C.c_int],
        "st_link_local": [C.POINTER(P), C.POINTER(i32), C.c_int],
        "st_multi_create": [C.POINTER(C.c_int), C.c_int, C.POINTER(P)],
        "st_multi_insert_mesh": [P, u64, C.POINTER(_MeshTriangle), C.c_size_t], "st_multi_remove_mesh": [P, u64],
        "st_multi_insert_material": [P, u64, C.POINTER(_Material)], "st_multi_has_material": [P, u64], "st_multi_remove_material": [P, u64],
        "st_multi_insert_image": [P, u64, C.c_void_p, u32, u32], "st_multi_remove_image": [P, u64],
        "st_multi_insert_dynamic_image": [P, u64, C.c_void_p, C.c_size_t, u32, u32], "st_multi_set_material_textures": [P, u64, C.POINTER(_MaterialTextures)],
        "st_multi_insert_instance": [P, u64, u64, u64, f32p], "st_multi_remove_instance": [P, u64],
        "st_multi_insert_light": [P, u64, C.POINTER(_Light)], "st_multi_remove_light": [P, u64], "st_multi_update_sun": [P, C.c_float, C.c_float],
        "st_multi_create_camera": [P, C.POINTER(_Camera), C.POINTER(i32)], "st_multi_update_camera": [P, i32, C.POINTER(_Camera)], "st_multi_delete_camera": [P, i32],
        "st_multi_tick": [P], "st_multi_render_camera": [P, i32, P, C.c_int], "st_multi_synchronize": [P],
        "st_multi_set_option": [P, C.c_int, C.c_int], "st_multi_set_seed_base": [P, u32], "st_multi_set_blue_noise": [P, C.c_void_p],
        "st_multi_read_buffer": [P, i32, C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)], "st_multi_peer_errors": [P, i32, C.POINTER(u32)],
        "st_multi_size": [P], "st_multi_member_camera": [P, i32, C.c_int],
        "st_multi_create_camera_on": [P, C.POINTER(_Camera), C.c_int, C.POINTER(i32)], "st_multi_camera_rank": [P, i32, C.POINTER(C.c_int)],
        "st_multi_move_camera": [P, i32, C.c_int],
        "st_multi_render_cameras": [P, C.POINTER(i32), C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int],
        "st_bvh_builder_create": [C.POINTER(P)], "st_bvh_builder_read": [P, C.c_void_p, C.c_size_t],
        "st_bvh_builder_build": [P, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(u32), C.POINTER(C.c_int)],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = None if name == "st_engine_destroy" else C.c_int
    lib.st_bvh_builder_destroy.argtypes = [P]
    lib.st_bvh_builder_destroy.restype = None
    lib.st_multi_destroy.argtypes = [P]
    lib.st_multi_destroy.restype = None
    lib.st_multi_engine.argtypes = [P, C.c_int]
    lib.st_multi_engine.restype = P
    lib.st_last_error.restype = C.c_char_p
    lib.st_pass_name.restype = C.c_char_p
    lib.st_pass_name.argtypes = [C.c_int]
    lib.st_frame.restype = C.c_uint32
    lib.st_frame.argtypes = [P]
    lib.st_set_frame.argtypes = [P, u32]
    lib.st_set_frame.restype = C.c_int
    _LIB = lib
    return lib


def _pass_names():
    lib = load_library()
    return [lib.st_pass_name(i).decode() for i in range(PASS_COUNT)]


class _LazyNames(list):
    def _fill(self):
        if not len(self):
            self.extend(_pass_names())

    def __getitem__(self, i):
        self._fill()
        return list.__getitem__(self, i)

    def __iter__(self):
        self._fill()
        return list.__iter__(self)


PASS_NAMES = _LazyNames()


def _f(a, n=None):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float32).reshape(-1))
    if n is not None and a.size != n:
        raise ValueError(f"expected {n} floats, got {a.size}")
    return a


class BvhBuilder:
    """The host-side BVH builder on its own (strolle/src/bvh/builder.rs + serializer.rs); needs no GPU.
    `build(prims)` takes an (n, 11) float32 array (triangle id bits, material id bits, centre, bounds min, bounds max)
    and returns the serialised float4 stream as an (m, 4) float32 array; the object keeps the previous tree, whose
    unchanged subtrees are grafted when `reuse` is true (`grafted` = how many)."""

    def __init__(self):
        self.lib = load_library()
        self._h = C.c_void_p()
        if self.lib.st_bvh_builder_create(C.byref(self._h)) != 0:
            raise StrolleError(self.lib.st_last_error().decode())
        self.grafted = 0
        self.depth = 0

    def build(self, prims, reuse=True):
        prims = np.ascontiguousarray(prims, dtype=np.float32).reshape(-1, 11)
        n = C.c_size_t(0); g = C.c_uint32(0); d = C.c_int(0)
        if self.lib.st_bvh_builder_build(self._h, prims.ctypes.data, prims.shape[0], int(reuse), None, 0, C.byref(n), C.byref(g), C.byref(d)) != 0:
            raise StrolleError(self.lib.st_last_error().decode())
        # the size query already built the tree; read it back without rebuilding (a second build would graft everything)
        out = np.zeros(n.value, dtype=np.float32)
        if self.lib.st_bvh_builder_read(self._h, out.ctypes.data, out.size) != 0:
            raise StrolleError(self.lib.st_last_error().decode())
        self.grafted, self.depth = int(g.value), int(d.value)
        return out.reshape(-1, 4)

    def close(self):
        if self._h:
            self.lib.st_bvh_builder_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_FORMAT_DTYPES = {FORMAT_RGBA32F: "float32", FORMAT_RGBA8_SRGB: "uint8", FORMAT_RGBA16F: "float16"}


class _Surface:
    """A caller's output surface: a numpy array or a torch tensor (CPU, pinned or not, or CUDA) of shape (h, w, 4) whose dtype matches
    the format, last two dimensions contiguous, any row stride.  `ptr` = address of pixel (0, 0), `pitch` = bytes between rows."""

    def __init__(self, out, fmt, size):
        if hasattr(out, "data_ptr"):   # torch.Tensor
            dtype, itemsize = str(out.dtype).replace("torch.", ""), out.element_size()
            self.ptr, self.cuda = out.data_ptr(), out.is_cuda
            shape, strides = tuple(out.shape), tuple(st * itemsize for st in out.stride())
            self.device = out.device if out.is_cuda else None
        else:
            out = out if isinstance(out, np.ndarray) else np.asarray(out)
            dtype, itemsize = out.dtype.name, out.itemsize
            self.ptr, self.cuda, self.device = out.ctypes.data, False, None
            shape, strides = out.shape, out.strides
        want = _FORMAT_DTYPES.get(fmt)
        if want is not None and dtype != want:
            raise ValueError(f"output format {fmt} needs a {want} surface, got {dtype}")
        if size is not None and shape != (size[1], size[0], 4):
            raise ValueError(f"output surface must have shape (h, w, 4) = {(size[1], size[0], 4)}, got {shape}")
        if len(shape) != 3 or shape[2] != 4 or strides[2] != itemsize or strides[1] != 4 * itemsize:
            raise ValueError(f"output surface must have contiguous pixels and channels (strides (*, {4 * itemsize}, {itemsize}) bytes), got strides {strides}")
        if strides[0] < 0:
            raise ValueError(f"output surface rows must run forward in memory, got a row stride of {strides[0]} bytes")
        self.pitch = strides[0]
        self.packed = strides[0] == shape[1] * 4 * itemsize

    def render(self, fn_packed, fn_to, synchronize):
        """Host surfaces without row padding go through the packed entry point; everything else through the *_to one.  A CUDA surface
        is ordered after the torch work queued on it before the engine writes, and holds the frame when this returns."""
        if not self.cuda and self.packed:
            return fn_packed(self.ptr)
        if self.cuda:
            import torch
            torch.cuda.current_stream(self.device).synchronize()
        fn_to(self.ptr, self.pitch)
        if self.cuda:
            synchronize()


def _render_cameras(render, synchronize, sizes, cams, outs, fmt):
    """The Python side of st_render_cameras / st_multi_render_cameras: checks every surface, orders the torch work queued on the CUDA ones
    before the call `render(handles, n, dsts, pitches)`, and returns once they hold their frames."""
    cams = [int(c) for c in cams]
    n = len(cams)
    if outs is not None and len(outs) != n:
        raise ValueError(f"{n} cameras but {len(outs)} output surfaces")
    surfaces = [None if o is None else _Surface(o, fmt, sizes.get(c)) for c, o in zip(cams, outs or [None] * n)]
    handles = (C.c_int32 * max(n, 1))(*cams)
    dsts = (C.c_void_p * max(n, 1))(*[s.ptr if s is not None else None for s in surfaces])
    pitches = (C.c_size_t * max(n, 1))(*[s.pitch if s is not None else 0 for s in surfaces])
    cuda = [s for s in surfaces if s is not None and s.cuda]
    if cuda:
        import torch
        for d in {s.device for s in cuda}:
            torch.cuda.current_stream(d).synchronize()
    render(handles, n, dsts if outs is not None else None, pitches)
    if cuda:
        synchronize()


def _dynamic_source(surface):
    """A dynamic image's surface: a torch uint8 tensor of shape (h, w, 4) on CUDA or in pinned host memory, pixels and channels
    contiguous, any row stride (e.g. a slice of a larger tensor).  Returns the checked `_Surface`."""
    if not hasattr(surface, "data_ptr"):
        raise TypeError(f"a dynamic image's surface must be a torch tensor on CUDA or in pinned memory, got {type(surface).__name__}; "
                        "pass host pixels to insert_image instead")
    s = _Surface(surface, FORMAT_RGBA8_SRGB, None)
    if not s.cuda and not surface.is_pinned():
        raise ValueError("a dynamic image's surface must be on CUDA or in pinned memory (the engine reads it at every tick); "
                         "pass pageable pixels to insert_image instead")
    return s


def _order_dynamic_sources(dynamic):
    """Before a tick reads the dynamic surfaces: the torch work queued on them (current stream of every device holding one; for pinned
    sources, of the current device) must be done."""
    if not dynamic:
        return
    import torch
    devices = {t.device for t in dynamic.values() if t.is_cuda}
    if any(not t.is_cuda for t in dynamic.values()):
        devices.add(torch.device("cuda", torch.cuda.current_device()))
    for d in devices:
        torch.cuda.current_stream(d).synchronize()


class Engine:
    """strolle::Engine on one B200 (CUDA device `device`)."""

    def __init__(self, device=0, blue_noise=None, seed_base=0xC0FFEE, exact=False):
        """`exact=True` switches the SVGF weights and the ReSTIR shading kernels to strict IEEE arithmetic (bit-identical to the CPU oracle)."""
        self.lib = load_library()
        h = C.c_void_p()
        self._h = None
        self._check(self.lib.st_engine_create(device, C.byref(h)))
        self._h = h
        if blue_noise is None:
            from . import scenes
            blue_noise = scenes.blue_noise()
        bn = np.ascontiguousarray(blue_noise, dtype=np.uint8).reshape(-1)
        self._check(self.lib.st_set_blue_noise(self._h, bn.ctypes.data))
        self._check(self.lib.st_set_seed_base(self._h, seed_base))
        if exact:
            self.set_option(OPT_SVGF_FAST_MATH, 0)
            self.set_option(OPT_SHADING_FAST_MATH, 0)
            self.set_option(OPT_FUSED_PASSES, 0)
        self._cams = {}
        self._images = {}    # handle -> (w, h) of every image inserted here
        self._dynamic = {}   # handle -> the tensor a dynamic image refreshes from: kept alive while the engine reads it

    def _check(self, rc):
        if rc != 0:
            raise StrolleError(f"strolle_b200 error {rc}: {self.lib.st_last_error().decode()}")

    def close(self):
        if self._h:
            self.lib.st_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- scene ------------------------------------------------------------------------------
    def insert_mesh(self, handle, triangles36):
        t = _f(triangles36)
        n = t.size // 36
        self._check(self.lib.st_insert_mesh(self._h, handle, t.ctypes.data_as(C.POINTER(_MeshTriangle)), n))

    def insert_material(self, handle, params12, alpha_blend=False):
        p = _f(params12, 12)
        m = _Material((C.c_float * 4)(*p[0:4]), (C.c_float * 4)(*p[4:8]), p[8], p[9], p[10], p[11], int(alpha_blend))
        self._check(self.lib.st_insert_material(self._h, handle, C.byref(m)))

    def insert_image(self, handle, rgba8):
        a = np.ascontiguousarray(rgba8, dtype=np.uint8)
        self._check(self.lib.st_insert_image(self._h, handle, a.ctypes.data, a.shape[1], a.shape[0]))
        self._images[handle] = (a.shape[1], a.shape[0])
        self._dynamic.pop(handle, None)

    def insert_dynamic_image(self, handle, surface):
        """ImageData::Texture { is_dynamic: true }: every `tick()` copies `surface` into the image's atlas rectangle, so cameras rendered after
        the tick see what the surface held then (e.g. another camera's `render_camera(out=surface, fmt=FORMAT_RGBA8_SRGB)` of the frame
        before).  `surface`: a torch uint8 tensor (h, w, 4) of Rgba8UnormSrgb texels on CUDA or in pinned memory, any row stride.  The
        engine keeps a reference to it until `remove_image`, `insert_image` or another `insert_dynamic_image` on the handle."""
        s = _dynamic_source(surface)
        h, w = int(surface.shape[0]), int(surface.shape[1])
        self._check(self.lib.st_insert_dynamic_image(self._h, handle, s.ptr, s.pitch, w, h))
        self._images[handle] = (w, h)
        self._dynamic[handle] = surface

    def remove_image(self, handle):
        self._check(self.lib.st_remove_image(self._h, handle))
        self._images.pop(handle, None)
        self._dynamic.pop(handle, None)

    def read_image(self, handle):
        """The image's atlas rectangle as an (h, w, 4) uint8 array, after the work queued on the engine."""
        w, h = self._images[handle]
        out = np.empty((h, w, 4), dtype=np.uint8)
        n = C.c_size_t()
        self._check(self.lib.st_read_image(self._h, handle, out.ctypes.data, out.nbytes, C.byref(n)))
        return out

    def set_material_textures(self, handle, base_color=None, emissive=None, metallic_roughness=None, normal_map=None):
        t = [base_color, emissive, metallic_roughness, normal_map]
        mask = sum((1 << i) for i, v in enumerate(t) if v is not None)
        mt = _MaterialTextures(*[v or 0 for v in t], mask)
        self._check(self.lib.st_set_material_textures(self._h, handle, C.byref(mt)))

    def insert_instance(self, handle, mesh, material, affine12):
        a = _f(affine12, 12)
        self._check(self.lib.st_insert_instance(self._h, handle, mesh, material, a.ctypes.data_as(C.POINTER(C.c_float))))

    def remove_instance(self, handle):
        self._check(self.lib.st_remove_instance(self._h, handle))

    def insert_light(self, handle, kind, params12):
        p = _f(params12, 12)
        l = _Light(kind, (C.c_float * 3)(*p[0:3]), p[3], (C.c_float * 3)(*p[4:7]), p[7], (C.c_float * 3)(*p[8:11]), p[11])
        self._check(self.lib.st_insert_light(self._h, handle, C.byref(l)))

    def remove_light(self, handle):
        self._check(self.lib.st_remove_light(self._h, handle))

    def update_sun(self, azimuth, altitude):
        self._check(self.lib.st_update_sun(self._h, azimuth, altitude))

    # ---- cameras ----------------------------------------------------------------------------
    @staticmethod
    def _cam(mode, denoise, ref_depth, w, h, transform16, projection16):
        return _Camera(mode, int(denoise), ref_depth, w, h, (C.c_float * 16)(*_f(transform16, 16)), (C.c_float * 16)(*_f(projection16, 16)))

    def create_camera(self, mode, denoise, ref_depth, w, h, transform16, projection16):
        c = self._cam(mode, denoise, ref_depth, w, h, transform16, projection16)
        out = C.c_int32()
        self._check(self.lib.st_create_camera(self._h, C.byref(c), C.byref(out)))
        self._cams[out.value] = (w, h)
        return out.value

    def update_camera(self, cam, mode, denoise, ref_depth, w, h, transform16, projection16):
        c = self._cam(mode, denoise, ref_depth, w, h, transform16, projection16)
        self._check(self.lib.st_update_camera(self._h, cam, C.byref(c)))
        self._cams[cam] = (w, h)

    def set_strip(self, cam, y0, y1):
        self._check(self.lib.st_camera_set_strip(self._h, cam, y0, y1))

    # ---- frame ------------------------------------------------------------------------------
    def tick(self):
        _order_dynamic_sources(self._dynamic)
        self._check(self.lib.st_tick(self._h))

    def render_camera(self, cam, out=None, fmt=FORMAT_RGBA32F):
        """Runs the frame's passes.  With `out` the composed frame is stored there in format `fmt`: a numpy array or torch tensor of shape
        (h, w, 4) and dtype float32 / uint8 / float16 (FORMAT_RGBA32F / FORMAT_RGBA8_SRGB / FORMAT_RGBA16F), in host memory or on a CUDA
        device, with any row stride; `out=big[y:y + h, x:x + w]` composes into a viewport of a larger surface and leaves the rest of it
        untouched.  A CUDA `out` holds the frame when this returns."""
        if out is None:
            self._check(self.lib.st_render_camera(self._h, cam, None, fmt))
            return
        _Surface(out, fmt, self._cams.get(cam)).render(lambda p: self._check(self.lib.st_render_camera(self._h, cam, p, fmt)),
                                                       lambda p, pitch: self._check(self.lib.st_render_camera_to(self._h, cam, p, pitch, fmt)),
                                                       self.synchronize)

    def render_cameras(self, cams, outs=None, fmt=FORMAT_RGBA32F):
        """Renders the cameras `cams` for this frame; cameras of one size, mode, denoise and ref_depth run as one launch per pass.  Each
        camera's buffers and output are bit for bit what `render_camera` gives when called for the cameras one after another.  `outs`:
        None, or one entry per camera, each None (no output) or a surface as `render_camera`'s `out`, in format `fmt`.  CUDA surfaces
        hold their frames when this returns."""
        _render_cameras(lambda *a: self._check(self.lib.st_render_cameras(self._h, *a, fmt)), self.synchronize, self._cams, cams, outs, fmt)

    def render_camera_to(self, cam, ptr, pitch_bytes, fmt):
        """st_render_camera_to on a raw address (pixel (0, 0) of the camera inside the surface); returns once enqueued for device memory."""
        self._check(self.lib.st_render_camera_to(self._h, cam, ptr, pitch_bytes, fmt))

    def copy_output(self, cam, out, fmt=FORMAT_RGBA32F):
        self._check(self.lib.st_copy_output(self._h, cam, out.ctypes.data, fmt))

    def render_range(self, cam, first, last):
        self._check(self.lib.st_render_range(self._h, cam, first, last))

    def frame_schedule(self, cam):
        ids = (C.c_int * 64)()
        n = C.c_int()
        self._check(self.lib.st_frame_schedule(self._h, cam, ids, 64, C.byref(n)))
        return list(ids[: n.value])

    def synchronize(self):
        self._check(self.lib.st_synchronize(self._h))

    def frame(self):
        return self.lib.st_frame(self._h)

    def set_frame(self, frame):
        self._check(self.lib.st_set_frame(self._h, frame))

    # ---- hooks ------------------------------------------------------------------------------
    def read_buffer(self, cam, name):
        n = C.c_size_t()
        self._check(self.lib.st_read_buffer(self._h, cam, name.encode(), None, 0, C.byref(n)))
        out = np.empty(n.value, dtype=np.float32)
        self._check(self.lib.st_read_buffer(self._h, cam, name.encode(), out.ctypes.data, n.value, C.byref(n)))
        return out

    def buffer_device_ptr(self, cam, name):
        p, n = C.c_void_p(), C.c_size_t()
        self._check(self.lib.st_buffer_device_ptr(self._h, cam, name.encode(), C.byref(p), C.byref(n)))
        return p.value, n.value

    def read_scene(self, name):
        n = C.c_size_t()
        self._check(self.lib.st_read_scene(self._h, name.encode(), None, 0, C.byref(n)))
        out = np.empty(n.value, dtype=np.float32)
        if n.value:
            self._check(self.lib.st_read_scene(self._h, name.encode(), out.ctypes.data, n.value, C.byref(n)))
        return out

    def bvh_depth(self):
        d = C.c_int()
        self._check(self.lib.st_bvh_depth(self._h, C.byref(d)))
        return d.value

    def trace_closest(self, rays8, return_ms=False):
        r = _f(rays8)
        n = r.size // 8
        out = np.empty(n * 12, dtype=np.float32)
        ms = C.c_float()
        self._check(self.lib.st_trace_closest(self._h, r.ctypes.data, n, out.ctypes.data, C.byref(ms)))
        out = out.reshape(n, 12)
        return (out, ms.value) if return_ms else out

    def trace_any(self, rays8, return_ms=False):
        r = _f(rays8)
        n = r.size // 8
        out = np.empty(n, dtype=np.uint32)
        ms = C.c_float()
        self._check(self.lib.st_trace_any(self._h, r.ctypes.data, n, out.ctypes.data, C.byref(ms)))
        return (out, ms.value) if return_ms else out

    def device_math(self, op, a, b=None):
        ops = {"sin": 0, "cos": 1, "acos": 2, "atan2": 3, "exp": 4, "pow": 5, "acos_approx": 6}
        a = _f(a)
        b = _f(b) if b is not None else np.zeros_like(a)
        out = np.empty_like(a)
        self._check(self.lib.st_device_math(self._h, ops[op], a.ctypes.data, b.ctypes.data, out.ctypes.data, a.size))
        return out

    def set_option(self, option, value):
        self._check(self.lib.st_set_option(self._h, option, int(value)))

    def get_stat(self, stat):
        v = C.c_uint64(0)
        self._check(self.lib.st_get_stat(self._h, int(stat), C.byref(v)))
        return int(v.value)

    def set_stream(self, cuda_stream_ptr, external=True):
        """Runs the engine on a caller-owned stream (handle 0/None = the legacy default stream)."""
        self._check(self.lib.st_set_stream(self._h, cuda_stream_ptr or None, int(external)))

    def count_rays(self, enabled=True):
        self._check(self.lib.st_count_rays(self._h, int(enabled)))

    def ray_count(self, reset=False):
        n = C.c_uint64()
        self._check(self.lib.st_ray_count(self._h, C.byref(n), int(reset)))
        return n.value

    def nccl_init(self, id128, rank, world):
        buf = (C.c_uint8 * 128)(*bytes(id128))
        self._check(self.lib.st_nccl_init(self._h, buf, rank, world))

    def peer_export(self, cam):
        buf = (C.c_uint8 * 192)()
        self._check(self.lib.st_peer_export(self._h, cam, buf))
        return bytes(buf)

    def peer_import(self, cam, handles, rank, world):
        blob = b"".join(handles)
        buf = (C.c_uint8 * len(blob))(*blob)
        self._check(self.lib.st_peer_import(self._h, cam, buf, rank, world))

    def peer_errors(self, cam):
        n = C.c_uint32()
        self._check(self.lib.st_peer_errors(self._h, cam, C.byref(n)))
        return n.value

    def render_strips(self, cam, out=None, fmt=FORMAT_RGBA32F, temporal_reach=16, gather=False):
        ptr = out.ctypes.data if out is not None else None
        self._check(self.lib.st_render_strips(self._h, cam, ptr, fmt, temporal_reach, int(gather) if gather else (1 if out is not None else 0)))

    def halo_bytes(self):
        n = C.c_uint64()
        self._check(self.lib.st_halo_bytes(self._h, C.byref(n)))
        return n.value

    def mark_begin(self):
        self._check(self.lib.st_mark_begin(self._h))

    def mark_end(self):
        ms = C.c_float()
        self._check(self.lib.st_mark_end(self._h, C.byref(ms)))
        return ms.value

    def enable_timing(self, enabled=True):
        self._check(self.lib.st_enable_timing(self._h, int(enabled)))

    def pass_times(self, reset=False):
        ms = np.zeros(PASS_COUNT, dtype=np.float32)
        launches = np.zeros(PASS_COUNT, dtype=np.uint32)
        self._check(self.lib.st_pass_times(self._h, ms.ctypes.data, launches.ctypes.data, int(reset)))
        return ms, launches

    def wavelet_times(self, reset=False):
        """K22 per à-trous iteration (stride 1, 2, 4, 8, 16): (ms[5], launches[5]) while timing is enabled."""
        ms = np.zeros(5, dtype=np.float32)
        launches = np.zeros(5, dtype=np.uint32)
        self._check(self.lib.st_wavelet_times(self._h, ms.ctypes.data, launches.ctypes.data, int(reset)))
        return ms, launches


class MultiEngine:
    """strolle::Engine over several devices of ONE process (st_multi_*): the frame is partitioned into row strips, one per
    device; same method names as `Engine`, so `scenes.apply` and the tests drive it unchanged.  `devices` may repeat an
    ordinal (several strips on one GPU: exercises the whole strip protocol on a single-GPU box)."""

    def __init__(self, devices=(0, 1), blue_noise=None, seed_base=0xC0FFEE, exact=False):
        self.lib = load_library()
        self._h = None
        arr = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        self._check(self.lib.st_multi_create(arr, len(devices), C.byref(h)))
        self._h = h
        self.n = len(devices)
        self._cams = {}
        self._images, self._dynamic = {}, {}   # as Engine's
        if blue_noise is None:
            from . import scenes
            blue_noise = scenes.blue_noise()
        bn = np.ascontiguousarray(blue_noise, dtype=np.uint8).reshape(-1)
        self._check(self.lib.st_multi_set_blue_noise(self._h, bn.ctypes.data))
        self._check(self.lib.st_multi_set_seed_base(self._h, seed_base))
        if exact:
            self.set_option(OPT_SVGF_FAST_MATH, 0)
            self.set_option(OPT_SHADING_FAST_MATH, 0)
            self.set_option(OPT_FUSED_PASSES, 0)

    _check = Engine._check

    def close(self):
        if self._h:
            self.lib.st_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def member(self, rank):
        """Borrowed `Engine` view of member `rank` (statistics, per-strip buffers, the buffers of the cameras placed there under their member
        handles, `member_camera`); do not close it."""
        e = Engine.__new__(Engine)
        e.lib, e._h, e._cams = self.lib, C.c_void_p(self.lib.st_multi_engine(self._h, rank)), {}
        e._images, e._dynamic = self._images, {}
        e.close = lambda: None
        return e

    def member_camera(self, cam, rank):
        return self.lib.st_multi_member_camera(self._h, cam, rank)

    def insert_mesh(self, handle, triangles36):
        t = _f(triangles36)
        self._check(self.lib.st_multi_insert_mesh(self._h, handle, t.ctypes.data_as(C.POINTER(_MeshTriangle)), t.size // 36))

    def insert_material(self, handle, params12, alpha_blend=False):
        p = _f(params12, 12)
        m = _Material((C.c_float * 4)(*p[0:4]), (C.c_float * 4)(*p[4:8]), p[8], p[9], p[10], p[11], int(alpha_blend))
        self._check(self.lib.st_multi_insert_material(self._h, handle, C.byref(m)))

    def insert_image(self, handle, rgba8):
        a = np.ascontiguousarray(rgba8, dtype=np.uint8)
        self._check(self.lib.st_multi_insert_image(self._h, handle, a.ctypes.data, a.shape[1], a.shape[0]))
        self._images[handle] = (a.shape[1], a.shape[0])
        self._dynamic.pop(handle, None)

    def insert_dynamic_image(self, handle, surface):
        """As `Engine.insert_dynamic_image`; every member refreshes its own atlas from `surface`, which every member's device must reach."""
        s = _dynamic_source(surface)
        h, w = int(surface.shape[0]), int(surface.shape[1])
        self._check(self.lib.st_multi_insert_dynamic_image(self._h, handle, s.ptr, s.pitch, w, h))
        self._images[handle] = (w, h)
        self._dynamic[handle] = surface

    def remove_image(self, handle):
        self._check(self.lib.st_multi_remove_image(self._h, handle))
        self._images.pop(handle, None)
        self._dynamic.pop(handle, None)

    def read_image(self, handle, rank=0):
        """Member `rank`'s atlas rectangle of the image (every member holds the same texels)."""
        return self.member(rank).read_image(handle)

    def set_material_textures(self, handle, base_color=None, emissive=None, metallic_roughness=None, normal_map=None):
        t = [base_color, emissive, metallic_roughness, normal_map]
        mask = sum((1 << i) for i, v in enumerate(t) if v is not None)
        mt = _MaterialTextures(*[v or 0 for v in t], mask)
        self._check(self.lib.st_multi_set_material_textures(self._h, handle, C.byref(mt)))

    def insert_instance(self, handle, mesh, material, affine12):
        a = _f(affine12, 12)
        self._check(self.lib.st_multi_insert_instance(self._h, handle, mesh, material, a.ctypes.data_as(C.POINTER(C.c_float))))

    def remove_instance(self, handle):
        self._check(self.lib.st_multi_remove_instance(self._h, handle))

    def insert_light(self, handle, kind, params12):
        p = _f(params12, 12)
        l = _Light(kind, (C.c_float * 3)(*p[0:3]), p[3], (C.c_float * 3)(*p[4:7]), p[7], (C.c_float * 3)(*p[8:11]), p[11])
        self._check(self.lib.st_multi_insert_light(self._h, handle, C.byref(l)))

    def remove_light(self, handle):
        self._check(self.lib.st_multi_remove_light(self._h, handle))

    def update_sun(self, azimuth, altitude):
        self._check(self.lib.st_multi_update_sun(self._h, azimuth, altitude))

    def _rank(self, rank, what):
        if rank == "auto":
            return PLACE_AUTO
        if isinstance(rank, bool) or not isinstance(rank, numbers.Integral):
            raise TypeError(f"{what}: rank must be a member index or \"auto\", got {rank!r}")
        if not 0 <= rank < self.n:
            raise ValueError(f"{what}: rank {rank} is not a member of this group of {self.n}")
        return int(rank)

    def create_camera(self, mode, denoise, ref_depth, w, h, transform16, projection16, rank=None):
        """`rank=None`: a strip camera, rows split across every member.  An int or "auto": the camera lives whole on that member (view
        parallelism; "auto" = the member with the fewest pixels of placed cameras, the lowest rank on a tie)."""
        c = Engine._cam(mode, denoise, ref_depth, w, h, transform16, projection16)
        out = C.c_int32()
        if rank is None:
            self._check(self.lib.st_multi_create_camera(self._h, C.byref(c), C.byref(out)))
        else:
            self._check(self.lib.st_multi_create_camera_on(self._h, C.byref(c), self._rank(rank, "create_camera"), C.byref(out)))
        self._cams[out.value] = (w, h)
        return out.value

    def camera_rank(self, cam):
        """The member a placed camera lives on, or PLACE_STRIPS for a strip camera."""
        r = C.c_int()
        self._check(self.lib.st_multi_camera_rank(self._h, cam, C.byref(r)))
        return r.value

    def move_camera(self, cam, rank):
        """Moves a placed camera with all of its temporal state to member `rank`; its next frame is the one it would have rendered where
        it was."""
        self._check(self.lib.st_multi_move_camera(self._h, cam, self._rank(rank, "move_camera")))

    def update_camera(self, cam, mode, denoise, ref_depth, w, h, transform16, projection16):
        c = Engine._cam(mode, denoise, ref_depth, w, h, transform16, projection16)
        self._check(self.lib.st_multi_update_camera(self._h, cam, C.byref(c)))
        self._cams[cam] = (w, h)

    def tick(self):
        _order_dynamic_sources(self._dynamic)
        self._check(self.lib.st_multi_tick(self._h))

    def render_camera(self, cam, out=None, fmt=FORMAT_RGBA32F):
        """As `Engine.render_camera`; every member stores its own rows of the frame into `out`."""
        if out is None:
            self._check(self.lib.st_multi_render_camera(self._h, cam, None, fmt))
            return
        _Surface(out, fmt, self._cams.get(cam)).render(lambda p: self._check(self.lib.st_multi_render_camera(self._h, cam, p, fmt)),
                                                       lambda p, pitch: self._check(self.lib.st_multi_render_camera_to(self._h, cam, p, pitch, fmt)),
                                                       self.synchronize)

    def render_cameras(self, cams, outs=None, fmt=FORMAT_RGBA32F):
        """As `Engine.render_cameras`, for cameras placed on members of the group: every member renders its cameras of the list as batched
        groups, all members at once.  Each camera's buffers and output are bit for bit what one `Engine` gives for it.  A CUDA surface may
        be on any device the camera's member reaches; every one holds its frame when this returns."""
        _render_cameras(lambda *a: self._check(self.lib.st_multi_render_cameras(self._h, *a, fmt)), self.synchronize, self._cams, cams, outs, fmt)

    def render_camera_to(self, cam, ptr, pitch_bytes, fmt):
        self._check(self.lib.st_multi_render_camera_to(self._h, cam, ptr, pitch_bytes, fmt))

    def synchronize(self):
        self._check(self.lib.st_multi_synchronize(self._h))

    def set_option(self, option, value):
        self._check(self.lib.st_multi_set_option(self._h, option, int(value)))

    def read_buffer(self, cam, name):
        """The whole frame's buffer, each strip read from the member that owns it."""
        n = C.c_size_t()
        self._check(self.lib.st_multi_read_buffer(self._h, cam, name.encode(), None, 0, C.byref(n)))
        out = np.empty(n.value, dtype=np.float32)
        self._check(self.lib.st_multi_read_buffer(self._h, cam, name.encode(), out.ctypes.data, n.value, C.byref(n)))
        return out

    def peer_errors(self, cam):
        n = C.c_uint32()
        self._check(self.lib.st_multi_peer_errors(self._h, cam, C.byref(n)))
        return n.value


def nccl_unique_id():
    lib = load_library()
    buf = (C.c_uint8 * 128)()
    rc = lib.st_nccl_unique_id(buf)
    if rc != 0:
        raise StrolleError(lib.st_last_error().decode())
    return bytes(buf)


def strip_bounds_native(height, world):
    """The engine's row partition [(y0, y1), ...] (st_strip_bounds; no GPU needed) — multigpu.strip_bounds must agree."""
    lib = load_library()
    out = (C.c_int * (2 * world))()
    if lib.st_strip_bounds(int(height), int(world), out) != 0:
        raise StrolleError(lib.st_last_error().decode())
    return [(out[2 * r], out[2 * r + 1]) for r in range(world)]


def plan_strip_order(schedule, dma=True, still=False):
    """The fused strip transport's op order for a pass schedule, as a list of strings (st_plan_strip_order; no GPU needed).
    `dma`: ST_OPT_STRIP_DMA (0 / False, 1 / True, 2); `still`: the order of a frame on which neither the camera nor an instance moved."""
    lib = load_library()
    arr = (C.c_int * len(schedule))(*schedule)
    out = C.create_string_buffer(8192)
    rc = lib.st_plan_strip_order(arr, len(schedule), (int(dma) & 3) | (4 if still else 0), out, 8192)
    if rc != 0:
        raise StrolleError(lib.st_last_error().decode())
    return [x for x in out.value.decode().split(";") if x]


def plan_frame_native(schedule, frame, temporal_reach=16):
    """The engine's C++ exchange plan as [(before_step, name, reach), ...] (for tests against multigpu.plan_frame)."""
    lib = load_library()
    arr = (C.c_int * len(schedule))(*schedule)
    out = C.create_string_buffer(8192)
    rc = lib.st_plan_frame(arr, len(schedule), frame, temporal_reach, out, 8192)
    if rc != 0:
        raise StrolleError(lib.st_last_error().decode())
    items = [x for x in out.value.decode().split(";") if x]
    return [(int(a), b, int(c)) for a, b, c in (i.split(":") for i in items)]
