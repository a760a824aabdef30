"""gs_b200 -- thin ctypes binding over the C ABI of libgsb200.so (include/gs_b200.h) and the
C bridge of the C++ host library libgsb200_host.so (host/gs_b200_host.h).

This is plumbing for tests and bench.py only: the product is the CUDA library + the C++ host.
There is NO fallback: if libgsb200.so is missing this module raises at import, and without a
CUDA device `Context()` raises (gsb_create -> GSB_ERR_NO_DEVICE).  Nothing here touches oracle/.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_ROOT = Path(__file__).resolve().parents[2]  # .../3dgs.cpp_b200
LIB_PATH = Path(os.environ.get("GSB200_LIB", PKG_ROOT / "libgsb200.so"))  # override only for A/B experiments
HOST_LIB_PATH = PKG_ROOT / "libgsb200_host.so"

if not LIB_PATH.exists():
    raise ImportError(f"{LIB_PATH} not built: run `python __graft_entry__.py build` (nvcc, sm_100a)")
if not HOST_LIB_PATH.exists():
    raise ImportError(f"{HOST_LIB_PATH} not built: run `python __graft_entry__.py build`")

lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_GLOBAL)
host = C.CDLL(str(HOST_LIB_PATH))

# ---- enums (gs_b200.h) ----
OK = 0
ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_NO_SCENE, ERR_OOM, ERR_OVERFLOW = -1, -2, -3, -4, -5, -6
FORMAT_RGBA32F, FORMAT_RGBA8, FORMAT_BGRA8 = 0, 1, 2
MODE_EXACT, MODE_FAST = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
(BUF_COV3D, BUF_ATTR, BUF_TILES_OVERLAP, BUF_PREFIX_SUM, BUF_KEYS_UNSORTED, BUF_VALS_UNSORTED,
 BUF_KEYS_SORTED, BUF_VALS_SORTED, BUF_TILE_BOUNDARY, BUF_DEPTH_ORDER, BUF_EMIT_OFFSETS) = range(11)
ALL_ROWS = 0xFFFFFFFF

EXPORTED_SYMBOLS = [  # every symbol include/gs_b200.h declares
    "gsb_abi_version", "gsb_device_count", "gsb_create", "gsb_destroy", "gsb_last_error",
    "gsb_scene_upload", "gsb_scene_size", "gsb_set_mode", "gsb_set_debug", "gsb_set_timers", "gsb_set_tile_cull", "gsb_set_sh_storage",
    "gsb_reserve_instances", "gsb_render", "gsb_render_aux", "gsb_render_async", "gsb_get_stats", "gsb_debug_size",
    "gsb_debug_download", "gsb_sort_pairs", "gsb_sort_pairs32", "gsb_set_graph", "gsb_host_alloc", "gsb_host_free",
    # frame sharding over several GPUs
    "gsb_group_create", "gsb_group_destroy", "gsb_group_size", "gsb_group_context", "gsb_group_last_error",
    "gsb_group_scene_upload", "gsb_group_render", "gsb_group_render_async",
    "gsb_shard_unique_id", "gsb_shard_last_error", "gsb_create_sharded", "gsb_shard_rank", "gsb_shard_world", "gsb_shard_slice",
    "gsb_shard_band", "gsb_scene_upload_sharded", "gsb_render_sharded", "gsb_render_sharded_async", "gsb_shard_frame",
]
HOST_EXPORTED_SYMBOLS = [  # host/gs_b200_host.h
    "gsh_last_error", "gsh_initialize", "gsh_draw", "gsh_pan_translation", "gsh_movement", "gsh_cleanup",
    "gsh_set_camera", "gsh_get_camera", "gsh_key_input", "gsh_render", "gsh_render_aux", "gsh_frame", "gsh_stats",
    "gsh_num_vertices", "gsh_context", "gsh_uniforms_from_camera", "gsh_camera_translate",
    "gsh_activate_records", "gsh_load_ply", "gsh_free", "gsh_write_ply", "gsh_synth_default_params",
    "gsh_synth_records",
]


class Uniforms(C.Structure):
    """gsb_uniforms == Renderer::UniformBuffer (src/Renderer.h:21-29), 160 bytes."""
    _fields_ = [("camera_position", C.c_float * 4), ("proj_mat", C.c_float * 16), ("view_mat", C.c_float * 16),
                ("width", C.c_uint32), ("height", C.c_uint32), ("tan_fovx", C.c_float), ("tan_fovy", C.c_float)]


assert C.sizeof(Uniforms) == 160


class Stats(C.Structure):
    _fields_ = [("num_gaussians", C.c_uint64), ("num_visible", C.c_uint64), ("num_instances", C.c_uint64), ("num_instances_aabb", C.c_uint64),
                ("blend_consumed", C.c_uint64), ("instance_capacity", C.c_uint64), ("sort_passes", C.c_uint32),
                ("regrow_count", C.c_uint32), ("preprocess_ms", C.c_float), ("prefix_sum_ms", C.c_float),
                ("preprocess_sort_ms", C.c_float), ("sort_ms", C.c_float), ("tile_boundary_ms", C.c_float),
                ("render_ms", C.c_float), ("frame_ms", C.c_float), ("sort_depth_ms", C.c_float),
                ("sort_tile_ms", C.c_float), ("sort_hist_ms", C.c_float), ("sort_pass_ms", C.c_float * 8),
                ("sort_depth_passes", C.c_uint32), ("pad_", C.c_uint32), ("blend_warp_visits", C.c_uint64), ("blend_pixel_hits", C.c_uint64), ("blend_staged", C.c_uint64), ("shard_blend_ms", C.c_float), ("shard_wait_ms", C.c_float)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["sort_pass_ms"] = list(self.sort_pass_ms)[:self.sort_passes]
        return d


class SynthParams(C.Structure):
    _fields_ = [("center", C.c_float * 3), ("half_extent", C.c_float * 3), ("log_scale_min", C.c_float),
                ("log_scale_max", C.c_float), ("opacity_min", C.c_float), ("opacity_max", C.c_float),
                ("sh_dc_range", C.c_float), ("sh_rest_sigma", C.c_float)]


ATTR_DTYPE = np.dtype([("conic_opacity", "<f4", 4), ("color_radii", "<f4", 4), ("aabb", "<u4", 4),
                       ("uv", "<f4", 2), ("depth", "<f4"), ("magic", "<u4")])
assert ATTR_DTYPE.itemsize == 64

_vp = C.c_void_p
lib.gsb_abi_version.restype = C.c_int
lib.gsb_device_count.restype = C.c_int
lib.gsb_create.argtypes = [C.c_int, C.POINTER(_vp)]
lib.gsb_destroy.argtypes = [_vp]
lib.gsb_destroy.restype = None
lib.gsb_last_error.argtypes = [_vp]
lib.gsb_last_error.restype = C.c_char_p
lib.gsb_scene_upload.argtypes = [_vp, _vp, C.c_uint64, C.c_int]
lib.gsb_scene_size.argtypes = [_vp]
lib.gsb_scene_size.restype = C.c_uint64
lib.gsb_set_mode.argtypes = [_vp, C.c_int]
lib.gsb_set_debug.argtypes = [_vp, C.c_int]
lib.gsb_set_timers.argtypes = [_vp, C.c_int]
lib.gsb_set_tile_cull.argtypes = [_vp, C.c_int]
lib.gsb_set_sh_storage.argtypes = [_vp, C.c_int]
lib.gsb_set_graph.argtypes = [_vp, C.c_int]
lib.gsb_host_alloc.argtypes = [C.POINTER(_vp), C.c_size_t]
lib.gsb_host_free.argtypes = [_vp]
lib.gsb_host_free.restype = None
lib.gsb_reserve_instances.argtypes = [_vp, C.c_uint64]
lib.gsb_render.argtypes = [_vp, C.POINTER(Uniforms), C.c_uint32, C.c_uint32, _vp, C.c_size_t, C.c_int, C.c_int, _vp]
lib.gsb_render_aux.argtypes = [_vp, C.POINTER(Uniforms), C.c_uint32, C.c_uint32, _vp, C.c_size_t, _vp, C.c_size_t, C.c_int,
                                C.c_int, _vp]
lib.gsb_render_async.argtypes = [_vp, C.POINTER(Uniforms), C.c_uint32, C.c_uint32, _vp, C.c_size_t, C.c_int, _vp]
lib.gsb_get_stats.argtypes = [_vp, C.POINTER(Stats)]
lib.gsb_debug_size.argtypes = [_vp, C.c_int]
lib.gsb_debug_size.restype = C.c_size_t
lib.gsb_debug_download.argtypes = [_vp, C.c_int, _vp, C.c_size_t]
lib.gsb_sort_pairs.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_uint64, C.c_uint32, _vp]
lib.gsb_sort_pairs32.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_uint64, C.c_uint32, _vp]

lib.gsb_group_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(_vp)]
lib.gsb_group_destroy.argtypes = [_vp]
lib.gsb_group_destroy.restype = None
lib.gsb_group_size.argtypes = [_vp]
lib.gsb_group_context.argtypes = [_vp, C.c_int]
lib.gsb_group_context.restype = _vp
lib.gsb_group_last_error.argtypes = [_vp]
lib.gsb_group_last_error.restype = C.c_char_p
lib.gsb_group_scene_upload.argtypes = [_vp, _vp, C.c_uint64, C.c_int]
lib.gsb_group_render.argtypes = [_vp, C.POINTER(Uniforms), _vp, C.c_size_t, C.c_int, C.c_int]
lib.gsb_group_render_async.argtypes = [_vp, C.POINTER(Uniforms), C.c_int]
lib.gsb_shard_unique_id.argtypes = [_vp]
lib.gsb_shard_last_error.restype = C.c_char_p
lib.gsb_create_sharded.argtypes = [C.c_int, C.c_int, C.c_int, _vp, C.POINTER(_vp)]
lib.gsb_shard_rank.argtypes = [_vp]
lib.gsb_shard_world.argtypes = [_vp]
lib.gsb_shard_slice.argtypes = [C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
lib.gsb_shard_band.argtypes = [_vp, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
lib.gsb_scene_upload_sharded.argtypes = [_vp, _vp, C.c_uint64, C.c_int]
lib.gsb_render_sharded.argtypes = [_vp, C.POINTER(Uniforms), _vp, C.c_size_t, C.c_int, C.c_int, _vp]
lib.gsb_render_sharded_async.argtypes = [_vp, C.POINTER(Uniforms), C.c_int, _vp]
lib.gsb_shard_frame.argtypes = [_vp]
lib.gsb_shard_frame.restype = _vp

host.gsh_last_error.restype = C.c_char_p
host.gsh_initialize.argtypes = [C.c_char_p, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_int]
host.gsh_initialize.restype = _vp
host.gsh_draw.argtypes = [_vp]
host.gsh_pan_translation.argtypes = [_vp, C.c_float, C.c_float]
host.gsh_movement.argtypes = [_vp, C.c_float, C.c_float, C.c_float]
host.gsh_key_input.argtypes = [_vp, C.POINTER(C.c_int)]
host.gsh_cleanup.argtypes = [_vp]
host.gsh_cleanup.restype = None
host.gsh_set_camera.argtypes = [_vp, _vp, _vp, C.c_float, C.c_float, C.c_float]
host.gsh_get_camera.argtypes = [_vp, _vp, _vp, C.POINTER(C.c_float)]
host.gsh_render.argtypes = [_vp, C.c_uint32, C.c_uint32, C.c_int, _vp, C.c_size_t]
host.gsh_render_aux.argtypes = [_vp, C.c_uint32, C.c_uint32, C.c_int, _vp, C.c_size_t, _vp, C.c_size_t]
host.gsh_frame.argtypes = [_vp, C.POINTER(C.c_size_t)]
host.gsh_frame.restype = _vp
host.gsh_stats.argtypes = [_vp, C.POINTER(Stats)]
host.gsh_num_vertices.argtypes = [_vp]
host.gsh_num_vertices.restype = C.c_uint64
host.gsh_context.argtypes = [_vp]
host.gsh_context.restype = _vp
host.gsh_uniforms_from_camera.argtypes = [_vp, _vp, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint32,
                                          C.POINTER(Uniforms)]
host.gsh_uniforms_from_camera.restype = None
host.gsh_camera_translate.argtypes = [_vp, _vp, _vp]
host.gsh_camera_translate.restype = None
host.gsh_activate_records.argtypes = [_vp, C.c_uint64, _vp]
host.gsh_activate_records.restype = None
host.gsh_load_ply.argtypes = [C.c_char_p, C.POINTER(C.c_uint64)]
host.gsh_load_ply.restype = C.POINTER(C.c_float)
host.gsh_free.argtypes = [_vp]
host.gsh_free.restype = None
host.gsh_write_ply.argtypes = [C.c_char_p, _vp, C.c_uint64]
host.gsh_synth_default_params.argtypes = [C.POINTER(SynthParams)]
host.gsh_synth_default_params.restype = None
host.gsh_synth_records.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(SynthParams), _vp]
host.gsh_synth_records.restype = None


class GsbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gsb error {code}: {msg}")
        self.code = code


def _f32(a, n=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if n is not None:
        assert a.size == n
    return a


# ---------------------------------------------------------------- host-only helpers (no GPU)
def uniforms_from_camera(pos, quat_wxyz, fov_deg, near, far, width, height) -> Uniforms:
    """Renderer::updateUniforms via the C++ host (src/Renderer.cpp:719-754)."""
    u = Uniforms()
    p, q = _f32(pos, 3), _f32(quat_wxyz, 4)
    host.gsh_uniforms_from_camera(p.ctypes.data, q.ctypes.data, fov_deg, near, far, width, height, C.byref(u))
    return u


def camera_translate(pos, quat_wxyz, t):
    p, q, tt = _f32(pos, 3).copy(), _f32(quat_wxyz, 4), _f32(t, 3)
    host.gsh_camera_translate(p.ctypes.data, q.ctypes.data, tt.ctypes.data)
    return p


def activate_records(records: np.ndarray) -> np.ndarray:
    rec = _f32(records).reshape(-1, 62)
    out = np.empty((rec.shape[0], 60), np.float32)
    host.gsh_activate_records(rec.ctypes.data, rec.shape[0], out.ctypes.data)
    return out


def load_ply(path) -> np.ndarray:
    n = C.c_uint64(0)
    p = host.gsh_load_ply(str(path).encode(), C.byref(n))
    if not p:
        raise RuntimeError(host.gsh_last_error().decode())
    try:
        return np.ctypeslib.as_array(p, shape=(n.value, 60)).copy() if n.value else np.empty((0, 60), np.float32)
    finally:
        host.gsh_free(p)


def write_ply(path, records: np.ndarray):
    rec = _f32(records).reshape(-1, 62)
    if host.gsh_write_ply(str(path).encode(), rec.ctypes.data, rec.shape[0]) != 0:
        raise RuntimeError(host.gsh_last_error().decode())


def synth_params(**kw) -> SynthParams:
    p = SynthParams()
    host.gsh_synth_default_params(C.byref(p))
    for k, v in kw.items():
        if k in ("center", "half_extent"):
            getattr(p, k)[:] = list(v)
        else:
            setattr(p, k, v)
    return p


def synth_records(seed: int, n: int, params: SynthParams | None = None, first: int = 0) -> np.ndarray:
    """Deterministic synthetic PLY records (n x 62 float32), SURVEY 8d."""
    params = params or synth_params()
    out = np.empty((n, 62), np.float32)
    host.gsh_synth_records(seed, first, n, C.byref(params), out.ctypes.data)
    return out


def band_for_rank(height: int, rank: int, world: int):
    """Tile-row band [begin, end) of `rank` for frame sharding (SURVEY 8e): equal-height bands of
    R = ceil(ceil(H/16) / world) tile rows (NCCL all-gather needs equal counts); trailing ranks may be
    short or empty.  Returns (begin, end, rows_per_rank)."""
    tiles_y = (height + 15) // 16
    rows_per = (tiles_y + world - 1) // world
    begin = min(tiles_y, rank * rows_per)
    return begin, min(tiles_y, begin + rows_per), rows_per


def stream_ptr(stream=None):
    """cudaStream_t of a torch stream (or None -> the context's own stream)."""
    return None if stream is None else C.c_void_p(stream.cuda_stream)


# ---------------------------------------------------------------- the C ABI context
class Context:
    """gsb_ctx wrapper.  All compute happens in libgsb200's CUDA kernels."""

    def __init__(self, device: int = 0, handle=None):
        self._own = handle is None
        if handle is None:
            h = _vp()
            rc = lib.gsb_create(device, C.byref(h))
            if rc != OK:
                raise GsbError(rc, lib.gsb_last_error(None).decode())
            handle = h
        self.h = handle
        self.device = device

    def close(self):
        if self.h and self._own:
            lib.gsb_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != OK:
            raise GsbError(rc, lib.gsb_last_error(self.h).decode())

    def upload(self, vertices):
        """vertices: (n, 60) float32 numpy array (host) or torch CUDA tensor (device)."""
        if isinstance(vertices, np.ndarray):
            v = _f32(vertices).reshape(-1, 60)
            self._ck(lib.gsb_scene_upload(self.h, v.ctypes.data, v.shape[0], MEM_HOST))
        else:  # torch tensor on this device
            assert vertices.is_cuda and vertices.is_contiguous() and vertices.dtype.itemsize == 4
            self._ck(lib.gsb_scene_upload(self.h, vertices.data_ptr(), vertices.numel() // 60, MEM_DEVICE))

    @property
    def num_gaussians(self):
        return lib.gsb_scene_size(self.h)

    def set_mode(self, mode):
        self._ck(lib.gsb_set_mode(self.h, mode))

    def set_debug(self, on=True):
        self._ck(lib.gsb_set_debug(self.h, int(on)))

    def set_tile_cull(self, level=1):
        """gsb_set_tile_cull: 0 reference lists, 1 (True) exact per-tile instance culling, 2 coarse 4x4-tile bins."""
        self._ck(lib.gsb_set_tile_cull(self.h, int(level)))

    def set_sh_storage(self, half=True):
        """gsb_set_sh_storage: fp16 SH coefficients from the next upload on (NOT a parity mode)."""
        self._ck(lib.gsb_set_sh_storage(self.h, int(half)))

    def set_timers(self, on=True):
        self._ck(lib.gsb_set_timers(self.h, int(on)))

    def set_graph(self, on=True):
        self._ck(lib.gsb_set_graph(self.h, int(on)))

    def reserve(self, capacity):
        self._ck(lib.gsb_reserve_instances(self.h, capacity))

    @staticmethod
    def band_rows(u: Uniforms, rows):
        tiles_y = (u.height + 15) // 16
        rb, re = (0, tiles_y) if rows is None else rows
        re = min(re, tiles_y)
        return rb, re, min(u.height, re * 16) - rb * 16

    def render(self, u: Uniforms, fmt=FORMAT_RGBA32F, rows=None) -> np.ndarray:
        """Render to a HOST numpy array through gsb_render (band = tile rows [rb, re))."""
        rb, re, nrows = self.band_rows(u, rows)
        out = np.empty((nrows, u.width, 4), np.float32 if fmt == FORMAT_RGBA32F else np.uint8)
        self._ck(lib.gsb_render(self.h, C.byref(u), rb, re, out.ctypes.data, 0, MEM_HOST, fmt, None))
        return out

    def render_into(self, u: Uniforms, out_ptr: int, fmt=FORMAT_RGBA32F, rows=None, stream=None, sync=True):
        """Render into DEVICE memory at out_ptr (e.g. tensor.data_ptr())."""
        rb, re, _ = self.band_rows(u, rows)
        if sync:
            self._ck(lib.gsb_render(self.h, C.byref(u), rb, re, out_ptr, 0, MEM_DEVICE, fmt, stream_ptr(stream)))
        else:
            self._ck(lib.gsb_render_async(self.h, C.byref(u), rb, re, out_ptr, 0, fmt, stream_ptr(stream)))

    def render_aux(self, u: Uniforms, fmt=FORMAT_RGBA32F, rows=None):
        """gsb_render_aux to HOST numpy arrays: (img, aux) with aux of shape (rows, W, 2) float32 = (opacity, expected depth)
        per pixel; img is exactly what render() returns."""
        rb, re, nrows = self.band_rows(u, rows)
        out = np.empty((nrows, u.width, 4), np.float32 if fmt == FORMAT_RGBA32F else np.uint8)
        aux = np.empty((nrows, u.width, 2), np.float32)
        self._ck(lib.gsb_render_aux(self.h, C.byref(u), rb, re, out.ctypes.data, 0, aux.ctypes.data, 0, MEM_HOST, fmt, None))
        return out, aux

    def render_aux_into(self, u: Uniforms, out_ptr: int, aux_ptr: int, fmt=FORMAT_RGBA32F, rows=None, stream=None,
                        aux_row_pitch=0):
        """gsb_render_aux into DEVICE memory (e.g. tensor.data_ptr()); aux_row_pitch in bytes, 0 = tight."""
        rb, re, _ = self.band_rows(u, rows)
        self._ck(lib.gsb_render_aux(self.h, C.byref(u), rb, re, out_ptr, 0, aux_ptr, aux_row_pitch, MEM_DEVICE, fmt,
                                    stream_ptr(stream)))

    def stats(self) -> Stats:
        s = Stats()
        self._ck(lib.gsb_get_stats(self.h, C.byref(s)))
        return s

    def download(self, which) -> np.ndarray:
        nbytes = lib.gsb_debug_size(self.h, which)
        dt = {BUF_COV3D: np.float32, BUF_ATTR: ATTR_DTYPE, BUF_TILES_OVERLAP: np.uint32, BUF_PREFIX_SUM: np.uint32,
              BUF_KEYS_UNSORTED: np.uint64, BUF_VALS_UNSORTED: np.uint32, BUF_KEYS_SORTED: np.uint64,
              BUF_VALS_SORTED: np.uint32, BUF_TILE_BOUNDARY: np.uint32, BUF_DEPTH_ORDER: np.uint32,
              BUF_EMIT_OFFSETS: np.uint64}[which]
        out = np.empty(nbytes // np.dtype(dt).itemsize, dt)
        if nbytes or which == BUF_COV3D:
            self._ck(lib.gsb_debug_download(self.h, which, out.ctypes.data, nbytes))
        if which == BUF_COV3D:
            out = out.reshape(-1, 6)
        if which == BUF_TILE_BOUNDARY:
            out = out.reshape(-1, 2)
        return out

    def sort_pairs(self, keys_ptr, vals_ptr, keys_tmp_ptr, vals_tmp_ptr, m, key_bits=64, stream=None):
        self._ck(lib.gsb_sort_pairs(self.h, keys_ptr, vals_ptr, keys_tmp_ptr, vals_tmp_ptr, m, key_bits,
                                    stream_ptr(stream)))

    def sort_pairs32(self, keys_ptr, vals_ptr, keys_tmp_ptr, vals_tmp_ptr, m, key_bits=32, stream=None):
        self._ck(lib.gsb_sort_pairs32(self.h, keys_ptr, vals_ptr, keys_tmp_ptr, vals_tmp_ptr, m, key_bits,
                                      stream_ptr(stream)))


# ---------------------------------------------------------------- one frame over several GPUs
def shard_slice(n_total: int, rank: int, world: int):
    """(first, count) of the Gaussians rank `rank` holds (gsb_shard_slice)."""
    first, count = C.c_uint64(), C.c_uint64()
    assert lib.gsb_shard_slice(n_total, rank, world, C.byref(first), C.byref(count)) == OK
    return first.value, count.value


def _frame_shape(u: Uniforms, fmt):
    return (u.height, u.width, 4), (np.float32 if fmt == FORMAT_RGBA32F else np.uint8)


class Group:
    """gsb_group: one process drives `devices` (ids may repeat: several ranks on one GPU)."""

    def __init__(self, devices):
        devices = list(devices)
        arr = (C.c_int * len(devices))(*devices)
        h = _vp()
        rc = lib.gsb_group_create(len(devices), arr, C.byref(h))
        if rc != OK:
            raise GsbError(rc, lib.gsb_shard_last_error().decode())
        self.h = h
        self.size = len(devices)

    def close(self):
        if self.h:
            lib.gsb_group_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != OK:
            raise GsbError(rc, lib.gsb_group_last_error(self.h).decode())

    def context(self, rank) -> "Context":
        return Context(handle=_vp(lib.gsb_group_context(self.h, rank)))

    def upload(self, vertices: np.ndarray):
        v = _f32(vertices).reshape(-1, 60)
        self._ck(lib.gsb_group_scene_upload(self.h, v.ctypes.data, v.shape[0], MEM_HOST))

    def render(self, u: Uniforms, fmt=FORMAT_RGBA32F) -> np.ndarray:
        shape, dt = _frame_shape(u, fmt)
        out = np.empty(shape, dt)
        self._ck(lib.gsb_group_render(self.h, C.byref(u), out.ctypes.data, 0, MEM_HOST, fmt))
        return out

    def render_async(self, u: Uniforms, fmt=FORMAT_BGRA8):
        self._ck(lib.gsb_group_render_async(self.h, C.byref(u), fmt))


def shard_unique_id() -> bytes:
    buf = (C.c_ubyte * 128)()
    rc = lib.gsb_shard_unique_id(buf)
    if rc != OK:
        raise GsbError(rc, lib.gsb_shard_last_error().decode())
    return bytes(buf)


class ShardedContext(Context):
    """gsb_create_sharded: this process is rank `rank` of `world` (one process per GPU)."""

    def __init__(self, device, rank, world, unique_id: bytes):
        h = _vp()
        idbuf = (C.c_ubyte * 128).from_buffer_copy(unique_id)
        rc = lib.gsb_create_sharded(device, rank, world, idbuf, C.byref(h))
        if rc != OK:
            raise GsbError(rc, lib.gsb_shard_last_error().decode() or lib.gsb_last_error(None).decode())
        super().__init__(device, handle=h)
        self._own = True
        self.rank, self.world = rank, world

    def upload_slice(self, slice_vertices: np.ndarray, n_total: int):
        v = _f32(slice_vertices).reshape(-1, 60)
        self._ck(lib.gsb_scene_upload_sharded(self.h, v.ctypes.data, n_total, MEM_HOST))

    def render_sharded(self, u: Uniforms, fmt=FORMAT_RGBA32F, stream=None) -> np.ndarray:
        shape, dt = _frame_shape(u, fmt)
        out = np.empty(shape, dt)
        self._ck(lib.gsb_render_sharded(self.h, C.byref(u), out.ctypes.data, 0, MEM_HOST, fmt, stream_ptr(stream)))
        return out

    def render_sharded_into(self, u: Uniforms, out_ptr, fmt, mem=MEM_DEVICE, stream=None):
        self._ck(lib.gsb_render_sharded(self.h, C.byref(u), out_ptr, 0, mem, fmt, stream_ptr(stream)))

    def render_sharded_async(self, u: Uniforms, fmt, stream=None):
        self._ck(lib.gsb_render_sharded_async(self.h, C.byref(u), fmt, stream_ptr(stream)))

    def frame_ptr(self) -> int:
        return lib.gsb_shard_frame(self.h)


# ---------------------------------------------------------------- the C++ host Renderer (vkgs_* style bridge)
class HostRenderer:
    """C++ `Renderer` (3dgs.cpp_b200/host/Renderer.h) driven through the gsh_* C bridge."""

    def __init__(self, scene_path, device=0, width=1280, height=720, fmt=FORMAT_BGRA8, mode=MODE_EXACT):
        self.h = host.gsh_initialize(str(scene_path).encode(), device, width, height, fmt, mode)
        if not self.h:
            raise RuntimeError(host.gsh_last_error().decode())
        self.width, self.height, self.fmt = width, height, fmt

    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError(host.gsh_last_error().decode())

    def close(self):
        if self.h:
            host.gsh_cleanup(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_camera(self, pos, quat_wxyz, fov=45.0, near=0.1, far=1000.0):
        p, q = _f32(pos, 3), _f32(quat_wxyz, 4)
        self._ck(host.gsh_set_camera(self.h, p.ctypes.data, q.ctypes.data, fov, near, far))

    def get_camera(self):
        p, q, f = np.zeros(3, np.float32), np.zeros(4, np.float32), C.c_float()
        self._ck(host.gsh_get_camera(self.h, p.ctypes.data, q.ctypes.data, C.byref(f)))
        return p, q, f.value

    def movement(self, x, y, z):
        self._ck(host.gsh_movement(self.h, x, y, z))

    def pan(self, dx, dy):
        self._ck(host.gsh_pan_translation(self.h, dx, dy))

    def keys(self, keys):
        arr = (C.c_int * 6)(*[int(k) for k in keys])
        self._ck(host.gsh_key_input(self.h, arr))

    def draw(self) -> np.ndarray:
        self._ck(host.gsh_draw(self.h))
        return self._frame(self.width, self.height, self.fmt)

    def render(self, width, height, fmt=FORMAT_RGBA32F) -> np.ndarray:
        self._ck(host.gsh_render(self.h, width, height, fmt, None, 0))
        return self._frame(width, height, fmt)

    def render_aux(self, width, height, fmt=FORMAT_RGBA32F):
        """Renderer::renderAux: (img, aux) with aux of shape (height, width, 2) float32 = (opacity, expected depth)."""
        dt = np.float32 if fmt == FORMAT_RGBA32F else np.uint8
        img = np.empty((height, width, 4), dt)
        aux = np.empty((height, width, 2), np.float32)
        self._ck(host.gsh_render_aux(self.h, width, height, fmt, img.ctypes.data, img.nbytes, aux.ctypes.data, aux.nbytes))
        return img, aux

    def _frame(self, w, h, fmt):
        n = C.c_size_t()
        p = host.gsh_frame(self.h, C.byref(n))
        dt = np.float32 if fmt == FORMAT_RGBA32F else np.uint8
        buf = (C.c_char * n.value).from_address(p)
        return np.frombuffer(buf, dtype=dt).reshape(h, w, 4).copy()

    def stats(self) -> Stats:
        s = Stats()
        self._ck(host.gsh_stats(self.h, C.byref(s)))
        return s

    @property
    def num_vertices(self):
        return host.gsh_num_vertices(self.h)
