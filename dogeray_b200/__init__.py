"""dogeray_b200 -- host-side mirror of the reference's hot-path interface over the C ABI.

The product is ``libdogeray_b200.so`` (``include/dogeray_b200.h``); this module is a thin ctypes
binding whose names follow the reference's own vocabulary (raygpu/kernel.cu): a *scene* is what
``getnum``/``read``/``readtextures``/``build_bvh`` produce, ``Scene.frame_i3`` is one
``CudaStarter`` call, ``Scene.render`` is the accumulate loop of ``main``.

There is no CPU path: the library is loaded on import and the import fails loudly if it has not
been built (``python dogeray_b200/build.py``); every device entry point raises ``DogerayError``
when no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdogeray_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "dogeray_b200: %s is missing -- build it with `python dogeray_b200/build.py` "
        "(there is no CPU fallback)" % LIB_PATH
    )
_lib = C.CDLL(LIB_PATH)

OK, ERR_ARG, ERR_IO, ERR_PARSE, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
FLAG_ACCUMULATE = 1
FLAG_EXACT_SAMPLES = 2
FLAG_DYNAMIC_TILES = 4
FLAG_SHARD_SAMPLES = 8
BUILD_LBVH_ONLY = 1
BUILD_KEEP_DEBUG = 2


class DogerayError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__("dogeray_b200 error %d: %s" % (status, message))
        self.status = status


class Settings(C.Structure):
    """The `*` settings line of a .rts file (SURVEY.md App. A.1; kernel.cu:1223-1299)."""
    _fields_ = [
        ("cam", C.c_float * 3), ("aperture", C.c_float), ("look", C.c_float * 3), ("focus", C.c_float),
        ("fov", C.c_int32), ("max_depth", C.c_int32), ("spp", C.c_int32), ("bg_intensity", C.c_float),
        ("backtex", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
    ]

    def copy(self) -> "Settings":
        s = Settings()
        C.memmove(C.byref(s), C.byref(self), C.sizeof(Settings))
        return s

    def replace(self, **kw) -> "Settings":
        s = self.copy()
        for k, v in kw.items():
            if k in ("cam", "look"):
                getattr(s, k)[:] = list(v)
            else:
                setattr(s, k, v)
        return s

    def as_dict(self):
        return {
            "cam": list(self.cam), "aperture": self.aperture, "look": list(self.look), "focus": self.focus,
            "fov": self.fov, "max_depth": self.max_depth, "spp": self.spp, "bg_intensity": self.bg_intensity,
            "backtex": self.backtex, "width": self.width, "height": self.height,
        }


# numpy view of drb_object (one object line, SURVEY.md App. A.2)
OBJECT_DTYPE = np.dtype([
    ("pos", "<f4", 3), ("type", "<i4"), ("col", "<f4", 3), ("add_y", "<f4"), ("add_x", "<f4"),
    ("dim", "<f4", 3), ("mat", "<i4"), ("rot", "<f4", 3), ("norm", "<f4", 3),
    ("n1", "<f4", 3), ("n2", "<f4", 3), ("n3", "<f4", 3), ("t1", "<f4", 2), ("t2", "<f4", 2), ("t3", "<f4", 2),
    ("smooth", "<i4"), ("checker", "<i4"), ("texnum", "<i4"), ("rtexnum", "<i4"), ("ncols", "<i4"),
])
assert OBJECT_DTYPE.itemsize == 156


class Opts(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("sample_base", C.c_uint32), ("sample_count", C.c_uint32),
        ("batch_paths", C.c_uint32), ("flags", C.c_uint32), ("stream", C.c_void_p),
        ("tile_rank", C.c_uint32), ("tile_count", C.c_uint32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("paths", C.c_uint64), ("rays", C.c_uint64), ("trace_ms", C.c_float), ("total_ms", C.c_float),
        ("trace_launches", C.c_uint32), ("kernel_launches", C.c_uint32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class BuildInfo(C.Structure):
    _fields_ = [
        ("nprims", C.c_int64), ("nnodes", C.c_int64), ("bounds_min", C.c_float * 3), ("bounds_max", C.c_float * 3),
        ("upload_ms", C.c_float), ("build_ms", C.c_float), ("max_depth", C.c_int32), ("rebuild_iterations", C.c_int32),
        ("nwide", C.c_int64), ("wide_levels", C.c_int32), ("stack_levels", C.c_int32),
    ]


def _sig(name, restype, *argtypes):
    f = getattr(_lib, name)
    f.restype = restype
    f.argtypes = list(argtypes)
    return f


_vp, _cp, _i, _i64, _u32, _u64 = C.c_void_p, C.c_char_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64
_pp = C.POINTER(C.c_void_p)

# every symbol include/dogeray_b200.h declares
_sig("drb_host_scene_load", _i, _cp, _cp, _pp)
_sig("drb_host_scene_load_cached", _i, _cp, _cp, _cp, _pp, C.POINTER(C.c_int))
_sig("drb_hash_bytes", _u64, _vp, C.c_size_t)
_sig("drb_host_scene_parse", _i, _cp, C.c_size_t, _cp, _pp)
_sig("drb_host_scene_create", _i, C.POINTER(Settings), _vp, _i64, C.POINTER(_cp), _i, _pp)
_sig("drb_host_scene_free", None, _vp)
_sig("drb_host_scene_num_objects", _i64, _vp)
_sig("drb_host_scene_objects", _vp, _vp)
_sig("drb_host_scene_settings", _i, _vp, C.POINTER(Settings))
_sig("drb_host_scene_num_textures", _i, _vp)
_sig("drb_host_scene_texture_path", _cp, _vp, _i)
_sig("drb_host_scene_num_skipped", _i64, _vp)
_sig("drb_host_scene_num_renderable", _i64, _vp)
_sig("drb_rts_write", _i, _cp, C.POINTER(Settings), _vp, _i64, C.POINTER(_cp), _i, _cp)
_sig("drb_settings_default", None, C.POINTER(Settings))
_sig("drb_scene_create", _i, _vp, _i, _pp)
_sig("drb_scene_create_ex", _i, _vp, _i, _u32, _pp)
_sig("drb_scene_create_from_device", _i, _vp, _i, _u32, _vp, _vp, _pp)
_sig("drb_scene_tree", _i, _vp, _vp, _vp, _vp, _vp)
_sig("drb_scene_wide", _i, _vp, _vp, _vp)
_sig("drb_scene_refit_device", _i, _vp, _vp, _i64, _vp)
_sig("drb_scene_refit", _i, _vp, _vp, _i64)
_sig("drb_scene_load", _i, _cp, _cp, _i, _pp)
_sig("drb_scene_free", None, _vp)
_sig("drb_scene_settings", _i, _vp, C.POINTER(Settings))
_sig("drb_scene_num_prims", _i64, _vp)
_sig("drb_scene_num_objects", _i64, _vp)
_sig("drb_scene_build_info", _i, _vp, C.POINTER(BuildInfo))
_sig("drb_scene_lbvh", _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
_sig("drb_opts_default", None, C.POINTER(Opts))
_sig("drb_render_device", _i, _vp, C.POINTER(Settings), C.POINTER(Opts), _vp, C.POINTER(Stats))
_sig("drb_render", _i, _vp, C.POINTER(Settings), C.POINTER(Opts), _vp, C.POINTER(Stats))
_sig("drb_render_multi", _i, C.POINTER(C.c_void_p), _i, C.POINTER(Settings), C.POINTER(Opts), _vp, C.POINTER(Stats))
_sig("drb_render_multi_times", _i, C.POINTER(C.c_float), _i)
_sig("drb_scene_create_multi", _i, _vp, C.POINTER(C.c_int), _i, _u32, C.POINTER(C.c_void_p))
_sig("drb_frame_i3", _i, _vp, C.POINTER(Settings), C.POINTER(Opts), _i, _vp)
_sig("drb_trace_ids", _i, _vp, _vp, _vp, _i64, _vp, _vp)
_sig("drb_trace_device", _i, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp)
_sig("drb_occluded_device", _i, _vp, _vp, _vp, _vp, _i64, _vp, _vp)
_sig("drb_primary_rays", _i, _vp, C.POINTER(Settings), C.POINTER(Opts), _u32, _vp, _vp)
_sig("drb_tonemap", _i, _vp, _i, _i, C.c_double, _vp)
_sig("drb_tonemap_device", _i, _vp, _i, _i, C.c_double, _vp, _vp)
_sig("drb_write_bmp", _i, _cp, _vp, _i, _i)
_sig("drb_write_ppm", _i, _cp, _vp, _i, _i)
_sig("drb_read_ppm", _i, _cp, _pp, C.POINTER(_i), C.POINTER(_i))
_sig("drb_free", None, _vp)
_sig("drb_last_error", _cp)
_sig("drb_abi_version", _i)
_sig("drb_device_count", _i)
_sig("drb_trim", _i, _i)
_sig("drb_philox_word", _u32, _u64, _u32, _u32, _u32, _u32)

EXPORTED_SYMBOLS = [
    "drb_host_scene_load", "drb_host_scene_load_cached", "drb_hash_bytes", "drb_host_scene_parse", "drb_host_scene_create",
    "drb_host_scene_free",
    "drb_host_scene_num_objects", "drb_host_scene_objects", "drb_host_scene_settings",
    "drb_host_scene_num_textures", "drb_host_scene_texture_path", "drb_host_scene_num_skipped", "drb_host_scene_num_renderable",
    "drb_scene_create_from_device", "drb_scene_create_multi", "drb_render_multi_times",
    "drb_rts_write", "drb_settings_default", "drb_scene_create", "drb_scene_create_ex", "drb_scene_tree", "drb_scene_wide", "drb_scene_refit_device", "drb_scene_refit", "drb_scene_load", "drb_scene_free",
    "drb_scene_settings", "drb_scene_num_prims", "drb_scene_num_objects", "drb_scene_build_info",
    "drb_scene_lbvh", "drb_opts_default", "drb_render_device", "drb_render", "drb_render_multi", "drb_frame_i3",
    "drb_trace_ids", "drb_trace_device", "drb_occluded_device", "drb_primary_rays", "drb_tonemap", "drb_tonemap_device", "drb_write_bmp",
    "drb_write_ppm", "drb_read_ppm", "drb_free", "drb_last_error", "drb_abi_version",
    "drb_device_count", "drb_trim", "drb_philox_word",
]


def last_error() -> str:
    return _lib.drb_last_error().decode("utf-8", "replace")


def _check(rc: int):
    if rc != 0:
        raise DogerayError(rc, last_error())


def _b(s: Optional[str]):
    return None if s is None else os.fsencode(s)


def _stream_handle(stream: Optional[int]):
    """None -> the scene's own (non-blocking) stream.  0 is how torch names the legacy default stream
    (torch.cuda.current_stream().cuda_stream outside a stream context); the C ABI reads a NULL stream as "the scene's own",
    so the legacy default stream travels as its CUDA handle cudaStreamLegacy (0x1)."""
    return None if stream is None else (1 if stream == 0 else stream)


def _record(stream, *tensors):
    """keeps tensors that work on `stream` reads or writes alive until it is done when they belong to another stream"""
    import torch
    if stream != torch.cuda.current_stream(stream.device):
        for x in tensors:
            if x is not None:
                x.record_stream(stream)


def default_settings() -> Settings:
    s = Settings()
    _lib.drb_settings_default(C.byref(s))
    return s


def device_count() -> int:
    return int(_lib.drb_device_count())


def render_multi(scenes: Sequence["Scene"], settings: Optional[Settings] = None, *, seed=0, sample_base=0, sample_count=None,
                 batch_paths=0, accumulate_into: Optional[np.ndarray] = None, dynamic=False, shard="tiles") -> Tuple[np.ndarray, Stats]:
    """One frame over several resident scenes (the same scene on different devices) from this process, one host thread per
    handle.  shard="tiles" (default): interleaved tiles, bit-identical to Scene.render on one handle; with dynamic=True the
    tile shards are claimed from a shared queue.  shard="samples": sample ranges, summed in handle order.  With peer access
    the image lives in one buffer on the first handle's device and the other devices write / are read over NVLink."""
    assert len(scenes) >= 1 and shard in ("tiles", "samples")
    st = settings if settings is not None else scenes[0].settings
    flags = (FLAG_DYNAMIC_TILES if dynamic else 0) | (FLAG_SHARD_SAMPLES if shard == "samples" else 0)
    if accumulate_into is not None:
        out = np.ascontiguousarray(accumulate_into, dtype=np.float32)
        assert out.shape == (st.height, st.width, 3)
        flags |= FLAG_ACCUMULATE
    else:
        out = np.zeros((st.height, st.width, 3), np.float32)
    o = Scene._opts(seed, sample_base, sample_count, batch_paths, flags, None, 0, 0)
    handles = (C.c_void_p * len(scenes))(*[sc.handle for sc in scenes])
    stats = Stats()
    _check(_lib.drb_render_multi(handles, len(scenes), C.byref(st), C.byref(o), out.ctypes.data, C.byref(stats)))
    return out, stats


def render_multi_times() -> list:
    """device time (ms) each handle spent in this thread's last render_multi call (load-balance measurements)"""
    buf = (C.c_float * 64)()
    n = _lib.drb_render_multi_times(buf, 64)
    return [float(buf[k]) for k in range(min(n, 64))]


def create_multi(hs: "HostScene", devices: Sequence[int], build_flags: int = 0) -> list:
    """The same scene on several devices; the object lines cross PCIe once (each device uploads a share, the devices
    exchange shares over NVLink) and every device builds its own tree."""
    devs = (C.c_int * len(devices))(*devices)
    out = (C.c_void_p * len(devices))()
    _check(_lib.drb_scene_create_multi(hs.handle, devs, len(devices), build_flags, out))
    return [Scene(C.c_void_p(out[k]), devices[k]) for k in range(len(devices))]


def hash_bytes(data: bytes) -> int:
    """the 64-bit content hash the scene cache is keyed by"""
    return int(_lib.drb_hash_bytes(data, len(data)))


def trim(device: int = 0):
    """Return all idle device memory of `device` to the driver."""
    _check(_lib.drb_trim(device))


def philox_word(seed: int, x: int, y: int, sample: int, n: int) -> int:
    return int(_lib.drb_philox_word(seed, x, y, sample, n))


def philox_uniform(seed: int, x: int, y: int, sample: int, n: int) -> float:
    return float((np.float32(philox_word(seed, x, y, sample, n) >> 8) + np.float32(0.5)) * np.float32(1.0 / 16777216.0))


class HostScene:
    """Parsed .rts scene on the host (what getnum + read + getppmpaths leave behind)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def load(cls, rts_path: str, tex_dir: Optional[str] = None, cache=None) -> "HostScene":
        """`cache`: None = parse the text; True = binary cache next to the scene (`<scene>.drbcache`);
        a path = that cache file.  `cache_hit` on the result says whether the cache served the load."""
        h = C.c_void_p()
        if cache is None or cache is False:
            _check(_lib.drb_host_scene_load(_b(rts_path), _b(tex_dir), C.byref(h)))
            hs = cls(h)
            hs.cache_hit = False
            return hs
        hit = C.c_int(0)
        _check(_lib.drb_host_scene_load_cached(_b(rts_path), _b(tex_dir), None if cache is True else _b(cache), C.byref(h), C.byref(hit)))
        hs = cls(h)
        hs.cache_hit = bool(hit.value)
        return hs

    @classmethod
    def parse(cls, text: bytes, tex_dir: Optional[str] = None) -> "HostScene":
        h = C.c_void_p()
        _check(_lib.drb_host_scene_parse(text, len(text), _b(tex_dir), C.byref(h)))
        return cls(h)

    @classmethod
    def from_objects(cls, objects: np.ndarray, settings: Optional[Settings] = None, tex_paths: Sequence[str] = ()) -> "HostScene":
        objects = np.ascontiguousarray(objects, dtype=OBJECT_DTYPE)
        arr = (C.c_char_p * max(len(tex_paths), 1))(*[_b(p) for p in tex_paths])
        h = C.c_void_p()
        _check(_lib.drb_host_scene_create(C.byref(settings) if settings is not None else None, objects.ctypes.data,
                                          len(objects), arr if tex_paths else None, len(tex_paths), C.byref(h)))
        return cls(h)

    def close(self):
        if self._h and _lib is not None:             # _lib is None while the interpreter shuts down
            _lib.drb_host_scene_free(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    @property
    def num_objects(self) -> int:
        return int(_lib.drb_host_scene_num_objects(self._h))

    @property
    def num_renderable(self) -> int:
        return int(_lib.drb_host_scene_num_renderable(self._h))

    @property
    def num_skipped(self) -> int:
        return int(_lib.drb_host_scene_num_skipped(self._h))

    @property
    def settings(self) -> Settings:
        s = Settings()
        _check(_lib.drb_host_scene_settings(self._h, C.byref(s)))
        return s

    @property
    def texture_paths(self):
        n = _lib.drb_host_scene_num_textures(self._h)
        return [os.fsdecode(_lib.drb_host_scene_texture_path(self._h, i)) for i in range(n)]

    def objects(self) -> np.ndarray:
        n = self.num_objects
        if n == 0:
            return np.zeros(0, dtype=OBJECT_DTYPE)
        p = _lib.drb_host_scene_objects(self._h)
        buf = (C.c_char * (n * OBJECT_DTYPE.itemsize)).from_address(p)
        return np.frombuffer(buf, dtype=OBJECT_DTYPE).copy()


def write_rts(path: str, settings: Settings, objects: np.ndarray, tex_names: Sequence[str] = (), backtex_name: Optional[str] = None):
    """Write a scene in the exporter's format (plugin/rtsexport.py:207, 312-314)."""
    objects = np.ascontiguousarray(objects, dtype=OBJECT_DTYPE)
    arr = (C.c_char_p * max(len(tex_names), 1))(*[_b(p) for p in tex_names])
    _check(_lib.drb_rts_write(_b(path), C.byref(settings), objects.ctypes.data, len(objects), arr if tex_names else None,
                              len(tex_names), _b(backtex_name)))


def make_objects(n: int) -> np.ndarray:
    """n object records with the reference's struct defaults (kernel.cu:55-71), type 2."""
    o = np.zeros(n, dtype=OBJECT_DTYPE)
    o["type"] = 2
    for k in ("norm", "n1", "n2", "n3"):
        o[k] = (-2.0, -3.0, -20.0)
    o["t1"] = (0.0, 1.0)
    o["t2"] = (0.0, 0.0)
    o["t3"] = (1.0, 0.0)
    o["texnum"] = -1
    o["rtexnum"] = -1
    return o


class Scene:
    """Device-resident scene: textures uploaded, LBVH built on the GPU, everything kept in HBM."""

    def __init__(self, handle, device: int = 0):
        self._h = handle
        self.device = device                         # the CUDA device the scene lives on

    @classmethod
    def load(cls, rts_path: str, tex_dir: Optional[str] = None, device: int = 0) -> "Scene":
        h = C.c_void_p()
        _check(_lib.drb_scene_load(_b(rts_path), _b(tex_dir), device, C.byref(h)))
        return cls(h, device)

    @classmethod
    def from_host(cls, hs: HostScene, device: int = 0, build_flags: int = 0) -> "Scene":
        h = C.c_void_p()
        _check(_lib.drb_scene_create_ex(hs.handle, device, build_flags, C.byref(h)))
        return cls(h, device)

    @classmethod
    def from_device_objects(cls, hs: HostScene, objects_ptr: int, device: int = 0, build_flags: int = 0, stream: Optional[int] = None) -> "Scene":
        """The object lines are already in device memory (hs.num_objects records of OBJECT_DTYPE at `objects_ptr`, e.g.
        all-gathered over NVLink from per-rank partial uploads); `stream` is the stream that produced them."""
        h = C.c_void_p()
        _check(_lib.drb_scene_create_from_device(hs.handle, device, build_flags, objects_ptr, _stream_handle(stream), C.byref(h)))
        return cls(h, device)

    def close(self):
        if self._h and _lib is not None:             # _lib is None while the interpreter shuts down
            _lib.drb_scene_free(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    @property
    def settings(self) -> Settings:
        s = Settings()
        _check(_lib.drb_scene_settings(self._h, C.byref(s)))
        return s

    @property
    def num_prims(self) -> int:
        return int(_lib.drb_scene_num_prims(self._h))

    @property
    def num_objects(self) -> int:
        return int(_lib.drb_scene_num_objects(self._h))

    @property
    def build_info(self) -> BuildInfo:
        b = BuildInfo()
        _check(_lib.drb_scene_build_info(self._h, C.byref(b)))
        return b

    def lbvh(self):
        """Integer outputs of the GPU build: keys, order, parent, left, right, node_min, node_max."""
        n = self.num_prims
        ni = max(n - 1, 0)
        keys = np.zeros(n, np.uint64); order = np.zeros(n, np.int32)
        parent = np.zeros(ni, np.int32); left = np.zeros(ni, np.int32); right = np.zeros(ni, np.int32)
        nmin = np.zeros((ni, 3), np.float32); nmax = np.zeros((ni, 3), np.float32)
        _check(_lib.drb_scene_lbvh(self._h, keys.ctypes.data, order.ctypes.data, parent.ctypes.data, left.ctypes.data,
                                   right.ctypes.data, nmin.ctypes.data, nmax.ctypes.data))
        return dict(keys=keys, order=order, parent=parent, left=left, right=right, node_min=nmin, node_max=nmax)

    def tree(self):
        """The hierarchy the traversal nodes were emitted from (root = node 0): left, right, node_min, node_max."""
        ni = max(self.num_prims - 1, 0)
        left = np.zeros(ni, np.int32); right = np.zeros(ni, np.int32)
        nmin = np.zeros((ni, 3), np.float32); nmax = np.zeros((ni, 3), np.float32)
        _check(_lib.drb_scene_tree(self._h, left.ctypes.data, right.ctypes.data, nmin.ctypes.data, nmax.ctypes.data))
        return dict(left=left, right=right, node_min=nmin, node_max=nmax)

    def wide(self):
        """The four-wide traversal nodes: child (n,4) int32 and boxes (n,4,3) uint32 (min_q | max_q << 16)."""
        n = int(self.build_info.nwide)
        child = np.zeros((n, 4), np.int32); boxes = np.zeros((n, 4, 3), np.uint32)
        _check(_lib.drb_scene_wide(self._h, child.ctypes.data, boxes.ctypes.data))
        return dict(child=child, boxes=boxes)

    def refit_device(self, objects_ptr: int, n: int, stream: Optional[int] = None):
        """New object lines for the same tree: n (== num_objects) records of OBJECT_DTYPE in DEVICE memory at `objects_ptr`,
        produced on `stream` (a raw handle; None -> the scene's own).  Synchronous: the scene is updated when it returns."""
        _check(_lib.drb_scene_refit_device(self._h, objects_ptr, n, _stream_handle(stream)))

    def refit(self, objects, *, stream=None):
        """Update the resident scene in place from new object lines, keeping its tree (drb_scene_refit): a host OBJECT_DTYPE
        array of num_objects records, or a contiguous CUDA tensor on the scene's device holding them (nbytes ==
        num_objects * 156, e.g. float32 (n, 39)) written on `stream` (a torch.cuda.Stream, default the current one)."""
        n = self.num_objects
        if isinstance(objects, np.ndarray):
            if objects.dtype != OBJECT_DTYPE or objects.ndim != 1 or len(objects) != n:
                raise ValueError("refit takes %d records of OBJECT_DTYPE, got %s %s" % (n, objects.dtype, objects.shape))
            a = np.ascontiguousarray(objects)
            _check(_lib.drb_scene_refit(self._h, a.ctypes.data, n))
            return
        import torch
        if not isinstance(objects, torch.Tensor):
            raise ValueError("refit takes a numpy OBJECT_DTYPE array or a CUDA tensor, got %s" % type(objects).__name__)
        dev = torch.device("cuda", self.device)
        if objects.device != dev or not objects.is_contiguous() or objects.nbytes != n * OBJECT_DTYPE.itemsize:
            raise ValueError("refit takes a contiguous tensor of %d bytes on %s, got %d bytes on %s" %
                             (n * OBJECT_DTYPE.itemsize, dev, objects.nbytes, objects.device))
        if stream is None:
            stream = torch.cuda.current_stream(dev)
        self.refit_device(objects.data_ptr(), n, stream.cuda_stream)

    @staticmethod
    def _opts(seed=0, sample_base=0, sample_count=None, batch_paths=0, flags=0, stream=None, tile_rank=0, tile_count=0) -> Opts:
        """sample_count None -> the settings' spp; an integer is taken literally (0 traces nothing: the empty share of
        a sharded frame, distributed.shard_samples with spp < ranks)"""
        o = Opts()
        _lib.drb_opts_default(C.byref(o))
        if sample_count is not None:
            flags |= FLAG_EXACT_SAMPLES
        o.seed, o.sample_base, o.sample_count, o.batch_paths, o.flags = seed, sample_base, int(sample_count or 0), batch_paths, flags
        o.stream = _stream_handle(stream)
        o.tile_rank, o.tile_count = tile_rank, tile_count
        return o

    def render(self, settings: Optional[Settings] = None, *, seed=0, sample_base=0, sample_count=None, batch_paths=0,
               accumulate_into: Optional[np.ndarray] = None, want_stats=True, tile_rank=0, tile_count=0) -> Tuple[np.ndarray, Optional[Stats]]:
        """Sum of radiance per pixel, float32 (H, W, 3), host buffers (device->host copy included)."""
        st = settings if settings is not None else self.settings
        flags = 0
        if accumulate_into is not None:
            out = np.ascontiguousarray(accumulate_into, dtype=np.float32)
            assert out.shape == (st.height, st.width, 3)
            flags |= FLAG_ACCUMULATE
        else:
            out = np.zeros((st.height, st.width, 3), np.float32)
        o = self._opts(seed, sample_base, sample_count, batch_paths, flags, None, tile_rank, tile_count)
        stats = Stats() if want_stats else None
        _check(_lib.drb_render(self._h, C.byref(st), C.byref(o), out.ctypes.data, C.byref(stats) if stats is not None else None))
        return out, stats

    def render_device(self, accum_ptr: int, settings: Optional[Settings] = None, *, seed=0, sample_base=0, sample_count=None,
                      batch_paths=0, accumulate=False, stream: Optional[int] = None, want_stats=False, tile_rank=0, tile_count=0) -> Optional[Stats]:
        """Same into a DEVICE buffer of H*W*3 float32 (e.g. torch tensor .data_ptr()); asynchronous unless want_stats."""
        st = settings if settings is not None else self.settings
        o = self._opts(seed, sample_base, sample_count, batch_paths, FLAG_ACCUMULATE if accumulate else 0, stream, tile_rank, tile_count)
        stats = Stats() if want_stats else None
        _check(_lib.drb_render_device(self._h, C.byref(st), C.byref(o), accum_ptr, C.byref(stats) if stats is not None else None))
        return stats

    def frame_i3(self, settings: Optional[Settings] = None, divisor: int = 1, *, seed=0, sample_base=0, sample_count=None,
                 out: Optional[np.ndarray] = None) -> np.ndarray:
        """One CudaStarter call: int32 (W, H, 3) indexed [x, y] = outputr[x*H + y] (kernel.cu:1006, 1083-1085)."""
        st = settings if settings is not None else self.settings
        if out is None:
            out = np.zeros((st.width, st.height, 3), np.int32)
        assert out.dtype == np.int32 and out.shape == (st.width, st.height, 3) and out.flags.c_contiguous
        o = self._opts(seed, sample_base, sample_count)
        _check(_lib.drb_frame_i3(self._h, C.byref(st), C.byref(o), divisor, out.ctypes.data))
        return out

    def trace_ids(self, origins: np.ndarray, dirs: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """Closest-hit object ids (-1 = miss) and t for explicit rays: hit() of kernel.cu:468-512."""
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        assert o.shape == d.shape
        ids = np.empty(len(o), np.int32); t = np.empty(len(o), np.float32)
        _check(_lib.drb_trace_ids(self._h, o.ctypes.data, d.ctypes.data, len(o), ids.ctypes.data, t.ctypes.data))
        return ids, t

    def trace_device(self, o_ptr: int, d_ptr: int, n: int, ids_ptr: int, t_ptr: Optional[int] = None, uv_ptr: Optional[int] = None,
                     stream: Optional[int] = None):
        """Closest hit for n rays in DEVICE arrays (n*3 float32 each): ids int32 (-1 = miss), optionally t float32 (-1 on a miss)
        and (u, v) float32 pairs of the hit triangle.  Enqueued on `stream` (a raw handle; None -> the scene's own), asynchronous."""
        _check(_lib.drb_trace_device(self._h, o_ptr, d_ptr, n, ids_ptr, t_ptr, uv_ptr, _stream_handle(stream)))

    def occluded_device(self, o_ptr: int, d_ptr: int, n: int, out_ptr: int, tmax_ptr: Optional[int] = None, stream: Optional[int] = None):
        """Any hit below tmax (n float32 in device memory; None -> 10000) for n rays in DEVICE arrays: n bytes 0 / 1 at
        `out_ptr`.  Enqueued on `stream` (a raw handle; None -> the scene's own), asynchronous."""
        _check(_lib.drb_occluded_device(self._h, o_ptr, d_ptr, tmax_ptr, n, out_ptr, _stream_handle(stream)))

    def _query_args(self, stream, *tensors):
        """(torch, stream, contiguous inputs): float32 CUDA tensors on the scene's device, the stream defaulting to the
        caller's current torch stream"""
        import torch
        dev = torch.device("cuda", self.device)
        out = []
        for x in tensors:
            if not isinstance(x, torch.Tensor):
                raise ValueError("ray queries take torch tensors, got %s" % type(x).__name__)
            if x.dtype != torch.float32 or x.device != dev:
                raise ValueError("ray queries take float32 tensors on %s, got %s on %s" % (dev, x.dtype, x.device))
            out.append(x.contiguous())
        if stream is None:
            stream = torch.cuda.current_stream(dev)
        return torch, stream, out

    def trace(self, origins, dirs, *, with_uv: bool = True, stream=None):
        """Closest hit for torch rays: origins and dirs float32 (..., 3) on the scene's device.  Returns (ids int32 (...),
        t float32 (...), uv float32 (..., 2) or None), allocated on that device and enqueued on `stream` (a torch.cuda.Stream,
        default the current one) without synchronising."""
        torch, stream, (o, d) = self._query_args(stream, origins, dirs)
        if o.shape != d.shape or o.shape[-1:] != (3,):
            raise ValueError("origins and dirs must have the same shape (..., 3), got %s and %s" % (tuple(o.shape), tuple(d.shape)))
        lead = o.shape[:-1]
        ids = torch.empty(lead, dtype=torch.int32, device=o.device)
        t = torch.empty(lead, dtype=torch.float32, device=o.device)
        uv = torch.empty(lead + (2,), dtype=torch.float32, device=o.device) if with_uv else None
        self.trace_device(o.data_ptr(), d.data_ptr(), o.numel() // 3, ids.data_ptr(), t.data_ptr(), uv.data_ptr() if with_uv else None,
                          stream.cuda_stream)
        _record(stream, o, d, ids, t, uv)
        return ids, t, uv

    def occluded(self, origins, dirs, tmax=None, *, stream=None):
        """Any hit at t < tmax for torch rays: origins and dirs float32 (..., 3), tmax float32 (...) or None (10000), all on
        the scene's device.  Returns bool (...), enqueued on `stream` (a torch.cuda.Stream, default the current one) without
        synchronising."""
        torch, stream, xs = self._query_args(stream, origins, dirs, *(() if tmax is None else (tmax,)))
        o, d = xs[0], xs[1]
        tm = xs[2] if tmax is not None else None
        if o.shape != d.shape or o.shape[-1:] != (3,) or (tm is not None and tm.shape != o.shape[:-1]):
            raise ValueError("origins and dirs must have the same shape (..., 3) and tmax their leading shape")
        out = torch.empty(o.shape[:-1], dtype=torch.bool, device=o.device)
        self.occluded_device(o.data_ptr(), d.data_ptr(), o.numel() // 3, out.data_ptr(), tm.data_ptr() if tm is not None else None,
                             stream.cuda_stream)
        _record(stream, o, d, tm, out)
        return out

    def primary_rays(self, settings: Optional[Settings] = None, sample: int = 0, seed: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """Camera rays of one sample index, (H, W, 3) each: kernel.cu:1067-1076."""
        st = settings if settings is not None else self.settings
        o = np.empty((st.height, st.width, 3), np.float32); d = np.empty((st.height, st.width, 3), np.float32)
        op = self._opts(seed)
        _check(_lib.drb_primary_rays(self._h, C.byref(st), C.byref(op), sample, o.ctypes.data, d.ctypes.data))
        return o, d


def tonemap(accum: np.ndarray, nsamples: float) -> np.ndarray:
    """clamp(trunc(255 * sum / n), 0, 255), linear (kernel.cu:1083-1085, 2287) -> uint8 (H, W, 3)."""
    a = np.ascontiguousarray(accum, np.float32)
    h, w, _ = a.shape
    out = np.empty((h, w, 3), np.uint8)
    _check(_lib.drb_tonemap(a.ctypes.data, w, h, float(nsamples), out.ctypes.data))
    return out


def tonemap_device(accum_ptr: int, width: int, height: int, nsamples: float, rgb8_ptr: int, stream: Optional[int] = None):
    _check(_lib.drb_tonemap_device(accum_ptr, width, height, float(nsamples), rgb8_ptr, stream))


def write_bmp(path: str, rgb8: np.ndarray):
    a = np.ascontiguousarray(rgb8, np.uint8)
    _check(_lib.drb_write_bmp(_b(path), a.ctypes.data, a.shape[1], a.shape[0]))


def write_ppm(path: str, rgb8: np.ndarray):
    a = np.ascontiguousarray(rgb8, np.uint8)
    _check(_lib.drb_write_ppm(_b(path), a.ctypes.data, a.shape[1], a.shape[0]))


def read_ppm(path: str) -> np.ndarray:
    p = C.c_void_p(); w = C.c_int(); h = C.c_int()
    _check(_lib.drb_read_ppm(_b(path), C.byref(p), C.byref(w), C.byref(h)))
    try:
        buf = (C.c_uint8 * (w.value * h.value * 4)).from_address(p.value)
        return np.frombuffer(buf, np.uint8).reshape(h.value, w.value, 4).copy()
    finally:
        _lib.drb_free(p)
