"""TEST INFRASTRUCTURE -- ctypes access to oracle/libdogeray_oracle.so (the plain-C restatement in
dogeray_oracle.c and the host LBVH mirror in lbvh_host.c).  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs may import this module."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libdogeray_oracle.so")


def build():
    subprocess.run(["make", "-s", "-C", HERE], check=True)
    return LIB


def _load():
    if not os.path.exists(LIB):
        build()
    L = C.CDLL(LIB)
    L.orc_load.argtypes = [C.c_char_p, C.c_char_p]; L.orc_load.restype = C.c_void_p
    L.orc_free.argtypes = [C.c_void_p]
    L.orc_num_objects.argtypes = [C.c_void_p]
    L.orc_num_nodes.argtypes = [C.c_void_p]
    L.orc_get_settings.argtypes = [C.c_void_p, C.c_void_p]
    L.orc_set_settings.argtypes = [C.c_void_p, C.c_void_p]
    L.orc_set_seed.argtypes = [C.c_void_p, C.c_uint64]
    L.orc_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.orc_hit_brute.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.orc_brute_tris.argtypes = [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 2 + [C.c_int]
    L.orc_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_int]; L.orc_frame.restype = C.c_uint64
    L.orc_primary_rays.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p]
    L.orc_philox_word.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]; L.orc_philox_word.restype = C.c_uint32
    L.lbvh_host_build.argtypes = [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 8
    L.lbvh_host_build.restype = C.c_int
    L.ploc_host_build.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5
    L.ploc_host_build.restype = C.c_int
    L.wide_host_build.argtypes = [C.c_void_p] * 6 + [C.c_int] + [C.c_void_p] * 4
    L.wide_host_build.restype = C.c_int
    return L


class Restated:
    """A scene inside the C restatement."""

    def __init__(self, rts_path: str, tex_dir: str = ""):
        self.L = _load()
        self.h = self.L.orc_load(os.fsencode(rts_path), os.fsencode(tex_dir or ""))
        if not self.h:
            raise IOError("oracle could not open %s" % rts_path)

    def close(self):
        if self.h:
            self.L.orc_free(self.h)
            self.h = None

    __del__ = close

    @property
    def num_objects(self):
        return self.L.orc_num_objects(self.h)

    @property
    def num_nodes(self):
        return self.L.orc_num_nodes(self.h)

    def get_settings(self):
        s = np.zeros(16, np.float32)
        self.L.orc_get_settings(self.h, s.ctypes.data)
        return s

    def set_settings(self, s):
        s = np.ascontiguousarray(s, np.float32)
        self.L.orc_set_settings(self.h, s.ctypes.data)

    def apply(self, st):
        self.set_settings([st.cam[0], st.cam[1], st.cam[2], st.aperture, st.look[0], st.look[1], st.look[2], st.focus,
                           st.fov, st.max_depth, st.spp, st.bg_intensity, st.backtex, st.width, st.height, 0])

    def set_seed(self, seed):
        self.L.orc_set_seed(self.h, seed)

    def _hit(self, fn, origins, dirs):
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        t = np.empty(len(o), np.float32); ids = np.empty(len(o), np.int32)
        fn(self.h, o.ctypes.data, d.ctypes.data, len(o), t.ctypes.data, ids.ctypes.data)
        return ids, t

    def hit(self, origins, dirs):
        return self._hit(self.L.orc_hit, origins, dirs)

    def hit_brute(self, origins, dirs):
        return self._hit(self.L.orc_hit_brute, origins, dirs)

    def frame(self, divisor=1, sample_base=0, threads=0):
        s = self.get_settings()
        W, H = int(s[13]), int(s[14])
        f = np.zeros((W, H, 3), np.float32); i = np.zeros((W, H, 3), np.int32)
        rays = self.L.orc_frame(self.h, f.ctypes.data, i.ctypes.data, divisor, sample_base, threads or (os.cpu_count() or 1))
        return f, i, int(rays)

    def primary_rays(self, sample=0):
        s = self.get_settings()
        W, H = int(s[13]), int(s[14])
        o = np.empty((H, W, 3), np.float32); d = np.empty((H, W, 3), np.float32)
        self.L.orc_primary_rays(self.h, sample, o.ctypes.data, d.ctypes.data)
        return o, d


def brute_tris(v0, v1, v2, origins, dirs, threads=0):
    """Closest hit by definition over triangle arrays (n,3) x3: (ids, t), -1 = miss; lowest index keeps exact ties."""
    L = _load()
    v0 = np.ascontiguousarray(v0, np.float32); v1 = np.ascontiguousarray(v1, np.float32); v2 = np.ascontiguousarray(v2, np.float32)
    o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3); d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
    t = np.empty(len(o), np.float32); ids = np.empty(len(o), np.int32)
    L.orc_brute_tris(v0.ctypes.data, v1.ctypes.data, v2.ctypes.data, len(v0), o.ctypes.data, d.ctypes.data, len(o), t.ctypes.data, ids.ctypes.data,
                     threads or (os.cpu_count() or 1))
    return ids, t


def philox_word(seed, x, y, sample, n):
    return int(_load().orc_philox_word(seed, x, y, sample, n))


def lbvh_host(bmin: np.ndarray, bmax: np.ndarray):
    """Host LBVH over primitive boxes (n,3): dict like dogeray_b200.Scene.lbvh() plus height / scene_bounds."""
    L = _load()
    bmin = np.ascontiguousarray(bmin, np.float32); bmax = np.ascontiguousarray(bmax, np.float32)
    n = len(bmin); ni = max(n - 1, 0)
    keys = np.zeros(n, np.uint64); order = np.zeros(n, np.int32)
    parent = np.zeros(ni, np.int32); left = np.zeros(ni, np.int32); right = np.zeros(ni, np.int32)
    nmin = np.zeros((ni, 3), np.float32); nmax = np.zeros((ni, 3), np.float32); sb = np.zeros(6, np.float32)
    h = L.lbvh_host_build(bmin.ctypes.data, bmax.ctypes.data, n, keys.ctypes.data, order.ctypes.data, parent.ctypes.data,
                          left.ctypes.data, right.ctypes.data, nmin.ctypes.data, nmax.ctypes.data, sb.ctypes.data)
    return dict(keys=keys, order=order, parent=parent, left=left, right=right, node_min=nmin, node_max=nmax, height=h, scene_bounds=sb)


def ploc_host(lmin_sorted: np.ndarray, lmax_sorted: np.ndarray, radius: int = 16):
    """Host mirror of the SAH-guided rebuild over sorted leaf boxes: dict(left, right, node_min, node_max, height, rounds)."""
    L = _load()
    lmin = np.ascontiguousarray(lmin_sorted, np.float32); lmax = np.ascontiguousarray(lmax_sorted, np.float32)
    n = len(lmin); ni = max(n - 1, 0)
    left = np.zeros(ni, np.int32); right = np.zeros(ni, np.int32)
    nmin = np.zeros((ni, 3), np.float32); nmax = np.zeros((ni, 3), np.float32)
    rounds = C.c_int(0)
    h = L.ploc_host_build(lmin.ctypes.data, lmax.ctypes.data, n, radius, left.ctypes.data, right.ctypes.data, nmin.ctypes.data, nmax.ctypes.data,
                          C.byref(rounds))
    return dict(left=left, right=right, node_min=nmin, node_max=nmax, height=h, rounds=rounds.value)


def wide_host(left, right, node_min, node_max, lmin_sorted, lmax_sorted, scene_bounds):
    """Host mirror of the four-wide collapse: dict(child (n,4), boxes (n,4,3), levels)."""
    L = _load()
    left = np.ascontiguousarray(left, np.int32); right = np.ascontiguousarray(right, np.int32)
    nmin = np.ascontiguousarray(node_min, np.float32); nmax = np.ascontiguousarray(node_max, np.float32)
    lmin = np.ascontiguousarray(lmin_sorted, np.float32); lmax = np.ascontiguousarray(lmax_sorted, np.float32)
    sb = np.ascontiguousarray(scene_bounds, np.float32)
    n = len(lmin)
    child = np.zeros((max(n - 1, 1), 4), np.int32); boxes = np.zeros((max(n - 1, 1), 4, 3), np.uint32)
    lev = C.c_int(0)
    nw = L.wide_host_build(left.ctypes.data, right.ctypes.data, nmin.ctypes.data, nmax.ctypes.data, lmin.ctypes.data, lmax.ctypes.data, n,
                           sb.ctypes.data, child.ctypes.data, boxes.ctypes.data, C.byref(lev))
    return dict(child=child[:nw], boxes=boxes[:nw], levels=lev.value)
