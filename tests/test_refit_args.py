"""The refit entry points are exported and reject bad arguments before touching CUDA (no GPU needed)."""
import ctypes

import numpy as np
import pytest

import dogeray_b200 as drb


def test_refit_symbols_exported():
    lib = ctypes.CDLL(drb.LIB_PATH)
    for name in ("drb_scene_refit_device", "drb_scene_refit"):
        assert hasattr(lib, name) and name in drb.EXPORTED_SYMBOLS


def test_refit_argument_errors():
    L = drb._lib
    buf = ctypes.create_string_buffer(156 * 4)
    p = ctypes.addressof(buf)
    # null scene
    assert L.drb_scene_refit_device(None, p, 1, None) == drb.ERR_ARG
    assert L.drb_scene_refit(None, p, 1) == drb.ERR_ARG
    assert b"bad argument" in L.drb_last_error()
    # null objects and n < 0 are refused before the handle is used
    fake = ctypes.create_string_buffer(4096)
    s = ctypes.addressof(fake)
    assert L.drb_scene_refit_device(s, None, 1, None) == drb.ERR_ARG
    assert L.drb_scene_refit(s, None, 1) == drb.ERR_ARG
    assert L.drb_scene_refit_device(s, p, -1, None) == drb.ERR_ARG
    assert L.drb_scene_refit(s, p, -1) == drb.ERR_ARG


def test_refit_rejects_bad_host_arrays_before_the_library():
    fake = ctypes.create_string_buffer(4096)                                  # a zeroed handle: num_objects == 0
    sc = drb.Scene(ctypes.c_void_p(ctypes.addressof(fake)))
    called = []
    real = drb._lib.drb_scene_refit
    try:
        drb._lib.drb_scene_refit = lambda *a: called.append(a) or 0
        for bad in (np.zeros(0, np.float32), np.zeros(3, drb.OBJECT_DTYPE), np.zeros((0, 2), drb.OBJECT_DTYPE), [1, 2]):
            with pytest.raises(ValueError):
                sc.refit(bad)
        assert not called
        sc.refit(np.zeros(0, drb.OBJECT_DTYPE))                               # right dtype and length reaches the library
        assert len(called) == 1
    finally:
        drb._lib.drb_scene_refit = real
        sc._h = None                                                          # not a real scene: nothing to free
