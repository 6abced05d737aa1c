"""The device ray-query entry points are exported and reject bad arguments before touching CUDA (no GPU needed)."""
import ctypes

import dogeray_b200 as drb


def test_ray_query_symbols_exported():
    lib = ctypes.CDLL(drb.LIB_PATH)
    for name in ("drb_trace_device", "drb_occluded_device"):
        assert hasattr(lib, name) and name in drb.EXPORTED_SYMBOLS


def test_ray_query_argument_errors():
    L = drb._lib
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    # null scene
    assert L.drb_trace_device(None, p, p, 1, p, None, None, None) == drb.ERR_ARG
    assert L.drb_occluded_device(None, p, p, None, 1, p, None) == drb.ERR_ARG
    assert b"bad argument" in L.drb_last_error()
    # negative n and null required pointers are refused before the handle is used; n == 0 does nothing
    fake = ctypes.create_string_buffer(4096)
    s = ctypes.addressof(fake)
    assert L.drb_trace_device(s, p, p, -1, p, None, None, None) == drb.ERR_ARG
    assert L.drb_occluded_device(s, p, p, None, -1, p, None) == drb.ERR_ARG
    assert L.drb_trace_device(s, p, p, 1, None, p, p, None) == drb.ERR_ARG
    assert L.drb_trace_device(s, None, p, 1, p, None, None, None) == drb.ERR_ARG
    assert L.drb_occluded_device(s, p, None, p, 1, p, None) == drb.ERR_ARG
    assert L.drb_occluded_device(s, p, p, p, 1, None, None) == drb.ERR_ARG
    assert L.drb_trace_device(s, None, None, 0, None, None, None, None) == drb.OK
    assert L.drb_occluded_device(s, None, None, None, 0, None, None) == drb.OK
