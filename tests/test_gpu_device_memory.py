"""Device memory comes back (`pytest -m gpu` on a B200).

Every device array the library allocates -- scene arrays, build scratch, render queues, query buffers, per-call uploads --
goes back to the block cache, and from there to the pool with drb_trim.  A leak on the create -> render -> free cycle would
stay hidden behind the cache until the device runs out of memory, so this reads the default pool's own counters through
the driver: the process-local used memory, which other users of the GPU do not change (cudaMemGetInfo would see them), and
the reserved high-water mark, which grows only when the pool asks the driver for more.  torch's default allocator does not
use the default pool."""
import ctypes
import os

import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth

pytestmark = pytest.mark.gpu

CU_MEMPOOL_ATTR_RESERVED_MEM_HIGH = 6
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


class Pool:
    """device 0's default memory pool, read through libcuda"""

    def __init__(self):
        self.cu = ctypes.CDLL("libcuda.so.1")
        assert self.cu.cuInit(0) == 0
        dev = ctypes.c_int()
        assert self.cu.cuDeviceGet(ctypes.byref(dev), 0) == 0
        self.pool = ctypes.c_void_p()
        assert self.cu.cuDeviceGetDefaultMemPool(ctypes.byref(self.pool), dev) == 0

    def attr(self, which):
        v = ctypes.c_uint64()
        assert self.cu.cuMemPoolGetAttribute(self.pool, which, ctypes.byref(v)) == 0
        return v.value

    def used(self):
        return self.attr(CU_MEMPOOL_ATTR_USED_MEM_CURRENT)

    def reserved_high(self):
        return self.attr(CU_MEMPOOL_ATTR_RESERVED_MEM_HIGH)


def settings(w, h):
    st = drb.default_settings()
    st.cam[:] = [0.0, 3.0, 12.0]
    st.width, st.height, st.spp, st.max_depth = w, h, 2, 4
    return st


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    torch = pytest.importorskip("torch")
    if "cudaMallocAsync" in os.environ.get("PYTORCH_CUDA_ALLOC_CONF", ""):
        pytest.skip("torch allocates from the default pool (PYTORCH_CUDA_ALLOC_CONF selects cudaMallocAsync)")
    td = str(tmp_path_factory.mktemp("memory"))
    tex = synth.write_test_textures(td)
    objs, st, tp = synth.materials_scene(tex, width=64, height=40, spp=2, max_depth=4, nu=24, nv=12)
    one = drb.make_objects(1)
    one["pos"], one["dim"], one["rot"] = (-1, -1, 0), (1, -1, 0), (0, 1, 0)
    bad = objs.copy()
    bad["texnum"] = len(tp)                                  # every line names a texture that does not load
    rng = np.random.default_rng(0)
    n = 5000
    o = np.tile(np.asarray(st.cam, np.float32), (n, 1))
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    # every torch tensor exists before the baseline
    dev = torch.device("cuda", 0)
    return dict(objs=objs, st=st, tp=tuple(tp), one=one, bad=bad, bad_tp=tuple(tp) + (os.path.join(td, "missing.ppm"),),
                o=o, d=d, to=torch.from_numpy(o).to(dev), td=torch.from_numpy(d).to(dev),
                tobjs=torch.from_numpy(objs.view(np.uint8).copy()).to(dev), torch=torch)


def cycle(x):
    """one round of everything that owns device memory"""
    torch, objs, st, tp = x["torch"], x["objs"], x["st"], x["tp"]
    hs = drb.HostScene.from_objects(objs, st, tp)
    for flags in (0, drb.BUILD_KEEP_DEBUG, drb.BUILD_LBVH_ONLY):
        drb.Scene.from_host(hs, build_flags=flags).close()
    for lines in (drb.make_objects(0), x["one"]):
        sc = drb.Scene.from_host(drb.HostScene.from_objects(lines, settings(32, 24)))
        sc.render(settings(32, 24))
        sc.trace_ids(x["o"][:100], x["d"][:100])
        sc.close()
    torch.cuda.synchronize()
    drb.Scene.from_device_objects(hs, x["tobjs"].data_ptr()).close()
    sc = drb.Scene.from_host(hs)
    sc.render(settings(32, 24))
    sc.render(settings(96, 64))                              # larger queues: the first set goes back
    ids, t, uv = sc.trace(x["to"], x["td"])
    occ = sc.occluded(x["to"], x["td"])
    torch.cuda.synchronize()
    del ids, t, uv, occ
    sc.trace_ids(x["o"], x["d"])
    sc.primary_rays(settings(48, 32))
    sc.frame_i3(settings(48, 32), divisor=1)
    sc.refit(objs)
    refused = objs.copy()
    refused["pos"][:, 0] = np.nan                           # every rendered line
    with pytest.raises(drb.DogerayError):
        sc.refit(refused)
    sc.close()
    with pytest.raises(drb.DogerayError):
        drb.Scene.from_host(drb.HostScene.from_objects(x["bad"], st, x["bad_tp"]))


def test_every_cycle_returns_its_memory_and_reuses_the_cache(inputs):
    pool = Pool()
    cycle(inputs)                                            # lazy module loading, the facts cache, torch's own set-up
    drb.trim(0)
    base = pool.used()
    cycle(inputs)
    high = pool.reserved_high()
    for k in range(3):
        cycle(inputs)
        assert pool.reserved_high() == high, "cycle %d asked the pool for more memory (%d -> %d bytes)" % (k + 2, high, pool.reserved_high())
    drb.trim(0)
    assert pool.used() == base, "%d bytes of device memory did not come back" % (pool.used() - base)
