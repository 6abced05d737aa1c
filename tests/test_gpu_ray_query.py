"""Device-resident ray queries (drb_trace_device, drb_occluded_device and the torch wrappers Scene.trace / Scene.occluded)
against the host query drb_trace_ids, the brute-force definition and a float32 restatement of the barycentrics
(`pytest -m gpu` on a B200).

Bars: closest-hit ids and t bit-identical to drb_trace_ids; (u, v) bit-identical to intersect_prim's arithmetic;
occluded == (id >= 0) & (t < min(tmax, 1e4)) bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth
from oracle import restated
from conftest import HAVE_REF, ROOT, SAMPLES, sample

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
F = np.float32


def _torch():
    import torch
    return torch


def cuda(a):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda()


def query(sc, o, d, tmax=None):
    """closest hit (ids, t, uv) and occlusion through the torch wrappers, as numpy"""
    torch = _torch()
    to, td = cuda(o), cuda(d)
    ids, t, uv = sc.trace(to, td)
    occ = sc.occluded(to, td, None if tmax is None else cuda(tmax))
    torch.cuda.synchronize()
    return ids.cpu().numpy(), t.cpu().numpy(), uv.cpu().numpy(), occ.cpu().numpy()


def expected_occluded(ids, t, tmax):
    with np.errstate(invalid="ignore"):
        return (ids >= 0) & (t < np.minimum(tmax, F(1e4)))


def restated_uv(objs, ids, o, d):
    """intersect_prim's (u, v) in float32, operation by operation (-fmad=false), for the object each ray hit"""
    def cross(a, b):
        return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2], a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], 1)

    def dot(a, b):
        return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]

    uv = np.zeros((len(ids), 2), F)
    k = np.flatnonzero(ids >= 0)
    k = k[objs["type"][ids[k]] == 2]
    ob = objs[ids[k]]
    v0 = ob["pos"].astype(F)
    e1 = ob["dim"].astype(F) - v0
    e2 = ob["rot"].astype(F) - v0
    oo, dd = o[k].astype(F), d[k].astype(F)
    h = cross(dd, e2)
    f = F(1) / dot(e1, h)
    sv = oo - v0
    uv[k, 0] = f * dot(sv, h)
    uv[k, 1] = f * dot(dd, cross(sv, e1))
    return uv


def check_scene(sc, objs, o, d, rng, min_hits=1):
    """every query of this file on one scene and one ray set; returns (ids, t)"""
    o = np.ascontiguousarray(o, F).reshape(-1, 3); d = np.ascontiguousarray(d, F).reshape(-1, 3)
    hid, ht = sc.trace_ids(o, d)
    ids, t, uv, occ = query(sc, o, d)
    assert np.array_equal(ids, hid) and np.array_equal(t, ht)
    assert (ids >= 0).sum() >= min_hits
    assert np.array_equal(occ, ids >= 0)                                      # tmax NULL: 10000
    assert np.array_equal(uv.view(np.uint32), restated_uv(objs, ids, o, d).view(np.uint32))
    n = len(o)
    for tmax in (t.copy(),                                                    # exactly t: the hit is not below it
                 np.nextafter(t, F(np.inf)),                                  # one ulp above: it is
                 rng.uniform(0, 2 * max(float(t.max()), 1.0), n).astype(F),
                 np.zeros(n, F), np.full(n, -1.0, F), np.full(n, np.inf, F),
                 np.choose(rng.integers(0, 4, n), [t, np.full(n, np.nan, F), np.full(n, -np.inf, F), np.full(n, 2e4, F)]).astype(F)):
        _, _, _, occ = query(sc, o, d, tmax)
        assert np.array_equal(occ, expected_occluded(ids, t, tmax))
    return ids, t


def scene_from(objs, st=None):
    return drb.Scene.from_host(drb.HostScene.from_objects(objs, st))


def sphere_objects(rng, n, spheres_every=1):
    o = drb.make_objects(n)
    c = rng.uniform(-4, 4, (n, 3)).astype(F)
    o["pos"] = c
    o["dim"] = c + rng.uniform(-0.6, 0.6, (n, 3)).astype(F)
    o["rot"] = c + rng.uniform(-0.6, 0.6, (n, 3)).astype(F)
    sph = np.arange(n) % spheres_every == 0
    o["type"][sph] = 0
    o["dim"][sph, 0] = rng.uniform(0.1, 0.5, int(sph.sum()))
    return o


def random_rays(rng, n, spread=6.0):
    o = rng.uniform(-spread, spread, (n, 3)).astype(F)
    d = rng.normal(size=(n, 3)).astype(F)
    d[::7, 0] = 0.0; d[::11, 2] = 0.0; d[::13] = (0.0, 0.0, 0.0)              # axis-parallel and zero directions
    return o, d


def test_golden_heightfield_and_materials_rays(tmp_path):
    rng = np.random.default_rng(1)
    g = np.load(os.path.join(GOLDEN, "synth_heightfield.npz"))
    objs, st = synth.heightfield_scene(n=24, width=48, height=40, spp=3, max_depth=5)
    p = str(tmp_path / "hf.rts")
    drb.write_rts(p, st, objs)
    hs = drb.HostScene.load(p)
    ids, t = check_scene(drb.Scene.from_host(hs), hs.objects(), g["origins"], g["dirs"], rng, min_hits=100)
    assert np.array_equal(ids, g["ids"].reshape(-1)) and np.array_equal(t, g["t"].reshape(-1))

    g = np.load(os.path.join(GOLDEN, "synth_materials.npz"))
    tex = synth.write_test_textures(str(tmp_path))
    objs, st, tp = synth.materials_scene(tex, width=96, height=56, spp=3, max_depth=6, nu=24, nv=12)
    p = str(tmp_path / "mats.rts")
    drb.write_rts(p, st, objs, tex_names=[os.path.basename(x) for x in tp], backtex_name=os.path.basename(tp[0]))
    hs = drb.HostScene.load(p, str(tmp_path))
    ids, t = check_scene(drb.Scene.from_host(hs), hs.objects(), g["origins"], g["dirs"], rng, min_hits=100)
    assert np.array_equal(ids, g["ids"].reshape(-1)) and np.array_equal(t, g["t"].reshape(-1))


def test_incoherent_rays_against_brute_force(tmp_path):
    rng = np.random.default_rng(5)
    objs, st = synth.heightfield_scene(n=60)
    p = str(tmp_path / "hf.rts")
    drb.write_rts(p, st, objs)
    hs = drb.HostScene.load(p)
    n = 20000
    o = rng.uniform(-6, 6, (n, 3)).astype(F); o[:, 1] = -np.abs(o[:, 1]) - 0.5
    d = rng.normal(size=(n, 3)).astype(F); d[:, 1] = np.abs(d[:, 1])
    d[::7, 0] = 0.0; d[::11, 2] = 0.0; d[::13] = 0.0
    ids, t = check_scene(drb.Scene.from_host(hs), hs.objects(), o, d, rng, min_hits=n // 10)
    bid, bt = restated.Restated(p).hit_brute(o, d)
    bad = np.flatnonzero(ids != bid)                                          # only an exact tie in t may pick another object
    assert len(bad) <= 5 and all(ids[k] >= 0 and bid[k] >= 0 and t[k] == bt[k] for k in bad)
    same = (ids == bid) & (bid >= 0)
    assert np.array_equal(t[same], bt[same])


@pytest.mark.parametrize("spheres_every", [1, 3])
def test_sphere_and_mixed_scenes(spheres_every):
    rng = np.random.default_rng(spheres_every)
    objs = sphere_objects(rng, 300, spheres_every)
    o, d = random_rays(rng, 20000)
    check_scene(scene_from(objs), objs, o, d, rng, min_hits=1000)


def test_empty_one_object_and_far_scenes():
    rng = np.random.default_rng(7)
    o, d = random_rays(rng, 3000)
    empty = drb.make_objects(0)
    ids, _ = check_scene(scene_from(empty), empty, o, d, rng, min_hits=0)
    assert (ids == -1).all()
    one = drb.make_objects(1)
    one["pos"], one["dim"], one["rot"] = (-1, -1, 0), (1, -1, 0), (0, 1, 0)
    o1 = np.concatenate([o, np.tile(F([[0.2, 0.1, 2.0]]), (500, 1))]); d1 = np.concatenate([d, np.tile(F([[0, 0, -1]]), (500, 1))])
    check_scene(scene_from(one), one, o1, d1, rng, min_hits=500)
    # the small scene ~10^5 scene sizes from the origin of test_small_scene_far_from_the_origin
    n = 7
    far = drb.make_objects(n)
    c = (np.array([4000.0, -3000.0, 5000.0]) + rng.uniform(-0.004, 0.004, (n, 3))).astype(F)
    far["pos"] = c; far["dim"] = c + rng.uniform(-0.004, 0.004, (n, 3)).astype(F); far["rot"] = c + rng.uniform(-0.004, 0.004, (n, 3)).astype(F)
    m = 4096
    ro = (np.array([4000.0, -3000.0, 5000.0]) + rng.normal(size=(m, 3)) * 3).astype(F)
    rd = ((c[rng.integers(0, n, m)] + rng.uniform(-0.003, 0.003, (m, 3)) - ro) * 40).astype(F)
    ids, t = check_scene(scene_from(far), far, ro, rd, rng, min_hits=50)
    bid, bt = restated.brute_tris(far["pos"], far["dim"], far["rot"], ro, rd)
    same = ids == bid
    assert (same | ((ids >= 0) & (bid >= 0) & (t == bt))).all() and np.array_equal(t[same & (bid >= 0)], bt[same & (bid >= 0)])


def test_scene_on_the_sorted_push_variant():
    """above DRB_SORTED_PUSH_FROM (4 Mi primitives) the closest-hit query runs k_trace<true>"""
    rng = np.random.default_rng(11)
    objs, st = synth.instanced_grid_scene(grid=8, width=160, height=90)
    sc = scene_from(objs, st)
    assert sc.num_prims >= 4 << 20
    o, d = sc.primary_rays(st, 0, seed=1)
    check_scene(sc, objs, o, d, rng, min_hits=5000)


@pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref not available")
def test_sample_scenes():
    rng = np.random.default_rng(3)
    for name in ("cube.rts", "mats.rts", "SPERSSSSS.rts", "cow.rts"):
        hs = drb.HostScene.load(sample(name), SAMPLES)
        objs = hs.objects()
        sc = drb.Scene.from_host(hs)
        st = sc.settings.replace(width=96, height=64)
        o, d = sc.primary_rays(st, 0, seed=2)
        check_scene(sc, objs, o, d, rng)


_CHUNK_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
import dogeray_b200 as drb
from dogeray_b200 import synth
objs, st = synth.heightfield_scene(n=30)
sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
rng = np.random.default_rng(9)
n = 2731
o = torch.from_numpy(rng.uniform(-6, 6, (n, 3)).astype(np.float32)).cuda(); o[:, 1] = -o[:, 1].abs() - 0.5
d = torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32)).cuda(); d[:, 1] = d[:, 1].abs()
tmax = torch.from_numpy(rng.uniform(0, 12, n).astype(np.float32)).cuda()
ids, t, uv = sc.trace(o, d)
occ = sc.occluded(o, d, tmax)
torch.cuda.synchronize()
np.savez(sys.argv[2], ids=ids.cpu().numpy(), t=t.cpu().numpy(), uv=uv.cpu().numpy(), occ=occ.cpu().numpy())
"""


def test_chunked_queries_equal_one_chunk(tmp_path):
    out = {}
    for chunk in (None, "1000"):
        env = dict(os.environ)
        env.pop("DOGERAY_B200_QUERY_CHUNK", None)
        if chunk:
            env["DOGERAY_B200_QUERY_CHUNK"] = chunk
        path = str(tmp_path / ("r%s.npz" % chunk))
        r = subprocess.run([sys.executable, "-c", _CHUNK_SCRIPT, ROOT, path], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        out[chunk] = np.load(path)
    a, b = out[None], out["1000"]
    assert (a["ids"] >= 0).sum() > 200 and a["occ"].any() and not a["occ"].all()
    for k in ("ids", "t", "uv", "occ"):
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), k


def test_queries_leave_renders_and_host_queries_alone():
    torch = _torch()
    objs, st = synth.heightfield_scene(n=20, width=64, height=40, spp=2, max_depth=4)
    sc = scene_from(objs, st)
    o, d = sc.primary_rays(st, 0, seed=5)
    ids0, t0 = sc.trace_ids(o, d)
    ref = scene_from(objs, st)
    a1, s1 = ref.render(st, seed=8)
    a2, s2 = ref.render(st, seed=8)
    b1, r1 = sc.render(st, seed=8)
    rng = np.random.default_rng(2)
    n = 64 * 40 * 2 * 3                                                       # more rays than the render's batch holds
    qo = cuda(rng.uniform(-6, 6, (n, 3)).astype(F)); qd = cuda(rng.normal(size=(n, 3)).astype(F))
    sc.trace(qo, qd); sc.occluded(qo, qd)
    torch.cuda.synchronize()
    b2, r2 = sc.render(st, seed=8)
    assert np.array_equal(a1, b1) and np.array_equal(a2, b2)
    for x, y in ((s1, r1), (s2, r2)):
        assert (x.paths, x.rays, x.kernel_launches, x.trace_launches) == (y.paths, y.rays, y.kernel_launches, y.trace_launches)
    ids1, t1 = sc.trace_ids(o, d)
    assert np.array_equal(ids0, ids1) and np.array_equal(t0, t1)


def test_torch_wrappers_shapes_pointers_streams_and_errors():
    torch = _torch()
    objs, st = synth.heightfield_scene(n=24, width=48, height=40)
    sc = scene_from(objs, st)
    o, d = sc.primary_rays(st, 0, seed=3)                                     # (H, W, 3)
    to, td = cuda(o), cuda(d)
    tmax = torch.rand(40, 48, device="cuda") * 8
    ids, t, uv = sc.trace(to, td)
    occ = sc.occluded(to, td, tmax)
    assert ids.shape == (40, 48) and t.shape == (40, 48) and uv.shape == (40, 48, 2) and occ.shape == (40, 48)
    assert ids.dtype == torch.int32 and occ.dtype == torch.bool
    assert sc.trace(to, td, with_uv=False)[2] is None
    # pointer level on the caller's stream
    n = 40 * 48
    pids = torch.empty(n, dtype=torch.int32, device="cuda"); pt = torch.empty(n, device="cuda"); puv = torch.empty(n, 2, device="cuda")
    pocc = torch.empty(n, dtype=torch.uint8, device="cuda")
    cs = torch.cuda.current_stream().cuda_stream
    sc.trace_device(to.data_ptr(), td.data_ptr(), n, pids.data_ptr(), pt.data_ptr(), puv.data_ptr(), stream=cs)
    sc.occluded_device(to.data_ptr(), td.data_ptr(), n, pocc.data_ptr(), tmax.data_ptr(), stream=cs)
    torch.cuda.synchronize()
    assert torch.equal(pids, ids.reshape(-1)) and torch.equal(pt, t.reshape(-1)) and torch.equal(puv, uv.reshape(-1, 2))
    assert torch.equal(pocc.bool(), occ.reshape(-1))
    assert (ids >= 0).sum() > 100
    # rays produced on a side stream and queried there, read after that stream synchronises
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        so = torch.from_numpy(o).to("cuda", non_blocking=False) * 1.0
        sd = torch.from_numpy(d).to("cuda") + 0.0
        sids, stt, suv = sc.trace(so, sd)
        socc = sc.occluded(so, sd, tmax * 1.0)
    s.synchronize()
    assert torch.equal(sids, ids) and torch.equal(stt, t) and torch.equal(suv, uv) and torch.equal(socc, occ)
    # an explicit stream argument outside a stream context
    s2 = torch.cuda.Stream()
    s2.wait_stream(torch.cuda.current_stream())
    xids, _, _ = sc.trace(to, td, stream=s2)
    s2.synchronize()
    assert torch.equal(xids, ids)
    # wrong dtype / device / shape
    for bad in (to.double(), to.cpu()):
        with pytest.raises(ValueError):
            sc.trace(bad, td)
        with pytest.raises(ValueError):
            sc.occluded(bad, td)
    with pytest.raises(ValueError):
        sc.occluded(to, td, tmax.double())
    with pytest.raises(ValueError):
        sc.trace(to[..., :2], td[..., :2])
    # n == 0 and argument errors through the C ABI
    assert drb._lib.drb_trace_device(sc.handle, None, None, 0, None, None, None, None) == drb.OK
    assert drb._lib.drb_occluded_device(sc.handle, None, None, None, -1, None, None) == drb.ERR_ARG
    assert drb._lib.drb_trace_device(sc.handle, to.data_ptr(), None, 5, pids.data_ptr(), None, None, None) == drb.ERR_ARG
