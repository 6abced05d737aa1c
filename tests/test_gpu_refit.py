"""Scene refit (drb_scene_refit / drb_scene_refit_device, Scene.refit) against the build it started from, a numpy mirror
of the integer-union box update, a fresh build of the moved geometry and the brute-force hit (`pytest -m gpu` on a B200).

Bars: refitting unchanged lines changes no bit of the nodes, bounds, queries or renders; after any move every node box
equals the float32 mirror (leaf boxes quantised on the grid of the new bounds, integer union bottom-up over the unchanged
links); queries equal a fresh build's up to exact-t ties; refused refits leave the scene untouched."""
import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth
from oracle import restated

pytestmark = pytest.mark.gpu

F = np.float32
EMPTY = np.int32(-2 ** 31)
DEBUG = drb.BUILD_KEEP_DEBUG


def _torch():
    import torch
    return torch


# ---- scenes ---------------------------------------------------------------------------------------------

def settings(w=48, h=32, spp=2, depth=4):
    st = drb.default_settings()
    st.cam[:] = [0.0, 3.0, 12.0]
    st.width, st.height, st.spp, st.max_depth = w, h, spp, depth
    return st


def heightfield():
    objs, st = synth.heightfield_scene(n=24, width=48, height=32, spp=2, max_depth=4)
    return objs, st, ()


def mixed(seed=4):
    rng = np.random.default_rng(seed)
    n = 300
    o = drb.make_objects(n)
    c = rng.uniform(-4, 4, (n, 3)).astype(F)
    o["pos"] = c
    o["dim"] = c + rng.uniform(-0.6, 0.6, (n, 3)).astype(F)
    o["rot"] = c + rng.uniform(-0.6, 0.6, (n, 3)).astype(F)
    sph = np.arange(n) % 3 == 0
    o["type"][sph] = 0
    o["dim"][sph, 0] = rng.uniform(0.1, 0.5, int(sph.sum()))
    o["col"] = rng.uniform(0.2, 0.9, (n, 3)).astype(F)
    o["mat"][::7] = 1
    return o, settings(), ()


def materials(tmp_path):
    tex = synth.write_test_textures(str(tmp_path))
    objs, st, tp = synth.materials_scene(tex, width=64, height=40, spp=2, max_depth=4, nu=24, nv=12)
    return objs, st, tuple(tp)


def one():
    o = drb.make_objects(1)
    o["pos"], o["dim"], o["rot"] = (-1, -1, 0), (1, -1, 0), (0, 1, 0)
    st = settings()
    st.cam[:] = [0.0, 0.0, 4.0]
    return o, st, ()


def build(objs, st, tp=(), flags=DEBUG):
    return drb.Scene.from_host(drb.HostScene.from_objects(objs, st, tp), build_flags=flags)


def renderable(objs):
    r = ((objs["type"] == 2) & ((objs["ncols"] == 0) | (objs["ncols"] >= 16))) | ((objs["type"] == 0) & ((objs["ncols"] == 0) | (objs["ncols"] >= 10)))
    return np.flatnonzero(r)


# ---- the numpy mirror -----------------------------------------------------------------------------------

def leaf_boxes(objs):
    p, d, r = objs["pos"].astype(F), objs["dim"].astype(F), objs["rot"].astype(F)
    lo = np.minimum(p, np.minimum(d, r)); hi = np.maximum(p, np.maximum(d, r))
    sph = objs["type"] == 0
    rad = np.abs(d[:, :1])
    lo[sph] = (p - rad)[sph]; hi[sph] = (p + rad)[sph]
    return lo, hi


def mirror(sc, objs):
    """(boxes (nwide, 4, 3) uint32, bounds min, bounds max) the refit must produce for `objs` on `sc`'s links"""
    child = sc.wide()["child"]
    lines = renderable(objs)[sc.lbvh()["order"]]                             # slot -> object line
    lo, hi = leaf_boxes(objs[lines])
    bmin, bmax = lo.min(0), hi.max(0)
    ext = bmax - bmin
    ext = np.where(ext > 0, ext, F(1)).astype(F)
    qs = (ext / F(65527)).astype(F)
    qlo = (bmin - F(4) * qs).astype(F)
    a = np.clip(np.floor((lo - qlo) / qs).astype(np.int64) - 1, 0, 65535)
    b = np.clip(np.ceil((hi - qlo) / qs).astype(np.int64) + 1, 0, 65535)
    leaf_q = (a | (b << 16)).astype(np.uint32)
    levels = [np.array([0])] if len(child) else []
    while levels:
        c = child[levels[-1]].reshape(-1)
        nxt = np.sort(c[c >= 0])
        if not len(nxt):
            break
        levels.append(nxt)
    boxes = np.zeros((len(child), 4, 3), np.uint32)
    for lv in reversed(levels):
        for k in range(4):
            c = child[lv, k]
            q = np.full((len(lv), 3), 0xFFFF, np.uint32)
            leaf = (c < 0) & (c != EMPTY)
            q[leaf] = leaf_q[~c[leaf]]
            inner = c >= 0
            cb = boxes[c[inner]]
            q[inner] = (cb & 0xFFFF).min(1) | ((cb >> 16).max(1) << 16)
            boxes[lv, k] = q
    return boxes, bmin, bmax


# ---- observations ---------------------------------------------------------------------------------------

def rays(st, n=4000, seed=0):
    rng = np.random.default_rng(seed)
    cam = np.array(st.cam, F)
    o = (cam + rng.normal(size=(n, 3)) * 0.5).astype(F)
    d = (rng.uniform(-6, 6, (n, 3)).astype(F) - o).astype(F)
    return o, d


def query(sc, o, d):
    torch = _torch()
    to, td = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    ids, t, uv = sc.trace(to, td)
    occ = sc.occluded(to, td)
    torch.cuda.synchronize()
    return ids.cpu().numpy(), t.cpu().numpy(), uv.cpu().numpy(), occ.cpu().numpy()


def snapshot(sc, st, o, d):
    w = sc.wide()
    bi = sc.build_info
    ids, t, uv, occ = query(sc, o, d)
    img, stats = sc.render(st, seed=3)
    return dict(child=w["child"], boxes=w["boxes"], bmin=np.array(bi.bounds_min, F), bmax=np.array(bi.bounds_max, F),
                info=(bi.nprims, bi.nnodes, bi.nwide, bi.wide_levels, bi.stack_levels, bi.max_depth, bi.rebuild_iterations),
                ids=ids, t=t, uv=uv, occ=occ, img=img, rays=np.array([stats.rays, stats.paths]))


def assert_same(a, b):
    for k in a:
        if k == "info":
            assert a[k] == b[k]
        else:
            assert np.array_equal(np.ascontiguousarray(a[k]).view(np.uint8), np.ascontiguousarray(b[k]).view(np.uint8)), k


def agree(a, b, ties_ok=True):
    """closest hits of two scenes over the same geometry: equal, except another id at an exact tie in t"""
    ids, t, uv, occ = a
    jds, s, vu, occ2 = b
    assert np.array_equal(t.view(np.uint32), s.view(np.uint32)) and np.array_equal(occ, occ2)
    same = ids == jds
    assert np.array_equal(uv[same].view(np.uint32), vu[same].view(np.uint32))
    bad = ~same
    assert ties_ok or not bad.any()
    assert bad.sum() <= max(5, len(ids) // 1000) and ((ids[bad] >= 0) & (jds[bad] >= 0)).all()


def images_agree(a, b, exact):
    ia, sa = a
    ib, sb = b
    if exact:
        assert np.array_equal(ia.view(np.uint32), ib.view(np.uint32)) and sa.rays == sb.rays
    else:
        same = np.all(ia.view(np.uint32) == ib.view(np.uint32), axis=-1).mean()
        assert same >= 0.999, same
        if same == 1.0:
            assert sa.rays == sb.rays


# ---- deformations ---------------------------------------------------------------------------------------

def deform(objs, kind, rng):
    o = objs.copy()
    tri = o["type"] == 2
    if kind == "jitter":
        for f in ("pos", "dim", "rot"):
            o[f][tri] += rng.normal(0, 0.01, (int(tri.sum()), 3)).astype(F)
        o["pos"][~tri] += rng.normal(0, 0.05, (int((~tri).sum()), 3)).astype(F)
        o["dim"][~tri, 0] *= rng.uniform(0.8, 1.2, int((~tri).sum())).astype(F)
    elif kind == "rigid":
        part = np.arange(len(o)) < len(o) // 2
        c, s = np.cos(0.7), np.sin(0.7)
        R = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]], F)
        for f in ("pos", "dim", "rot"):
            m = part & (tri | (f == "pos"))
            o[f][m] = (o[f][m] @ R.T + F([1.5, 0.25, -0.5])).astype(F)
    elif kind == "translate":
        for f in ("pos", "dim", "rot"):
            m = tri | (f == "pos")
            o[f][m] = (o[f][m] + F([1e3, -1e3, 1e3])).astype(F)
    elif kind == "scale":
        for f in ("pos", "dim", "rot"):
            m = tri | (f == "pos")
            o[f][m] = (o[f][m] * F(1e-3)).astype(F)
        o["dim"][~tri, 0] *= F(1e-3)
    return o


def moved_rays(st, objs, kind, n=4000, seed=1):
    """rays aimed at the moved geometry (the camera moves with a translation or scaling)"""
    rng = np.random.default_rng(seed)
    lines = renderable(objs)
    lo, hi = leaf_boxes(objs[lines])
    c = ((lo + hi) * F(0.5))[rng.integers(0, len(lines), n)]
    ext = float((hi.max(0) - lo.min(0)).max())
    o = (c + rng.normal(size=(n, 3)) * ext).astype(F)
    d = (c + rng.normal(size=(n, 3)) * ext * 0.01 - o).astype(F)
    return o, d


# ---- 1. identity ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["heightfield", "mixed", "materials", "one", "empty", "lbvh_only"])
def test_refit_with_unchanged_lines_changes_nothing(name, tmp_path):
    flags = DEBUG
    if name == "materials":
        objs, st, tp = materials(tmp_path)
    elif name == "one":
        objs, st, tp = one()
    elif name == "empty":
        objs, st, tp = drb.make_objects(0), settings(), ()
    elif name == "mixed":
        objs, st, tp = mixed()
    else:
        objs, st, tp = heightfield()
        if name == "lbvh_only":
            flags |= drb.BUILD_LBVH_ONLY
    sc = build(objs, st, tp, flags)
    o, d = rays(st)
    before = snapshot(sc, st, o, d)
    sc.refit(objs)
    assert_same(before, snapshot(sc, st, o, d))
    torch = _torch()
    sc.refit(torch.from_numpy(objs.view(np.uint8).copy()).cuda())
    assert_same(before, snapshot(sc, st, o, d))


# ---- 2 + 3. deformed geometry: the mirror and a fresh build ---------------------------------------------

@pytest.mark.parametrize("scene", ["heightfield", "mixed", "lbvh_only"])
@pytest.mark.parametrize("kind", ["jitter", "rigid", "translate", "scale"])
def test_deformed_geometry_matches_mirror_and_fresh_build(scene, kind):
    rng = np.random.default_rng(sum(map(ord, scene + kind)))
    objs, st, tp = mixed() if scene == "mixed" else heightfield()
    flags = DEBUG | (drb.BUILD_LBVH_ONLY if scene == "lbvh_only" else 0)
    sc = build(objs, st, tp, flags)
    child0 = sc.wide()["child"].copy()
    moved = deform(objs, kind, rng)
    sc.refit(moved)
    w = sc.wide()
    assert np.array_equal(w["child"], child0)
    boxes, bmin, bmax = mirror(sc, moved)
    assert np.array_equal(w["boxes"], boxes)
    bi = sc.build_info
    assert np.array_equal(np.array(bi.bounds_min, F), bmin) and np.array_equal(np.array(bi.bounds_max, F), bmax)
    fresh = build(moved, st, tp, flags)
    o, d = moved_rays(st, moved, kind)
    a, b = query(sc, o, d), query(fresh, o, d)
    # hit_tri's absolute epsilons (|det| >= 1e-4, t > 1e-4) make triangles of a 1e-3-scaled heightfield unhittable for any
    # ray scale, so there only the nodes, the bounds and the (empty) query results are compared
    assert (a[0] >= 0).sum() > (-1 if kind == "scale" and scene != "mixed" else 100)
    agree(a, b)
    if scene != "mixed":                                                      # triangles only: the brute-force hit
        bid, bt = restated.brute_tris(moved["pos"], moved["dim"], moved["rot"], o, d)
        ids, t = a[0], a[1]
        same = ids == bid
        assert (same | ((ids >= 0) & (bid >= 0) & (t == bt))).all()
        assert np.array_equal(t[bid >= 0], bt[bid >= 0])
    if kind in ("jitter", "rigid"):                                           # the camera still sees the scene
        images_agree(sc.render(st, seed=5), fresh.render(st, seed=5), exact=scene == "mixed")


# ---- 4. materials ---------------------------------------------------------------------------------------

def test_changed_materials_render_like_a_fresh_build(tmp_path):
    objs, st, tp = materials(tmp_path)
    sc = build(objs, st, tp, 0)
    rng = np.random.default_rng(8)
    m = objs.copy()
    n = len(m)
    m["col"] = rng.uniform(0.1, 1.0, (n, 3)).astype(F)
    m["mat"] = rng.choice([0, 1, 2, 3, 4, 5], n)
    m["add_y"] = rng.uniform(0.0, 0.5, n).astype(F)
    m["texnum"] = rng.choice([-1, 1], n)
    m["rtexnum"] = rng.choice([-1, 1], n)
    m["checker"] = rng.integers(0, 2, n)
    sc.refit(m)
    fresh = build(m, st, tp, 0)
    images_agree(sc.render(st, seed=2), fresh.render(st, seed=2), exact=True)


# ---- 5. refusals ----------------------------------------------------------------------------------------

def test_refused_refits_leave_the_scene_untouched():
    torch = _torch()
    objs, st, _ = heightfield()
    extra = drb.make_objects(3)
    extra["type"] = 1                                                         # not renderable
    objs = np.concatenate([objs, extra])
    sc = build(objs, st)
    o, d = rays(st)
    base = snapshot(sc, st, o, d)
    n = len(objs)
    cases = []
    b = objs.copy(); b["type"][17] = 0; cases.append((b, 17))               # kind change
    b = objs.copy(); b["type"][n - 2] = 2; cases.append((b, n - 2))         # a line becomes renderable
    b = objs.copy(); b["ncols"][5] = 3; cases.append((b, 5))                # a line stops being renderable
    b = objs.copy(); b["dim"][40, 1] = np.nan; cases.append((b, 40))        # NaN vertex
    b = objs.copy(); b["rot"][41, 0] = np.inf; b["pos"][60, 2] = np.nan; cases.append((b, 41))
    for bad, line in cases:
        moved = deform(bad, "jitter", np.random.default_rng(line))
        moved["type"], moved["ncols"] = bad["type"], bad["ncols"]
        with pytest.raises(drb.DogerayError) as e:
            sc.refit(moved)
        assert e.value.status == drb.ERR_ARG and ("line %d " % line) in str(e.value), str(e.value)
        assert_same(base, snapshot(sc, st, o, d))
        tb = torch.from_numpy(moved.view(np.uint8).copy()).cuda()
        assert drb._lib.drb_scene_refit_device(sc.handle, tb.data_ptr(), n, None) == drb.ERR_ARG
        assert_same(base, snapshot(sc, st, o, d))
    more = torch.from_numpy(np.concatenate([objs, objs[:1]]).view(np.uint8).copy()).cuda()
    assert drb._lib.drb_scene_refit_device(sc.handle, more.data_ptr(), n + 1, None) == drb.ERR_ARG
    assert drb._lib.drb_scene_refit(sc.handle, objs.ctypes.data, n - 1) == drb.ERR_ARG
    assert_same(base, snapshot(sc, st, o, d))


# ---- 6. many steps --------------------------------------------------------------------------------------

def test_fifty_refits_then_fresh_build_and_mirror():
    objs, st, _ = mixed(9)
    sc = build(objs, st)
    o, d = rays(st)
    query(sc, o, d); sc.render(st, seed=1)                                   # query and render buffers exist
    rng = np.random.default_rng(10)
    cur = objs
    for step in range(50):
        cur = deform(cur, ("jitter", "rigid")[step % 2], rng)
        sc.refit(cur)
    boxes, bmin, bmax = mirror(sc, cur)
    assert np.array_equal(sc.wide()["boxes"], boxes)
    assert np.array_equal(np.array(sc.build_info.bounds_min, F), bmin)
    fresh = build(cur, st)
    o, d = moved_rays(st, cur, "jitter")
    agree(query(sc, o, d), query(fresh, o, d))
    images_agree(sc.render(st, seed=4), fresh.render(st, seed=4), exact=True)


# ---- 7. torch and streams -------------------------------------------------------------------------------

def test_torch_side_stream_refit_then_queries():
    torch = _torch()
    objs, st, _ = heightfield()
    sc = build(objs, st)
    n = len(objs)
    base = torch.from_numpy(objs.view(F).reshape(n, 39).copy()).cuda()
    delta = torch.tensor([0.25, -0.5, 0.125], device="cuda")
    moved = objs.copy()
    for f in ("pos", "dim", "rot"):
        moved[f] = (moved[f] + np.array([0.25, -0.5, 0.125], F)).astype(F)
    o, d = moved_rays(st, moved, "translate")
    to, td = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    expect = query(build(moved, st), o, d)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        t = base.clone()
        for c in (0, 9, 13):                                                  # v0, v1, v2
            t[:, c:c + 3] += delta
        sc.refit(t, stream=s)
        ids, tt, uv = sc.trace(to, td)
    s.synchronize()
    got = (ids.cpu().numpy(), tt.cpu().numpy(), uv.cpu().numpy())
    assert np.array_equal(got[0], expect[0]) and np.array_equal(got[1], expect[1]) and np.array_equal(got[2], expect[2])
    # the scene's own stream
    pids = torch.empty(len(o), dtype=torch.int32, device="cuda")
    pt = torch.empty(len(o), device="cuda")
    sc.trace_device(to.data_ptr(), td.data_ptr(), len(o), pids.data_ptr(), pt.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(pids.cpu().numpy(), expect[0]) and np.array_equal(pt.cpu().numpy(), expect[1])
    # host arrays work too, and bring the scene back
    sc.refit(objs)
    assert_same(snapshot(build(objs, st), st, o, d), snapshot(sc, st, o, d))
    # wrong device, size or dtype
    with pytest.raises(ValueError):
        sc.refit(base.cpu())
    with pytest.raises(ValueError):
        sc.refit(base[:-1])
    with pytest.raises(ValueError):
        sc.refit(base[:, :38])
    with pytest.raises(ValueError):
        sc.refit(objs.view(F))
    with pytest.raises(ValueError):
        sc.refit(objs[:-1])
