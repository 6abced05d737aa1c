"""The cooperative tree build (k_ploc_all, k_wide_all) and the refit (k_refit_wide) against their host mirrors at the sizes
where the kernels change shape, and scenes whose primitive boxes are all the same (`pytest -m gpu` on a B200).

The small scenes of test_gpu_parity.py and test_gpu_refit.py leave every block with one 256-wide tile and fewer than 256
blocks.  Here:
  * 2 048 / 2 049 primitives: the clustering starts in (or one cluster above) block 0's solo mode;
  * 65 537 primitives: 257 clustering blocks, so one thread sums two block totals;
  * 100 000 primitives and up: chunks of several tiles, so the running carry between tiles is used;
  * a flat regular grid: many exact area ties;
  * 1 M and 10 M triangles (the benchmark scenes): wide levels above 148 x 256 nodes for the collapse, and above one
    grid stride for the refit's box update.
Bars: keys, order, both binary trees, all float boxes, the four-wide nodes, the level and stack counts, the tree height
and the number of clustering rounds equal the mirrors' bit for bit; a refit equals the numpy mirror of the box update."""
import math

import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth
from oracle import restated
from test_gpu_parity import wide_stack_need
from test_gpu_refit import agree, deform, leaf_boxes, mirror, moved_rays, query, renderable, settings

pytestmark = pytest.mark.gpu

F = np.float32
EMPTY = -2 ** 31
DEBUG = drb.BUILD_KEEP_DEBUG


# ---- the host mirror of the whole build -----------------------------------------------------------------

def stack_need(child):
    """wide_stack_need of test_gpu_parity, one numpy pass per level: (need of the root, number of levels).  Breadth-first
    ids put the internal children of one level, in order, right after it."""
    bounds = [0, 1]
    while True:
        c = child[bounds[-2]:bounds[-1]]
        inner = c[c >= 0]
        if not len(inner):
            break
        assert inner[0] == bounds[-1] and inner[-1] == bounds[-1] + len(inner) - 1
        bounds.append(bounds[-1] + len(inner))
    assert bounds[-1] == len(child)
    need = np.zeros(len(child), np.int64)
    for lv in range(len(bounds) - 2, -1, -1):
        c = child[bounds[lv]:bounds[lv + 1]]
        kids = (c != EMPTY).sum(1)
        deepest = np.where(c >= 0, need[np.maximum(c, 0)], 0).max(1)
        need[bounds[lv]:bounds[lv + 1]] = np.maximum(kids - 1, 0) + deepest
    return int(need[0]), len(bounds) - 1


def host_build(objs):
    lo, hi = leaf_boxes(objs[renderable(objs)])
    h = restated.lbvh_host(lo, hi)
    lmin, lmax = lo[h["order"]], hi[h["order"]]
    p = restated.ploc_host(lmin, lmax)
    w = restated.wide_host(p["left"], p["right"], p["node_min"], p["node_max"], lmin, lmax, h["scene_bounds"])
    need, levels = stack_need(w["child"])
    assert levels == w["levels"]
    return dict(lbvh=h, ploc=p, wide=w, need=need)


def same(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s, mirror %s" % (what, a.shape, b.shape)
    bad = np.flatnonzero(np.any((a != b).reshape(len(a), -1), axis=1)) if a.ndim else ([0] if a != b else [])
    assert not len(bad), "%s differs from the mirror at %d of %d entries, first %d: %r vs %r" % (what, len(bad), len(a), bad[0], a[bad[0]], b[bad[0]])


def assert_build_matches_mirror(sc, m):
    h, p, w = m["lbvh"], m["ploc"], m["wide"]
    dev = sc.lbvh()
    for k in ("keys", "order", "parent", "left", "right", "node_min", "node_max"):
        same(dev[k], h[k], "lbvh " + k)
    bi = sc.build_info
    same(np.array(list(bi.bounds_min) + list(bi.bounds_max), F), h["scene_bounds"], "scene bounds")
    t = sc.tree()
    for k in ("left", "right", "node_min", "node_max"):
        same(t[k], p[k], "tree " + k)
    dw = sc.wide()
    same(dw["child"], w["child"], "wide child")
    same(dw["boxes"], w["boxes"], "wide boxes")
    assert bi.nwide == len(w["child"]), "nwide"
    assert bi.wide_levels == w["levels"], "wide_levels"
    assert bi.stack_levels == m["need"] + 2, "stack_levels"
    assert bi.max_depth == p["height"], "max_depth"
    assert bi.rebuild_iterations == p["rounds"], "rebuild_iterations"


def assert_plain_build_same_nodes(objs, st, sc):
    plain = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    pw, dw = plain.wide(), sc.wide()
    same(pw["child"], dw["child"], "wide child without the debug flag")
    same(pw["boxes"], dw["boxes"], "wide boxes without the debug flag")
    a, b = plain.build_info, sc.build_info
    assert (a.stack_levels, a.max_depth, a.rebuild_iterations) == (b.stack_levels, b.max_depth, b.rebuild_iterations)


def info_bytes(sc):
    bi = sc.build_info
    bi.upload_ms = bi.build_ms = 0.0                                          # wall-clock fields
    return bytes(bi)


# ---- scenes ---------------------------------------------------------------------------------------------

def random_tris(n, seed, spheres=0.0):
    rng = np.random.default_rng(seed)
    o = drb.make_objects(n)
    c = rng.uniform(-20, 20, (n, 3)).astype(F)
    o["pos"] = c
    o["dim"] = c + rng.uniform(-1, 1, (n, 3)).astype(F)
    o["rot"] = c + rng.uniform(-1, 1, (n, 3)).astype(F)
    if spheres:
        sph = rng.uniform(size=n) < spheres
        o["type"][sph] = 0
        o["dim"][sph, 0] = rng.uniform(0.2, 1.0, int(sph.sum())).astype(F)
    return o


def scale_scene(name):
    if name.startswith("random"):
        n = int(name[len("random"):])
        return random_tris(n, seed=n, spheres=0.02), settings()
    if name == "flat_grid":
        return synth.heightfield_scene(n=200, amp=0.0)
    if name == "grid1m":
        return synth.instanced_grid_scene(spp=1, max_depth=4)
    raise KeyError(name)


class Built:
    def __init__(self, objs, st):
        self.objs, self.st = objs, st
        self.hs = drb.HostScene.from_objects(objs, st)
        self.sc = drb.Scene.from_host(self.hs, build_flags=DEBUG)
        self.m = host_build(objs)


@pytest.fixture(scope="module")
def grid1m():
    return Built(*scale_scene("grid1m"))


@pytest.fixture(scope="module")
def city10m():
    return Built(*synth.city_scene())


# ---- a. the build against the mirror --------------------------------------------------------------------

def test_per_level_stack_need_equals_the_node_by_node_sweep():
    m = host_build(random_tris(3000, seed=1, spheres=0.02))
    assert m["need"] == wide_stack_need(m["wide"]["child"])


@pytest.mark.parametrize("name", ["random2048", "random2049", "random65537", "random100000", "flat_grid"])
def test_build_matches_mirror(name):
    b = Built(*scale_scene(name))
    assert_build_matches_mirror(b.sc, b.m)
    assert_plain_build_same_nodes(b.objs, b.st, b.sc)


def test_million_triangle_build_matches_mirror(grid1m):
    assert grid1m.sc.num_prims == 16 * 65536 + 4
    assert_build_matches_mirror(grid1m.sc, grid1m.m)
    assert_plain_build_same_nodes(grid1m.objs, grid1m.st, grid1m.sc)


def test_ten_million_triangle_build_matches_mirror(city10m):
    assert city10m.sc.num_prims > 10_000_000 - 8
    assert_build_matches_mirror(city10m.sc, city10m.m)
    assert_plain_build_same_nodes(city10m.objs, city10m.st, city10m.sc)


# ---- b. determinism -------------------------------------------------------------------------------------

def test_million_triangle_build_is_deterministic(grid1m):
    again = drb.Scene.from_host(grid1m.hs, build_flags=DEBUG)
    a, b = grid1m.sc.wide(), again.wide()
    assert a["child"].tobytes() == b["child"].tobytes() and a["boxes"].tobytes() == b["boxes"].tobytes()
    assert info_bytes(grid1m.sc) == info_bytes(again)


# ---- c. refit -------------------------------------------------------------------------------------------

def assert_identity_refit(b):
    w0, i0 = b.sc.wide(), info_bytes(b.sc)
    b.sc.refit(b.objs)
    w1 = b.sc.wide()
    assert w0["child"].tobytes() == w1["child"].tobytes() and w0["boxes"].tobytes() == w1["boxes"].tobytes()
    assert info_bytes(b.sc) == i0


def test_million_triangle_identity_refit(grid1m):
    assert_identity_refit(grid1m)


def test_ten_million_triangle_identity_refit(city10m):
    assert_identity_refit(city10m)


@pytest.mark.parametrize("kind", ["jitter", "rigid", "translate"])
def test_million_triangle_deformed_refit(grid1m, kind):
    b = grid1m
    moved = deform(b.objs, kind, np.random.default_rng(sum(map(ord, kind))))
    try:
        b.sc.refit(moved)
        w = b.sc.wide()
        same(w["child"], b.m["wide"]["child"], "links after the refit")
        boxes, bmin, bmax = mirror(b.sc, moved)
        same(w["boxes"], boxes, "refitted boxes")
        bi = b.sc.build_info
        same(np.array(bi.bounds_min, F), bmin, "refitted bounds min")
        same(np.array(bi.bounds_max, F), bmax, "refitted bounds max")
        fresh = drb.Scene.from_host(drb.HostScene.from_objects(moved, b.st))
        o, d = moved_rays(b.st, moved, kind, n=4000)
        got = query(b.sc, o, d)
        assert (got[0] >= 0).sum() > 1000
        agree(got, query(fresh, o, d))
        bid, bt = restated.brute_tris(moved["pos"], moved["dim"], moved["rot"], o[:256], d[:256])
        ids, t = got[0][:256], got[1][:256]
        assert (bid >= 0).sum() > 64
        assert ((ids == bid) | ((ids >= 0) & (bid >= 0) & (t == bt))).all()
        assert np.array_equal(t[bid >= 0], bt[bid >= 0])
    finally:
        b.sc.refit(b.objs)                                                    # the next test starts from the built scene


# ---- d. identical primitive boxes -----------------------------------------------------------------------

def coincident(n, kind):
    o = drb.make_objects(n)
    if kind == "triangles":
        o["pos"], o["dim"], o["rot"] = (0, 0, 0), (1, 0, 0), (0, 1, 0)
    elif kind == "points":                                                    # zero-size triangles at one point
        o["pos"] = o["dim"] = o["rot"] = (0.25, 0.5, 0)
    elif kind == "spheres":
        o["type"] = 0
        o["pos"] = (0.5, 0.5, 0)
        o["dim"][:, 0] = 0.5
    return o


def identical_scene(name):
    """(objects, ids of the coincident lines)"""
    kind, n = name.split("_")
    n = int(n)
    if kind == "mixed":
        o = np.concatenate([coincident(n, "triangles"), random_tris(n, seed=3)])
        return o, np.arange(n)
    return coincident(n, kind), np.arange(n)


def identical_rays(n=4096, seed=6):
    """rays from both sides of z = 0 through the unit square the coincident primitives cover, and a little beyond it"""
    rng = np.random.default_rng(seed)
    tgt = np.concatenate([rng.uniform(-0.2, 1.2, (n, 2)), np.zeros((n, 1))], 1)
    o = np.concatenate([rng.uniform(-2, 3, (n, 2)), rng.choice([-4.0, 4.0], (n, 1))], 1)
    return o.astype(F), (tgt - o).astype(F)


@pytest.mark.parametrize("name", ["triangles_64", "triangles_400", "triangles_600", "triangles_2000", "triangles_100000",
                                  "points_2000", "spheres_2000", "mixed_2000"])
def test_identical_boxes_build_a_balanced_tree(name):
    objs, tie_ids = identical_scene(name)
    n = len(objs)
    st = settings(w=32, h=24, spp=2, depth=3)
    st.cam[:] = [0.5, 0.5, 6.0]
    st.look[:] = [0.5, 0.5, 0.0]
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st), build_flags=DEBUG)
    m = host_build(objs)
    assert_build_matches_mirror(sc, m)
    bi = sc.build_info
    log2n = math.ceil(math.log2(n))
    # a run of identical boxes halves every round; mixed into random triangles, its subtree hangs below a path of theirs
    # (stack 29 alone, 26 for the random half, 47 together; a chain gave 2 016)
    assert bi.stack_levels <= (4 if name.startswith("mixed") else 3) * log2n + 8, (bi.stack_levels, n)
    assert bi.rebuild_iterations <= 4 * math.log2(n), (bi.rebuild_iterations, n)
    o, d = identical_rays()
    ids, t, _, occ = query(sc, o, d)
    if name.startswith("spheres"):
        # every sphere is the same sphere: the hit of any one of them, by a scene holding only it
        ref_ids, ref_t, _, _ = query(drb.Scene.from_host(drb.HostScene.from_objects(objs[:1], st)), o, d)
        bid, bt = np.where(ref_ids >= 0, 0, -1), ref_t
    else:
        bid, bt = restated.brute_tris(objs["pos"], objs["dim"], objs["rot"], o, d)
    hit = bid >= 0
    if name.startswith("points"):
        assert not hit.any()                                                  # a zero-size triangle has det 0: never hit
    else:
        assert hit.sum() > 500
    assert np.array_equal(ids >= 0, hit)
    assert np.array_equal(t[hit].view(np.uint32), bt[hit].view(np.uint32))
    tie = np.isin(ids, tie_ids) & np.isin(bid, tie_ids)                       # same box, same vertices: the same t
    assert ((ids == bid) | tie).all()
    assert np.array_equal(occ, hit)                                           # tmax 1e4, and the hit test takes t < 1e4 only
    img, stats = sc.render(st, seed=2)
    assert np.isfinite(img).all() and stats.paths == 32 * 24 * 2
