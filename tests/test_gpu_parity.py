"""Parity of the CUDA path against the oracle, all through the C ABI (`pytest -m gpu` on a B200).

Oracle = oracle/_ref (the reference's own kernel.cu compiled for the host) where present, else the C
restatement that is pinned to it (tests/test_oracle_pin.py).  Bars:
  closest-hit object ids   bit-exact (a mismatch is tolerated only as an exact-t tie, and counted)
  hit distances            bit-exact
  radiance                 the stated tolerance is <= 1e-3 RMSE (BASELINE.json north_star); the tests
                           additionally require >= 99.9 % of pixels to be bit-identical, because both
                           sides consume the same Philox stream
"""
import os

import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth
from oracle import restated
from conftest import HAVE_REF, ROOT, SAMPLES, needs_ref, sample

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RMSE_TOL = 1e-3            # in [0,1] radiance units
SCENES = [("cube.rts", dict(cam=(6.0, -5.0, 9.0))), ("cube.rts", {}), ("mats.rts", {}), ("glass.rts", dict(max_depth=8)),
          ("bolter2.blend.rts", {}), ("rough.blend.rts", {}), ("gloss.rts", {}), ("uv2.rts", {}), ("lots.rts", {}), ("cow.rts", {}),
          ("textest.rts", {}), ("smoothdiff.rts", {}), ("glasstest.rts", dict(max_depth=8)), ("corvette.blend.rts", {}),
          ("eorovan.blend.rts", {}), ("SPERSSSSS.rts", {}), ("HIGH.rts", {}), ("light.rts", {})]


class Oracle:
    """the reference build if present, else the restatement"""

    def __init__(self, path, texdir, ref):
        self.ref = ref if HAVE_REF else None
        if self.ref is not None:
            self.ref.load(path, texdir)
        else:
            self.r = restated.Restated(path, texdir)

    def apply(self, st, seed):
        if self.ref is not None:
            self.ref.apply(st); self.ref.set_seed(seed)
        else:
            self.r.apply(st); self.r.set_seed(seed)

    def hit(self, o, d):
        return self.ref.hit(o, d) if self.ref is not None else self.r.hit(o, d)

    def frame(self, div=1, base=0):
        return self.ref.frame(div, base) if self.ref is not None else self.r.frame(div, base)

    def singlehit(self, o, d, k):
        return self.ref.singlehit(o, d, k) if self.ref is not None else None


@pytest.fixture(scope="module")
def maybe_ref():
    if HAVE_REF:
        from oracle import refhost
        return refhost.RefHost()
    return None


def assert_ids_match(ids, t, oid, ot, orc=None, o=None, d=None):
    ids, oid = ids.reshape(-1), oid.reshape(-1)
    bad = np.flatnonzero(ids != oid)
    for k in bad:            # only an exact tie in t may pick a different object (SURVEY.md hard part 1)
        assert ids[k] >= 0 and oid[k] >= 0 and t.reshape(-1)[k] == ot.reshape(-1)[k], \
            "ray %d: ours (%d, %r) oracle (%d, %r)" % (k, ids[k], t.reshape(-1)[k], oid[k], ot.reshape(-1)[k])
    same = ids == oid
    hit = same & (oid >= 0)
    assert np.array_equal(t.reshape(-1)[hit], ot.reshape(-1)[hit])
    return len(bad)


def assert_frames_match(ours_255, theirs_255):
    diff = (ours_255.astype(np.float64) - theirs_255.astype(np.float64)) / 255.0
    rmse = float(np.sqrt(np.mean(diff ** 2)))
    identical = float(np.mean(np.all(ours_255 == theirs_255, axis=-1)))
    assert rmse <= RMSE_TOL, "RMSE %g" % rmse
    assert identical >= 0.999, "only %.4f of pixels bit-identical (rmse %g)" % (identical, rmse)
    return rmse, identical


@needs_ref
@pytest.mark.parametrize("name,over", SCENES)
def test_sample_scene_ids_and_radiance(maybe_ref, name, over):
    sc = drb.Scene.load(sample(name), SAMPLES)
    st = sc.settings.replace(width=96, height=64, spp=3, max_depth=over.get("max_depth", 5))
    if "cam" in over:
        st = st.replace(cam=over["cam"])
    orc = Oracle(sample(name), SAMPLES, maybe_ref)
    orc.apply(st, 21)
    o, d = sc.primary_rays(st, sample=0, seed=21)
    ids, t = sc.trace_ids(o, d)
    oid, ot = orc.hit(o, d)
    assert_ids_match(ids, t, oid, ot)
    f, fi, rays = orc.frame()
    acc, stats = sc.render(st, seed=21)
    assert stats.rays == rays and stats.paths == 96 * 64 * 3
    ours = acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / 3)
    assert_frames_match(ours, f)
    ints = sc.frame_i3(st, 1, seed=21)
    assert np.mean(ints == fi) >= 0.999


def test_golden_synthetic_scene(tmp_path):
    """no reference needed at run time: scene regenerated, expected values came from the reference"""
    g = np.load(os.path.join(GOLDEN, "synth_heightfield.npz"))
    objs, st = synth.heightfield_scene(n=24, width=48, height=40, spp=3, max_depth=5)
    p = str(tmp_path / "hf.rts")
    drb.write_rts(p, st, objs)                       # the golden was made from this text (6-decimal %f), not from the float arrays
    sc = drb.Scene.load(p)
    o, d = sc.primary_rays(st, sample=0, seed=int(g["seed"]))
    assert np.array_equal(o, g["origins"]) and np.array_equal(d, g["dirs"])          # camera rays bit-exact
    ids, t = sc.trace_ids(o, d)
    assert np.array_equal(ids, g["ids"]) and np.array_equal(t, g["t"])
    acc, stats = sc.render(st, seed=int(g["seed"]))
    assert stats.rays == int(g["rays"])
    ours = acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / 3)
    assert np.array_equal(ours, g["frame"])
    assert np.array_equal(sc.frame_i3(st, 1, seed=int(g["seed"])), g["frame_i"])


def test_golden_materials_scene(tmp_path):
    """BASELINE config 4 in small against numbers that came from the reference: no oracle needed at run time"""
    g = np.load(os.path.join(GOLDEN, "synth_materials.npz"))
    tex = synth.write_test_textures(str(tmp_path))
    objs, st, tp = synth.materials_scene(tex, width=96, height=56, spp=3, max_depth=6, nu=24, nv=12)
    p = str(tmp_path / "mats.rts")
    drb.write_rts(p, st, objs, tex_names=[os.path.basename(t) for t in tp], backtex_name=os.path.basename(tp[0]))
    sc = drb.Scene.load(p, str(tmp_path))
    st = sc.settings
    seed = int(g["seed"])
    o, d = sc.primary_rays(st, sample=0, seed=seed)
    assert np.array_equal(o, g["origins"]) and np.array_equal(d, g["dirs"])
    ids, t = sc.trace_ids(o, d)
    assert np.array_equal(ids, g["ids"]) and np.array_equal(t, g["t"])
    acc, stats = sc.render(st, seed=seed)
    assert stats.rays == int(g["rays"])
    assert np.array_equal(acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / 3), g["frame"])
    assert np.array_equal(sc.frame_i3(st, 1, seed=seed), g["frame_i"])


@needs_ref
def test_golden_cube():
    g = np.load(os.path.join(GOLDEN, "cube_frame.npz"))
    sc = drb.Scene.load(sample("cube.rts"))
    st = sc.settings.replace(cam=(6.0, -5.0, 9.0), width=40, height=32, spp=3, max_depth=4)
    ids, t = sc.trace_ids(g["origins"], g["dirs"])
    assert np.array_equal(ids, g["ids"]) and np.array_equal(t, g["t"])
    acc, _ = sc.render(st, seed=int(g["seed"]))
    assert np.array_equal(acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / 3), g["frame"])


def test_incoherent_rays_against_brute_force(tmp_path):
    """random rays through a 7 200-triangle scene: ids equal the BVH-independent brute-force definition"""
    objs, st = synth.heightfield_scene(n=60)
    p = str(tmp_path / "hf.rts")
    drb.write_rts(p, st, objs)
    sc = drb.Scene.load(p)
    r = restated.Restated(p)
    rng = np.random.default_rng(5)
    n = 20000
    o = rng.uniform(-6, 6, (n, 3)).astype(np.float32); o[:, 1] = -np.abs(o[:, 1]) - 0.5
    d = rng.normal(size=(n, 3)).astype(np.float32); d[:, 1] = np.abs(d[:, 1])
    d[::7, 0] = 0.0; d[::11, 2] = 0.0                                        # axis-parallel components
    ids, t = sc.trace_ids(o, d)
    bid, bt = r.hit_brute(o, d)
    ties = assert_ids_match(ids, t, bid, bt)
    assert ties <= 5 and (ids >= 0).sum() > n // 10


def test_frame_i3_divisor_and_partial_blocks(maybe_ref, tmp_path):
    objs, st = synth.heightfield_scene(n=12, width=72, height=50, spp=2, max_depth=4)     # 50 % 8 != 0
    p = str(tmp_path / "s.rts")
    drb.write_rts(p, st, objs)
    sc = drb.Scene.load(p)
    orc = Oracle(p, "", maybe_ref)
    for div in (1, 2, 4):
        orc.apply(st, 2)
        f, fi, _ = orc.frame(div, 0)
        out = np.full((72, 50, 3), -7, np.int32)
        sc.frame_i3(st, div, seed=2, out=out)
        gw, gh = 72 // div // 8 * 8, 50 // div // 8 * 8
        assert np.array_equal(out[:gw, :gh], fi[:gw, :gh])
        mask = np.ones((72, 50), bool); mask[:gw, :gh] = False
        assert (out[mask] == -7).all()                                       # untouched outside the launched grid


def test_render_properties_batches_shards_accumulate():
    objs, st = synth.heightfield_scene(n=20, width=64, height=40, spp=8, max_depth=5)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    full, s_full = sc.render(st, seed=4)
    again, _ = sc.render(st, seed=4)
    assert np.array_equal(full, again)                                       # deterministic
    small, s_small = sc.render(st, seed=4, batch_paths=64 * 40 * 2)          # 4 wavefront batches instead of 1
    assert s_small.rays == s_full.rays and np.array_equal(small, full)       # one running sum per pixel: batching does not show
    a, sa = sc.render(st, seed=4, sample_base=0, sample_count=3)             # two sample shards ...
    b, sb = sc.render(st, seed=4, sample_base=3, sample_count=5)
    assert sa.rays + sb.rays == s_full.rays and np.allclose(a + b, full, rtol=0, atol=2e-5)
    acc = a.copy()
    acc, _ = sc.render(st, seed=4, sample_base=3, sample_count=5, accumulate_into=acc)   # ... or accumulated in place
    assert np.array_equal(acc, full)                                         # ... which continues the same running sum
    other, _ = sc.render(st, seed=5)
    assert not np.array_equal(other, full)


def test_edge_scenes_empty_single_and_spheres():
    st = drb.default_settings().replace(width=32, height=24, spp=2, max_depth=3)
    empty = drb.Scene.from_host(drb.HostScene.from_objects(drb.make_objects(0), st))
    acc, stats = empty.render(st, seed=1)
    assert stats.rays == 32 * 24 * 2 and (acc > 0).all()                     # every path sees the sky once
    one = drb.make_objects(1)
    one["pos"], one["dim"], one["rot"] = (-1, -1, 0), (1, -1, 0), (0, 1, 0)
    one["col"] = 0.5; one["mat"] = 1
    sc = drb.Scene.from_host(drb.HostScene.from_objects(one, st))
    ids, t = sc.trace_ids(np.array([[0, 0, 2], [5, 5, 2]], np.float32), np.array([[0, 0, -1], [0, 0, -1]], np.float32))
    assert ids.tolist() == [0, -1] and t[0] == 2.0
    junk = drb.make_objects(3); junk["type"] = [1, 2, 3]                     # unsupported types stay out of the tree, ids keep line numbers
    junk["pos"][1], junk["dim"][1], junk["rot"][1] = (-1, -1, 0), (1, -1, 0), (0, 1, 0)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(junk, st))
    assert sc.num_prims == 1 and sc.num_objects == 3
    ids, _ = sc.trace_ids(np.array([[0, 0, 2]], np.float32), np.array([[0, 0, -1]], np.float32))
    assert ids.tolist() == [1]


def wide_stack_need(child):
    """Exact bound of traversal pushes over a four-wide tree (the host side of k_wide_all's last pass): a visit pushes all
    but one of a node's children, so need(node) = (children - 1) + max over internal children of need(child).  Children
    have larger ids than their parent (breadth-first ids), so one backwards sweep does it."""
    EMPTY = -2 ** 31
    need = np.zeros(len(child), np.int64)
    for i in range(len(child) - 1, -1, -1):
        kids = [c for c in child[i] if c != EMPTY]
        need[i] = max(len(kids) - 1, 0) + max([need[c] for c in kids if c >= 0], default=0)
    return int(need[0])


def test_gpu_lbvh_bit_exact_against_host_build():
    rng = np.random.default_rng(8)
    cases = []
    objs, _ = synth.heightfield_scene(n=40)
    cases.append(objs)
    dup = drb.make_objects(64)                                               # 64 coincident triangles: every key ties
    dup["pos"], dup["dim"], dup["rot"] = (0, 0, 0), (1, 0, 0), (0, 1, 0)
    cases.append(dup)
    for n in (2, 3, 1000):
        o = drb.make_objects(n)
        c = rng.uniform(-20, 20, (n, 3)).astype(np.float32)
        o["pos"] = c; o["dim"] = c + rng.uniform(-1, 1, (n, 3)).astype(np.float32); o["rot"] = c + rng.uniform(-1, 1, (n, 3)).astype(np.float32)
        if n == 1000:
            o["type"][::50] = 0; o["dim"][::50, 0] = 0.7                     # a few spheres
        cases.append(o)
    if HAVE_REF:
        cases.append(drb.HostScene.load(sample("SPERSSSSS.rts")).objects())
    for objs in cases:
        sc = drb.Scene.from_host(drb.HostScene.from_objects(objs), build_flags=drb.BUILD_KEEP_DEBUG)
        tri = objs["type"] == 2
        v = np.stack([objs["pos"], objs["dim"], objs["rot"]], 1)
        bmin = np.where(tri[:, None], v.min(1), objs["pos"] - np.abs(objs["dim"][:, :1]))
        bmax = np.where(tri[:, None], v.max(1), objs["pos"] + np.abs(objs["dim"][:, :1]))
        host = restated.lbvh_host(bmin, bmax)
        dev = sc.lbvh()
        for k in ("keys", "order", "parent", "left", "right"):
            assert np.array_equal(dev[k], host[k]), k
        assert np.array_equal(dev["node_min"], host["node_min"]) and np.array_equal(dev["node_max"], host["node_max"])
        bi = sc.build_info
        assert np.array_equal(np.array(list(bi.bounds_min) + list(bi.bounds_max), np.float32), host["scene_bounds"])
        # the SAH-guided rebuild over the same sorted leaves, against its host mirror
        if len(objs) > 1:
            lmin, lmax = bmin[host["order"]], bmax[host["order"]]
            ph = restated.ploc_host(lmin, lmax)
            dt = sc.tree()
            assert np.array_equal(dt["left"], ph["left"]) and np.array_equal(dt["right"], ph["right"])
            assert np.array_equal(dt["node_min"], ph["node_min"]) and np.array_equal(dt["node_max"], ph["node_max"])
            assert bi.max_depth == ph["height"] and bi.rebuild_iterations > 0
            # ... and the four-wide collapse of that tree (ids, links, 16-bit boxes)
            wh = restated.wide_host(ph["left"], ph["right"], ph["node_min"], ph["node_max"], lmin, lmax, host["scene_bounds"])
            dw = sc.wide()
            assert bi.nwide == len(wh["child"]) and bi.wide_levels == wh["levels"]
            assert np.array_equal(dw["child"], wh["child"]) and np.array_equal(dw["boxes"], wh["boxes"])
            assert bi.stack_levels == wide_stack_need(wh["child"]) + 2 <= 3 * wh["levels"] + 2
            # the default build keeps none of the debug arrays, and emits the same traversal nodes
            plain = drb.Scene.from_host(drb.HostScene.from_objects(objs))
            pw = plain.wide()
            assert np.array_equal(pw["child"], wh["child"]) and np.array_equal(pw["boxes"], wh["boxes"])
            assert plain.build_info.stack_levels == bi.stack_levels and plain.build_info.max_depth == bi.max_depth
            with pytest.raises(drb.DogerayError):
                plain.lbvh()
            with pytest.raises(drb.DogerayError):
                plain.tree()
            lb = drb.Scene.from_host(drb.HostScene.from_objects(objs), build_flags=drb.BUILD_LBVH_ONLY | drb.BUILD_KEEP_DEBUG)
            assert lb.build_info.max_depth == host["height"] and lb.build_info.rebuild_iterations == 0
            lt = lb.tree()
            assert np.array_equal(lt["left"], host["left"]) and np.array_equal(lt["right"], host["right"])


def test_scene_from_object_lines_already_on_the_device():
    """drb_scene_create_from_device: the build reads an array some other stream produced (e.g. an all-gather of per-rank
    partial uploads) and gives the scene the host upload gives"""
    import torch
    objs, st = synth.heightfield_scene(n=48, width=64, height=40, spp=2, max_depth=4)
    objs = np.concatenate([objs, drb.make_objects(3)])                     # degenerate + a legacy type that stays out of the tree
    objs["type"][-1] = 1
    hs = drb.HostScene.from_objects(objs, st)
    assert hs.num_renderable == len(objs) - 1
    a = drb.Scene.from_host(hs)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        halves = [torch.from_numpy(objs[:1000].view(np.uint8)).cuda(non_blocking=True), torch.from_numpy(objs[1000:].view(np.uint8)).cuda(non_blocking=True)]
        dev = torch.cat(halves)                                            # stands in for the all-gather
        b = drb.Scene.from_device_objects(hs, dev.data_ptr(), stream=side.cuda_stream)
    wa, wb = a.wide(), b.wide()
    assert np.array_equal(wa["child"], wb["child"]) and np.array_equal(wa["boxes"], wb["boxes"])
    fa, sa = a.render(st, seed=2); fb, sb = b.render(st, seed=2)
    assert np.array_equal(fa, fb) and sa.rays == sb.rays
    # a host scene whose count disagrees with the device array is refused, not overrun
    wrong = objs.copy(); wrong["type"][:10] = 1
    with pytest.raises(drb.DogerayError):
        drb.Scene.from_device_objects(drb.HostScene.from_objects(wrong, st), dev.data_ptr(), stream=side.cuda_stream)


def test_zero_samples_means_zero_samples():
    """an integer sample_count is literal (DRB_FLAG_EXACT_SAMPLES): the empty share of a sharded frame traces nothing"""
    objs, st = synth.heightfield_scene(n=12, width=40, height=24, spp=3, max_depth=4)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    full, sf = sc.render(st, seed=9)                                        # sample_count=None -> settings.spp
    assert sf.paths == 40 * 24 * 3
    none, sn = sc.render(st, seed=9, sample_count=0)
    assert sn.paths == 0 and sn.rays == 0 and not none.any()
    kept, _ = sc.render(st, seed=9, sample_count=0, accumulate_into=full.copy())
    assert np.array_equal(kept, full)
    # no bounce at all: raycolor's loop never runs and returns black (kernel.cu:793, 981); twice, so stale buffers would show
    for _ in range(2):
        black, sb = sc.render(st.replace(max_depth=0), seed=9)
        assert sb.rays == 0 and not black.any()
    one, s1 = sc.render(st.replace(max_depth=1), seed=9)                     # only misses shine at depth 1
    assert s1.rays == 40 * 24 * 3 and one.max() > 0
    # spp < ranks: the shares of 8 ranks, summed, are the 3-sample frame
    from dogeray_b200.distributed import shard_samples
    acc = np.zeros_like(full)
    for r in range(8):
        base, count = shard_samples(st.spp, r, 8)
        part, _ = sc.render(st, seed=9, sample_base=base, sample_count=count)
        acc += part
    assert np.allclose(acc, full, rtol=0, atol=1e-5)


def test_small_scene_far_from_the_origin():
    """ray padding larger than the scene (origin ~10^5 scene sizes away): an empty child slot's inverted box then passes
    the slab test; its link has the stack sentinel's bits and must be dropped, not end the traversal"""
    rng = np.random.default_rng(5)
    n = 7                                                                    # 7 leaves: the four-wide tree has empty slots
    o = drb.make_objects(n)
    c = (np.array([4000.0, -3000.0, 5000.0]) + rng.uniform(-0.004, 0.004, (n, 3))).astype(np.float32)
    o["pos"] = c; o["dim"] = c + rng.uniform(-0.004, 0.004, (n, 3)).astype(np.float32); o["rot"] = c + rng.uniform(-0.004, 0.004, (n, 3)).astype(np.float32)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(o))
    assert (sc.wide()["child"] == -2 ** 31).any()
    m = 4096
    ro = (np.array([4000.0, -3000.0, 5000.0]) + rng.normal(size=(m, 3)) * 3).astype(np.float32)
    tgt = c[rng.integers(0, n, m)] + rng.uniform(-0.003, 0.003, (m, 3))
    rd = ((tgt - ro) * 40).astype(np.float32)                                # long directions: |det| clears hit_tri's epsilon
    ids, t = sc.trace_ids(ro, rd)
    bid, bt = restated.brute_tris(o["pos"], o["dim"], o["rot"], ro, rd)
    assert (bid >= 0).sum() > 50
    assert_ids_match(ids, t, bid, bt)


def test_tonemap_device_matches_host():
    import torch
    rng = np.random.default_rng(3)
    acc = (rng.uniform(-0.2, 1.4, (20, 30, 3)) * 6).astype(np.float32)
    t = torch.from_numpy(acc).cuda()
    out = torch.empty(20, 30, 3, dtype=torch.uint8, device="cuda")
    drb.tonemap_device(t.data_ptr(), 30, 20, 6, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), drb.tonemap(acc, 6))


def test_render_device_into_torch_tensor_matches_host_api():
    import torch
    objs, st = synth.heightfield_scene(n=16, width=40, height=24, spp=4, max_depth=4)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    host, _ = sc.render(st, seed=6)
    t = torch.zeros(24, 40, 3, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    sc.render_device(t.data_ptr(), st, seed=6, stream=stream)
    torch.cuda.synchronize()
    assert np.array_equal(t.cpu().numpy(), host)


def test_tree_variant_and_traversal_knobs_do_not_change_results(tmp_path):
    """the Karras-only tree and the traversal's refill / leaf-batch / step thresholds are scheduling choices: same ids,
    same image"""
    import subprocess, sys, hashlib
    objs, st = synth.heightfield_scene(n=40, width=80, height=48, spp=4, max_depth=5)
    hs = drb.HostScene.from_objects(objs, st)
    a = drb.Scene.from_host(hs)
    b = drb.Scene.from_host(hs, build_flags=drb.BUILD_LBVH_ONLY)
    o, d = a.primary_rays(st, 0, seed=3)
    ia, ta = a.trace_ids(o, d); ib, tb = b.trace_ids(o, d)
    assert np.array_equal(ia, ib) and np.array_equal(ta, tb)
    fa, sa = a.render(st, seed=3); fb, sb = b.render(st, seed=3)
    assert np.array_equal(fa, fb) and sa.rays == sb.rays
    p = str(tmp_path / "s.rts"); drb.write_rts(p, st, objs)
    code = ("import sys,hashlib; sys.path.insert(0, %r); import dogeray_b200 as drb; sc = drb.Scene.load(%r); "
            "st = sc.settings.replace(width=80, height=48, spp=4, max_depth=5); acc, s = sc.render(st, seed=3); "
            "print(hashlib.sha256(acc.tobytes()).hexdigest(), s.rays)") % (ROOT, p)
    outs = []
    for env in ({}, {"DOGERAY_B200_REFILL": "32", "DOGERAY_B200_LEAF_BATCH": "1", "DOGERAY_B200_STEP_MIN": "1"}):
        r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs.append(r.stdout.strip())
    assert outs[0] == outs[1]


def test_all_material_classes_textures_and_env_map(tmp_path, maybe_ref):
    """BASELINE config 4 in small: diffuse / mirror / metal / glass / glossy / emissive, colour + roughness textures,
    checker, smooth normals, environment map -- against the oracle, bit for bit"""
    tex = synth.write_test_textures(str(tmp_path))
    objs, st, tp = synth.materials_scene(tex, width=96, height=56, spp=3, max_depth=6, nu=24, nv=12)
    p = str(tmp_path / "mats.rts")
    drb.write_rts(p, st, objs, tex_names=[os.path.basename(t) for t in tp], backtex_name=os.path.basename(tp[0]))
    sc = drb.Scene.load(p, str(tmp_path))
    assert sc.settings.backtex == 0 and set(np.unique(drb.HostScene.load(p, str(tmp_path)).objects()["mat"])) == {0, 1, 2, 3, 4, 5}
    orc = Oracle(p, str(tmp_path), maybe_ref)
    stt = sc.settings
    orc.apply(stt, 13)
    o, d = sc.primary_rays(stt, sample=0, seed=13)
    ids, t = sc.trace_ids(o, d)
    oid, ot = orc.hit(o, d)
    assert_ids_match(ids, t, oid, ot)
    f, fi, rays = orc.frame()
    acc, stats = sc.render(stt, seed=13)
    assert stats.rays == rays
    assert_frames_match(acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / 3), f)


def test_trim_releases_cached_memory_and_rendering_still_works():
    import torch
    objs, st = synth.heightfield_scene(n=16, width=64, height=40, spp=2, max_depth=3)
    hs = drb.HostScene.from_objects(objs, st)
    sc = drb.Scene.from_host(hs); a, _ = sc.render(st, seed=1); sc.close()
    free0, _ = torch.cuda.mem_get_info()
    drb.trim(0)
    free1, _ = torch.cuda.mem_get_info()
    assert free1 >= free0
    sc = drb.Scene.from_host(hs); b, _ = sc.render(st, seed=1); sc.close()
    assert np.array_equal(a, b)


def test_converged_radiance_4096spp_rmse_and_psnr(tmp_path, maybe_ref):
    """north_star's radiance bar, literally: <= 1e-3 per-pixel RMSE / >= 45 dB PSNR against a 4096-spp reference image
    of the same scene and seed (the reference image comes from the oracle; both sides use the same Philox stream)"""
    objs, st = synth.heightfield_scene(n=16, width=32, height=24, spp=4096, max_depth=6)
    p = str(tmp_path / "conv.rts")
    drb.write_rts(p, st, objs)
    sc = drb.Scene.load(p)
    orc = Oracle(p, "", maybe_ref)
    orc.apply(st, 77)
    f, _, rays = orc.frame()
    ref_img = f.transpose(1, 0, 2) / 255.0                                  # mean radiance, (H, W, 3)
    acc, stats = sc.render(st, seed=77)
    img = acc / np.float32(4096)
    rmse = float(np.sqrt(np.mean((img - ref_img) ** 2)))
    peak = float(max(ref_img.max(), 1.0))
    psnr = float("inf") if rmse == 0 else 20 * np.log10(peak / rmse)
    assert stats.rays == rays
    assert rmse <= 1e-3 and psnr >= 45.0, (rmse, psnr)
    # and a 256-spp image with another seed is an unbiased estimate of the same picture (noise ~ 1/sqrt(256))
    other, _ = sc.render(st.replace(spp=256), seed=78)
    noisy = float(np.sqrt(np.mean((other / np.float32(256) - ref_img) ** 2)))
    assert noisy < 0.08, noisy
    assert abs(float((other / np.float32(256)).mean()) - float(ref_img.mean())) < 0.01


def test_non_finite_coordinates_do_not_hang(tmp_path):
    """NaN / inf vertices (a text file can say `nan`) must end in an image or an error code, never in a hang"""
    import subprocess, sys
    code = """
import sys, numpy as np
sys.path.insert(0, %r)
import dogeray_b200 as drb
from dogeray_b200 import synth
objs, st = synth.heightfield_scene(n=12, width=48, height=32, spp=2, max_depth=4)
objs["pos"][5] = np.nan; objs["dim"][17, 1] = np.inf; objs["rot"][40] = -np.inf; objs["pos"][99, 0] = 3e38
try:
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    acc, stats = sc.render(st, seed=1)
    ids, t = sc.trace_ids(np.array([[0, -5, 7]], np.float32), np.array([[0, 5, -7]], np.float32))
    print("RENDERED", stats.rays, float(np.nanmean(acc)))
except drb.DogerayError as e:
    print("ERROR", e.status)
""" % ROOT
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr[-1500:]
    assert "RENDERED" in p.stdout or "ERROR" in p.stdout


def test_render_error_paths_return_codes():
    import ctypes as C
    objs, st = synth.heightfield_scene(n=4, width=16, height=8, spp=1, max_depth=2)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    dummy = np.zeros(16 * 8 * 3, np.float32)
    for bad in (st.replace(width=0), st.replace(height=-3), st.replace(width=40000), st.replace(max_depth=-1)):
        assert drb._lib.drb_render(sc.handle, C.byref(bad), None, dummy.ctypes.data, None) == drb.ERR_ARG
        assert drb.last_error() != ""
    with pytest.raises(drb.DogerayError) as e:
        sc.render(st.replace(backtex=3))                      # the scene has no textures
    assert e.value.status == drb.ERR_ARG and "backtex" in str(e.value)
    assert drb._lib.drb_render(sc.handle, C.byref(st), None, None, None) == drb.ERR_ARG
    assert drb._lib.drb_render(None, C.byref(st), None, None, None) == drb.ERR_ARG
    assert drb._lib.drb_trace_ids(sc.handle, None, None, 5, None, None) == drb.ERR_ARG
    assert drb._lib.drb_frame_i3(sc.handle, C.byref(st), None, 0, None) == drb.ERR_ARG
    with pytest.raises(drb.DogerayError):
        drb.Scene.from_host(drb.HostScene.from_objects(objs, st), device=99)
    # spp = 0: a black accumulator, no rays
    acc, stats = sc.render(st.replace(spp=0))
    assert stats.rays == 0 and not acc.any()
    # depth 0: every path ends black immediately (kernel.cu:793 loop does not run)
    acc, stats = sc.render(st.replace(max_depth=0))
    assert stats.rays == 0 and not acc.any()


def test_tile_sharding_is_bit_identical_to_the_whole_image():
    """interleaved 8x4-pixel tiles over 3 "ranks": the partial images are disjoint and their sum IS the 1-GPU image"""
    objs, st = synth.heightfield_scene(n=20, width=70, height=45, spp=5, max_depth=5)      # not a multiple of the tile size
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    full, sf = sc.render(st, seed=8)
    parts, rays, paths = [], 0, 0
    for r in range(3):
        p, s = sc.render(st, seed=8, tile_rank=r, tile_count=3)
        parts.append(p); rays += s.rays; paths += s.paths
    assert rays == sf.rays and paths == sf.paths
    nz = [(p != 0).any(axis=2) for p in parts]
    assert not (nz[0] & nz[1]).any() and not (nz[0] & nz[2]).any() and not (nz[1] & nz[2]).any()      # disjoint pixels
    assert np.array_equal(parts[0] + parts[1] + parts[2], full)                                        # bit-identical
    from dogeray_b200.distributed import tile_owner_mask
    for r in range(3):                                                                                  # the host-side ownership formula is the kernel's
        m = tile_owner_mask(st.width, st.height, r, 3)
        assert not nz[r][~m].any() and np.array_equal(parts[r][m], full[m])
    with pytest.raises(drb.DogerayError):
        sc.render(st, tile_rank=3, tile_count=3)


def test_render_multi_over_several_handles_is_bit_identical_to_one_handle():
    """drb_render_multi: one host thread per handle, interleaved tiles resolved straight into one device image.  Two and
    three handles on device 0 stand in for two and three GPUs (same code path; test_render_multi_on_two_devices runs it
    across real peers)."""
    objs, st = synth.heightfield_scene(n=24, width=83, height=47, spp=6, max_depth=5)      # ragged right and bottom tiles
    hs = drb.HostScene.from_objects(objs, st)
    scenes = [drb.Scene.from_host(hs) for _ in range(3)]
    full, sf = scenes[0].render(st, seed=21)
    for n in (1, 2, 3):
        img, sm = drb.render_multi(scenes[:n], st, seed=21)
        assert np.array_equal(img, full), n
        assert sm.rays == sf.rays and sm.paths == sf.paths == 83 * 47 * 6
        assert sm.kernel_launches >= sf.kernel_launches
    # accumulate: two half-frames over two handles == the two half-frames on one handle
    a, _ = scenes[0].render(st, seed=21, sample_base=0, sample_count=3)
    a, _ = scenes[0].render(st, seed=21, sample_base=3, sample_count=3, accumulate_into=a)
    b, _ = drb.render_multi(scenes[:2], st, seed=21, sample_base=0, sample_count=3)
    b, _ = drb.render_multi(scenes[:2], st, seed=21, sample_base=3, sample_count=3, accumulate_into=b)
    assert np.array_equal(a, b)
    # small batches inside every shard
    c, _ = drb.render_multi(scenes, st, seed=21, batch_paths=4096)
    assert np.array_equal(c, full)
    # tile shards claimed from the shared queue: whoever renders a shard, the bits are the same
    for n in (2, 3):
        d, sd = drb.render_multi(scenes[:n], st, seed=21, dynamic=True)
        assert np.array_equal(d, full) and sd.rays == sf.rays and sd.paths == sf.paths
        assert len(drb.render_multi_times()) == n
    d, _ = drb.render_multi(scenes[:2], st, seed=21, sample_base=0, sample_count=3, dynamic=True)
    d, _ = drb.render_multi(scenes[:2], st, seed=21, sample_base=3, sample_count=3, accumulate_into=d, dynamic=True)
    assert np.array_equal(d, a)
    # sample shards: handle k traces sample range k, the parts are added in handle order by one kernel
    e, se = drb.render_multi(scenes, st, seed=21, shard="samples")
    assert se.rays == sf.rays and se.paths == sf.paths
    parts = [scenes[0].render(st, seed=21, sample_base=2 * k, sample_count=2)[0] for k in range(3)]
    assert np.array_equal(e, (parts[0] + parts[1]) + parts[2])
    assert np.allclose(e, full, rtol=0, atol=1e-5)
    e2, _ = drb.render_multi(scenes[:2], st, seed=21, shard="samples", accumulate_into=full.copy())
    assert np.allclose(e2, 2 * full, rtol=0, atol=2e-5)
    g, sg = drb.render_multi(scenes, st.replace(spp=2), seed=21, shard="samples")          # fewer samples than handles: an empty share
    assert sg.paths == 83 * 47 * 2 and np.allclose(g, parts[0], rtol=0, atol=1e-6)
    with pytest.raises(drb.DogerayError):
        bad = drb.Settings.from_buffer_copy(bytes(st)); bad.width = 0
        drb.render_multi(scenes[:2], bad)


def test_render_multi_on_two_devices():
    """the same through real peers: the scene created on device 0 and on device 1"""
    if drb.device_count() < 2:
        pytest.skip("needs two GPUs")
    objs, st = synth.heightfield_scene(n=32, width=130, height=75, spp=8, max_depth=6)
    hs = drb.HostScene.from_objects(objs, st)
    s0, s1 = drb.Scene.from_host(hs, device=0), drb.Scene.from_host(hs, device=1)
    full, sf = s0.render(st, seed=5)
    other, _ = s1.render(st, seed=5)
    assert np.array_equal(full, other)                                     # the build and the frame do not depend on the device
    img, sm = drb.render_multi([s0, s1], st, seed=5)
    assert np.array_equal(img, full) and sm.rays == sf.rays
    # the same scene made by ONE sharded upload + peer exchange; dynamic tiles and sample shards across real peers
    ndev = min(drb.device_count(), 4)
    scenes = drb.create_multi(hs, list(range(ndev)))
    w0 = s0.wide()
    for sc in scenes:
        w = sc.wide()
        assert np.array_equal(w["child"], w0["child"]) and np.array_equal(w["boxes"], w0["boxes"])
    for kw in (dict(), dict(dynamic=True)):
        img, sm = drb.render_multi(scenes, st, seed=5, **kw)
        assert np.array_equal(img, full) and sm.rays == sf.rays
    img, sm = drb.render_multi(scenes, st, seed=5, shard="samples")
    assert sm.rays == sf.rays and np.allclose(img, full, rtol=0, atol=1e-5)
    again, _ = drb.render_multi(scenes, st, seed=5, shard="samples")
    assert np.array_equal(again, img)                                      # fixed summation order

