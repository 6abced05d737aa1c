"""Wider parity sweep: every shipped sample scene, generated stand-ins for them, and randomised scenes, against the
oracle (bit-exact bars as in test_gpu_parity.py)."""
import os

import numpy as np
import pytest

import dogeray_b200 as drb
from dogeray_b200 import synth
from oracle import restated
from conftest import HAVE_REF, SAMPLES, all_sample_scenes, needs_ref, sample
from test_gpu_parity import Oracle, assert_frames_match, assert_ids_match

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def maybe_ref():
    if HAVE_REF:
        from oracle import refhost
        return refhost.RefHost()
    return None


def renderable_count(path):
    o = drb.HostScene.load(path, SAMPLES).objects()
    return int((((o["type"] == 2) & (o["ncols"] >= 16)) | ((o["type"] == 0) & (o["ncols"] >= 10))).sum())


def check_scene_file(maybe_ref, path, texdir, seed, max_depth=5):
    """a scene file at 64x48, 2 spp against the oracle: bit-exact ids and distances of every primary ray, equal ray
    counts, the frame within the bars of assert_frames_match"""
    sc = drb.Scene.load(path, texdir or None)
    st = sc.settings.replace(width=64, height=48, spp=2, max_depth=max_depth)
    orc = Oracle(path, texdir, maybe_ref)
    orc.apply(st, seed)
    ro, rd = sc.primary_rays(st, sample=0, seed=seed)
    ids, t = sc.trace_ids(ro, rd)
    oid, ot = orc.hit(ro, rd)
    # junk lines (HIGH.rts, light.rts) leave an indeterminate object in the reference's tree; ids of real objects must agree
    assert_ids_match(ids, t, oid, ot)
    f, fi, rays = orc.frame()
    acc, stats = sc.render(st, seed=seed)
    assert stats.rays == rays
    assert_frames_match(acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(0.5), f)
    return ids


@needs_ref
@pytest.mark.parametrize("name", all_sample_scenes())
def test_every_sample_scene(maybe_ref, name):
    path = sample(name)
    if os.path.getsize(path) == 0 or renderable_count(path) < 2:
        pytest.skip("the reference's build_bvh does not terminate on fewer than two objects")
    o = drb.HostScene.load(path, SAMPLES).objects()
    if ((o["type"] != 0) & (o["type"] != 2)).any():
        pytest.skip("legacy object types: undefined behaviour in the reference (SURVEY App. B.9)")
    check_scene_file(maybe_ref, path, SAMPLES, 31)


# Scenes generated here that stand in for the reference's sample scenes, which are not part of this repository: one kind
# per feature class those scenes exercise, each in several seeded variants of size, layout, materials and camera.
STAND_IN_KINDS = ("heightfield", "boxes", "soup", "blobs", "glass", "materials")
STAND_INS = [(kind, v) for kind in STAND_IN_KINDS for v in range(14)]


def box_quads(lo, hi, col, mat, rough):
    """the six faces of an axis-aligned box as twelve triangles, wound outwards"""
    (x0, y0, z0), (x1, y1, z1) = lo, hi
    faces = [((x0, y0, z0), (x0, y1, z0), (x1, y1, z0), (x1, y0, z0)), ((x0, y0, z1), (x1, y0, z1), (x1, y1, z1), (x0, y1, z1)),
             ((x0, y0, z0), (x0, y0, z1), (x0, y1, z1), (x0, y1, z0)), ((x1, y0, z0), (x1, y1, z0), (x1, y1, z1), (x1, y0, z1)),
             ((x0, y0, z0), (x1, y0, z0), (x1, y0, z1), (x0, y0, z1)), ((x0, y1, z0), (x0, y1, z1), (x1, y1, z1), (x1, y1, z0))]
    return np.concatenate([synth.quad(*f, col, mat, rough) for f in faces])


def write_stand_in(d, kind, v):
    """writes stand-in scene `kind` variant `v` as d/scene.rts (textures beside it); returns (path, texdir, max_depth)"""
    rng = np.random.default_rng(7000 + 100 * STAND_IN_KINDS.index(kind) + v)
    view = dict(look=(0, 0, 0), focus=3.0, aperture=float(rng.choice([0.0, 0.01, 0.1])), fov=int(rng.choice([35, 45, 60])))
    tex, backtex, depth = [], None, 5
    if kind == "heightfield":                   # one mesh, diffuse and metal facets (as the exported meshes)
        objs, st = synth.heightfield_scene(n=6 + 2 * v, seed=v, metal_every=2 + v % 5)
        st = st.replace(aperture=view["aperture"], fov=view["fov"])
    elif kind == "boxes":                       # axis-aligned boxes of quads (as cube.rts), half with the normalised diffuse lobe
        objs = np.concatenate([box_quads(c - h, c + h, rng.uniform(0.2, 0.95, 3), int(rng.choice([0, 0, 2, 3, 5])), float(rng.uniform(0, 0.3)))
                               for c, h in zip(rng.uniform(-3, 3, (8, 3)), rng.uniform(0.3, 1.2, (8, 3)))])
        objs["add_x"] = 0.5 * (v % 2)
        st = drb.default_settings().replace(cam=(float(rng.uniform(-5, 5)), -4.0, 7.0), **view)
    elif kind == "soup":                        # unstructured triangles of every material class, checker and smooth normals
        scale = float(rng.choice([0.5, 3.0, 40.0]))
        objs = random_scene(rng, int(rng.choice([64, 300, 1500])), scale, spheres=False, duplicates=False)
        st = drb.default_settings().replace(cam=(0.3 * scale, -0.2 * scale, 2.8 * scale), **view)
    elif kind in ("blobs", "glass"):            # closed smooth or flat meshes on a floor; glass at depth 8 (as glass.rts)
        mats = [(4, float(rng.uniform(1.2, 1.7)), 1)] * 3 if kind == "glass" else \
               [(0, 0.0, v % 2), (2, 0.0, 0), (3, float(rng.uniform(0.02, 0.3)), 1), (5, 0.05, v % 2), (1, 0.0, 0)]
        parts = []
        for k, (mat, rough, smooth) in enumerate(mats):
            v0, v1, v2, vn = synth.bumpy_torus(12 + 2 * v, 6 + v, R=1.6, r=0.7, seed=v * 10 + k)
            off = np.array([(k - (len(mats) - 1) / 2) * 4.5, -1.2, rng.uniform(-2, 2)], np.float32)
            o = drb.make_objects(len(v0))
            v0, v1, v2 = v0 + off, v1 + off, v2 + off
            o["pos"], o["dim"], o["rot"] = v0, v1, v2
            o["n1"], o["n2"], o["n3"] = vn
            fn = np.cross(v1 - v0, v2 - v0)
            o["norm"] = fn / np.maximum(np.linalg.norm(fn, axis=1, keepdims=True), 1e-30)
            o["col"] = (3.0, 2.4, 1.8) if mat == 1 else rng.uniform(0.3, 1.0, 3)
            o["mat"], o["add_y"], o["smooth"], o["ncols"] = mat, rough, smooth, 38
            parts.append(o)
        parts.append(synth.quad((-40, 0, -40), (40, 0, -40), (40, 0, 40), (-40, 0, 40), (0.7, 0.7, 0.7)))
        objs = np.concatenate(parts)
        st = drb.default_settings().replace(cam=(float(rng.uniform(-6, 6)), -6.0, 14.0), **dict(view, look=(0, -1, 0)))
        depth = 8 if kind == "glass" else 5
    else:                                       # textures, roughness map, checker and environment map (as bolter2 / rough / gloss)
        tex = synth.write_test_textures(d)
        objs, st, tex = synth.materials_scene(tex, nu=8 + 2 * (v % 4), nv=4 + v % 3)
        st = st.replace(cam=(float(v - 7), -7.0, 17.0), aperture=view["aperture"], fov=view["fov"])
        backtex = os.path.basename(tex[0])
    path = os.path.join(d, "scene.rts")
    drb.write_rts(path, st, objs, tex_names=[os.path.basename(t) for t in tex], backtex_name=backtex)
    return path, d if tex else "", depth


@pytest.mark.parametrize("kind,variant", STAND_INS)
def test_sample_scene_stand_ins(tmp_path, maybe_ref, kind, variant):
    """test_every_sample_scene's bars on the stand-in scenes, which run wherever the repository does"""
    path, texdir, depth = write_stand_in(str(tmp_path), kind, variant)
    ids = check_scene_file(maybe_ref, path, texdir, 31 + variant, depth)
    assert (ids >= 0).mean() > 0.2                                     # the camera sees the scene


def random_scene(rng, n, scale, spheres=True, duplicates=True):
    o = drb.make_objects(n)
    c = rng.uniform(-1, 1, (n, 3)) * scale
    o["pos"] = c
    o["dim"] = c + rng.normal(size=(n, 3)) * scale * 0.3
    o["rot"] = c + rng.normal(size=(n, 3)) * scale * 0.3
    o["col"] = rng.uniform(0.1, 1.0, (n, 3))
    o["mat"] = rng.choice([0, 0, 0, 1, 2, 3, 4, 5, 7], n)
    o["add_y"] = np.where(o["mat"] == 4, rng.uniform(1.1, 1.8, n), rng.uniform(0, 0.5, n))
    o["add_x"] = rng.choice([0.0, 0.5], n)
    fn = np.cross(o["dim"] - o["pos"], o["rot"] - o["pos"])
    fn /= np.maximum(np.linalg.norm(fn, axis=1, keepdims=True), 1e-20)
    has_n = rng.uniform(size=n) < 0.7
    o["norm"][has_n] = fn[has_n]
    vn = fn + rng.normal(size=(n, 3)) * 0.2
    for k in ("n1", "n2", "n3"):
        o[k][has_n] = (vn + rng.normal(size=(n, 3)) * 0.05)[has_n]
    o["smooth"] = rng.integers(0, 2, n)
    o["checker"] = (rng.uniform(size=n) < 0.2).astype(np.int32)
    o["t1"], o["t2"], o["t3"] = rng.uniform(0, 3, (n, 2)), rng.uniform(0, 3, (n, 2)), rng.uniform(0, 3, (n, 2))
    sph = (rng.uniform(size=n) < 0.1) & spheres                       # some spheres
    o["type"][sph] = 0
    o["dim"][sph, 0] = rng.uniform(0.05, 0.4, int(sph.sum())) * scale
    o["mat"][sph & (o["mat"] == 4)] = 3                               # glass spheres need an inside hit the reference does not have
    o["checker"][sph] = 0                                             # getnormal leaves texco uninitialised for spheres (kernel.cu:707-710): UB with the checker
    deg = rng.uniform(size=n) < 0.05                                  # zero-area triangles
    o["rot"][deg] = o["dim"][deg]
    dup = (rng.uniform(size=n) < 0.05) & duplicates                   # exact duplicates (all keys tie, equal t)
    src = rng.integers(0, n, n)
    for k in ("pos", "dim", "rot", "type"):
        o[k][dup] = o[k][src[dup]]
    o["ncols"] = 38
    return o


@pytest.mark.parametrize("seed", range(12))
def test_random_scenes(tmp_path, maybe_ref, seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.choice([3, 17, 64, 300, 1500]))
    scale = float(rng.choice([0.5, 3.0, 40.0]))
    # seeds 0-5: triangles only, no exact duplicates -> the strict bar; 6-8: + spheres; 9-11: + duplicated objects
    spheres, duplicates = seed >= 6, seed >= 9
    objs = random_scene(rng, n, scale, spheres, duplicates)
    st = drb.default_settings().replace(cam=(0.3 * scale, -0.2 * scale, 2.8 * scale), look=(0, 0, 0), width=72, height=48, spp=2, max_depth=6,
                                        focus=3.0, aperture=float(rng.choice([0.0, 0.01, 0.2])), fov=int(rng.choice([30, 45, 70])))
    p = str(tmp_path / "r.rts")
    drb.write_rts(p, st, objs)
    sc = drb.Scene.load(p)
    # closest hit: camera rays and random rays against the BVH-independent brute-force definition
    r = restated.Restated(p)
    ro, rd = sc.primary_rays(st, sample=0, seed=seed)
    o2 = rng.uniform(-2, 2, (4000, 3)).astype(np.float32) * scale
    d2 = rng.normal(size=(4000, 3)).astype(np.float32)
    allo = np.concatenate([ro.reshape(-1, 3), o2]); alld = np.concatenate([rd.reshape(-1, 3), d2])
    ids, t = sc.trace_ids(allo, alld)
    bid, bt = r.hit_brute(allo, alld)
    assert_ids_match(ids, t, bid, bt)
    # radiance against the oracle frame (same tree-independent semantics); duplicates make exact-t ties, whose winner
    # depends on the tree, so frames are compared only when the scene has no such tie among primary hits
    orc = Oracle(p, "", maybe_ref)
    orc.apply(st, seed)
    oid, ot = orc.hit(ro, rd)
    f, fi, rays = orc.frame()
    acc, stats = sc.render(st, seed=seed)
    ours = acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(0.5)
    identical = float(np.mean(np.all(ours == f, axis=-1)))
    rmse = float(np.sqrt(np.mean(((ours - f) / 255.0) ** 2)))
    assert np.isfinite(acc).all()
    if not spheres:
        # nothing tree-dependent, nothing library-dependent: the stated tolerance and the bit-identity bar
        assert stats.rays == rays
        assert identical >= 0.999 and rmse <= 1e-3, (identical, rmse)
    elif not duplicates:
        # hit_sphere squares lengths with powf(len, 2) (kernel.cu:320, 324); the device squares with one multiply, which is
        # the correctly rounded value glibc's powf misses by an ulp now and then -- a path may then take another branch
        # (at 2 spp one such path in a 72x48 image is already 5e-3 of RMSE).  Nearly every pixel is still bit-identical,
        # and the tolerance north_star states for CONVERGED radiance holds with room to spare at 64 spp.
        assert abs(stats.rays - rays) <= 0.002 * rays and identical >= 0.99, (stats.rays, rays, identical)
        st64 = st.replace(spp=64)
        orc.apply(st64, seed)
        f64, _, _ = orc.frame()
        acc64, _ = sc.render(st64, seed=seed)
        rmse64 = float(np.sqrt(np.mean(((acc64.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / 64) - f64) / 255.0) ** 2)))
        assert rmse64 <= 1e-3, rmse64
    else:
        # exact-t ties on duplicated objects keep the first one VISITED, which depends on the tree (the reference's median
        # split vs the LBVH): the twin may carry another material.  ids were checked above under the tie rule.
        assert identical >= 0.97 and rmse < 0.02, (identical, rmse)
