"""Refit against rebuild on one GPU, on the bench's 1 048 580-triangle scene (synth.instanced_grid_scene), object lines
already in device memory:

  refit     Scene.refit(tensor) (drb_scene_refit_device): host wall clock around the synchronous call, CUDA events
            around it on the caller's stream, and the summed device time of its kernels (torch.profiler); medians after
            a warm-up.  Nominal bytes moved: object lines read twice (validation, packing), the line -> slot map read
            twice, leaf boxes written and read (32 B per primitive), primitives and shading records written (192 B),
            nodes read and written (64 B each) and read once more as children.
  build     drb_scene_create_from_device on the same device array: host wall clock and the build's own device time
            (drb_build_info.build_ms).
  quality   closest-hit and occlusion Grays/s on a primary set and an ambient-occlusion set (built as in
            tools/ray_query_bench.py), and render Mrays/s on a reduced frame, after a refit and after a fresh build of
            the same moved geometry: every torus rotated about its own axis by 0, 10, 45 and 90 degrees, and a per-vertex
            jitter.

Prints one JSON line per record, with the device name and power limit read in the same run.

    python tools/refit_bench.py [--reps 7] [--samples 2] [--label TEXT] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dogeray_b200 as drb  # noqa: E402
from dogeray_b200 import synth  # noqa: E402
from ray_query_bench import event_ms, gpu_facts  # noqa: E402

GRID, NU, NV, SPACING = 4, 256, 128, 10.0
PER_TORUS = 2 * NU * NV


def torus_frames(seed=0):
    """centre and axis of every torus of instanced_grid_scene (same random tilts)"""
    rng = np.random.default_rng(seed)
    half = (GRID - 1) * SPACING / 2
    out = []
    for i in range(GRID):
        for j in range(GRID):
            ang = rng.uniform(-0.6, 0.6)
            c, s = np.cos(ang), np.sin(ang)
            out.append((np.array([i * SPACING - half, -2.2, j * SPACING - half]), np.array([0.0, c, s])))
    return out


def rotate_tori(objs, degrees):
    o = objs.copy()
    th = np.radians(degrees)
    for k, (c, a) in enumerate(torus_frames()):
        K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        R = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K                # Rodrigues
        sl = slice(k * PER_TORUS, (k + 1) * PER_TORUS)
        for f in ("pos", "dim", "rot"):
            o[f][sl] = ((o[f][sl] - c) @ R.T + c).astype(np.float32)
        for f in ("n1", "n2", "n3", "norm"):
            m = o[f][sl, 2] != -20.0
            v = o[f][sl]
            v[m] = (v[m] @ R.T).astype(np.float32)
            o[f][sl] = v
    return o


def jitter(objs, sigma=0.02, seed=3):
    o = objs.copy()
    rng = np.random.default_rng(seed)
    n = GRID * GRID * PER_TORUS
    for f in ("pos", "dim", "rot"):
        o[f][:n] += rng.normal(0, sigma, (n, 3)).astype(np.float32)
    return o


def to_dev(objs):
    return torch.from_numpy(objs.view(np.uint8).copy()).cuda()


def wall(fn, reps):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ms))


def kernel_ms(fn, prefix, reps):
    """summed device time of the kernels whose name contains `prefix`, per call (torch.profiler, CUPTI)"""
    fn()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    total_us = sum(e.self_device_time_total for e in prof.key_averages() if prefix in e.key)
    if total_us <= 0:
        raise RuntimeError("the profiler saw no %s* kernel" % prefix)
    return total_us / 1e3 / reps


def query_sets(sc, st, samples, dev):
    H, W = st.height, st.width
    O = torch.empty(samples, H, W, 3, device=dev); D = torch.empty_like(O)
    for s in range(samples):
        o, d = sc.primary_rays(st, s, seed=1)
        O[s] = torch.from_numpy(o); D[s] = torch.from_numpy(d)
    O = O.reshape(-1, 3); D = D.reshape(-1, 3)
    ids, t, uv = sc.trace(O, D)
    hit = ids >= 0
    info = sc.build_info
    extent = max(info.bounds_max[k] - info.bounds_min[k] for k in range(3))
    # geometric normal from the hit's ray: the occluder side does not matter for the rate
    Dh = D[hit]
    P = O[hit] + t[hit, None] * Dh
    N = -Dh / Dh.norm(dim=1, keepdim=True)
    P = P + N * (1e-4 * extent)
    gen = torch.Generator(device=dev); gen.manual_seed(7)
    u1 = torch.rand(len(P), device=dev, generator=gen); u2 = torch.rand(len(P), device=dev, generator=gen)
    helper = torch.where(N[:, :1].abs() < 0.9, torch.tensor([1.0, 0.0, 0.0], device=dev), torch.tensor([0.0, 1.0, 0.0], device=dev))
    T = torch.linalg.cross(helper, N); T = T / T.norm(dim=1, keepdim=True)
    B = torch.linalg.cross(N, T)
    r, phi = u1.sqrt(), 2 * np.pi * u2
    ao = T * (r * phi.cos())[:, None] + B * (r * phi.sin())[:, None] + N * (1 - u1).clamp_min(0).sqrt()[:, None]
    return [("primary", O.contiguous(), D.contiguous(), None),
            ("ao", P.contiguous(), ao.contiguous(), torch.full((len(P),), 0.05 * extent, device=dev))]


def rates(sc, sets, st_small, reps, dev):
    stream = torch.cuda.current_stream().cuda_stream
    out = {}
    for name, so, sd, tmax in sets:
        n = len(so)
        ids = torch.empty(n, dtype=torch.int32, device=dev); t = torch.empty(n, device=dev)
        occ = torch.empty(n, dtype=torch.bool, device=dev)
        c = event_ms(lambda: sc.trace_device(so.data_ptr(), sd.data_ptr(), n, ids.data_ptr(), t.data_ptr(), None, stream), reps)
        o = event_ms(lambda: sc.occluded_device(so.data_ptr(), sd.data_ptr(), n, occ.data_ptr(),
                                                tmax.data_ptr() if tmax is not None else None, stream), reps)
        out[name + "_closest_grays"] = round(n / c / 1e6, 4)
        out[name + "_occluded_grays"] = round(n / o / 1e6, 4)
    sc.render(st_small, seed=1)
    ms = []
    for _ in range(3):
        _, stats = sc.render(st_small, seed=1)
        ms.append(stats.total_ms)
    out["render_mrays"] = round(stats.rays / float(np.median(ms)) / 1e3, 1)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--samples", type=int, default=2)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    if drb.device_count() < 1:
        raise SystemExit("refit_bench needs a CUDA device")
    name, power = gpu_facts()
    dev = torch.device("cuda", 0)
    objs, st = synth.instanced_grid_scene(grid=GRID, nu=NU, nv=NV, width=1920, height=1080)
    hs = drb.HostScene.from_objects(objs, st)
    d_objs = to_dev(objs)
    stream = torch.cuda.current_stream()
    torch.cuda.synchronize()
    lines = []

    def emit(rec):
        rec.update(label=a.label, scene_prims=int(hs.num_renderable), device=name, power_limit_w=power)
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    # refit vs build on the same device array
    def create():
        return drb.Scene.from_device_objects(hs, d_objs.data_ptr(), stream=stream.cuda_stream)
    build_wall = wall(lambda: create().close(), a.reps)
    build_dev = []
    for _ in range(a.reps):
        s = create(); build_dev.append(s.build_info.build_ms); s.close()
    sc = create()
    refit_wall = wall(lambda: sc.refit(d_objs, stream=stream), a.reps)
    refit_event = event_ms(lambda: sc.refit(d_objs, stream=stream), a.reps)
    refit_kernels = kernel_ms(lambda: sc.refit(d_objs, stream=stream), "k_refit_", a.reps)
    bi = sc.build_info
    nobj, nprims, nwide = len(objs), bi.nprims, bi.nwide
    nbytes = 2 * 156 * nobj + 2 * 4 * nobj + 2 * 32 * nprims + 192 * nprims + 3 * 64 * nwide
    emit({"record": "refit_vs_build", "objects": nobj, "nwide": int(nwide), "wide_levels": int(bi.wide_levels),
          "refit_wall_ms": round(refit_wall, 3), "refit_event_ms": round(refit_event, 3), "refit_kernel_ms": round(refit_kernels, 3),
          "build_wall_ms": round(build_wall, 3), "build_device_ms": round(float(np.median(build_dev)), 3),
          "refit_bytes_nominal": int(nbytes), "refit_gbps_over_kernels": round(nbytes / refit_kernels / 1e6, 1),
          "speedup_wall": round(build_wall / refit_wall, 2)})

    # tree quality after a refit vs a fresh build of the same geometry
    st_small = st.replace(width=480, height=270, spp=4)
    for label, moved in [("rotate_0", rotate_tori(objs, 0.0)), ("rotate_10", rotate_tori(objs, 10.0)),
                         ("rotate_45", rotate_tori(objs, 45.0)), ("rotate_90", rotate_tori(objs, 90.0)), ("jitter_0.02", jitter(objs))]:
        dm = to_dev(moved)
        sc.refit(objs)                                                          # back to the build's geometry, then one step
        sc.refit(dm, stream=stream)
        fresh = drb.Scene.from_device_objects(hs, dm.data_ptr(), stream=stream.cuda_stream)
        sets = query_sets(fresh, st, a.samples, dev)
        r_refit = rates(sc, sets, st_small, a.reps, dev)
        r_fresh = rates(fresh, sets, st_small, a.reps, dev)
        rec = {"record": "quality", "deformation": label}
        rec.update({"refit_" + k: v for k, v in r_refit.items()})
        rec.update({"fresh_" + k: v for k, v in r_fresh.items()})
        rec["refit_over_fresh_primary_closest"] = round(r_refit["primary_closest_grays"] / r_fresh["primary_closest_grays"], 3)
        emit(rec)
        fresh.close()
        del sets, dm
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
