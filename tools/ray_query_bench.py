"""Ray-query rates on one GPU: closest hit (drb_trace_device), any hit (drb_occluded_device) and the host-array query
(drb_trace_ids, copies and synchronisation included) on three ray sets of the bench's 1 048 580-triangle scene
(synth.instanced_grid_scene):

  primary   `--samples` samples of 1920x1080 camera rays (primary_rays), tmax = 10000
  shadow    from every primary hit (offset along the face normal, toward the ray's side) to a point light above the grid,
            tmax = distance to the light
  ao        one cosine-distributed hemisphere ray per primary hit, tmax = 0.05 x the scene's largest extent

Each query is timed with CUDA events on one stream after one warm-up call (median of `--reps`); the host query with a wall
clock.  Every set is checked ray for ray: occluded == (closest id >= 0) & (closest t < tmax).  Prints one JSON line per set
with the device name and power limit read in the same run.

    python tools/ray_query_bench.py [--samples 16] [--reps 5] [--label TEXT] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dogeray_b200 as drb  # noqa: E402
from dogeray_b200 import synth  # noqa: E402


def gpu_facts():
    name = torch.cuda.get_device_name(0)
    power = None
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power = float(r.stdout.split()[0])
    except Exception:                                                   # noqa: BLE001  (reported as null)
        pass
    return name, power


def event_ms(fn, reps):
    fn()                                                                # warm-up
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def wall_ms(fn, reps):
    fn()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ms))


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=2)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    if drb.device_count() < 1:
        raise SystemExit("ray_query_bench needs a CUDA device")
    name, power = gpu_facts()
    objs, st = synth.instanced_grid_scene(grid=4, nu=256, nv=128, width=1920, height=1080)
    sc = drb.Scene.from_host(drb.HostScene.from_objects(objs, st))
    info = sc.build_info
    extent = max(info.bounds_max[k] - info.bounds_min[k] for k in range(3))
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream

    # primary rays
    H, W = st.height, st.width
    O = torch.empty(a.samples, H, W, 3, device=dev); D = torch.empty_like(O)
    for s in range(a.samples):
        o, d = sc.primary_rays(st, s, seed=1)
        O[s] = torch.from_numpy(o); D[s] = torch.from_numpy(d)
    O = O.reshape(-1, 3); D = D.reshape(-1, 3)
    ids, t, _ = sc.trace(O, D, with_uv=False)
    hit = ids >= 0
    # secondary rays from the hit points
    v0 = torch.from_numpy(objs["pos"].astype(np.float32)).to(dev)
    nrm = torch.linalg.cross(torch.from_numpy(objs["dim"].astype(np.float32)).to(dev) - v0,
                             torch.from_numpy(objs["rot"].astype(np.float32)).to(dev) - v0)
    nrm = nrm / nrm.norm(dim=1, keepdim=True).clamp_min(1e-30)
    N = nrm[ids[hit].long()]
    Dh = D[hit]
    N = torch.where(((N * Dh).sum(1, keepdim=True) > 0), -N, N)               # the face side the ray came from
    P = O[hit] + t[hit, None] * Dh + N * (1e-4 * extent)
    light = torch.tensor([5.0, -40.0, 8.0], device=dev)                         # above the grid (up is -y)
    toL = light - P
    dist = toL.norm(dim=1)
    gen = torch.Generator(device=dev); gen.manual_seed(7)
    u1 = torch.rand(len(P), device=dev, generator=gen); u2 = torch.rand(len(P), device=dev, generator=gen)
    helper = torch.where(N[:, :1].abs() < 0.9, torch.tensor([1.0, 0.0, 0.0], device=dev), torch.tensor([0.0, 1.0, 0.0], device=dev))
    T = torch.linalg.cross(helper, N); T = T / T.norm(dim=1, keepdim=True)
    B = torch.linalg.cross(N, T)
    r, phi = u1.sqrt(), 2 * np.pi * u2
    ao_d = T * (r * phi.cos())[:, None] + B * (r * phi.sin())[:, None] + N * (1 - u1).clamp_min(0).sqrt()[:, None]
    sets = [
        ("primary", O, D, None),
        ("shadow", P.contiguous(), (toL / dist[:, None]).contiguous(), dist.contiguous()),
        ("ao", P.contiguous(), ao_d.contiguous(), torch.full((len(P),), 0.05 * extent, device=dev)),
    ]
    del O, D, ids, t, hit, N, Dh, toL, u1, u2, helper, T, B, r, phi, ao_d
    torch.cuda.synchronize()

    lines = []
    for set_name, so, sd, tmax in sets:
        n = len(so)
        ids = torch.empty(n, dtype=torch.int32, device=dev); t = torch.empty(n, device=dev)
        occ = torch.empty(n, dtype=torch.bool, device=dev)
        closest_ms = event_ms(lambda: sc.trace_device(so.data_ptr(), sd.data_ptr(), n, ids.data_ptr(), t.data_ptr(), None, stream), a.reps)
        occ_ms = event_ms(lambda: sc.occluded_device(so.data_ptr(), sd.data_ptr(), n, occ.data_ptr(),
                                                     tmax.data_ptr() if tmax is not None else None, stream), a.reps)
        torch.cuda.synchronize()
        tm = tmax if tmax is not None else torch.full((n,), 1e4, device=dev)
        want = (ids >= 0) & (t < tm)
        mismatches = int((occ != want).sum())
        ho, hd = so.cpu().numpy(), sd.cpu().numpy()
        host_ms = wall_ms(lambda: sc.trace_ids(ho, hd), a.host_reps)
        hids, ht = sc.trace_ids(ho, hd)
        host_same = bool(np.array_equal(hids, ids.cpu().numpy()) and np.array_equal(ht, t.cpu().numpy()))
        rec = {
            "set": set_name, "rays": n, "label": a.label,
            "closest_ms": round(closest_ms, 3), "occluded_ms": round(occ_ms, 3), "host_trace_ids_ms": round(host_ms, 3),
            "closest_grays": round(n / closest_ms / 1e6, 4), "occluded_grays": round(n / occ_ms / 1e6, 4),
            "host_trace_ids_grays": round(n / host_ms / 1e6, 4),
            "hit_fraction": round(float((ids >= 0).float().mean()), 5), "occluded_fraction": round(float(occ.float().mean()), 5),
            "occluded_mismatches": mismatches, "host_ids_t_identical": host_same,
            "tmax": "1e4" if tmax is None else ("distance to light" if set_name == "shadow" else "%.4g" % (0.05 * extent)),
            "scene_prims": sc.num_prims, "device": name, "power_limit_w": power,
        }
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        assert mismatches == 0 and host_same, rec
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
