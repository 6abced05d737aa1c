#!/usr/bin/env python3
"""Headline benchmark: Mrays/s of the path-tracing hot path on BASELINE.json's million-triangle config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload grid1m|bunny|cube] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step is one full frame of the workload (all pixels x all samples).  With N > 1 the scene is replicated,
each rank traces spp/N of the sample indices and the radiance sums are reduced to rank 0 with one NCCL
reduce (strong scaling: the frame is fixed).  Rank 0 prints ONE JSON line.

  value      Mrays/s, whole job, scene resident in HBM, CUDA events on the launching stream, max over ranks
  e2e        same metric through the host-buffer API: every step uploads the object lines, rebuilds the LBVH
             on the GPU, renders, reduces and reads the float image back to the host (what one CudaStarter
             call of the reference spans, kernel.cu:2562-2669)
  roofline   the closest-hit kernel (k_trace): algorithmic bytes per ray (SURVEY.md 8d:
             32*ceil(log2 Ntris) + 36 + 64) x rays / its summed CUDA-event duration, against the measured
             HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline / --impl reference
             the reference's own trace function compiled for the host (oracle/_ref; else the C restatement)
             on all host cores, on a bounded sample (fewer samples per pixel) of the same frame
  ref_gpu    the reference's kernel.cu rebuilt unmodified for sm_100 (oracle/_ref), kernel-only and as one
             CudaStarter call, on a bounded sample of the same frame (north_star's first baseline)
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/s"
HBM_FALLBACK_GBS = 6650.0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


WORKLOAD_TEXTURES = []


def workload(name):
    from dogeray_b200 import synth
    if name == "grid1m":
        objs, st = synth.instanced_grid_scene(grid=4, nu=256, nv=128, width=1920, height=1080, spp=256, max_depth=10)
        desc = "synthetic 1M-triangle instanced grid (16 x 65536-tri bumpy tori + floor + wall), 1920x1080, 256 spp, 10 bounces"
    elif name == "bunny":
        objs, st = synth.bunny_class_scene(width=1920, height=1080, spp=64, max_depth=8)
        desc = "bunny-class stand-in (3 x 81920-tri blobs + floor + wall; sanford.blend.rts is a missing blob), 1920x1080, 64 spp, 8 bounces"
    elif name == "city10m":
        objs, st = synth.city_scene(width=3840, height=2160, spp=1024, max_depth=10)
        desc = "synthetic ~10M-triangle city grid, 3840x2160, 1024 spp, 10 bounces (BASELINE config 5 stand-in)"
    elif name == "mats":
        import tempfile
        d = tempfile.mkdtemp(prefix="drb_tex_")
        objs, st, tex = synth.materials_scene(synth.write_test_textures(d))
        WORKLOAD_TEXTURES[:] = tex
        desc = "material/texture/env-map divergence scene (10 material classes, 92k triangles), 1920x1080, 256 spp, 10 bounces (BASELINE config 4 stand-in)"
    elif name == "cube":
        objs, st = synth.heightfield_scene(n=8, width=256, height=256, spp=16, max_depth=4)
        desc = "small smoke workload, 256x256, 16 spp, 4 bounces"
    else:
        raise SystemExit("unknown workload %s" % name)
    return objs, st, desc


def bytes_per_ray(ntris):
    return 32 * math.ceil(math.log2(max(ntris, 2))) + 36 + 64


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_counters():
    """ncu counters of k_trace from this round's committed capture (profiles/trace_counters.json): what actually limits it"""
    p = os.path.join(ROOT, "profiles", "trace_counters.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


def profiled_traffic():
    """dram bytes per k_trace launch from the committed ncu capture, if one was recorded"""
    p = os.path.join(ROOT, "profiles", "trace_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.first = 0
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """the timed region starts here: earlier rows (the sampler's own start-up, the warm-up steps) do not count"""
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.first:] or self.rows[-1:]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class StdoutToStderr:
    """The reference prints banners to stdout (e.g. "N textures total", kernel.cu:1995); keep our stdout to the one
    JSON line by pointing file descriptor 1 at stderr while reference code runs."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


_SCENE_FILE = {}
LAST_CPU_FRAME = {}      # the CPU baseline's last frame (255 * mean, (W, H, 3)) with its sample range: the bench line's parity check


def scene_file(objs, st):
    """the workload as a .rts text file in its own directory (written once; the reference only reads files)"""
    import dogeray_b200 as drb
    if "path" not in _SCENE_FILE:
        tmp = tempfile.mkdtemp(prefix="drb_bench_")
        path = os.path.join(tmp, "scene.rts")
        t0 = time.time()
        drb.write_rts(path, st, objs)
        log("[bench] wrote %s (%.0f MB) in %.1f s" % (path, os.path.getsize(path) / 1e6, time.time() - t0))
        _SCENE_FILE["path"], _SCENE_FILE["dir"] = path, tmp
    return _SCENE_FILE["path"], _SCENE_FILE["dir"]


def scene_file_cleanup():
    if "path" in _SCENE_FILE:
        try:
            os.remove(_SCENE_FILE["path"]); os.rmdir(_SCENE_FILE["dir"])
        except OSError:
            pass
        _SCENE_FILE.clear()


def cpu_reference_arm(objs, st, desc, spp_sample, steps, warmup, threads):
    """the reference's host-compiled trace function (or the restatement) on a bounded sample: `spp_sample`
    samples per pixel of the same frame.  Returns (Mrays/s, ms per step, kind, rays per path)."""
    from oracle import refhost, restated
    path, tmp = scene_file(objs, st)
    t0 = time.time()
    s = st.replace(spp=spp_sample)
    if refhost.available():
        kind = "reference"
        eng = refhost.RefHost()
        eng.load(path, "")
        eng.apply(s); eng.set_seed(0)
        frame = lambda base: eng.frame(1, base, threads)
    else:
        kind = "port"
        eng = restated.Restated(path, "")
        eng.apply(s); eng.set_seed(0)
        frame = lambda base: eng.frame(1, base, threads)
    log("[cpu %s] scene parsed + host BVH built in %.1f s" % (kind, time.time() - t0))
    for w in range(warmup):
        frame(1000 + w)
    rays = 0; t1 = time.time()
    for k in range(steps):
        f, _, r = frame(k * spp_sample)
        rays += r
    dt = time.time() - t1
    paths = st.width * st.height * spp_sample * steps
    LAST_CPU_FRAME["frame"], LAST_CPU_FRAME["base"], LAST_CPU_FRAME["spp"], LAST_CPU_FRAME["rays"] = f, (steps - 1) * spp_sample, spp_sample, r
    return rays / dt / 1e6, dt / steps * 1e3, kind, rays / max(paths, 1)


def ref_gpu_baseline(objs, st, spp_sample):
    """kernel.cu rebuilt for sm_100, kernel-only (CUDA events, resident buffers) at `spp_sample` spp of the same frame.
    Rays are the reference's OWN count: the same launch of the instrumented build (a counter in front of raycolor's
    hit() call, oracle/make_ref.py build_gpu_counting), which is never the build that is timed."""
    import ctypes as C
    import numpy as np
    lib = os.path.join(ROOT, "oracle", "_ref", "libdogeray_ref_gpu.so")
    lib_count = os.path.join(ROOT, "oracle", "_ref", "libdogeray_ref_gpu_count.so")
    if not os.path.exists(lib):
        return {"unavailable": "oracle/_ref/libdogeray_ref_gpu.so not built"}
    path, tmp = scene_file(objs, st)
    sv = np.array([st.cam[0], st.cam[1], st.cam[2], st.aperture, st.look[0], st.look[1], st.look[2], st.focus, st.fov, st.max_depth,
                   spp_sample, st.bg_intensity, st.backtex, st.width, st.height, 0], np.float32)
    out = np.zeros((st.width, st.height, 3), np.int32)
    paths = st.width * st.height * spp_sample

    def load(libpath):
        L = C.CDLL(libpath)
        L.refgpu_load.argtypes = [C.c_char_p, C.c_char_p]
        L.refgpu_set_settings.argtypes = [C.c_void_p]
        L.refgpu_kernel_only.argtypes = [C.c_void_p, C.c_int, C.c_int]; L.refgpu_kernel_only.restype = C.c_float
        L.refgpu_rays.argtypes = [C.c_int]; L.refgpu_rays.restype = C.c_longlong
        t0 = time.time()
        n = L.refgpu_load(os.fsencode(path), os.fsencode(tmp))
        if n <= 0:
            raise RuntimeError("refgpu_load returned %d" % n)
        L.refgpu_set_settings(sv.ctypes.data)
        return L, time.time() - t0

    rays, rays_src = None, None
    if os.path.exists(lib_count):
        Lc, _ = load(lib_count)
        Lc.refgpu_rays(1)
        if Lc.refgpu_kernel_only(out.ctypes.data, 1, 1) > 0:
            rays = int(Lc.refgpu_rays(1))
            rays_src = "counted by the reference's own raycolor (instrumented build, separate untimed launch at the same spp)"
        Lc.refgpu_free()
    L, load_s = load(lib)
    L.refgpu_kernel_only(out.ctypes.data, 1, 1)                       # warm-up
    launches = 3
    ms = L.refgpu_kernel_only(out.ctypes.data, 1, launches)
    L.refgpu_free()
    if rays is None:
        return {"unavailable": "the ray-counting build of the reference is missing: no ray count of its own"}
    return {"kernel_only_mrays_s": rays / (ms * 1e-3) / 1e6 if ms > 0 else None, "kernel_ms": ms, "launches_timed": launches,
            "spp": spp_sample, "paths": paths, "rays": rays, "rays_per_path": rays / paths, "rays_source": rays_src,
            "sample": "same frame at %d of %d spp (kernel.cu unmodified, nvcc -arch=sm_100, kernel only from resident buffers, mean of %d launches after one warm-up)"
                      % (spp_sample, st.spp, launches),
            "host_parse_build_s": round(load_s, 2), "mean_pixel": float(out.mean())}


def parity_against_cpu_frame(drb, device, kind):
    """The CPU baseline leg rendered `spp` samples of the frame from the .rts text with the reference's own code; render
    the same sample range of the same text on the GPU and compare: the bench line carries its own parity evidence."""
    import numpy as np
    if "frame" not in LAST_CPU_FRAME or "path" not in _SCENE_FILE:
        return None
    f, base, spp, cpu_rays = LAST_CPU_FRAME["frame"], LAST_CPU_FRAME["base"], LAST_CPU_FRAME["spp"], LAST_CPU_FRAME["rays"]
    hs = drb.HostScene.load(_SCENE_FILE["path"], _SCENE_FILE["dir"])
    sc = drb.Scene.from_host(hs, device=device)
    st = sc.settings
    acc, stats = sc.render(st, seed=0, sample_base=base, sample_count=spp)
    sc.close(); hs.close()
    ours = acc.transpose(1, 0, 2) * np.float32(255.0) * np.float32(1.0 / spp)
    diff = (ours.astype(np.float64) - f.astype(np.float64)) / 255.0
    return {"against": "cpu_baseline frame (%s), samples [%d, %d) of every pixel, %d x %d" % (kind, base, base + spp, st.width, st.height),
            "identical": float(np.mean(np.all(ours == f, axis=-1))), "rmse": float(np.sqrt(np.mean(diff ** 2))),
            "max_abs": float(np.abs(diff).max()), "rays_equal": bool(stats.rays == cpu_rays), "rays": int(stats.rays), "cpu_rays": int(cpu_rays)}


DUMP_LIMIT_BYTES = 30 << 20          # per array; a dump holds at most two images, so it stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy.  An array larger than DUMP_LIMIT_BYTES is kept as every k-th row of its
    flattening to (-1, last axis), i.e. every k-th pixel of an image in row-major order: the same pixels for the same
    arguments, whichever build wrote them."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if a.nbytes > DUMP_LIMIT_BYTES:
            a = a.reshape(-1, a.shape[-1])[::-(-a.nbytes // DUMP_LIMIT_BYTES)]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
        log("[bench] dumped %s %s %s to %s" % (name, a.dtype, a.shape, out_dir))


def emit(line):
    """the ONE line on the real stdout"""
    os.write(REAL_STDOUT, (json.dumps(line) + "\n").encode())


REAL_STDOUT = 1


def main():
    # Libraries print banners to stdout (NCCL's version line, the reference's "N textures total"); keep the real
    # stdout for the one JSON line and point file descriptor 1 at stderr for everything else.
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="grid1m")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-spp", type=int, default=0, help="samples per pixel of the CPU baseline's bounded sample (0 = auto)")
    ap.add_argument("--no-baselines", action="store_true", help="skip cpu_baseline / ref_gpu (profiling runs)")
    ap.add_argument("--shard", default="samples", choices=["samples", "tiles"],
                    help="N > 1: shard sample indices (default) or interleaved 8x4-pixel tiles (bit-identical to the 1-GPU image)")
    ap.add_argument("--batch-paths", type=int, default=0, help="paths in flight per wavefront batch (0 = library default)")
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (profiling runs only; invalidates the metric)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step of each timed loop computed as DIR/<name>.npy: "
                         "resident_* for the scene-resident loop behind 'value', e2e_* for the host-buffer loop behind 'e2e' "
                         "(--impl reference: the last CPU frame), so that two builds can be compared output for output (the "
                         "inputs depend on the arguments only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    K, W = args.steps, args.warmup

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    objs, st, desc = workload(args.workload)
    if args.spp:
        st = st.replace(spp=args.spp)
    ntris = int((objs["type"] == 2).sum())
    config = {"workload": desc, "triangles": ntris, "width": st.width, "height": st.height, "spp": st.spp, "max_depth": st.max_depth,
              "seed": 0, "sharding": "samples, contiguous ranges per rank, one NCCL reduce of the float radiance sums to rank 0" if world > 1 else "none",
              "l2": "working set per step (ray queues: 120 B per path slot, 64 GB for the frame; scene 225 MB) exceeds the 126 MB L2; no explicit flush"}
    ncores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return 0
        spp_s = args.cpu_spp or 8
        with StdoutToStderr():
            v, ms, kind, rpp = cpu_reference_arm(objs, st, desc, spp_s, K, W, ncores)
        sample = "%d of %d spp per step on %d host threads (same scene, camera, depth)" % (spp_s, st.spp, ncores)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": ncores, "kind": kind, "sample": sample},
                "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "rays_per_path": rpp, "gpu_launches": 0}
        if args.dump_outputs:
            # the last timed CPU frame (the reference's Kernel(), or its C restatement): 255 * mean radiance, indexed [x, y]
            dump_outputs(args.dump_outputs, {"frame_255": LAST_CPU_FRAME["frame"], "rays": [float(LAST_CPU_FRAME["rays"])]})
        scene_file_cleanup()
        emit(line)
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    import dogeray_b200 as drb
    from dogeray_b200.distributed import shard_samples

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: dogeray_b200 has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    t0 = time.time()
    hs = drb.HostScene.from_objects(objs, st, WORKLOAD_TEXTURES)
    scene = drb.Scene.from_host(hs, device=local)
    bi = scene.build_info
    log("[rank %d] scene: %d prims, %d nodes, height %d, upload %.1f ms, GPU LBVH build %.1f ms (host wall %.2f s)" %
        (rank, bi.nprims, bi.nnodes, bi.max_depth, bi.upload_ms, bi.build_ms, time.time() - t0))

    if args.shard == "tiles" and world > 1:
        base, count, tile_kw = 0, st.spp, dict(tile_rank=rank, tile_count=world)
        config["sharding"] = "interleaved 8x4-pixel tiles (tile t -> rank t mod N), one NCCL reduce of the disjoint partial images to rank 0"
    else:
        (base, count), tile_kw = shard_samples(st.spp, rank, world), {}
    accum = torch.zeros(st.height, st.width, 3, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        if tile_kw:
            accum.zero_()
        s = scene.render_device(accum.data_ptr(), st, seed=0, sample_base=base, sample_count=count, batch_paths=args.batch_paths, stream=stream, want_stats=True, **tile_kw)
        if world > 1:
            dist.reduce(accum, dst=0)
        return s

    # nvidia-smi is started BEFORE the warm-up: its NVML start-up holds driver locks for tens of milliseconds, which
    # showed up as a ~85 ms hole in the kernel launches of the first timed step when it was started after it
    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(W):
        step_resident()
    barrier()
    if clocks:
        clocks.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rays = 0; paths = 0; trace_ms = 0.0; launches = 0; trace_launches = 0
    e0.record()
    for _ in range(K):
        s = step_resident()
        log("[rank %d] resident step: %.1f ms total, %.1f ms in k_trace" % (rank, s.total_ms, s.trace_ms))
        rays += s.rays; paths += s.paths; trace_ms += s.trace_ms; launches += s.kernel_launches; trace_launches += s.trace_launches
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if clocks else None

    def step_outputs(stats, img):
        """what one step hands its caller: the radiance sums of the frame (rank 0, after the reduce) and the rays and
        paths traced, summed over ranks"""
        counts = torch.tensor([float(stats.rays), float(stats.paths)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(counts)
        return img.cpu().numpy() if rank == 0 else None, counts.cpu().numpy()

    if args.dump_outputs:
        resident_out = step_outputs(s, accum)          # the e2e steps below overwrite accum
    tot = torch.tensor([float(rays), float(paths), ms, trace_ms, float(launches), float(trace_launches)], device=dev, dtype=torch.float64)
    if world > 1:
        mx = tot.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tot.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        rays_all, paths_all, ms_max, trace_ms_max, launches_all = sm[0].item(), sm[1].item(), mx[2].item(), mx[3].item(), sm[4].item()
    else:
        rays_all, paths_all, ms_max, trace_ms_max, launches_all = float(rays), float(paths), ms, trace_ms, float(launches)
    value = rays_all / (ms_max * 1e-3) / 1e6
    image_mean = float(accum.mean().item()) / max(st.spp, 1) if rank == 0 else 0.0

    # ---- e2e: host buffers in, host image out, every step -------------------------------------------------
    # One CudaStarter call of the reference uploads the whole scene, renders and downloads (kernel.cu:2604-2651).  Here,
    # per step: the object lines go host -> device from pinned memory (N > 1: rank r uploads lines [r*chunk, (r+1)*chunk)
    # and ONE all-gather over NVLink completes the array on every GPU, so the node pays the PCIe upload once, not N
    # times), the tree is rebuilt on the GPU, the frame is rendered, reduced, and the float image is read back.
    host_img = torch.empty(st.height, st.width, 3, pin_memory=True)
    nobj = hs.num_objects
    rec = drb.OBJECT_DTYPE.itemsize
    d2h = st.height * st.width * 3 * 4
    if world > 1:
        chunk = (nobj + world - 1) // world
        lo, hi = min(nobj, rank * chunk), min(nobj, (rank + 1) * chunk)
        mine = torch.zeros(chunk * rec, dtype=torch.uint8).pin_memory()
        mine[: (hi - lo) * rec] = torch.from_numpy(hs.objects()[lo:hi].view(np.uint8).copy())
        gathered = torch.empty(world * chunk * rec, dtype=torch.uint8, device=dev)
        h2d = world * chunk * rec                                  # whole job, per step
        config["e2e_upload"] = "each rank uploads 1/%d of the object lines (%d B), one NCCL all-gather completes the array on every GPU" % (world, chunk * rec)
    else:
        h2d = nobj * rec

    e2e_parts = {"create_ms": 0.0, "render_ms": 0.0, "reduce_readback_ms": 0.0, "free_ms": 0.0}

    def step_e2e():
        t0 = time.perf_counter()
        if world > 1:
            part = mine.to(dev, non_blocking=True)                # H2D of this rank's share
            dist.all_gather_into_tensor(gathered, part)
            sc = drb.Scene.from_device_objects(hs, gathered.data_ptr(), device=local, stream=stream)   # GPU LBVH build
        else:
            sc = drb.Scene.from_host(hs, device=local)            # H2D of every object line + GPU LBVH build
        t1 = time.perf_counter()
        if tile_kw:
            accum.zero_()
        s = sc.render_device(accum.data_ptr(), st, seed=0, sample_base=base, sample_count=count, batch_paths=args.batch_paths, stream=stream, want_stats=True, **tile_kw)
        t2 = time.perf_counter()
        if world > 1:
            dist.reduce(accum, dst=0)
        if rank == 0:
            host_img.copy_(accum, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        t3 = time.perf_counter()
        sc.close()
        t4 = time.perf_counter()
        for k, v in zip(e2e_parts, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            e2e_parts[k] += v * 1e3
        log("[rank %d] e2e step: create %.1f ms, render %.1f ms (device %.1f, k_trace %.1f), reduce+readback %.1f ms, free %.1f ms" %
            (rank, (t1 - t0) * 1e3, (t2 - t1) * 1e3, s.total_ms, s.trace_ms, (t3 - t2) * 1e3, (t4 - t3) * 1e3))
        return s

    scene.close()
    for _ in range(min(W, 1)):
        step_e2e()
    barrier()
    for k in e2e_parts:
        e2e_parts[k] = 0.0
    t_e = time.perf_counter(); e_rays = 0
    for _ in range(K):
        last = step_e2e()
        e_rays += last.rays
    barrier()
    e_ms = (time.perf_counter() - t_e) * 1e3
    if args.dump_outputs:
        e2e_out = step_outputs(last, host_img)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"resident_radiance_sum": resident_out[0], "resident_rays_paths": resident_out[1],
                                             "e2e_radiance_sum": e2e_out[0], "e2e_rays_paths": e2e_out[1]})
    et = torch.tensor([float(e_rays), e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        es = et.clone(); dist.all_reduce(es, op=dist.ReduceOp.SUM)
        em = et.clone(); dist.all_reduce(em, op=dist.ReduceOp.MAX)
        e_rays_all, e_ms_max = es[0].item(), em[1].item()
    else:
        e_rays_all, e_ms_max = float(e_rays), e_ms
    e2e_value = e_rays_all / (e_ms_max * 1e-3) / 1e6

    free_b, total_b = torch.cuda.mem_get_info(dev)
    hbm_used_gb = (total_b - free_b) / 1e9                         # scene + ray queues + cached blocks, after the last step

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        bpr = bytes_per_ray(ntris)
        # k_trace runs on every rank at once: per-GPU achieved bandwidth = this rank's rays x bytes / its trace time
        achieved = (rays * bpr) / (trace_ms * 1e-3) / 1e9 if trace_ms > 0 else 0.0
        traffic = profiled_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "spp_per_s_1080p": paths_all / (ms_max * 1e-3) / 2073600.0, "rays_per_path": rays_all / max(paths_all, 1.0),
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e_ms_max / K,
                    "what": "per step: upload object lines, GPU LBVH build, render, reduce, float image to pinned host memory",
                    "parts_ms_per_step_rank0": {k: v / K for k, v in e2e_parts.items()}},
            "gpu_launches": int(launches_all),
            "roofline": {"bound": "hbm", "kernel": "k_trace", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (traffic["dram_bytes_per_second"] * (trace_ms / max(trace_launches, 1)) * 1e-3) if traffic and "dram_bytes_per_second" in traffic else None,
                         "traffic_source": ("DRAM bytes/s of k_trace in the committed ncu capture (%s) x this run's mean launch duration" % traffic["source"]) if traffic else None,
                         "algorithmic_bytes_per_launch": bpr * rays / max(trace_launches, 1), "peak_source": peak_src,
                         "bytes_per_ray": bpr, "rays_per_launch": rays / max(trace_launches, 1), "trace_ms_per_step": trace_ms / K,
                         "trace_share_of_step": trace_ms / ms if ms > 0 else None,
                         "note": "algorithmic bytes = 32*ceil(log2 Ntris) + 36 + 64 per ray (SURVEY.md 8d); scenes of this size are largely L2-resident, see profiles/"},
            "clocks": clk, "image_mean_radiance": image_mean,
            "build": {"upload_ms": bi.upload_ms, "lbvh_build_ms": bi.build_ms, "tree_height": bi.max_depth, "wide_nodes": int(bi.nwide),
                      "wide_levels": bi.wide_levels, "stack_levels": bi.stack_levels},
            "hbm_in_use_gb": hbm_used_gb,
        }
        counters = profiled_counters()
        if counters:
            line["roofline"].update(counters)
        if world == 1 and not args.no_baselines:
            rpp = rays_all / max(paths_all, 1.0)
            try:
                spp_s = args.cpu_spp or 8
                with StdoutToStderr():
                    v, cms, kind, _ = cpu_reference_arm(objs, st, desc, spp_s, 1, 0, ncores)
                line["cpu_baseline"] = {"value": v, "unit": "Mrays/s", "cores": ncores, "kind": kind,
                                        "sample": "%d of %d spp of the same frame on %d host threads, %.1f s" % (spp_s, st.spp, ncores, cms / 1e3)}
                line["parity"] = parity_against_cpu_frame(drb, local, kind)
            except Exception as ex:                                  # the baseline must never cost the measurement
                line["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "cores": ncores, "kind": "port", "sample": "failed: %r" % (ex,)}
            try:
                with StdoutToStderr():
                    line["ref_gpu"] = ref_gpu_baseline(objs, st, 32)
            except Exception as ex:
                line["ref_gpu"] = {"unavailable": repr(ex)}
            scene_file_cleanup()
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
