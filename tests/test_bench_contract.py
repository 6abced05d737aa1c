"""bench.py prints exactly one JSON line on stdout with the contract's keys (checked here through the reference
arm on the small workload, which needs no GPU; the GPU arm is checked by the gpu-marked test)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e"}


def run_bench(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one line, got %d" % len(lines)
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--workload", "cube", "--steps", "1", "--warmup", "0", "--cpu-spp", "1")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["metric"] == "Mrays/s" and d["unit"] == "Mrays/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_dumps_the_frame_of_its_last_step(tmp_path):
    import dogeray_b200 as drb
    from dogeray_b200 import synth
    from oracle import restated
    K = 3
    args = ["--impl", "reference", "--workload", "cube", "--steps", str(K), "--warmup", "1", "--cpu-spp", "1", "--dump-outputs"]
    dumps = []
    for k in range(2):
        d = tmp_path / str(k)
        assert run_bench(*args, str(d))["steps"] == K
        assert sorted(p.name for p in d.iterdir()) == ["frame_255.npy", "rays.npy"]
        dumps.append({p.stem: np.load(p) for p in d.iterdir()})
    for name in dumps[0]:
        assert np.array_equal(dumps[0][name], dumps[1][name]), name
    # the same frame computed here: the workload's text, 1 spp, seed 0, the last timed step's sample (K - 1)
    objs, st = synth.heightfield_scene(n=8, width=256, height=256, spp=16, max_depth=4)      # bench.py's "cube" workload
    p = str(tmp_path / "cube.rts")
    drb.write_rts(p, st, objs)
    r = restated.Restated(p, "")
    r.apply(st.replace(spp=1)); r.set_seed(0)
    f, _, rays = r.frame(1, K - 1)
    assert dumps[0]["frame_255"].dtype == np.float32 and np.array_equal(dumps[0]["frame_255"], f)
    assert dumps[0]["rays"].dtype == np.float64 and dumps[0]["rays"].tolist() == [rays]
    r.apply(st.replace(spp=1)); r.set_seed(0)
    assert not np.array_equal(r.frame(1, 0)[0], f)                                          # another step's frame would differ


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cube", "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "--steps" in p.stderr and p.stdout.strip() == ""


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cube", "--gpus", "2"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_line():
    d = run_bench("--workload", "cube", "--steps", "2", "--warmup", "3")
    assert BASE_KEYS <= set(d) and "impl" not in d and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3
    assert d["value"] > 0 and d["gpu_launches"] > 0 and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and "traffic" in r
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert d["parity"]["identical"] >= 0.999 and d["parity"]["rmse"] <= 1e-3          # the bench line carries its own parity evidence
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])


@pytest.mark.gpu
def test_gpu_arm_dumps_the_frame_of_its_last_step(tmp_path):
    import dogeray_b200 as drb
    from dogeray_b200 import synth
    d = run_bench("--workload", "cube", "--steps", "2", "--warmup", "1", "--no-baselines", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    assert sorted(p.name for p in tmp_path.iterdir()) == ["e2e_radiance_sum.npy", "e2e_rays_paths.npy",
                                                         "resident_radiance_sum.npy", "resident_rays_paths.npy"]
    objs, st = synth.heightfield_scene(n=8, width=256, height=256, spp=16, max_depth=4)      # bench.py's "cube" workload
    acc, stats = drb.Scene.from_host(drb.HostScene.from_objects(objs, st)).render(st, seed=0)
    for loop in ("resident", "e2e"):
        img, counts = np.load(tmp_path / (loop + "_radiance_sum.npy")), np.load(tmp_path / (loop + "_rays_paths.npy"))
        assert img.dtype == np.float32 and np.array_equal(img, acc), loop
        assert counts.dtype == np.float64 and counts.tolist() == [stats.rays, stats.paths], loop
