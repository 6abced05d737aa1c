#!/usr/bin/env python3
"""TEST / BASELINE INFRASTRUCTURE -- build the reference itself as the parity oracle.

Nothing of /root/reference is copied into the repository.  This recipe compiles the
reference's single translation unit, raygpu/kernel.cu, WHERE IT LIES, three ways, and
writes only binaries (and staged sample DATA files) into the git-ignored
``oracle/_ref/`` directory, which travels to the GPU box with the gpurun snapshot:

``libdogeray_ref_host.so``
    The reference's device + host functions as plain host C++ (SURVEY.md section 8c).
    ``kernel.cu`` cannot be handed to g++ whole (it includes SDL/Windows headers and
    contains a <<<>>> launch), so the line ranges that hold the data types, the device
    functions, ``Kernel`` and the loader / BVH builder are streamed through ``sed`` into
    the compiler's stdin between ``ref_host_shim.h`` and ``ref_host_api.inc``.  The only
    edit made to the stream is one instrumentation token: a thread-local ray counter
    bumped in front of the single ``hit()`` call in ``raycolor`` (kernel.cu:800), so the
    CPU baseline can report rays/s.  No sliced source is written to disk.

``libdogeray_ref_gpu.so``
    ``kernel.cu`` compiled UNMODIFIED by nvcc for sm_100 behind three stub headers
    (``oracle/stubs``) with ``-Dmain=ref_main``, plus the headless driver
    ``ref_gpu_driver.cu``.  This is the "reference kernel rebuilt for sm_100" baseline.

``libdogeray_ref_gpu_count.so``
    The same build with ONE call inserted in front of ``raycolor``'s ``hit()`` call (kernel.cu:800) that bumps a device
    counter, so that the GPU baseline's Mrays/s uses the reference's OWN ray count.  The edited stream lives in a
    temporary file outside the repo for the duration of the compile; this build is never the one that is timed.

``samples/``
    The reference's sample scenes and textures (DATA, not source), staged so that a
    machine without a checkout of the reference can render the same inputs.  Beside them,
    ``bolter2.blend.rts.bmp``: one of the reference's screenshots (SDL_SaveBMP output).

Run:  python oracle/make_ref.py [--reference /root/reference] [--no-gpu]
"""
import argparse
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")

# kernel.cu line ranges (1-based, inclusive) that make up the host slice:
#   27-32     render size globals
#   47-134    singleobject, bvh, file-scope settings
#   144-1093  vector helpers ... Kernel
#   1096-1909 random_double, getnum, gettexnum, read, pairsort ... build_bvh
SLICE = [(27, 32), (47, 134), (144, 1093), (1096, 1909)]
# the one instrumentation edit (see module docstring)
COUNT_SED = r"s/float3 hitoride = hit(rayo, raydir, bvhtree, b);/orc_rays++; &/"


def run(cmd, **kw):
    print("+", cmd if isinstance(cmd, str) else " ".join(cmd), flush=True)
    subprocess.run(cmd, check=True, **kw)


def build_host(ref_root):
    src = os.path.join(ref_root, "raygpu", "kernel.cu")
    ranges = ";".join("%d,%dp" % r for r in SLICE)
    out = os.path.join(OUT, "libdogeray_ref_host.so")
    shell = (
        "( echo '#include \"ref_host_shim.h\"';"
        " sed -n '{ranges}' '{src}' | sed '{count}';"
        " cat '{api}' ) |"
        " g++ -std=c++17 -O2 -ffp-contract=off -fPIC -shared -pthread -w -I'{here}' -x c++ - -o '{out}'"
    ).format(ranges=ranges, src=src, count=COUNT_SED, api=os.path.join(HERE, "ref_host_api.inc"), here=HERE, out=out)
    run(["bash", "-o", "pipefail", "-c", shell])
    return out


def build_gpu(ref_root):
    src = os.path.join(ref_root, "raygpu", "kernel.cu")
    out = os.path.join(OUT, "libdogeray_ref_gpu.so")
    run([
        "nvcc", "-std=c++17", "-O3", "-arch=sm_100", "-w", "-Xcompiler", "-fPIC", "-shared",
        "-I" + os.path.join(HERE, "stubs"), "-D_USE_MATH_DEFINES", "-Dmain=ref_main",
        '-DREF_KERNEL_CU="%s"' % src,
        os.path.join(HERE, "ref_gpu_driver.cu"), "-o", out,
    ])
    return out


def build_gpu_counting(ref_root):
    """the same build with a ray counter in front of raycolor's hit() call (kernel.cu:800).  The edited stream goes to a
    temporary file outside the repo, which is gone when the compile is; only the .so lands in oracle/_ref."""
    import tempfile
    src = os.path.join(ref_root, "raygpu", "kernel.cu")
    out = os.path.join(OUT, "libdogeray_ref_gpu_count.so")
    with tempfile.TemporaryDirectory(prefix="drb_refcount_") as td:
        edited = os.path.join(td, "kernel_counted.cu")
        run(["bash", "-o", "pipefail", "-c", "sed '%s' '%s' > '%s'" % (COUNT_SED.replace("orc_rays++;", "refgpu_count_ray();"), src, edited)])
        with open(edited) as f:
            if "refgpu_count_ray();" not in f.read():
                raise RuntimeError("the ray-counter edit did not apply (kernel.cu:800 changed?)")
        run([
            "nvcc", "-std=c++17", "-O3", "-arch=sm_100", "-w", "-Xcompiler", "-fPIC", "-shared",
            "-I" + os.path.join(HERE, "stubs"), "-D_USE_MATH_DEFINES", "-Dmain=ref_main", "-DREF_COUNT_RAYS",
            '-DREF_KERNEL_CU="%s"' % edited,
            os.path.join(HERE, "ref_gpu_driver.cu"), "-o", out,
        ])
    return out


def stage_samples(ref_root):
    src = os.path.join(ref_root, "samples")
    dst = os.path.join(OUT, "samples")
    os.makedirs(dst, exist_ok=True)
    n = 0
    for name in sorted(os.listdir(src)):
        low = name.lower()
        if low.endswith(".rts") or low.endswith(".ppm"):
            s, d = os.path.join(src, name), os.path.join(dst, name)
            if not os.path.exists(d) or os.path.getsize(d) != os.path.getsize(s):
                shutil.copyfile(s, d)
            n += 1
    extra = os.path.join(ref_root, "raygpu", "scene.rts")
    if os.path.exists(extra):
        shutil.copyfile(extra, os.path.join(dst, "_raygpu_scene.rts"))
        n += 1
    shot = os.path.join(ref_root, "images", "bolter2.blend.rts.bmp")      # the BMP writer's byte-for-byte fixture
    if os.path.exists(shot):
        shutil.copyfile(shot, os.path.join(OUT, "bolter2.blend.rts.bmp"))
        n += 1
    return n


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    ap.add_argument("--no-gpu", action="store_true", help="skip the nvcc build of the unmodified reference")
    args = ap.parse_args(argv)
    if not os.path.exists(os.path.join(args.reference, "raygpu", "kernel.cu")):
        print("reference not present at %s: keeping whatever is already in %s" % (args.reference, OUT))
        return 0
    os.makedirs(OUT, exist_ok=True)
    build_host(args.reference)
    if not args.no_gpu:
        build_gpu(args.reference)
        build_gpu_counting(args.reference)
    n = stage_samples(args.reference)
    print("staged %d sample files into %s" % (n, os.path.join(OUT, "samples")))
    return 0


if __name__ == "__main__":
    sys.exit(main())
