"""Builds neural_raytracing_b200/lib/libnrt_b200.so with nvcc for sm_100a (in-tree, so the
built library travels to the GPU box with the repo snapshot).  No torch involved: the library is
a plain C-ABI shared object (include/nrt_b200.h)."""
import concurrent.futures
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
# NRT_BUILD_TAG (development): kernel variants (NRT_EXTRA_NVCC_FLAGS=-D...) built side by side as
# lib/libnrt_b200_<tag>.so; NRT_LIB_TAG selects one at load time (_native.py).  The product is the untagged build.
TAG = os.environ.get("NRT_BUILD_TAG", "")
OBJ = os.path.join(ROOT, "build", "nrt_obj" + ("_" + TAG if TAG else ""))
LIB = os.path.join(HERE, "lib", "libnrt_b200%s.so" % ("_" + TAG if TAG else ""))

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"),
          "-I" + CSRC]
# per-translation-unit extra flags.  The fp32 "exact" path must not contract a*b+c on its own:
# every fused multiply-add there is an explicit fmaf (see include/nrt_detmath.h).
EXTRA_ENV = os.environ.get("NRT_EXTRA_NVCC_FLAGS", "").split()
EXTRA = {
    "nrt_f32.cu": ["-fmad=false"],
    "nrt_f32_bwd.cu": ["-fmad=false"],
    "nrt_sdf_grad.cu": ["-fmad=false"],
    "nrt_shade.cu": ["-fmad=false"],
    "nrt_shade_direct.cu": ["-fmad=false"],
    "nrt_camera.cu": ["-fmad=false"],
    "nrt_mesh.cu": ["-fmad=false"],
}


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _digest(path, flags):
    h = hashlib.sha256()
    h.update(" ".join(flags).encode())
    for p in [path] + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))) + \
            sorted(os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))):
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _compile(src):
    name = os.path.basename(src)
    flags = ARCH + COMMON + EXTRA.get(name, []) + EXTRA_ENV
    obj = os.path.join(OBJ, name + ".o")
    stamp = obj + ".sha"
    dg = _digest(src, flags)
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dg:
        return obj, False
    cmd = [_nvcc()] + flags + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (name, r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(dg)
    return obj, True


def build(verbose=True):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    srcs = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        res = list(ex.map(_compile, srcs))
    objs = [o for o, _ in res]
    changed = any(c for _, c in res)
    if changed or not os.path.exists(LIB):
        cmd = [_nvcc()] + ARCH + ["-shared", "-cudart", "static", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        print("libnrt_b200: %d sources, %s -> %s" % (len(srcs), "rebuilt" if changed else "up to date", LIB))
    return LIB


if __name__ == "__main__":
    build()
    sys.exit(0)
