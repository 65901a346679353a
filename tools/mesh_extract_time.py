"""Times mesh extraction from a SphereSDF of the nerf_synthetic.py shape (128 spheres, randomly initialised non-zero
residual net) at 256^3, 512^3 and, if the memory fits, 1024^3: the lattice evaluation at f16 and f32, each extraction
kernel from the library's profile tags (iso_count, iso_scan, iso_emit), V and F, the extraction's bytes over its kernel
time against the measured device-to-device copy bandwidth, and peak memory.  The GPU name, power limit and SM clock are
read in the same run.  Prints one JSON object and writes it to --out.

    python tools/mesh_extract_time.py --out profiles/r04_mesh_extract_time.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from neural_raytracing_b200 import config, ops  # noqa: E402
from neural_raytracing_b200.pathtracer import mesh  # noqa: E402
from neural_raytracing_b200.pathtracer.shapes.sdfs import SphereSDF  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:       # the numbers are still valid; the record says why the card was not identified
        return {"name": torch.cuda.get_device_name(), "error": str(e)}


def shape(seed=0):
    torch.manual_seed(seed)
    s = SphereSDF(n=128, device="cuda")
    with torch.no_grad():
        for lin in s.shift._linears():
            lin.reset_parameters()
        s.shift.out.weight.mul_(0.1)
    s.invalidate_packed()
    return s


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return sorted(ms)[len(ms) // 2], out


def copy_bandwidth(nbytes=4 << 30):
    x = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    y.copy_(x)
    ms, _ = timed(lambda: y.copy_(x), 5)
    del x, y
    return 2 * nbytes / (ms * 1e-3)       # read + write


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="256,512,1024")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    s = shape()
    res = {"gpu": gpu_info(), "copy_bandwidth_GBps": copy_bandwidth() / 1e9, "sizes": []}
    for n in [int(x) for x in args.sizes.split(",")]:
        P = n ** 3
        free = torch.cuda.mem_get_info()[0]
        if 4 * P + 20 * P + (8 << 30) > free:          # values + extraction workspace + outputs, with margin
            res["sizes"].append({"n": n, "skipped": "needs more than the %.0f GB free" % (free / 1e9)})
            continue
        reps = 5 if n <= 256 else (3 if n <= 512 else 1)
        row = {"n": n}
        for prec in ("f16", "f32"):
            config.precision = prec
            mesh.sdf_grid(s, min(n, 64))                  # warm-up: module load, tensor-core blob
            ms, values = timed(lambda: mesh.sdf_grid(s, n), reps)
            row["lattice_eval_ms_" + prec] = ms
            row["lattice_eval_TFLOPs_" + prec] = P * 331e3 / (ms * 1e-3) / 1e12
        config.precision = "f16"
        values = mesh.sdf_grid(s, n)
        mesh.isosurface(values)                           # warm-up: workspace, CUB
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        ops.profile_enable(True)
        ops.profile_collect()
        kern = {"iso_count": [], "iso_scan": [], "iso_emit": []}
        for _ in range(reps):
            verts, faces = mesh.isosurface(values)
            torch.cuda.synchronize()
            prof = ops.profile_collect()
            for k in kern:
                kern[k].append(prof[k][0])
        ops.profile_enable(False)
        for k, v in kern.items():
            row[k + "_ms"] = sorted(v)[len(v) // 2]
        V, F = verts.shape[0], faces.shape[0]
        ext_ms = sum(row[k + "_ms"] for k in kern)
        # bytes the extraction must move: count reads values and writes 3 one-byte arrays; the scans read 2 and write
        # 16 bytes per point; emit reads values, mask and both offsets and writes the vertices and faces
        nbytes = P * (4 + 3) + P * (2 + 16) + P * (4 + 1 + 8 + 8) + 12 * V + 24 * F
        row.update(V=V, F=F, extraction_ms=ext_ms, extraction_bytes=nbytes,
                   extraction_GBps=nbytes / (ext_ms * 1e-3) / 1e9,
                   extraction_over_lattice_eval_f16=ext_ms / row["lattice_eval_ms_f16"],
                   peak_memory_GB_extraction=torch.cuda.max_memory_allocated() / 1e9)
        torch.cuda.reset_peak_memory_stats()
        ms, _ = timed(lambda: mesh.extract_mesh(s, n), reps)
        row["extract_mesh_end_to_end_ms_f16"] = ms
        row["peak_memory_GB_extract_mesh"] = torch.cuda.max_memory_allocated() / 1e9
        res["sizes"].append(row)
        del values, verts, faces
        ops._iso_ws_cache.clear()
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
