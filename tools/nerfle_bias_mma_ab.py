"""A/B of the NRT_BIAS_MMA switch (csrc/tc_core.cuh) on the cfg2 frame that bench.py measures.

    python tools/nerfle_bias_mma_ab.py [--pairs 3] [--steps 10] [--warmup 3] [--base bm0] [--new ""] [--extra main,bm2]
                                       [--out DIR]

Each build is a library variant next to the product one (build_native.py: NRT_BUILD_TAG=<tag>
NRT_EXTRA_NVCC_FLAGS=-DNRT_BIAS_MMA=<v> builds lib/libnrt_b200_<tag>.so; "" is the untagged product build), selected per
run with NRT_LIB_TAG.  The script runs `bench.py --gpus 1` for the base and the new build in alternation, `--pairs`
times, reads `ms_per_step` and the per-kernel `kernel_ms` of every JSON line, and reports per build the median, the
spread between its own runs ((max - min) / median) and the change of the new build against the base.  Every build,
including the `--extra` ones, also runs once with `--dump-outputs`, and the frames are compared with the base build's:
max-abs and RMS difference, and whether they are bit-identical.  The GPU name, its power limit and SM clocks are read
in the same run.  Writes ab.json and the dumped frames under --out (default: a new temporary directory)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = ("mlp_tc_nerf_first", "mlp_tc_nerf_second")


def lib_path(tag):
    return os.path.join(ROOT, "neural_raytracing_b200", "lib", "libnrt_b200%s.so" % ("_" + tag if tag else ""))


def run_bench(tag, args, dump=None):
    env = dict(os.environ, NRT_LIB_TAG=tag)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(args.steps), "--warmup",
           str(args.warmup), "--no-also", "--no-cpu-baseline"]
    if dump:
        cmd += ["--dump-outputs", dump]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError("bench.py failed for build %r:\n%s" % (tag, r.stderr[-4000:]))
    line = json.loads(r.stdout.strip().splitlines()[-1])
    rec = {"ms_per_step": line["ms_per_step"], "clocks": line.get("clocks")}
    for k in KERNELS:
        rec[k] = line["kernel_ms"][k]
    return rec


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")])) if r.returncode == 0 else {}


def summary(runs):
    out = {}
    for key in ("ms_per_step",) + KERNELS:
        v = [r[key] for r in runs]
        med = statistics.median(v)
        out[key] = {"runs": v, "median": med, "spread": (max(v) - min(v)) / med}
    out["sm_mhz"] = [(r.get("clocks") or {}).get("sm_mhz") for r in runs]   # bench.py's clock samples of each run
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--base", default="bm0", help="library tag of the reference build (NRT_BIAS_MMA=0)")
    ap.add_argument("--new", default="", help="library tag of the build under test (default: the product build)")
    ap.add_argument("--extra", default="", help="comma-separated further tags whose frames are compared with the base")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    args.out = args.out or tempfile.mkdtemp(prefix="nrt_bias_mma_ab_")
    extra = [t for t in args.extra.split(",") if t]
    for tag in [args.base, args.new] + extra:
        if not os.path.exists(lib_path(tag)):
            sys.exit("missing %s: build it first (build_native.py with NRT_BUILD_TAG)" % lib_path(tag))
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "steps": args.steps, "warmup": args.warmup, "base": args.base, "new": args.new}

    # outputs: one dump per build, compared with the base build's frame
    frames = {}
    for tag in [args.base, args.new] + extra:
        d = os.path.join(args.out, "dump_" + (tag or "product"))
        run_bench(tag, args, dump=d)
        frames[tag] = np.load(os.path.join(d, "rgb.npy"))
    ref = frames[args.base]
    res["outputs_vs_base"] = {}
    for tag, f in frames.items():
        diff = (f.astype(np.float64) - ref.astype(np.float64))
        res["outputs_vs_base"][tag or "product"] = {
            "bit_identical": bool(np.array_equal(f.view(np.uint32), ref.view(np.uint32))),
            "max_abs": float(np.abs(diff).max()), "rms": float(np.sqrt(np.mean(diff ** 2))),
            "n_differing": int((f != ref).sum())}

    # timing: base and new in alternation
    runs = {args.base: [], args.new: []}
    for p in range(args.pairs):
        for tag in (args.base, args.new):
            runs[tag].append(run_bench(tag, args))
            print("pair %d %-8s %s" % (p, tag or "product", json.dumps(runs[tag][-1])), file=sys.stderr)
    sb, sn = summary(runs[args.base]), summary(runs[args.new])
    res["base_runs"], res["new_runs"] = sb, sn
    res["change"] = {}
    for key in ("ms_per_step",) + KERNELS:
        ch = sn[key]["median"] / sb[key]["median"] - 1.0
        res["change"][key] = {"relative": ch, "larger_than_spread": abs(ch) > max(sb[key]["spread"], sn[key]["spread"])}
    res["gpu_after"] = gpu_info()
    with open(os.path.join(args.out, "ab.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
