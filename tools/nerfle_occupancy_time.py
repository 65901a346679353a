"""Times the occupancy-culled NeRFLE render against the unculled one on a scene with empty space.  NeRFLE.first's density
is fitted (f16 training kernels, random points) to three balls of radius 0.25-0.4 in [-1,1]^3; NeRFLE.second stays random.
Then 800x800 frames from the cfg2 camera (bench.py's camera_matrix(0)), for uniform 64 samples and for 64 + 128
hierarchical samples, without a grid and with a 128^3 grid over [-1.5,1.5]^3 at threshold 0 and 0.01: the kept fraction,
the first / second / cull kernel times per frame (profile tags, a run of their own), the frame time (CUDA events, the
conditions alternating, L2 flushed), and the PSNR of the culled frame against the unculled one.  Also the update time
at 128^3 and 256^3 with 4 points per cell.  The GPU name, power limit and SM clock are read in the same run.  Prints one
JSON object and writes it to --out.

    python tools/nerfle_occupancy_time.py --out profiles/r09_nerfle_occupancy_time.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from neural_raytracing_b200 import config, ops  # noqa: E402
from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE, OccupancyGrid  # noqa: E402

IMG = 800
BALLS = ((-0.45, 0.1, 0.2, 0.4), (0.4, -0.3, -0.1, 0.3), (0.15, 0.45, -0.5, 0.25))   # centre, radius


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:
        return {"name": torch.cuda.get_device_name(), "error": str(e)}


def camera_matrix(view=0):
    """bench.py's cfg2 camera (NeRF convention, -z forward, on the unit sphere looking at the origin)."""
    az, el = 0.7 * view + 0.3, 0.4
    c = np.array([np.cos(el) * np.sin(az), np.sin(el), np.cos(el) * np.cos(az)], np.float64)
    fwd = -c / np.linalg.norm(c)
    right = np.cross(fwd, [0, 1, 0]); right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    m = np.eye(4)
    m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = right, up, -fwd, c
    return m[None].astype(np.float32)


def fit_density(model, steps, batch=65536):
    """sigma_raw -> 10 inside the balls, -1 outside (Adam, f16 training kernels of SkipConnMLP)."""
    opt = torch.optim.Adam(model.first.parameters(), lr=1e-3)
    ctr = torch.tensor([b[:3] for b in BALLS], device="cuda")
    rad = torch.tensor([b[3] for b in BALLS], device="cuda")
    g = torch.Generator("cuda").manual_seed(0)
    loss = None
    for _ in range(steps):
        p = torch.rand(batch, 3, device="cuda", generator=g) * 3.0 - 1.5
        inside = ((p[:, None, :] - ctr[None]).norm(dim=-1) < rad[None]).any(dim=1)
        target = torch.where(inside, 10.0, -1.0)
        loss = ((model.first(p)[:, 0] - target) ** 2).mean()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
    return float(loss.item())


def psnr(a, b):
    mse = float(((a.double() - b.double()) ** 2).mean().item())
    return 200.0 if mse == 0 else -10.0 * math.log10(mse)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--fit-steps", type=int, default=3000)
    ap.add_argument("--reps", type=int, default=6)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    config.precision = "f16"
    torch.manual_seed(0)
    model = NeRFLE(device="cuda")
    loss = fit_density(model, args.fit_steps)
    first, second = model.first.packed(), model.second.packed()
    cam = ops.CameraDesc(ops.CAM_NERF, torch.from_numpy(camera_matrix(0)).cuda(), None,
                         focal=0.5 * IMG / np.tan(np.radians(30)), size=IMG, nx=IMG, ny=IMG)
    code = torch.tensor([[0.4, 1.0, 0.3]], device="cuda")
    samplings = {"uniform64": dict(ts=torch.linspace(0, 2.05, 64, device="cuda")),
                 "hier64_128": dict(ts=None, n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=0x5EED)}
    grids = {}
    for thr in (0.0, 0.01):
        grids[thr] = OccupancyGrid(resolution=128, bbox_min=(-1.5,) * 3, bbox_max=(1.5,) * 3, threshold=thr)
        grids[thr].update(model, points_per_cell=4, decay=0.0, seed=1)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    conds = [("none", None)] + [("grid_thr%g" % t, g) for t, g in grids.items()]

    def frame(kw, grid, counter=None):
        kw = dict(kw)
        ts = kw.pop("ts")
        return ops.nerfle_render_camera(first, second, cam, ts, code, prec="f16", occupancy=grid, samples_done=counter, **kw)

    result = {"gpu": gpu_info(), "scene": {"balls": BALLS, "fit_steps": args.fit_steps, "fit_loss": loss,
                                           "image": [IMG, IMG], "grid": "128^3 over [-1.5,1.5]^3, 4 points per cell, seed 1",
                                           "occupied_fraction": {str(t): g.occupied_fraction() for t, g in grids.items()}},
              "renders": {}}
    for sname, kw in samplings.items():
        S = 64 + (kw.get("n_fine", 0))
        base = frame(kw, None)
        rec = {}
        for cname, g in conds:
            counter = torch.zeros(1, dtype=torch.int64, device="cuda")
            img = frame(kw, g, counter if g is not None else None)
            r = {"kept_fraction": (float(counter.item()) / (IMG * IMG * S)) if g is not None else 1.0,
                 "psnr_vs_unculled_db": psnr(img, base), "max_abs_vs_unculled": float((img - base).abs().max().item())}
            ops.profile_collect(); ops.profile_enable(True)
            for _ in range(3):
                frame(kw, g)
            torch.cuda.synchronize()
            prof = ops.profile_collect(); ops.profile_enable(False)
            for tag in ("mlp_tc_nerf_first", "mlp_tc_nerf_second", "occupancy_cull", "camera_rays", "sample_pdf",
                        "merge_composite", "stratified_ts"):
                if prof.get(tag, (0, 0))[1]:
                    r[tag + "_ms"] = prof[tag][0] / 3
            rec[cname] = r
        # frame times: the conditions alternating, L2 flushed outside the event bracket
        times = {c: [] for c, _ in conds}
        for _ in range(2):
            for _, g in conds:
                frame(kw, g)
        for _ in range(args.reps):
            for cname, g in conds:
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                frame(kw, g)
                b.record()
                torch.cuda.synchronize()
                times[cname].append(a.elapsed_time(b))
        for cname, _ in conds:
            t = sorted(times[cname])
            rec[cname]["frame_ms_median"] = t[len(t) // 2]
            rec[cname]["frame_ms_all"] = times[cname]
        for cname, _ in conds[1:]:
            rec[cname]["speedup_vs_unculled"] = rec["none"]["frame_ms_median"] / rec[cname]["frame_ms_median"]
        result["renders"][sname] = rec
    upd = {}
    for res in (128, 256):
        g = OccupancyGrid(resolution=res, bbox_min=(-1.5,) * 3, bbox_max=(1.5,) * 3, threshold=0.01)
        g.update(model, points_per_cell=4, seed=1)
        ts = []
        for k in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.update(model, points_per_cell=4, seed=2 + k)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        upd["%d^3" % res] = {"ms_median": sorted(ts)[2], "ms_all": ts, "points": res ** 3 * 4}
    result["update"] = upd
    result["gpu_after"] = gpu_info()
    s = json.dumps(result, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
