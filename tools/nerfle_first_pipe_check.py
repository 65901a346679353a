"""Outputs of NeRFLE.first's inference kernels under two library builds, compared bit for bit (NRT_FIRST_PIPE,
csrc/tc_core.cuh: the change moves work across the tile boundary and must not change a single bit).

    python tools/nerfle_first_pipe_check.py --base fp0 [--new ""] [--out FILE]

Each build (build_native.py with NRT_BUILD_TAG, selected with NRT_LIB_TAG) renders, in a process of its own:
  * the 4K leg of bench.py: 3840 x 2160 rays, one uniform pass of 64 samples, f16;
  * the same 4K frame from its camera (rays generated inside the kernels);
  * a 400 x 400 camera-fed frame with 64 + 128 hierarchical sampling, f16 and bf16;
  * the plain [M, 3] -> [M, 65] forward of NeRFLE.first on 2^20 + 77 points, f16.
Writes a JSON line per output: n_differing, max-abs difference and whether the two builds agree bit for bit."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def render(out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import bench
    from neural_raytracing_b200 import ops
    dev = torch.device("cuda")
    w1, w2 = bench.synthetic_weights(0)

    def to_packed(w):
        Ws = [torch.from_numpy(x).to(dev) for x in w["W"]]
        bs = [torch.from_numpy(x).to(dev) for x in w["b"]]
        return ops.PackedMLP(w["in_size"], 0, w["freqs"], w["hidden"], w["num_layers"], w["skip"], w["out"],
                             ops.ACT_LEAKY_RELU, torch.from_numpy(w["basis"]).to(dev), ops.PackedMLP.pack(Ws, bs))
    m1, m2 = to_packed(w1), to_packed(w2)
    code = torch.tensor([[0.4, 1.0, 0.3]], device=dev)
    ts = torch.linspace(0, 2.05, 64, device=dev)
    res = {}
    base = torch.from_numpy(bench.camera_rays(1080, 0)).to(dev)
    rays4k = base[torch.arange(3840 * 2160, device=dev) % base.shape[0]].contiguous()
    res["render_4k"] = ops.nerfle_render(m1, m2, rays4k, ts, code, prec="f16")
    del rays4k, base
    ops.set_camera_rays_mode(True)      # the camera-fed kernels (IoNerfFirst<64, true>) rather than k_camera_rays
    c2w = torch.from_numpy(bench.camera_matrix(0)).to(dev)
    cam = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=0.5 * 3840 / np.tan(np.radians(30)), size=3840, x0=0, y0=840,
                         nx=3840, ny=2160)
    res["render_4k_camera"] = ops.nerfle_render_camera(m1, m2, cam, ts, code, prec="f16")
    cam = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=0.5 * 400 / np.tan(np.radians(30)), size=400, nx=400, ny=400)
    for prec in ("f16", "bf16"):
        res["camera_hier_" + prec] = ops.nerfle_render_camera(m1, m2, cam, None, code, prec=prec, n_coarse=64, n_fine=128,
                                                              t_near=0.0, t_far=2.05, jitter_seed=5)
    ops.set_camera_rays_mode(False)
    x = (0.8 * torch.randn((1 << 20) + 77, 3, generator=torch.Generator().manual_seed(4))).to(dev)
    res["first_forward_f16"] = ops.mlp_forward(m1, x, prec="f16")
    torch.cuda.synchronize()
    for k, v in res.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default="fp0")
    ap.add_argument("--new", default="")
    ap.add_argument("--out", default=None)
    ap.add_argument("--render-into", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.render_into:
        render(args.render_into)
        return
    tmp = tempfile.mkdtemp(prefix="nrt_first_pipe_")
    dirs = {}
    for tag in (args.base, args.new):
        d = os.path.join(tmp, tag or "product")
        os.makedirs(d, exist_ok=True)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--render-into", d], check=True,
                       env=dict(os.environ, NRT_LIB_TAG=tag), cwd=ROOT)
        dirs[tag] = d
    lines = []
    for f in sorted(os.listdir(dirs[args.base])):
        a = np.load(os.path.join(dirs[args.base], f))
        b = np.load(os.path.join(dirs[args.new], f))
        rec = {"output": f[:-4], "shape": list(a.shape), "base": args.base, "new": args.new or "product",
               "bit_identical": bool(np.array_equal(a.view(np.uint32), b.view(np.uint32))),
               "n_differing": int((a.view(np.uint32) != b.view(np.uint32)).sum()),
               "max_abs": float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max()),
               "finite": bool(np.isfinite(b).all())}
        lines.append(json.dumps(rec))
        print(lines[-1])
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
