#!/usr/bin/env python
"""Benchmark of the B200-native neural_raytracing hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision f16|bf16|f32]
                    [--dump-outputs DIR]

Workload at N = 1 (BASELINE.json configs[1]): nerf_synthetic-shape NeRF volumetric render, 800x800 rays,
64 coarse + 128 importance-resampled fine samples per ray, random-init NeRFLE-architecture MLPs
(pytorch3d/pathtracer/shapes/nerf.py:153-214), forward only.  One "step" = one full frame.

Workload at N > 1 (BASELINE.json configs[4], the multi-GPU configuration): the 65,536-ray nerfle.py-style
training step (4 views x 128x128 rays, S = 64: forward + backward + AdamW) under STRONG scaling -- rank g
takes 65,536/N rays, the MLP weight gradients are all-reduced with NCCL on ONE flat buffer -- with the
ray-sharded 4K (3840x2160) render as the second number.  The same step is also timed on rank 0 alone in
the same run (`single_gpu_same_run`), and N-rank gradients / images are checked against the 1-rank ones.

Prints ONE JSON line (rank 0):
  value      rays/s, whole job, inputs resident in HBM, CUDA-event timed (max over ranks)
  e2e        same through the public host-buffer entry point (pinned rays H2D + rgb D2H inside)
  roofline   dominant kernel (tcgen05 fused first MLP): algorithmic FLOP / event-timed duration
             against the measured bf16 peak in MEASURED_PEAKS.json
  cpu_baseline  the reference's eager-PyTorch op sequence re-stated in oracle/port.py, timed on
             the host cores on a bounded sample of the same workload (rank 0, N=1 only)

`--impl reference` times only that CPU restatement (the reference is pure Python/PyTorch and does
not exist on the GPU box; oracle/ is its pinned restatement) and prints the same line shape.

`--steps K` is the number of timed steps behind `value` and `ms_per_step`.  The secondary legs pick their own counts:
`e2e` (and `e2e.from_camera`) times max(3, min(K, 10)) steps; at N > 1 the eager per-kernel split and
`single_gpu_same_run` time max(3, K // 2) steps; the configs under `also` and the 4K render have fixed counts.

`--dump-outputs DIR` writes what the last timed step computed, float32, once per run:
  N = 1   rgb.npy     the radiance of the frame, [640000, 3]
  N > 1   loss.npy    the loss of rank 0's slice; grad.npy the all-reduced flat gradient and params.npy the flat
                      parameters after the AdamW update (both in the layout of training.FlatParameters)
The inputs are fixed by seeds, so two builds run with the same arguments can be compared output for output: the
render is reproducible bit for bit; the training step's weight gradients are accumulated with atomics, so its outputs
agree from run to run only to the order of fp32 summation (about 1e-3 of the largest element).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
# version banner there at the first collective, whatever NCCL_DEBUG says on this image), so descriptor 1 is pointed at
# stderr for the whole run and the result line goes to a private duplicate of the original stdout.
_RESULT_FD = os.dup(1)
os.dup2(2, 1)
sys.stdout = sys.stderr


def emit_result(line: dict):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


import numpy as np  # noqa: E402

IMG = 800
N_COARSE, N_FINE = 64, 128
T_NEAR, T_FAR = 0.0, 2.05
JITTER_SEED = 7
# algorithmic FLOP per MLP sample = 2 * MAC of the Linear layers (SURVEY.md section 8d)
FLOP_FIRST, FLOP_SECOND = 2 * 103680, 2 * 59072
CPU_SAMPLE_RAYS = 4096
# cfg5 (BASELINE.json configs[4]): nerfle.py-style training step, 4 views x 128x128 rays, S = 64
TRAIN_RAYS, TRAIN_VIEWS, TRAIN_S = 65536, 4, 64
CPU_TRAIN_SAMPLE_RAYS = 1024
# algorithmic bytes the weight-gradient kernel reads per sample: 2 B x (fan-in + fan-out) of every Linear (both MLPs)
WGRAD_BYTES_PER_SAMPLE = 2 * (1706 + 1563)


def synthetic_weights(seed):
    """Random-init weights with nn.Linear's default distribution U(-1/sqrt(K), 1/sqrt(K)) for the
    NeRFLE architecture (first: 3->65, 5x128; second: 70->3, 8x64; sigma=32, 16 frequencies)."""
    def mlp(seed, in_size, out, num_layers, hidden, freqs, sigma, skip=3):
        rs = np.random.RandomState(seed)
        basis = (sigma * rs.standard_normal((freqs, in_size))).astype(np.float32).T.copy()
        dim_p = in_size + 2 * freqs
        shapes = [(hidden, dim_p)]
        for i in range(num_layers):
            sk = (i % skip) == 0 and i != num_layers - 1
            shapes.append((hidden, hidden + (dim_p if sk else 0)))
        shapes.append((out, hidden))
        W = [rs.uniform(-1 / np.sqrt(k), 1 / np.sqrt(k), size=(n, k)).astype(np.float32) for n, k in shapes]
        b = [rs.uniform(-1 / np.sqrt(k), 1 / np.sqrt(k), size=(n,)).astype(np.float32) for n, k in shapes]
        return dict(in_size=in_size, out=out, num_layers=num_layers, hidden=hidden, freqs=freqs, latent=0,
                    skip=skip, basis=basis, W=W, b=b)
    w1 = mlp(seed, 3, 65, 5, 128, 16, 32.0)
    w2 = mlp(seed + 1, 70, 3, 8, 64, 16, 32.0)
    w1["b"][-1][0] = 0.5   # non-trivial densities
    return w1, w2


def camera_rays(size, view):
    """Pinhole camera on the unit sphere looking at the origin (fov 60 deg), one ray per pixel."""
    az = 0.7 * view + 0.3
    el = 0.4
    c = np.array([np.cos(el) * np.sin(az), np.sin(el), np.cos(el) * np.cos(az)], np.float64)
    fwd = -c / np.linalg.norm(c)
    right = np.cross(fwd, [0, 1, 0]); right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    u = (np.arange(size) + 0.5) / size * 2 - 1
    xx, yy = np.meshgrid(u, u, indexing="ij")
    t = np.tan(np.radians(30))
    d = fwd[None, None] + t * xx[..., None] * right[None, None] + t * yy[..., None] * up[None, None]
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    o = np.broadcast_to(c, d.shape)
    return np.concatenate([o, d], -1).reshape(-1, 6).astype(np.float32)


def camera_matrix(view):
    """cam_to_world [1,4,4] (NeRF convention, -z forward) of the camera camera_rays() looks through."""
    az = 0.7 * view + 0.3
    el = 0.4
    c = np.array([np.cos(el) * np.sin(az), np.sin(el), np.cos(el) * np.cos(az)], np.float64)
    fwd = -c / np.linalg.norm(c)
    right = np.cross(fwd, [0, 1, 0]); right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    m = np.eye(4)
    m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = right, up, -fwd, c
    return m[None].astype(np.float32)


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = None
        self.p = None

    def start(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        try:
            self.p.terminate(); self.p.wait(timeout=5)
            self.f.flush(); self.f.seek(0)
            sm, mx, reasons = [], [], set()
            for line in self.f.read().strip().splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); mx.append(float(c[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            if sm:
                busy = [s for s in sm if s >= 0.5 * max(sm)] or sm
                out = {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                       "samples": len(sm)}
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.f.name)
            except Exception:
                pass
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1384.0), d.get("hbm_gbs", 6532.5), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def cpu_reference_rate(w1, w2, rays, steps, warmup):
    """rays/s of the reference's eager op sequence (oracle/port.py) on the host cores."""
    import torch
    from oracle import port
    code = np.array([[0.4, 1.0, 0.3]], np.float32)
    torch.set_num_threads(os.cpu_count() or 1)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        port.torch_nerfle_render(w1, w2, rays, code, N_COARSE, N_FINE, T_NEAR, T_FAR, seed=JITTER_SEED)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    return rays.shape[0] / (ms / 1e3), ms, torch.get_num_threads()


def run_reference(args, rank, world=1):
    """The reference's own CPU implementation of the path (it is eager PyTorch: oracle/port.py re-states its op
    sequence; /root/reference does not exist on the GPU box) on the host cores, on this arm's config / metric / unit.
    Under torchrun rank 0 alone runs it."""
    if rank != 0:
        return
    if max(world, args.gpus) > 1:
        return run_reference_train(args, max(world, args.gpus))
    w1, w2 = synthetic_weights(0)
    rays = camera_rays(IMG, 0)
    sel = np.linspace(0, rays.shape[0] - 1, CPU_SAMPLE_RAYS).astype(np.int64)
    rate, ms, threads = cpu_reference_rate(w1, w2, rays[sel], args.steps, args.warmup)
    sample = "%d of the %d rays of the frame (evenly strided), full 64+128 samples/ray, per step" % (CPU_SAMPLE_RAYS, IMG * IMG)
    line = {
        "impl": "reference", "metric": "rays_per_sec", "value": rate, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "mlp_samples_per_sec": rate * (N_COARSE + N_FINE),
        "config": workload_config("f16"),
        "arithmetic": "f32 (CPU, eager PyTorch op sequence)",
        "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_result(line)


def run_reference_train(args, world):
    """CPU arm of the N > 1 workload (cfg5 training step): the reference's eager step (oracle/port.py::TorchNerfleTrainer)
    on a bounded sample of the batch, all host threads."""
    import torch
    from oracle import port
    torch.set_num_threads(os.cpu_count() or 1)
    w1, w2 = synthetic_weights(0)
    w1["b"][-1][0] = 0.5
    tr = port.TorchNerfleTrainer(w1, w2)
    per = CPU_TRAIN_SAMPLE_RAYS // TRAIN_VIEWS
    all_rays = train_rays_np()
    sel = np.linspace(0, all_rays.shape[1] - 1, per).astype(np.int64)
    rays = torch.from_numpy(all_rays[:, sel].copy())
    ts = torch.linspace(0, 2.05, TRAIN_S)
    loc = torch.from_numpy(TRAIN_LIGHTS.copy())
    target = torch.full((TRAIN_VIEWS, per, 3), 0.5)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        tr.step(rays, ts, loc, target, CPU_TRAIN_SAMPLE_RAYS * 3)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    ms = 1e3 * sum(times) / len(times)
    rate = CPU_TRAIN_SAMPLE_RAYS / (ms / 1e3)
    sample = "%d of the %d rays of the batch (%d evenly strided rays of each view), S = %d, forward + backward + AdamW per step" % (
        CPU_TRAIN_SAMPLE_RAYS, TRAIN_RAYS, per, TRAIN_S)
    emit_result({
        "impl": "reference", "metric": "train_rays_per_sec", "value": rate, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "mlp_samples_per_sec": rate * TRAIN_S,
        "config": train_workload_config("f16 operands / fp32 accumulate (tcgen05 training kernels)", world),
        "arithmetic": "f32 (CPU, eager PyTorch op sequence + autograd)",
        "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def workload_config(precision):
    return {"workload": "cfg2 nerf_synthetic-shape NeRF volumetric render %dx%d, %d coarse + %d fine samples/ray, "
                        "NeRFLE MLPs (3->65 5x128, 70->3 8x64), random init, forward only" % (IMG, IMG, N_COARSE, N_FINE),
            "rays_per_step_per_gpu": IMG * IMG, "samples_per_ray": N_COARSE + N_FINE, "precision": precision,
            "l2": "flushed (256 MiB memset) between timed iterations; per-step intermediates (>1 GB) exceed L2",
            "sharding": "one frame per rank, no data-path collective"}


NO_CPU = [False]


def supplementary(dev, rank, world, steps=5, warmup=3):
    """Other BASELINE.json configs, measured after the headline run (reported under "also"; never part of `value`).
      cfg5_train: nerfle.py-style training step on 65,536 rays IN TOTAL (strong scaling: rank g takes 65,536/N rays),
                  S = 64, mse, AdamW, tensor-core training kernels (fp16 operands), ONE flat NCCL all-reduce of the
                  164,164 MLP gradients per step;
      cfg3_train: the same step at 4,096 rays (N = 1 only);
      cfg1_sdf_march: sphere-trace + min-along-ray scan of a random-init SphereSDF (64 spheres + 8x128 softplus MLP),
                  512x512 rays, max_steps 64, tensor-core march (N = 1 only)."""
    import random
    import torch
    import torch.distributed as dist
    from neural_raytracing_b200 import config, distributed as D, ops
    from neural_raytracing_b200.pathtracer.lights import PointLights
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    from neural_raytracing_b200.pathtracer.shapes.sdfs import SDF, SphereSDF
    out = {}
    peak_tf, peak_gbs, peak_src = measured_peaks()

    def roof(kernel, bound, work, ms, note=None):
        """roofline entry of a supplementary config's dominant kernel: work = algorithmic TFLOP (tensor) or GB (hbm) done in
        `ms` milliseconds of that kernel's CUDA-event time"""
        if not ms or ms <= 0:
            return None
        ach = work / (ms * 1e-3)
        peak = peak_tf if bound == "tensor" else peak_gbs
        r = {"kernel": kernel, "bound": bound, "achieved": ach, "peak": peak, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
             "frac": ach / peak, "peak_source": peak_src, "kernel_ms": ms}
        if note:
            r["algorithmic_work"] = note
        return r

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def train_bench(total_rays, side):
        torch.manual_seed(1)
        net = NeRFLE(device=dev)
        with torch.no_grad():
            net.first.out.bias[0] = 0.5
        opt = torch.optim.AdamW(net.parameters(), lr=8e-5, weight_decay=0)
        rays_all = torch.from_numpy(camera_rays(side, 0)).to(dev)
        lo, hi = D.shard_range(total_rays, rank, world)
        rays = rays_all[lo:hi].reshape(1, hi - lo, 1, 1, 6).contiguous()
        lights = PointLights(device=dev, location=torch.tensor([[0.4, 1.0, 0.3]], device=dev), scale=10)
        target = torch.full((1, hi - lo, 1, 1, 3), 0.5, device=dev)
        ar = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]

        def one(i=None):
            random.seed(0)
            opt.zero_grad(set_to_none=True)
            loss = (net(rays, lights) - target).square().sum() / (total_rays * 3)
            loss.backward()
            if i is not None:
                ar[i][0].record()
            D.allreduce_gradients(net.parameters(), average=False)
            if i is not None:
                ar[i][1].record()
            opt.step()
            return loss.detach()     # do not keep the autograd graph (and its 28 GB of saved tiles) alive across steps
        for _ in range(warmup):
            one()
        sync()
        ops.profile_collect(); ops.profile_enable(True)
        for i, (a, b) in enumerate(ev):
            a.record(); loss = one(i); b.record()
        sync()
        prof = ops.profile_collect(); ops.profile_enable(False)
        ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) / steps)
        ar_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ar) / steps)
        loss_val = float(loss)
        del loss
        wg_ms = prof.get("mlp_tc_wgrad", (0.0, 0))[0] / steps
        return {"ms_per_step": ms, "rays_per_sec": total_rays / ms * 1e3, "mlp_samples_per_sec": total_rays * 64 / ms * 1e3,
                "roofline": roof("k_mlp_wgrad_tc (tcgen05; the saved 16-bit activation / gradient tiles read once)", "hbm",
                                 (hi - lo) * 64 * WGRAD_BYTES_PER_SAMPLE / 1e9, wg_ms,
                                 "%d samples x %d B of saved tiles" % ((hi - lo) * 64, WGRAD_BYTES_PER_SAMPLE)),

                "model_tflops_fwd_bwd": total_rays * 64 * (FLOP_FIRST + FLOP_SECOND) * 3 / ms / 1e9,
                "grad_allreduce_ms": ar_ms, "grad_bucket_bytes": 4 * sum(p.numel() for p in net.parameters()),
                "kernel_ms_per_step": {k: round(v[0] / steps, 3) for k, v in prof.items() if v[1]},
                "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1),
                "loss": loss_val, "scaling": "strong", "train_precision": config.train_precision}

    def graph_bench(total_rays, side):
        """The same step captured in CUDA graphs (training.GraphedStep): zero_grad + forward + backward | all-reduce | AdamW."""
        import gc
        from neural_raytracing_b200.training import GraphedStep
        gc.collect()
        torch.manual_seed(1)
        net = NeRFLE(device=dev)
        with torch.no_grad():
            net.first.out.bias[0] = 0.5
        net.far_jitter = torch.full((1,), 0.5, device=dev)
        opt_g = torch.optim.AdamW(net.parameters(), lr=8e-5, weight_decay=0, capturable=True)
        rays_all = torch.from_numpy(camera_rays(side, 0)).to(dev)
        lo, hi = D.shard_range(total_rays, rank, world)
        rays = rays_all[lo:hi].reshape(1, hi - lo, 1, 1, 6).contiguous()
        lights = PointLights(device=dev, location=torch.tensor([[0.4, 1.0, 0.3]], device=dev), scale=10)
        target = torch.full((1, hi - lo, 1, 1, 3), 0.5, device=dev)
        gstep = GraphedStep(lambda: (net(rays, lights) - target).square().sum() / (total_rays * 3), opt_g, modules=[net],
                            allreduce=(lambda: D.allreduce_gradients(net.parameters(), average=False)) if world > 1 else None)
        for _ in range(2):
            gstep()
        sync()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(steps):
            gstep()
        g1.record()
        sync()
        ms = max_over_ranks(g0.elapsed_time(g1) / steps)
        return {"ms_per_step": ms, "rays_per_sec": total_rays / ms * 1e3, "loss": float(gstep.loss.detach())}

    prev = config.train_precision
    try:
        config.set_train_precision("f16")
        try:
            out["cfg5_train_65536rays"] = train_bench(65536, 256)
        except Exception as e:   # noqa: BLE001 -- supplementary numbers must never break the headline line
            out["cfg5_train_65536rays"] = {"error": repr(e)[:300]}
        if world == 1:
            try:
                out["cfg3_train_4096rays"] = train_bench(4096, 64)
            except Exception as e:   # noqa: BLE001
                out["cfg3_train_4096rays"] = {"error": repr(e)[:300]}
    finally:
        config.set_train_precision(prev)
    if world == 1:
        try:
            torch.manual_seed(2)
            sphere = SphereSDF(n=64, device=dev)
            with torch.no_grad():
                for q in sphere.shift.parameters():
                    q.normal_(0, 0.02)   # the reference zero-initialises the residual MLP (sdfs.py:30): perturb it
                sphere.shift.out.weight.mul_(0.1); sphere.shift.out.bias.zero_()   # residual of a few mm, like a trained SDF
                sphere.radii.abs_().add_(0.05)   # sdfs.py:20 draws radii in [-0.1, 0.1]: make the object visible
            shape = SDF(device=dev, sdf=sphere, max_steps=64)
            packed = sphere.packed()
            rays = torch.from_numpy(camera_rays(512, 0)).to(dev)
            R = rays.shape[0]
            res = {}
            for prec in ("f16", "f32"):
                cnt = torch.zeros(1, dtype=torch.int64, device=dev)
                def fn():
                    d, h = ops.sphere_trace(packed, rays, shape.epsilon, 64, 10.0, prec=prec, steps_counter=cnt)
                    ops.min_scan(packed, rays, 2.2 / 128, 128, prec=prec)
                    return h
                fn(); torch.cuda.synchronize(); cnt.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); h = fn(); b.record(); torch.cuda.synchronize()
                ms = a.elapsed_time(b)
                evals = int(cnt.item()) + R * 129
                res[prec] = {"ms": ms, "rays_per_sec": R / ms * 1e3, "sdf_samples_per_sec": evals / ms * 1e3,
                             "tflops": evals * 331008 / ms / 1e9, "hit_fraction": float(h.float().mean())}
            res["roofline"] = roof("k_mlp_tc<SphereSDF.shift 8x128 softplus; IoMarch + IoScanEval> (tcgen05, weights streamed)", "tensor",
                                   res["f16"]["tflops"] * res["f16"]["ms"] * 1e-3, res["f16"]["ms"],
                                   "live march evaluations + 129 scan evaluations per ray, 331,008 FLOP each")
            out["cfg1_sdf_march_512x512"] = res
            # the same at cfg1's NAMED size (64x64 = 4,096 rays), next to the CPU: the reference's lock-step march (64
            # evaluations of every ray) + scan (129) on the host cores (oracle/port.py, the reference's eager op sequence)
            rays64 = torch.from_numpy(camera_rays(64, 0)).to(dev)
            r64 = {}
            for prec in ("f16", "f32"):
                def fn64():
                    ops.sphere_trace(packed, rays64, shape.epsilon, 64, 10.0, prec=prec)
                    ops.min_scan(packed, rays64, 2.2 / 128, 128, prec=prec)
                fn64(); torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(5):
                    fn64()
                b.record(); torch.cuda.synchronize()
                r64[prec] = {"ms": a.elapsed_time(b) / 5, "rays_per_sec": 4096 / (a.elapsed_time(b) / 5) * 1e3}
            if rank == 0 and not NO_CPU[0]:
                from oracle import port
                lin = [sphere.shift.init] + list(sphere.shift.layers) + [sphere.shift.out]
                wcpu = {"centers": sphere.centers.detach().cpu().numpy(), "radii": sphere.radii.detach().cpu().numpy(),
                        "tfs": sphere.tfs.detach().cpu().numpy(),
                        "shift": {"basis": sphere.shift.basis_p.detach().cpu().numpy(), "num_layers": len(sphere.shift.layers),
                                  "skip": sphere.shift.skip, "W": [l.weight.detach().cpu().numpy() for l in lin],
                                  "b": [l.bias.detach().cpu().numpy() for l in lin]}}
                r_cpu = rays64.cpu().numpy()
                port.torch_sdf_march_and_scan(wcpu, r_cpu[:256])     # warm-up
                t0 = time.perf_counter()
                _d, h_cpu, _i = port.torch_sdf_march_and_scan(wcpu, r_cpu)
                cpu_ms = (time.perf_counter() - t0) * 1e3
                d_gpu, h_gpu = ops.sphere_trace(packed, rays64, shape.epsilon, 64, 10.0, prec="f32")
                r64["cpu_port"] = {"ms": cpu_ms, "rays_per_sec": 4096 / cpu_ms * 1e3, "cores": torch.get_num_threads(), "kind": "port",
                                   "sample": "the whole 64x64 frame: 64 lock-step march + 129 scan evaluations of every ray (193 of the "
                                             "~200 network evaluations per ray of the colocate pipeline), torch CPU, all host threads",
                                   "hit_mask_xor_vs_gpu_f32": int((h_cpu.numpy() ^ h_gpu.cpu().numpy().astype(bool)).sum())}
            out["cfg1_sdf_march_64x64"] = r64
        except Exception as e:   # noqa: BLE001
            out["cfg1_sdf_march_512x512"] = {"error": repr(e)[:300]}
    # cfg1: the whole colocate.py-style pipeline through the drop-in pathtrace() (sphere-trace + normals + 2 NeuralBSDF +
    # diffuse + conductor mixed by the 16x256 sp_var MLP, point light, learned-occlusion MLP + shadow march, silhouette
    # scan), 512x512 rays in one chunk, forward, tensor-core precision vs the exact fp32 kernels
    if world == 1:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import scenes
            import synth
            import neural_raytracing_b200.pathtracer as P
            from neural_raytracing_b200.pathtracer.cameras import NeRFCamera
            shape_c, _sph, bsdf_c, lights_c, integ_c, w_isect = scenes.build_pipeline(P, "colocate", device=dev)
            c2w, focal = synth.nerf_cameras(1, 512, device=dev)
            cam = NeRFCamera(cam_to_world=c2w, focal=focal, device=dev)
            res = {}
            prev_p = config.precision
            for prec in ("f16", "f32"):
                config.set_precision(prec)

                def frame():
                    with torch.no_grad():
                        return P.pathtrace(shape_c, size=512, chunk_size=512, bundle_size=1, bsdf=bsdf_c, integrator=integ_c,
                                           lights=lights_c, cameras=cam, device=dev, silent=True, background=0, w_isect=w_isect,
                                           with_noise=False)
                frame(); frame()
                torch.cuda.synchronize()
                ops.profile_collect(); ops.profile_enable(True)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n_it = 3 if prec == "f16" else 1
                a.record()
                for _ in range(n_it):
                    img = frame()
                b.record(); torch.cuda.synchronize()
                pr = ops.profile_collect(); ops.profile_enable(False)
                ms = a.elapsed_time(b) / n_it
                res[prec] = {"ms_per_frame": ms, "rays_per_sec": 512 * 512 / ms * 1e3,
                             "kernel_ms_per_frame": {k: round(v[0] / n_it, 3) for k, v in pr.items() if v[1]},
                             "library_launches_per_frame": sum(v[1] for v in pr.values()) // n_it}
                if prec == "f16":
                    res["roofline"] = roof("k_mlp_tc<SphereSDF.shift; IoScanEval> (min-along-ray scan, tcgen05)", "tensor",
                                           512 * 512 * 129 * 331008 / 1e12, pr.get("sdf_min_scan_tc", (0.0, 0))[0] / n_it,
                                           "262,144 rays x 129 evaluations x 331,008 FLOP")
            config.set_precision(prev_p)
            out["cfg1_colocate_pipeline_512x512"] = res
        except Exception as e:   # noqa: BLE001
            out["cfg1_colocate_pipeline_512x512"] = {"error": repr(e)[:300]}
    # cfg2b: the pipeline nerf_synthetic.py itself builds (nerf_synthetic.py:61-75): SDF(SphereSDF(n=128), max_steps=64) +
    # Direct + LightField + ComposeSpatialVarying of 8 NeuralBSDF(Softplus), NeRFCamera, 800x800 rays, forward
    if world == 1:
        try:
            import torch.nn as nn
            import synth
            import neural_raytracing_b200.pathtracer as P
            from neural_raytracing_b200.pathtracer.cameras import NeRFCamera
            torch.manual_seed(3)
            sph = SphereSDF(n=128, device=dev)
            with torch.no_grad():
                for q in sph.shift.parameters():
                    q.normal_(0, 0.02)
                sph.shift.out.weight.mul_(0.1); sph.shift.out.bias.zero_()
                sph.radii.abs_().add_(0.05)
            shp = SDF(device=dev, sdf=sph, max_steps=64)
            kids = [P.bsdf.NeuralBSDF(activation=nn.Softplus(), device=dev) for _ in range(8)]
            bsdf8 = P.bsdf.ComposeSpatialVarying(kids, device=dev)
            lf = P.lights.LightField(device=dev)
            with torch.no_grad():
                lf.light_field_approx.out.bias.add_(0.5)
            c2w, focal = synth.nerf_cameras(1, 800, device=dev)
            cam8 = NeRFCamera(cam_to_world=c2w, focal=focal, device=dev)
            res = {}
            prev_p = config.precision
            for prec in ("f16", "f32"):
                config.set_precision(prec)

                def frame8():
                    with torch.no_grad():
                        return P.pathtrace(shp, size=800, chunk_size=800, bundle_size=1, bsdf=bsdf8, integrator=P.integrators.Direct(),
                                           lights=lf, cameras=cam8, device=dev, silent=True, background=0, with_noise=False)
                # median of five frames after two warm-ups (one for the 2 s fp32 frame): a single frame right after the other
                # configs' allocations measured anything between 111 and 158 ms for a frame that takes 80 ms in steady state
                n_warm, n_timed = (2, 5) if prec == "f16" else (1, 1)
                for _ in range(n_warm):
                    frame8()
                torch.cuda.synchronize()
                times = []
                for _ in range(n_timed):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); img8, _ = frame8(); b.record(); torch.cuda.synchronize()
                    times.append(a.elapsed_time(b))
                ms = sorted(times)[len(times) // 2]
                res[prec] = {"ms_per_frame": ms, "frames_ms": [round(t, 2) for t in times], "rays_per_sec": 800 * 800 / ms * 1e3,
                             "finite": bool(torch.isfinite(img8).all()),
                             "lit_fraction": float((img8.abs().sum(-1) > 0).float().mean())}
            config.set_precision(prev_p)
            out["cfg2b_nerf_synthetic_pipeline_800x800"] = res
        except Exception as e:   # noqa: BLE001
            out["cfg2b_nerf_synthetic_pipeline_800x800"] = {"error": repr(e)[:300]}
    # cfg4 (BASELINE.json configs[3]) at its NAMED size and model: dtu.py's scene (dtu.py:93-108: SDF(SphereSDF(n=64), 64 steps),
    # ComposeSpatialVarying of 10 NeuralBSDF + 6 Diffuse under the 16-way 16x256 sp_var MLP, LightField, NeRFIntegrator(Direct),
    # DTUCamera) trained on ONE 1600x1200 image = 1,920,000 rays per step, rendered as 12 crops of 400x400 through
    # pathtrace_sample (gradients accumulate over the crops), masked_loss (no SSIM) + eikonal_loss on the analytic normals,
    # ONE fused AdamW step on the flat parameter buffer.  Tensor-core inference AND training kernels (f16).
    if world == 1:
        try:
            if os.path.join(ROOT, "tests", "golden") not in sys.path:
                sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import scenes
            import neural_raytracing_b200.pathtracer as P
            from neural_raytracing_b200 import training
            from neural_raytracing_b200.pathtracer.cameras import DTUCamera
            from neural_raytracing_b200.pathtracer.utils import eikonal_loss, masked_loss
            prev_p, prev_t = config.precision, config.train_precision
            config.set_precision("f16"); config.set_train_precision("f16")
            random.seed(0)
            torch.manual_seed(4)
            shape_d, sphere_d, bsdf_d, lights_d, integ_d = scenes.build_dtu16(P, device=dev)
            mlps = [sphere_d.shift, bsdf_d.sp_var_fn, lights_d.light_field_approx] + [k.mlp for k in bsdf_d.bsdfs if hasattr(k, "mlp")]
            mlp_params = {id(q) for m in mlps for q in m.parameters()}
            others = [q for q in list(sphere_d.parameters()) + list(bsdf_d.parameters()) + list(lights_d.parameters())
                      if id(q) not in mlp_params]
            flat = training.FlatParameters(mlps, others)
            opt_d = torch.optim.AdamW([flat.param], lr=8e-5, weight_decay=0, fused=True)
            pose, Kmat = scenes.dtu_cameras(1, device=dev)
            cam_d = DTUCamera(pose=pose, intrinsic=Kmat, device=dev)
            CROP, NX, NY = 400, 4, 3
            exp_d, mask_d = scenes.dtu_targets(1, CROP, device=dev)
            hits = [0]

            def dtu_step():
                flat.zero_grad()
                tot = 0.0
                for cx in range(NX):
                    for cy in range(NY):
                        got, mi = P.pathtrace_sample(shape_d, size=1600, chunk_size=CROP, bundle_size=1, crop_size=CROP, bsdf=bsdf_d,
                                                     integrator=integ_d, cameras=cam_d, lights=lights_d, device=dev,
                                                     uv=(cx * CROP, cy * CROP), background=0, addition=lambda mi: mi,
                                                     squeeze_first=False, silent=True)
                        loss = masked_loss(got[..., :3], exp_d, mi.throughput.squeeze(-1), mask_d, mask_weight=10,
                                           with_logits=mi.with_logits, ssim_fn=None) / (NX * NY)
                        if hasattr(mi, "raw_normals"):
                            loss = loss + eikonal_loss(mi.raw_normals) / (NX * NY)
                            hits[0] += mi.raw_normals.shape[0]
                        loss.backward()
                        tot = tot + loss.detach()
                opt_d.step()
                return tot
            dtu_step()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            hits[0] = 0
            ops.profile_collect(); ops.profile_enable(True)
            n_it = 2
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record()
            for _ in range(n_it):
                l_d = dtu_step()
            b.record(); torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3 / n_it
            pr = ops.profile_collect(); ops.profile_enable(False)
            ms = a.elapsed_time(b) / n_it
            rays_d = CROP * CROP * NX * NY
            kms = {k: round(v[0] / n_it, 3) for k, v in pr.items() if v[1]}
            out["cfg4_dtu_step_1600x1200"] = {
                "ms_per_step": ms, "wall_ms_per_step": wall, "rays_per_sec": rays_d / ms * 1e3, "rays_per_step": rays_d,
                "hit_fraction": hits[0] / n_it / rays_d, "crops": "%d x %d crops of %dx%d" % (NX, NY, CROP, CROP),
                "loss": float(l_d), "finite": bool(torch.isfinite(flat.grad).all()), "parameters": int(flat.flat.numel()),
                "kernel_ms_per_step": kms, "library_launches_per_step": sum(v[1] for v in pr.values()) // n_it,
                "library_kernel_ms_per_step": round(sum(kms.values()), 2),
                "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1),
                "precision": "f16 operands / fp32 accumulate: march, min scan, training forward, dgrad, wgrad of every network on "
                             "tcgen05, incl. the normals (value + Jacobian of SphereSDF.shift and its reverse pass); the sphere set "
                             "and the shading stages in fp32",
                "roofline": roof("k_mlp_tc<SphereSDF.shift; IoScanEval> (min-along-ray scan of SDF.throughput, tcgen05)", "tensor",
                                 rays_d * 129 * 331008 / 1e12, pr.get("sdf_min_scan_tc", (0.0, 0))[0] / n_it,
                                 "1,920,000 rays x 129 evaluations x 331,008 FLOP")}
            config.set_precision(prev_p); config.set_train_precision(prev_t)
            del flat, opt_d, shape_d, sphere_d, bsdf_d, lights_d
            torch.cuda.empty_cache()
        except Exception as e:   # noqa: BLE001
            out["cfg4_dtu_step_1600x1200"] = {"error": repr(e)[:400]}
            config.set_precision("f32"); config.set_train_precision("f32")
    # cfg5 (i): ray-sharded 4K render (3840x2160 = 8,294,400 rays, the reference's single uniform pass of 64 samples,
    # nerf.py:175-214) on the tensor-core kernels: rank g renders its contiguous slice, no data-path collective
    try:
        w1, w2 = synthetic_weights(0)

        def to_packed(w):
            Ws = [torch.from_numpy(x).to(dev) for x in w["W"]]
            bs = [torch.from_numpy(x).to(dev) for x in w["b"]]
            return ops.PackedMLP(w["in_size"], 0, w["freqs"], w["hidden"], w["num_layers"], w["skip"], w["out"],
                                 ops.ACT_LEAKY_RELU, torch.from_numpy(w["basis"]).to(dev), ops.PackedMLP.pack(Ws, bs))
        m1, m2 = to_packed(w1), to_packed(w2)
        total = 3840 * 2160
        lo, hi = D.shard_range(total, rank, world)
        base = torch.from_numpy(camera_rays(1080, 0)).to(dev)                 # 1,166,400 distinct rays, tiled to the slice
        rays4k = base.repeat((hi - lo + base.shape[0] - 1) // base.shape[0], 1)[: hi - lo].contiguous()
        ts = torch.linspace(0, 2.05, 64, device=dev)
        code = torch.tensor([[0.4, 1.0, 0.3]], device=dev)
        ops.nerfle_render(m1, m2, rays4k, ts, code, prec="f16")
        sync()
        ops.profile_collect(); ops.profile_enable(True)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        img = ops.nerfle_render(m1, m2, rays4k, ts, code, prec="f16")
        b.record()
        sync()
        prof4k = ops.profile_collect(); ops.profile_enable(False)
        ms = max_over_ranks(a.elapsed_time(b))
        out["cfg5_render_4k_64samples"] = {"ms_per_frame": ms, "rays_per_sec": total / ms * 1e3, "mlp_samples_per_sec": total * 64 / ms * 1e3,
                                           "model_tflops": total * 64 * (FLOP_FIRST + FLOP_SECOND) / ms / 1e9, "scaling": "strong",
                                           "finite": bool(torch.isfinite(img).all()),
                                           "kernel_ms": {k: round(v[0], 3) for k, v in prof4k.items() if v[1]},
                                           "roofline": roof("k_mlp_tc<NeRFLE.first> (tcgen05)", "tensor", (hi - lo) * 64 * FLOP_FIRST / 1e12,
                                                            prof4k.get("mlp_tc_nerf_first", (0.0, 0))[0],
                                                            "%d samples x %d FLOP (this rank's slice)" % ((hi - lo) * 64, FLOP_FIRST))}
        del rays4k, img, base
    except Exception as e:   # noqa: BLE001
        out["cfg5_render_4k_64samples"] = {"error": repr(e)[:300]}
    # CUDA-graph captured steps last: a failed capture must not disturb the measurements above
    try:
        config.set_train_precision("f16")
        for name, total, side in (("cfg5_train_65536rays", 65536, 256),) + ((("cfg3_train_4096rays", 4096, 64),) if world == 1 else ()):
            try:
                out[name]["cuda_graph"] = graph_bench(total, side)
            except Exception as e:   # noqa: BLE001
                out[name]["cuda_graph"] = {"error": repr(e)[:300]}
                break
    finally:
        config.set_train_precision(prev)
    return out


# ---------------------------------------------------------------------------------------------------------------
# cfg5 (BASELINE.json configs[4]): the multi-GPU configuration
# ---------------------------------------------------------------------------------------------------------------
def train_workload_config(precision, world):
    return {"workload": "cfg5 (BASELINE.json configs[4]) nerfle.py-style NeRF+PT training step, %d rays in total (%d views x "
                        "128x128), S = %d, forward + backward + AdamW, NeRFLE MLPs (3->65 5x128, 70->3 8x64), random init; "
                        "second number: ray-sharded 4K (3840x2160) render" % (TRAIN_RAYS, TRAIN_VIEWS, TRAIN_S),
            "rays_per_step_total": TRAIN_RAYS, "samples_per_ray": TRAIN_S, "precision": precision,
            "l2": "inputs larger than L2: every step streams %.1f GB of saved activation tiles per %d rays" % (
                TRAIN_RAYS * TRAIN_S * 6.6e3 / 1e9, TRAIN_RAYS),
            "sharding": "strong scaling: rank g takes a contiguous 1/N of the rays; ONE flat NCCL all-reduce of the %d "
                        "MLP weight gradients per step" % 164164}


def train_rays_np():
    """[views, rays_per_view, 6]: 128x128 rays of each of the 4 views."""
    side = int(round((TRAIN_RAYS // TRAIN_VIEWS) ** 0.5))
    return np.stack([camera_rays(side, v) for v in range(TRAIN_VIEWS)])


TRAIN_LIGHTS = np.array([[0.4, 1.0, 0.3], [0.9, 0.5, -0.2], [-0.3, 0.8, 0.6], [0.1, 1.1, -0.5]], np.float32)


class TrainBench:
    """The cfg5 training step on the rays [lo, hi) of the flattened batch: NeRFLE model, flat parameter / gradient
    buffers (training.FlatParameters), fused AdamW, optional CUDA-graph capture of the whole step incl. the all-reduce."""

    def __init__(self, dev, lo, hi, distributed, graph=True):
        import torch
        from neural_raytracing_b200 import config, training
        from neural_raytracing_b200.pathtracer.lights import PointLights
        from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
        self.torch, self.dev, self.lo, self.hi = torch, dev, lo, hi
        config.set_train_precision("f16")
        torch.manual_seed(1)
        self.net = NeRFLE(device=dev)
        with torch.no_grad():
            self.net.first.out.bias[0] = 0.5
        self.net.far_jitter = torch.full((1,), 0.5, device=dev)
        self.flat = training.FlatParameters([self.net.first, self.net.second])
        self.opt = torch.optim.AdamW([self.flat.param], lr=8e-5, weight_decay=0, fused=True, capturable=True)
        per = TRAIN_RAYS // TRAIN_VIEWS
        n = hi - lo
        assert n > 0 and (n % per == 0 or per % n == 0), "slices must be whole views or whole fractions of a view"
        all_rays = train_rays_np().reshape(-1, 6)
        v0, v1 = lo // per, (hi - 1) // per + 1
        self.shape = (v1 - v0, n // (v1 - v0), 1, 1, 6)
        self.rays_host = torch.from_numpy(all_rays[lo:hi].reshape(self.shape).copy()).pin_memory()
        self.rays = self.rays_host.to(dev)
        self.lights = PointLights(device=dev, location=torch.from_numpy(TRAIN_LIGHTS[v0:v1].copy()).to(dev), scale=10)
        self.target = torch.full(self.shape[:-1] + (3,), 0.5, device=dev)
        self.allreduce = (lambda: self.flat.allreduce(average=False)) if distributed else None
        self.graph = None
        self.graph_error = None
        if graph:
            try:
                self.graph = training.GraphedStep(self.loss_fn, self.opt, modules=[self.net], allreduce=self.allreduce,
                                                  flat=self.flat, single_graph=True)
            except Exception as e:    # noqa: BLE001 -- fall back to the eager step, say so in the line
                self.graph_error = repr(e)[:300]
                torch.cuda.synchronize()

    def loss_fn(self):
        return (self.net(self.rays, self.lights) - self.target).square().sum() / (TRAIN_RAYS * 3)

    def eager_step(self):
        self.flat.zero_grad()
        loss = self.loss_fn()
        loss.backward()
        if self.allreduce is not None:
            self.allreduce()
        self.opt.step()
        return loss.detach()

    def step(self):
        return self.graph() if self.graph is not None else self.eager_step()

    def e2e_step(self):
        """Public API with HOST inputs: this rank's rays from pinned host memory, the loss read back."""
        self.rays.copy_(self.rays_host, non_blocking=True)
        return float(self.step().detach())

    def gradients_only(self):
        """Flat gradient of the current weights on this slice (no optimizer step, no all-reduce)."""
        self.flat.zero_grad()
        self.loss_fn().backward()
        return self.flat.grad.clone()


def _time_steps(torch, fn, steps, warmup, barrier):
    for _ in range(warmup):
        fn()
    barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        a.record(); fn(); b.record()
    barrier()
    return sum(a.elapsed_time(b) for a, b in evs) / steps


def run_multi_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from neural_raytracing_b200 import config, distributed as D, ops
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if "MASTER_ADDR" not in os.environ:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", RANK="0", WORLD_SIZE="1")
    dist.init_process_group("nccl", device_id=dev)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    assert TRAIN_RAYS % world == 0
    lo, hi = D.shard_range(TRAIN_RAYS, rank, world)
    sampler = ClockSampler(local_rank)
    sampler.start()
    tb = TrainBench(dev, lo, hi, distributed=True, graph=True)

    # ---- parity: the all-reduced N-rank gradient equals the 1-rank gradient of the whole batch (same weights) ----
    g_local = tb.gradients_only()
    g_sum = g_local.clone()
    dist.all_reduce(g_sum, op=dist.ReduceOp.SUM)
    parity = None
    single = None
    if rank == 0:
        one = TrainBench(dev, 0, TRAIN_RAYS, distributed=False, graph=True)
        g_one = one.gradients_only()
        a, b = g_sum.double(), g_one.double()
        parity = {"grad_cosine_nrank_vs_1rank": float((a @ b) / (a.norm() * b.norm())),
                  "grad_max_abs_diff_over_max_abs": float((a - b).abs().max() / b.abs().max()),
                  "note": "fp32 sums in a different order (per-rank partial sums + NCCL ring vs one kernel's atomics)"}
    barrier()

    # ---- the headline: K timed steps, barrier + synchronize on both sides, CUDA events, max over ranks ----
    last = [None]

    def timed_step():
        last[0] = tb.step()
    ms = max_over_ranks(_time_steps(torch, timed_step, args.steps, args.warmup, barrier))
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss=last[0], grad=tb.flat.grad, params=tb.flat.flat)
    del last
    # per-kernel split: the library's event brackets do not fire inside a graph replay, so the same step is also run
    # eagerly (its kernels are the ones the graph holds)
    n_eager = max(3, args.steps // 2)
    tb.eager_step(); tb.eager_step()
    barrier()
    ops.profile_collect(); ops.profile_enable(True)
    ms_eager = max_over_ranks(_time_steps(torch, tb.eager_step, n_eager, 0, barrier))
    prof_all = ops.profile_collect(); ops.profile_enable(False)
    prof = {k: (v[0] * args.steps / n_eager, int(round(v[1] * args.steps / n_eager))) for k, v in prof_all.items()}
    # all-reduce alone (eager, bracketed by events on the same stream)
    ar = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record(); tb.flat.allreduce(); b.record()
        torch.cuda.synchronize()
        ar.append(a.elapsed_time(b))
    ar_ms = max_over_ranks(sorted(ar)[len(ar) // 2])
    # ---- e2e: host rays in (pinned, H2D inside), loss out (D2H inside), wall clock over the steps ----
    e2e_steps = max(3, min(args.steps, 10))
    tb.e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        tb.e2e_step()
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps)
    loss_val = float(tb.step().detach())

    # ---- the same step on rank 0 alone, same run, same box (what N = 1 costs) ----
    if rank == 0:
        nobar = torch.cuda.synchronize
        ms1 = _time_steps(torch, one.step, max(3, args.steps // 2), 3, nobar)
        ms1_eager = _time_steps(torch, one.eager_step, 3, 1, nobar)
        single = {"ms_per_step": ms1, "ms_per_step_eager": ms1_eager, "rays_per_sec": TRAIN_RAYS / ms1 * 1e3,
                  "speedup_at_n": ms1 / ms, "cuda_graph": one.graph is not None}
        del one
        torch.cuda.empty_cache()
    barrier()

    # ---- second number: ray-sharded 4K render (the reference's single uniform pass of 64 samples), strong scaling ----
    render = None
    try:
        w1, w2 = synthetic_weights(0)

        def to_packed(w):
            Ws = [torch.from_numpy(x).to(dev) for x in w["W"]]
            bs = [torch.from_numpy(x).to(dev) for x in w["b"]]
            return ops.PackedMLP(w["in_size"], 0, w["freqs"], w["hidden"], w["num_layers"], w["skip"], w["out"],
                                 ops.ACT_LEAKY_RELU, torch.from_numpy(w["basis"]).to(dev), ops.PackedMLP.pack(Ws, bs))
        m1, m2 = to_packed(w1), to_packed(w2)
        total = 3840 * 2160
        rlo, rhi = D.shard_range(total, rank, world)
        base = torch.from_numpy(camera_rays(1080, 0)).to(dev)     # 1,166,400 distinct rays; ray i of the 4K frame = base[i % len]
        idx = torch.arange(rlo, rhi, device=dev) % base.shape[0]
        rays4k = base[idx].contiguous()
        ts = torch.linspace(0, 2.05, 64, device=dev)
        code = torch.tensor([[0.4, 1.0, 0.3]], device=dev)
        ops.nerfle_render(m1, m2, rays4k, ts, code, prec="f16")
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        img = ops.nerfle_render(m1, m2, rays4k, ts, code, prec="f16")
        b.record()
        barrier()
        rms = max_over_ranks(a.elapsed_time(b))
        # N-rank image == 1-rank image: rank 0 renders ANOTHER rank's slice and compares bit for bit
        chk = torch.zeros(2, device=dev, dtype=torch.float64)
        other = world - 1
        olo, ohi = D.shard_range(total, other, world)
        n_cmp = min(65536, ohi - olo)
        if rank == other and world > 1:
            sample = img[:n_cmp].contiguous()
            dist.send(sample, dst=0)
        if rank == 0:
            theirs = torch.empty(n_cmp, 3, device=dev)
            if world > 1:
                dist.recv(theirs, src=other)
            else:
                theirs.copy_(img[:n_cmp])
            mine = ops.nerfle_render(m1, m2, base[torch.arange(olo, olo + n_cmp, device=dev) % base.shape[0]].contiguous(), ts,
                                     code, prec="f16")
            chk[0] = float((mine - theirs).abs().max())
            chk[1] = float(torch.equal(mine, theirs))
        render = {"ms_per_frame": rms, "rays_per_sec": total / rms * 1e3, "mlp_samples_per_sec": total * 64 / rms * 1e3,
                  "model_tflops": total * 64 * (FLOP_FIRST + FLOP_SECOND) / rms / 1e9, "scaling": "strong",
                  "nrank_vs_1rank_max_abs_diff": float(chk[0]) if rank == 0 else None,
                  "nrank_vs_1rank_bit_identical": bool(chk[1]) if rank == 0 else None,
                  "compared": "%d pixels of rank %d's slice re-rendered by rank 0" % (n_cmp, other)}
        del rays4k, img, base
        # the same 4K frame from its camera (SURVEY f4): rank g renders its pixel rows, generating the rays on its own
        # device inside the library call -- no ray array is built, sharded or copied anywhere
        try:
            c2w = torch.from_numpy(camera_matrix(0)).to(dev)
            xlo, xhi = D.shard_range(3840, rank, world)

            def rows(x0, n):
                cam = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=0.5 * 3840 / np.tan(np.radians(30)), size=3840, x0=x0,
                                     y0=840, nx=n, ny=2160)
                return ops.nerfle_render_camera(m1, m2, cam, ts, code, prec="f16")
            rows(xlo, xhi - xlo)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            mine_rows = rows(xlo, xhi - xlo)
            b.record()
            barrier()
            cms = max_over_ranks(a.elapsed_time(b))
            same = torch.zeros(1, device=dev, dtype=torch.float64)
            n_cmp = min(16, xhi - xlo)
            if rank == world - 1 and world > 1:
                dist.send(mine_rows[:, :n_cmp].contiguous(), dst=0)
            if rank == 0:
                olo, _ = D.shard_range(3840, world - 1, world)
                theirs = torch.empty((1, n_cmp, 2160, 1, 3), device=dev)
                if world > 1:
                    dist.recv(theirs, src=world - 1)
                else:
                    theirs.copy_(mine_rows[:, :n_cmp])
                same[0] = float(torch.equal(rows(olo, n_cmp), theirs))
            render["from_camera"] = {"ms_per_frame": cms, "rays_per_sec": total / cms * 1e3,
                                     "nrank_vs_1rank_bit_identical": bool(same[0]) if rank == 0 else None,
                                     "note": "rank g renders pixel rows shard_range(3840, g, N) of the 3840x2160 window through "
                                             "nrt_nerfle_render_camera (rays generated on its own device)"}
            del mine_rows
        except Exception as e:   # noqa: BLE001
            render["from_camera"] = {"error": repr(e)[:300]}
    except Exception as e:   # noqa: BLE001
        render = {"error": repr(e)[:300]}

    if rank == 0:
        peak_tf, peak_gbs, peak_src = measured_peaks()
        value = TRAIN_RAYS / ms * 1e3
        wg_ms, wg_n = prof.get("mlp_tc_wgrad", (0.0, 0))
        roof = None
        if wg_n and wg_ms > 0:
            bytes_per_launch = (hi - lo) * TRAIN_S * WGRAD_BYTES_PER_SAMPLE / 2.0     # two launches per step (second, first)
            gbs = bytes_per_launch / (wg_ms / wg_n * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "k_mlp_wgrad_tc (tcgen05, saved 16-bit activation / gradient tiles read once)",
                    "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs, "traffic": None,
                    "peak_source": peak_src.replace("sustained bf16", "copy bandwidth"), "launches": wg_n,
                    "avg_launch_ms": wg_ms / wg_n,
                    "algorithmic_bytes_per_sample": WGRAD_BYTES_PER_SAMPLE,
                    "share_of_step": wg_ms / (ms * args.steps),
                    "note": "per rank; at N ranks every kernel works on 1/N of the batch",
                    "other_kernels": {k: {"ms_per_step": round(v[0] / args.steps, 4), "launches": v[1],
                                          "tflops": (round((hi - lo) * TRAIN_S * (FLOP_FIRST + FLOP_SECOND) / (v[0] / args.steps) / 1e9, 1)
                                                     if k in ("mlp_tc_train_fwd", "mlp_tc_dgrad") else None)}
                                      for k, v in prof.items() if v[1] and k != "mlp_tc_wgrad"}}
        line = {
            "metric": "train_rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "mlp_samples_per_sec": value * TRAIN_S,
            "model_tflops_fwd_bwd": value * TRAIN_S * (FLOP_FIRST + FLOP_SECOND) * 3 / 1e12,
            "config": train_workload_config("f16 operands / fp32 accumulate (tcgen05 training kernels)", world),
            "e2e": {"value": TRAIN_RAYS / e2e_ms * 1e3, "unit": "rays/s", "h2d_bytes_per_step": (hi - lo) * 24,
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms,
                    "api": "training.GraphedStep (one CUDA graph: zero_grad, NeRFLE forward, loss, backward, NCCL all-reduce, "
                           "fused AdamW); rays copied from pinned host memory and the loss read back every step"},
            "gpu_launches": sum(n for _, n in prof.values()),
            "gpu_launches_note": "library kernels per step x steps (the timed steps replay a CUDA graph holding exactly these kernels)",
            "kernel_ms_per_step": {k: round(v[0] / args.steps, 4) for k, v in prof.items() if v[1]},
            "cuda_graph": tb.graph is not None, "cuda_graph_error": tb.graph_error,
            "ms_per_step_eager": ms_eager, "grad_allreduce_ms": ar_ms,
            "grad_bucket_bytes": int(tb.flat.grad.numel() * 4),
            "loss": loss_val,
            "single_gpu_same_run": single,
            "parity_nrank_vs_1rank": parity,
            "render_4k": render,
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": None,
        }
        emit_result(line)
    # tear-down: the captured graphs hold NCCL kernels; release them before the communicator, and never let a stuck
    # communicator tear-down keep the job alive after the result line is out
    barrier()
    tb.graph = None
    del tb
    torch.cuda.synchronize()
    import threading
    threading.Timer(20.0, lambda: os._exit(0)).start()
    try:
        dist.destroy_process_group()
    finally:
        os._exit(0)


def ncu_traffic():
    """Per-launch DRAM bytes of the dominant kernel from the committed `ncu --set full` capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("mlp_tc_nerf_first_dram_bytes_per_launch")
        except Exception:
            return None
    return None


def dump_outputs(directory, **arrays):
    """Writes each tensor as DIR/<name>.npy in float32."""
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline number (value, ms_per_step); the secondary legs pick their own counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="f16", choices=["f16", "bf16", "f32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the supplementary configs reported under `also`")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    multi_gpu = world > 1 or os.environ.get("NRT_BENCH_FORCE_CFG5") == "1"     # (the env switch is a development aid)
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference arm times a sample of the rays only")

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if multi_gpu:
        run_multi_gpu(args, rank, world, local_rank)
        return

    import torch
    import torch.distributed as dist
    from neural_raytracing_b200 import ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    w1, w2 = synthetic_weights(0)

    def to_packed(w):
        Ws = [torch.from_numpy(x).to(dev) for x in w["W"]]
        bs = [torch.from_numpy(x).to(dev) for x in w["b"]]
        return ops.PackedMLP(w["in_size"], 0, w["freqs"], w["hidden"], w["num_layers"], w["skip"], w["out"],
                             ops.ACT_LEAKY_RELU, torch.from_numpy(w["basis"]).to(dev), ops.PackedMLP.pack(Ws, bs))
    m1, m2 = to_packed(w1), to_packed(w2)
    rays_np = camera_rays(IMG, rank)
    R = rays_np.shape[0]
    rays = torch.from_numpy(rays_np).to(dev)
    code = torch.tensor([[0.4, 1.0, 0.3]], device=dev)
    rays_host = torch.from_numpy(rays_np).pin_memory()
    out_host = torch.empty(R, 3).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    kw = dict(prec=args.precision, n_coarse=N_COARSE, n_fine=N_FINE, t_near=T_NEAR, t_far=T_FAR, jitter_seed=JITTER_SEED)

    def step():
        return ops.nerfle_render(m1, m2, rays, None, code, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()            # nvidia-smi needs ~1 s to come up: start it before the warm-up
    # the warm-up also keeps each step's rgb alive until the next one returns, so the timed loop reuses cached blocks
    for _ in range(args.warmup):
        rgb = step()
    barrier()
    ops.profile_collect()
    ops.profile_enable(True)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in evs:
        flush.zero_()          # L2 flush, outside the event bracket
        a.record()
        rgb = step()
        b.record()
    barrier()
    clocks = sampler.stop()
    prof = ops.profile_collect()
    ops.profile_enable(False)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rgb=rgb)
    del rgb
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * R / (ms_per_step / 1e3)

    # ---- end to end: pinned host rays in, host rgb out, copies inside the timed region ----
    e2e_steps = max(3, min(args.steps, 10))
    ops.nerfle_render_host(m1, m2, rays_host, None, code, out_host, **kw)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ops.nerfle_render_host(m1, m2, rays_host, None, code, out_host, **kw)   # synchronises before returning
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_value = world * R / (e2e_ms / 1e3)

    # ---- the same frame from its camera (SURVEY f4): rays generated on the device inside the call, nothing but the
    #      camera descriptor goes in, the image comes back to pinned host memory ----
    cam = ops.CameraDesc(ops.CAM_NERF, torch.from_numpy(camera_matrix(rank)).to(dev), None,
                         focal=0.5 * IMG / np.tan(np.radians(30)), size=IMG, nx=IMG, ny=IMG)
    ops.nerfle_render_camera_host(m1, m2, cam, None, code, out_host, **kw)
    cam_finite = bool(torch.isfinite(out_host).all())
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ops.nerfle_render_camera_host(m1, m2, cam, None, code, out_host, **kw)
    torch.cuda.synchronize()
    cam_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    t = torch.tensor([cam_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    cam_ms = float(t.item())

    also = None
    NO_CPU[0] = bool(args.no_cpu_baseline)
    if not args.no_also:
        del flush
        torch.cuda.empty_cache()
        also = supplementary(dev, rank, world)

    # ---- CPU baseline last (rank 0, N=1 only): it must not overlap the GPU timing, and running it first leaves the
    # host's OpenMP pool spinning under the launch-bound training steps of `also` ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sel = np.linspace(0, R - 1, CPU_SAMPLE_RAYS).astype(np.int64)
        rate, ms, threads = cpu_reference_rate(w1, w2, rays_np[sel], 2, 1)
        cpu = {"value": rate, "unit": "rays/s", "cores": threads, "kind": "port",
               "sample": "%d evenly strided rays of the frame, 64+128 samples/ray, mean of 2 runs after 1 warm-up "
                         "(oracle/port.py: the reference's eager PyTorch op sequence on the host cores)" % CPU_SAMPLE_RAYS}

    if rank == 0:
        peak_tf, peak_gbs, peak_src = measured_peaks()
        first_ms, first_n = prof.get("mlp_tc_nerf_first", (0.0, 0))
        launches = sum(n for _, n in prof.values())
        roof = None
        if first_n and first_ms > 0:
            samples_per_launch = R * (N_COARSE + N_FINE) * args.steps / first_n
            tf = samples_per_launch * FLOP_FIRST / (first_ms / first_n * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": "k_mlp_tc<NeRFLE.first> (tcgen05, %s operands)" % args.precision,
                    "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf, "traffic": ncu_traffic(),
                    "peak_source": peak_src, "launches": first_n, "avg_launch_ms": first_ms / first_n,
                    "algorithmic_flop_per_sample": FLOP_FIRST,
                    "share_of_step": first_ms / total_ms if total_ms else None}
        # the other kernels of the step, each against the roof that bounds it (live CUDA-event times of this run)
        others = {}

        def _other(tag, kernel, bound, work_per_step, peak, unit, note):
            t_ms, n = prof.get(tag, (0.0, 0))
            if n and t_ms > 0:
                ach = work_per_step * args.steps / (t_ms * 1e-3)
                others[tag] = {"kernel": kernel, "bound": bound, "achieved": ach, "peak": peak, "unit": unit,
                               "frac": ach / peak, "launches": n, "share_of_step": t_ms / total_ms if total_ms else None,
                               "algorithmic_work_per_step": note}
        _other("mlp_tc_nerf_second", "k_mlp_tc<NeRFLE.second>", "tensor", R * (N_COARSE + N_FINE) * FLOP_SECOND / 1e12, peak_tf,
               "TFLOP/s", "%d samples x %d FLOP" % (R * (N_COARSE + N_FINE), FLOP_SECOND))
        _other("merge_composite", "k_merge_composite", "hbm", R * ((N_COARSE + N_FINE) * 20 + 12) / 1e9, peak_gbs, "GB/s",
               "%d rays x (192 samples x 20 B (t, sigma, rgb) + 12 B out)" % R)
        _other("sample_pdf", "k_sample_pdf", "hbm", R * (N_COARSE * 8 + N_FINE * 4) / 1e9, peak_gbs, "GB/s",
               "%d rays x (64 x 8 B (t, sigma) read + 128 x 4 B written)" % R)
        _other("stratified_ts", "k_stratified_ts", "hbm", R * N_COARSE * 4 / 1e9, peak_gbs, "GB/s", "%d rays x 64 x 4 B written" % R)
        if roof is not None:
            roof["other_kernels"] = others
        elif args.precision == "f32":
            fm, fn = prof.get("nerfle_fused_f32", (0.0, 0))
            if fn and fm > 0:
                tf = R * (N_COARSE + N_FINE) * args.steps / fn * (FLOP_FIRST + FLOP_SECOND) / (fm / fn * 1e-3) / 1e12
                roof = {"bound": "tensor", "kernel": "k_nerfle (fp32 FMA, exact path)", "achieved": tf, "peak": peak_tf,
                        "unit": "TFLOP/s", "frac": tf / peak_tf, "traffic": None, "peak_source": peak_src}
        line = {
            "metric": "rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "mlp_samples_per_sec": value * (N_COARSE + N_FINE),
            "model_tflops": value * (N_COARSE + N_FINE) * (FLOP_FIRST + FLOP_SECOND) / 1e12,
            "config": workload_config(args.precision),
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": R * 24, "d2h_bytes_per_step": R * 12,
                    "ms_per_step": e2e_ms,
                    "from_camera": {"value": world * R / (cam_ms / 1e3), "unit": "rays/s", "ms_per_step": cam_ms,
                                    "h2d_bytes_per_step": 0, "d2h_bytes_per_step": R * 12, "finite": cam_finite,
                                    "note": "nrt_nerfle_render_camera_host: pixel -> ray inside the library "
                                            "(k_camera_rays per 262,144-ray chunk), no ray array crosses PCIe"}},
            "gpu_launches": launches,
            "kernel_ms": {k: round(v[0], 3) for k, v in prof.items() if v[1]},
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "also": also,
        }
        emit_result(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
