"""Time a NeRFLE training step (forward -> MSE -> backward -> AdamW, tensor-core training kernels, f16) with the
reference's 64 shared uniform samples against hierarchical sampling (HierarchicalSampling: 64 stratified coarse + 128
importance-resampled fine samples), eager and captured by training.GraphedStep, at R = 4,096 and 16,384 rays.

Prints ONE JSON line: the GPU's name and power limit (read in the same run), and per case
  * ms_per_step: device events around `--steps` steps after `--warmup` steps;
  * kernel_ms_per_step: the per-kernel split of an eager step (ops.profile_enable; a separate, profiled run -- graph
    replays launch nothing from the host, so the split of a graphed step is that of the eager one);
  * peak_mem_gb: torch.cuda.max_memory_allocated over the timed steps;
  * vs_fp32: max |rgb| difference of the forward and the smallest per-tensor gradient cosine of the f16 step against
    the exact fp32 kernels on the same rays and the same sample distances.
65,536 rays are not timed by default: the saved activation tiles take ~6.6 KB per sample, ~83 GB at 192 samples.
Needs a CUDA device; there is no CPU mode."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)


def gpu_info():
    import torch
    idx = torch.cuda.current_device()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(idx)],
                           capture_output=True, text=True, timeout=60)
        power = r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        power = "unavailable (%s)" % e
    return {"gpu": torch.cuda.get_device_name(idx), "power_limit_and_max_sm_clock": power}


def make_model(hier):
    import torch
    import helpers
    from neural_raytracing_b200.pathtracer.shapes.nerf import HierarchicalSampling, NeRFLE
    n = NeRFLE(device="cuda")
    w1, w2 = helpers.nerfle_weights(False)
    for mod, w in ((n.first, w1), (n.second, w2)):
        mod.basis_p = torch.from_numpy(w["basis"]).cuda()
        for lin, W, b in zip([mod.init] + list(mod.layers) + [mod.out], w["W"], w["b"]):
            with torch.no_grad():
                lin.weight.copy_(torch.from_numpy(W)); lin.bias.copy_(torch.from_numpy(b))
    if hier:
        n.sampling = HierarchicalSampling()
    else:
        n.far_jitter = torch.full((1,), 0.37, device="cuda")     # device-side far-plane draw: capturable
    return n


def scene(R):
    import torch
    import synth
    from neural_raytracing_b200.pathtracer.lights import PointLights
    rays = torch.from_numpy(synth.camera_rays(5, R).reshape(1, R, 1, 1, 6)).cuda()
    lights = PointLights(device="cuda", location=torch.tensor([[0.4, 1.0, 0.3]], device="cuda"), scale=10)
    target = torch.full((1, R, 1, 1, 3), 0.5, device="cuda")
    return rays, lights, target


def time_case(R, hier, graphed, steps, warmup):
    import torch
    from neural_raytracing_b200 import config, ops
    from neural_raytracing_b200.training import GraphedStep
    n = make_model(hier)
    rays, lights, target = scene(R)
    opt = torch.optim.AdamW(n.parameters(), lr=8e-5, weight_decay=0, capturable=True)
    loss_fn = lambda: torch.nn.functional.mse_loss(n(rays, lights), target)
    config.set_train_precision("f16")
    try:
        if graphed:
            fn = GraphedStep(loss_fn, opt, modules=[n], warmup=warmup)
        else:
            def fn():
                opt.zero_grad(set_to_none=True)
                loss = loss_fn()
                loss.backward()
                opt.step()
                return loss
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res = {"ms_per_step": round(e0.elapsed_time(e1) / steps, 3),
               "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 1e9, 3)}
        if not graphed:
            ops.profile_collect()
            ops.profile_enable(True)
            k = max(1, min(steps, 5))
            for _ in range(k):
                fn()
            torch.cuda.synchronize()
            prof = ops.profile_collect()
            ops.profile_enable(False)
            res["kernel_ms_per_step"] = {t: round(ms / k, 3) for t, (ms, c) in prof.items() if c}
    finally:
        config.set_train_precision("f32")
    del fn, opt, n
    torch.cuda.empty_cache()
    return res


def vs_fp32(R, hier):
    """f16 step against the exact fp32 kernels on the same distances (the hierarchical ones from the f16 coarse pass)."""
    import torch
    from neural_raytracing_b200 import config, ops
    n = make_model(hier)
    rays, lights, target = scene(R)
    real = ops.nerfle_sample_hierarchical
    ops.nerfle_sample_hierarchical = lambda *a, **k: real(*a, **dict(k, prec="f16"))
    res = {}
    try:
        for prec in ("f32", "f16"):
            config.set_train_precision(prec)
            if hier:
                n.sampling.train_seed("cuda").fill_(5)
            n.zero_grad()
            out = n(rays, lights)
            torch.nn.functional.mse_loss(out, target).backward()
            res[prec] = (out.detach().clone(), [p.grad.clone() for p in n.parameters()])
    finally:
        ops.nerfle_sample_hierarchical = real
        config.set_train_precision("f32")
    cos = []
    for a, b in zip(res["f32"][1], res["f16"][1]):
        if float(a.norm()) > 0:
            a, b = a.double().flatten(), b.double().flatten()
            cos.append(float(a @ b / (a.norm() * b.norm())))
    return {"max_abs_rgb_diff": float((res["f32"][0] - res["f16"][0]).abs().max()), "min_grad_cosine": round(min(cos), 6)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rays", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nerfle_hier_train_time.py needs a CUDA device")
    out = dict(gpu_info(), train_precision="f16", steps=args.steps, warmup=args.warmup, cases=[])
    for R in args.rays:
        for hier in (False, True):
            case = {"rays": R, "sampling": "64+128 hierarchical" if hier else "64 uniform",
                    "samples_per_ray": 192 if hier else 64}
            for graphed in (False, True):
                case["graphed" if graphed else "eager"] = time_case(R, hier, graphed, args.steps, args.warmup)
            case["vs_fp32"] = vs_fp32(R, hier)
            out["cases"].append(case)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
