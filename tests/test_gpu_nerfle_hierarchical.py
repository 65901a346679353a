"""GPU tests (-m gpu) of training NeRFLE on hierarchical samples (NeRFLE.sampling = HierarchicalSampling(...)):
the merged distances of nrt_nerfle_sample_hierarchical against the numpy restatement (oracle/port.py), the per-sample
compositing pair, the trained function against the rendered one, gradients against float64 autograd, kernel routing,
a production-size step, CUDA-graph capture, and the one-call camera frame of pathtrace."""
import copy

import numpy as np
import pytest

import helpers
import synth
from oracle import c_oracle, port

pytestmark = pytest.mark.gpu

KW = dict(n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05)


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-300))


def _model(envmap=False, jitter=True):
    import torch
    from neural_raytracing_b200.pathtracer.shapes.nerf import HierarchicalSampling, NeRFLE
    n = NeRFLE(envmap=envmap, device="cuda")
    w1, w2 = helpers.nerfle_weights(envmap)
    for mod, w in ((n.first, w1), (n.second, w2)):
        mod.basis_p = torch.from_numpy(w["basis"]).cuda()
        for lin, W, b in zip([mod.init] + list(mod.layers) + [mod.out], w["W"], w["b"]):
            with torch.no_grad():
                lin.weight.copy_(torch.from_numpy(W)); lin.bias.copy_(torch.from_numpy(b))
    n.sampling = HierarchicalSampling(jitter=jitter, **KW)
    return n


def _scene(n_views, W, H, seed=5):
    import torch
    from neural_raytracing_b200.pathtracer.lights import PointLights
    rays = _t(synth.camera_rays(seed, n_views * W * H).reshape(n_views, W, H, 1, 6))
    g = torch.Generator(device="cuda").manual_seed(seed)
    lights = PointLights(device="cuda", location=torch.randn(n_views, 3, device="cuda", generator=g), scale=10)
    return rays, lights


def _inputs(n, rays, lights):
    code = n._code_rows(n._light_code(lights, rays.device), rays.shape[0]).detach().float()
    return code, n._view_index(rays)


@pytest.mark.parametrize("seed", [0, 7])
def test_distances_vs_restatement(seed):
    """Stratified coarse distances, the coarse sigma of the C oracle, port.sample_pdf and a stable merge: every ray's
    merged list is ascending, the coarse distances are the restatement's bit for bit, and the merged lists agree to 1e-5
    except where a fine sample falls into a near-empty bin: there the pdf is ~the 1e-5 weight floor and the inverse CDF
    divides by it, so the few-ulp difference between the kernel's warp-scan cdf and numpy's sequential cumsum moves the
    sample within its bin (measured on B200 at seed 7: 89.6 % of the rays within 1e-5, the worst 1.9e-3; seed 0: all within
    1e-5).  The gate keeps a margin of 2.6x over that worst case, far below the 0.032 of one coarse bin, so a sample placed
    in the wrong bin fails."""
    from neural_raytracing_b200 import ops
    w1, w2 = helpers.nerfle_weights(False)
    R = 192
    rays = synth.camera_rays(55, R)
    code = np.array([[0.4, 1.0, 0.3]], np.float32)
    ts = ops.nerfle_sample_hierarchical(helpers.cuda_mlp(w1), helpers.cuda_mlp(w2), _t(rays), _t(code), prec="f32",
                                        jitter_seed=seed, **KW)
    assert tuple(ts.shape) == (192, R)
    got = ts.cpu().numpy().T
    ts_c = port.stratified_ts(R, 64, 0.0, 2.05, seed)
    _, sig_c, _ = c_oracle.nerfle_render(helpers.oracle_mlp(w1), helpers.oracle_mlp(w2), rays, ts_per_ray=ts_c,
                                         light_code=code, store=True)
    ts_f = port.sample_pdf(sig_c, ts_c, 128, seed)
    ref = np.sort(np.concatenate([ts_c, ts_f], axis=1), axis=1, kind="stable")
    assert (np.diff(got, axis=1) >= 0).all()
    assert all(np.isin(ts_c[r], got[r]).all() for r in range(R))
    err = np.abs(got - ref).max(axis=1)
    assert (err <= 1e-5).mean() >= (1.0 if seed == 0 else 0.85), np.sort(err)[-10:]
    assert err.max() <= 5e-3, err.max()


def test_composite_ts_vs_shared_and_float64():
    import torch
    from neural_raytracing_b200 import ops, torch_ops  # noqa: F401  (registers torch.ops.nrt_b200.composite_ts)
    g = torch.Generator(device="cuda").manual_seed(0)
    S, R = 192, 3000
    sigma = torch.randn(S, R, device="cuda", generator=g) * 2
    rgb = torch.rand(S, R, 3, device="cuda", generator=g)
    go = torch.randn(R, 3, device="cuda", generator=g)
    ts = torch.sort(torch.rand(S, device="cuda", generator=g) * 2.05).values
    tsr = ts[:, None].expand(S, R).contiguous()
    assert torch.equal(ops.composite_forward_ts(sigma, rgb, tsr), ops.composite_forward(sigma, rgb, ts))
    a, b = ops.composite_backward(sigma, rgb, ts, go), ops.composite_backward_ts(sigma, rgb, tsr, go)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    tpr = torch.sort(torch.rand(S, R, device="cuda", generator=g) * 2.05, dim=0).values
    out = ops.composite_forward_ts(sigma, rgb, tpr)
    gs, gc = ops.composite_backward_ts(sigma, rgb, tpr, go)
    s64, c64, t64 = sigma.double().requires_grad_(), rgb.double().requires_grad_(), tpr.double()
    al = 1 - torch.exp(-torch.relu(s64) * t64)
    cp = torch.roll(torch.cumprod((1 - al).clamp(min=1e-10), dim=0), 1, 0)
    cp = torch.cat([cp[:-1], torch.ones_like(cp[:1])])
    ref = ((al * cp)[..., None] * c64).sum(0)
    (ref * go.double()).sum().backward()
    for got, want in ((out, ref.detach()), (gs, s64.grad), (gc, c64.grad)):
        assert torch.allclose(got.double(), want, atol=1e-6, rtol=1e-5), float((got.double() - want).abs().max())
    # through the registered operator and its backward
    s2 = sigma.clone().requires_grad_()
    (torch.ops.nrt_b200.composite_ts(s2, rgb, tpr) * go).sum().backward()
    assert torch.equal(s2.grad, gs)


@pytest.mark.parametrize("envmap", [False, True])
@pytest.mark.parametrize("tprec,tol", [("f32", 1e-5), ("f16", 2e-3)])
def test_trained_function_is_rendered_function(envmap, tprec, tol):
    """The differentiable forward with seed s equals ops.nerfle_render(n_coarse, n_fine, t_near, t_far, jitter_seed=s) at
    the same precision: a 2-view [2,W,H,1,6] batch with per-view light codes."""
    from neural_raytracing_b200 import config, ops
    n = _model(envmap)
    rays, lights = _scene(2, 12, 10)
    seed = 7
    n.sampling.train_seed("cuda").fill_(seed)
    try:
        config.set_train_precision(tprec)
        out = n(rays, lights)
    finally:
        config.set_train_precision("f32")
    assert out.requires_grad and tuple(out.shape) == (2, 12, 10, 1, 3)
    assert int(n.sampling.seed.item()) == seed + 1
    code, view = _inputs(n, rays, lights)
    ref = ops.nerfle_render(n.first.packed(), n.second.packed(), rays, None, code, view, prec=tprec, jitter_seed=seed, **KW)
    assert float((out.detach() - ref).abs().max()) <= tol


@pytest.mark.parametrize("tprec,tol", [("f32", 1e-5), ("f16", 2e-3)])
@pytest.mark.parametrize("n_coarse,n_fine", [(1, 0), (64, 0), (16, 16), (4, 128), (128, 384)])
def test_every_accepted_configuration_trains(n_coarse, n_fine, tprec, tol):
    """Configurations at the edges of what HierarchicalSampling accepts -- one stratified sample, a single stratified pass
    (n_fine = 0: no coarse pass, the stratified distances are trained on as they are), the fewest coarse samples the
    resampling allows -- train, and the trained function is the rendered one."""
    import torch
    from neural_raytracing_b200 import config, ops
    from neural_raytracing_b200.pathtracer.shapes.nerf import HierarchicalSampling
    n = _model()
    n.sampling = HierarchicalSampling(n_coarse=n_coarse, n_fine=n_fine, t_near=0.0, t_far=2.05)
    rays, lights = _scene(2, 8, 8)
    target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
    n.sampling.train_seed("cuda").fill_(9)
    try:
        config.set_train_precision(tprec)
        out = n(rays, lights)
        torch.nn.functional.mse_loss(out, target).backward()
    finally:
        config.set_train_precision("f32")
    grads = [p.grad for p in n.parameters()]
    assert all(g is not None and torch.isfinite(g).all() for g in grads)
    assert sum(float(g.norm()) for g in grads) > 0
    code, view = _inputs(n, rays, lights)
    ref = ops.nerfle_render(n.first.packed(), n.second.packed(), rays, None, code, view, prec=tprec, n_coarse=n_coarse,
                            n_fine=n_fine, t_near=0.0, t_far=2.05, jitter_seed=9)
    assert float((out.detach() - ref).abs().max()) <= tol


def _ref_grads64(n, rays, ts, code, view, target, chunk=1024):
    """float64 torch autograd of both MLPs + compositing over the fixed distances ts [S,R], loss = MSE to target.  Rays
    are independent, so the loss is accumulated chunk by chunk of rays (memory stays a few GB at 16,384 rays)."""
    import torch
    mods = []
    for m in (n.first, n.second):
        d = copy.deepcopy(m).double()
        d.basis_p = m.basis_p.detach().double()
        mods.append(d)
    f, s2 = mods
    r_all = rays.double().reshape(-1, 6)
    S, R = ts.shape
    tgt = target.double().reshape(R, 3)
    light_all = code.double()[view.long()]
    for r0 in range(0, R, chunk):
        r, t, light = r_all[r0:r0 + chunk], ts[:, r0:r0 + chunk].double(), light_all[r0:r0 + chunk]
        k = r.shape[0]
        pts = r[None, :, :3] + t[..., None] * r[None, :, 3:]
        fo = f.forward_reference_ops(pts)
        lat, sig = fo[..., 1:], fo[..., 0]
        x2 = torch.cat([lat, r[None, :, 3:].expand(S, k, 3), light[None].expand(S, k, -1)], -1)
        rgb = s2.forward_reference_ops(x2).sigmoid()
        al = 1 - torch.exp(-torch.relu(sig) * t)
        cp = torch.roll(torch.cumprod((1 - al).clamp(min=1e-10), dim=0), 1, 0)
        cp = torch.cat([cp[:-1], torch.ones_like(cp[:1])])
        out = ((al * cp)[..., None] * rgb).sum(0)
        (((out - tgt[r0:r0 + chunk]) ** 2).sum() / (R * 3)).backward()
    return [p.grad for p in list(f.parameters()) + list(s2.parameters())]


@pytest.mark.parametrize("envmap", [False, True])
@pytest.mark.parametrize("tprec,gate,shape", [("f32", 0.99999, (2, 16, 8)), ("f16", 0.999, (2, 128, 64))])
def test_gradients_vs_float64(envmap, tprec, gate, shape):
    """Cosine per parameter tensor against float64 autograd on the same merged distances.
    f32 (exact kernels): 0.99999 on every tensor at 256 rays x 192 samples.  (At 16,384 rays the fp32 sum of 3.1 M
    per-sample contributions in NeRFLE.first's init-layer gradient drifts: measured 0.999978 on B200.)
    f16: 0.999 on every tensor, the NeRFLE gate of test_gpu_tc_train.py, at a training batch of 16,384 rays x 192 samples.
    (The forward's 16-bit rounding decides which leaky_relu kinks NeRFLE.first's input-side layers pass through; a flipped
    kink is an error of one sample, so it takes a realistic batch for the gradient to average over them: at 256 rays those
    two tensors measured 0.9964 / 0.9986 on B200.)"""
    import torch
    from neural_raytracing_b200 import config, ops
    n = _model(envmap)
    rays, lights = _scene(*shape, seed=9)
    target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
    code, view = _inputs(n, rays, lights)
    seed = 3
    n.sampling.train_seed("cuda").fill_(seed)
    ts = ops.nerfle_sample_hierarchical(n.first.packed(), n.second.packed(), rays, code, view, prec=tprec, jitter_seed=seed,
                                        **KW)
    try:
        config.set_train_precision(tprec)
        n.zero_grad()
        torch.nn.functional.mse_loss(n(rays, lights), target).backward()
    finally:
        config.set_train_precision("f32")
    refs = _ref_grads64(n, rays, ts, code, view, target)
    cos = {name: _cos(p.grad, ref) for (name, p), ref in zip(n.named_parameters(), refs) if float(ref.norm()) > 0}
    assert len(cos) >= 30
    low = {k: c for k, c in cos.items() if c < gate}
    assert not low, (tprec, low, min(cos.values()))


def _tags(counts):
    return {k for k, (_, c) in counts.items() if c}


@pytest.mark.parametrize("tprec", ["f32", "f16"])
def test_kernel_routing(tprec):
    import torch
    from neural_raytracing_b200 import config, ops
    n = _model()
    rays, lights = _scene(1, 16, 16)
    target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
    try:
        config.set_train_precision(tprec)
        torch.nn.functional.mse_loss(n(rays, lights), target).backward()   # first call: packing, lazy set-up
        n.zero_grad()
        torch.cuda.synchronize()
        ops.profile_collect()
        torch.nn.functional.mse_loss(n(rays, lights), target).backward()
        torch.cuda.synchronize()
        ran = _tags(ops.profile_collect())
    finally:
        config.set_train_precision("f32")
    tc_train = {"mlp_tc_train_fwd", "mlp_tc_dgrad", "mlp_tc_wgrad"}
    assert {"stratified_ts", "sample_pdf", "merge_ts", "composite_ts_fwd", "composite_ts_bwd"} <= ran, ran
    assert "merge_composite" not in ran and "composite_fwd" not in ran
    if tprec == "f16":
        assert tc_train <= ran and not any(t.endswith("_f32") for t in ran), ran
    else:
        assert not (tc_train & ran), ran


def test_realistic_tile_count_f16_vs_fp32_kernels(monkeypatch):
    """4,096 rays x 192 samples = 6,144 tiles of 128: the f16 step's gradients against the exact fp32 kernels on the same
    merged distances (the gate of test_nerfle_training_step_tc_vs_fp32)."""
    import torch
    from neural_raytracing_b200 import config, ops
    real = ops.nerfle_sample_hierarchical
    monkeypatch.setattr(ops, "nerfle_sample_hierarchical", lambda *a, **k: real(*a, **dict(k, prec="f16")))
    n = _model()
    rays, lights = _scene(4, 32, 32, seed=11)
    target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
    res = {}
    try:
        for prec in ("f32", "f16"):
            config.set_train_precision(prec)
            n.sampling.train_seed("cuda").fill_(5)
            n.zero_grad()
            loss = torch.nn.functional.mse_loss(n(rays, lights), target)
            loss.backward()
            res[prec] = (float(loss.detach()), [p.grad.clone() for p in n.parameters()])
    finally:
        config.set_train_precision("f32")
    assert abs(res["f32"][0] - res["f16"][0]) < 1e-3 * max(1.0, abs(res["f32"][0]))
    cs = [_cos(a, b) for a, b in zip(res["f32"][1], res["f16"][1]) if float(a.norm()) > 0]
    assert min(cs) >= 0.995 and float(np.median(cs)) >= 0.9995, (min(cs), float(np.median(cs)))


def _graphed(n, rays, lights, target, lr):
    import torch
    from neural_raytracing_b200.training import GraphedStep
    opt = torch.optim.AdamW(n.parameters(), lr=lr, weight_decay=0, capturable=True)
    return GraphedStep(lambda: torch.nn.functional.mse_loss(n(rays, lights), target), opt, modules=[n], warmup=3)


def test_graphed_step(monkeypatch):
    """GraphedStep on a hierarchical NeRFLE: replayed losses equal eager ones, training lowers the loss, the device seed
    advances by one per step and new jitter is drawn per replay; without jitter the distances repeat."""
    import torch
    from neural_raytracing_b200 import config, ops
    real = ops.nerfle_sample_hierarchical
    seen = {}

    def spy(*a, **k):
        ts = real(*a, **k)
        if "buf" not in seen:
            seen["buf"] = torch.empty_like(ts)
        seen["buf"].copy_(ts)          # captured too: every replay leaves its distances here
        return ts
    monkeypatch.setattr(ops, "nerfle_sample_hierarchical", spy)
    a = _model()
    b = copy.deepcopy(a)
    rays, lights = _scene(1, 32, 32, seed=13)
    target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
    try:
        config.set_train_precision("f16")
        oa = torch.optim.AdamW(a.parameters(), lr=1e-3, weight_decay=0, capturable=True)
        step = _graphed(b, rays, lights, target, 1e-3)
        losses_b, seeds, dists = [], [], []
        for _ in range(4):
            losses_b.append(float(step().detach()))
            seeds.append(int(b.sampling.seed.item()))
            dists.append(seen["buf"].clone())
        losses_a = []
        for i in range(7):
            oa.zero_grad(set_to_none=True)
            loss = torch.nn.functional.mse_loss(a(rays, lights), target)
            loss.backward(); oa.step()
            if i >= 3:
                losses_a.append(float(loss.detach()))
        assert np.allclose(losses_a, losses_b, rtol=2e-3), (losses_a, losses_b)
        assert losses_b[-1] < losses_b[0]
        assert np.diff(seeds).tolist() == [1, 1, 1], seeds
        assert not torch.equal(dists[0], dists[1])
        # without jitter and with unchanged weights (lr = 0) consecutive replays see the same distances
        c = _model(jitter=False)
        seen.clear()
        step0 = _graphed(c, rays, lights, target, 0.0)
        step0(); d0 = seen["buf"].clone()
        step0(); d1 = seen["buf"].clone()
        assert c.sampling.seed is None and torch.equal(d0, d1)
    finally:
        config.set_train_precision("f32")


@pytest.mark.parametrize("prec", ["f32", "f16"])
def test_pathtrace_camera_frame_uses_the_sampling(prec):
    """pathtrace + NeRFReproduce with `sampling` set: one camera_rays launch per frame, and the frame equals ops.nerfle_render
    of ops.camera_rays' rays with the same sampling, bit for bit."""
    import torch
    import neural_raytracing_b200.pathtracer as P
    from neural_raytracing_b200 import config, ops
    from neural_raytracing_b200.pathtracer.cameras import NeRFCamera
    from neural_raytracing_b200.pathtracer.integrators import NeRFReproduce
    n = _model()
    _, lights = _scene(2, 1, 1)
    c2w, focal = synth.nerf_cameras(2, 16, device="cuda")
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cuda")
    try:
        config.set_precision(prec)
        ops.profile_collect()
        with torch.no_grad():
            img, extra = P.pathtrace(n, size=16, chunk_size=8, bundle_size=1, bsdf=None, integrator=NeRFReproduce(),
                                     lights=lights, cameras=cam, device="cuda", silent=True, with_noise=False)
        counts = {k: c for k, (_, c) in ops.profile_collect().items() if c}
        assert extra is None and counts.get("camera_rays") == 1, counts
        assert counts.get("sample_pdf", 0) >= 1, counts
        rays, view = ops.camera_rays(cam.device_desc(16, nx=16, ny=16), want_view=True)
        code, _ = _inputs(n, rays, lights)
        with torch.no_grad():
            ref = ops.nerfle_render(n.first.packed(), n.second.packed(), rays, None, code, view, prec=prec,
                                    **n._render_sampling())
            again = n(rays, lights)
    finally:
        config.set_precision("f32")
    assert torch.equal(img.reshape(-1), ref.mean(dim=-2).reshape(-1))
    assert torch.equal(again, ref)        # the gradient-free forward renders the same samples (render_seed)
