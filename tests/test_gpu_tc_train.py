"""GPU tests (-m gpu) of the tensor-core TRAINING path: forward that saves activation tiles, fused dgrad chain,
wgrad kernel (csrc/nrt_tc_train.cu), for the two NeRFLE networks.

Yardsticks (float64 torch autograd on the GPU):
  * "quantised reference": the same network with its weights and every activation rounded to fp16 the way the kernel
    rounds them (straight-through rounding).  leaky_relu has a kink at 0, so WHICH units sit on the 0.01 slope is
    decided by the forward's rounding; against a reference that rounds identically the kernels must agree tightly:
    cosine >= 0.9995 per parameter tensor.  This is the implementation-correctness gate.
  * exact reference (no rounding): the precision claim of the 16-bit path, SURVEY 8d's gate: cosine >= 0.999 per
    parameter tensor for both NeRFLE networks with fp16 operands (measured on B200: first >= 0.9994, second >= 0.9995,
    environment-light second >= 0.9994; the second MLP's Fourier phases come from a hi+lo split GEMM and the latent
    reaches it as fp32).  bf16 operands are 8x coarser (>= 0.995) and do not meet the gate: fp16 is the training mode.
"""
import numpy as np
import pytest

import helpers
import synth

pytestmark = pytest.mark.gpu


def _q(v):
    """straight-through fp16 rounding"""
    return v + (v.detach().half().double() - v.detach())


def _ref(w, x, out_act_sigmoid, quantised, split_inputs, softplus=False):
    import torch
    Ws = [torch.tensor(a, dtype=torch.float64, device="cuda") for a in w["W"]]
    bs = [torch.tensor(a, dtype=torch.float64, device="cuda", requires_grad=True) for a in w["b"]]
    if quantised:
        Ws = [a.half().double() for a in Ws]
    for a in Ws:
        a.requires_grad_()
    B = torch.tensor(w["basis"], dtype=torch.float64, device="cuda")
    x = x.double().requires_grad_()
    act = torch.nn.functional.softplus if softplus else torch.nn.functional.leaky_relu
    # Fourier phases keep ~fp32 accuracy for every network (fp32 FMAs for 3..5-D inputs, hi+lo split phase GEMM
    # otherwise); the raw inputs enter the init / skip layers as hi + lo columns (<= 5-D) or rounded once (wider)
    xq = _q(x) if (quantised and not split_inputs) else x
    ph = x @ B
    s, c = ph.sin(), ph.cos()
    if quantised:
        s, c = _q(s), _q(c)
    enc = torch.cat([xq, s, c], -1)
    enc_act = act(enc)
    if quantised:
        enc_act = torch.cat([enc_act[:, :x.shape[1]] if split_inputs else _q(enc_act[:, :x.shape[1]]), _q(enc_act[:, x.shape[1]:])], -1)
    h = enc @ Ws[0].t() + bs[0]
    L = w["num_layers"]
    for i in range(L):
        a = act(h)
        if quantised:
            a = _q(a)
        if i != L - 1 and i % w["skip"] == 0:
            a = torch.cat([a, enc_act], -1)
        h = a @ Ws[1 + i].t() + bs[1 + i]
    a = act(h)
    if quantised:
        a = _q(a)
    y = a @ Ws[-1].t() + bs[-1]
    if out_act_sigmoid:
        y = y.sigmoid()
    return y, x, Ws, bs


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a @ b) / (a.norm() * b.norm() + 1e-300))


LE_KW = dict(seed=33, in_size=115, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0)   # NeRFLE.second, envmap code


# the 256-wide nets (nrt_tc_train_wide.cu): sp_var_fn with 4 / 16 bases (bsdfs.py:487-496), LightField (lights.py:159-164)
WIDE_KW = {"sp_var4": dict(seed=41, in_size=3, out=4, num_layers=16, hidden=256, freqs=128, sigma=128.0),
           "sp_var16": dict(seed=42, in_size=3, out=16, num_layers=16, hidden=256, freqs=128, sigma=128.0),
           "light_field": dict(seed=43, in_size=3, out=3, num_layers=10, hidden=256, freqs=16, sigma=32.0)}
OCC_KW = dict(seed=18, in_size=5, out=1, num_layers=8, hidden=64, freqs=16, sigma=32.0)      # occlusion MLP (colocate.py:82-85)


@pytest.mark.parametrize("name,sig,need_x,gate_exact", [("nerf_first", False, False, 0.999), ("nerf_second", True, False, 0.999),
                                                        ("nerf_second", True, True, 0.999), ("nerf_second_le", True, True, 0.999),
                                                        ("neural_bsdf", True, True, 0.999), ("neural_bsdf", False, False, 0.999),
                                                        ("occ", True, True, 0.999),
                                                        # 16 layers of 16-bit rounding and 4,096 leaky_relu kinks (default init, not the
                                                        # reference's xavier): measured >= 0.9981 exact, >= 0.9993 quantised
                                                        ("sp_var4", True, False, 0.998), ("sp_var16", False, True, 0.998),
                                                        ("light_field", True, True, 0.999),
                                                        # SphereSDF.shift (softplus, no kinks): first-order path of sdf(best_pos)
                                                        ("sdf_shift", False, False, 0.9999)])
@pytest.mark.parametrize("M", [1, 129, 5000])
def test_tc_train_gradients(name, sig, need_x, gate_exact, M):
    import torch
    from neural_raytracing_b200 import ops
    kw = LE_KW if name == "nerf_second_le" else OCC_KW if name == "occ" else WIDE_KW[name] if name in WIDE_KW else \
        helpers.MLP_CASES[name][0]
    w = synth.mlp_weights(**kw)
    m = helpers.cuda_mlp(w, "softplus" if name == "sdf_shift" else None)
    out_act = ops.OUT_SIGMOID if sig else ops.OUT_NONE
    g = torch.Generator(device="cuda").manual_seed(M + 5)
    x = (0.6 if kw["in_size"] <= 5 else 0.1) * torch.randn(M, kw["in_size"], device="cuda", generator=g)
    gy = torch.randn(M, kw["out"], device="cuda", generator=g) * 3e-4    # realistic: small loss gradients
    out, ws = ops.mlp_forward_train_tc(m, x, out_act, prec="f16")
    gp, gx = ops.mlp_backward_tc(m, M, out, gy, ws, out_act, need_input_grad=need_x, prec="f16")
    gW, gb = m.unpack(gp)
    assert torch.isfinite(gp).all()
    for quantised, gate in ((True, 0.999 if name.startswith("sp_var") else 0.9995), (False, gate_exact)):
        y, xr, Ws, bs = _ref(w, x, sig, quantised, split_inputs=kw["in_size"] <= 5, softplus=name == "sdf_shift")
        (y * gy.double()).sum().backward()
        # (sdf_shift: the kernel's fp32 output layer sees the unrounded last activations, the quantised reference rounds them)
        assert float((out.double() - y.detach()).abs().max()) < (2e-4 if quantised and name != "sdf_shift" else 1e-3)
        if M < 100 and not quantised:
            continue   # a single sample: one flipped kink moves the cosine; the quantised gate still applies
        if M < 1000 and not quantised:
            gate = min(gate, 0.998)   # 129 samples: a few flipped kinks still move the cosine of the input-side layers
        for i, (a, b, ra, rb) in enumerate(zip(gW, gb, Ws, bs)):
            assert _cos(a, ra.grad) > gate, (name, "W", i, quantised, _cos(a, ra.grad))
            assert _cos(b, rb.grad) > gate, (name, "b", i, quantised, _cos(b, rb.grad))
            if quantised:
                scale = float(ra.grad.abs().max())
                # (256-wide nets: a kink that flips on one of few samples shows in single entries; the cosine gates above hold)
                assert float((a.double() - ra.grad).abs().max()) <= (0.15 if kw["hidden"] == 256 else 0.05) * scale + 1e-12
        if need_x:
            # d/dx of NeRFLE.second multiplies by the sigma = 32 basis (measured 0.9999)
            assert _cos(gx, xr.grad) > 0.999, (_cos(gx, xr.grad), quantised)


def test_tc_train_bf16_runs_and_is_coarser():
    import torch
    from neural_raytracing_b200 import ops
    kw, _ = helpers.MLP_CASES["nerf_first"]
    w = synth.mlp_weights(**kw)
    m = helpers.cuda_mlp(w)
    M = 4000
    g = torch.Generator(device="cuda").manual_seed(3)
    x = 0.6 * torch.randn(M, 3, device="cuda", generator=g)
    gy = torch.randn(M, 65, device="cuda", generator=g) * 1e-3
    y, xr, Ws, bs = _ref(w, x, False, False, True)
    (y * gy.double()).sum().backward()
    out, ws = ops.mlp_forward_train_tc(m, x, prec="bf16")
    gp, _ = ops.mlp_backward_tc(m, M, out, gy, ws, prec="bf16")
    gW, gb = m.unpack(gp)
    assert min(_cos(a, r.grad) for a, r in zip(gW, Ws)) > 0.98


def test_tc_train_loss_scale_handles_tiny_and_zero_gradients():
    """fp16 gradients: the device-side power-of-two loss scale keeps 1e-9-sized gradients exact in direction, and an
    all-zero upstream gradient gives exactly zero."""
    import torch
    from neural_raytracing_b200 import ops
    kw, _ = helpers.MLP_CASES["nerf_first"]
    m = helpers.cuda_mlp(synth.mlp_weights(**kw))
    M = 2000
    g = torch.Generator(device="cuda").manual_seed(4)
    x = 0.6 * torch.randn(M, 3, device="cuda", generator=g)
    gy = torch.randn(M, 65, device="cuda", generator=g)
    out, ws = ops.mlp_forward_train_tc(m, x)
    ga, _ = ops.mlp_backward_tc(m, M, out, gy, ws)
    out, ws = ops.mlp_forward_train_tc(m, x)
    gb, _ = ops.mlp_backward_tc(m, M, out, gy * 1e-9, ws)
    assert _cos(ga, gb) > 0.999999 and abs(float(gb.norm() / ga.norm()) / 1e-9 - 1) < 1e-3
    out, ws = ops.mlp_forward_train_tc(m, x)
    gz, _ = ops.mlp_backward_tc(m, M, out, gy * 0, ws)
    assert float(gz.abs().max()) == 0.0


def test_nerfle_training_step_tc_vs_fp32():
    """nerfle.py-style step (4 views x 16x16 crop, S = 64, mse): loss and parameter gradients of the tensor-core
    training path against the fused fp32 path."""
    import random
    import torch
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer.lights import PointLights
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    n = NeRFLE(device="cuda")
    synth.fill_module(n, 3)
    with torch.no_grad():
        n.first.out.bias[0] = 0.8     # positive density, otherwise relu(sigma) = 0 and every gradient vanishes
    rays = torch.from_numpy(synth.camera_rays(5, 4 * 16 * 16).reshape(4, 16, 16, 1, 6)).cuda()
    lights = PointLights(device="cuda", location=torch.randn(4, 3, device="cuda"), scale=10)
    target = torch.full((4, 16, 16, 1, 3), 0.5, device="cuda")
    res = {}
    try:
        for prec in ("f32", "f16"):
            config.set_train_precision(prec)
            random.seed(0)
            n.zero_grad()
            loss = torch.nn.functional.mse_loss(n(rays, lights), target)
            loss.backward()
            res[prec] = (float(loss.detach()), [p.grad.clone() for p in n.parameters()])
    finally:
        config.set_train_precision("f32")
    assert abs(res["f32"][0] - res["f16"][0]) < 1e-3 * max(1.0, abs(res["f32"][0]))
    cs = [_cos(a, b) for a, b in zip(res["f32"][1], res["f16"][1]) if float(b.norm()) > 0]
    assert min(cs) > 0.995 and float(np.median(cs)) > 0.9995, (min(cs), float(np.median(cs)))


def test_graphed_training_step_matches_eager():
    """CUDA-graph-captured NeRFLE step (training.GraphedStep) against the same steps run eagerly."""
    import copy
    import torch
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer.lights import PointLights
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    from neural_raytracing_b200.training import GraphedStep
    a = NeRFLE(device="cuda")
    synth.fill_module(a, 3)
    with torch.no_grad():
        a.first.out.bias[0] = 0.8
    b = copy.deepcopy(a)
    rays = torch.from_numpy(synth.camera_rays(5, 1024).reshape(1, 1024, 1, 1, 6)).cuda()
    lights = PointLights(device="cuda", location=torch.randn(1, 3, device="cuda"), scale=10)
    target = torch.full((1, 1024, 1, 1, 3), 0.5, device="cuda")
    jit = torch.full((1,), 0.37, device="cuda")
    a.far_jitter, b.far_jitter = jit, jit
    try:
        config.set_train_precision("f16")
        oa = torch.optim.AdamW(a.parameters(), lr=1e-3, weight_decay=0, capturable=True)
        ob = torch.optim.AdamW(b.parameters(), lr=1e-3, weight_decay=0, capturable=True)
        # GraphedStep runs 3 warm-up steps before capturing; do the same eagerly on the other copy
        step = GraphedStep(lambda: torch.nn.functional.mse_loss(b(rays, lights), target), ob, modules=[b], warmup=3)
        losses_b = [float(step().detach()) for _ in range(4)]
        losses_a = []
        for i in range(7):
            oa.zero_grad(set_to_none=True)
            loss = torch.nn.functional.mse_loss(a(rays, lights), target)
            loss.backward(); oa.step()
            if i >= 3:
                losses_a.append(float(loss.detach()))
    finally:
        config.set_train_precision("f32")
    assert np.allclose(losses_a, losses_b, rtol=2e-3), (losses_a, losses_b)
    assert losses_b[-1] < losses_b[0]      # it trains
    with torch.no_grad():
        ra, rb = a(rays, lights), b(rays, lights)
        eager_loss = float(torch.nn.functional.mse_loss(rb, target))
    # AdamW normalises the update, so last-bit gradient differences (atomics order) move individual weights; the two
    # trajectories stay close but not identical
    assert float((ra - rb).abs().max()) < 0.05
    # eager inference after the replays must see the UPDATED weights (the replays do not bump tensor versions; the
    # packed-parameter caches are invalidated by GraphedStep): its loss equals what the next replay computes
    next_loss = float(step().detach())
    assert abs(eager_loss - next_loss) < 2e-3 * max(1.0, next_loss), (eager_loss, next_loss, losses_b)


@pytest.mark.parametrize("envmap", [False, True])
@pytest.mark.parametrize("tprec,loss_tol,min_cos,min_cos_tensor", [("f32", 2e-5, 0.9999, 0.9999), ("f16", 1e-4, 0.9998, 0.997)])
def test_nerfle_training_step_vs_unmodified_reference(envmap, tprec, loss_tol, min_cos, min_cos_tensor):
    """Loss and the gradient of every Linear of a nerfle.py-style step (NeRFLE forward -> mse -> backward) against the
    fixture produced by the UNMODIFIED reference on CPU fp32 (tests/golden/make_golden.py::gen_nerfle_train).  Exact
    fp32 kernels: cosine >= 0.9999; tensor-core training kernels (fp16 operands): >= 0.9998 over all weights / all
    biases of an MLP (SURVEY 8d: 0.999), point-light and environment-light model alike, and per parameter tensor
    >= 0.999 everywhere except NeRFLE.first's init layer (35 inputs, 1 % of that MLP's gradient norm: 0.9977 / 0.9989;
    the forward's 16-bit rounding decides which leaky_relu kinks its few large contributions pass through)."""
    import random
    import torch
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer.lights import PointLights
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    g = helpers.golden("nerfle_train")
    tag = "le" if envmap else "pt"
    random.random = lambda: float(g["fixed_random"])
    n = NeRFLE(envmap=envmap, device="cuda")
    w1, w2 = helpers.nerfle_weights(envmap)
    for mod, w in ((n.first, w1), (n.second, w2)):
        mod.basis_p = torch.from_numpy(w["basis"]).cuda()
        for lin, W, b in zip([mod.init] + list(mod.layers) + [mod.out], w["W"], w["b"]):
            with torch.no_grad():
                lin.weight.copy_(torch.from_numpy(W)); lin.bias.copy_(torch.from_numpy(b))
    rays = torch.from_numpy(g[tag + "_rays"]).cuda()
    lights = PointLights(device="cuda", location=torch.from_numpy(g[tag + "_light_loc"]).cuda(), scale=10)
    target = torch.full(tuple(rays.shape[:-1]) + (3,), 0.5, device="cuda")
    try:
        config.set_train_precision(tprec)
        loss = torch.nn.functional.mse_loss(n(rays, lights), target)
        loss.backward()
    finally:
        config.set_train_precision("f32")
    ref_loss = float(g[tag + "_loss"])
    assert abs(float(loss.detach()) - ref_loss) <= loss_tol * max(1.0, ref_loss), (float(loss.detach()), ref_loss)
    for name, mod in (("first", n.first), ("second", n.second)):
        lins = [mod.init] + list(mod.layers) + [mod.out]
        gw = torch.cat([l.weight.grad.reshape(-1) for l in lins]).cpu().numpy().astype(np.float64)
        gb = torch.cat([l.bias.grad.reshape(-1) for l in lins]).cpu().numpy().astype(np.float64)
        for got, key, sizes in ((gw, "%s_g_%s_w" % (tag, name), [l.weight.numel() for l in lins]),
                                (gb, "%s_g_%s_b" % (tag, name), [l.bias.numel() for l in lins])):
            ref = synth.unpack_grad(g, key)
            cos = float(got @ ref / (np.linalg.norm(got) * np.linalg.norm(ref) + 1e-300))
            assert cos > min_cos, (key, tprec, cos)
            assert abs(np.linalg.norm(got) / float(g[key + "_norm"]) - 1) < (1e-3 if tprec == "f32" else 5e-3), key
            off = 0
            for i, k in enumerate(sizes):       # per parameter tensor
                a, b = got[off:off + k], ref[off:off + k]
                off += k
                c = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-300))
                gate = min_cos_tensor if (name == "first" and i == 0) else max(min_cos_tensor, 0.999)
                assert c > gate, (key, i, tprec, c)


def test_tc_train_large_weights_do_not_overflow():
    """A network whose layers amplify activations and gradients (weights 3x the default init: ~700x over the chain): the
    fp16 forward and data-gradient chain must stay finite (loss-scale head-room + saturating conversion) and agree with
    float64 autograd of the identically rounded network."""
    import torch
    from neural_raytracing_b200 import ops
    kw, _ = helpers.MLP_CASES["nerf_first"]
    w = synth.mlp_weights(**kw)
    w["W"] = [3.0 * a for a in w["W"]]
    m = helpers.cuda_mlp(w)
    M = 1500
    g = torch.Generator(device="cuda").manual_seed(8)
    x = 0.6 * torch.randn(M, 3, device="cuda", generator=g)
    gy = torch.randn(M, 65, device="cuda", generator=g)
    out, ws = ops.mlp_forward_train_tc(m, x)
    gp, _ = ops.mlp_backward_tc(m, M, out, gy, ws)
    assert torch.isfinite(out).all() and torch.isfinite(gp).all()
    y, xr, Ws, bs = _ref(w, x, False, True, True)
    (y * gy.double()).sum().backward()
    gW, gb = m.unpack(gp)
    assert min(_cos(a, r.grad) for a, r in zip(gW, Ws)) > 0.995


@pytest.mark.parametrize("K", [1, 32, 203, 3000])
def test_tc_value_jacobian_matches_double_backward(K):
    """nrt_mlp_value_jac_forward_tc / _backward_tc (SphereSDF.shift on the tensor cores: four rows per point, coupled
    softplus / sigmoid activation, shuffle-coupled reverse pass) vs FLOAT64 torch autograd: jac = autograd.grad(y, p,
    create_graph=True) and a loss on (y, jac) back-propagated into the weights -- the double backward the reference runs
    through SDF.autograd_diff (sdfs.py:184-197) for eikonal_loss (utils.py:294) and the shading normals."""
    import copy
    import torch
    import torch.nn.functional as F
    from neural_raytracing_b200 import ops
    from neural_raytracing_b200.pathtracer import neural_blocks as nb
    torch.manual_seed(0)
    mlp = nb.SkipConnMLP(device="cuda", in_size=3, out=1, num_layers=8, hidden_size=128, freqs=32, activation=F.softplus).to("cuda")
    synth.fill_module(mlp, 11)
    g = torch.Generator("cuda").manual_seed(K + 1)
    p = 0.5 * torch.randn(K, 3, device="cuda", generator=g)
    gv = torch.randn(K, 1, device="cuda", generator=g) * 1e-3
    gj = torch.randn(K, 1, 3, device="cuda", generator=g) * 1e-3
    pk = mlp.packed()
    val, jac, ws = ops.mlp_value_jac_forward_tc(pk, p, prec="f16")
    g_params = ops.mlp_value_jac_backward_tc(pk, K, ws, gv, gj, prec="f16")
    assert torch.isfinite(g_params).all()
    gW, gb = pk.unpack(g_params)
    m64 = copy.deepcopy(mlp).cpu().double()
    m64.basis_p = mlp.basis_p.detach().cpu().double()
    p64 = p.detach().cpu().double().requires_grad_()
    y64 = m64.forward_reference_ops(p64)
    j64, = torch.autograd.grad(y64[:, 0].sum(), p64, create_graph=True)
    scale_v, scale_j = y64.abs().max().item() + 1e-6, j64.abs().max().item() + 1e-6
    assert (val.cpu().double() - y64.detach()).abs().max().item() < 1e-3 * max(1.0, scale_v)
    assert (jac.cpu().double()[:, 0] - j64.detach()).abs().max().item() < 3e-3 * max(1.0, scale_j)
    assert _cos(jac[:, 0], j64.detach().cuda()) > 0.99999
    ((y64 * gv.cpu().double()).sum() + (j64 * gj.cpu().double()[:, 0]).sum()).backward()
    lin64 = [m64.init] + list(m64.layers) + [m64.out]
    for i, (w, b, l64) in enumerate(zip(gW, gb, lin64)):
        assert _cos(w, l64.weight.grad.cuda()) > 0.9995, ("W", i, _cos(w, l64.weight.grad.cuda()))
        assert _cos(b, l64.bias.grad.cuda()) > 0.9995, ("b", i, _cos(b, l64.bias.grad.cuda()))
