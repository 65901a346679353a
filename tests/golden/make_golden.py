"""Generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference/pytorch3d/pathtracer, imported through oracle/ref_shim.py) on CPU fp32.

Run in the build container only:   python tests/golden/make_golden.py
The fixtures pin the oracle (tests/test_oracle_vs_golden.py) and, through it, the CUDA path.
Every fixture stores the reference file:line of the function that produced it in `src`.
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
from oracle import ref_shim  # noqa: E402
import synth  # noqa: E402

pt = ref_shim.load()
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from pytorch3d.pathtracer.neural_blocks import SkipConnMLP  # noqa: E402
from pytorch3d.pathtracer.shapes.sdfs import SDF, SphereSDF  # noqa: E402
from pytorch3d.pathtracer.shapes.nerf import NeRFLE  # noqa: E402
from pytorch3d.pathtracer.lights import PointLights, LightField  # noqa: E402
from pytorch3d.pathtracer.bsdf import Diffuse, Conductor, NeuralBSDF, ComposeSpatialVarying  # noqa: E402
from pytorch3d.pathtracer.integrators import Direct, NeRFIntegrator, NeRFReproduce  # noqa: E402
from pytorch3d.pathtracer.interaction import coordinate_system, to_local  # noqa: E402
from pytorch3d.pathtracer.utils import param_rusin2, dir_to_elev_azim  # noqa: E402

torch.set_num_threads(8)
FIXED_RANDOM = 0.37  # value returned by the patched random.random (sdfs.py:236, nerf.py:178)


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def load_mlp(mod, w):
    """Copies synth weights into a reference SkipConnMLP (attribute assignment only)."""
    mod.basis_p = T(w["basis"]).clone()
    lins = [mod.init] + list(mod.layers) + [mod.out]
    assert len(lins) == len(w["W"])
    with torch.no_grad():
        for lin, W, b in zip(lins, w["W"], w["b"]):
            assert tuple(lin.weight.shape) == W.shape, (lin.weight.shape, W.shape)
            lin.weight.copy_(T(W))
            lin.bias.copy_(T(b))
    return mod


def ref_mlp(w, act=None):
    kw = {}
    if act == "softplus":
        kw["activation"] = F.softplus
    m = SkipConnMLP(num_layers=w["num_layers"], hidden_size=w["hidden"], in_size=w["in_size"],
                    out=w["out"], skip=w["skip"], freqs=w["freqs"], device="cpu",
                    latent_size=w["latent"], **kw)
    return load_mlp(m, w)


def ref_sdf(w, max_steps=64):
    s = SphereSDF(n=w["n"], device="cpu")
    with torch.no_grad():
        s.centers.copy_(T(w["centers"]))
        s.radii.copy_(T(w["radii"]))
        s.tfs.copy_(T(w["tfs"]))
    load_mlp(s.shift, w["shift"])
    return SDF(sdf=s, device="cpu", max_steps=max_steps), s


MLP_CASES = {
    # name: (synth kwargs, activation, M)
    "sdf_shift": (dict(seed=11, in_size=3, out=1, num_layers=8, hidden=128, freqs=32, sigma=32.0), "softplus", 130),
    "nerf_first": (dict(seed=12, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0), None, 257),
    "nerf_second": (dict(seed=13, in_size=70, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0), None, 200),
    "neural_bsdf": (dict(seed=14, in_size=3, out=3, num_layers=6, hidden=96, freqs=64, sigma=32.0), None, 100),
    "latent_small": (dict(seed=15, in_size=3, out=9, num_layers=5, hidden=32, freqs=16, sigma=32.0, latent=8), None, 77),
    "sp_var_small": (dict(seed=16, in_size=3, out=4, num_layers=7, hidden=256, freqs=128, sigma=128.0), None, 70),
    "one_layer": (dict(seed=17, in_size=5, out=1, num_layers=1, hidden=64, freqs=16, sigma=32.0), None, 64),
}


def gen_mlp():
    out = {}
    for name, (kw, act, M) in MLP_CASES.items():
        w = synth.mlp_weights(**kw)
        m = ref_mlp(w, act)
        rs = np.random.RandomState(kw["seed"] + 100)
        x = (0.6 * rs.standard_normal((M, kw["in_size"]))).astype(np.float32)
        lat = (0.5 * rs.standard_normal((M, kw.get("latent", 0)))).astype(np.float32) if kw.get("latent", 0) else None
        with torch.no_grad():
            y = m(T(x), T(lat) if lat is not None else None).numpy()
        out[name + "_x"] = x
        if lat is not None:
            out[name + "_latent"] = lat
        out[name + "_y"] = y
    out["src"] = np.array("neural_blocks.py:75-86 SkipConnMLP.forward; utils.py:37-40 fourier2")
    np.savez_compressed(os.path.join(HERE, "mlp.npz"), **out)
    print("mlp.npz", {k: v.shape for k, v in out.items() if k != "src"})


def gen_sdf():
    w = synth.sdf_weights(seed=21)
    sdf, sphere = ref_sdf(w, max_steps=64)
    rays = synth.camera_rays(22, 384)
    rays[:8, 3:] = -rays[:8, 3:]          # a few rays pointing away: guaranteed misses
    rs = np.random.RandomState(23)
    pts = (0.5 * rs.standard_normal((300, 3))).astype(np.float32)
    random.random = lambda: FIXED_RANDOM
    out = {}
    with torch.no_grad():
        out["pts"] = pts
        out["sdf_vals"] = sphere(T(pts)).numpy()
    r5 = T(rays).reshape(1, 384, 1, 1, 6)
    si, active = sdf.intersect(r5, max_t=10, primary=True)
    out["rays"] = rays
    out["hit"] = active.reshape(-1).numpy()
    out["depth"] = si.t.detach().reshape(-1).numpy()
    out["throughput"] = si.throughput.detach().reshape(-1).numpy()       # = -1000 * sdf(best_pos)
    out["p_after"] = si.p.detach().reshape(-1, 3).numpy()                 # hit points pushed along n
    out["normals"] = si.n.detach().reshape(-1, 3).numpy()
    out["raw_normals"] = si.raw_normals.detach().numpy()
    out["frame"] = si.frame.detach().reshape(-1, 3, 3).numpy()
    out["wi"] = si.wi.detach().reshape(-1, 3).numpy()
    # the min scan internals (sdfs.py:232-249), re-run to expose idx/best_pos
    thr, best_pos = sdf.throughput(r5[..., :3], r5[..., 3:])
    out["best_pos"] = best_pos.detach().reshape(-1, 3).numpy()
    out["scan_dist"] = np.array(sdf.dist, np.float64)
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    # shadow rays from the hit points towards a point light (scene.py:290-299)
    light = torch.tensor([[0.3, 1.1, 0.2]])
    d = light[:, None, None, None, :] - si.p.detach()
    dist = torch.linalg.norm(d, dim=-1, keepdim=True)
    d = F.normalize(d, eps=1e-6, dim=-1)
    srays = torch.cat([si.p.detach(), d], dim=-1)
    with torch.no_grad():
        nb = sdf.intersect_test(srays, max_t=dist.reshape_as(active)[..., None])
    out["shadow_rays"] = srays.reshape(-1, 6).numpy()
    out["shadow_max_t"] = dist.reshape(-1).numpy()
    out["not_blocked"] = nb.reshape(-1).numpy()
    # value + autograd gradient at arbitrary points (sdfs.py:184-197)
    g = sdf.autograd_diff(T(pts[:96]).clone())
    out["grad_pts"] = g.detach().numpy()
    out["src"] = np.array("shapes/sdfs.py:37-46,111-160,162-181,184-197,232-249; interaction.py:9-41")
    np.savez_compressed(os.path.join(HERE, "sdf.npz"), **out)
    print("sdf.npz hits", int(out["hit"].sum()), "of", len(out["hit"]), "not_blocked", int(out["not_blocked"].sum()))


def gen_nerfle():
    out = {}
    random.random = lambda: FIXED_RANDOM
    for tag, envmap in (("pt", False), ("le", True)):
        n = NeRFLE(envmap=envmap, device="cpu")
        w1 = synth.mlp_weights(seed=31, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0)
        in2 = 64 + (6 if not envmap else 3 + 16 * 3)
        w2 = synth.mlp_weights(seed=32 + envmap, in_size=in2, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0)
        # make densities non-trivial: bias the sigma output channel upwards
        w1["b"][-1][0] = 0.8
        load_mlp(n.first, w1)
        load_mlp(n.second, w2)
        N, Wd, Hd = 2, 6, 4
        rays = synth.camera_rays(33, N * Wd * Hd).reshape(N, Wd, Hd, 1, 6)
        loc = np.array([[0.4, 1.0, 0.3], [-0.8, 0.5, 0.6]], np.float32)
        lights = PointLights(device="cpu", location=T(loc), scale=10)
        with torch.no_grad():
            rgb = n(T(rays), lights)
        out[tag + "_rays"] = rays
        out[tag + "_light_loc"] = loc
        out[tag + "_rgb"] = rgb.numpy()
        if envmap:
            # the 48-float light code of nerf.py:184-195
            from pytorch3d.pathtracer.utils import elev_azim_to_dir
            points = torch.stack(torch.meshgrid(torch.linspace(0, 180, 4), torch.linspace(0, 45, 4)), dim=-1).reshape(-1, 2)
            with torch.no_grad():
                out[tag + "_light_code"] = lights.envmap(elev_azim_to_dir(points)).reshape(N, -1).numpy()
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("shapes/nerf.py:175-214 NeRFLE.forward; lights/lights.py:81-88 envmap")
    np.savez_compressed(os.path.join(HERE, "nerfle.npz"), **out)
    print("nerfle.npz rgb mean", float(out["pt_rgb"].mean()), float(out["le_rgb"].mean()))


def gen_nerfle_train():
    """nerfle.py:104-116-style step on the UNMODIFIED reference: NeRFLE forward -> mse -> backward.  Stores the loss and
    the gradient of every Linear (flattened in module order, synth.pack_grad, with its float64 norm as `<key>_norm`)
    for the point-light and the environment-light model."""
    out = {}
    random.random = lambda: FIXED_RANDOM
    for tag, envmap in (("pt", False), ("le", True)):
        n = NeRFLE(envmap=envmap, device="cpu")
        w1 = synth.mlp_weights(seed=31, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0)
        in2 = 64 + (6 if not envmap else 3 + 16 * 3)
        w2 = synth.mlp_weights(seed=32 + envmap, in_size=in2, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0)
        w1["b"][-1][0] = 0.8
        load_mlp(n.first, w1)
        load_mlp(n.second, w2)
        N, Wd, Hd = 2, 16, 12
        rays = synth.camera_rays(35, N * Wd * Hd).reshape(N, Wd, Hd, 1, 6)
        loc = np.array([[0.4, 1.0, 0.3], [-0.8, 0.5, 0.6]], np.float32)
        lights = PointLights(device="cpu", location=T(loc), scale=10)
        target = torch.full((N, Wd, Hd, 1, 3), 0.5)
        rgb = n(T(rays), lights)
        loss = F.mse_loss(rgb, target)           # nerfle.py:113
        loss.backward()
        out[tag + "_rays"] = rays
        out[tag + "_light_loc"] = loc
        out[tag + "_loss"] = np.array(loss.item(), np.float64)
        out[tag + "_rgb"] = rgb.detach().numpy()
        for name, mod in (("first", n.first), ("second", n.second)):
            lins = [mod.init] + list(mod.layers) + [mod.out]
            for kind in ("w", "b"):
                key = "%s_g_%s_%s" % (tag, name, kind)
                grad = np.concatenate([(l.weight if kind == "w" else l.bias).grad.numpy().ravel() for l in lins])
                out[key], out[key + "_scale"] = synth.pack_grad(grad)
                out[key + "_norm"] = np.array(np.linalg.norm(grad.astype(np.float64)), np.float64)
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("shapes/nerf.py:175-214 NeRFLE.forward + torch autograd of F.mse_loss (scripts/nerfle.py:113-116)")
    np.savez_compressed(os.path.join(HERE, "nerfle_train.npz"), **out)
    print("nerfle_train.npz: loss pt %.6f le %.6f, |g first| %.3e" % (out["pt_loss"], out["le_loss"],
                                                                      out["pt_g_first_w_norm"]))


def gen_composite():
    rs = np.random.RandomState(41)
    out = {}
    for tag, S, R in (("s64", 64, 50), ("s5", 5, 7), ("s1", 1, 3)):
        sigma = (2.0 * rs.standard_normal((S, R))).astype(np.float32)
        rgb = rs.uniform(size=(S, R, 3)).astype(np.float32)
        ts = np.linspace(0, 2.037, S).astype(np.float32) if S > 1 else np.array([0.7], np.float32)
        sg = T(sigma).clone().requires_grad_(True)
        cg = T(rgb).clone().requires_grad_(True)
        tt = T(ts)
        # nerf.py:205-213 verbatim semantics
        sigma_a = F.relu(sg)
        alpha = 1 - torch.exp(-sigma_a * tt[:, None].expand_as(sigma_a))
        cp = torch.cumprod((1 - alpha).clamp(min=1e-10), dim=0)
        cp = torch.roll(cp, 1, 0)
        cp[-1, ...] = 1
        weights = alpha * cp
        res = (weights[..., None] * cg).sum(dim=0)
        go = T(rs.standard_normal((R, 3)).astype(np.float32))
        res.backward(go)
        out.update({tag + "_sigma": sigma, tag + "_rgb": rgb, tag + "_ts": ts, tag + "_out": res.detach().numpy(),
                    tag + "_gout": go.numpy(), tag + "_gsigma": sg.grad.numpy(), tag + "_grgb": cg.grad.numpy()})
    out["src"] = np.array("shapes/nerf.py:205-213")
    np.savez_compressed(os.path.join(HERE, "composite.npz"), **out)
    print("composite.npz ok")


def gen_shading():
    rs = np.random.RandomState(51)
    out = {}
    n = rs.standard_normal((64, 3)).astype(np.float32)
    n[:4] = 0.0                      # zero normals (missed rays) go through the same code
    n[4] = [0, 0, -1]; n[5] = [0, 0, 1]
    v = rs.standard_normal((64, 3)).astype(np.float32)
    frame = coordinate_system(T(n))
    out["n"] = n; out["v"] = v
    out["frame"] = frame.numpy()
    out["to_local"] = to_local(frame, T(v)).numpy()
    a = rs.standard_normal((64, 3)).astype(np.float32); b = rs.standard_normal((64, 3)).astype(np.float32)
    a[0] = [0, 0, 1]; b[0] = [0, 0, 1]
    out["rusin_a"] = a; out["rusin_b"] = b
    out["rusin"] = param_rusin2(T(a), T(b)).numpy()
    out["elev_azim"] = dir_to_elev_azim(T(v)).numpy()
    out["src"] = np.array("interaction.py:9-41; utils.py:233-258,490-494")
    np.savez_compressed(os.path.join(HERE, "shading.npz"), **out)
    print("shading.npz ok")


def gen_lights_bsdf():
    """a9 / a14: PointLights.sample_direction (lights.py:89-110), Diffuse.eval_and_pdf (bsdfs.py:108-118) with the three
    preprocess functions the scripts use, Conductor.eval_and_pdf (bsdfs.py:364-388), each with the gradients of a fixed
    scalar loss to every leaf the scripts optimise (PYTORCH_JIT=0 in the shim: Conductor.eta DOES receive a gradient)."""
    from types import SimpleNamespace
    from pytorch3d.pathtracer.bsdf.bsdfs import identity_div_pi
    rs = np.random.RandomState(77)
    out = {}
    N, W, H = 2, 6, 5
    p = (0.6 * rs.standard_normal((N, W, H, 1, 3))).astype(np.float32)
    active = rs.uniform(size=(N, W, H, 1)) > 0.3
    wgt = rs.standard_normal((N, W, H, 1, 3)).astype(np.float32)           # dL/dspectrum
    wgt_d = rs.standard_normal((N, W, H, 1, 3)).astype(np.float32)         # dL/dd
    out.update(p=p, active=active, wgt=wgt, wgt_d=wgt_d)
    loc = np.array([[0.3, 1.2, 0.4], [-0.8, 0.5, 1.1]], np.float32)
    lights = PointLights(device="cpu", scale=5.0, intensity=[0.9, 0.7, 0.8], location=loc.tolist(), const=0.3, linear=0.05, square=0.7)
    lights.location = T(loc).clone().requires_grad_(True)
    pt_ = T(p).clone().requires_grad_(True)
    ds, spec = lights.sample_direction(SimpleNamespace(p=pt_), None, T(active))
    loss = (spec * T(wgt)).sum() + (ds.d * T(wgt_d)).sum() + 0.1 * ds.dist.sum()
    loss.backward()
    out.update(light_loc=loc, pl_d=ds.d.detach().numpy(), pl_dist=ds.dist.detach().numpy(), pl_spectrum=spec.detach().numpy(),
               pl_g_p=pt_.grad.numpy(), pl_g_location=lights.location.grad.numpy(), pl_g_intensity=lights.intensity.grad.numpy(),
               pl_g_scale=lights.scale.grad.numpy(), pl_g_const=lights.const.grad.numpy(), pl_g_linear=lights.linear.grad.numpy(),
               pl_g_square=lights.square.grad.numpy())
    # local directions
    wi = rs.standard_normal((N, W, H, 1, 3)).astype(np.float32); wi /= np.linalg.norm(wi, axis=-1, keepdims=True)
    wo = rs.standard_normal((N, W, H, 1, 3)).astype(np.float32); wo /= np.linalg.norm(wo, axis=-1, keepdims=True)
    # a few mirror configurations so that the conductor lobe (reflect(wi) . wo > 0.94) is hit
    for j in range(8):
        wo[0, j % W, j % H, 0] = wi[0, j % W, j % H, 0] * np.array([-1, -1, 1], np.float32)
    out.update(wi=wi, wo=wo)
    refl = rs.uniform(0.05, 0.95, 3).astype(np.float32)
    out["reflectance"] = refl
    for name, pre in (("div_pi", identity_div_pi), ("softplus", torch.nn.Softplus()), ("sigmoid", torch.sigmoid)):
        d = Diffuse(reflectance=refl.tolist(), preprocess=pre, device="cpu")
        wo_t = T(wo).clone().requires_grad_(True)
        spec, pdf = d.eval_and_pdf(SimpleNamespace(wi=T(wi), p=T(p)), wo_t, T(active))
        ((spec * T(wgt)).sum() + pdf.sum()).backward()
        out["df_%s_spectrum" % name] = spec.detach().numpy(); out["df_%s_pdf" % name] = pdf.detach().numpy()
        out["df_%s_g_reflectance" % name] = d.reflectance.grad.numpy(); out["df_%s_g_wo" % name] = wo_t.grad.numpy()
    spc = rs.uniform(-1, 1, 3).astype(np.float32)
    out["specular"] = spc
    for name, act in (("sigmoid", torch.sigmoid), ("softplus", torch.nn.Softplus())):
        c = Conductor(specular=spc.tolist(), eta=1.3, k=1.0, device="cpu", activation=act)
        wi_t = T(wi).clone().requires_grad_(True)
        spec, pdf = c.eval_and_pdf(SimpleNamespace(wi=wi_t, p=T(p)), T(wo), T(active))
        (spec * T(wgt)).sum().backward()
        out["cd_%s_spectrum" % name] = spec.detach().numpy(); out["cd_%s_pdf" % name] = pdf.detach().numpy()
        out["cd_%s_g_specular" % name] = c.specular.grad.numpy(); out["cd_%s_g_wi" % name] = wi_t.grad.numpy()
        out["cd_%s_g_eta" % name] = np.float32(0.0) if c.eta.grad is None else c.eta.grad.numpy()
        out["cd_%s_eta_has_grad" % name] = np.bool_(c.eta.grad is not None)
        out["cd_%s_k_has_grad" % name] = np.bool_(c.k.grad is not None)
    out["lobe_pixels"] = np.int64(int((out["cd_sigmoid_pdf"] > 0).sum()))
    out["src"] = np.array("lights.py:89-110; bsdfs.py:108-118, 327-341, 364-388 (PYTORCH_JIT=0)")
    np.savez_compressed(os.path.join(HERE, "lights_bsdf.npz"), **out)
    print("lights_bsdf.npz ok, conductor lobe pixels:", int(out["lobe_pixels"]), "eta grad:", bool(out["cd_sigmoid_eta_has_grad"]))


from scenes import build_pipeline  # noqa: E402


def gen_pipeline():
    """Full reference renders: colocate-style pathtrace (main.py:13-93 + integrators.py:156-206 + scene.py:301-318)
    and a DTU-style pathtrace_sample with LightField + eikonal/BCE-style gradients."""
    import pytorch3d.pathtracer as P
    import pytorch3d.pathtracer.shapes.sdfs, pytorch3d.pathtracer.bsdf, pytorch3d.pathtracer.lights  # noqa: F401
    import pytorch3d.pathtracer.integrators, pytorch3d.pathtracer.neural_blocks, pytorch3d.pathtracer.cameras  # noqa: F401
    from pytorch3d.pathtracer.cameras import NeRFCamera
    from pytorch3d.pathtracer.utils import eikonal_loss
    out = {}
    random.random = lambda: FIXED_RANDOM
    size = 16
    c2w, focal = synth.nerf_cameras(1, size)
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cpu")
    # ---- colocate-style forward
    shape, sphere, bsdf, lights, integrator, w_isect = build_pipeline(P, "colocate")
    with torch.no_grad():
        img, mi = P.pathtrace(shape, size=size, chunk_size=size, bundle_size=1, bsdf=bsdf, integrator=integrator,
                              lights=lights, cameras=cam, device="cpu", silent=True, background=0, w_isect=w_isect,
                              with_noise=False, addition=lambda it: it)
    out["colocate_img"] = img.numpy()
    out["colocate_throughput"] = mi.throughput.reshape(-1).numpy()
    out["colocate_weights"] = mi.normalized_weights.reshape(-1, 4).numpy()
    out["colocate_raw_normals"] = mi.raw_normals.detach().numpy()
    # ---- DTU-style forward + backward
    shape, sphere, bsdf, lights, integrator, w_isect = build_pipeline(P, "dtu")
    c2w2, focal2 = synth.nerf_cameras(2, size)
    cam2 = NeRFCamera(cam_to_world=c2w2, focal=focal2, device="cpu")
    got, mi = P.pathtrace_sample(shape, size=size, chunk_size=size, bundle_size=1, crop_size=8, uv=(3, 5), bsdf=bsdf,
                                 integrator=integrator, lights=lights, cameras=cam2, device="cpu", silent=True,
                                 background=0, w_isect=w_isect, with_noise=False, addition=lambda it: it,
                                 squeeze_first=False)
    out["dtu_img"] = got.detach().numpy()
    out["dtu_throughput"] = mi.throughput.detach().reshape(-1).numpy()
    loss = (got[..., :3] - 0.5).square().mean() + 0.1 * eikonal_loss(mi.raw_normals) + \
        torch.nn.functional.binary_cross_entropy_with_logits(mi.throughput.reshape(-1), torch.ones(mi.throughput.numel()) * 0.5)
    loss.backward()
    out["dtu_loss"] = np.array(loss.item(), np.float64)
    out["dtu_g_sdf_out_w"] = sphere.shift.out.weight.grad.numpy()
    out["dtu_g_sdf_l3_w"] = sphere.shift.layers[3].weight.grad.numpy()
    out["dtu_g_centers"] = sphere.centers.grad.numpy()
    out["dtu_g_bsdf0_init_w"] = bsdf.bsdfs[0].mlp.init.weight.grad.numpy()
    out["dtu_g_spvar_out_w"] = bsdf.sp_var_fn.out.weight.grad.numpy()
    out["dtu_g_light_out_w"] = lights.light_field_approx.out.weight.grad.numpy()
    out["dtu_g_light_color"] = lights.color.grad.numpy()
    out["dtu_g_reflectance"] = bsdf.bsdfs[2].reflectance.grad.numpy()
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("main.py:13-179; integrators/integrators.py:156-257; scene.py:290-324; bsdf/bsdfs.py; lights/lights.py")
    np.savez_compressed(os.path.join(HERE, "pipeline.npz"), **out)
    print("pipeline.npz: colocate img mean %.4f hits %d; dtu loss %.5f" % (out["colocate_img"].mean(), len(out["colocate_raw_normals"]), loss.item()))


def gen_cameras():
    """look_at_view_transform + OpenGLPerspectiveCameras.sample_positions as colocate.py:54-56 / nerfle.py:96 /
    training_utils.py:198 use them (renderer/cameras.py:539-575, 1313-1422)."""
    from pytorch3d.renderer import OpenGLPerspectiveCameras, look_at_view_transform
    from pytorch3d.pathtracer.samplers import Sampler
    out = {}
    elev = torch.linspace(0, 45, 5)
    azim = torch.linspace(-90, 90, 5)
    R, Tt = look_at_view_transform(dist=1.0, elev=elev, azim=azim)
    out["elev"], out["azim"], out["R"], out["T"] = elev.numpy(), azim.numpy(), R.numpy(), Tt.numpy()
    R2, T2 = look_at_view_transform(dist=2.7, elev=30.0, azim=200.0, at=((0.1, -0.2, 0.05),))
    out["R2"], out["T2"] = R2.numpy(), T2.numpy()
    R3, T3 = look_at_view_transform(eye=((0.0, 1.5, 0.0), (0.4, 0.3, -1.0)), at=((0.0, 0.0, 0.0),))   # first one: up || view
    out["R3"], out["T3"] = R3.numpy(), T3.numpy()
    cams = OpenGLPerspectiveCameras(device="cpu", R=R, T=Tt)
    out["centers"] = cams.get_camera_center().numpy()
    size = 16
    gx, gy = torch.meshgrid(torch.arange(4, 12, dtype=torch.float), torch.arange(2, 10, dtype=torch.float))
    pos = torch.stack([gy, gx], dim=-1)
    out["positions"] = pos.numpy()
    rays = cams.sample_positions(pos, Sampler(device="cpu"), bundle_size=2, size=size, N=len(cams), with_noise=False)
    out["rays"] = rays.numpy()
    cam1 = OpenGLPerspectiveCameras(device="cpu", R=R2, T=T2, fov=45.0, znear=0.5, zfar=20.0)
    out["rays_fov45"] = cam1.sample_positions(pos, Sampler(device="cpu"), bundle_size=1, size=size, N=1, with_noise=False).numpy()
    out["center_fov45"] = cam1.get_camera_center().numpy()
    out["src"] = np.array("pytorch3d/renderer/cameras.py:125-150, 539-575, 1284-1422")
    np.savez_compressed(os.path.join(HERE, "cameras.npz"), **out)
    print("cameras.npz: rays", out["rays"].shape, "dir norm", np.linalg.norm(out["rays"][..., 3:], axis=-1).mean())


def gen_camera_rays():
    """f4 fixtures: rays of NeRFCamera / DTUCamera on a pixel window (cameras.py:23-54, 132-192), and the reference's
    own pathtrace of a NeRFLE under NeRFReproduce through a NeRFCamera and through OpenGLPerspectiveCameras
    (main.py:13-93; nerfle.py:130-135 is this call) -- what the camera-driven whole-frame render must reproduce."""
    import scenes
    from pytorch3d.pathtracer.cameras import NeRFCamera, DTUCamera
    from pytorch3d.pathtracer.integrators import NeRFReproduce
    from pytorch3d.pathtracer.samplers import Sampler
    from pytorch3d.renderer import OpenGLPerspectiveCameras, look_at_view_transform
    import pytorch3d.pathtracer as P
    out = {}
    size = 16
    gx, gy = torch.meshgrid(torch.arange(3, 13, dtype=torch.float), torch.arange(2, 8, dtype=torch.float))
    pos = torch.stack([gy, gx], dim=-1)                      # window x0 = 3, y0 = 2, nx = 10, ny = 6
    out["window"] = np.array([3, 2, 10, 6], np.int32)
    c2w, focal = synth.nerf_cameras(3, size)
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cpu")
    out["nerf_rays"] = cam.sample_positions(pos, Sampler(device="cpu"), bundle_size=1, size=size, N=3, with_noise=False).numpy()
    pose, K = scenes.dtu_cameras(2, device="cpu")
    dcam = DTUCamera(pose=pose, intrinsic=K, device="cpu")
    out["dtu_rays"] = dcam.sample_positions(pos, Sampler(device="cpu"), bundle_size=2, size=size, N=2, with_noise=False).numpy()
    # whole frames of a NeRFLE
    random.random = lambda: FIXED_RANDOM
    n = NeRFLE(envmap=False, device="cpu")
    w1 = synth.mlp_weights(seed=31, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0)
    w2 = synth.mlp_weights(seed=32, in_size=70, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0)
    w1["b"][-1][0] = 0.8
    load_mlp(n.first, w1)
    load_mlp(n.second, w2)
    loc = np.array([[0.4, 1.0, 0.3], [-0.8, 0.5, 0.6]], np.float32)
    lights = PointLights(device="cpu", location=T(loc), scale=10)
    cam2 = NeRFCamera(cam_to_world=c2w[:2], focal=focal, device="cpu")
    with torch.no_grad():
        img, _ = P.pathtrace(n, size=size, chunk_size=8, bundle_size=1, bsdf=None, integrator=NeRFReproduce(),
                             lights=lights, cameras=cam2, device="cpu", silent=True, with_noise=False)
        R, Tt = look_at_view_transform(dist=1.6, elev=torch.tensor([20.0, 35.0]), azim=torch.tensor([-40.0, 70.0]))
        fcam = OpenGLPerspectiveCameras(device="cpu", R=R, T=Tt)
        img_f, _ = P.pathtrace(n, size=size, chunk_size=8, bundle_size=2, bsdf=None, integrator=NeRFReproduce(),
                               lights=lights, cameras=fcam, device="cpu", silent=True, with_noise=False)
    out["light_loc"] = loc
    out["frame_nerf"], out["frame_fov"] = img.numpy(), img_f.numpy()
    out["fov_R"], out["fov_T"] = R.numpy(), Tt.numpy()
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("pathtracer/cameras/cameras.py:23-54, 132-192; pathtracer/main.py:13-93; shapes/nerf.py:175-214")
    np.savez_compressed(os.path.join(HERE, "camera_rays.npz"), **out)
    print("camera_rays.npz:", out["nerf_rays"].shape, out["dtu_rays"].shape, out["frame_nerf"].shape, out["frame_fov"].shape,
          "frame means %.4f %.4f" % (img.mean(), img_f.mean()))


def gen_vis():
    """The visualisation integrators of dtu_vis.py / nerv_vis.py / visualize.py on the pipeline test scenes
    (integrators.py:25-136): BasisBRDF weight map, Debug normals, Depth, Illumination, Luminance."""
    import pytorch3d.pathtracer as P
    from pytorch3d.pathtracer.cameras import NeRFCamera
    from pytorch3d.pathtracer.integrators import BasisBRDF, Debug, Depth, Illumination, Luminance, Mask
    from scenes import build_pipeline
    out = {}
    random.random = lambda: FIXED_RANDOM
    size = 16
    c2w, focal = synth.nerf_cameras(1, size)
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cpu")

    def render(scene, integrator):
        shape, sphere, bsdf, lights, _integ, _w = build_pipeline(P, scene)
        integ = integrator(bsdf)
        with torch.no_grad():
            img, _ = P.pathtrace(shape, size=size, chunk_size=size, bundle_size=1, bsdf=bsdf, integrator=integ,
                                 lights=lights, cameras=cam, device="cpu", silent=True, background=0, with_noise=False)
        return img.numpy()
    out["dtu_basis"] = render("dtu", lambda b: BasisBRDF(b))
    out["dtu_debug_mask"] = render("dtu", lambda b: Mask(Debug()))
    out["dtu_depth"] = render("dtu", lambda b: Depth())
    out["colocate_basis"] = render("colocate", lambda b: BasisBRDF(b))
    out["colocate_illumination"] = render("colocate", lambda b: Illumination())
    out["colocate_luminance"] = render("colocate", lambda b: Luminance())
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("pytorch3d/pathtracer/integrators/integrators.py:25-136")
    np.savez_compressed(os.path.join(HERE, "vis.npz"), **out)
    print("vis.npz:", {k: (v.shape, float(np.mean(v))) for k, v in out.items() if hasattr(v, "shape") and v.ndim > 1})


def gen_sphere_examples():
    """utils.sphere_examples (utils.py:409-431) as dtu_vis.py:108 / nerv_vis.py / visualize.py call it: every basis of the
    spatially varying BSDF on the analytic unit sphere (shapes/shapes.py:31-68) under the fork's renderer.PointLights
    (renderer/lighting.py:289-305), Direct lighting; plus depth_image (utils.py:441-445).  pathtrace's default pixel jitter
    (1e-3 pixel) stays on, as in the scripts: the fixture is compared with a tolerance that covers it."""
    import pytorch3d.pathtracer as P
    from pytorch3d.pathtracer.utils import sphere_examples, depth_image
    from pytorch3d.pathtracer.shapes.shapes import Sphere
    from scenes import build_pipeline
    out = {}
    _shape, _sphere, bsdf, _lights, _integ, _w = build_pipeline(P, "dtu")
    with torch.no_grad():
        imgs = sphere_examples(bsdf, device="cpu", size=24, chunk_size=12, scale=100)
    out["bases"] = np.stack([i.numpy() for i in imgs])
    rays = T(synth.camera_rays(91, 300))
    rays[:, :3] *= 2.5
    ball = Sphere([0.1, -0.2, 0.05], 0.8, device="cpu")
    si, hit = ball.intersect(rays.clone())
    out["rays"], out["hit"], out["t"], out["p"], out["n"], out["wi"] = rays.numpy(), hit.numpy(), si.t.numpy(), si.p.numpy(), si.n.numpy(), si.wi.numpy()
    lo, hi, m = ball.intersect_limits(rays.clone())
    out["lo"], out["hi"] = lo.numpy(), hi.numpy()
    d = torch.rand(5, 7, 2) + 0.1
    out["depth_in"], out["depth_out"] = d.numpy(), depth_image(d).numpy()
    out["src"] = np.array("pytorch3d/pathtracer/utils.py:409-445; shapes/shapes.py:9-97; renderer/lighting.py:220-305")
    np.savez_compressed(os.path.join(HERE, "sphere_examples.npz"), **out)
    print("sphere_examples.npz:", out["bases"].shape, out["bases"].mean(axis=(1, 2, 3)), "hits", int(hit.sum()), "of", len(hit))


def gen_dataset_loaders():
    """training_utils.test_nerf_resources / test_colocate_resources (training_utils.py:538-595) on the miniature datasets of
    tests/golden/tiny_datasets.py: what the reference's loaders return for them."""
    import tempfile
    import tiny_datasets
    from pytorch3d.pathtracer.training_utils import test_nerf_resources, test_colocate_resources
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        d = tiny_datasets.write_nerf_synthetic(os.path.join(tmp, "lego")) + os.sep
        c2w, focal, imgs, masks = test_nerf_resources(d, size=8, kind="test", device="cpu")
        out["nerf_c2w"], out["nerf_focal"] = torch.stack(c2w).numpy(), np.array(focal, np.float64)
        out["nerf_imgs"], out["nerf_masks"] = torch.stack(imgs).numpy(), torch.stack(masks).numpy()
        cwd = os.getcwd()
        os.chdir(tmp)
        try:
            tiny_datasets.write_colocate(os.path.join("mitsuba_scenes", "cbox_relight"), "bunny")
            Rs, Ts, imgs, masks, xyzs = test_colocate_resources("bunny", size=4, dist=1.3, device="cpu")
        finally:
            os.chdir(cwd)
        out["col_R"], out["col_T"] = torch.cat(Rs).numpy(), torch.cat(Ts).numpy()
        out["col_imgs"], out["col_masks"], out["col_xyz"] = torch.stack(imgs).numpy(), torch.stack(masks).numpy(), torch.stack(xyzs).numpy()
    out["src"] = np.array("pytorch3d/pathtracer/training_utils.py:538-595; utils.py:365-369")
    np.savez_compressed(os.path.join(HERE, "dataset_loaders.npz"), **out)
    print("dataset_loaders.npz:", out["nerf_c2w"].shape, float(out["nerf_focal"]), out["col_R"].shape, out["col_xyz"].shape,
          "mask values", np.unique(out["nerf_masks"]))


def train_loop_case(P, train_nerf, device):
    """The tiny nerf_synthetic.py-style problem both the reference and the mirror train on (shared by the test)."""
    import scenes
    shape, sphere, bsdf, lights, _integ, _w = scenes.build_pipeline(P, "dtu", device=device)
    size, crop = 16, 4
    c2w, focal = synth.nerf_cameras(3, size, device=device)
    gx, gy = np.meshgrid(np.linspace(0, 1, size), np.linspace(0, 1, size), indexing="ij")
    imgs, masks = [], []
    for i in range(3):
        img = np.stack([0.3 + 0.4 * gx, 0.5 + 0.0 * gy, 0.6 - 0.3 * gy], axis=-1) * (0.8 + 0.1 * i)
        m = ((gx - 0.5) ** 2 + (gy - 0.5) ** 2 < 0.2).astype(np.float32)
        imgs.append(torch.tensor(img, dtype=torch.float, device=device))
        masks.append(torch.tensor(m, dtype=torch.float, device=device))
    params = list(sphere.parameters()) + list(bsdf.parameters()) + list(lights.parameters())
    opt = torch.optim.AdamW(params, lr=8e-5, weight_decay=0)
    random.seed(5); np.random.seed(5); torch.manual_seed(5)
    losses = train_nerf(shape, bsdf, P.integrators.Direct(), lights, [c for c in c2w], focal, imgs, masks, opt, size, crop,
                        N=2, iters=3, num_ckpts=1, save_freq=10**6, valid_freq=10**6, silent=True)
    return losses, sphere, bsdf


def gen_train_loop():
    """Three iterations of the UNMODIFIED reference's train_nerf (training_utils.py:211-300) on a 16x16, 3-view
    problem.  Patched for the run: save_image (matplotlib is stubbed) and the `ssim` that utils.masked_loss imports
    from the absent pytorch_msssim, which is replaced by the in-repo restatement (so the SSIM term itself stays
    unpinned; on 4x4 crops it is the per-pixel formula without any window)."""
    import pytorch3d.pathtracer as P
    import pytorch3d.pathtracer.training_utils as TU
    import pytorch3d.pathtracer.utils as RU
    import pytorch3d.pathtracer.shapes.sdfs, pytorch3d.pathtracer.bsdf, pytorch3d.pathtracer.lights  # noqa: F401
    import pytorch3d.pathtracer.integrators, pytorch3d.pathtracer.neural_blocks, pytorch3d.pathtracer.cameras  # noqa: F401
    from neural_raytracing_b200.pathtracer.ssim import ssim as our_ssim
    RU.ssim = our_ssim
    TU.ssim = our_ssim
    TU.save_image = lambda *a, **k: None
    random.random = lambda: FIXED_RANDOM
    losses, sphere, bsdf = train_loop_case(P, TU.train_nerf, "cpu")
    out = {"losses": np.array(losses, np.float64),
           "sdf_out_w_after": sphere.shift.out.weight.detach().numpy().copy(),
           "spvar_out_b_after": bsdf.sp_var_fn.out.bias.detach().numpy().copy(),
           "fixed_random": np.array(FIXED_RANDOM, np.float64),
           "src": np.array("pytorch3d/pathtracer/training_utils.py:211-300; utils.py:134-147, 307-359, 378-383")}
    np.savez_compressed(os.path.join(HERE, "train_loop.npz"), **out)
    print("train_loop.npz: losses", losses)


def gen_plain_nerf():
    """PlainNeRF.forward (shapes/nerf.py:46-74) with its density noise (:66) switched off (torch.randn_like -> 0 for
    the call) and the far-plane jitter fixed; plus the parameter names / shapes of every learned component of the path
    (what a checkpoint of the reference holds: dtu.py:93-108 pickles / jit-saves these modules)."""
    from pytorch3d.pathtracer.shapes.nerf import PlainNeRF
    out = {}
    random.random = lambda: FIXED_RANDOM
    n = PlainNeRF(device="cpu")
    synth.fill_module(n, 81)
    with torch.no_grad():
        n.first.out.bias[0] = 0.8        # positive density, otherwise every weight is 0 and the image is 0.5
    rays = T(synth.camera_rays(9, 2 * 6 * 5).reshape(2, 6, 5, 1, 6))
    latent = T(np.random.RandomState(4).standard_normal((2, 32)).astype(np.float32) * 0.5)
    n.assign_latent(latent)
    real = torch.randn_like
    torch.randn_like = lambda t, **k: torch.zeros_like(t)
    try:
        with torch.no_grad():
            rgb = n(rays, None)
    finally:
        torch.randn_like = real
    out["rays"], out["latent"], out["rgb"] = rays.numpy(), latent.numpy(), rgb.numpy()
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    # parameter inventory of the learned components
    mods = {"SphereSDF": SphereSDF(n=64, device="cpu"), "NeRFLE": NeRFLE(device="cpu"), "NeRFLE_envmap": NeRFLE(envmap=True, device="cpu"),
            "PlainNeRF": n, "NeuralBSDF": NeuralBSDF(device="cpu"), "LightField": LightField(device="cpu"),
            "ComposeSpatialVarying": ComposeSpatialVarying([NeuralBSDF(device="cpu"), Diffuse(device="cpu")], device="cpu")}
    for name, m in mods.items():
        sd = m.state_dict()
        out["sd_" + name] = np.array([k + ":" + "x".join(str(d) for d in v.shape) for k, v in sd.items()])
    out["src"] = np.array("pytorch3d/pathtracer/shapes/nerf.py:9-74; state_dict() of sdfs.py:16-31, nerf.py:153-172, bsdfs.py:482-496, 613-621, lights.py:155-164")
    np.savez_compressed(os.path.join(HERE, "plain_nerf.npz"), **out)
    print("plain_nerf.npz: rgb", out["rgb"].shape, "mean", out["rgb"].mean(), "std", out["rgb"].std(), "; state dicts", {k: len(out["sd_" + k]) for k in mods})


def gen_colocate64():
    """BASELINE configs[0] at its named size: colocate.py-style forward render, 64x64 camera rays, one chunk, bundle 1
    (SURVEY 8d cfg1): SDF(SphereSDF(n=64), max_steps=64), ComposeSpatialVarying([NeuralBSDF x2, Diffuse(Softplus),
    Conductor(Softplus)]), Direct, PointLights(scale=5), learned-occlusion MLP as w_isect."""
    import pytorch3d.pathtracer as P
    import pytorch3d.pathtracer.shapes.sdfs, pytorch3d.pathtracer.bsdf, pytorch3d.pathtracer.lights  # noqa: F401
    import pytorch3d.pathtracer.integrators, pytorch3d.pathtracer.neural_blocks, pytorch3d.pathtracer.cameras  # noqa: F401
    from pytorch3d.pathtracer.cameras import NeRFCamera
    out = {}
    random.random = lambda: FIXED_RANDOM
    size = 64
    c2w, focal = synth.nerf_cameras(1, size)
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cpu")
    shape, sphere, bsdf, lights, integrator, w_isect = build_pipeline(P, "colocate")
    with torch.no_grad():
        img, mi = P.pathtrace(shape, size=size, chunk_size=size, bundle_size=1, bsdf=bsdf, integrator=integrator,
                              lights=lights, cameras=cam, device="cpu", silent=True, background=0, w_isect=w_isect,
                              with_noise=False, addition=lambda it: it)
    out["img"] = img.numpy()
    out["throughput"] = mi.throughput.reshape(-1).numpy()
    out["weights"] = mi.normalized_weights.reshape(-1, 4).numpy().astype(np.float16)
    out["raw_normals"] = mi.raw_normals.detach().numpy()
    out["depth"] = mi.t.reshape(-1).numpy()
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("main.py:13-93; integrators/integrators.py:156-206; scene.py:301-318; shapes/sdfs.py:102-249; bsdf/bsdfs.py")
    np.savez_compressed(os.path.join(HERE, "colocate64.npz"), **out)
    print("colocate64.npz: img mean %.4f, %d hits of %d" % (out["img"].mean(), len(out["raw_normals"]), size * size))


def gen_dtu16():
    """BASELINE configs[3] with its named model (dtu.py:93-108: 10 NeuralBSDF + 6 Diffuse under a 16-way sp_var MLP,
    LightField, NeRFIntegrator(Direct()), DTUCamera) on 2 views x 64x64 rays (the whole 1600x1200 field of view): one train_dtu iteration
    (training_utils.py:385-405) -- pathtrace_sample, masked_loss(mask_weight=10) + eikonal_loss(raw_normals) --
    forward and backward.  The SSIM term of masked_loss comes from the absent, unpinned pytorch_msssim: it is patched
    to the constant 1 (-log 1 = 0) for the run, i.e. "masked_loss without SSIM" (SURVEY 8d cfg4).  Gradients are kept
    as scenes.grad_block() of every parameter tensor, stored with synth.pack_grad."""
    import pytorch3d.pathtracer as P
    import pytorch3d.pathtracer.utils as RU
    import pytorch3d.pathtracer.shapes.sdfs, pytorch3d.pathtracer.bsdf, pytorch3d.pathtracer.lights  # noqa: F401
    import pytorch3d.pathtracer.integrators, pytorch3d.pathtracer.neural_blocks, pytorch3d.pathtracer.cameras  # noqa: F401
    from pytorch3d.pathtracer.cameras import DTUCamera
    import scenes
    RU.ssim = lambda *a, **k: torch.ones(())
    random.random = lambda: FIXED_RANDOM
    out = {}
    n_views, size, crop, uv = 2, 64, 64, (0, 0)
    shape, sphere, bsdf, lights, integrator = scenes.build_dtu16(P)
    pose, K = scenes.dtu_cameras(n_views)
    cam = DTUCamera(pose=pose, intrinsic=K, device="cpu")
    exp, mask = scenes.dtu_targets(n_views, crop)
    got, mi = P.pathtrace_sample(shape, size=size, chunk_size=size, bundle_size=1, crop_size=crop, bsdf=bsdf,
                                 integrator=integrator, cameras=cam, lights=lights, device="cpu", uv=uv, background=0,
                                 addition=lambda mi: mi, squeeze_first=False, silent=True)
    loss_img = RU.masked_loss(got[..., :3], exp, mi.throughput.squeeze(-1), mask, mask_weight=10, with_logits=mi.with_logits)
    loss_eik = RU.eikonal_loss(mi.raw_normals)
    loss = loss_img + loss_eik
    loss.backward()
    out["img"] = got.detach().numpy()
    out["throughput"] = mi.throughput.detach().reshape(-1).numpy()
    out["n_hits"] = np.array(len(mi.raw_normals))
    out["loss"] = np.array([loss.item(), loss_img.item(), loss_eik.item()], np.float64)
    groups = {"sdf": sphere, "spvar": bsdf.sp_var_fn, "light": lights}
    for i, b in enumerate(bsdf.bsdfs[:10]):
        groups["bsdf%d" % i] = b.mlp
    names = []
    for gname, mod in groups.items():
        for pname, p in mod.named_parameters():
            assert p.grad is not None, (gname, pname)
            key = "g_%s.%s" % (gname, pname)
            out[key], out[key + "_scale"] = synth.pack_grad(scenes.grad_block(p.grad).numpy())
            out["n_" + key[2:]] = np.array(float(p.grad.norm()), np.float64)
            names.append(key)
    out["g_reflectance"] = np.stack([b.reflectance.grad.numpy() for b in bsdf.bsdfs[10:]])
    out["grad_keys"] = np.array(names)
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["config"] = np.array([n_views, size, crop, uv[0], uv[1]])
    out["src"] = np.array("scripts/dtu.py:93-146; training_utils.py:347-405; main.py:97-179; utils.py:294-359; cameras/cameras.py:132-192")
    np.savez_compressed(os.path.join(HERE, "dtu16.npz"), **out)
    print("dtu16.npz: loss %.5f (image %.5f, eikonal %.5f), %d hits of %d rays, %d gradient tensors" %
          (loss.item(), loss_img.item(), loss_eik.item(), len(mi.raw_normals), n_views * crop * crop, len(names)))


class GoldenRatioSampler:
    """Deterministic stand-in for Sampler (samplers.py:14-20): call c returns frac((i + 1 + 977 c) * phi), i the flat
    index.  Shared by the reference run and the GPU test so that both trace the same bounces."""

    def __init__(self):
        self.calls = 0

    def sample(self, shape, device="cpu"):
        n = int(np.prod(shape))
        i = torch.arange(n, dtype=torch.float64) + 1 + 977 * self.calls
        self.calls += 1
        return ((i * 0.6180339887498949) % 1.0).float().reshape(tuple(shape)).to(device)


def gen_path():
    """Path integrator (integrators.py:274-354) with two bounces on the DTU-style scene: ComposeSpatialVarying of two
    NeuralBSDFs and a Diffuse (a Conductor child makes the reference raise: bsdfs.py:395 calls reflect() with one
    argument), learned light field, deterministic sampler, torch.multinomial replaced by argmax for the run.
    Also the warp fixtures (warps.py:10-52)."""
    import pytorch3d.pathtracer as P
    import pytorch3d.pathtracer.shapes.sdfs, pytorch3d.pathtracer.bsdf, pytorch3d.pathtracer.lights  # noqa: F401
    import pytorch3d.pathtracer.integrators, pytorch3d.pathtracer.neural_blocks, pytorch3d.pathtracer.cameras  # noqa: F401
    from pytorch3d.pathtracer.cameras import NeRFCamera
    from pytorch3d.pathtracer.integrators import Path
    from pytorch3d.pathtracer.warps import square_to_cos_hemisphere, square_to_uniform_disk_concentric
    import scenes
    out = {}
    u = GoldenRatioSampler().sample((257, 2))
    u[0] = 0.5                                       # the centre of the square (v == 0 branch)
    out["warp_u"] = u.numpy()
    out["warp_disk"] = square_to_uniform_disk_concentric(u).numpy()
    out["warp_hemi"] = square_to_cos_hemisphere(u).numpy()
    random.random = lambda: FIXED_RANDOM
    shape, sphere, bsdf, lights, _integ, _w = scenes.build_pipeline(P, "dtu", device="cpu")
    size = 16
    c2w, focal = synth.nerf_cameras(1, size)
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cpu")
    real = torch.multinomial
    torch.multinomial = lambda k, num_samples=1, **kw: k.argmax(dim=-1, keepdim=True)
    try:
        with torch.no_grad():
            img, _ = P.pathtrace(shape, size=size, chunk_size=size, bundle_size=1, bsdf=bsdf, integrator=Path(max_depth=2),
                                 lights=lights, cameras=cam, device="cpu", silent=True, background=0, with_noise=False,
                                 sampler=GoldenRatioSampler())
            img1, _ = P.pathtrace(shape, size=size, chunk_size=size, bundle_size=1, bsdf=bsdf, integrator=Path(max_depth=1),
                                  lights=lights, cameras=cam, device="cpu", silent=True, background=0, with_noise=False,
                                  sampler=GoldenRatioSampler())
    finally:
        torch.multinomial = real
    out["img_depth2"], out["img_depth1"] = img.numpy(), img1.numpy()
    out["fixed_random"] = np.array(FIXED_RANDOM, np.float64)
    out["src"] = np.array("pytorch3d/pathtracer/integrators/integrators.py:274-354; bsdf/bsdfs.py:22-63, 88-106, 500-513, 625-633; warps.py:10-52")
    np.savez_compressed(os.path.join(HERE, "path.npz"), **out)
    print("path.npz: depth2 mean %.5f depth1 mean %.5f, second bounce adds %.5f on %d pixels" %
          (img.mean(), img1.mean(), (img - img1).abs().max(), int(((img - img1).abs().max(-1)[0] > 1e-6).sum())))


if __name__ == "__main__":
    which = sys.argv[1:] or ["mlp", "sdf", "nerfle", "nerfle_train", "composite", "shading", "pipeline", "cameras",
                             "train_loop", "plain_nerf", "path", "colocate64", "dtu16", "lights_bsdf", "camera_rays", "vis", "sphere_examples", "dataset_loaders"]
    for w in which:
        torch.manual_seed(0); random.seed(0); np.random.seed(0)
        globals()["gen_" + w]()
