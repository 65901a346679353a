"""Scene construction shared by tests/golden/make_golden.py (run on the UNMODIFIED reference package)
and the GPU pipeline tests (run on the drop-in mirror): the same code builds both, which is itself a
check of the drop-in surface (constructor kwargs, attributes that scripts mutate)."""
import numpy  # noqa: F401
import torch

import synth


def build_pipeline(P, kind, device="cpu"):
    """Builds the colocate-style ('colocate') or DTU-style ('dtu') scene out of the package `P`
    (either the reference `pytorch3d.pathtracer` or the drop-in mirror): identical code for both."""
    import torch.nn as nn
    sdfs, bsdfm, lightsm, integ = P.shapes.sdfs, P.bsdf, P.lights, P.integrators
    sphere = sdfs.SphereSDF(n=64, device=device)
    synth.fill_module(sphere, 61, shift_std=0.02)
    shape = sdfs.SDF(sdf=sphere, device=device, max_steps=64)
    if kind == "colocate":
        # colocate.py:63-85: 2 neural + diffuse + conductor bases, point light, learned occlusion MLP
        kids = [bsdfm.NeuralBSDF(device=device), bsdfm.NeuralBSDF(device=device),
                bsdfm.Diffuse(preprocess=nn.Softplus(), device=device), bsdfm.Conductor(activation=nn.Softplus(), device=device)]
        kids[2].reflectance = torch.tensor([0.3, 0.6, 0.2], device=device, requires_grad=True)
        kids[3].specular = torch.tensor([0.7, 0.4, 0.9], device=device, requires_grad=True)
        lights = lightsm.PointLights(device=device, location=[[0.9, 0.5, 0.7]], scale=5)
        occ = P.neural_blocks.SkipConnMLP(in_size=5, out=1, device=device).to(device)
        synth.fill_module(occ, 65)
        integrator, w_isect = integ.Direct(), occ
    else:
        # dtu.py:95-106: neural + diffuse(sigmoid) bases, learned light field, NeRFIntegrator(Direct())
        kids = [bsdfm.NeuralBSDF(activation=nn.Sigmoid(), device=device), bsdfm.NeuralBSDF(activation=nn.Sigmoid(), device=device),
                bsdfm.Diffuse(preprocess=torch.sigmoid, device=device)]
        kids[2].reflectance = torch.tensor([0.2, -0.4, 0.5], device=device, requires_grad=True)
        lights = lightsm.LightField(device=device)
        synth.fill_module(lights, 66)
        integrator, w_isect = integ.NeRFIntegrator(integ.Direct()), False
    for i, k in enumerate(kids[:2]):
        synth.fill_module(k, 62 + i)
    bsdf = bsdfm.ComposeSpatialVarying(kids, device=device)
    bsdf.sp_var_fn._synth_sigma = 128.0
    synth.fill_module(bsdf, 64)
    return shape, sphere, bsdf, lights, integrator, w_isect




def build_dtu16(P, device="cpu"):
    """The scene dtu.py trains (dtu.py:93-108): SDF(SphereSDF(n=2<<5), max_steps=64), ComposeSpatialVarying of
    10 NeuralBSDF + 6 Diffuse(sigmoid).random() with every child's `act` set to nn.Sigmoid() (dtu.py:101-106),
    LightField, NeRFIntegrator(Direct()) as train_dtu wraps it (training_utils.py:369)."""
    import torch.nn as nn
    sdfs, bsdfm, lightsm, integ = P.shapes.sdfs, P.bsdf, P.lights, P.integrators
    sphere = sdfs.SphereSDF(n=2 << 5, device=device)
    synth.fill_module(sphere, 71, shift_std=0.02)
    with torch.no_grad():
        # the k = 32 smooth-min of 64 spheres inflates the union by log(64)/32 = 0.13: pull the centres in and use the
        # negative half of sdfs.py:20's radius range so that the object covers ~2/3 of the view (hit AND miss pixels)
        sphere.centers.mul_(0.6)
        sphere.radii.abs_().mul_(-0.48)
    shape = sdfs.SDF(sdf=sphere, device=device)
    shape.max_steps = 64
    kids = [bsdfm.NeuralBSDF(device=device) for _ in range(10)] + \
           [bsdfm.Diffuse(preprocess=torch.sigmoid, device=device).random() for _ in range(6)]
    for i, k in enumerate(kids):
        setattr(k, "act", nn.Sigmoid())
        if i < 10:
            synth.fill_module(k, 72 + i)
        else:
            rs = synth.np.random.RandomState(900 + i)
            k.reflectance = torch.tensor(rs.uniform(-1, 1, 3).astype("float32"), device=device, requires_grad=True)
    bsdf = bsdfm.ComposeSpatialVarying(kids, device=device)
    bsdf.sp_var_fn._synth_sigma = 128.0
    synth.fill_module(bsdf.sp_var_fn, 90)
    lights = lightsm.LightField(device=device)
    synth.fill_module(lights, 91)
    with torch.no_grad():
        lights.light_field_approx.out.bias.add_(0.3)     # a light direction with positive components (lights.py:191 clamps)
    return shape, sphere, bsdf, lights, integ.NeRFIntegrator(integ.Direct())


def dtu_cameras(n_views, device="cpu"):
    """Synthetic DTU-style cameras (dtu.py:69-87): intrinsics of the 1600x1200 DTU images (fx = fy = 2892, principal
    point at the centre) and camera-to-world poses at distance 1 looking at the origin (+z forward, as IDR)."""
    import numpy as np
    poses, Ks = [], []
    for i in range(n_views):
        az, el = 0.4 + 1.1 * i, 0.3 + 0.15 * i
        c = np.array([np.cos(el) * np.sin(az), np.sin(el), np.cos(el) * np.cos(az)])
        fwd = -c / np.linalg.norm(c)
        right = np.cross([0, 1, 0], fwd); right /= np.linalg.norm(right)
        down = np.cross(fwd, right)
        m = np.eye(4, dtype=np.float32)
        m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = right, down, fwd, c
        K = np.eye(4, dtype=np.float32)
        K[0, 0] = K[1, 1] = 2892.0
        K[0, 2], K[1, 2] = 800.0, 600.0
        poses.append(m); Ks.append(K)
    return torch.tensor(np.stack(poses), device=device), torch.tensor(np.stack(Ks), device=device)


def dtu_targets(n_views, crop, device="cpu"):
    """Expected colours / masks of the crop: smooth colour ramps and a disc mask (so that both the hit and the miss
    branch of masked_loss, utils.py:307-359, are exercised)."""
    import numpy as np
    gx, gy = np.meshgrid(np.linspace(0, 1, crop), np.linspace(0, 1, crop), indexing="ij")
    exp = np.stack([np.stack([0.3 + 0.4 * gx, 0.5 + 0.0 * gy, 0.6 - 0.3 * gy], -1) * (0.8 + 0.1 * i) for i in range(n_views)])
    mask = np.stack([((gx - 0.5) ** 2 + (gy - 0.47 - 0.04 * i) ** 2 < 0.2).astype(np.float32) for i in range(n_views)])
    return torch.tensor(exp, dtype=torch.float, device=device), torch.tensor(mask, dtype=torch.float, device=device)


def grad_block(t):
    """The part of a gradient tensor the fixtures keep: the first 16 output rows of a weight matrix, everything of a
    vector / small tensor (with synth.pack_grad this keeps the dtu16 fixture under 1 MB; every kept element is an
    independent check)."""
    return t[:16] if t.dim() == 2 and t.shape[0] > 16 else t
