"""NeRFLE.second with the layer biases as one more K-chunk of each tcgen05 MMA (NRT_BIAS_MMA, csrc/tc_core.cuh) and the
zero x_lo chunks of the phase GEMM skipped for the packed 16-bit latent: point and environment light, f16 and bf16,
tile counts that are not a multiple of 128 samples x 148 SMs x tile slots, against the exact fp32 kernels with the
tolerances of the other tensor-core tests (max-abs 1e-3 f16, 5e-3 bf16).  The camera-fed kernels (rays computed in the
MLP kernels) must give the ray-fed image bit for bit."""
import numpy as np
import pytest

import helpers
import synth

pytestmark = pytest.mark.gpu

TOL = {"f16": 1e-3, "bf16": 5e-3}
SECOND = {
    "point": dict(seed=41, in_size=70, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0),
    "envmap": dict(seed=42, in_size=115, out=3, num_layers=8, hidden=64, freqs=16, sigma=32.0),
}


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("name", list(SECOND))
@pytest.mark.parametrize("M", [1, 148 * 3 * 128 + 77, 148 * 2 * 128 * 2 + 129])
def test_second_mlp_vs_exact(name, prec, M):
    """The plain [M, in] -> [M, 3] forward of the NeRFLE.second nets (every stage takes its bias from the MMA)."""
    from neural_raytracing_b200 import ops
    kw = SECOND[name]
    m = helpers.cuda_mlp(synth.mlp_weights(**kw))
    x = _t((0.6 * np.random.RandomState(M).standard_normal((M, kw["in_size"]))).astype(np.float32))
    y32 = ops.mlp_forward(m, x, prec="f32").cpu().numpy()
    y = ops.mlp_forward(m, x, prec=prec).cpu().numpy()
    assert y.shape == y32.shape and np.isfinite(y).all()
    assert np.abs(y - y32).max() < TOL[prec], np.abs(y - y32).max()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("envmap", [False, True])
def test_render_vs_exact(envmap, prec):
    """The render path (IoNerfSecond with the packed 16-bit latent: bias K-chunks and the shortened phase GEMM), one
    uniform pass of 192 samples (the frame's per-ray sample count; the same distances in both precisions) on 1,337 rays
    (256,704 samples: 2,005.5 tiles)."""
    from neural_raytracing_b200 import ops
    w1, w2 = helpers.nerfle_weights(envmap)
    m1, m2 = helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)
    rays = _t(synth.camera_rays(35, 1337))
    ld = 48 if envmap else 3
    code = _t((0.3 * np.random.RandomState(5).standard_normal((1, ld))).astype(np.float32))
    ts = _t(np.linspace(0.0, 2.05, 192).astype(np.float32))
    r32 = ops.nerfle_render(m1, m2, rays, ts, code, prec="f32").cpu().numpy()
    r = ops.nerfle_render(m1, m2, rays, ts, code, prec=prec).cpu().numpy()
    assert np.isfinite(r).all()
    assert np.abs(r - r32).max() < TOL[prec], np.abs(r - r32).max()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_camera_fed_equals_ray_fed(prec):
    import torch
    from neural_raytracing_b200 import ops
    w1, w2 = helpers.nerfle_weights(False)
    m1, m2 = helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)
    c2w, focal = synth.nerf_cameras(1, 400, device="cuda")
    desc = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=400, x0=11, y0=7, nx=37, ny=29)
    code = _t(np.array([[0.4, 1.0, 0.3]], np.float32))
    kw = dict(prec=prec, n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=5)
    ray_fed = ops.nerfle_render(m1, m2, ops.camera_rays(desc), None, code, **kw)
    try:
        ops.set_camera_rays_mode(True)
        cam_fed = ops.nerfle_render_camera(m1, m2, desc, None, code, **kw)
    finally:
        ops.set_camera_rays_mode(False)
    assert torch.isfinite(cam_fed).all()
    assert torch.equal(cam_fed.reshape(-1, 3), ray_fed.reshape(-1, 3))
