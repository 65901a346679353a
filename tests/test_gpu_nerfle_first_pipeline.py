"""NeRFLE.first's inference kernels with the tile boundary pipelined (NRT_FIRST_PIPE, csrc/tc_core.cuh): a slot fetches
its next tile's inputs one tile ahead, computes that tile's encoding while the output layer runs, and hands it to the
MMA warp before it stores the current tile's outputs.  Checked here, at tile counts that reach every tail of that
hand-off (a single tile; an odd tile count, so that one slot of the last CTA gets no tile; one tile more than the grid
has slots; several tiles per slot; sample counts that are not a multiple of 128): the plain forward and the render pass
(uniform and 64 + 128 hierarchical ts), f16 and bf16, against the exact fp32 kernels; the camera-fed frame against the
ray-fed one, bit for bit; and results that do not depend on the launch -- the same rays or points evaluated whole and as
two windows, bit for bit."""
import numpy as np
import pytest

import helpers
import synth

pytestmark = pytest.mark.gpu

TOL = {"f16": 1e-3, "bf16": 5e-3}
RENDER_S = 192


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _slots():
    """tile slots of one full grid: one CTA per SM, two tile slots each"""
    import torch
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count


def _first_mlp():
    w = synth.mlp_weights(seed=31, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0)
    return helpers.cuda_mlp(w)


def _sample_counts():
    g = _slots()
    return {"one_tile": 77, "odd_tiles": 128 * 36 + 5, "grid_plus_one": g * 128 + 1, "several_per_slot": g * 128 * 3 + 77}


def _ray_counts():
    g = _slots()
    # 192 samples per ray = 1.5 tiles per ray
    return {"two_tiles": 1, "odd_tiles": 23, "grid_plus_one": (2 * (g + 1) + 2) // 3, "several_per_slot": 2001}


@pytest.fixture(scope="module")
def nets():
    w1, w2 = helpers.nerfle_weights(False)
    return helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("case", ["one_tile", "odd_tiles", "grid_plus_one", "several_per_slot"])
def test_first_forward_vs_exact(prec, case):
    from neural_raytracing_b200 import ops
    M = _sample_counts()[case]
    m = _first_mlp()
    x = _t((0.8 * np.random.RandomState(M).standard_normal((M, 3))).astype(np.float32))
    y32 = ops.mlp_forward(m, x, prec="f32").cpu().numpy()
    y = ops.mlp_forward(m, x, prec=prec).cpu().numpy()
    assert y.shape == y32.shape and np.isfinite(y).all()
    assert np.abs(y - y32).max() < TOL[prec], np.abs(y - y32).max()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("case", ["two_tiles", "odd_tiles", "grid_plus_one", "several_per_slot"])
@pytest.mark.parametrize("sampling", ["uniform", "hierarchical"])
def test_render_vs_exact(nets, prec, case, sampling):
    from neural_raytracing_b200 import ops
    m1, m2 = nets
    R = _ray_counts()[case]
    rays = _t(synth.camera_rays(35, R))
    code = _t(np.array([[0.4, 1.0, 0.3]], np.float32))
    if sampling == "uniform":
        ts, kw = _t(np.linspace(0.0, 2.05, RENDER_S).astype(np.float32)), {}
    else:
        ts, kw = None, dict(n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=3)
    r32 = ops.nerfle_render(m1, m2, rays, ts, code, prec="f32", **kw).cpu().numpy()
    r = ops.nerfle_render(m1, m2, rays, ts, code, prec=prec, **kw).cpu().numpy()
    assert r.shape == r32.shape and np.isfinite(r).all()
    assert np.abs(r - r32).max() < TOL[prec], np.abs(r - r32).max()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_camera_fed_equals_ray_fed(nets, prec):
    """IoNerfFirst<64, true> computes the rays inside the kernel; its fetch runs the camera arithmetic a tile ahead"""
    import torch
    from neural_raytracing_b200 import ops
    m1, m2 = nets
    c2w, focal = synth.nerf_cameras(1, 400, device="cuda")
    desc = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=400, x0=7, y0=3, nx=97, ny=61)
    code = _t(np.array([[0.4, 1.0, 0.3]], np.float32))
    for kw in (dict(ts=_t(np.linspace(0.0, 2.05, RENDER_S).astype(np.float32))),
               dict(ts=None, n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=8)):
        ts = kw.pop("ts")
        ray_fed = ops.nerfle_render(m1, m2, ops.camera_rays(desc), ts, code, prec=prec, **kw)
        try:
            ops.set_camera_rays_mode(True)
            cam_fed = ops.nerfle_render_camera(m1, m2, desc, ts, code, prec=prec, **kw)
        finally:
            ops.set_camera_rays_mode(False)
        assert torch.isfinite(cam_fed).all()
        assert torch.equal(cam_fed.reshape(-1, 3), ray_fed.reshape(-1, 3))


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_render_does_not_depend_on_the_launch(nets, prec):
    """The same rays rendered in one call and as two windows (the split puts every sample in another tile and lane)"""
    import torch
    from neural_raytracing_b200 import ops
    m1, m2 = nets
    R, R0 = 2001, 677                       # 677 * 192 samples is not a multiple of 128
    rays = _t(synth.camera_rays(36, R))
    code = _t(np.array([[0.4, 1.0, 0.3]], np.float32))
    ts = _t(np.linspace(0.0, 2.05, RENDER_S).astype(np.float32))
    whole = ops.nerfle_render(m1, m2, rays, ts, code, prec=prec)
    parts = torch.cat([ops.nerfle_render(m1, m2, rays[:R0].contiguous(), ts, code, prec=prec),
                       ops.nerfle_render(m1, m2, rays[R0:].contiguous(), ts, code, prec=prec)])
    assert torch.isfinite(whole).all()
    assert torch.equal(whole, parts)


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_forward_does_not_depend_on_the_launch(prec):
    import torch
    from neural_raytracing_b200 import ops
    m = _first_mlp()
    M, M0 = _slots() * 128 * 2 + 301, 12345
    x = _t((0.8 * np.random.RandomState(5).standard_normal((M, 3))).astype(np.float32))
    whole = ops.mlp_forward(m, x, prec=prec)
    parts = torch.cat([ops.mlp_forward(m, x[:M0].contiguous(), prec=prec), ops.mlp_forward(m, x[M0:].contiguous(), prec=prec)])
    assert torch.isfinite(whole).all()
    assert torch.equal(whole, parts)
