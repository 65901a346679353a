"""Occupancy grid on the GPU: the update against the plain forward of NeRFLE.first, the cull decision against the numpy
restatement (tests/occupancy_port.py), the culled render against the unculled one (every cell occupied: bit for bit; no
cell: zero; a partial grid: kept samples bit for bit, culled samples exactly 0, the image a float64 composite of them),
the culled hierarchical render against the restatement, and the public layer (NeRFLE.occupancy, pathtrace, opcheck)."""
import functools

import numpy as np
import pytest

import helpers
import occupancy_port as occ
import synth

pytestmark = pytest.mark.gpu

PRECS = ("f16", "bf16")
BOX = ((-1.5, -1.5, -1.5), (1.5, 1.5, 1.5))
CHUNK = 262144          # kRayChunk, csrc/nrt_render.cu


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@functools.lru_cache(maxsize=None)
def _nets(envmap):
    w1, w2 = helpers.nerfle_weights(envmap)
    return helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)


def _code(envmap):
    if envmap:
        return _t((0.5 * np.random.RandomState(7).standard_normal((1, 48))).astype(np.float32))
    return _t(np.array([[0.4, 1.0, 0.3]], np.float32))


class Grid:
    """A grid given by its bits (what ops reads: res, bbox_min, bbox_max, bits)."""

    def __init__(self, occupied, res=32, box=BOX):
        self.res, self.bbox_min, self.bbox_max = res, box[0], box[1]
        self.occupied = np.asarray(occupied, bool).reshape(-1)
        self.words = occ.pack_bits(self.occupied)
        self.bits = _t(self.words)


def _full(res=32, box=BOX):
    return Grid(np.ones(res ** 3, bool), res, box)


def _ball(res=32, radius=0.8):
    c = (np.arange(res) + 0.5) / res * 3.0 - 1.5
    x, y, z = np.meshgrid(c, c, c, indexing="ij")
    return Grid(x * x + y * y + z * z < radius * radius, res)


def _random(res=32, p=0.4, seed=5):
    return Grid(np.random.RandomState(seed).rand(res ** 3) < p, res)


def _counter():
    import torch
    return torch.zeros(1, dtype=torch.int64, device="cuda")


# ---- update -----------------------------------------------------------------------------------------------------------
def _update(first, res, ppc, seed, prec, decay=0.0, density=None, threshold=0.01, box=BOX):
    import torch
    from neural_raytracing_b200 import ops
    d = torch.zeros(res ** 3, dtype=torch.float32, device="cuda") if density is None else density.clone()
    b = torch.zeros(ops.occupancy_words(res), dtype=torch.int32, device="cuda")
    ops.occupancy_update(first, res, box[0], box[1], d, b, points_per_cell=ppc, decay=decay, threshold=threshold, seed=seed,
                         prec=prec)
    return d, b


@pytest.mark.parametrize("prec", ("f16", "bf16", "f32"))
def test_update_centres_equal_plain_forward(prec):
    """seed 0, one point per cell: density = relu(column 0 of the plain forward of first) on torch-computed cell centres,
    bit for bit; bits = density > threshold"""
    import torch
    from neural_raytracing_b200 import ops
    first, _ = _nets(False)
    res = 32
    lo, _, h = occ.box(res, *BOX)
    idx = torch.arange(res, device="cuda", dtype=torch.float32)
    axes = [torch.tensor(lo[a], device="cuda") + (idx + 0.5) * torch.tensor(h[a], device="cuda") for a in range(3)]
    pts = torch.stack(torch.meshgrid(*axes, indexing="ij"), dim=-1).reshape(-1, 3).contiguous()
    assert np.array_equal(pts.cpu().numpy(), occ.update_points(res, *BOX, 1, 0))
    want = torch.relu(ops.mlp_forward(first, pts, prec=prec)[:, 0])
    thr = float(want.median().item())           # a threshold that leaves both kinds of cells
    d, b = _update(first, res, 1, 0, prec, threshold=thr)
    assert torch.equal(d, want)
    occupied = (d > thr).cpu().numpy()
    assert np.array_equal(b.cpu().numpy(), occ.pack_bits(occupied))
    assert 0.3 < occupied.mean() < 0.7


def test_update_jitter_decay_and_seeds():
    """jittered points are the restatement's (so they lie in their cells: test_occupancy_cpu), the decay rule holds,
    equal seeds give equal grids and different seeds different ones"""
    import torch
    from neural_raytracing_b200 import ops
    first, _ = _nets(False)
    res, ppc = 16, 4
    pts = _t(occ.update_points(res, *BOX, ppc, 7))
    raw = ops.mlp_forward(first, pts, prec="f16")[:, 0].reshape(-1, ppc).cpu().numpy()
    d7, b7 = _update(first, res, ppc, 7, "f16")
    want, wbits = occ.update_rule(np.zeros(res ** 3, np.float32), raw, 0.0, 0.01)
    assert np.array_equal(d7.cpu().numpy(), want) and np.array_equal(b7.cpu().numpy(), occ.pack_bits(wbits))
    d7b, b7b = _update(first, res, ppc, 7, "f16")
    assert torch.equal(d7, d7b) and torch.equal(b7, b7b)
    d8, _ = _update(first, res, ppc, 8, "f16")
    assert not torch.equal(d7, d8)
    d78, b78 = _update(first, res, ppc, 8, "f16", decay=0.5, density=d7)
    want2, wbits2 = occ.update_rule(d7.cpu().numpy(), np.zeros((res ** 3, 1), np.float32), 0.5, 0.01)
    want2 = np.maximum(want2, d8.cpu().numpy())
    assert np.array_equal(d78.cpu().numpy(), want2)
    assert np.array_equal(b78.cpu().numpy(), occ.pack_bits(want2 > np.float32(0.01)))


# ---- the cull decision ---------------------------------------------------------------------------------------------------
def test_mask_equals_restatement():
    from neural_raytracing_b200 import ops
    g = _random(res=32)
    rays = synth.camera_rays(61, 4000)
    rays[:7, 0] = np.nan                                   # non-finite rays are kept
    rays[7:11, 3] = np.inf
    ts = np.linspace(0, 2.05, 64).astype(np.float32)
    keep = ops.occupancy_mask(g, _t(rays), _t(ts)).cpu().numpy()
    want = occ.keep_mask(g.words, g.res, g.bbox_min, g.bbox_max, rays, ts)
    p = occ.sample_points(rays, ts)
    face = occ.near_face(p, g.res, g.bbox_min, g.bbox_max)
    assert np.array_equal(keep[~face], want[~face])
    assert face.sum() <= 1e-3 * face.size, face.sum()
    assert keep[:11].all()
    _, inside = occ.cell_coords(p, g.res, g.bbox_min, g.bbox_max)
    assert keep[~inside].all() and 0.2 < (~keep).mean() < 0.8 and (~inside).any()
    # per-ray distances take the same path
    tpr = occ.port.stratified_ts(4000, 64, 0.0, 2.05, 9)
    keep2 = ops.occupancy_mask(g, _t(rays), _t(tpr)).cpu().numpy()
    face2 = occ.near_face(occ.sample_points(rays, tpr), g.res, g.bbox_min, g.bbox_max)
    assert np.array_equal(keep2[~face2], occ.keep_mask(g.words, g.res, g.bbox_min, g.bbox_max, rays, tpr)[~face2])


# ---- renders ----------------------------------------------------------------------------------------------------------
SAMPLINGS = {"uniform64": dict(), "stratified64": dict(n_coarse=64, t_near=0.0, t_far=2.05, jitter_seed=11),
             "hier64_128": dict(n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=13)}


def _samples_per_ray(kw):
    return kw.get("n_coarse", 64) + kw.get("n_fine", 0)


def _render(envmap, prec, kw, rays=None, cam=None, occupancy=None, samples_done=None):
    from neural_raytracing_b200 import ops
    m1, m2 = _nets(envmap)
    ts = None if kw else _t(np.linspace(0, 2.05, 64).astype(np.float32))
    if cam is not None:
        return ops.nerfle_render_camera(m1, m2, cam, ts, _code(envmap), prec=prec, occupancy=occupancy,
                                        samples_done=samples_done, **kw)
    return ops.nerfle_render(m1, m2, rays, ts, _code(envmap), prec=prec, occupancy=occupancy, samples_done=samples_done, **kw)


@pytest.mark.parametrize("source", ("rays", "camera"))
@pytest.mark.parametrize("envmap", (False, True), ids=("pt", "le"))
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("sampling", tuple(SAMPLINGS))
def test_all_occupied_is_bit_identical(sampling, prec, envmap, source):
    import torch
    from neural_raytracing_b200 import ops
    kw = SAMPLINGS[sampling]
    rays = cam = None
    if source == "rays":
        rays = _t(synth.camera_rays(62, 3001))
        R = 3001
    else:
        c2w, focal = synth.nerf_cameras(1, 200, device="cuda")
        cam = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=200, x0=5, y0=9, nx=61, ny=53)
        R = cam.n_rays
    base = _render(envmap, prec, kw, rays, cam)
    n = _counter()
    got = _render(envmap, prec, kw, rays, cam, occupancy=_full(), samples_done=n)
    assert torch.equal(got, base)
    assert int(n.item()) == R * _samples_per_ray(kw)


def test_all_occupied_across_the_chunk_boundary():
    """R = 262,144 + 1,001 rays (two chunks, odd tile tails in the second), hierarchical 64 + 128"""
    import torch
    rays = _t(synth.camera_rays(63, CHUNK + 1001))
    kw = SAMPLINGS["hier64_128"]
    base = _render(False, "f16", kw, rays)
    n = _counter()
    assert torch.equal(_render(False, "f16", kw, rays, occupancy=_full(), samples_done=n), base)
    assert int(n.item()) == (CHUNK + 1001) * 192


@pytest.mark.parametrize("sampling", tuple(SAMPLINGS))
def test_no_cell_occupied_gives_zero(sampling):
    """every sample inside the box and culled: both MLPs see no row at all"""
    import torch
    g = Grid(np.zeros(16 ** 3, bool), 16, ((-3.2,) * 3, (3.2,) * 3))
    rays = _t(synth.camera_rays(64, 2000))
    n = _counter()
    img = _render(False, "f16", SAMPLINGS[sampling], rays, occupancy=g, samples_done=n)
    assert torch.equal(img, torch.zeros_like(img)) and int(n.item()) == 0


@pytest.mark.parametrize("grid", ("ball", "random"))
@pytest.mark.parametrize("prec", PRECS)
def test_partial_grid_samples_and_image(grid, prec):
    """kept samples bit for bit those of the unculled pass, culled ones exactly 0 (the kernel's own mask); the image a
    float64 composite of the culled per-sample arrays"""
    import torch
    from neural_raytracing_b200 import ops
    g = _ball() if grid == "ball" else _random()
    m1, m2 = _nets(False)
    rays = _t(synth.camera_rays(65, 5003))
    ts = _t(np.linspace(0, 2.05, 64).astype(np.float32))
    code = _code(False)
    sig0, rgb0 = ops.nerfle_render_samples(m1, m2, rays, ts, code, prec=prec)
    n = _counter()
    sig, rgb = ops.nerfle_render_samples(m1, m2, rays, ts, code, prec=prec, occupancy=g, samples_done=n)
    keep = ops.occupancy_mask(g, rays, ts)
    assert 0.1 < keep.float().mean().item() < 0.9
    assert int(n.item()) == int(keep.sum().item())
    assert torch.equal(sig[keep], sig0[keep]) and torch.equal(rgb[keep], rgb0[keep])
    assert (sig[~keep] == 0).all() and (rgb[~keep] == 0).all()
    img = ops.nerfle_render(m1, m2, rays, ts, code, prec=prec, occupancy=g).cpu().numpy()
    ref = occ.composite64(sig.cpu().numpy(), rgb.cpu().numpy(), ts.cpu().numpy()[None, :])
    assert np.abs(img - ref).max() < 1e-6
    assert not np.array_equal(img, ops.nerfle_render(m1, m2, rays, ts, code, prec=prec).cpu().numpy())


def test_hierarchical_culled_vs_restatement():
    """64 + 128 with a ball grid against the restatement (culled sigma = 0 in both passes; the tolerances of
    test_gpu_tensorcore.py::test_hierarchical_render_vs_restatement for f16), excluding the rays with a sample within
    1e-6 h of a cell face"""
    from neural_raytracing_b200 import ops
    g = _ball(res=32, radius=0.6)
    w1, w2 = helpers.nerfle_weights(False)
    rays = synth.camera_rays(55, 192)
    code = np.array([[0.4, 1.0, 0.3]], np.float32)
    ref, ts_c, ts_f = occ.render_hierarchical_culled(helpers.oracle_mlp(w1), helpers.oracle_mlp(w2), rays, code, 64, 128,
                                                     0.0, 2.05, 3, g.words, g.res, g.bbox_min, g.bbox_max)
    m1, m2 = _nets(False)
    rgb = ops.nerfle_render(m1, m2, _t(rays), None, _t(code), prec="f16", n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05,
                            jitter_seed=3, occupancy=g).cpu().numpy()
    face = np.zeros(rays.shape[0], bool)
    for t in (ts_c, ts_f):
        face |= occ.near_face(occ.sample_points(rays, t), g.res, g.bbox_min, g.bbox_max).any(axis=1)
    assert face.sum() <= 4, face.sum()
    culled = ~occ.keep_mask(g.words, g.res, g.bbox_min, g.bbox_max, rays, ts_c)
    assert culled.mean() > 0.05
    err = np.abs(rgb - ref).max(axis=-1)[~face]
    assert err.max() < 5e-4, err.max()
    assert helpers.psnr(rgb[~face], ref[~face]) > 85


# ---- public layer ------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _model():
    import torch
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    torch.manual_seed(3)
    m = NeRFLE(device="cuda")
    with torch.no_grad():
        m.first.out.bias[0] = 0.8        # a visible density (the randomly initialised one renders black)
    return m


def _lights():
    from neural_raytracing_b200.pathtracer.lights import PointLights
    return PointLights(location=[[0.4, 1.0, 0.3]], device="cuda")


class _Scene:
    """_model() at f16 with a fixed far plane (far_jitter) and a fresh grid; restored on exit"""

    def __enter__(self):
        import torch
        from neural_raytracing_b200 import config
        from neural_raytracing_b200.pathtracer.shapes.nerf import OccupancyGrid
        self.model, self.old = _model(), config.precision
        config.precision = "f16"
        self.model.far_jitter = torch.tensor([0.3], device="cuda")
        probe = OccupancyGrid(resolution=32, threshold=0.0).update(self.model, points_per_cell=2, seed=1)
        thr = float(probe.density.quantile(0.7).item())     # 30 % of the cells occupied
        self.grid = OccupancyGrid(resolution=32, threshold=thr).update(self.model, points_per_cell=2, seed=1)
        self.model.occupancy = self.grid
        return self

    def __exit__(self, *exc):
        from neural_raytracing_b200 import config
        config.precision = self.old
        self.model.occupancy = None
        self.model.far_jitter = None
        self.model.zero_grad(set_to_none=True)


def test_model_forward():
    import torch
    from neural_raytracing_b200 import config, ops
    with _Scene() as sc:
        model, grid = sc.model, sc.grid
        assert 0.0 < grid.occupied_fraction() < 1.0 and "OccupancyGrid(resolution=32" in repr(grid)
        rays = _t(synth.camera_rays(66, 1500))
        lc = _lights().location
        ts = model._sample_ts("cuda")
        ops.profile_collect()
        with torch.no_grad():
            got = model(rays, _lights())
        prof = ops.profile_collect()
        assert prof["occupancy_cull"][1] == 1 and prof["mlp_tc_nerf_first"][1] == 1 and prof["mlp_tc_nerf_second"][1] == 1
        want = ops.nerfle_render(model.first.packed(), model.second.packed(), rays, ts, lc, prec="f16", occupancy=grid)
        assert torch.equal(got, want)
        assert not torch.equal(got, ops.nerfle_render(model.first.packed(), model.second.packed(), rays, ts, lc, prec="f16"))
        # the hierarchical no-grad branch culls too
        from neural_raytracing_b200.pathtracer.shapes.nerf import HierarchicalSampling
        model.sampling = HierarchicalSampling(64, 128)
        try:
            with torch.no_grad():
                got = model(rays, _lights())
            want = ops.nerfle_render(model.first.packed(), model.second.packed(), rays, None, lc, prec="f16", occupancy=grid,
                                     **model._render_sampling())
            assert torch.equal(got, want)
        finally:
            model.sampling = None
        # a stale grid raises until it is updated
        with torch.no_grad():
            model.first.out.bias.add_(0.0)
        with pytest.raises(ops.NrtError, match="update"):
            with torch.no_grad():
                model(rays, _lights())
        grid.update(model, points_per_cell=2, seed=1)
        with torch.no_grad():
            model(rays, _lights())
        # f32 with a grid raises (NRT_E_UNSUPPORTED from the library)
        config.precision = "f32"
        grid.update(model, points_per_cell=1, seed=0)
        with pytest.raises(ops.NrtError, match="tensor-core"):
            with torch.no_grad():
                model(rays, _lights())


def test_pathtrace_frame_culls():
    """pathtrace under NeRFReproduce (one render_camera call per frame, main.py) equals nerfle_render_camera with the grid"""
    import torch
    from neural_raytracing_b200 import ops
    from neural_raytracing_b200.pathtracer import main as pt
    from neural_raytracing_b200.pathtracer.cameras import NeRFCamera
    from neural_raytracing_b200.pathtracer.integrators import NeRFReproduce
    with _Scene() as sc:
        model = sc.model
        c2w, focal = synth.nerf_cameras(1, 48, device="cuda")
        cams = NeRFCamera(cam_to_world=c2w, focal=focal, device="cuda")
        with torch.no_grad():
            img = pt.pathtrace(model, _lights(), cams, NeRFReproduce(), size=48, chunk_size=48, bundle_size=1,
                               device="cuda", with_noise=0, silent=True)
        img = img[0] if isinstance(img, tuple) else img
        cam = cams.device_desc(48, nx=48, ny=48, bundle_size=1)
        want = ops.nerfle_render_camera(model.first.packed(), model.second.packed(), cam, model._sample_ts("cuda"),
                                        _lights().location, prec="f16", occupancy=sc.grid)
        assert torch.equal(img.reshape(-1), want.mean(dim=-2).reshape(-1))


def test_training_ignores_the_grid():
    """the differentiable forward: no cull kernel runs, the loss is identical with and without the grid, and so are the
    gradients up to the run-to-run order of the wgrad kernels' fp32 atomics"""
    import torch
    from neural_raytracing_b200 import ops
    with _Scene() as sc:
        model = sc.model
        rays = _t(synth.camera_rays(67, 512))
        target = torch.rand(512, 3, device="cuda", generator=torch.Generator("cuda").manual_seed(1))

        def loss_and_grads():
            model.zero_grad(set_to_none=True)
            loss = ((model(rays, _lights()) - target) ** 2).mean()
            loss.backward()
            return loss.detach().clone(), [p.grad.clone() for p in model.parameters()]
        ops.profile_collect()
        l1, g1 = loss_and_grads()
        assert ops.profile_collect()["occupancy_cull"][1] == 0
        model.occupancy = None
        l0, g0 = loss_and_grads()
        assert torch.equal(l0, l1)
        for a, b in zip(g0, g1):
            torch.testing.assert_close(b, a, rtol=1e-4, atol=1e-7)


def test_opcheck():
    import torch
    from neural_raytracing_b200 import torch_ops
    from neural_raytracing_b200.pathtracer.shapes.nerf import NeRFLE
    torch.manual_seed(4)
    m = NeRFLE(device="cuda")
    p1, b1, a1 = torch_ops.pack_module(m.first).detach(), m.first.basis_p, torch_ops.arch_of(m.first)
    p2, b2, a2 = torch_ops.pack_module(m.second).detach(), m.second.basis_p, torch_ops.arch_of(m.second)
    res = 16
    dens = torch.zeros(res ** 3, device="cuda")
    bits = torch.zeros((res ** 3 + 31) // 32, dtype=torch.int32, device="cuda")
    box = ([-1.5] * 3, [1.5] * 3)
    torch.library.opcheck(torch.ops.nrt_b200.occupancy_update.default,
                          (dens, bits, p1, b1, a1, res, box[0], box[1], 2, 0.0, 0.01, 1, 1))
    d2, b2_ = torch.ops.nrt_b200.occupancy_update(dens, bits, p1, b1, a1, res, box[0], box[1], 2, 0.0, 0.01, 1, 1)
    rays = _t(synth.camera_rays(68, 300))
    ts = torch.linspace(0, 2.05, 64, device="cuda")
    code = torch.tensor([[0.4, 1.0, 0.3]], device="cuda")
    torch.library.opcheck(torch.ops.nrt_b200.nerfle_render.default,
                          (rays, ts, code, p1, b1, a1, p2, b2, a2, 1, b2_, res, box[0], box[1]))
    c2w, focal = synth.nerf_cameras(1, 64, device="cuda")
    torch.library.opcheck(torch.ops.nrt_b200.nerfle_render_camera.default,
                          (0, c2w, None, float(focal), 64.0, 0, 0, 20, 16, 1, 0.0, 0, ts, code, p1, b1, a1, p2, b2, a2, 1,
                           b2_, res, box[0], box[1]))
