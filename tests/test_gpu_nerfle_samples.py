"""Every sample of the NeRFLE tensor-core render pass and of the fused training forward against float64.

A composited pixel hides most of what the two NeRFLE kernels compute: with the reference's compositing (alpha from the
absolute distance, nerf.py:205-213) transmittance is gone after ~40 of 192 samples, and the test networks of the frame
tests barely depend on their inputs.  So this module compares per-sample sigma (pre-relu) and rgb (sigmoid), output by
output, with a float64 restatement of nerf.py:175-203 (`_reference`), on networks whose outputs vary: NeRFLE.first drawn
with w_scale 0.75, NeRFLE.second with w_scale 2.5 (rgb spans 0.20..0.77, std 0.07, against 0.47..0.50 at w_scale 1).  The
next sample on a ray, the neighbouring ray, the sample one tile later, another view's light code and another tile's latent
each move some sample of every tile they touch by more than 10x the f16 gates and 3x the bf16 gates, which
tests/test_nerfle_samples_cpu.py checks on the C oracle.  Steeper networks do not test more: NeRFLE.second takes Fourier
features (sigma 32) of the latent, so the kernels' 16-bit rounding grows with the weights faster than the outputs spread.
At w_scale 2 / 3 the rgb error measured on the B200 reached 0.16 (f16) and 0.64 (bf16), as large as the errors a wrong index
makes; 0.75 / 2.5 was chosen from a CPU emulation of 16-bit operand rounding (weights, activations, encoding) that matched
the B200's errors to within 1.6x (at 2 / 3 and at 0.75 / 2.5), for the widest margin over the planted errors.

The render pass is reached through nrt_nerfle_render_samples, the render's own chunk loop with the compositing left out.
Cases (each at f16 and bf16): tile tails (one partial tile, an odd tile count, grid slots + 1 tiles, several tiles per
slot) at S = 192 (the division in ray_of) and S = 64 (the power-of-two shift); per-ray distances (jittered stratified and
the merged 64 + 128 hierarchical ones); both second nets with three views and view_of_ray = r % 3; the camera-fed kernels
against the ray-fed pass on the same camera, bit for bit, also across the 262,144-ray chunk boundary (cam_r0); the chunk
boundary of a ray array, bit-identical to the two halves rendered apart; and the fp32 pass equal to the C oracle.  IO
policies reached: IoNerfFirst<64> and <64, true>, IoNerfSecond<64,3,true>, <64,3,true,true> and <64,48,true>.
The training forward (nrt_nerfle_train_forward / _ts, sample-major, fp32 latent hand-off) is checked the same way, and
against the render pass on the same inputs: the function trained is the function rendered.

Gates (GATES below): max-abs and RMS error per output, also over the tail tiles of every launch (the last 3 x SMs tiles of
a 262,144-ray chunk hold the last tile of every slot of both kernels, which run at most three slots a CTA), so that an
error growing with the tile index shows.  Measured on NVIDIA B200 (power limit 1000 W), largest over all cases and over
the tail tiles (max-abs / RMS):
    render pass  f16   sigma 4.1e-5 / 1.1e-5   rgb 2.6e-3 / 3.0e-4
                 bf16  sigma 2.5e-4 / 4.6e-5   rgb 2.0e-2 / 2.7e-3
    training     f16   sigma 3.8e-5 / 1.0e-5   rgb 1.5e-3 / 2.0e-4
                 bf16  sigma 2.4e-4 / 4.4e-5   rgb 1.3e-2 / 1.5e-3
The gates are twice these, rounded up to two digits.  The whole module ran in 4.4 s there."""
import functools

import numpy as np
import pytest

import helpers
import synth

pytestmark = pytest.mark.gpu

PRECS = ("f16", "bf16")
W_SCALE_FIRST, W_SCALE_SECOND = 0.75, 2.5
T_FAR = 2.05
N_VIEWS = 3
CHUNK = 262144          # kRayChunk, csrc/nrt_render.cu
TAIL_SLOTS = 3          # slots a CTA of the NeRFLE kernels runs at most (tc_core.cuh, kMaxSlots)

# per-sample error against float64: (max-abs, RMS), for sigma and for each rgb channel
GATES = {
    "render": {"f16": {"sigma": (8.2e-5, 2.3e-5), "rgb": (5.2e-3, 6.1e-4)},
               "bf16": {"sigma": (5.1e-4, 9.2e-5), "rgb": (4.1e-2, 5.5e-3)}},
    "train": {"f16": {"sigma": (7.7e-5, 2.1e-5), "rgb": (3.1e-3, 4.0e-4)},
              "bf16": {"sigma": (4.9e-4, 8.9e-5), "rgb": (2.6e-2, 3.1e-3)}},
}
OUTPUTS = ("sigma", "r", "g", "b")


def gate(kind, prec, output):
    return GATES[kind][prec]["sigma" if output == "sigma" else "rgb"]


def weights(envmap):
    """synth weights of NeRFLE.first and NeRFLE.second (point light: 70 inputs; environment code: 115)"""
    w1 = synth.mlp_weights(seed=31, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0,
                           w_scale=W_SCALE_FIRST)
    w2 = synth.mlp_weights(seed=32 + int(envmap), in_size=64 + 3 + (48 if envmap else 3), out=3, num_layers=8, hidden=64,
                           freqs=16, sigma=32.0, w_scale=W_SCALE_SECOND)
    return w1, w2


def light_codes(envmap):
    """one distinct light code per view"""
    if envmap:
        return (0.5 * np.random.RandomState(7).standard_normal((N_VIEWS, 48))).astype(np.float32)
    return np.array([[0.4, 1.0, 0.3], [-0.8, 0.3, 0.9], [0.2, -1.1, -0.5]], np.float32)


def ray_counts(S, slots):
    """rays per tile-tail case; slots = tile slots of one full grid (two per SM); 128-sample tiles"""
    if S == 192:        # 1.5 tiles per ray: the division in ray_of
        return {"one_tile": 1, "odd_tiles": 23, "grid_plus_one": (2 * (slots + 1) + 2) // 3, "several_per_slot": 2001}
    assert S == 64      # half a tile per ray: the shift
    return {"one_tile": 1, "odd_tiles": 69, "grid_plus_one": 2 * slots + 1, "several_per_slot": 6 * slots + 3}


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@functools.lru_cache(maxsize=None)
def _nets(envmap):
    w1, w2 = weights(envmap)
    return helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)


# ---- float64 reference: nerf.py:175-203 per sample, on the GPU ----------------------------------------------------
@functools.lru_cache(maxsize=None)
def _weights64(envmap):
    import torch

    def dev(w):
        d = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64, device="cuda")
        return dict(basis=d(w["basis"]), W=[d(x) for x in w["W"]], b=[d(x) for x in w["b"]], L=w["num_layers"],
                    skip=w["skip"])
    return tuple(dev(w) for w in weights(envmap))


def _mlp64(w, x):
    """neural_blocks.py:75-86 (the op order of oracle/port.py::torch_mlp) in float64"""
    import torch
    import torch.nn.functional as Fn
    xb = x @ w["basis"]
    enc = torch.cat([x, xb.sin(), xb.cos()], dim=-1)
    h = Fn.linear(enc, w["W"][0], w["b"][0])
    L = w["L"]
    for i in range(L):
        if i != L - 1 and (i % w["skip"]) == 0:
            h = torch.cat([h, enc], dim=-1)
        h = Fn.linear(Fn.leaky_relu(h), w["W"][1 + i], w["b"][1 + i])
    return Fn.linear(Fn.leaky_relu(h), w["W"][L + 1], w["b"][L + 1])


def _reference(envmap, rays, ts, codes, view):
    """rays [n,6], ts [n,S] (fp32 CUDA, as the kernels get them), codes [V,ld], view [n] int or None ->
    sigma [n,S], rgb [n,S,3] in float64: p = o + t d, NeRFLE.first (sigma = output 0, latent = 1..64),
    NeRFLE.second on [latent | r_d | code[view]], sigmoid"""
    import torch
    w1, w2 = _weights64(envmap)
    n, S = ts.shape
    sig = torch.empty((n, S), dtype=torch.float64, device="cuda")
    rgb = torch.empty((n, S, 3), dtype=torch.float64, device="cuda")
    codes = codes.double()
    step = max(1, 131072 // S)
    with torch.no_grad():
        for r0 in range(0, n, step):
            r = rays[r0:r0 + step].double()
            t = ts[r0:r0 + step].double()
            k = r.shape[0]
            o, d = r[:, :3], r[:, 3:]
            f = _mlp64(w1, (o[:, None, :] + t[..., None] * d[:, None, :]).reshape(-1, 3)).reshape(k, S, 65)
            c = codes[view[r0:r0 + step].long()] if view is not None else codes[:1].expand(k, -1)
            x2 = torch.cat([f[..., 1:], d[:, None, :].expand(k, S, 3), c[:, None, :].expand(k, S, c.shape[-1])], dim=-1)
            sig[r0:r0 + k] = f[..., 0]
            rgb[r0:r0 + k] = torch.sigmoid(_mlp64(w2, x2.reshape(k * S, -1))).reshape(k, S, 3)
    return sig, rgb


# ---- gates ---------------------------------------------------------------------------------------------------------
def _render_tail(R, S, rows):
    """[len(rows), S] mask of the samples in the tail tiles of their 262,144-ray chunk (ray-major, m = ray * S + s)"""
    import torch
    rows = rows.long()
    c0 = rows // CHUNK * CHUNK
    n = torch.clamp(R - c0, max=CHUNK)
    T = (n * S + 127) // 128
    tile = ((rows - c0)[:, None] * S + torch.arange(S, device=rows.device)[None, :]) // 128
    return tile >= (T - TAIL_SLOTS * _sms())[:, None]


def _train_tail(R, S):
    """[R, S] mask of the tail tiles of the training forward (one launch over m = s * R + ray)"""
    import torch
    T = (R * S + 127) // 128
    m = torch.arange(S, device="cuda")[None, :] * R + torch.arange(R, device="cuda")[:, None]
    return m // 128 >= T - TAIL_SLOTS * _sms()


def _stats(sig, rgb, rsig, rrgb, tail):
    """per output: (max-abs, RMS, tail max-abs, tail RMS); all inputs ray-major [n,S] / [n,S,3]"""
    errs = {"sigma": (sig.double() - rsig).abs()}
    for j, name in enumerate(OUTPUTS[1:]):
        errs[name] = (rgb[..., j].double() - rrgb[..., j]).abs()
    out = {}
    for name, e in errs.items():
        te = e[tail]
        out[name] = (float(e.max()), float(e.square().mean().sqrt()),
                     float(te.max()) if te.numel() else 0.0, float(te.square().mean().sqrt()) if te.numel() else 0.0)
    return out


def _assert_gates(kind, prec, label, stats):
    for name, (mx, rms, tmx, trms) in stats.items():
        gmax, grms = gate(kind, prec, name)
        assert np.isfinite([mx, rms, tmx, trms]).all(), (label, name, stats)
        assert mx <= gmax, "%s %s: max error %.3g > %.3g" % (label, name, mx, gmax)
        assert rms <= grms, "%s %s: RMS error %.3g > %.3g" % (label, name, rms, grms)
        assert tmx <= gmax and trms <= grms, "%s %s: tail tiles max %.3g / RMS %.3g" % (label, name, tmx, trms)


def _check(kind, prec, label, sig, rgb, envmap, rays, ts, codes, view, tail):
    rsig, rrgb = _reference(envmap, rays, ts, codes, view)
    _assert_gates(kind, prec, label, _stats(sig, rgb, rsig, rrgb, tail))


def _check_render(prec, label, envmap, rays, ts, codes, view=None, rows=None, R=None, **kw):
    """the render pass on all rays; compared with float64 on `rows` (default all)"""
    import torch
    from neural_raytracing_b200 import ops
    m1, m2 = _nets(envmap)
    sig, rgb = ops.nerfle_render_samples(m1, m2, rays, ts, codes, view_of_ray=view, prec=prec)
    R = rays.shape[0]
    if rows is None:
        rows = torch.arange(R, device="cuda")
    ts_rows = ts[rows] if ts.dim() == 2 else ts[None, :].expand(rows.numel(), -1)
    _check("render", prec, label, sig[rows], rgb[rows], envmap, rays[rows], ts_rows, codes,
           view[rows] if view is not None else None, _render_tail(R, ts.shape[-1], rows))
    return sig, rgb


def _views(R):
    return _t((np.arange(R) % N_VIEWS).astype(np.int32))


def _uniform(S):
    return _t(np.linspace(0.0, T_FAR, S).astype(np.float32))


# ---- B: the render pass --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", ["one_tile", "odd_tiles", "grid_plus_one", "several_per_slot"])
@pytest.mark.parametrize("S", [192, 64])
def test_render_tile_tails(prec, case, S):
    R = ray_counts(S, 2 * _sms())[case]
    rays = _t(synth.camera_rays(40 + S, R))
    _check_render(prec, "render %s S=%d" % (case, S), False, rays, _uniform(S), _t(light_codes(False)[:1]))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("envmap", [False, True], ids=["point_light", "envmap"])
def test_render_views(prec, envmap):
    R = 2001
    rays = _t(synth.camera_rays(41, R))
    _check_render(prec, "render views envmap=%d" % envmap, envmap, rays, _uniform(192), _t(light_codes(envmap)), _views(R))


def _hierarchical_ts(prec, rays, codes, view):
    """the merged 64 + 128 distances the hierarchical render composites over and training trains on: [192, R]"""
    from neural_raytracing_b200 import ops
    m1, m2 = _nets(False)
    return ops.nerfle_sample_hierarchical(m1, m2, rays, codes, view_of_ray=view, prec=prec, n_coarse=64, n_fine=128,
                                          t_near=0.0, t_far=T_FAR, jitter_seed=3)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("sampling", ["stratified", "hierarchical"])
def test_render_per_ray_ts(prec, sampling):
    from oracle import port
    R = 2001
    rays = _t(synth.camera_rays(42, R))
    codes, view = _t(light_codes(False)), _views(R)
    if sampling == "stratified":
        ts = _t(port.stratified_ts(R, 192, 0.0, T_FAR, seed=5))
    else:
        ts = _hierarchical_ts(prec, rays, codes, view).t().contiguous()
    assert ts.shape == (R, 192)
    _check_render(prec, "render %s ts" % sampling, False, rays, ts, codes, view)


def _camera_both_modes(prec, desc, ts, codes):
    import torch
    from neural_raytracing_b200 import ops
    m1, m2 = _nets(False)
    ray_fed = ops.nerfle_render_samples(m1, m2, desc, ts, codes, prec=prec)
    try:
        ops.set_camera_rays_mode(True)
        cam_fed = ops.nerfle_render_samples(m1, m2, desc, ts, codes, prec=prec)
    finally:
        ops.set_camera_rays_mode(False)
    for a, b in zip(ray_fed, cam_fed):
        assert torch.equal(a, b)
    rays, view = ops.camera_rays(desc, want_view=True)
    return ray_fed, rays.reshape(-1, 6), view


@pytest.mark.parametrize("prec", PRECS)
def test_camera_fed_equals_ray_fed(prec):
    """IoNerfFirst<64, true> / IoNerfSecond<64,3,true,true> against k_camera_rays + the ray-fed pass; 2 views with their
    own codes; 2 * 97 * 61 rays * 96 samples is not a multiple of 128"""
    from neural_raytracing_b200 import ops
    c2w, focal = synth.nerf_cameras(2, 400, device="cuda")
    desc = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=400, x0=7, y0=3, nx=97, ny=61)
    S, codes = 96, _t(light_codes(False)[1:])
    assert desc.n_rays * S % 128 != 0
    (sig, rgb), rays, view = _camera_both_modes(prec, desc, _uniform(S), codes)
    _check("render", prec, "camera", sig, rgb, False, rays, _uniform(S)[None, :].expand(rays.shape[0], -1), codes, view,
           _render_tail(rays.shape[0], S, _t(np.arange(rays.shape[0]))))


@pytest.mark.parametrize("prec", PRECS)
def test_camera_chunk_boundary(prec):
    """a camera block of more than 262,144 rays: the second chunk's kernels compute their rays from cam_r0 on"""
    import torch
    from neural_raytracing_b200 import ops
    c2w, focal = synth.nerf_cameras(2, 400, device="cuda")
    desc = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=400, x0=18, y0=18, nx=363, ny=363)
    S, codes = 64, _t(light_codes(False)[:2])
    R = desc.n_rays
    assert CHUNK < R < 2 * CHUNK
    (sig, rgb), rays, view = _camera_both_modes(prec, desc, _uniform(S), codes)
    rows = torch.arange(CHUNK - 2048, R, device="cuda")
    _check("render", prec, "camera chunks", sig[rows], rgb[rows], False, rays[rows],
           _uniform(S)[None, :].expand(rows.numel(), -1), codes, view[rows], _render_tail(R, S, rows))


@pytest.mark.parametrize("prec", PRECS)
def test_render_chunk_boundary(prec):
    """R = 262,144 + 301: the second chunk's rays, views and outputs are offset by r0; the pass is the same as two calls
    split at the boundary, bit for bit"""
    import torch
    from neural_raytracing_b200 import ops
    R, S = CHUNK + 301, 64
    rays = _t(synth.camera_rays(43, R))
    codes, view, ts = _t(light_codes(False)), _views(R), _uniform(S)
    rs = np.random.RandomState(9)
    rows = torch.from_numpy(np.unique(np.concatenate([np.arange(CHUNK - 2048, R), rs.randint(0, R, 4096)]))).cuda()
    sig, rgb = _check_render(prec, "render chunks", False, rays, ts, codes, view, rows=rows)
    m1, m2 = _nets(False)
    parts = [ops.nerfle_render_samples(m1, m2, rays[a:b].contiguous(), ts, codes, view_of_ray=view[a:b].contiguous(),
                                       prec=prec) for a, b in ((0, CHUNK), (CHUNK, R))]
    assert torch.equal(sig, torch.cat([p[0] for p in parts]))
    assert torch.equal(rgb, torch.cat([p[1] for p in parts]))


@pytest.mark.parametrize("envmap", [False, True], ids=["point_light", "envmap"])
def test_f32_equals_oracle(envmap):
    """the fp32 pass through the same entry equals the C oracle bit for bit (per-ray ts for the point light, shared for
    the environment code; three views)"""
    from neural_raytracing_b200 import ops
    from oracle import c_oracle, port
    R, S = 23, 64
    w1, w2 = weights(envmap)
    m1, m2 = _nets(envmap)
    rays = synth.camera_rays(44, R)
    codes = light_codes(envmap)
    view = (np.arange(R) % N_VIEWS).astype(np.int32)
    if envmap:
        ts = np.linspace(0.0, T_FAR, S).astype(np.float32)
        kw = dict(ts=ts)
    else:
        ts = port.stratified_ts(R, S, 0.0, T_FAR, seed=6)
        kw = dict(ts_per_ray=ts)
    _, osig, orgb = c_oracle.nerfle_render(helpers.oracle_mlp(w1), helpers.oracle_mlp(w2), rays, light_code=codes,
                                           view_of_ray=view, store=True, **kw)
    sig, rgb = ops.nerfle_render_samples(m1, m2, _t(rays), _t(ts), _t(codes), view_of_ray=_t(view), prec="f32")
    assert np.array_equal(sig.cpu().numpy(), osig)
    assert np.array_equal(rgb.cpu().numpy(), orgb)


# ---- C: the fused training forward ---------------------------------------------------------------------------------
def _check_train(prec, label, envmap, rays, ts, codes, view):
    """ts [S] or [S,R]; the training forward's sample-major outputs against float64 and against the render pass"""
    from neural_raytracing_b200 import ops
    m1, m2 = _nets(envmap)
    R = rays.shape[0]
    sig_t, rgb_t, _ = ops.nerfle_train_forward(m1, m2, rays, ts, codes, view_of_ray=view, prec=prec)
    sig, rgb = sig_t.t(), rgb_t.transpose(0, 1)                       # ray-major
    S = sig.shape[1]
    ts_r = ts.t().contiguous() if ts.dim() == 2 else ts
    ts_rows = ts_r if ts_r.dim() == 2 else ts_r[None, :].expand(R, -1)
    _check("train", prec, label, sig, rgb, envmap, rays, ts_rows, codes, view, _train_tail(R, S))
    rsig, rrgb = ops.nerfle_render_samples(m1, m2, rays, ts_r, codes, view_of_ray=view, prec=prec)
    for name, a, b in (("sigma", sig, rsig), ("rgb", rgb, rrgb)):
        limit = gate("train", prec, name)[0] + gate("render", prec, name)[0]
        d = float((a - b).abs().max())
        assert d <= limit, "%s: training and render pass differ by %.3g in %s (> %.3g)" % (label, d, name, limit)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", ["one_tile", "odd_tiles", "grid_plus_one", "several_per_slot"])
@pytest.mark.parametrize("S", [192, 64])
def test_train_tile_tails(prec, case, S):
    R = ray_counts(S, 2 * _sms())[case]
    rays = _t(synth.camera_rays(50 + S, R))
    _check_train(prec, "train %s S=%d" % (case, S), False, rays, _uniform(S), _t(light_codes(False)), _views(R))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("envmap", [False, True], ids=["point_light", "envmap"])
@pytest.mark.parametrize("ts_kind", ["shared", "per_sample"])
def test_train_nets(prec, envmap, ts_kind):
    R = 2001
    rays = _t(synth.camera_rays(51, R))
    codes, view = _t(light_codes(envmap)), _views(R)
    ts = _uniform(192) if ts_kind == "shared" else _hierarchical_ts(prec, rays, _t(light_codes(False)), view)
    _check_train(prec, "train %s envmap=%d" % (ts_kind, envmap), envmap, rays, ts, codes, view)
