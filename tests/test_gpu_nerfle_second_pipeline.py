"""NeRFLE.second's point-light kernels with the tile boundary pipelined (NRT_SECOND_PIPE, csrc/tc_core.cuh): a slot copies
its next tile's packed latent into shared memory one tile ahead, writes that tile's x_hi / x_lo while its current tile's
last hidden layer runs, and hands the next tile's phase GEMM to the MMA warp before its own fused output layer.  A sample
evaluated on the wrong tile's latent is invisible in a composited frame, so every sample is compared with float64 here,
through the render's own chunk loop (nrt_nerfle_render_samples) and the reference and gates of
test_gpu_nerfle_samples.py, at tile counts that reach every tail of that hand-off:
  * a sample count that is not a multiple of 128;
  * fewer tiles than 3 x grid (three slots per CTA, one CTA per SM): slots with no tile and with exactly one;
  * exactly 3 x grid tiles, and one tile fewer and more (one slot with a second tile); two and four tiles per slot
    (from the third tile on, a slot's latent was prefetched under the tile before the previous one);
  * S = 64 and S = 192;
  * three views with their own light codes (view_of_ray = r % 3);
  * the 262,144-ray chunk boundary.
The camera-fed kernels (IoNerfSecond<64, 3, true, true>) equal the ray-fed ones bit for bit at the same tile counts, and
the pass does not depend on the launch: the same rays rendered whole and as two windows, bit for bit."""
import numpy as np
import pytest

import synth
import test_gpu_nerfle_samples as ns

pytestmark = pytest.mark.gpu

SLOTS_PER_CTA = 3      # NetNerfSecondPT: 3 x 160 TMEM columns


def _tiles_to_rays(ntiles, S):
    """smallest ray count whose R * S samples take at least `ntiles` 128-sample tiles.  S = 64: exactly `ntiles`, the
    last one half full; S = 192 (1.5 tiles a ray) reaches only tile counts that are not 1 mod 3: one more there"""
    R = (ntiles * 128 + S - 1) // S
    while ((R - 1) * S + 127) // 128 >= ntiles:
        R -= 1
    if S == 64:
        R = 2 * ntiles - 1
        assert (R * S + 127) // 128 == ntiles and (R * S) % 128 != 0
    return R


def _cases():
    g = SLOTS_PER_CTA * ns._sms()
    return {"partial_tile": 35, "below_grid": g - 2, "grid_minus_one": g - 1, "grid": g, "grid_plus_one": g + 1,
            "two_per_slot": 2 * g + 5, "four_per_slot": 4 * g + 7}


@pytest.mark.parametrize("prec", ns.PRECS)
@pytest.mark.parametrize("case", ["partial_tile", "below_grid", "grid_minus_one", "grid", "grid_plus_one", "two_per_slot",
                                  "four_per_slot"])
@pytest.mark.parametrize("S", [64, 192])
def test_tile_counts_vs_float64(prec, case, S):
    R = _tiles_to_rays(_cases()[case], S)
    rays = ns._t(synth.camera_rays(60 + S, R))
    ns._check_render(prec, "second pipe %s S=%d" % (case, S), False, rays, ns._uniform(S), ns._t(ns.light_codes(False)),
                     ns._views(R))


@pytest.mark.parametrize("prec", ns.PRECS)
def test_chunk_boundary_vs_float64(prec):
    """R = 262,144 + 301 at S = 64: the second chunk's launch starts over at tile 0 of its own latent"""
    import torch
    R, S = ns.CHUNK + 301, 64
    rays = ns._t(synth.camera_rays(61, R))
    rs = np.random.RandomState(11)
    rows = torch.from_numpy(np.unique(np.concatenate([np.arange(ns.CHUNK - 4096, R), rs.randint(0, R, 4096)]))).cuda()
    ns._check_render(prec, "second pipe chunks", False, rays, ns._uniform(S), ns._t(ns.light_codes(False)), ns._views(R),
                     rows=rows)


@pytest.mark.parametrize("prec", ns.PRECS)
@pytest.mark.parametrize("case", ["below_grid", "grid_plus_one"])
def test_camera_fed_equals_ray_fed(prec, case):
    """the camera-fed kernels compute direction and view a tile ahead with cam_ray; 2 views with their own codes"""
    from neural_raytracing_b200 import ops
    c2w, focal = synth.nerf_cameras(2, 400, device="cuda")
    S = 64
    R = _tiles_to_rays(_cases()[case], S)
    nx = 61
    ny = max(1, R // (2 * nx))
    desc = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=400, x0=5, y0=9, nx=nx, ny=ny)
    codes = ns._t(ns.light_codes(False)[:2])
    (sig, rgb), rays, view = ns._camera_both_modes(prec, desc, ns._uniform(S), codes)
    ns._check("render", prec, "second pipe camera", sig, rgb, False, rays,
              ns._uniform(S)[None, :].expand(rays.shape[0], -1), codes, view,
              ns._render_tail(rays.shape[0], S, ns._t(np.arange(rays.shape[0]))))


@pytest.mark.parametrize("prec", ns.PRECS)
def test_does_not_depend_on_the_launch(prec):
    """the same rays whole and as two windows (four tiles per slot): 1,001 * 192 samples are not a multiple of 128, so
    every sample of the second window sits in another tile, lane and slot"""
    import torch
    from neural_raytracing_b200 import ops
    m1, m2 = ns._nets(False)
    R0 = 1001
    R = _tiles_to_rays(4 * SLOTS_PER_CTA * ns._sms() + 7, 192)
    assert R0 < R
    rays = ns._t(synth.camera_rays(62, R))
    codes, view, ts = ns._t(ns.light_codes(False)), ns._views(R), ns._uniform(192)
    whole = ops.nerfle_render_samples(m1, m2, rays, ts, codes, view_of_ray=view, prec=prec)
    parts = [ops.nerfle_render_samples(m1, m2, rays[a:b].contiguous(), ts, codes, view_of_ray=view[a:b].contiguous(),
                                       prec=prec) for a, b in ((0, R0), (R0, R))]
    for k in range(2):
        assert torch.isfinite(whole[k]).all()
        assert torch.equal(whole[k], torch.cat([p[k] for p in parts]))
