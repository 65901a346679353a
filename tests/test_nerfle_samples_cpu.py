"""The per-sample gates of tests/test_gpu_nerfle_samples.py have power: on its networks and inputs (C oracle, fp32), the
errors an indexing bug in the NeRFLE render or training kernels would make -- a sample evaluated on the next sample of its
ray, on the same sample of the neighbouring ray, on the sample one 128-sample tile later, rgb with another view's light
code, rgb from the latent of the sample one tile later with its own direction -- move at least one sample of every tile they touch by
more than 10x the f16 gate and 3x the bf16 gate, and move at least 90 % of the samples they touch beyond the f16 gate.
A later change that loosens a gate or swaps in flatter networks fails here."""
import numpy as np
import pytest

import helpers
import synth
import test_gpu_nerfle_samples as G
from oracle import c_oracle

R, S = 48, 192


def _scene(envmap):
    w1, w2 = G.weights(envmap)
    o1, o2 = helpers.oracle_mlp(w1), helpers.oracle_mlp(w2)
    rays = synth.camera_rays(60 + int(envmap), R)
    ts = np.linspace(0.0, G.T_FAR, S).astype(np.float32)
    codes = G.light_codes(envmap)
    view = (np.arange(R) % G.N_VIEWS).astype(np.int32)
    _, sig, rgb = c_oracle.nerfle_render(o1, o2, rays, ts=ts, light_code=codes, view_of_ray=view, store=True)
    return o1, o2, rays, ts, codes, view, sig.astype(np.float64), rgb.astype(np.float64)


def _second(o2, latent, d, code):
    """NeRFLE.second on [latent | r_d | code], sigmoid; all [R,S,...]"""
    x = np.concatenate([latent, d, code], axis=-1).reshape(R * S, -1)
    return c_oracle.mlp_forward(o2, x, out_act=c_oracle.OUT_SIGMOID).reshape(R, S, 3).astype(np.float64)


def _planted(envmap):
    """name -> (sigma, rgb, affected [R,S] bool) with the error planted"""
    o1, o2, rays, ts, codes, view, sig, rgb = _scene(envmap)
    flat = lambda a: a.reshape((R * S,) + a.shape[2:])
    out = {}
    s2, r2 = sig.copy(), rgb.copy()
    s2[:, :-1], r2[:, :-1] = sig[:, 1:], rgb[:, 1:]
    aff = np.zeros((R, S), bool)
    aff[:, :-1] = True
    out["next sample on the ray"] = (s2, r2, aff)
    s2, r2 = sig.copy(), rgb.copy()
    s2[:-1], r2[:-1] = sig[1:], rgb[1:]
    aff = np.zeros((R, S), bool)
    aff[:-1] = True
    out["same sample of the next ray"] = (s2, r2, aff)
    s2, r2 = flat(sig).copy(), flat(rgb).copy()
    s2[:-128], r2[:-128] = flat(sig)[128:], flat(rgb)[128:]
    aff = np.zeros(R * S, bool)
    aff[:-128] = True
    out["sample one tile later"] = (s2.reshape(R, S), r2.reshape(R, S, 3), aff.reshape(R, S))
    p = (rays[:, None, :3] + ts[None, :, None] * rays[:, None, 3:]).astype(np.float32)
    latent = c_oracle.mlp_forward(o1, p.reshape(-1, 3)).reshape(R, S, 65)[..., 1:]
    d = np.broadcast_to(rays[:, None, 3:], (R, S, 3))
    code = lambda v: np.broadcast_to(codes[v][:, None, :], (R, S, codes.shape[1]))
    assert np.abs(_second(o2, latent, d, code(view)) - rgb).max() < 1e-5     # the restatement is the render's
    out["another view's light code"] = (sig, _second(o2, latent, d, code((view + 1) % G.N_VIEWS)), np.ones((R, S), bool))
    lat2 = latent.reshape(R * S, -1).copy()
    lat2[:-128] = lat2[128:]
    aff = np.zeros(R * S, bool)
    aff[:-128] = True
    out["the latent of the sample one tile later"] = (sig, _second(o2, lat2.reshape(R, S, -1), d, code(view)), aff.reshape(R, S))
    return sig, rgb, out


@pytest.fixture(scope="module", params=[False, True], ids=["point_light", "envmap"])
def planted(request):
    return _planted(request.param)


def _score(kind, prec, sig, rgb, s2, r2):
    """per sample: the largest output change in units of that output's max-abs gate"""
    sc = np.abs(s2 - sig) / G.gate(kind, prec, "sigma")[0]
    return np.maximum(sc, (np.abs(r2 - rgb) / G.gate(kind, prec, "rgb")[0]).max(axis=-1))


@pytest.mark.parametrize("kind", ["render", "train"])
def test_planted_errors_exceed_the_gates(planted, kind):
    sig, rgb, cases = planted
    for name, (s2, r2, aff) in cases.items():
        f16 = _score(kind, "f16", sig, rgb, s2, r2).reshape(-1)
        bf16 = _score(kind, "bf16", sig, rgb, s2, r2).reshape(-1)
        a = aff.reshape(-1)
        tiles = np.unique(np.nonzero(a)[0] // 128)
        for t in tiles:
            sl = slice(t * 128, (t + 1) * 128)
            assert (f16[sl][a[sl]] > 10).any() and (bf16[sl][a[sl]] > 3).any(), \
                "%s: tile %d moves by at most %.2fx the f16 gate / %.2fx the bf16 gate" % (
                    name, t, f16[sl][a[sl]].max(), bf16[sl][a[sl]].max())
        share = float((f16[a] > 1).mean())
        assert share >= 0.9, "%s: only %.3f of the affected samples exceed the f16 gate" % (name, share)
