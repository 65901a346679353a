"""Numpy restatement of the occupancy grid (include/nrt_b200.h, nrt_occupancy_t): the update points, the cell of a sample
point, the cull decision, the update rule and the bit words; and a restatement of the culled hierarchical render."""
import numpy as np

from oracle import port

F32 = np.float32


def box(res, bbox_min, bbox_max):
    """(lo, inv, h) per axis as the library rounds them: inv = res / (hi - lo), h = (hi - lo) / res in double, then fp32."""
    lo = np.asarray(bbox_min, F32)
    span = np.asarray(bbox_max, F32).astype(np.float64) - lo.astype(np.float64)
    return lo, (float(res) / span).astype(F32), (span / float(res)).astype(F32)


def update_points(res, bbox_min, bbox_max, points_per_cell, seed):
    """[res^3 * ppc, 3]: point q of cell c at lo + (idx + u) * h, every operation rounded in fp32."""
    lo, _, h = box(res, bbox_min, bbox_max)
    c = np.repeat(np.arange(res ** 3, dtype=np.int64), points_per_cell)
    q = np.tile(np.arange(points_per_cell, dtype=np.int64), res ** 3)
    idx = np.stack([c // (res * res), (c // res) % res, c % res], axis=-1)
    out = np.empty((c.size, 3), F32)
    for a in range(3):
        u = port.hash_u01(seed, c, 3 * q + a) if seed else np.full(c.size, 0.5, F32)
        out[:, a] = lo[a] + (idx[:, a].astype(F32) + u.astype(F32)) * h[a]
    return out


def sample_points(rays, ts):
    """p = o + t d of every sample [R,S,3] as the kernels form it (one fused multiply-add per axis)."""
    rays = np.asarray(rays, F32).reshape(-1, 6)
    t = np.asarray(ts, F32)
    t = np.broadcast_to(t[None, :], (rays.shape[0], t.size)) if t.ndim == 1 else t
    o, d = rays[:, None, :3].astype(np.float64), rays[:, None, 3:].astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        return (t[..., None].astype(np.float64) * d + o).astype(F32)


def cell_coords(p, res, bbox_min, bbox_max):
    """u = (p - lo) * inv per axis in fp32 (cell units); inside iff every axis is in [0, res)."""
    lo, inv, _ = box(res, bbox_min, bbox_max)
    with np.errstate(invalid="ignore", over="ignore"):
        u = ((np.asarray(p, F32) - lo) * inv).astype(F32)
        inside = np.all((u >= 0) & (u < F32(res)), axis=-1)
    return u, inside


def cell_index(p, res, bbox_min, bbox_max):
    """(inside [..], linear cell index [..], -1 outside) of points p [..., 3]."""
    u, inside = cell_coords(p, res, bbox_min, bbox_max)
    ijk = np.where(inside[..., None], np.floor(np.nan_to_num(u)), 0).astype(np.int64)
    c = (ijk[..., 0] * res + ijk[..., 1]) * res + ijk[..., 2]
    return inside, np.where(inside, c, -1)


def near_face(p, res, bbox_min, bbox_max, rel=1e-6):
    """Samples within rel * h of a cell face (where fp32 rounding may put them in either cell), in float64."""
    lo = np.asarray(bbox_min, np.float64)
    span = np.asarray(bbox_max, np.float64) - lo
    with np.errstate(invalid="ignore"):
        u = (np.asarray(p, np.float64) - lo) / span * res
        return np.any(np.abs(u - np.round(u)) < rel, axis=-1) & np.all(np.isfinite(u), axis=-1)


def pack_bits(occ):
    """bool [res^3] -> int32 words [ceil(res^3 / 32)]: bit c & 31 of word c >> 5."""
    occ = np.asarray(occ, bool).reshape(-1)
    pad = np.zeros((occ.size + 31) // 32 * 32, bool)
    pad[:occ.size] = occ
    w = (pad.reshape(-1, 32).astype(np.uint64) << np.arange(32, dtype=np.uint64)).sum(axis=1)
    return w.astype(np.uint32).view(np.int32)


def unpack_bits(words, n):
    w = np.asarray(words).view(np.uint32).astype(np.uint64)
    return ((w[:, None] >> np.arange(32, dtype=np.uint64)) & 1).astype(bool).reshape(-1)[:n]


def keep_mask(words, res, bbox_min, bbox_max, rays, ts):
    """bool [R,S]: False iff the sample's point is inside the box and its cell's bit is clear."""
    p = sample_points(rays, ts)
    inside, c = cell_index(p, res, bbox_min, bbox_max)
    occ = unpack_bits(words, res ** 3)
    return ~inside | occ[np.maximum(c, 0)]


def update_rule(density, sigma_raw, decay, threshold):
    """density [res^3], sigma_raw [res^3, ppc] -> (density', occupied bool): max(decay * density, max_q relu(sigma))."""
    m = np.max(np.maximum(np.asarray(sigma_raw, F32), F32(0)), axis=1)
    d = np.maximum((F32(decay) * np.asarray(density, F32)).astype(F32), m)
    return d, d > F32(threshold)


def render_hierarchical_culled(first, second, rays, light_code, n_coarse, n_fine, t_near, t_far, seed, words, res,
                               bbox_min, bbox_max):
    """port.nerfle_render_hierarchical with sigma_raw = 0 at culled samples of both passes (alpha = 0 there, so their
    rgb does not matter).  -> (rgb [R,3], ts_c [R,Sc], ts_f [R,Sf])."""
    from oracle import c_oracle
    rays = np.ascontiguousarray(rays, F32).reshape(-1, 6)
    R = rays.shape[0]
    ts_c = port.stratified_ts(R, n_coarse, t_near, t_far, seed)
    _, sig_c, rgb_c = c_oracle.nerfle_render(first, second, rays, ts_per_ray=ts_c, light_code=light_code, store=True)
    sig_c = np.where(keep_mask(words, res, bbox_min, bbox_max, rays, ts_c), sig_c, F32(0))
    ts_f = port.sample_pdf(sig_c, ts_c, n_fine, seed)
    _, sig_f, rgb_f = c_oracle.nerfle_render(first, second, rays, ts_per_ray=ts_f, light_code=light_code, store=True)
    sig_f = np.where(keep_mask(words, res, bbox_min, bbox_max, rays, ts_f), sig_f, F32(0))
    t_all = np.concatenate([ts_c, ts_f], axis=1)
    order = np.argsort(t_all, axis=1, kind="stable")
    rows = np.arange(R)[:, None]
    sig = np.concatenate([sig_c, sig_f], axis=1)[rows, order]
    rgb = np.concatenate([rgb_c, rgb_f], axis=1)[rows, order]
    return port.composite_ray_major(sig, rgb, t_all[rows, order]), ts_c, ts_f


def composite64(sigma_raw, rgb, ts):
    """The render's compositing (nerf.py:205-213, k_merge_composite) in float64 on ray-major arrays."""
    s = np.asarray(sigma_raw, np.float64)
    t = np.broadcast_to(np.asarray(ts, np.float64), s.shape)
    a = 1.0 - np.exp(-np.maximum(s, 0.0) * t)
    cp = np.roll(np.cumprod(np.maximum(1.0 - a, 1e-10), axis=1), 1, axis=1)
    cp[:, -1] = 1.0
    return ((a * cp)[..., None] * np.asarray(rgb, np.float64)).sum(axis=1)
