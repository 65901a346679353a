"""Deterministic synthetic weights / rays shared by tests/golden/make_golden.py (which loads them
into the UNMODIFIED reference modules) and by the tests (which load them into the oracle and
into the CUDA path).  numpy's legacy RandomState stream is frozen across numpy versions, so
fixtures only need to store inputs and reference outputs, never weights."""
import numpy as np


def mlp_weights(seed, in_size, out, num_layers, hidden, freqs, sigma, latent=0, skip=3,
                w_scale=1.0, zero=False):
    """torch-layout weights of a SkipConnMLP (neural_blocks.py:36-55): list order
    [init, layers[0..L-1], out]; W [N,K] ~ U(-1/sqrt(K), 1/sqrt(K)) * w_scale."""
    rs = np.random.RandomState(seed)
    basis = (sigma * rs.standard_normal((freqs, in_size))).astype(np.float32).T.copy()  # [in, freqs]
    dim_p = in_size + 2 * freqs + latent
    shapes = [(hidden, dim_p)]
    for i in range(num_layers):
        sk = (i % skip) == 0 and i != num_layers - 1
        shapes.append((hidden, hidden + (dim_p if sk else 0)))
    shapes.append((out, hidden))
    W, b = [], []
    for (n, k) in shapes:
        bound = w_scale / np.sqrt(k)
        W.append(rs.uniform(-bound, bound, size=(n, k)).astype(np.float32) * (0 if zero else 1))
        b.append(rs.uniform(-bound, bound, size=(n,)).astype(np.float32) * (0 if zero else 1))
    return dict(in_size=in_size, out=out, num_layers=num_layers, hidden=hidden, freqs=freqs,
                latent=latent, skip=skip, basis=basis, W=W, b=b)


def sdf_weights(seed, n=64, hidden=128, num_layers=8, freqs=32, shift_std=0.02):
    """SphereSDF parameters (sdfs.py:17-31): centers 0.3U-0.15, radii 0.2U-0.1, tfs small
    (the constructor uses zeros; a small perturbation exercises the affine warp), and the
    residual MLP `shift` ~ N(0, shift_std) instead of the constructor's zero-init, which would
    hide MLP errors (SURVEY.md section 8c)."""
    rs = np.random.RandomState(seed)
    centers = (0.3 * rs.uniform(size=(n, 3)) - 0.15).astype(np.float32)
    radii = (0.2 * rs.uniform(size=(n,)) - 0.1).astype(np.float32)
    tfs = (0.05 * rs.standard_normal((n, 3, 3))).astype(np.float32)
    m = mlp_weights(seed + 1, 3, 1, num_layers, hidden, freqs, 32.0)
    for i in range(len(m["W"])):
        m["W"][i] = (shift_std * rs.standard_normal(m["W"][i].shape)).astype(np.float32)
        m["b"][i] = (shift_std * rs.standard_normal(m["b"][i].shape)).astype(np.float32)
    return dict(n=n, centers=centers, radii=radii, tfs=tfs, shift=m)


def camera_rays(seed, n_rays, dist=1.0, jitter=0.35):
    """Rays from points on a sphere of radius `dist` looking roughly at the origin."""
    rs = np.random.RandomState(seed)
    o = rs.standard_normal((n_rays, 3))
    o = dist * o / np.linalg.norm(o, axis=-1, keepdims=True)
    d = -o + jitter * rs.standard_normal((n_rays, 3))
    d = d / np.linalg.norm(d, axis=-1, keepdims=True)
    return np.concatenate([o, d], -1).astype(np.float32)


def _name_seed(name, seed):
    h = 2166136261
    for ch in (name + "#%d" % seed).encode():
        h = ((h ^ ch) * 16777619) & 0xFFFFFFFF
    return h


def fill_module(mod, seed, shift_std=None):
    """Deterministically (re)initialises every nn.Parameter and every SkipConnMLP.basis_p of `mod`
    from the parameter NAME, so a reference module and its drop-in mirror (same attribute names)
    receive identical weights.  Linear weights ~ U(+-1/sqrt(fan_in)); if shift_std is given every
    parameter whose name contains 'shift.' is N(0, shift_std) instead (SphereSDF residual MLP)."""
    import torch
    with torch.no_grad():
        for name, p in sorted(mod.named_parameters(), key=lambda kv: kv[0]):
            rs = np.random.RandomState(_name_seed(name, seed))
            if shift_std is not None and "shift." in name:
                v = shift_std * rs.standard_normal(tuple(p.shape))
            elif name.endswith("centers"):
                v = 0.3 * rs.uniform(size=tuple(p.shape)) - 0.15
            elif name.endswith("radii"):
                v = 0.2 * rs.uniform(size=tuple(p.shape)) - 0.1
            elif name.endswith("tfs"):
                v = 0.05 * rs.standard_normal(tuple(p.shape))
            elif name.endswith("color"):
                v = rs.uniform(-0.5, 0.5, size=tuple(p.shape))
            else:
                fan_in = p.shape[1] if p.dim() >= 2 else max(1, p.shape[0])
                b = 1.0 / np.sqrt(fan_in)
                v = rs.uniform(-b, b, size=tuple(p.shape))
            p.copy_(torch.from_numpy(np.asarray(v, np.float32)).to(p.device))
        for name, m in sorted(mod.named_modules(), key=lambda kv: kv[0]):
            if hasattr(m, "basis_p") and hasattr(m, "dim_p"):
                rs = np.random.RandomState(_name_seed(name + ".basis_p", seed))
                shape = tuple(m.basis_p.shape)            # [in, freqs]
                sigma = float(getattr(m, "_synth_sigma", 32.0))
                m.basis_p = torch.from_numpy((sigma * rs.standard_normal(shape)).astype(np.float32)).to(m.basis_p.device)
    return mod


def nerf_cameras(n_views, size, device="cpu"):
    """cam_to_world [N,4,4] on the unit sphere looking at the origin (NeRF convention: -z forward) + focal."""
    import torch
    mats = []
    for i in range(n_views):
        az, el = 0.5 + 0.9 * i, 0.35 + 0.1 * i
        c = np.array([np.cos(el) * np.sin(az), np.sin(el), np.cos(el) * np.cos(az)])
        fwd = -c / np.linalg.norm(c)
        right = np.cross(fwd, [0, 1, 0]); right /= np.linalg.norm(right)
        up = np.cross(right, fwd)
        m = np.eye(4)
        m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = right, up, -fwd, c
        mats.append(m)
    return torch.tensor(np.stack(mats), dtype=torch.float, device=device), 0.5 * size / np.tan(np.radians(25))


class GoldenRatioSampler:
    """Deterministic stand-in for the path tracer's Sampler (samplers.py:14-20): call c returns
    frac((i + 1 + 977 c) * phi), i the flat index.  The same class body is used by tests/golden/make_golden.py for the
    reference run, so both sides trace the same bounces."""

    def __init__(self):
        self.calls = 0

    def sample(self, shape, device="cpu"):
        import torch
        n = int(np.prod(shape))
        i = torch.arange(n, dtype=torch.float64) + 1 + 977 * self.calls
        self.calls += 1
        return ((i * 0.6180339887498949) % 1.0).float().reshape(tuple(shape)).to(device)


def pack_grad(x):
    """A reference gradient as float16 times a power-of-two float32 scale (stored as `<key>` and `<key>_scale`): every
    element is kept, at half the bytes of float32, so the gradient fixtures stay under 1 MB.  The scale maps the largest
    magnitude into [2**14, 2**15]: every element above 2**-29 of it keeps 11 significant bits (relative error <= 2**-11),
    smaller ones lose precision down to zero, and decoding is exact.  On the stored reference gradients this moves every
    cosine (whole vector and per tensor) by less than 1e-7; the norm checks use norms stored in float64."""
    x = np.asarray(x, np.float32)
    m = float(np.abs(x).max()) if x.size else 0.0
    scale = np.float32(2.0 ** (int(np.ceil(np.log2(m))) - 15)) if m > 0 else np.float32(1.0)
    return (x / scale).astype(np.float16), scale


def unpack_grad(g, key):
    """float64 value of a gradient stored with pack_grad."""
    return g[key].astype(np.float64) * float(g[key + "_scale"])
