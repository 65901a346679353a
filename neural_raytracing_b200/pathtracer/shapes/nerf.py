"""Volumetric NeRF models (pytorch3d/pathtracer/shapes/nerf.py): NeRFLE and PlainNeRF."""
import random

import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import config, ops
from ..neural_blocks import SkipConnMLP
from ..utils import dir_to_elev_azim, elev_azim_to_dir


def composite_reference_ops(sigma_raw, rgb, ts):
    """nerf.py:205-213 on sample-major tensors with torch ops (differentiable)."""
    sigma_a = F.relu(sigma_raw)
    shape = (-1,) + (1,) * (sigma_a.dim() - 1)
    alpha = 1 - torch.exp(-sigma_a * ts.reshape(shape))
    cp = torch.cumprod((1 - alpha).clamp(min=1e-10), dim=0)
    cp = torch.roll(cp, 1, 0)
    cp[-1, ...] = 1
    return ((alpha * cp)[..., None] * rgb).sum(dim=0)


class _Composite(torch.autograd.Function):
    """Compositing through the HBM-bound CUDA kernels (forward + backward)."""

    @staticmethod
    def forward(ctx, sigma_raw, rgb, ts):
        s, c, t = sigma_raw.contiguous().float(), rgb.contiguous().float(), ts.contiguous().float()
        ctx.save_for_backward(s, c, t)
        return ops.composite_forward(s, c, t)

    @staticmethod
    def backward(ctx, g):
        s, c, t = ctx.saved_tensors
        gs, gc = ops.composite_backward(s, c, t, g.contiguous().float())
        return gs, gc, None


def composite(sigma_raw, rgb, ts):
    if sigma_raw.is_cuda:
        return _Composite.apply(sigma_raw, rgb, ts)
    return composite_reference_ops(sigma_raw, rgb, ts)


class _CompositeTs(torch.autograd.Function):
    """_Composite with per-sample distances ts [S,...] (hierarchical sampling)."""

    @staticmethod
    def forward(ctx, sigma_raw, rgb, ts):
        s, c, t = sigma_raw.contiguous().float(), rgb.contiguous().float(), ts.contiguous().float()
        ctx.save_for_backward(s, c, t)
        return ops.composite_forward_ts(s, c, t)

    @staticmethod
    def backward(ctx, g):
        s, c, t = ctx.saved_tensors
        gs, gc = ops.composite_backward_ts(s, c, t, g.contiguous().float())
        return gs, gc, None


class HierarchicalSampling:
    """Opt-in NeRF sampling for NeRFLE: n_coarse stratified distances in [t_near, t_far) (jittered within their bins when
    `jitter`), a coarse pass, n_fine distances drawn by inverse-CDF resampling of the coarse weights, and compositing over
    all n_coarse + n_fine samples in ascending order (n_fine = 0: one stratified pass).  An extension: the reference uses
    64 shared uniform distances (nerf.py:178).  Assign an instance to `NeRFLE.sampling`.  CUDA only: the sampling, the
    resampling and the compositing over per-sample distances exist as CUDA kernels alone, so a NeRFLE whose rays are on
    the CPU raises NrtError while `sampling` is set.

    Seeds: gradient-free renders use `render_seed` (fixed, so a frame renders the same image every time); training
    reads the device tensor `train_seed(device)` and advances it by one per forward, so a step captured by
    training.GraphedStep draws new coarse and fine jitter on every replay."""

    def __init__(self, n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter=True):
        n_coarse, n_fine, t_near, t_far = int(n_coarse), int(n_fine), float(t_near), float(t_far)
        if n_coarse < 1 or n_fine < 0:
            raise ValueError("HierarchicalSampling: n_coarse must be >= 1 and n_fine >= 0, got %d / %d" % (n_coarse, n_fine))
        if n_fine > 0 and n_coarse < 3:
            raise ValueError("HierarchicalSampling: n_coarse must be >= 3 when n_fine > 0 (the resampling uses the interior "
                             "coarse samples), got %d" % n_coarse)
        if not t_far > t_near:
            raise ValueError("HierarchicalSampling: t_far (%g) must be greater than t_near (%g)" % (t_far, t_near))
        for name, k in (("n_coarse", n_coarse), ("n_fine", n_fine)):
            if k > 0 and 64 % k != 0 and k % 64 != 0:
                raise ValueError("HierarchicalSampling: %s = %d must divide 64 or be a multiple of 64 (the sample tiling of "
                                 "the fp32 NeRFLE kernel that renders it and runs the fp32 coarse pass)" % (name, k))
        if n_coarse + n_fine > ops.N.MAX_HIER_SAMPLES:
            raise ValueError("HierarchicalSampling: n_coarse + n_fine = %d exceeds %d, the samples per ray the merge kernels "
                             "hold in shared memory" % (n_coarse + n_fine, ops.N.MAX_HIER_SAMPLES))
        self.n_coarse, self.n_fine, self.t_near, self.t_far, self.jitter = n_coarse, n_fine, t_near, t_far, bool(jitter)
        self.render_seed = 0x5EED if self.jitter else 0
        self.seed = None      # device int64 [1], created on the module's device by train_seed()

    @property
    def n_samples(self):
        return self.n_coarse + self.n_fine

    def train_seed(self, device):
        """The device seed of the differentiable forward (None without jitter)."""
        if not self.jitter:
            return None
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if self.seed is None or self.seed.device != device:
            self.seed = torch.ones(1, dtype=torch.int64, device=device)
        return self.seed

    def __repr__(self):
        return "HierarchicalSampling(n_coarse=%d, n_fine=%d, t_near=%g, t_far=%g, jitter=%s)" % (
            self.n_coarse, self.n_fine, self.t_near, self.t_far, self.jitter)


class _NerfleFused(torch.autograd.Function):
    """first MLP -> [latent | r_d | light] -> second MLP -> sigmoid on the tensor-core training kernels, nothing but
    sigma [S,...] and rgb [S,...,3] materialised in fp32 (ops.nerfle_train_forward / _backward).  Gradients reach the
    weights of both MLPs; rays, ts and the light code are treated as constants (as in nerfle.py, where only
    `model.parameters()` are optimised)."""

    @staticmethod
    def forward(ctx, module, rays, ts, code, view, prec, *params):
        p1, p2 = module.first.packed(), module.second.packed()
        sigma, rgb, state = ops.nerfle_train_forward(p1, p2, rays.detach().float(), ts.detach().float(), code.detach().float(), view, prec)
        ctx.p1, ctx.p2, ctx.state, ctx.prec = p1, p2, state, prec
        ctx.fg1, ctx.fg2 = getattr(module.first, "_flat_grad", None), getattr(module.second, "_flat_grad", None)
        if (ctx.fg1 is None) != (ctx.fg2 is None):
            ctx.fg1 = ctx.fg2 = None
        ctx.n1 = len(module.first._flat_params())
        ctx.save_for_backward(rgb)
        lead = tuple(rays.shape[:-1])
        return sigma.reshape((sigma.shape[0],) + lead), rgb.reshape((sigma.shape[0],) + lead + (3,))

    @staticmethod
    def backward(ctx, g_sigma, g_rgb):
        rgb, = ctx.saved_tensors
        g1, g2 = ops.nerfle_train_backward(ctx.p1, ctx.p2, rgb, g_sigma.contiguous().float(), g_rgb.contiguous().float(),
                                           ctx.state, ctx.prec, ctx.fg1, ctx.fg2)
        if ctx.fg1 is not None:      # accumulated straight into training.FlatParameters' gradient buffer
            return (None,) * (6 + 2 * (len(ctx.p1.dims) + len(ctx.p2.dims)))
        flat = []
        for pk, g in ((ctx.p1, g1), (ctx.p2, g2)):
            gW, gb = pk.unpack(g)
            for w, b in zip(gW, gb):
                flat += [w, b]
        return (None, None, None, None, None, None) + tuple(flat)


class NeRFLE(nn.Module):
    """NeRF with a point light / environment-light code (nerf.py:153-214)."""

    def __init__(self, envmap=False, bins=4, device="cuda"):
        super().__init__()
        self.latent_size = 64
        self.first = SkipConnMLP(num_layers=5, hidden_size=128, in_size=3, out=1 + self.latent_size,
                                 device=device).to(device)
        self.bins = bins
        self.second = SkipConnMLP(in_size=self.latent_size + (6 if not envmap else 3 + bins * bins * 3), out=3,
                                  device=device).to(device)
        self.envmap = envmap
        # optional device tensor in [0,1): when set, replaces random.random() of the far-plane jitter (nerf.py:178) so
        # that a CUDA-graph-captured step (neural_raytracing_b200.training.GraphedStep) still jitters per replay
        self.far_jitter = None
        # optional HierarchicalSampling (not a constructor argument: the constructor keeps the reference's signature;
        # not in state_dict).  None: the reference's 64 shared uniform distances.
        self.sampling = None

    def _sample_ts(self, device):
        if getattr(self, "far_jitter", None) is not None:
            return torch.linspace(0, 1, 64, device=device) * (2 + self.far_jitter.reshape(()).to(device) * 0.1)
        return torch.linspace(0, 2 + random.random() * 0.1, 64, device=device)

    def _light_code(self, lights, device):
        """[n_views, 3] light location, or the [n_views, 3*bins^2] environment code (nerf.py:184-197)."""
        if getattr(self, "envmap", False):
            grid = torch.stack(torch.meshgrid(torch.linspace(0, 180, self.bins, device=device),
                                              torch.linspace(0, 45, self.bins, device=device), indexing="ij"),
                               dim=-1).reshape(-1, 2)
            code = lights.envmap(elev_azim_to_dir(grid))
            return code.reshape(code.shape[0], -1)
        return lights.location

    @staticmethod
    def _code_rows(code, n_views):
        """One light-code row per view: a single light broadcasts over the views as it does in nerf.py:199-201 (`expand`)."""
        if code.shape[0] == 1 and n_views > 1:
            return code.expand(n_views, code.shape[-1])
        if code.shape[0] != n_views:
            raise ValueError("light code has %d rows for %d views" % (code.shape[0], n_views))
        return code

    def _view_index(self, rays):
        """[R] int32: which view (light code row) each ray belongs to; cached per batch shape."""
        key = (rays.shape[0], rays[0].numel() // 6, rays.device)
        cache = self.__dict__.setdefault("_view_cache", {})
        if key not in cache:
            cache.clear()
            cache[key] = torch.arange(key[0], device=rays.device, dtype=torch.int32).repeat_interleave(key[1])
        return cache[key]

    def _needs_grad(self, rays):
        return torch.is_grad_enabled() and (rays.requires_grad or any(p.requires_grad for p in self.parameters()))

    def _render_sampling(self):
        """nerfle_render keyword arguments of `sampling` for a gradient-free render."""
        s = self.sampling
        return dict(n_coarse=s.n_coarse, n_fine=s.n_fine, t_near=s.t_near, t_far=s.t_far, jitter_seed=s.render_seed)

    def render_camera(self, cam, lights):
        """The frame of `cam` (ops.CameraDesc) in one library call, rays generated on the device inside it (f4):
        what pathtrace's tile loop + sample_positions + forward compute for an inference render (main.py:57-88,
        nerf.py:175-214), with ONE far-plane draw (nerf.py:178) per frame instead of one per tile (with `sampling` set:
        its hierarchical samples, seeded by sampling.render_seed).
        -> rgb [n_views, nx, ny, bundle, 3]."""
        device = cam.device
        code = self._code_rows(self._light_code(lights, device), cam.n_views)
        prec = config.precision if self.first.precision() != "f32" and self.second.precision() != "f32" else "f32"
        if getattr(self, "sampling", None) is not None:
            return ops.nerfle_render_camera(self.first.packed(), self.second.packed(), cam, None, code.detach().float(),
                                            prec=prec, **self._render_sampling())
        ts = self._sample_ts(device)
        return ops.nerfle_render_camera(self.first.packed(), self.second.packed(), cam, ts, code.detach().float(),
                                        prec=prec)

    def forward(self, rays, lights):
        """nerf.py:175-214.  With `sampling` (a HierarchicalSampling) set, the samples are its stratified coarse +
        importance-resampled fine distances instead of the reference's 64 shared ones, and neither `far_jitter` nor
        random.random() is used: a gradient-free forward renders with sampling.render_seed; a differentiable one takes
        the merged distances from a no-grad coarse pass (at the train precision) seeded by the device tensor
        sampling.train_seed(), advances that seed by one, and trains both MLPs on all n_coarse + n_fine samples (the
        light code is a constant there, as on the fused path)."""
        if getattr(self, "sampling", None) is not None:
            return self._forward_hierarchical(rays, lights)
        r_o, r_d = rays.split([3, 3], dim=-1)
        device = r_o.device
        ts = self._sample_ts(device)
        code = self._code_rows(self._light_code(lights, device), rays.shape[0])
        if rays.is_cuda and not self._needs_grad(rays):
            # fused render: rays in, rgb out
            view = self._view_index(rays)
            # the fused tensor-core render instantiates the point-light and the bins = 4 environment net only: any
            # other shape keeps the exact fp32 kernel (SkipConnMLP.precision() knows which shapes are instantiated)
            prec = config.precision if self.first.precision() != "f32" and self.second.precision() != "f32" else "f32"
            return ops.nerfle_render(self.first.packed(), self.second.packed(), rays.detach().float(), ts,
                                     code.detach().float(), view, prec=prec)
        # differentiable path: fused MLP kernels where available + CUDA compositing
        tprec = self.first.train_precision()
        if rays.is_cuda and tprec != "f32" and self.second.train_precision() == tprec and not rays.requires_grad \
                and not code.requires_grad:
            view = self._view_index(rays)
            alpha, rgb = _NerfleFused.apply(self, rays, ts, code, view, tprec, *self.first._flat_params(),
                                            *self.second._flat_params())
            return composite(alpha, rgb, ts)
        pts = r_o.unsqueeze(0) + torch.tensordot(ts, r_d, dims=0)
        first_out = self.first(pts)
        latent, alpha = first_out[..., 1:], first_out[..., 0]
        lead = latent.shape[:-1]
        light = code.reshape((1, code.shape[0]) + (1,) * (len(lead) - 2) + (-1,)).expand(lead + (-1,))
        rgb = self.second(torch.cat([latent, r_d[None, ...].expand(lead + (3,)), light], dim=-1), out_act=ops.OUT_SIGMOID)
        return composite(alpha, rgb, ts)

    def _forward_hierarchical(self, rays, lights):
        s = self.sampling
        if not rays.is_cuda:
            raise ops.NrtError("NeRFLE.sampling (%r) runs on the CUDA kernels only; the rays are on %s -- set "
                               "sampling = None for the reference's sampling on the CPU" % (s, rays.device))
        r_o, r_d = rays.split([3, 3], dim=-1)
        # the light code is a constant here, as on the fused path (nerfle.py optimises model.parameters() only)
        code = self._code_rows(self._light_code(lights, rays.device), rays.shape[0]).detach().float()
        view = self._view_index(rays)
        if not self._needs_grad(rays):
            prec = config.precision if self.first.precision() != "f32" and self.second.precision() != "f32" else "f32"
            return ops.nerfle_render(self.first.packed(), self.second.packed(), rays.detach().float(), None, code, view,
                                     prec=prec, **self._render_sampling())
        tprec = self.first.train_precision()
        fused = tprec != "f32" and self.second.train_precision() == tprec and not rays.requires_grad
        seed = s.train_seed(rays.device)
        with torch.no_grad():
            ts = ops.nerfle_sample_hierarchical(self.first.packed(), self.second.packed(), rays.detach().float(), code,
                                                view, prec=tprec if fused else "f32",
                                                n_coarse=s.n_coarse, n_fine=s.n_fine, t_near=s.t_near, t_far=s.t_far,
                                                seed=seed)
            if seed is not None:
                seed.add_(1)
        lead = tuple(rays.shape[:-1])
        if fused:
            alpha, rgb = _NerfleFused.apply(self, rays, ts, code, view, tprec, *self.first._flat_params(),
                                            *self.second._flat_params())
            return _CompositeTs.apply(alpha, rgb, ts.reshape(alpha.shape))
        ts = ts.reshape((s.n_samples,) + lead)
        pts = r_o.unsqueeze(0) + ts[..., None] * r_d.unsqueeze(0)
        first_out = self.first(pts)
        latent, alpha = first_out[..., 1:], first_out[..., 0]
        light = code.reshape((1, code.shape[0]) + (1,) * (len(lead) - 1) + (-1,)).expand(latent.shape[:-1] + (-1,))
        rgb = self.second(torch.cat([latent, r_d[None, ...].expand(latent.shape[:-1] + (3,)), light], dim=-1),
                          out_act=ops.OUT_SIGMOID)
        return _CompositeTs.apply(alpha, rgb, ts)


class PlainNeRF(nn.Module):
    """Per-image-latent NeRF (nerf.py:9-74)."""

    def __init__(self, latent_size: int = 32, intermediate_size: int = 32, steps=32, device="cuda"):
        super().__init__()
        self.latent = None
        self.latent_size = latent_size
        self.steps = steps
        self.first = SkipConnMLP(in_size=3, out=1 + intermediate_size, latent_size=latent_size, num_layers=5,
                                 hidden_size=32, device=device).to(device)
        self.second = SkipConnMLP(in_size=2, out=3, latent_size=latent_size + intermediate_size, num_layers=5,
                                  hidden_size=32, device=device).to(device)

    def assign_latent(self, latent):
        assert latent.shape[-1] == self.latent_size
        assert len(latent.shape) == 2, "expected latent in [B, L]"
        self.latent = latent

    def forward(self, rays, lights):
        assert self.latent is not None
        r_o, r_d = rays.split([3, 3], dim=-1)
        ts = torch.linspace(0.4, 2 + random.random() * 0.1, self.steps, device=r_o.device)
        pts = r_o.unsqueeze(0) + torch.tensordot(ts, r_d, dims=0)
        latent = self.latent[None, :, None, None, None, :].expand(pts.shape[:-1] + (-1,))
        first_out = self.first(pts, latent)
        alpha, inter = first_out[..., 0], first_out[..., 1:]
        view = dir_to_elev_azim(r_d)[None, ...].expand(latent.shape[:-1] + (2,))
        rgb = self.second(view, torch.cat([inter, latent], dim=-1)).tanh()
        alpha = alpha + torch.randn_like(alpha) * 1e-3      # nerf.py:66
        return (composite(alpha, rgb, ts) + 1) / 2
