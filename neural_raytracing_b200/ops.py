"""Functional ops on CUDA tensors.  Thin marshalling over the C ABI of libnrt_b200.so
(include/nrt_b200.h): torch only provides device memory and the current stream.

No fallback exists: a non-CUDA / non-fp32 / non-contiguous tensor, a missing library or a failed
kernel raises."""
import ctypes
from typing import List, Optional, Sequence

import torch

from . import _native as N
from ._native import (ACT_LEAKY_RELU, ACT_SOFTPLUS, OUT_NONE, OUT_SIGMOID, OUT_SOFTPLUS, OUT_TANH,  # noqa: F401
                      PREC_BF16, PREC_F16, PREC_F32, NrtError)

# set once the analytic-Jacobian kernel is part of the library
HAS_SDF_VALUE_GRAD = True

_PREC_NAMES = {"f32": PREC_F32, "fp32": PREC_F32, "f16": PREC_F16, "fp16": PREC_F16, "bf16": PREC_BF16}


def prec_id(p) -> int:
    if isinstance(p, str):
        return _PREC_NAMES[p.lower()]
    return int(p)


def _chk(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise NrtError("%s must be a CUDA tensor (there is no CPU path)" % name)
    if t.dtype != dtype:
        raise NrtError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        t = t.contiguous()
    return t


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def mlp_layer_dims(in_size, latent_size, freqs, hidden, num_layers, skip, out_size):
    """(K, N) of every Linear in evaluation order [init, layers..., out] (neural_blocks.py:36-55)."""
    dim_p = in_size + 2 * freqs + latent_size
    dims = [(dim_p, hidden)]
    for i in range(num_layers):
        sk = (i % skip) == 0 and i != num_layers - 1
        dims.append((hidden + (dim_p if sk else 0), hidden))
    dims.append((hidden, out_size))
    return dims


class PackedMLP:
    """Device parameters of one SkipConnMLP in the packed-f32 layout of nrt_mlp_t."""

    def __init__(self, in_size, latent_size, freqs, hidden, num_layers, skip, out_size, act,
                 basis: torch.Tensor, params: torch.Tensor):
        self.in_size, self.latent_size, self.freqs, self.hidden = in_size, latent_size, freqs, hidden
        self.num_layers, self.skip, self.out_size, self.act = num_layers, skip, out_size, act
        self.basis = _chk(basis, "basis").reshape(in_size, freqs)
        self.params = _chk(params, "params")
        self.dims = mlp_layer_dims(in_size, latent_size, freqs, hidden, num_layers, skip, out_size)
        n = sum(k * n_ + n_ for k, n_ in self.dims)
        if self.params.numel() != n:
            raise NrtError("packed params have %d floats, expected %d" % (self.params.numel(), n))
        self.tc_blobs = {}   # prec -> uint8 tensor (tensor-core layout), built on demand
        self.dgrad_blobs = {}   # need_x -> uint8 tensor (transposed weights for the tensor-core backward)
        self._params_nk = None

    @staticmethod
    def pack(weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor]) -> torch.Tensor:
        """torch-layout weights (W [N,K]) in order [init, layers..., out] -> flat packed-f32 blob."""
        chunks = []
        for W, b in zip(weights, biases):
            chunks.append(W.detach().t().contiguous().reshape(-1))
            chunks.append(b.detach().reshape(-1))
        return torch.cat(chunks).to(torch.float32).contiguous()

    def unpack(self, flat: torch.Tensor):
        """Inverse of pack for a gradient blob: returns ([gW [N,K]], [gb [N]])."""
        gW, gb, off = [], [], 0
        for (k, n) in self.dims:
            gW.append(flat[off:off + k * n].reshape(k, n).t())
            off += k * n
            gb.append(flat[off:off + n])
            off += n
        return gW, gb

    def params_nk(self) -> torch.Tensor:
        """The weights in nn.Linear's [N][K] layout (per layer, no biases) for the backward's data-gradient GEMM."""
        if self._params_nk is None:
            chunks, off = [], 0
            for (k, n) in self.dims:
                chunks.append(self.params[off:off + k * n].reshape(k, n).t().contiguous().reshape(-1))
                off += k * n + n
            self._params_nk = torch.cat(chunks).contiguous()
        return self._params_nk

    def c_struct(self, prec=PREC_F32) -> N.NrtMlp:
        tc = None
        if prec != PREC_F32:
            tc = self.tc_blob(prec).data_ptr()
        return N.NrtMlp(self.in_size, self.latent_size, self.freqs, self.hidden, self.num_layers, self.skip,
                        self.out_size, self.act, self.basis.data_ptr(), self.params.data_ptr(), tc)

    def tc_blob(self, prec) -> torch.Tensor:
        if prec not in self.tc_blobs:
            c = N.NrtMlp(self.in_size, self.latent_size, self.freqs, self.hidden, self.num_layers, self.skip,
                         self.out_size, self.act, self.basis.data_ptr(), self.params.data_ptr(), None)
            nbytes = N.lib().nrt_mlp_tc_blob_bytes(ctypes.byref(c), prec)
            if nbytes < 0:
                N.check(int(nbytes))
            blob = torch.empty(int(nbytes), dtype=torch.uint8, device=self.params.device)
            N.check(N.lib().nrt_mlp_pack_tc(ctypes.byref(c), prec, _ptr(blob), _stream()))
            self.tc_blobs[prec] = blob
        return self.tc_blobs[prec]


    def dgrad_blob(self, need_x: bool, prec=PREC_F16) -> torch.Tensor:
        key = (bool(need_x), prec)
        if key not in self.dgrad_blobs:
            c = self.c_struct()
            nbytes = N.lib().nrt_mlp_tc_dgrad_blob_bytes(ctypes.byref(c), int(key[0]))
            if nbytes < 0:
                N.check(int(nbytes))
            blob = torch.empty(int(nbytes), dtype=torch.uint8, device=self.params.device)
            N.check(N.lib().nrt_mlp_pack_tc_dgrad(ctypes.byref(c), prec, int(key[0]), _ptr(blob), _stream()))
            self.dgrad_blobs[key] = blob
        return self.dgrad_blobs[key]


class PackedSDF:
    """Device parameters of a SphereSDF (sdfs.py:16-46)."""

    def __init__(self, centers, radii, tfs, shift: PackedMLP):
        self.centers = _chk(centers.detach(), "centers")
        self.radii = _chk(radii.detach(), "radii")
        self.tfs = _chk(tfs.detach(), "tfs")
        self.shift = shift
        self.n = self.radii.shape[0]

    def c_struct(self, prec=PREC_F32) -> N.NrtSphereSdf:
        return N.NrtSphereSdf(self.n, self.centers.data_ptr(), self.radii.data_ptr(), self.tfs.data_ptr(),
                              self.shift.c_struct(prec))


# ---------------------------------------------------------------------------------------------
def mlp_forward(m: PackedMLP, x: torch.Tensor, latent: Optional[torch.Tensor] = None, out_act=OUT_NONE,
                prec=PREC_F32, save_acts=False):
    """SkipConnMLP.forward (neural_blocks.py:75-86) on [..., in_size] -> [..., out_size]."""
    prec = prec_id(prec)
    batch = x.shape[:-1]
    x2 = _chk(x, "x").reshape(-1, m.in_size)
    M = x2.shape[0]
    lat = None
    if m.latent_size:
        if latent is None:
            raise NrtError("this MLP needs a latent of size %d" % m.latent_size)
        lat = _chk(latent, "latent").reshape(M, m.latent_size)
    out = torch.empty((M, m.out_size), dtype=torch.float32, device=x.device)
    acts = None
    if save_acts:
        acts = torch.empty(((m.num_layers + 1) * m.hidden, M), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        c = m.c_struct(prec)
        N.check(N.lib().nrt_mlp_forward(ctypes.byref(c), prec, out_act, _ptr(x2), _ptr(lat), M, _ptr(out),
                                        _ptr(acts), _stream()))
    out = out.reshape(batch + (m.out_size,))
    return (out, acts) if save_acts else out


def _grad_out(m: PackedMLP, g_params):
    """The packed-f32 gradient the kernels ACCUMULATE into: a fresh zero blob, or the caller's buffer (e.g. the slice
    of training.FlatParameters' flat gradient that belongs to this MLP)."""
    if g_params is None:
        return torch.zeros_like(m.params)
    if g_params.numel() != m.params.numel() or not g_params.is_contiguous() or g_params.dtype != torch.float32:
        raise NrtError("g_params must be a contiguous fp32 buffer of %d floats" % m.params.numel())
    return g_params


def mlp_backward(m: PackedMLP, x, latent, out, acts, g_out, out_act=OUT_NONE, need_input_grad=False, g_params=None):
    x2 = _chk(x, "x").reshape(-1, m.in_size)
    M = x2.shape[0]
    lat = _chk(latent, "latent").reshape(M, m.latent_size) if m.latent_size else None
    out2 = _chk(out, "out").reshape(M, m.out_size)
    g2 = _chk(g_out, "g_out").reshape(M, m.out_size)
    g_params = _grad_out(m, g_params)
    g_x = torch.empty_like(x2) if need_input_grad else None
    g_lat = torch.empty_like(lat) if (need_input_grad and lat is not None) else None
    with torch.cuda.device(x.device):
        c = m.c_struct()
        N.check(N.lib().nrt_mlp_backward(ctypes.byref(c), out_act, _ptr(x2), _ptr(lat), M, _ptr(out2), _ptr(acts),
                                         _ptr(g2), _ptr(m.params_nk()), _ptr(g_params), _ptr(g_x), _ptr(g_lat),
                                         _stream()))
    return g_params, g_x, g_lat


def mlp_forward_train_tc(m: PackedMLP, x: torch.Tensor, out_act=OUT_NONE, prec=PREC_F16):
    """Tensor-core training forward: returns (out [M,out], workspace) -- the workspace holds the saved
    activation tiles and must be handed to mlp_backward_tc unchanged."""
    prec = prec_id(prec)
    x2 = _chk(x, "x").reshape(-1, m.in_size)
    M = x2.shape[0]
    out = torch.empty((M, m.out_size), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        c = m.c_struct(prec)
        nbytes = N.lib().nrt_mlp_train_tc_workspace_bytes(ctypes.byref(c), M)
        if nbytes < 0:
            N.check(int(nbytes))
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=x.device)
        N.check(N.lib().nrt_mlp_forward_train_tc(ctypes.byref(c), prec, out_act, _ptr(x2), M, _ptr(out), _ptr(ws),
                                                 ws.numel(), _stream()))
    return out, ws


def mlp_backward_tc(m: PackedMLP, M: int, out: torch.Tensor, g_out: torch.Tensor, ws: torch.Tensor, out_act=OUT_NONE,
                    need_input_grad=False, prec=PREC_F16, g_params=None):
    """Tensor-core backward of mlp_forward_train_tc: (g_params packed-f32, g_x or None)."""
    prec = prec_id(prec)
    out2 = _chk(out, "out").reshape(M, m.out_size)
    g2 = _chk(g_out, "g_out").reshape(M, m.out_size)
    g_params = _grad_out(m, g_params)
    g_x = torch.empty((M, m.in_size), dtype=torch.float32, device=out.device) if need_input_grad else None
    with torch.cuda.device(out.device):
        c = m.c_struct(prec)
        blob = m.dgrad_blob(need_input_grad, prec)
        N.check(N.lib().nrt_mlp_backward_tc(ctypes.byref(c), prec, out_act, M, _ptr(out2), _ptr(g2), _ptr(blob), _ptr(ws),
                                            ws.numel(), _ptr(g_params), _ptr(g_x), _stream()))
    return g_params, g_x


def nerfle_train_forward(first: PackedMLP, second: PackedMLP, rays: torch.Tensor, ts: torch.Tensor, light_code: torch.Tensor,
                         view_of_ray: Optional[torch.Tensor] = None, prec=PREC_F16):
    """Both NeRFLE MLPs under autograd on the tensor cores (nrt_nerfle_train_forward): rays [R,6], ts [S] ->
    sigma [S,R], rgb [S,R,3] (sample-major) and the opaque state for nerfle_train_backward.  A 2-D ts [S,R] gives every
    sample its own distance (nrt_nerfle_train_forward_ts; the hierarchical samples of nerfle_sample_hierarchical)."""
    prec = prec_id(prec)
    r2 = _chk(rays, "rays").reshape(-1, 6)
    R = r2.shape[0]
    per_sample = ts.dim() == 2
    S = ts.shape[0] if per_sample else ts.numel()
    if per_sample and ts.shape[1] != R:
        raise NrtError("ts [S,R] has %d columns for %d rays" % (ts.shape[1], R))
    t = _chk(ts, "ts").reshape(ts.shape if per_sample else (S,))
    entry = N.lib().nrt_nerfle_train_forward_ts if per_sample else N.lib().nrt_nerfle_train_forward
    code = _chk(light_code, "light_code").reshape(-1, light_code.shape[-1])
    view = _chk(view_of_ray, "view_of_ray", torch.int32) if view_of_ray is not None else None
    dev = rays.device
    sigma = torch.empty((S, R), dtype=torch.float32, device=dev)
    rgb = torch.empty((S, R, 3), dtype=torch.float32, device=dev)
    lat = torch.empty((S * R + 127) // 128 * 128 * 64, dtype=torch.float32, device=dev)   # whole tiles (tile-interleaved)
    with torch.cuda.device(dev):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        n1 = N.lib().nrt_mlp_train_tc_workspace_bytes(ctypes.byref(c1), S * R)
        n2 = N.lib().nrt_mlp_train_tc_workspace_bytes(ctypes.byref(c2), S * R)
        if n1 < 0 or n2 < 0:
            N.check(int(min(n1, n2)))
        ws1 = torch.empty(int(n1), dtype=torch.uint8, device=dev)
        ws2 = torch.empty(int(n2), dtype=torch.uint8, device=dev)
        N.check(entry(ctypes.byref(c1), ctypes.byref(c2), prec, _ptr(r2), R, _ptr(t), S, _ptr(code), code.shape[-1], _ptr(view),
                      _ptr(sigma), _ptr(rgb), _ptr(lat), _ptr(ws1), ws1.numel(), _ptr(ws2), ws2.numel(), _stream()))
    return sigma, rgb, (ws1, ws2, R, S, code.shape[-1])


def nerfle_train_backward(first: PackedMLP, second: PackedMLP, rgb: torch.Tensor, g_sigma: torch.Tensor, g_rgb: torch.Tensor,
                          state, prec=PREC_F16, g_params_first=None, g_params_second=None):
    """(g_params_first, g_params_second), packed-f32 layout (accumulated into the given buffers if any)."""
    prec = prec_id(prec)
    ws1, ws2, R, S, light_dim = state
    dev = rgb.device
    gs = _chk(g_sigma, "g_sigma").reshape(S, R)
    gc = _chk(g_rgb, "g_rgb").reshape(S, R, 3)
    y = _chk(rgb, "rgb").reshape(S, R, 3)
    g1, g2 = _grad_out(first, g_params_first), _grad_out(second, g_params_second)
    scratch = torch.empty((S * R + 127) // 128 * 128 * 64, dtype=torch.float32, device=dev)   # whole tiles
    with torch.cuda.device(dev):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        b1, b2 = first.dgrad_blob(False, prec), second.dgrad_blob(True, prec)
        N.check(N.lib().nrt_nerfle_train_backward(ctypes.byref(c1), ctypes.byref(c2), prec, R, S, light_dim, _ptr(y), _ptr(gs),
                                                  _ptr(gc), _ptr(b1), _ptr(b2), _ptr(ws1), _ptr(ws2), _ptr(scratch), _ptr(g1),
                                                  _ptr(g2), _stream()))
    return g1, g2


def sdf_eval(s: PackedSDF, p: torch.Tensor, prec=PREC_F32) -> torch.Tensor:
    prec = prec_id(prec)
    batch = p.shape[:-1]
    p2 = _chk(p, "p").reshape(-1, 3)
    out = torch.empty(p2.shape[0], dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device):
        c = s.c_struct(prec)
        N.check(N.lib().nrt_sdf_eval(ctypes.byref(c), prec, _ptr(p2), p2.shape[0], _ptr(out), _stream()))
    return out.reshape(batch)


def sdf_value_grad(s: PackedSDF, p: torch.Tensor):
    batch = p.shape[:-1]
    p2 = _chk(p, "p").reshape(-1, 3)
    val = torch.empty(p2.shape[0], dtype=torch.float32, device=p.device)
    grad = torch.empty((p2.shape[0], 3), dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device):
        c = s.c_struct()
        N.check(N.lib().nrt_sdf_value_grad(ctypes.byref(c), _ptr(p2), p2.shape[0], _ptr(val), _ptr(grad), _stream()))
    return val.reshape(batch), grad.reshape(batch + (3,))


def mlp_value_jac_forward(m: PackedMLP, p: torch.Tensor, save_acts=False):
    """Forward-mode (value, d value / d p) of a SkipConnMLP with in_size 3: p [M,3] -> value [M,out], jac [M,out,3]
    (+ the saved four-column activations for mlp_value_jac_backward)."""
    p2 = _chk(p, "p").reshape(-1, 3)
    M = p2.shape[0]
    val = torch.empty((M, m.out_size), dtype=torch.float32, device=p.device)
    jac = torch.empty((M, m.out_size, 3), dtype=torch.float32, device=p.device)
    acts = torch.empty(((m.num_layers + 1) * m.hidden, 4 * M), dtype=torch.float32, device=p.device) if save_acts else None
    with torch.cuda.device(p.device):
        c = m.c_struct()
        N.check(N.lib().nrt_mlp_value_jac_forward(ctypes.byref(c), _ptr(p2), M, _ptr(val), _ptr(jac), _ptr(acts), _stream()))
    return val, jac, acts


def mlp_value_jac_backward(m: PackedMLP, p: torch.Tensor, acts: torch.Tensor, g_value: torch.Tensor, g_jac: torch.Tensor):
    """Reverse pass of mlp_value_jac_forward into the packed-f32 parameter gradient (the reference's double backward
    through SDF.autograd_diff, sdfs.py:184-197)."""
    p2 = _chk(p, "p").reshape(-1, 3)
    M = p2.shape[0]
    gv = _chk(g_value, "g_value").reshape(M, m.out_size)
    gj = _chk(g_jac, "g_jac").reshape(M, m.out_size, 3)
    g_params = torch.zeros_like(m.params)
    with torch.cuda.device(p.device):
        c = m.c_struct()
        N.check(N.lib().nrt_mlp_value_jac_backward(ctypes.byref(c), _ptr(p2), M, _ptr(acts), _ptr(gv), _ptr(gj),
                                                   _ptr(m.params_nk()), _ptr(g_params), _stream()))
    return g_params


def sphere_set_forward(centers, radii, tfs, p: torch.Tensor, want_grad=True):
    """Smooth-min of the warped spheres (sdfs.py:37-45) at p [K,3]: value [K] and d value / d p [K,3]."""
    p2 = _chk(p, "p").reshape(-1, 3)
    K = p2.shape[0]
    c, r, t = _chk(centers.detach(), "centers"), _chk(radii.detach(), "radii"), _chk(tfs.detach(), "tfs")
    val = torch.empty(K, dtype=torch.float32, device=p.device)
    grad = torch.empty((K, 3), dtype=torch.float32, device=p.device) if want_grad else None
    with torch.cuda.device(p.device):
        N.check(N.lib().nrt_sphere_set_forward(int(c.shape[0]), _ptr(c), _ptr(r), _ptr(t), _ptr(p2), K, _ptr(val), _ptr(grad), _stream()))
    return val, grad


def sphere_set_backward(centers, radii, tfs, p: torch.Tensor, g_value, g_grad):
    """Reverse pass of sphere_set_forward's two outputs into (g_centers, g_radii, g_tfs)."""
    p2 = _chk(p, "p").reshape(-1, 3)
    K = p2.shape[0]
    c, r, t = _chk(centers.detach(), "centers"), _chk(radii.detach(), "radii"), _chk(tfs.detach(), "tfs")
    gv = None if g_value is None else _chk(g_value, "g_value").reshape(K)
    gg = None if g_grad is None else _chk(g_grad, "g_grad").reshape(K, 3)
    gc, gr, gt = torch.zeros_like(c), torch.zeros_like(r), torch.zeros_like(t)
    with torch.cuda.device(p.device):
        N.check(N.lib().nrt_sphere_set_backward(int(c.shape[0]), _ptr(c), _ptr(r), _ptr(t), _ptr(p2), K, _ptr(gv), _ptr(gg), _ptr(gc),
                                                _ptr(gr), _ptr(gt), _stream()))
    return gc, gr, gt


def mlp_value_jac_forward_tc(m: PackedMLP, p: torch.Tensor, prec=PREC_F16):
    """Tensor-core (value, d value / d p) of SphereSDF.shift: p [K,3] -> value [K,1], jac [K,1,3] and the workspace of
    saved activation tiles for mlp_value_jac_backward_tc (nrt_mlp_value_jac_forward_tc)."""
    prec = prec_id(prec)
    p2 = _chk(p, "p").reshape(-1, 3)
    K = p2.shape[0]
    val = torch.empty((K, 1), dtype=torch.float32, device=p.device)
    jac = torch.empty((K, 1, 3), dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device):
        c = m.c_struct(prec)
        nbytes = N.lib().nrt_mlp_value_jac_tc_workspace_bytes(ctypes.byref(c), K)
        if nbytes < 0:
            N.check(int(nbytes))
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=p.device)
        N.check(N.lib().nrt_mlp_value_jac_forward_tc(ctypes.byref(c), prec, _ptr(p2), K, _ptr(val), _ptr(jac), _ptr(ws), ws.numel(),
                                                     _stream()))
    return val, jac, ws


def mlp_value_jac_backward_tc(m: PackedMLP, K: int, ws: torch.Tensor, g_value: Optional[torch.Tensor], g_jac: torch.Tensor,
                              prec=PREC_F16, g_params=None):
    """Reverse pass of mlp_value_jac_forward_tc into the packed-f32 parameter gradient."""
    prec = prec_id(prec)
    gv = None if g_value is None else _chk(g_value, "g_value").reshape(K)
    gj = _chk(g_jac, "g_jac").reshape(K, 3)
    g_params = _grad_out(m, g_params)
    with torch.cuda.device(gj.device):
        c = m.c_struct(prec)
        blob = m.dgrad_blob(False, prec)
        N.check(N.lib().nrt_mlp_value_jac_backward_tc(ctypes.byref(c), prec, K, _ptr(gv), _ptr(gj), _ptr(blob), _ptr(ws), ws.numel(),
                                                      _ptr(g_params), _stream()))
    return g_params


def sphere_trace(s: PackedSDF, rays: torch.Tensor, epsilon=1e-3, max_steps=64, max_t=10.0,
                 active: Optional[torch.Tensor] = None, prec=PREC_F32, steps_counter: Optional[torch.Tensor] = None):
    """SDF.intersect march loop (sdfs.py:111-131).  rays [...,6] -> depth [...], hit [...] (bool)."""
    prec = prec_id(prec)
    batch = rays.shape[:-1]
    r2 = _chk(rays, "rays").reshape(-1, 6)
    R = r2.shape[0]
    depth = torch.empty(R, dtype=torch.float32, device=rays.device)
    hit = torch.empty(R, dtype=torch.uint8, device=rays.device)
    act = _chk(active.reshape(-1).to(torch.uint8), "active", torch.uint8) if active is not None else None
    with torch.cuda.device(rays.device):
        c = s.c_struct(prec)
        N.check(N.lib().nrt_sdf_sphere_trace(ctypes.byref(c), prec, _ptr(r2), _ptr(act), R, float(epsilon),
                                             int(max_steps), float(max_t), _ptr(depth), _ptr(hit),
                                             _ptr(steps_counter), _stream()))
    return depth.reshape(batch), hit.bool().reshape(batch)


def shadow_test(s: PackedSDF, rays: torch.Tensor, max_t: torch.Tensor, epsilon=1e-3, max_steps=64,
                active: Optional[torch.Tensor] = None, prec=PREC_F32, steps_counter: Optional[torch.Tensor] = None):
    """SDF.intersect_test (sdfs.py:162-181).  Returns not_blocked [...] (bool)."""
    prec = prec_id(prec)
    batch = rays.shape[:-1]
    r2 = _chk(rays, "rays").reshape(-1, 6)
    R = r2.shape[0]
    mt = _chk(max_t, "max_t").reshape(-1)
    if mt.numel() != R:
        mt = mt.expand(R).contiguous()
    nb = torch.empty(R, dtype=torch.uint8, device=rays.device)
    act = _chk(active.reshape(-1).to(torch.uint8), "active", torch.uint8) if active is not None else None
    with torch.cuda.device(rays.device):
        c = s.c_struct(prec)
        N.check(N.lib().nrt_sdf_shadow_test(ctypes.byref(c), prec, _ptr(r2), _ptr(mt), _ptr(act), R, float(epsilon),
                                            int(max_steps), _ptr(nb), _ptr(steps_counter), _stream()))
    return nb.bool().reshape(batch)


def min_scan(s: PackedSDF, rays: torch.Tensor, step: float, n_steps=128, prec=PREC_F32):
    """SDF.throughput scan (sdfs.py:232-249).  Returns (best_idx int32 [...], best_pos [...,3], min [...])."""
    prec = prec_id(prec)
    batch = rays.shape[:-1]
    r2 = _chk(rays, "rays").reshape(-1, 6)
    R = r2.shape[0]
    idx = torch.empty(R, dtype=torch.int32, device=rays.device)
    pos = torch.empty((R, 3), dtype=torch.float32, device=rays.device)
    mv = torch.empty(R, dtype=torch.float32, device=rays.device)
    with torch.cuda.device(rays.device):
        c = s.c_struct(prec)
        N.check(N.lib().nrt_sdf_min_scan(ctypes.byref(c), prec, _ptr(r2), R, float(step), int(n_steps), _ptr(idx),
                                         _ptr(pos), _ptr(mv), _stream()))
    return idx.reshape(batch), pos.reshape(batch + (3,)), mv.reshape(batch)


def composite_forward(sigma_raw: torch.Tensor, rgb: torch.Tensor, ts: torch.Tensor) -> torch.Tensor:
    """nerf.py:206-213 on sample-major sigma_raw [S,R], rgb [S,R,3], ts [S] -> [R,3]."""
    sg = _chk(sigma_raw, "sigma_raw")
    S, R = sg.shape[0], sg[0].numel()
    c = _chk(rgb, "rgb").reshape(S, R, 3)
    t = _chk(ts, "ts").reshape(S)
    out = torch.empty((R, 3), dtype=torch.float32, device=sg.device)
    with torch.cuda.device(sg.device):
        N.check(N.lib().nrt_composite_forward(_ptr(sg), _ptr(c), _ptr(t), S, R, _ptr(out), _stream()))
    return out.reshape(tuple(sigma_raw.shape[1:]) + (3,))


def composite_backward(sigma_raw, rgb, ts, g_out):
    sg = _chk(sigma_raw, "sigma_raw")
    S, R = sg.shape[0], sg[0].numel()
    c = _chk(rgb, "rgb").reshape(S, R, 3)
    t = _chk(ts, "ts").reshape(S)
    go = _chk(g_out, "g_out").reshape(R, 3)
    g_s = torch.empty_like(sg)
    g_c = torch.empty_like(c)
    with torch.cuda.device(sg.device):
        N.check(N.lib().nrt_composite_backward(_ptr(sg), _ptr(c), _ptr(t), S, R, _ptr(go), _ptr(g_s), _ptr(g_c),
                                               _stream()))
    return g_s, g_c.reshape(rgb.shape)


def _ts_per_sample(ts, S, R):
    t = _chk(ts, "ts")
    if t.numel() != S * R:
        raise NrtError("ts must hold one distance per sample, [%d,%d]; got %s" % (S, R, tuple(ts.shape)))
    return t.reshape(S, R)


def composite_forward_ts(sigma_raw: torch.Tensor, rgb: torch.Tensor, ts: torch.Tensor) -> torch.Tensor:
    """composite_forward with per-sample distances: sigma_raw [S,...], rgb [S,...,3], ts [S,...] -> [...,3]
    (nrt_composite_forward_ts; the reference's quirks kept)."""
    sg = _chk(sigma_raw, "sigma_raw")
    S, R = sg.shape[0], sg[0].numel()
    c = _chk(rgb, "rgb").reshape(S, R, 3)
    t = _ts_per_sample(ts, S, R)
    out = torch.empty((R, 3), dtype=torch.float32, device=sg.device)
    with torch.cuda.device(sg.device):
        N.check(N.lib().nrt_composite_forward_ts(_ptr(sg), _ptr(c), _ptr(t), S, R, _ptr(out), _stream()))
    return out.reshape(tuple(sigma_raw.shape[1:]) + (3,))


def composite_backward_ts(sigma_raw, rgb, ts, g_out):
    sg = _chk(sigma_raw, "sigma_raw")
    S, R = sg.shape[0], sg[0].numel()
    c = _chk(rgb, "rgb").reshape(S, R, 3)
    t = _ts_per_sample(ts, S, R)
    go = _chk(g_out, "g_out").reshape(R, 3)
    g_s = torch.empty_like(sg)
    g_c = torch.empty_like(c)
    with torch.cuda.device(sg.device):
        N.check(N.lib().nrt_composite_backward_ts(_ptr(sg), _ptr(c), _ptr(t), S, R, _ptr(go), _ptr(g_s), _ptr(g_c),
                                                  _stream()))
    return g_s, g_c.reshape(rgb.shape)


def shading_frame(normals: torch.Tensor, rays: Optional[torch.Tensor] = None):
    """coordinate_system(normals) [..,3,3] and, if rays are given, wi = to_local(frame, -r_d)
    (interaction.py:9-27, 38-41; sdfs.py:158-159)."""
    batch = normals.shape[:-1]
    n2 = _chk(normals, "normals").reshape(-1, 3)
    R = n2.shape[0]
    frame = torch.empty((R, 3, 3), dtype=torch.float32, device=normals.device)
    wi = r2 = None
    if rays is not None:
        r2 = _chk(rays, "rays").reshape(-1, 6)
        wi = torch.empty((R, 3), dtype=torch.float32, device=normals.device)
    with torch.cuda.device(normals.device):
        N.check(N.lib().nrt_shading_frame(_ptr(n2), _ptr(r2), R, _ptr(frame), _ptr(wi), _stream()))
    frame = frame.reshape(batch + (3, 3))
    return (frame, wi.reshape(batch + (3,))) if rays is not None else frame


def to_local(frame: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    batch = v.shape[:-1]
    f2 = _chk(frame, "frame").reshape(-1, 9)
    v2 = _chk(v, "v").expand(batch + (3,)).reshape(-1, 3).contiguous()
    out = torch.empty_like(v2)
    with torch.cuda.device(v.device):
        N.check(N.lib().nrt_to_local(_ptr(f2), _ptr(v2), v2.shape[0], _ptr(out), _stream()))
    return out.reshape(batch + (3,))


def param_rusin2(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """utils.py:233-258 on [...,3] x [...,3]."""
    batch = a.shape[:-1]
    a2 = _chk(a, "a").reshape(-1, 3)
    b2 = _chk(b, "b").reshape(-1, 3)
    out = torch.empty_like(a2)
    with torch.cuda.device(a.device):
        N.check(N.lib().nrt_param_rusin2(_ptr(a2), _ptr(b2), a2.shape[0], _ptr(out), _stream()))
    return out.reshape(batch + (3,))


# ---- fused shading glue of the Direct integrator on compacted hits (nrt_shade_*; include/nrt_b200.h) ----------------
LIGHT_POINT, LIGHT_FIELD = 0, 1
BSDF_NEURAL, BSDF_DIFFUSE, BSDF_CONDUCTOR = 0, 1, 2


def _f32(t, name, shape=None):
    t = _chk(t, name)
    return t if shape is None else t.reshape(shape)


def shade_geom_forward(raw_n, p_hit, rays_hit, eps5, want_frame=True):
    K = raw_n.shape[0]
    rn, ph, rh = _f32(raw_n, "raw_n", (K, 3)), _f32(p_hit, "p_hit", (K, 3)), _f32(rays_hit, "rays_hit", (K, 6))
    n, p_off, wi = torch.empty_like(rn), torch.empty_like(rn), torch.empty_like(rn)
    frame = torch.empty((K, 3, 3), dtype=torch.float32, device=rn.device) if want_frame else None
    with torch.cuda.device(rn.device):
        N.check(N.lib().nrt_shade_geom_forward(_ptr(rn), _ptr(ph), _ptr(rh), K, float(eps5), _ptr(n), _ptr(p_off), _ptr(wi),
                                               _ptr(frame), _stream()))
    return n, p_off, wi, frame


def shade_geom_backward(raw_n, rays_hit, eps5, g_n, g_p_off, g_wi):
    K = raw_n.shape[0]
    rn, rh = _f32(raw_n, "raw_n", (K, 3)), _f32(rays_hit, "rays_hit", (K, 6))
    opt = lambda g, nm: None if g is None else _f32(g, nm, (K, 3))
    g = torch.empty_like(rn)
    with torch.cuda.device(rn.device):
        N.check(N.lib().nrt_shade_geom_backward(_ptr(rn), _ptr(rh), K, float(eps5), _ptr(opt(g_n, "g_n")),
                                                _ptr(opt(g_p_off, "g_p_off")), _ptr(opt(g_wi, "g_wi")), _ptr(g), _stream()))
    return g


def _light_struct(mode, location, amp, coef, view_of_hit, v, sig_color):
    n_views = 0 if location is None else location.shape[0]
    return N.NrtLight(mode, n_views, *[None if t is None else t.data_ptr() for t in (location, amp, coef, view_of_hit, v, sig_color)])


def shade_light_forward(mode, n, wi, p_off, location=None, amp=None, coef=None, view_of_hit=None, v=None, sig_color=None,
                        want_elaz=False):
    """-> d [K,3], dist [K], wo [K,3], rusin [K,3], e [K,3], elaz [K,2] or None."""
    K = n.shape[0]
    dev = n.device
    d, wo, ru, e = (torch.empty((K, 3), dtype=torch.float32, device=dev) for _ in range(4))
    dist = torch.empty(K, dtype=torch.float32, device=dev)
    elaz = torch.empty((K, 2), dtype=torch.float32, device=dev) if want_elaz else None
    L = _light_struct(mode, location, amp, coef, view_of_hit, v, sig_color)
    with torch.cuda.device(dev):
        N.check(N.lib().nrt_shade_light_forward(ctypes.byref(L), _ptr(n), _ptr(wi), _ptr(p_off), K, _ptr(d), _ptr(dist), _ptr(wo),
                                                _ptr(ru), _ptr(e), _ptr(elaz), _stream()))
    return d, dist, wo, ru, e, elaz


def shade_light_backward(mode, n, wi, p_off, g_wo, g_rusin, g_e, g_elaz, location=None, amp=None, coef=None, view_of_hit=None,
                         v=None, sig_color=None):
    """-> g_n, g_wi, g_pv [K,3], g_amp [n_views,3] | None, g_coef [3] | None, g_sig_color [3] | None."""
    K = n.shape[0]
    dev = n.device
    g_n, g_wi, g_pv = (torch.empty((K, 3), dtype=torch.float32, device=dev) for _ in range(3))
    g_amp = torch.zeros_like(amp) if mode == LIGHT_POINT else None
    g_coef = torch.zeros(3, dtype=torch.float32, device=dev) if mode == LIGHT_POINT else None
    g_sig = torch.zeros(3, dtype=torch.float32, device=dev) if mode == LIGHT_FIELD else None
    L = _light_struct(mode, location, amp, coef, view_of_hit, v, sig_color)
    with torch.cuda.device(dev):
        N.check(N.lib().nrt_shade_light_backward(ctypes.byref(L), _ptr(n), _ptr(wi), _ptr(p_off), K, _ptr(g_wo), _ptr(g_rusin),
                                                 _ptr(g_e), _ptr(g_elaz), _ptr(g_n), _ptr(g_wi), _ptr(g_pv), _ptr(g_amp),
                                                 _ptr(g_coef), _ptr(g_sig), _stream()))
    return g_n, g_wi, g_pv, g_amp, g_coef, g_sig


def _blend_struct(kinds, neural_act, diffuse_pre):
    arr = (ctypes.c_int32 * N.MAX_BSDFS)(*([int(k) for k in kinds] + [0] * (N.MAX_BSDFS - len(kinds))))
    return N.NrtBlend(len(kinds), arr, int(neural_act), int(diffuse_pre))


def shade_blend_forward(kinds, neural_act, diffuse_pre, logits, neural_raw, wi, wo, e, refl, cond_spec, cond_eta, inv_samples):
    K = logits.shape[0]
    out = torch.empty((K, 3), dtype=torch.float32, device=logits.device)
    B = _blend_struct(kinds, neural_act, diffuse_pre)
    with torch.cuda.device(logits.device):
        N.check(N.lib().nrt_shade_blend_forward(ctypes.byref(B), _ptr(logits), _ptr(neural_raw), _ptr(wi), _ptr(wo), _ptr(e),
                                                _ptr(refl), _ptr(cond_spec), _ptr(cond_eta), float(inv_samples), K, _ptr(out),
                                                _stream()))
    return out


def shade_blend_backward(kinds, neural_act, diffuse_pre, logits, neural_raw, wi, wo, e, refl, cond_spec, cond_eta, inv_samples,
                         g_out):
    K = logits.shape[0]
    dev = logits.device
    g_logits = torch.empty_like(logits)
    g_neural = torch.empty_like(neural_raw) if neural_raw is not None else None
    g_wi, g_wo, g_e = (torch.empty((K, 3), dtype=torch.float32, device=dev) for _ in range(3))
    g_refl = torch.zeros_like(refl) if refl is not None else None
    g_cs = torch.zeros_like(cond_spec) if cond_spec is not None else None
    g_ce = torch.zeros_like(cond_eta) if cond_eta is not None else None
    B = _blend_struct(kinds, neural_act, diffuse_pre)
    with torch.cuda.device(dev):
        N.check(N.lib().nrt_shade_blend_backward(ctypes.byref(B), _ptr(logits), _ptr(neural_raw), _ptr(wi), _ptr(wo), _ptr(e),
                                                 _ptr(refl), _ptr(cond_spec), _ptr(cond_eta), float(inv_samples), K, _ptr(g_out),
                                                 _ptr(g_logits), _ptr(g_neural), _ptr(g_wi), _ptr(g_wo), _ptr(g_e), _ptr(g_refl),
                                                 _ptr(g_cs), _ptr(g_ce), _stream()))
    return g_logits, g_neural, g_wi, g_wo, g_e, g_refl, g_cs, g_ce


_ws_cache = {}


def nerfle_render(first: PackedMLP, second: PackedMLP, rays: torch.Tensor, ts: Optional[torch.Tensor],
                  light_code: torch.Tensor, view_of_ray: Optional[torch.Tensor] = None, prec=PREC_F32,
                  n_coarse: Optional[int] = None, n_fine=0, t_near=0.0, t_far=0.0, jitter_seed=0) -> torch.Tensor:
    """NeRFLE.forward (nerf.py:175-214): rays [...,6] -> rgb [...,3].
    With n_fine == 0 and jitter_seed == 0 this is the reference's single uniform pass over `ts`."""
    prec = prec_id(prec)
    batch = rays.shape[:-1]
    r2 = _chk(rays, "rays").reshape(-1, 6)
    R = r2.shape[0]
    t = _chk(ts, "ts").reshape(-1) if ts is not None else None
    if n_coarse is None:
        if t is None:
            raise NrtError("either ts or n_coarse must be given")
        n_coarse = t.numel()
    lc = _chk(light_code, "light_code")
    lc = lc.reshape(-1, lc.shape[-1])
    vor = _chk(view_of_ray.reshape(-1), "view_of_ray", torch.int32) if view_of_ray is not None else None
    out = torch.empty((R, 3), dtype=torch.float32, device=rays.device)
    samp = N.NrtNerfSampling(int(n_coarse), int(n_fine), float(t_near), float(t_far), int(jitter_seed))
    with torch.cuda.device(rays.device):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        nbytes = N.lib().nrt_nerfle_render_workspace(ctypes.byref(c1), ctypes.byref(c2), prec, R, ctypes.byref(samp))
        key = (rays.device.index, torch.cuda.current_stream().cuda_stream)
        ws = _ws_cache.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=rays.device)
            _ws_cache[key] = ws
        N.check(N.lib().nrt_nerfle_render(ctypes.byref(c1), ctypes.byref(c2), prec, _ptr(r2), R, _ptr(t),
                                          ctypes.byref(samp), _ptr(lc), lc.shape[-1], _ptr(vor), _ptr(out),
                                          _ptr(ws), ws.numel(), _stream()))
    return out.reshape(batch + (3,))


_sample_ws_cache = {}


def nerfle_sample_hierarchical(first: PackedMLP, second: PackedMLP, rays: torch.Tensor, light_code: torch.Tensor,
                               view_of_ray: Optional[torch.Tensor] = None, prec=PREC_F32, n_coarse=64, n_fine=128,
                               t_near=0.0, t_far=2.05, jitter_seed=0, seed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The merged coarse + fine distances nerfle_render(n_coarse, n_fine, ...) composites over, for training on them
    (nrt_nerfle_sample_hierarchical): rays [...,6] -> ts [n_coarse + n_fine, R], ascending per ray, sample-major.
    `seed`, a one-element int64 CUDA tensor, replaces jitter_seed when given: the kernels read it on the device."""
    prec = prec_id(prec)
    r2 = _chk(rays, "rays").reshape(-1, 6)
    R = r2.shape[0]
    lc = _chk(light_code, "light_code")
    lc = lc.reshape(-1, lc.shape[-1])
    vor = _chk(view_of_ray.reshape(-1), "view_of_ray", torch.int32) if view_of_ray is not None else None
    sd = None
    if seed is not None:
        sd = _chk(seed, "seed", torch.int64)
        if sd.numel() != 1:
            raise NrtError("seed must hold one int64")
    out = torch.empty((int(n_coarse) + int(n_fine), R), dtype=torch.float32, device=rays.device)
    samp = N.NrtNerfSampling(int(n_coarse), int(n_fine), float(t_near), float(t_far), int(jitter_seed))
    with torch.cuda.device(rays.device):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        nbytes = N.lib().nrt_nerfle_sample_hierarchical_workspace(ctypes.byref(c1), ctypes.byref(c2), prec, R,
                                                                  ctypes.byref(samp))
        key = (rays.device.index, torch.cuda.current_stream().cuda_stream)
        ws = _sample_ws_cache.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=rays.device)
            _sample_ws_cache[key] = ws
        N.check(N.lib().nrt_nerfle_sample_hierarchical(ctypes.byref(c1), ctypes.byref(c2), prec, _ptr(r2), R,
                                                       ctypes.byref(samp), _ptr(sd), _ptr(lc), lc.shape[-1], _ptr(vor),
                                                       _ptr(out), _ptr(ws), ws.numel(), _stream()))
    return out


def nerfle_render_host(first: PackedMLP, second: PackedMLP, rays_host: torch.Tensor, ts_host: torch.Tensor,
                       light_code: torch.Tensor, out_host: torch.Tensor, prec=PREC_F32, n_coarse=None, n_fine=0,
                       t_near=0.0, t_far=0.0, jitter_seed=0):
    """End-to-end leg: HOST (pinned) rays in, HOST rgb out; H2D/D2H copies happen inside the call."""
    prec = prec_id(prec)
    assert not rays_host.is_cuda and not out_host.is_cuda
    R = rays_host.reshape(-1, 6).shape[0]
    S = ts_host.numel() if ts_host is not None else 0
    if n_coarse is None:
        n_coarse = S
    lc = _chk(light_code, "light_code")
    samp = N.NrtNerfSampling(int(n_coarse), int(n_fine), float(t_near), float(t_far), int(jitter_seed))
    with torch.cuda.device(lc.device):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        N.check(N.lib().nrt_nerfle_render_host(
            ctypes.byref(c1), ctypes.byref(c2), prec, ctypes.c_void_p(rays_host.data_ptr()), R,
            ctypes.c_void_p(ts_host.data_ptr()) if ts_host is not None else None, S, ctypes.byref(samp), _ptr(lc),
            lc.shape[-1], ctypes.c_void_p(out_host.data_ptr()), _stream()))
    return out_host


# ---- a21 / f4: ray generators on the device, camera-driven render --------------------------------
CAM_NERF, CAM_DTU, CAM_FOV = 0, 1, 2


class CameraDesc:
    """nrt_camera_t plus the tensors its device pointers borrow (kept alive for the duration of the call).

    kind: CAM_NERF (a = cam_to_world [n,3|4,4], focal), CAM_DTU (a = pose [n,4,4], b = intrinsics [n,3|4,3|4]) or
    CAM_FOV (a = inverse full projection [n,4,4] in the row-vector convention, b = camera centres [n,3]).  The block
    of rays is the reference's [n_views, nx, ny, bundle, 6]: pixel position (u, v) = (y0 + j, x0 + i) as in
    pathtrace (main.py:67-74), or `positions` [nx, ny(, bundle), 2] when given."""

    def __init__(self, kind, a, b=None, focal=1.0, size=1.0, x0=0, y0=0, nx=0, ny=0, bundle=1, positions=None,
                 jitter=0.0, jitter_seed=0):
        a = _chk(a, "camera matrix a")
        if a.dim() != 3:
            raise NrtError("camera matrix a must be [n_views, rows, cols], got %s" % (tuple(a.shape),))
        self.device = a.device
        self.n_views = a.shape[0]
        if b is not None:
            b = _chk(b, "camera matrix b")
            if b.dim() == 2:
                b = b.reshape(b.shape[0], 1, b.shape[1])
            if b.shape[0] != self.n_views:
                raise NrtError("camera matrices a and b disagree on the number of views")
        elif kind != CAM_NERF:
            raise NrtError("this camera kind needs the second matrix (intrinsics / centres)")
        ppp = 1
        if positions is not None:
            positions = _chk(positions, "positions")
            if positions.shape[-1] != 2 or positions.numel() not in (nx * ny * 2, nx * ny * bundle * 2):
                raise NrtError("positions must be [nx, ny(, bundle), 2]")
            ppp = positions.numel() // (nx * ny * 2) if nx * ny else 1
        self._keep = (a, b, positions)
        self.nx, self.ny, self.bundle = int(nx), int(ny), int(bundle)
        self.struct = N.NrtCamera(
            int(kind), int(self.n_views), _ptr(a), _ptr(b), a.shape[1] * a.shape[2], a.shape[2],
            (b.shape[1] * b.shape[2]) if b is not None else 0, b.shape[2] if b is not None else 0,
            float(focal), float(size), int(x0), int(y0), int(nx), int(ny), int(bundle), int(ppp), _ptr(positions),
            float(jitter), int(jitter_seed))

    @property
    def n_rays(self):
        return self.n_views * self.nx * self.ny * self.bundle


def camera_rays(cam: CameraDesc, want_view=False):
    """sample_positions of the three cameras as one kernel: rays [n_views, nx, ny, bundle, 6] (fp32, device)."""
    R = cam.n_rays
    out = torch.empty((cam.n_views, cam.nx, cam.ny, cam.bundle, 6), dtype=torch.float32, device=cam.device)
    view = torch.empty((R,), dtype=torch.int32, device=cam.device) if want_view else None
    with torch.cuda.device(cam.device):
        N.check(N.lib().nrt_camera_rays(ctypes.byref(cam.struct), 0, R, _ptr(out), _ptr(view), _stream()))
    return (out, view) if want_view else out


def set_camera_rays_mode(fused: bool):
    """False (default): every chunk's rays come from k_camera_rays; True: the tensor-core NeRF kernels compute each sample's
    ray from the camera themselves (no ray array; same image bit for bit; measured 2.5-3 % slower on B200)."""
    N.check(N.lib().nrt_set_camera_rays_mode(1 if fused else 0))


def nerfle_render_camera(first: PackedMLP, second: PackedMLP, cam: CameraDesc, ts: Optional[torch.Tensor],
                         light_code: torch.Tensor, prec=PREC_F32, n_coarse: Optional[int] = None, n_fine=0,
                         t_near=0.0, t_far=0.0, jitter_seed=0) -> torch.Tensor:
    """The frame of a volumetric shape from its camera in one call: rays are generated on the device inside the
    library (f4; replaces the tile loop of pathtrace, main.py:57-88).  -> rgb [n_views, nx, ny, bundle, 3]."""
    prec = prec_id(prec)
    t = _chk(ts, "ts").reshape(-1) if ts is not None else None
    if n_coarse is None:
        if t is None:
            raise NrtError("either ts or n_coarse must be given")
        n_coarse = t.numel()
    lc = _chk(light_code, "light_code")
    lc = lc.reshape(-1, lc.shape[-1])
    if lc.shape[0] < cam.n_views:
        raise NrtError("light_code has %d rows for %d views" % (lc.shape[0], cam.n_views))
    out = torch.empty((cam.n_views, cam.nx, cam.ny, cam.bundle, 3), dtype=torch.float32, device=cam.device)
    samp = N.NrtNerfSampling(int(n_coarse), int(n_fine), float(t_near), float(t_far), int(jitter_seed))
    with torch.cuda.device(cam.device):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        nbytes = N.lib().nrt_nerfle_render_camera_workspace(ctypes.byref(c1), ctypes.byref(c2), prec,
                                                            ctypes.byref(cam.struct), ctypes.byref(samp))
        key = (cam.device.index, torch.cuda.current_stream().cuda_stream)
        ws = _ws_cache.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=cam.device)
            _ws_cache[key] = ws
        N.check(N.lib().nrt_nerfle_render_camera(ctypes.byref(c1), ctypes.byref(c2), prec, ctypes.byref(cam.struct),
                                                 _ptr(t), ctypes.byref(samp), _ptr(lc), lc.shape[-1], _ptr(out),
                                                 _ptr(ws), ws.numel(), _stream()))
    return out


def nerfle_render_samples(first: PackedMLP, second: PackedMLP, rays_or_cam, ts: torch.Tensor, light_code: torch.Tensor,
                          view_of_ray: Optional[torch.Tensor] = None, prec=PREC_F32):
    """The per-sample values the render composites (nrt_nerfle_render_samples: the render's own chunks and kernels):
    rays [...,6] or a CameraDesc, ts [S] (shared) or [R,S] (per ray) -> sigma [R,S] (pre-relu), rgb [R,S,3] (sigmoid),
    ray-major.  A camera picks the light-code row of every ray from its view and takes the camera-fed kernels when
    set_camera_rays_mode(True) selected them, as nerfle_render_camera does."""
    prec = prec_id(prec)
    cam = rays_or_cam if isinstance(rays_or_cam, CameraDesc) else None
    if cam is not None:
        r2, R, dev = None, cam.n_rays, cam.device
        if view_of_ray is not None:
            raise NrtError("a camera gives every ray its view; view_of_ray must be None")
    else:
        r2 = _chk(rays_or_cam, "rays").reshape(-1, 6)
        R, dev = r2.shape[0], r2.device
    per_ray = ts.dim() == 2
    t = _chk(ts, "ts")
    if per_ray and t.shape[0] != R:
        raise NrtError("ts [R,S] has %d rows for %d rays" % (t.shape[0], R))
    S = t.shape[-1] if per_ray else t.numel()
    lc = _chk(light_code, "light_code")
    lc = lc.reshape(-1, lc.shape[-1])
    vor = _chk(view_of_ray.reshape(-1), "view_of_ray", torch.int32) if view_of_ray is not None else None
    sigma = torch.empty((R, S), dtype=torch.float32, device=dev)
    rgb = torch.empty((R, S, 3), dtype=torch.float32, device=dev)
    cs = ctypes.byref(cam.struct) if cam is not None else None
    with torch.cuda.device(dev):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        ws = _cached_ws(_ws_cache, dev, N.lib().nrt_nerfle_render_samples_workspace(ctypes.byref(c1), ctypes.byref(c2), prec,
                                                                                     R, S, cs))
        N.check(N.lib().nrt_nerfle_render_samples(ctypes.byref(c1), ctypes.byref(c2), prec, _ptr(r2), cs, R,
                                                  None if per_ray else _ptr(t), _ptr(t) if per_ray else None, S, _ptr(lc),
                                                  lc.shape[-1], _ptr(vor), _ptr(sigma), _ptr(rgb), _ptr(ws), ws.numel(),
                                                  _stream()))
    return sigma, rgb


def nerfle_render_camera_host(first: PackedMLP, second: PackedMLP, cam: CameraDesc, ts_host: Optional[torch.Tensor],
                              light_code: torch.Tensor, out_host: torch.Tensor, prec=PREC_F32, n_coarse=None,
                              n_fine=0, t_near=0.0, t_far=0.0, jitter_seed=0):
    """End-to-end leg of the camera-driven render: only the camera goes in, the image comes back to HOST memory."""
    prec = prec_id(prec)
    assert not out_host.is_cuda and out_host.numel() == cam.n_rays * 3
    S = ts_host.numel() if ts_host is not None else 0
    if n_coarse is None:
        n_coarse = S
    lc = _chk(light_code, "light_code")
    samp = N.NrtNerfSampling(int(n_coarse), int(n_fine), float(t_near), float(t_far), int(jitter_seed))
    with torch.cuda.device(cam.device):
        c1, c2 = first.c_struct(prec), second.c_struct(prec)
        N.check(N.lib().nrt_nerfle_render_camera_host(
            ctypes.byref(c1), ctypes.byref(c2), prec, ctypes.byref(cam.struct),
            ctypes.c_void_p(ts_host.data_ptr()) if ts_host is not None else None, S, ctypes.byref(samp), _ptr(lc),
            lc.shape[-1], ctypes.c_void_p(out_host.data_ptr()), _stream()))
    return out_host


# ---- meshes: a SphereSDF on a lattice, isosurface extraction (nrt_sdf_lattice_eval, nrt_isosurface_*) --------------
def lattice(shape, origin, spacing) -> N.NrtLattice:
    """nrt_lattice_t of a [nx, ny, nz] lattice with fp32 origin and spacing (validated by the library)."""
    nx, ny, nz = (int(n) for n in shape)
    return N.NrtLattice(nx, ny, nz, (ctypes.c_float * 3)(*[float(x) for x in origin]),
                        (ctypes.c_float * 3)(*[float(x) for x in spacing]))


def _cached_ws(cache, dev, nbytes):
    if nbytes < 0:
        N.check(int(nbytes))
    key = (dev.index, torch.cuda.current_stream().cuda_stream)
    ws = cache.get(key)
    if ws is None or ws.numel() < nbytes:
        cache.pop(key, None)
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        cache[key] = ws
    return ws


_lattice_ws_cache = {}
_iso_ws_cache = {}


def sdf_lattice(s: PackedSDF, g: N.NrtLattice, prec=PREC_F32) -> torch.Tensor:
    """SphereSDF.forward at every point of lattice g: values [nx, ny, nz] (nrt_sdf_lattice_eval, nrt_sdf_eval at `prec`)."""
    prec = prec_id(prec)
    dev = s.centers.device
    values = torch.empty((g.nx, g.ny, g.nz), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        c = s.c_struct(prec)
        ws = _cached_ws(_lattice_ws_cache, dev, N.lib().nrt_sdf_lattice_eval_workspace(ctypes.byref(g)))
        N.check(N.lib().nrt_sdf_lattice_eval(ctypes.byref(c), prec, ctypes.byref(g), _ptr(values), _ptr(ws), ws.numel(),
                                             _stream()))
    return values


def isosurface(values: torch.Tensor, origin, spacing, level=0.0):
    """Marching tetrahedra on the lattice values [nx, ny, nz] (point (i,j,k) at origin + (i,j,k) * spacing) ->
    verts [V,3] float32, faces [F,3] int64; conventions in include/nrt_b200.h.  Count pass, ONE device-to-host read of
    (V, F) (the only host synchronisation), allocation, emit pass.  The workspace (19 bytes per lattice point) is kept
    per device and stream."""
    v = _chk(values, "values")
    if v.dim() != 3:
        raise NrtError("values must be a 3-D [nx, ny, nz] lattice, got %s" % (tuple(values.shape),))
    g = lattice(v.shape, origin, spacing)
    dev = v.device
    with torch.cuda.device(dev):
        ws = _cached_ws(_iso_ws_cache, dev, N.lib().nrt_isosurface_workspace(ctypes.byref(g)))
        counts = torch.empty(2, dtype=torch.int64, device=dev)
        N.check(N.lib().nrt_isosurface_count(ctypes.byref(g), _ptr(v), float(level), _ptr(ws), ws.numel(), _ptr(counts),
                                             _stream()))
        nv, nf = counts.tolist()
        verts = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        faces = torch.empty((nf, 3), dtype=torch.int64, device=dev)
        N.check(N.lib().nrt_isosurface_emit(ctypes.byref(g), _ptr(v), float(level), _ptr(ws), ws.numel(), nv, nf,
                                            _ptr(verts), _ptr(faces), _stream()))
    return verts, faces


# ---- launch accounting / per-kernel timing ----------------------------------------------------
def profile_enable(on: bool):
    N.check(N.lib().nrt_profile_enable(1 if on else 0))


def profile_collect():
    """{kernel tag: (summed device ms [needs profile_enable], launches)} since the last collect."""
    n = N.lib().nrt_profile_num_tags()
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_longlong * n)()
    N.check(N.lib().nrt_profile_collect(n, ms, cnt))
    return {N.lib().nrt_profile_tag_name(i).decode(): (ms[i], int(cnt[i])) for i in range(n)}
