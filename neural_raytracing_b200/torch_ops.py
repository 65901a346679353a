"""`torch.ops.nrt_b200.*`: the hot path as registered PyTorch operators (SURVEY.md section 8b "custom-op layer").

Every operator is a thin functional wrapper (tensors, ints and floats only, no Python objects) over one or two entry
points of libnrt_b200's C ABI (include/nrt_b200.h) with
  * an implementation for CUDA tensors (ctypes -> the hand-written kernels; there is no CPU implementation),
  * a fake (meta) implementation, so shapes propagate under FakeTensor / torch.compile tracing,
  * a registered backward where the reference differentiates the function: the SkipConnMLP (neural_blocks.py:75-86),
    compositing (nerf.py:205-213) and the forward-mode (value, d value / d p) pair behind SDF.autograd_diff
    (sdfs.py:184-197).  The scan loops are `no_grad` in the reference (sdfs.py:119-131, 169-180, 237-245) and carry none.

A network is described by its packed-f32 parameter blob (`params`, layout of nrt_mlp_t: W^T [K][N] + bias per Linear in
evaluation order), its Fourier basis [in, freqs] and `arch = [in_size, latent_size, freqs, hidden, num_layers, skip,
out_size, activation]`.  `pack_module(mlp)` builds the blob from a SkipConnMLP with differentiable torch ops, so
gradients returned for `params` reach the nn.Linear weights.  The class layer (pathtracer/*) caches the packed and
tensor-core blobs per module; these functional operators re-derive them per call.
"""
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import ops

NS = "nrt_b200"


def _mlp(params: Tensor, basis: Tensor, arch: List[int]) -> "ops.PackedMLP":
    if len(arch) != 8:
        raise ops.NrtError("arch must be [in_size, latent_size, freqs, hidden, num_layers, skip, out_size, activation]")
    i, lat, f, h, L, sk, o, act = [int(v) for v in arch]
    return ops.PackedMLP(i, lat, f, h, L, sk, o, act, basis.detach().contiguous(), params.detach().contiguous())


def _sdf(centers, radii, tfs, params, basis, arch) -> "ops.PackedSDF":
    return ops.PackedSDF(centers, radii, tfs, _mlp(params, basis, arch))


def arch_of(mlp) -> List[int]:
    """`arch` of a pathtracer.neural_blocks.SkipConnMLP."""
    from .pathtracer.neural_blocks import _activation_id
    return [mlp.in_size, mlp.latent_size, int(mlp.basis_p.shape[-1]), mlp.init.out_features, len(mlp.layers), mlp.skip,
            mlp.out.out_features, _activation_id(mlp.activation)]


def pack_module(mlp) -> Tensor:
    """Packed-f32 parameter blob of a SkipConnMLP, differentiable w.r.t. its nn.Linear weights and biases."""
    chunks = []
    for lin in [mlp.init] + list(mlp.layers) + [mlp.out]:
        chunks.append(lin.weight.t().reshape(-1))
        chunks.append(lin.bias.reshape(-1))
    return torch.cat(chunks).float()


# ---- a2: SkipConnMLP ----------------------------------------------------------------------------------------
@torch.library.custom_op(NS + "::mlp_forward", mutates_args=())
def mlp_forward(x: Tensor, latent: Optional[Tensor], params: Tensor, basis: Tensor, arch: List[int], out_act: int,
                prec: int) -> Tuple[Tensor, Tensor]:
    """x [M,in] (+ latent [M,latent]) -> (out [M,out] with `out_act` applied, acts).  `acts` holds the post-activation
    layer inputs the fp32 backward needs (empty for the tensor-core precisions, which are inference-only here)."""
    m = _mlp(params, basis, arch)
    if prec == ops.PREC_F32:
        out, acts = ops.mlp_forward(m, x, latent, out_act=out_act, prec=prec, save_acts=True)
        return out.reshape(-1, m.out_size), acts
    out = ops.mlp_forward(m, x, latent, out_act=out_act, prec=prec)
    return out.reshape(-1, m.out_size), x.new_empty(0)


@mlp_forward.register_fake
def _(x, latent, params, basis, arch, out_act, prec):
    M = x.reshape(-1, arch[0]).shape[0]
    acts = x.new_empty(((arch[4] + 1) * arch[3], M)) if prec == ops.PREC_F32 else x.new_empty(0)
    return x.new_empty((M, arch[6])), acts


@torch.library.custom_op(NS + "::mlp_backward", mutates_args=())
def mlp_backward(x: Tensor, latent: Optional[Tensor], out: Tensor, acts: Tensor, g_out: Tensor, params: Tensor,
                 basis: Tensor, arch: List[int], out_act: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Reverse mode of mlp_forward (fp32): (g_params [P], g_x [M,in], g_latent [M,latent] or empty)."""
    m = _mlp(params, basis, arch)
    g_params, g_x, g_lat = ops.mlp_backward(m, x, latent, out, acts, g_out.contiguous(), out_act=out_act, need_input_grad=True)
    return g_params, g_x, g_lat if g_lat is not None else x.new_empty(0)


@mlp_backward.register_fake
def _(x, latent, out, acts, g_out, params, basis, arch, out_act):
    M = x.reshape(-1, arch[0]).shape[0]
    return params.new_empty(params.shape), x.new_empty((M, arch[0])), x.new_empty((M, arch[1]) if arch[1] else (0,))


def _mlp_setup(ctx, inputs, output):
    x, latent, params, basis, arch, out_act, prec = inputs
    if prec != ops.PREC_F32:
        raise ops.NrtError("nrt_b200::mlp_forward is differentiable in fp32 only; 16-bit training: "
                           "torch.ops.nrt_b200.mlp_forward_train_tc (forward and backward on the tensor cores)")
    out, acts = output
    ctx.save_for_backward(x, latent if latent is not None else x.new_empty(0), out, acts, params, basis)
    ctx.arch, ctx.out_act, ctx.has_latent = list(arch), out_act, latent is not None


def _mlp_bwd(ctx, g_out, g_acts):
    x, latent, out, acts, params, basis = ctx.saved_tensors
    lat = latent if ctx.has_latent else None
    g_params, g_x, g_lat = torch.ops.nrt_b200.mlp_backward(x, lat, out, acts, g_out, params, basis, ctx.arch, ctx.out_act)
    return g_x.reshape(x.shape), (g_lat.reshape(latent.shape) if ctx.has_latent else None), g_params, None, None, None, None


mlp_forward.register_autograd(_mlp_bwd, setup_context=_mlp_setup)


# ---- a2 under autograd on the tensor cores (north_star: forward and backward registered) ---------------------------------
@torch.library.custom_op(NS + "::mlp_forward_train_tc", mutates_args=())
def mlp_forward_train_tc(x: Tensor, params: Tensor, basis: Tensor, arch: List[int], out_act: int, prec: int) -> Tuple[Tensor, Tensor]:
    """Tensor-core training forward (tcgen05, 16-bit operands / fp32 accumulate): x [M,in] -> (out [M,out] with `out_act`
    applied, workspace of saved activation tiles for mlp_backward_tc).  The shapes the library instantiates: NeRFLE.first /
    .second, NeuralBSDF.mlp, the occlusion MLP, SphereSDF.shift, sp_var_fn (4 / 8 / 16 bases), LightField; others raise."""
    m = _mlp(params, basis, arch)
    out, ws = ops.mlp_forward_train_tc(m, x, out_act, prec=prec)
    return out, ws


@mlp_forward_train_tc.register_fake
def _(x, params, basis, arch, out_act, prec):
    M = x.reshape(-1, arch[0]).shape[0]
    ws = torch.empty(torch.library.get_ctx().new_dynamic_size(), dtype=torch.uint8, device=x.device)
    return x.new_empty((M, arch[6])), ws


@torch.library.custom_op(NS + "::mlp_backward_tc", mutates_args=())
def mlp_backward_tc(x: Tensor, out: Tensor, ws: Tensor, g_out: Tensor, params: Tensor, basis: Tensor, arch: List[int],
                    out_act: int, prec: int, need_input_grad: bool) -> Tuple[Tensor, Tensor]:
    """Reverse mode of mlp_forward_train_tc: streamed dgrad + wgrad on the tensor cores -> (g_params [P], g_x [M,in] or
    empty).  NeRFLE.first has no input gradient on this path (its inputs are ray samples; split-precision encoding)."""
    m = _mlp(params, basis, arch)
    M = x.reshape(-1, arch[0]).shape[0]
    g_params, g_x = ops.mlp_backward_tc(m, M, out, g_out.contiguous(), ws, out_act, need_input_grad=need_input_grad, prec=prec)
    return g_params, g_x if g_x is not None else x.new_empty(0)


@mlp_backward_tc.register_fake
def _(x, out, ws, g_out, params, basis, arch, out_act, prec, need_input_grad):
    M = x.reshape(-1, arch[0]).shape[0]
    return params.new_empty(params.shape), x.new_empty((M, arch[0]) if need_input_grad else (0,))


def _mlp_tc_setup(ctx, inputs, output):
    x, params, basis, arch, out_act, prec = inputs
    out, ws = output
    ctx.save_for_backward(x, out, ws, params, basis)
    ctx.arch, ctx.out_act, ctx.prec = list(arch), out_act, prec


def _mlp_tc_bwd(ctx, g_out, g_ws):
    x, out, ws, params, basis = ctx.saved_tensors
    need = bool(ctx.needs_input_grad[0])
    g_params, g_x = torch.ops.nrt_b200.mlp_backward_tc(x, out, ws, g_out, params, basis, ctx.arch, ctx.out_act, ctx.prec, need)
    return (g_x.reshape(x.shape) if need else None), g_params, None, None, None, None


mlp_forward_train_tc.register_autograd(_mlp_tc_bwd, setup_context=_mlp_tc_setup)


# ---- a19: compositing ------------------------------------------------------------------------------------------
@torch.library.custom_op(NS + "::composite", mutates_args=())
def composite(sigma_raw: Tensor, rgb: Tensor, ts: Tensor) -> Tensor:
    """nerf.py:205-213 on sample-major sigma_raw [S,R], rgb [S,R,3], ts [S] -> [R,3] (quirks kept, see DESIGN 4.4)."""
    return ops.composite_forward(sigma_raw, rgb, ts).reshape(-1, 3)


@composite.register_fake
def _(sigma_raw, rgb, ts):
    return sigma_raw.new_empty((sigma_raw[0].numel(), 3))


@torch.library.custom_op(NS + "::composite_backward", mutates_args=())
def composite_backward(sigma_raw: Tensor, rgb: Tensor, ts: Tensor, g_out: Tensor) -> Tuple[Tensor, Tensor]:
    g_s, g_c = ops.composite_backward(sigma_raw, rgb, ts, g_out.contiguous())
    return g_s.reshape(sigma_raw.shape), g_c.reshape(rgb.shape)


@composite_backward.register_fake
def _(sigma_raw, rgb, ts, g_out):
    return sigma_raw.new_empty(sigma_raw.shape), rgb.new_empty(rgb.shape)


def _comp_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _comp_bwd(ctx, g):
    s, c, t = ctx.saved_tensors
    g_s, g_c = torch.ops.nrt_b200.composite_backward(s, c, t, g)
    return g_s, g_c, None


composite.register_autograd(_comp_bwd, setup_context=_comp_setup)


@torch.library.custom_op(NS + "::composite_ts", mutates_args=())
def composite_ts(sigma_raw: Tensor, rgb: Tensor, ts: Tensor) -> Tensor:
    """composite with per-sample distances ts [S,R] (hierarchical sampling; the reference's quirks kept) -> [R,3]."""
    return ops.composite_forward_ts(sigma_raw, rgb, ts).reshape(-1, 3)


@composite_ts.register_fake
def _(sigma_raw, rgb, ts):
    return sigma_raw.new_empty((sigma_raw[0].numel(), 3))


@torch.library.custom_op(NS + "::composite_ts_backward", mutates_args=())
def composite_ts_backward(sigma_raw: Tensor, rgb: Tensor, ts: Tensor, g_out: Tensor) -> Tuple[Tensor, Tensor]:
    g_s, g_c = ops.composite_backward_ts(sigma_raw, rgb, ts, g_out.contiguous())
    return g_s.reshape(sigma_raw.shape), g_c.reshape(rgb.shape)


@composite_ts_backward.register_fake
def _(sigma_raw, rgb, ts, g_out):
    return sigma_raw.new_empty(sigma_raw.shape), rgb.new_empty(rgb.shape)


def _comp_ts_bwd(ctx, g):
    s, c, t = ctx.saved_tensors
    g_s, g_c = torch.ops.nrt_b200.composite_ts_backward(s, c, t, g)
    return g_s, g_c, None


composite_ts.register_autograd(_comp_ts_bwd, setup_context=_comp_setup)


# ---- a6 / a22: value and Jacobian of an in_size-3 SkipConnMLP (SphereSDF.shift) -----------------------------------
@torch.library.custom_op(NS + "::mlp_value_jac", mutates_args=())
def mlp_value_jac(p: Tensor, params: Tensor, basis: Tensor, arch: List[int]) -> Tuple[Tensor, Tensor, Tensor]:
    """p [M,3] -> (value [M,out], jac [M,out,3] = d value / d p, saved four-column activations)."""
    val, jac, acts = ops.mlp_value_jac_forward(_mlp(params, basis, arch), p, save_acts=True)
    return val, jac, acts


@mlp_value_jac.register_fake
def _(p, params, basis, arch):
    M = p.reshape(-1, 3).shape[0]
    return p.new_empty((M, arch[6])), p.new_empty((M, arch[6], 3)), p.new_empty(((arch[4] + 1) * arch[3], 4 * M))


@torch.library.custom_op(NS + "::mlp_value_jac_backward", mutates_args=())
def mlp_value_jac_backward(p: Tensor, acts: Tensor, g_value: Tensor, g_jac: Tensor, params: Tensor, basis: Tensor,
                           arch: List[int]) -> Tensor:
    """The hand-written reverse pass of mlp_value_jac into the packed parameters (the reference's double backward)."""
    return ops.mlp_value_jac_backward(_mlp(params, basis, arch), p, acts, g_value.contiguous(), g_jac.contiguous())


@mlp_value_jac_backward.register_fake
def _(p, acts, g_value, g_jac, params, basis, arch):
    return params.new_empty(params.shape)


def _vj_setup(ctx, inputs, output):
    p, params, basis, arch = inputs
    ctx.save_for_backward(p, output[2], params, basis)
    ctx.arch = list(arch)


def _vj_bwd(ctx, g_val, g_jac, g_acts):
    p, acts, params, basis = ctx.saved_tensors
    g_params = torch.ops.nrt_b200.mlp_value_jac_backward(p, acts, g_val, g_jac, params, basis, ctx.arch)
    return None, g_params, None, None          # p carries no gradient (the march is no_grad in the reference)


mlp_value_jac.register_autograd(_vj_bwd, setup_context=_vj_setup)


# ---- a3 / a4 / a5 / a7: SphereSDF evaluation and the three gradient-free scan loops -----------------------------------
@torch.library.custom_op(NS + "::sdf_eval", mutates_args=())
def sdf_eval(p: Tensor, centers: Tensor, radii: Tensor, tfs: Tensor, params: Tensor, basis: Tensor, arch: List[int],
             prec: int) -> Tensor:
    return ops.sdf_eval(_sdf(centers, radii, tfs, params, basis, arch), p, prec=prec).reshape(-1)


@sdf_eval.register_fake
def _(p, centers, radii, tfs, params, basis, arch, prec):
    return p.new_empty((p.reshape(-1, 3).shape[0],))


@torch.library.custom_op(NS + "::sdf_sphere_trace", mutates_args=())
def sdf_sphere_trace(rays: Tensor, centers: Tensor, radii: Tensor, tfs: Tensor, params: Tensor, basis: Tensor,
                     arch: List[int], epsilon: float, max_steps: int, max_t: float, prec: int) -> Tuple[Tensor, Tensor]:
    """SDF.intersect march (sdfs.py:111-131): rays [R,6] -> (depth [R], hit [R] bool)."""
    d, h = ops.sphere_trace(_sdf(centers, radii, tfs, params, basis, arch), rays, epsilon, max_steps, max_t, prec=prec)
    return d.reshape(-1), h.reshape(-1)


@sdf_sphere_trace.register_fake
def _(rays, centers, radii, tfs, params, basis, arch, epsilon, max_steps, max_t, prec):
    R = rays.reshape(-1, 6).shape[0]
    return rays.new_empty((R,)), rays.new_empty((R,), dtype=torch.bool)


@torch.library.custom_op(NS + "::sdf_shadow_test", mutates_args=())
def sdf_shadow_test(rays: Tensor, max_t: Tensor, centers: Tensor, radii: Tensor, tfs: Tensor, params: Tensor, basis: Tensor,
                    arch: List[int], epsilon: float, max_steps: int, prec: int) -> Tensor:
    """SDF.intersect_test (sdfs.py:162-181): rays [R,6], max_t [R] -> not_blocked [R] bool."""
    return ops.shadow_test(_sdf(centers, radii, tfs, params, basis, arch), rays, max_t, epsilon, max_steps, prec=prec).reshape(-1)


@sdf_shadow_test.register_fake
def _(rays, max_t, centers, radii, tfs, params, basis, arch, epsilon, max_steps, prec):
    return rays.new_empty((rays.reshape(-1, 6).shape[0],), dtype=torch.bool)


@torch.library.custom_op(NS + "::sdf_min_scan", mutates_args=())
def sdf_min_scan(rays: Tensor, centers: Tensor, radii: Tensor, tfs: Tensor, params: Tensor, basis: Tensor, arch: List[int],
                 step: float, n_steps: int, prec: int) -> Tuple[Tensor, Tensor, Tensor]:
    """SDF.throughput scan (sdfs.py:232-249): (best_idx int32 [R], best_pos [R,3], min value [R])."""
    i, pos, mv = ops.min_scan(_sdf(centers, radii, tfs, params, basis, arch), rays, step, n_steps, prec=prec)
    return i.reshape(-1), pos.reshape(-1, 3), mv.reshape(-1)


@sdf_min_scan.register_fake
def _(rays, centers, radii, tfs, params, basis, arch, step, n_steps, prec):
    R = rays.reshape(-1, 6).shape[0]
    return rays.new_empty((R,), dtype=torch.int32), rays.new_empty((R, 3)), rays.new_empty((R,))


# ---- a18: NeRFLE volumetric render ------------------------------------------------------------------------------
@torch.library.custom_op(NS + "::nerfle_render", mutates_args=())
def nerfle_render(rays: Tensor, ts: Tensor, light_code: Tensor, params1: Tensor, basis1: Tensor, arch1: List[int],
                  params2: Tensor, basis2: Tensor, arch2: List[int], prec: int) -> Tensor:
    """NeRFLE.forward (nerf.py:175-214) for one view / light code: rays [R,6], ts [S] -> rgb [R,3] (gradient-free)."""
    return ops.nerfle_render(_mlp(params1, basis1, arch1), _mlp(params2, basis2, arch2), rays, ts, light_code,
                             prec=prec).reshape(-1, 3)


@nerfle_render.register_fake
def _(rays, ts, light_code, params1, basis1, arch1, params2, basis2, arch2, prec):
    return rays.new_empty((rays.reshape(-1, 6).shape[0], 3))


@torch.library.custom_op(NS + "::nerfle_sample_hierarchical", mutates_args=())
def nerfle_sample_hierarchical(rays: Tensor, light_code: Tensor, view_of_ray: Optional[Tensor], params1: Tensor, basis1: Tensor,
                               arch1: List[int], params2: Tensor, basis2: Tensor, arch2: List[int], prec: int, n_coarse: int,
                               n_fine: int, t_near: float, t_far: float, jitter_seed: int, seed: Optional[Tensor]) -> Tensor:
    """The merged coarse + fine distances of nerfle_render's hierarchical mode (stratified coarse pass, inverse-CDF
    resampling; an extension, nerf.py:178 uses one shared ts) -> ts [n_coarse + n_fine, R], sample-major, ascending per
    ray (gradient-free).  `seed` (one int64 on the device) replaces jitter_seed when given."""
    return ops.nerfle_sample_hierarchical(_mlp(params1, basis1, arch1), _mlp(params2, basis2, arch2), rays, light_code,
                                          view_of_ray, prec=prec, n_coarse=n_coarse, n_fine=n_fine, t_near=t_near,
                                          t_far=t_far, jitter_seed=jitter_seed, seed=seed)


@nerfle_sample_hierarchical.register_fake
def _(rays, light_code, view_of_ray, params1, basis1, arch1, params2, basis2, arch2, prec, n_coarse, n_fine, t_near, t_far,
      jitter_seed, seed):
    return rays.new_empty((n_coarse + n_fine, rays.reshape(-1, 6).shape[0]))


# ---- a21 / f4: ray generators and the camera-driven render -------------------------------------------------------
def _cam(kind: int, a: Tensor, b: Optional[Tensor], focal: float, size: float, x0: int, y0: int, nx: int, ny: int, bundle: int,
         positions: Optional[Tensor], jitter: float, jitter_seed: int) -> "ops.CameraDesc":
    return ops.CameraDesc(int(kind), a, b, focal=focal, size=size, x0=x0, y0=y0, nx=nx, ny=ny, bundle=bundle,
                          positions=positions, jitter=jitter, jitter_seed=jitter_seed)


@torch.library.custom_op(NS + "::camera_rays", mutates_args=())
def camera_rays(kind: int, a: Tensor, b: Optional[Tensor], focal: float, size: float, x0: int, y0: int, nx: int, ny: int,
                bundle: int, positions: Optional[Tensor], jitter: float, jitter_seed: int) -> Tensor:
    """sample_positions of NeRFCamera (kind 0) / DTUCamera (1) / FoVPerspectiveCameras (2) for a pixel window or explicit
    positions (cameras.py:23-54, 132-192; renderer/cameras.py:539-575) -> rays [n_views, nx, ny, bundle, 6]."""
    return ops.camera_rays(_cam(kind, a, b, focal, size, x0, y0, nx, ny, bundle, positions, jitter, jitter_seed))


@camera_rays.register_fake
def _(kind, a, b, focal, size, x0, y0, nx, ny, bundle, positions, jitter, jitter_seed):
    return a.new_empty((a.shape[0], nx, ny, bundle, 6))


@torch.library.custom_op(NS + "::nerfle_render_camera", mutates_args=())
def nerfle_render_camera(kind: int, a: Tensor, b: Optional[Tensor], focal: float, size: float, x0: int, y0: int, nx: int,
                         ny: int, bundle: int, jitter: float, jitter_seed: int, ts: Tensor, light_code: Tensor,
                         params1: Tensor, basis1: Tensor, arch1: List[int], params2: Tensor, basis2: Tensor,
                         arch2: List[int], prec: int) -> Tensor:
    """The frame of a NeRFLE from its camera in one call, rays generated on the device inside the library (f4; what pathtrace
    + NeRFReproduce compute, main.py:57-88 + nerf.py:175-214) -> rgb [n_views, nx, ny, bundle, 3] (gradient-free)."""
    cam = _cam(kind, a, b, focal, size, x0, y0, nx, ny, bundle, None, jitter, jitter_seed)
    return ops.nerfle_render_camera(_mlp(params1, basis1, arch1), _mlp(params2, basis2, arch2), cam, ts, light_code, prec=prec)


@nerfle_render_camera.register_fake
def _(kind, a, b, focal, size, x0, y0, nx, ny, bundle, jitter, jitter_seed, ts, light_code, params1, basis1, arch1, params2,
      basis2, arch2, prec):
    return a.new_empty((a.shape[0], nx, ny, bundle, 3))


OPERATORS = ["camera_rays", "nerfle_render_camera", "mlp_forward", "mlp_backward", "mlp_forward_train_tc", "mlp_backward_tc", "composite", "composite_backward", "mlp_value_jac", "mlp_value_jac_backward",
             "sdf_eval", "sdf_sphere_trace", "sdf_shadow_test", "sdf_min_scan", "nerfle_render", "composite_ts",
             "composite_ts_backward", "nerfle_sample_hierarchical"]
