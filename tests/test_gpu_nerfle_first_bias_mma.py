"""NeRFLE.first's inference kernels on the render layout (NRT_BIAS_MMA bit 2, csrc/tc_core.cuh make_render_layout): the
init and skip layers take their biases from weight rows in the padding of the encoding's x segment, the other layers from
8-deep bias chunks, and no epilogue pre-loads a bias.  Checked here: the plain forward and the render pass (uniform and
64 + 128 hierarchical), f16 and bf16, sample counts that are not a multiple of 128 samples x 148 SMs x 2 tile slots,
against the exact fp32 kernels (max-abs 1e-3 f16, 5e-3 bf16); the camera-fed frame against the ray-fed one, bit for bit;
the blob, byte for byte, against a numpy restatement of both layouts; and the training forward, which must read only
the training layout at the front of the blob."""
import ctypes

import numpy as np
import pytest

import helpers
import synth

pytestmark = pytest.mark.gpu

TOL = {"f16": 1e-3, "bf16": 5e-3}
M_ODD = [1, 148 * 2 * 128 + 77, 148 * 2 * 128 * 2 + 129]
TRAIN_BYTES = 225280             # make_layout(3, 0, 16, 128, 5, 3, 65): 110,848 16-bit weights + 896 floats
RENDER_BYTES = 229312            # 3,712 16-bit chunk elements + the weights + 48 basis floats


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _first(seed=31):
    return synth.mlp_weights(seed=seed, in_size=3, out=65, num_layers=5, hidden=128, freqs=16, sigma=32.0)


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("M", M_ODD)
def test_first_mlp_vs_exact(prec, M):
    """The plain [M, 3] -> [M, 65] forward (every layer takes its bias from an MMA)."""
    from neural_raytracing_b200 import ops
    m = helpers.cuda_mlp(_first())
    x = _t((0.8 * np.random.RandomState(M).standard_normal((M, 3))).astype(np.float32))
    y32 = ops.mlp_forward(m, x, prec="f32").cpu().numpy()
    y = ops.mlp_forward(m, x, prec=prec).cpu().numpy()
    assert y.shape == y32.shape and np.isfinite(y).all()
    assert np.abs(y - y32).max() < TOL[prec], np.abs(y - y32).max()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("R", [1337, 3083])
def test_render_vs_exact(prec, R):
    """ops.nerfle_render: one uniform pass of 192 samples, and the 64 + 128 hierarchical frame (R * 192 samples is not
    a multiple of 128 x 148 x 2)."""
    from neural_raytracing_b200 import ops
    w1, w2 = helpers.nerfle_weights(False)
    m1, m2 = helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)
    rays = _t(synth.camera_rays(35, R))
    code = _t(np.array([[0.4, 1.0, 0.3]], np.float32))
    ts = _t(np.linspace(0.0, 2.05, 192).astype(np.float32))
    r32 = ops.nerfle_render(m1, m2, rays, ts, code, prec="f32").cpu().numpy()
    r = ops.nerfle_render(m1, m2, rays, ts, code, prec=prec).cpu().numpy()
    assert np.isfinite(r).all()
    assert np.abs(r - r32).max() < TOL[prec], np.abs(r - r32).max()
    kw = dict(n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=3)
    h32 = ops.nerfle_render(m1, m2, rays, None, code, prec="f32", **kw).cpu().numpy()
    h = ops.nerfle_render(m1, m2, rays, None, code, prec=prec, **kw).cpu().numpy()
    assert np.isfinite(h).all()
    assert np.abs(h - h32).max() < TOL[prec], np.abs(h - h32).max()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_camera_fed_equals_ray_fed(prec):
    import torch
    from neural_raytracing_b200 import ops
    w1, w2 = helpers.nerfle_weights(False)
    m1, m2 = helpers.cuda_mlp(w1), helpers.cuda_mlp(w2)
    c2w, focal = synth.nerf_cameras(1, 400, device="cuda")
    desc = ops.CameraDesc(ops.CAM_NERF, c2w, None, focal=focal, size=400, x0=5, y0=13, nx=41, ny=23)
    code = _t(np.array([[0.4, 1.0, 0.3]], np.float32))
    kw = dict(prec=prec, n_coarse=64, n_fine=128, t_near=0.0, t_far=2.05, jitter_seed=8)
    ray_fed = ops.nerfle_render(m1, m2, ops.camera_rays(desc), None, code, **kw)
    try:
        ops.set_camera_rays_mode(True)
        cam_fed = ops.nerfle_render_camera(m1, m2, desc, None, code, **kw)
    finally:
        ops.set_camera_rays_mode(False)
    assert torch.isfinite(cam_fed).all()
    assert torch.equal(cam_fed.reshape(-1, 3), ray_fed.reshape(-1, 3))


# ---- numpy restatement of the two layouts (UMMA canonical no-swizzle K-major: (n, k) at ((k/8)*N + n)*8 + k%8) ----
def _cvt(v, fmt):
    """float32 -> 16-bit operand bits (round to nearest even)"""
    v = np.asarray(v, np.float32)
    if fmt == "f16":
        return v.astype(np.float16).view(np.uint16)
    u = v.view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def _back(h, fmt):
    return h.view(np.float16).astype(np.float32) if fmt == "f16" else (h.astype(np.uint32) << 16).view(np.float32)


def _bias_terms(b, fmt):
    """b = b_hi + b_mid + b_lo, each the 16-bit rounding of what the previous terms left over"""
    out, res = [], np.asarray(b, np.float32)
    for _ in range(3):
        v = _back(_cvt(res, fmt), fmt)
        out.append(v)
        res = (res - v).astype(np.float32)
    return out


def _canon(dense):
    """dense [N, K] -> canonical element order"""
    N, K = dense.shape
    return dense.reshape(N, K // 8, 8).transpose(1, 0, 2).reshape(-1)


def _ops(w, fmt):
    """the 8 dense operands [N, K] of NeRFLE.first's training layout, as float32 values before rounding"""
    W, basis = w["W"], w["basis"]                     # W[i]: [N, K] (nn.Linear), basis [3, 16]
    ph = np.zeros((16, 16), np.float32)               # phase op: K = [x_hi | x_lo | x_hi] segments of 3
    hi = _back(_cvt(basis, fmt), fmt)
    for k in range(9):
        j = k % 3
        ph[:, k] = hi[j] if k < 6 else (basis[j] - hi[j])

    def enc(Wl, k0):                                  # reference encoding [x(3) | sin(16) | cos(16)] -> K = 48
        e = np.zeros((128, 48), np.float32)
        e[:, 0:3] = Wl[:, k0:k0 + 3]
        e[:, 3:6] = Wl[:, k0:k0 + 3]
        e[:, 16:48] = Wl[:, k0 + 3:k0 + 35]
        return e
    ops = [ph, enc(W[0], 0)]
    for i in range(5):
        Wl = W[1 + i]
        ops.append(np.concatenate([Wl[:, :128], enc(Wl, 128)], 1) if i in (0, 3) else Wl.copy())
    out = np.zeros((80, 128), np.float32)
    out[:65] = W[6]
    ops.append(out)
    return ops


def _train_blob(w, fmt):
    ops = _ops(w, fmt)
    wts = np.concatenate([_cvt(_canon(o), fmt) for o in ops])
    bias = np.concatenate([b if b.size == 128 else np.pad(b, (0, 80 - b.size)) for b in w["b"]]).astype(np.float32)
    basis = w["basis"].astype(np.float32).reshape(-1)
    return wts.tobytes() + bias.tobytes() + basis.tobytes()


def _render_blob(w, fmt):
    ops = _ops(w, fmt)
    for o, li in ((1, 0), (2, 1), (5, 4)):            # bias rows 9, 10, 11 of the encoding part
        k0 = 0 if o == 1 else 128
        for t, v in enumerate(_bias_terms(w["b"][li], fmt)):
            ops[o][:, k0 + 9 + t] = v
    chunks = []
    for o, li in ((7, 6), (3, 2), (4, 3), (6, 5)):    # 8-deep chunks: (n, k < 8) at n*8 + k
        N = ops[o].shape[0]
        c = np.zeros((N, 8), np.float32)
        for t, v in enumerate(_bias_terms(w["b"][li], fmt)):
            c[:v.size, t] = v
        chunks.append(_cvt(c.reshape(-1), fmt))
    wts = np.concatenate(chunks + [_cvt(_canon(o), fmt) for o in ops])
    return wts.tobytes() + w["basis"].astype(np.float32).reshape(-1).tobytes()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_blob_layouts(prec):
    """The blob holds the training layout, unchanged, then (128-byte aligned) the render layout."""
    from neural_raytracing_b200 import _native as N
    from neural_raytracing_b200 import ops
    w = _first()
    m = helpers.cuda_mlp(w)
    c = m.c_struct()
    assert N.lib().nrt_mlp_tc_blob_bytes(ctypes.byref(c), ops.prec_id(prec)) == TRAIN_BYTES + RENDER_BYTES
    blob = m.tc_blob(ops.prec_id(prec)).cpu().numpy().tobytes()
    assert len(blob) == TRAIN_BYTES + RENDER_BYTES
    assert blob[:TRAIN_BYTES] == _train_blob(w, prec)
    assert blob[TRAIN_BYTES:] == _render_blob(w, prec)


def _train_forward(m, x, blob):
    """nrt_mlp_forward_train_tc (f16) on the given blob, into a zeroed workspace: (out, workspace with the saved tiles)"""
    import torch
    from neural_raytracing_b200 import _native as N
    from neural_raytracing_b200 import ops
    p = ops.prec_id("f16")
    c = m.c_struct()
    c.params_tc = blob.data_ptr()
    M = x.shape[0]
    ws = torch.zeros(int(N.lib().nrt_mlp_train_tc_workspace_bytes(ctypes.byref(c), M)), dtype=torch.uint8, device="cuda")
    out = torch.zeros((M, 65), dtype=torch.float32, device="cuda")
    N.check(N.lib().nrt_mlp_forward_train_tc(ctypes.byref(c), p, ops.OUT_NONE, x.data_ptr(), M, out.data_ptr(), ws.data_ptr(),
                                             ws.numel(), ops._stream()))
    torch.cuda.synchronize()
    return out, ws


def test_training_forward_reads_the_training_layout():
    """The training forward (sigma / latent and the saved tiles) is bit-identical with a blob cut down to the training
    layout, i.e. with what a build without the render layout allocates and packs."""
    import torch
    from neural_raytracing_b200 import ops
    m = helpers.cuda_mlp(_first(seed=12))
    x = _t((0.8 * np.random.RandomState(3).standard_normal((148 * 2 * 128 + 77, 3))).astype(np.float32))
    full = m.tc_blob(ops.prec_id("f16"))
    out, ws = _train_forward(m, x, full)
    out2, ws2 = _train_forward(m, x, full[:TRAIN_BYTES].clone())
    assert torch.isfinite(out).all()
    assert torch.equal(out, out2) and torch.equal(ws, ws2)
