"""GPU tests of the mesh extraction (csrc/nrt_mesh.cu, ops.sdf_lattice / ops.isosurface, pathtracer/mesh.py): the kernels
against the numpy restatement (tests/mesh_port.py) bit for bit, determinism, the counts and capacities of the two passes,
the lattice evaluation against SphereSDF.forward, and the surface of an analytic sphere and of a trained-shape stand-in."""
import ctypes
import math

import numpy as np
import pytest

import mesh_port

pytestmark = pytest.mark.gpu


def _T(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _random_field(shape, seed, ties=False, nans=False):
    rng = np.random.RandomState(seed)
    origin, spacing = mesh_port.lattice_spacing(shape, (-1, -1, -1), (1, 1, 1))
    p = mesh_port.lattice_points(shape, origin, spacing).astype(np.float64)
    v = np.linalg.norm(p * [1.0, 1.2, 0.9], axis=-1) - 0.55 + 0.15 * rng.standard_normal(shape)
    if ties:
        v = np.round(v * 4) / 4
    v = v.astype(np.float32)
    if nans:
        flat = v.reshape(-1)
        idx = rng.choice(flat.size, flat.size // 50, replace=False)
        flat[idx[: len(idx) // 2]] = np.nan
        flat[idx[len(idx) // 2:: 2]] = np.inf
        flat[idx[len(idx) // 2 + 1:: 2]] = -np.inf
    return v, origin, spacing


def _same_f32(a, b):
    """Bit equality, with any NaN equal to any NaN (the hardware's and numpy's default NaNs differ in sign)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32)))


CASES = {
    "odd_dims": dict(shape=(37, 41, 29), seed=1, level=0.0),
    "level": dict(shape=(37, 41, 29), seed=2, level=0.35),
    "ties": dict(shape=(31, 26, 33), seed=3, level=0.0, ties=True),
    "nan_inf": dict(shape=(37, 41, 29), seed=4, level=0.0, nans=True),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_kernels_match_restatement_bit_for_bit(name):
    import torch
    from neural_raytracing_b200 import ops
    c = CASES[name]
    vals, origin, spacing = _random_field(c["shape"], c["seed"], c.get("ties", False), c.get("nans", False))
    if c.get("ties"):
        assert np.count_nonzero(vals == c["level"]) > 100
    rv, rf = mesh_port.isosurface(vals, origin, spacing, c["level"])
    assert rf.shape[0] > 0
    verts, faces = ops.isosurface(_T(vals), origin, spacing, c["level"])
    assert verts.dtype == torch.float32 and faces.dtype == torch.int64
    assert _same_f32(verts.cpu().numpy(), rv), name
    assert np.array_equal(faces.cpu().numpy(), rf), name
    if not c.get("nans"):
        _, counts, directed_unique = mesh_port.edge_counts(rf)
        assert directed_unique and np.all(counts <= 2)


@pytest.mark.parametrize("fill", [1.0, -1.0])
def test_empty_and_all_inside_give_typed_empty_outputs(fill):
    import torch
    from neural_raytracing_b200 import ops
    vals = np.full((9, 8, 7), fill, np.float32)
    verts, faces = ops.isosurface(_T(vals), (0, 0, 0), (0.1, 0.1, 0.1), 0.0)
    assert tuple(verts.shape) == (0, 3) and verts.dtype == torch.float32
    assert tuple(faces.shape) == (0, 3) and faces.dtype == torch.int64


def test_two_runs_are_identical():
    from neural_raytracing_b200 import ops
    vals, origin, spacing = _random_field((64, 64, 64), 5)
    v1, f1 = ops.isosurface(_T(vals), origin, spacing, 0.0)
    v2, f2 = ops.isosurface(_T(vals), origin, spacing, 0.0)
    assert np.array_equal(v1.cpu().numpy().view(np.uint32), v2.cpu().numpy().view(np.uint32))
    assert np.array_equal(f1.cpu().numpy(), f2.cpu().numpy())


def test_counts_equal_emitted_lengths_and_capacities_hold():
    import torch
    from neural_raytracing_b200 import _native as N, ops
    vals, origin, spacing = _random_field((37, 41, 29), 6)
    rv, rf = mesh_port.isosurface(vals, origin, spacing, 0.0)
    v = _T(vals)
    g = ops.lattice(vals.shape, origin, spacing)
    L = N.lib()
    nbytes = L.nrt_isosurface_workspace(ctypes.byref(g))
    assert nbytes >= 19 * vals.size
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    counts = torch.empty(2, dtype=torch.int64, device="cuda")
    N.check(L.nrt_isosurface_count(ctypes.byref(g), ops._ptr(v), 0.0, ops._ptr(ws), nbytes, ops._ptr(counts), ops._stream()))
    nv, nf = counts.tolist()
    assert (nv, nf) == (rv.shape[0], rf.shape[0])
    for cap_v, cap_f in ((nv, nf), (nv // 3, nf // 2), (0, 0)):
        verts = torch.full((nv + 7, 3), -7.0, device="cuda")
        faces = torch.full((nf + 7, 3), -7, dtype=torch.int64, device="cuda")
        N.check(L.nrt_isosurface_emit(ctypes.byref(g), ops._ptr(v), 0.0, ops._ptr(ws), nbytes, cap_v, cap_f, ops._ptr(verts),
                                      ops._ptr(faces), ops._stream()))
        vh, fh = verts.cpu().numpy(), faces.cpu().numpy()
        assert np.array_equal(vh[:cap_v].view(np.uint32), rv[:cap_v].view(np.uint32)) and np.all(vh[cap_v:] == -7.0)
        assert np.array_equal(fh[:cap_f], rf[:cap_f]) and np.all(fh[cap_f:] == -7)
    with pytest.raises(N.NrtError):
        N.check(L.nrt_isosurface_count(ctypes.byref(g), ops._ptr(v), 0.0, ops._ptr(ws), nbytes - 256, ops._ptr(counts),
                                       ops._stream()))


def _random_sphere_sdf(seed=0, n=128):
    """The shape nerf_synthetic.py trains: 128 spheres, with a randomly initialised, non-zero residual net."""
    import torch
    from neural_raytracing_b200.pathtracer.shapes.sdfs import SphereSDF
    torch.manual_seed(seed)
    s = SphereSDF(n=n, device="cuda")
    with torch.no_grad():
        for lin in s.shift._linears():
            lin.reset_parameters()
        s.shift.out.weight.mul_(0.1)
    s.invalidate_packed()
    return s


def _explicit_points(shape, origin, spacing):
    import torch
    axes = [torch.tensor(origin[a], dtype=torch.float32, device="cuda") +
            torch.arange(shape[a], device="cuda").float() * torch.tensor(spacing[a], dtype=torch.float32, device="cuda")
            for a in range(3)]
    return torch.stack(torch.meshgrid(*axes, indexing="ij"), -1)


@pytest.mark.parametrize("prec", ["f32", "f16"])
def test_sdf_grid_equals_forward_on_the_same_points(prec):
    import torch
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer import mesh
    s = _random_sphere_sdf(1)
    shape, lo, hi = (37, 41, 29), (-0.9, -1.1, -0.7), (1.0, 0.8, 1.2)
    old = config.precision
    config.precision = prec
    try:
        assert s.precision() == prec
        values = mesh.sdf_grid(s, shape, lo, hi)
        origin, spacing = mesh_port.lattice_spacing(shape, lo, hi)
        pts = _explicit_points(shape, origin.tolist(), spacing.tolist())
        assert np.array_equal(pts.cpu().numpy(), mesh_port.lattice_points(shape, origin, spacing))
        with torch.no_grad():
            ref = s(pts)
            ref_ops = s.forward_reference_ops(pts)
    finally:
        config.precision = old
    assert tuple(values.shape) == shape
    assert np.array_equal(values.cpu().numpy().view(np.uint32), ref.cpu().numpy().view(np.uint32))
    assert (values - ref_ops).abs().max().item() < (1e-4 if prec == "f32" else 5e-3)


def _unit_sphere_sdf(r=0.5):
    import torch
    from neural_raytracing_b200.pathtracer.shapes.sdfs import SphereSDF
    s = SphereSDF(n=1, device="cuda")
    with torch.no_grad():
        s.centers.zero_()
        s.radii.fill_(r)
        s.tfs.zero_()
    return s


def test_analytic_sphere_mesh():
    import torch
    from neural_raytracing_b200 import ops
    from neural_raytracing_b200.pathtracer import mesh
    r, n = 0.5, 128
    s = _unit_sphere_sdf(r)
    values = mesh.sdf_grid(s, n)
    origin, spacing = mesh_port.lattice_spacing((n,) * 3, (-1,) * 3, (1,) * 3)
    p = mesh_port.lattice_points((n,) * 3, origin, spacing).astype(np.float64)
    exact = np.linalg.norm(p, axis=-1) - r
    near = exact < 0.25                      # below the smooth-min clamp: log(1e4) / 32 = 0.288
    assert np.abs(values.cpu().numpy()[near] - exact[near]).max() < 2e-6
    verts, faces = mesh.extract_mesh(s, n)
    v, f = verts.cpu().numpy(), faces.cpu().numpy()
    edges, counts, directed_unique = mesh_port.edge_counts(f)
    assert np.all(counts == 2) and directed_unique
    assert v.shape[0] - edges.shape[0] + f.shape[0] == 2
    vol = mesh_port.signed_volume(v, f)
    assert vol > 0 and abs(vol / (4 / 3 * math.pi * r ** 3) - 1) < 2e-3
    h = float(spacing[0])
    assert np.abs(np.linalg.norm(v.astype(np.float64), axis=1) - r).max() <= h * h / r
    # every face normal agrees with the SDF gradient at its centroid
    vd = v.astype(np.float64)
    fn = np.cross(vd[f[:, 1]] - vd[f[:, 0]], vd[f[:, 2]] - vd[f[:, 0]])
    cen = vd[f].mean(axis=1)
    _, g = ops.sdf_value_grad(s.packed(), _T(cen.astype(np.float32)))
    dots = np.einsum("ij,ij->i", fn, g.cpu().numpy().astype(np.float64))
    assert np.all(dots > 0)


def test_normals_are_the_normalised_sdf_gradient():
    import torch
    from neural_raytracing_b200 import ops
    from neural_raytracing_b200.pathtracer import mesh
    s = _random_sphere_sdf(2)
    verts, faces, normals = mesh.extract_mesh(s, 64, normals=True)
    assert normals.shape == verts.shape and verts.shape[0] > 0
    assert (normals.norm(dim=-1) - 1).abs().max().item() < 1e-5
    _, g = ops.sdf_value_grad(s.packed(), verts)
    assert torch.equal(normals, torch.nn.functional.normalize(g, dim=-1))


def test_archive_extracts_the_same_mesh(tmp_path):
    import torch
    from neural_raytracing_b200.pathtracer import checkpoint, mesh
    from neural_raytracing_b200.pathtracer.shapes.sdfs import SDF
    s = _random_sphere_sdf(3)
    path = str(tmp_path / "shape.pt")
    checkpoint.save_sdf_archive(s, path)
    shape = SDF(sdf=torch.jit.load(path, "cuda"), device="cuda")
    v1, f1 = mesh.extract_mesh(s, 48)
    v2, f2 = mesh.extract_mesh(shape, 48)
    assert v1.shape[0] > 0
    assert torch.equal(v1, v2) and torch.equal(f1, f2)


def test_512_cubed_random_init_shape_f16():
    from neural_raytracing_b200 import config
    from neural_raytracing_b200.pathtracer import mesh
    s = _random_sphere_sdf(4)
    old = config.precision
    config.precision = "f16"
    try:
        verts, faces = mesh.extract_mesh(s, 512)
    finally:
        config.precision = old
    v, f = verts.cpu().numpy(), faces.cpu().numpy()
    assert f.shape[0] > 1000
    edges, counts, directed_unique = mesh_port.edge_counts(f)
    assert directed_unique and np.all(counts <= 2)
    origin, spacing = mesh_port.lattice_spacing((512,) * 3, (-1,) * 3, (1,) * 3)
    far = origin + np.float32(511) * spacing
    b = edges[counts == 1]
    a, c = v[b[:, 0]], v[b[:, 1]]
    on_face = np.zeros(len(b), bool)
    for bound in (origin, far):
        on_face |= np.any((a == bound) & (c == bound), axis=1)
    assert np.all(on_face)
