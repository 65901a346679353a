"""CPU tests (no GPU) of the mesh extraction: the numpy restatement of the marching-tetrahedra kernels (tests/mesh_port.py)
yields closed, consistently oriented, accurate surfaces; the public interface of pathtracer/mesh.py validates its input and
refuses CPU tensors; the isosurface operator's fake implementation has data-dependent sizes; write_ply round-trips."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import mesh_port  # noqa: E402
from neural_raytracing_b200 import _native as N, ops, torch_ops  # noqa: E402,F401
from neural_raytracing_b200.pathtracer import mesh  # noqa: E402


def _field(fn, n, lo=-1.0, hi=1.0):
    origin, spacing = mesh_port.lattice_spacing((n, n, n), (lo,) * 3, (hi,) * 3)
    p = mesh_port.lattice_points((n, n, n), origin, spacing).astype(np.float64)
    return fn(p).astype(np.float32), origin, spacing


def _closed_oriented(faces):
    _, counts, directed_unique = mesh_port.edge_counts(faces)
    return bool(np.all(counts == 2)) and directed_unique


def test_sphere_128_closed_euler_volume_radius():
    r, n = 0.5, 128
    vals, origin, spacing = _field(lambda p: np.linalg.norm(p, axis=-1) - r, n)
    verts, faces = mesh_port.isosurface(vals, origin, spacing, 0.0)
    assert verts.dtype == np.float32 and faces.dtype == np.int64
    edges, counts, directed_unique = mesh_port.edge_counts(faces)
    assert np.all(counts == 2) and directed_unique
    assert verts.shape[0] - edges.shape[0] + faces.shape[0] == 2
    vol = mesh_port.signed_volume(verts, faces)
    exact = 4.0 / 3.0 * np.pi * r ** 3
    assert vol > 0 and abs(vol / exact - 1) < 2e-3
    h = float(spacing[0])
    assert np.abs(np.linalg.norm(verts.astype(np.float64), axis=1) - r).max() <= h * h / r
    vd = verts.astype(np.float64)
    fn = np.cross(vd[faces[:, 1]] - vd[faces[:, 0]], vd[faces[:, 2]] - vd[faces[:, 0]])
    cen = vd[faces].mean(axis=1)
    assert np.all(np.einsum("ij,ij->i", fn, cen) > 0)          # outward: along the gradient p / |p|


def test_sum_of_gaussians_closed_and_positive():
    c = np.array([[0.3, 0.0, 0.1], [-0.35, 0.2, -0.1], [0.0, -0.3, 0.25]])
    def fn(p):
        s = sum(np.exp(-np.sum((p - ci) ** 2, -1) / 0.06) for ci in c)
        return 0.4 - s                                        # inside where the blobs exceed 0.4
    vals, origin, spacing = _field(fn, 57)
    verts, faces = mesh_port.isosurface(vals, origin, spacing, 0.0)
    assert faces.shape[0] > 1000 and _closed_oriented(faces)
    assert mesh_port.signed_volume(verts, faces) > 0


def test_nonzero_level_and_noncubic_lattice():
    rng = np.random.RandomState(3)
    shape = (23, 17, 29)
    origin, spacing = mesh_port.lattice_spacing(shape, (-1, -1, -1), (1, 1, 1))
    p = mesh_port.lattice_points(shape, origin, spacing).astype(np.float64)
    vals = (np.linalg.norm(p * [1.0, 1.3, 0.8], axis=-1) + 0.01 * rng.standard_normal(shape)).astype(np.float32)
    verts, faces = mesh_port.isosurface(vals, origin, spacing, 0.6)
    assert _closed_oriented(faces) and mesh_port.signed_volume(verts, faces) > 0


def test_field_cut_by_the_box_has_boundary_on_box_faces_only():
    n = 40
    vals, origin, spacing = _field(lambda p: np.linalg.norm(p - [0.8, 0.0, 0.0], axis=-1) - 0.6, n)
    verts, faces = mesh_port.isosurface(vals, origin, spacing, 0.0)
    edges, counts, directed_unique = mesh_port.edge_counts(faces)
    assert directed_unique and np.all(counts <= 2)
    boundary = edges[counts == 1]
    assert boundary.shape[0] > 0
    far = origin + (n - 1) * spacing
    for e in boundary:
        a, b = verts[e[0]], verts[e[1]]
        on_face = [(a[ax] == bound[ax] and b[ax] == bound[ax]) for ax in range(3) for bound in (origin, far)]
        assert any(on_face), (a, b)


def test_exact_ties_stay_closed():
    n = 33
    vals, origin, spacing = _field(lambda p: np.round(np.linalg.norm(p, axis=-1) * 8) / 8 - 0.5, n)
    assert np.count_nonzero(vals == 0) > 100
    verts, faces = mesh_port.isosurface(vals, origin, spacing, 0.0)
    assert faces.shape[0] > 0 and _closed_oriented(faces)
    edges, _, _ = mesh_port.edge_counts(faces)
    assert verts.shape[0] - edges.shape[0] + faces.shape[0] == 2


def test_empty_and_all_inside():
    vals = np.ones((5, 6, 7), np.float32)
    for level in (0.0, 2.0):
        v, f = mesh_port.isosurface(vals, (0, 0, 0), (1, 1, 1), level)
        assert v.shape == (0, 3) and f.shape == (0, 3)


def test_validation_errors():
    s = torch.zeros(4, 4, 4)
    with pytest.raises(ValueError):
        mesh.isosurface(torch.zeros(4, 4), level=0.0)
    with pytest.raises(ValueError):
        mesh.isosurface(torch.zeros(4, 4, 1))
    with pytest.raises(ValueError):
        mesh.isosurface(torch.zeros(4, 4, 1025))
    with pytest.raises(ValueError):
        mesh.isosurface(s, level=float("nan"))
    with pytest.raises(ValueError):
        mesh.isosurface(s, level=float("inf"))
    with pytest.raises(ValueError):
        mesh.isosurface(s, bbox_min=(0, 0, 0), bbox_max=(1, 0, 1))
    with pytest.raises(ops.NrtError):
        mesh.isosurface(s)                                   # CPU tensor: no CPU path
    with pytest.raises(TypeError, match="isosurface"):
        mesh.sdf_grid(lambda p: p.norm(dim=-1) - 1)
    with pytest.raises(TypeError):
        mesh.extract_mesh(object())


def test_sdf_grid_validates_resolution_and_box():
    from neural_raytracing_b200.pathtracer.shapes.sdfs import SphereSDF
    s = SphereSDF(n=4, device="cpu")
    for res in (1, 1025, (8, 8), (8, 8, 0), 2.5):
        with pytest.raises(ValueError):
            mesh.sdf_grid(s, res)
    with pytest.raises(ValueError):
        mesh.sdf_grid(s, 8, bbox_min=(0, 0, 0), bbox_max=(1, 1, -1))
    with pytest.raises(ops.NrtError):
        mesh.sdf_grid(s, 8)                                  # CPU parameters: no CPU path


def test_lattice_abi_validation_without_gpu():
    L = N.lib()
    ok = ops.lattice((4, 5, 6), (0, 0, 0), (0.1, 0.1, 0.1))
    assert L.nrt_sdf_lattice_eval_workspace(ctypes.byref(ok)) == 1536     # 120 points * 12 B, 256-byte aligned
    for g in (ops.lattice((1, 5, 6), (0, 0, 0), (1, 1, 1)), ops.lattice((4, 5, 1025), (0, 0, 0), (1, 1, 1)),
              ops.lattice((4, 5, 6), (0, 0, 0), (1, 0, 1)), ops.lattice((4, 5, 6), (0, 0, 0), (1, float("inf"), 1)),
              ops.lattice((4, 5, 6), (0, float("nan"), 0), (1, 1, 1))):
        assert L.nrt_sdf_lattice_eval_workspace(ctypes.byref(g)) == N.E_INVALID
        assert L.nrt_isosurface_workspace(ctypes.byref(g)) == N.E_INVALID


def test_profile_tags_appended():
    names = [N.lib().nrt_profile_tag_name(i).decode() for i in range(N.lib().nrt_profile_num_tags())]
    assert names[-4:] == ["lattice_points", "iso_count", "iso_scan", "iso_emit"]
    assert names.index("composite_ts_bwd") == len(names) - 5


def test_isosurface_fake_has_dynamic_sizes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from torch.fx.experimental.symbolic_shapes import ShapeEnv
    assert "isosurface" in torch_ops.OPERATORS
    with FakeTensorMode(shape_env=ShapeEnv()):
        v = torch.empty(9, 10, 11, device="cuda")
        verts, faces = torch.ops.nrt_b200.isosurface(v, [0.0, 0.0, 0.0], [0.1, 0.1, 0.1], 0.0)
        assert verts.dtype == torch.float32 and faces.dtype == torch.int64
        assert verts.shape[1] == 3 and faces.shape[1] == 3
        assert isinstance(verts.shape[0], torch.SymInt) and isinstance(faces.shape[0], torch.SymInt)


def test_write_ply_round_trip(tmp_path):
    vals, origin, spacing = _field(lambda p: np.linalg.norm(p, axis=-1) - 0.5, 12)
    verts, faces = mesh_port.isosurface(vals, origin, spacing, 0.0)
    normals = verts / np.linalg.norm(verts, axis=1, keepdims=True)
    for nrm in (None, normals):
        path = str(tmp_path / "m.ply")
        mesh.write_ply(path, torch.from_numpy(verts), torch.from_numpy(faces), None if nrm is None else torch.from_numpy(nrm))
        raw = open(path, "rb").read()
        end = raw.index(b"end_header\n") + len(b"end_header\n")
        header = raw[:end].decode("ascii").splitlines()
        assert header[:2] == ["ply", "format binary_little_endian 1.0"]
        assert "element vertex %d" % len(verts) in header and "element face %d" % len(faces) in header
        nprop = 6 if nrm is not None else 3
        vdat = np.frombuffer(raw, "<f4", count=len(verts) * nprop, offset=end).reshape(-1, nprop)
        assert np.array_equal(vdat[:, :3], verts)
        if nrm is not None:
            assert np.array_equal(vdat[:, 3:], nrm.astype(np.float32))
        frec = np.frombuffer(raw, [("n", "u1"), ("i", "<i4", (3,))], offset=end + vdat.nbytes)
        assert len(frec) == len(faces) and np.all(frec["n"] == 3)
        assert np.array_equal(frec["i"].astype(np.int64), faces)
