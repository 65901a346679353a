"""Triangle meshes from a trained signed distance field (an extension: the reference renders and trains its SDF but has
no surface output).

    verts, faces = extract_mesh(sdf, resolution=256)          # SphereSDF, or SDF(sdf=SphereSDF / torch.jit.load(...))
    write_ply("shape.ply", verts, faces)

`sdf_grid` evaluates the field on a lattice over a box (the SDF kernels at the field's gradient-free precision) and
`isosurface` extracts the level set of any lattice by marching tetrahedra on the GPU (csrc/nrt_mesh.cu).  The mesh is
indexed, consistently oriented (normals point toward values >= level, outward for an SDF) and closed wherever the surface
stays inside the box.  Output order is deterministic.  CUDA only, as everywhere in this library: a CPU tensor raises
NrtError."""
import math

import numpy as np
import torch
import torch.nn.functional as F

from .. import ops
from .._native import MAX_LATTICE_DIM
from .shapes.sdfs import SDF, SphereSDF


def _resolution(resolution):
    if isinstance(resolution, (int, np.integer)):
        res = (resolution,) * 3
    elif isinstance(resolution, (tuple, list, torch.Size)):
        res = tuple(resolution)
    else:
        res = ()
    if len(res) != 3:
        raise ValueError("resolution must be an int or a 3-tuple, got %r" % (resolution,))
    for n in res:
        if int(n) != n or not 2 <= int(n) <= MAX_LATTICE_DIM:
            raise ValueError("resolution: every dimension must be an integer in [2, %d], got %r" % (MAX_LATTICE_DIM, res))
    return tuple(int(n) for n in res)


def _box(shape, bbox_min, bbox_max):
    """(origin, spacing) of the lattice: spacing = (bbox_max - bbox_min) / (n - 1) in float64, rounded to fp32 once."""
    lo = [float(x) for x in bbox_min]
    hi = [float(x) for x in bbox_max]
    if len(lo) != 3 or len(hi) != 3:
        raise ValueError("bbox_min and bbox_max must have 3 components")
    if not all(math.isfinite(x) for x in lo + hi):
        raise ValueError("bbox_min and bbox_max must be finite")
    if any(h <= l for l, h in zip(lo, hi)):
        raise ValueError("bbox_max must exceed bbox_min on every axis, got %r and %r" % (tuple(lo), tuple(hi)))
    origin = np.asarray(lo, np.float64).astype(np.float32)
    spacing = ((np.asarray(hi, np.float64) - np.asarray(lo, np.float64)) / (np.asarray(shape, np.float64) - 1)).astype(np.float32)
    return origin.tolist(), spacing.tolist()


def _sphere_sdf(sdf) -> SphereSDF:
    if isinstance(sdf, SphereSDF):
        return sdf
    if isinstance(sdf, SDF) and isinstance(sdf._impl, SphereSDF):
        return sdf._impl
    raise TypeError("sdf_grid / extract_mesh evaluate a SphereSDF, or an SDF whose implementation is one (including "
                    "SDF(sdf=torch.jit.load(archive))); got %s.  For any other field, evaluate it on a lattice yourself "
                    "and call isosurface(values, bbox_min, bbox_max, level)." % type(sdf).__name__)


def sdf_grid(sdf, resolution=256, bbox_min=(-1.0, -1.0, -1.0), bbox_max=(1.0, 1.0, 1.0)) -> torch.Tensor:
    """The field at every lattice point of the box: values [nx, ny, nz], point (i,j,k) at bbox_min + (i,j,k) * spacing.
    Bit-identical to SphereSDF.forward on the same points (gradient-free, at sphere_sdf.precision())."""
    s = _sphere_sdf(sdf)
    shape = _resolution(resolution)
    origin, spacing = _box(shape, bbox_min, bbox_max)
    with torch.no_grad():
        return ops.sdf_lattice(s.packed(), ops.lattice(shape, origin, spacing), prec=s.precision())


def isosurface(values, bbox_min=(-1.0, -1.0, -1.0), bbox_max=(1.0, 1.0, 1.0), level=0.0):
    """The surface values == level of a lattice values [nx, ny, nz] spanning the box: verts [V,3] float32,
    faces [F,3] int64 (the convention of PyTorch3D's Meshes).  Inside is values < level."""
    if not isinstance(values, torch.Tensor):
        raise TypeError("values must be a torch.Tensor")
    if values.dim() != 3:
        raise ValueError("values must be a 3-D [nx, ny, nz] lattice, got shape %s" % (tuple(values.shape),))
    shape = _resolution(tuple(values.shape))
    level = float(level)
    if not math.isfinite(level):
        raise ValueError("level must be finite, got %r" % level)
    origin, spacing = _box(shape, bbox_min, bbox_max)
    return ops.isosurface(values, origin, spacing, level)


def extract_mesh(sdf, resolution=256, bbox_min=(-1.0, -1.0, -1.0), bbox_max=(1.0, 1.0, 1.0), level=0.0, normals=False):
    """sdf_grid + isosurface: (verts, faces), or (verts, faces, vertex normals) with normals=True -- the unit gradient of
    the field at each vertex (the exact fp32 value-and-gradient kernel, ops.sdf_value_grad)."""
    s = _sphere_sdf(sdf)
    values = sdf_grid(s, resolution, bbox_min, bbox_max)
    verts, faces = isosurface(values, bbox_min, bbox_max, level)
    if not normals:
        return verts, faces
    if verts.shape[0] == 0:
        return verts, faces, torch.empty_like(verts)
    with torch.no_grad():
        _, g = ops.sdf_value_grad(s.packed(), verts)
    return verts, faces, F.normalize(g, dim=-1)


def write_ply(path, verts, faces, normals=None):
    """Binary little-endian PLY: float x y z (+ nx ny nz) per vertex, a uchar-counted int list per face."""
    v = np.ascontiguousarray(torch.as_tensor(verts).detach().cpu().numpy(), np.float32).reshape(-1, 3)
    f = torch.as_tensor(faces).detach().cpu().numpy().reshape(-1, 3)
    if f.size and (f.min() < 0 or f.max() >= v.shape[0]):
        raise ValueError("faces reference vertices outside [0, %d)" % v.shape[0])
    if v.shape[0] > np.iinfo(np.int32).max:
        raise ValueError("PLY face indices are 32-bit; %d vertices do not fit" % v.shape[0])
    props = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    if normals is not None:
        props += [("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4")]
    vrec = np.empty(v.shape[0], dtype=props)
    vrec["x"], vrec["y"], vrec["z"] = v[:, 0], v[:, 1], v[:, 2]
    if normals is not None:
        n = np.ascontiguousarray(torch.as_tensor(normals).detach().cpu().numpy(), np.float32).reshape(-1, 3)
        if n.shape[0] != v.shape[0]:
            raise ValueError("normals must have one row per vertex")
        vrec["nx"], vrec["ny"], vrec["nz"] = n[:, 0], n[:, 1], n[:, 2]
    frec = np.empty(f.shape[0], dtype=[("n", "u1"), ("i", "<i4", (3,))])
    frec["n"] = 3
    frec["i"] = f
    header = ["ply", "format binary_little_endian 1.0", "element vertex %d" % v.shape[0]]
    header += ["property float %s" % name for name, _ in props]
    header += ["element face %d" % f.shape[0], "property list uchar int vertex_indices", "end_header"]
    with open(path, "wb") as fh:
        fh.write(("\n".join(header) + "\n").encode("ascii"))
        fh.write(vrec.tobytes())
        fh.write(frec.tobytes())
