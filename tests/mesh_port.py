"""numpy restatement of the isosurface extraction of csrc/nrt_mesh.cu (marching tetrahedra on the Freudenthal
triangulation of the lattice).  TEST INFRASTRUCTURE: only the tests import it.

Conventions (the same as include/nrt_b200.h, nrt_lattice_t):
  - values [nx,ny,nz] fp32, point (i,j,k) at origin + (i,j,k) * spacing, one rounded product and one rounded sum;
  - a point is inside iff value < level (NaN is outside);
  - the vertex of a crossing edge from a (lower end) to b is p_a + t (p_b - p_a), t = (level - a) / (b - a), every
    operation rounded in fp32;
  - vertices ascend by (lattice index of the lower end, direction 1..7 with bit 0 = +i, bit 1 = +j, bit 2 = +k);
  - faces ascend by (cell, tetrahedron, triangle), and (v1 - v0) x (v2 - v0) points toward value >= level.
"""
import itertools

import numpy as np

F32 = np.float32
PERMS = list(itertools.permutations(range(3)))      # (0,1,2), (0,2,1), (1,0,2), (1,2,0), (2,0,1), (2,1,0)


def tet_offsets():
    """[6][4] corner offsets (bit 0 = +i, bit 1 = +j, bit 2 = +k) of the Kuhn tetrahedra 0 -> e_a -> e_a+e_b -> 1."""
    return [[0, 1 << a, (1 << a) | (1 << b), 7] for a, b, _ in PERMS]


def _bits(o):
    return np.array([o & 1, (o >> 1) & 1, (o >> 2) & 1], np.int64)


def tet_table():
    """table[t][case] = list of triangles, each three vertex codes o_lo | (d << 3): the crossing edge from corner
    offset o_lo in direction d.  case bit v = corner v of tetrahedron t is inside.  Orientation is fixed with exact
    integer geometry at the edge midpoints: the normal must point from the inside corners to the outside ones."""
    offs = tet_offsets()
    table = []
    for t in range(6):
        o = offs[t]
        P = [_bits(x) for x in o]
        row = []
        for case in range(16):
            ins = [v for v in range(4) if (case >> v) & 1]
            out = [v for v in range(4) if not (case >> v) & 1]
            if len(ins) in (0, 4):
                row.append([])
                continue
            if len(ins) == 1 or len(ins) == 3:
                a = ins[0] if len(ins) == 1 else out[0]
                rest = [v for v in range(4) if v != a]
                tris = [[(a, rest[0]), (a, rest[1]), (a, rest[2])]]
            else:
                A, B = ins
                C, D = out
                tris = [[(A, C), (A, D), (B, D)], [(A, C), (B, D), (B, C)]]
            g = len(ins) * sum(P[v] for v in out) - len(out) * sum(P[v] for v in ins)
            coded = []
            for tri in tris:
                m = [P[x] + P[y] for x, y in tri]                # twice the midpoints
                n = np.cross(m[1] - m[0], m[2] - m[0])
                if int(n @ g) < 0:
                    tri = [tri[0], tri[2], tri[1]]
                code = []
                for x, y in tri:
                    lo, hi = min(x, y), max(x, y)                # path order: o[lo] is a subset of o[hi]
                    code.append(o[lo] | ((o[hi] ^ o[lo]) << 3))
                coded.append(code)
            row.append(coded)
        table.append(row)
    return table


def lattice_points(shape, origin, spacing):
    """[nx,ny,nz,3] fp32 lattice points: origin + idx * spacing, product and sum rounded separately."""
    axes = [F32(origin[a]) + np.arange(shape[a]).astype(F32) * F32(spacing[a]) for a in range(3)]
    gi, gj, gk = np.meshgrid(*axes, indexing="ij")
    return np.stack([gi, gj, gk], -1).astype(F32)


def isosurface(values, origin, spacing, level=0.0):
    """-> verts [V,3] float32, faces [F,3] int64 (what nrt_isosurface_count + _emit produce)."""
    v = np.ascontiguousarray(values, F32)
    nx, ny, nz = v.shape
    level = F32(level)
    flat = v.reshape(-1)
    P = flat.size
    with np.errstate(invalid="ignore"):
        inside = (flat < level)
    idx = np.arange(P, dtype=np.int64)
    ii, jj, kk = idx // (ny * nz), (idx // nz) % ny, idx % nz
    step = lambda o: ((o & 1) * ny * nz) + (((o >> 1) & 1) * nz) + ((o >> 2) & 1)
    valid = lambda o: (ii + (o & 1) < nx) & (jj + ((o >> 1) & 1) < ny) & (kk + ((o >> 2) & 1) < nz)

    mask = np.zeros(P, np.int64)
    for d in range(1, 8):
        ok = valid(d)
        q = np.where(ok, idx + step(d), 0)
        mask |= ((ok & (inside != inside[q])).astype(np.int64) << (d - 1))
    popc = np.array([bin(m).count("1") for m in range(128)], np.int64)
    vcnt = popc[mask]
    vbase = np.concatenate([[0], np.cumsum(vcnt)[:-1]]).astype(np.int64)

    # vertices, ascending by (lower end, direction)
    pts = lattice_points((nx, ny, nz), origin, spacing).reshape(-1, 3)
    vp, vd = [], []
    for d in range(1, 8):
        sel = np.nonzero((mask >> (d - 1)) & 1)[0]
        vp.append(sel)
        vd.append(np.full(sel.size, d, np.int64))
    vp, vd = np.concatenate(vp), np.concatenate(vd)
    order = np.lexsort((vd, vp))
    vp, vd = vp[order], vd[order]
    qb = vp + np.array([step(d) for d in range(8)], np.int64)[vd]
    a, b = flat[vp], flat[qb]
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        t = ((level - a).astype(F32) / (b - a).astype(F32)).astype(F32)
        pa, pb = pts[vp], pts[qb]
        verts = (pa + t[:, None] * (pb - pa)).astype(F32)

    # faces, ascending by (cell, tetrahedron, triangle)
    table = tet_table()
    offs = tet_offsets()
    cell = valid(7)
    cells = idx[cell]
    cin = np.zeros(cells.size, np.int64)
    for o in range(8):
        cin |= inside[cells + step(o)].astype(np.int64) << o
    fc, fk, fv = [], [], []
    for t_ in range(6):
        case = np.zeros(cells.size, np.int64)
        for vtx in range(4):
            case |= ((cin >> offs[t_][vtx]) & 1) << vtx
        for c in range(16):
            tris = table[t_][c]
            if not tris:
                continue
            sel = cells[case == c]
            for n, tri in enumerate(tris):
                ids = []
                for code in tri:
                    o_lo, d = code & 7, code >> 3
                    q = sel + step(o_lo)
                    ids.append(vbase[q] + popc[mask[q] & ((1 << (d - 1)) - 1)])
                fc.append(sel)
                fk.append(np.full(sel.size, t_ * 2 + n, np.int64))
                fv.append(np.stack(ids, -1))
    if fc:
        fc, fk, fv = np.concatenate(fc), np.concatenate(fk), np.concatenate(fv)
        faces = fv[np.lexsort((fk, fc))].astype(np.int64)
    else:
        faces = np.zeros((0, 3), np.int64)
    return verts.reshape(-1, 3), faces.reshape(-1, 3)


def lattice_spacing(shape, bbox_min, bbox_max):
    """(origin, spacing) fp32 of the lattice: spacing = (bbox_max - bbox_min) / (n - 1) in float64, rounded once."""
    origin = np.asarray(bbox_min, np.float64).astype(F32)
    spacing = ((np.asarray(bbox_max, np.float64) - np.asarray(bbox_min, np.float64)) /
               (np.asarray(shape, np.float64) - 1)).astype(F32)
    return origin, spacing


# ---- mesh checks shared by the CPU and GPU tests -------------------------------------------------------------------
def edge_counts(faces):
    """(undirected edge -> count, directed edges unique?)."""
    f = np.asarray(faces, np.int64)
    de = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    directed_unique = np.unique(de, axis=0).shape[0] == de.shape[0]
    und = np.sort(de, axis=1)
    u, c = np.unique(und, axis=0, return_counts=True)
    return u, c, directed_unique


def signed_volume(verts, faces):
    v = np.asarray(verts, np.float64)
    f = np.asarray(faces, np.int64)
    return float(np.einsum("ij,ij->i", v[f[:, 0]], np.cross(v[f[:, 1]], v[f[:, 2]])).sum() / 6.0)
