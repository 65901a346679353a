// Triangle meshes from a scalar lattice: a SphereSDF evaluated on a lattice (nrt_sdf_lattice_eval) and the isosurface of
// any fp32 lattice by marching tetrahedra on its Freudenthal (Kuhn) triangulation (nrt_isosurface_count / _emit).
//
// Every cube of the lattice is cut into the 6 tetrahedra 0 -> e_a -> e_a + e_b -> (1,1,1), one per permutation (a,b,c)
// of the axes.  Each tetrahedron edge is a lattice edge from a point p to p + d, d one of the 7 nonzero {0,1}^3 offsets
// (bit 0 = +i, bit 1 = +j, bit 2 = +k), so a surface vertex is named by (p, d) and neighbouring cells agree on it: the
// mesh is indexed and closed by construction.  Point p owns the vertices of its crossing outgoing edges, numbered
// vbase[p] + popc(mask[p] & ((1 << (d - 1)) - 1)), and cell p (its lowest corner) owns its triangles from fbase[p].
// Both offsets are exclusive scans (CUB) of per-point counts.  The arithmetic is explicitly rounded fp32
// (__fmul_rn / __fadd_rn / __fsub_rn / __fdiv_rn), so tests/mesh_port.py reproduces the output bit for bit.
#include <cub/device/device_scan.cuh>
#include <cuda/std/functional>

#include <math.h>

#include "nrt_common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int64_t kLatticeChunk = int64_t(1) << 22;   // points per nrt_sdf_eval call of nrt_sdf_lattice_eval

// The triangles of one Kuhn tetrahedron per sign case (bit v of the case: corner v is inside).  A vertex is coded as
// o_lo | (d << 3): the crossing edge from corner offset o_lo in direction d.  Passed to the kernels by value.
struct IsoTable {
  uint8_t off[6][4];          // corner offsets of tetrahedron t (bit 0 = +i, bit 1 = +j, bit 2 = +k)
  uint8_t ntri[6][16];
  uint8_t code[6][16][2][3];
};

// Built with exact integer geometry: each triangle is oriented so that its normal, taken at the edge midpoints,
// points from the inside corners to the outside ones.  That orientation holds for every crossing parameter in (0, 1),
// so (v1 - v0) x (v2 - v0) points toward value >= level.
IsoTable build_table() {
  static const int perms[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};
  IsoTable tb;
  memset(&tb, 0, sizeof(tb));
  for (int t = 0; t < 6; ++t) {
    const int a = perms[t][0], b = perms[t][1];
    const int o[4] = {0, 1 << a, (1 << a) | (1 << b), 7};
    int P[4][3];
    for (int v = 0; v < 4; ++v)
      for (int c = 0; c < 3; ++c) {
        tb.off[t][v] = (uint8_t)o[v];
        P[v][c] = (o[v] >> c) & 1;
      }
    for (int cs = 0; cs < 16; ++cs) {
      int ins[4], outs[4], ni = 0, no = 0;
      for (int v = 0; v < 4; ++v) {
        if ((cs >> v) & 1) ins[ni++] = v;
        else outs[no++] = v;
      }
      if (ni == 0 || ni == 4) continue;
      int tris[2][3][2], nt;
      if (ni == 1 || ni == 3) {
        const int lone = ni == 1 ? ins[0] : outs[0];
        int k = 0;
        for (int v = 0; v < 4; ++v)
          if (v != lone) { tris[0][k][0] = lone; tris[0][k][1] = v; ++k; }
        nt = 1;
      } else {
        const int A = ins[0], B = ins[1], C = outs[0], D = outs[1];
        const int q[2][3][2] = {{{A, C}, {A, D}, {B, D}}, {{A, C}, {B, D}, {B, C}}};
        memcpy(tris, q, sizeof(q));
        nt = 2;
      }
      int g[3];
      for (int c = 0; c < 3; ++c) {
        int so = 0, si = 0;
        for (int k = 0; k < no; ++k) so += P[outs[k]][c];
        for (int k = 0; k < ni; ++k) si += P[ins[k]][c];
        g[c] = ni * so - no * si;
      }
      for (int n = 0; n < nt; ++n) {
        int m[3][3];
        for (int k = 0; k < 3; ++k)
          for (int c = 0; c < 3; ++c) m[k][c] = P[tris[n][k][0]][c] + P[tris[n][k][1]][c];
        const int u[3] = {m[1][0] - m[0][0], m[1][1] - m[0][1], m[1][2] - m[0][2]};
        const int w[3] = {m[2][0] - m[0][0], m[2][1] - m[0][1], m[2][2] - m[0][2]};
        const int nrm[3] = {u[1] * w[2] - u[2] * w[1], u[2] * w[0] - u[0] * w[2], u[0] * w[1] - u[1] * w[0]};
        const bool flip = nrm[0] * g[0] + nrm[1] * g[1] + nrm[2] * g[2] < 0;
        for (int k = 0; k < 3; ++k) {
          const int kk = flip ? (k == 0 ? 0 : 3 - k) : k;
          int lo = tris[n][kk][0], hi = tris[n][kk][1];
          if (lo > hi) { const int s = lo; lo = hi; hi = s; }   // path order: o[lo] is a subset of o[hi]
          tb.code[t][cs][n][k] = (uint8_t)(o[lo] | ((o[hi] ^ o[lo]) << 3));
        }
      }
      tb.ntri[t][cs] = (uint8_t)nt;
    }
  }
  return tb;
}

const IsoTable& table() {
  static const IsoTable tb = build_table();
  return tb;
}

struct Grid {
  int64_t nx, ny, nz, P;
  float o[3], s[3];
};

Grid grid_of(const nrt_lattice_t* g) {
  Grid r;
  r.nx = g->nx; r.ny = g->ny; r.nz = g->nz; r.P = g->nx * g->ny * g->nz;
  for (int c = 0; c < 3; ++c) { r.o[c] = g->origin[c]; r.s[c] = g->spacing[c]; }
  return r;
}

__device__ __forceinline__ int64_t step_of(const Grid& g, int o) {
  return (int64_t)(o & 1) * g.ny * g.nz + (int64_t)((o >> 1) & 1) * g.nz + ((o >> 2) & 1);
}

__device__ __forceinline__ float coord(const Grid& g, int c, int64_t i) {
  return __fadd_rn(g.o[c], __fmul_rn((float)i, g.s[c]));
}

// bit o of *cin: corner p + o is inside; bit o of the return value: that corner exists
__device__ __forceinline__ unsigned corners(const Grid& g, const float* __restrict__ v, float level, int64_t p, int64_t i,
                                            int64_t j, int64_t k, unsigned* cin) {
  unsigned valid = 0, in = 0;
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    if (i + (o & 1) < g.nx && j + ((o >> 1) & 1) < g.ny && k + ((o >> 2) & 1) < g.nz) {
      valid |= 1u << o;
      if (__ldg(v + p + step_of(g, o)) < level) in |= 1u << o;   // NaN compares false: outside
    }
  }
  *cin = in;
  return valid;
}

__device__ __forceinline__ unsigned tet_case(const IsoTable& tb, int t, unsigned cin) {
  return ((cin >> tb.off[t][0]) & 1) | (((cin >> tb.off[t][1]) & 1) << 1) | (((cin >> tb.off[t][2]) & 1) << 2) |
         (((cin >> tb.off[t][3]) & 1) << 3);
}

__global__ void k_lattice_points(Grid g, int64_t p0, int64_t n, float* __restrict__ out) {
  for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < n; x += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = p0 + x;
    const int64_t k = p % g.nz, r = p / g.nz, j = r % g.ny, i = r / g.ny;
    out[3 * x + 0] = coord(g, 0, i);
    out[3 * x + 1] = coord(g, 1, j);
    out[3 * x + 2] = coord(g, 2, k);
  }
}

// one thread per lattice point, consecutive threads along z: the crossing mask of its 7 outgoing edges, its vertex
// count and the triangle count of the cell whose lowest corner it is
__global__ void k_iso_count(Grid g, IsoTable tb, const float* __restrict__ v, float level, uint8_t* __restrict__ mask,
                            uint8_t* __restrict__ vcnt, uint8_t* __restrict__ fcnt) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < g.P; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = p % g.nz, r = p / g.nz, j = r % g.ny, i = r / g.ny;
    unsigned cin;
    const unsigned valid = corners(g, v, level, p, i, j, k, &cin);
    const unsigned own = cin & 1u;
    unsigned m = 0;
#pragma unroll
    for (int d = 1; d < 8; ++d)
      if (((valid >> d) & 1u) && ((cin >> d) & 1u) != own) m |= 1u << (d - 1);
    unsigned nf = 0;
    if (valid == 0xFFu) {
#pragma unroll
      for (int t = 0; t < 6; ++t) nf += tb.ntri[t][tet_case(tb, t, cin)];
    }
    mask[p] = (uint8_t)m;
    vcnt[p] = (uint8_t)__popc(m);
    fcnt[p] = (uint8_t)nf;
  }
}

__global__ void k_iso_totals(const uint8_t* __restrict__ vcnt, const uint8_t* __restrict__ fcnt,
                             const int64_t* __restrict__ vbase, const int64_t* __restrict__ fbase, int64_t P,
                             int64_t* __restrict__ counts) {
  counts[0] = vbase[P - 1] + vcnt[P - 1];
  counts[1] = fbase[P - 1] + fcnt[P - 1];
}

__device__ __forceinline__ int64_t vertex_id(const Grid& g, const uint8_t* __restrict__ mask,
                                             const int64_t* __restrict__ vbase, int64_t p, unsigned code) {
  const int64_t q = p + step_of(g, code & 7u);
  const unsigned d = code >> 3;
  return vbase[q] + __popc(mask[q] & ((1u << (d - 1)) - 1u));
}

// one thread per lattice point: its crossing vertices, then the triangles of its cell; nothing is written at or past
// max_vertices / max_faces
__global__ void k_iso_emit(Grid g, IsoTable tb, const float* __restrict__ v, float level,
                           const uint8_t* __restrict__ mask, const int64_t* __restrict__ vbase,
                           const int64_t* __restrict__ fbase, int64_t max_v, int64_t max_f, float* __restrict__ verts,
                           int64_t* __restrict__ faces) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < g.P; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t k = p % g.nz, r = p / g.nz, j = r % g.ny, i = r / g.ny;
    const unsigned m = mask[p];
    if (m) {
      const float a = __ldg(v + p);
      const float pa[3] = {coord(g, 0, i), coord(g, 1, j), coord(g, 2, k)};
      const int64_t vb = vbase[p];
      for (int d = 1; d < 8; ++d) {
        if (!((m >> (d - 1)) & 1u)) continue;
        const int64_t id = vb + __popc(m & ((1u << (d - 1)) - 1u));
        if (id >= max_v) break;
        const float b = __ldg(v + p + step_of(g, d));
        const float t = __fdiv_rn(__fsub_rn(level, a), __fsub_rn(b, a));
        const float pb[3] = {coord(g, 0, i + (d & 1)), coord(g, 1, j + ((d >> 1) & 1)), coord(g, 2, k + ((d >> 2) & 1))};
#pragma unroll
        for (int c = 0; c < 3; ++c) verts[3 * id + c] = __fadd_rn(pa[c], __fmul_rn(t, __fsub_rn(pb[c], pa[c])));
      }
    }
    if (i + 1 < g.nx && j + 1 < g.ny && k + 1 < g.nz) {
      unsigned cin;
      corners(g, v, level, p, i, j, k, &cin);
      int64_t f = fbase[p];
      for (int t = 0; t < 6 && f < max_f; ++t) {
        const unsigned cs = tet_case(tb, t, cin);
        for (int n = 0; n < tb.ntri[t][cs] && f < max_f; ++n, ++f) {
#pragma unroll
          for (int c = 0; c < 3; ++c) faces[3 * f + c] = vertex_id(g, mask, vbase, p, tb.code[t][cs][n][c]);
        }
      }
    }
  }
}

int grid_blocks(int64_t n) { return (int)std::min<int64_t>((n + kThreads - 1) / kThreads, (int64_t)nrt_sm_count() * 16); }

int check_lattice(const nrt_lattice_t* g, const char* who) {
  NRT_REQUIRE(g != nullptr, "%s: lattice is NULL", who);
  const int64_t n[3] = {g->nx, g->ny, g->nz};
  for (int c = 0; c < 3; ++c) {
    NRT_REQUIRE(n[c] >= 2 && n[c] <= NRT_MAX_LATTICE_DIM, "%s: lattice dimension %d is %lld, must be in [2, %d]", who, c,
                (long long)n[c], NRT_MAX_LATTICE_DIM);
    NRT_REQUIRE(isfinite(g->spacing[c]) && g->spacing[c] > 0.0f, "%s: lattice spacing %d is %g, must be finite and > 0",
                who, c, (double)g->spacing[c]);
    NRT_REQUIRE(isfinite(g->origin[c]), "%s: lattice origin %d is not finite", who, c);
  }
  return NRT_OK;
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// workspace of the extraction: mask, vcnt, fcnt (1 byte each), vbase, fbase (int64 each), then CUB's scan storage
struct IsoWs {
  uint8_t *mask, *vcnt, *fcnt;
  int64_t *vbase, *fbase;
  void* temp;
  size_t temp_bytes, total;
};

int scan_temp_bytes(int64_t P, size_t* out) {
  size_t b = 0;
  NRT_CUDA(cub::DeviceScan::ExclusiveScan(nullptr, b, (const uint8_t*)nullptr, (int64_t*)nullptr,
                                          cuda::std::plus<int64_t>(), (int64_t)0, P, (cudaStream_t)0));
  *out = b;
  return NRT_OK;
}

int iso_layout(int64_t P, void* base, IsoWs* w) {
  int rc = scan_temp_bytes(P, &w->temp_bytes);
  if (rc != NRT_OK) return rc;
  char* b = (char*)base;
  size_t off = 0;
  w->mask = (uint8_t*)(b + off); off += align256(P);
  w->vcnt = (uint8_t*)(b + off); off += align256(P);
  w->fcnt = (uint8_t*)(b + off); off += align256(P);
  w->vbase = (int64_t*)(b + off); off += align256(8 * (size_t)P);
  w->fbase = (int64_t*)(b + off); off += align256(8 * (size_t)P);
  w->temp = b + off; off += align256(w->temp_bytes);
  w->total = off;
  return NRT_OK;
}

}  // namespace

extern "C" int64_t nrt_sdf_lattice_eval_workspace(const nrt_lattice_t* g) {
  int rc = check_lattice(g, "nrt_sdf_lattice_eval_workspace");
  if (rc != NRT_OK) return rc;
  return (int64_t)align256(12 * (size_t)std::min<int64_t>(grid_of(g).P, kLatticeChunk));
}

extern "C" int nrt_sdf_lattice_eval(const nrt_sphere_sdf_t* s, int prec, const nrt_lattice_t* g, float* values, void* ws,
                                    size_t ws_bytes, void* stream) {
  int rc = check_lattice(g, "nrt_sdf_lattice_eval");
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(values != nullptr && ws != nullptr, "nrt_sdf_lattice_eval: null values/workspace");
  const Grid gd = grid_of(g);
  const int64_t chunk = std::min<int64_t>(gd.P, kLatticeChunk);
  NRT_REQUIRE(ws_bytes >= 12 * (size_t)chunk, "nrt_sdf_lattice_eval: workspace of %zu bytes, needs %zu", ws_bytes,
              12 * (size_t)chunk);
  cudaStream_t st = (cudaStream_t)stream;
  float* pts = (float*)ws;
  for (int64_t p0 = 0; p0 < gd.P; p0 += chunk) {
    const int64_t n = std::min<int64_t>(chunk, gd.P - p0);
    {
      NrtProfScope _ps(TAG_LATTICE_POINTS, st);
      k_lattice_points<<<grid_blocks(n), kThreads, 0, st>>>(gd, p0, n, pts);
    }
    NRT_CUDA(cudaGetLastError());
    rc = nrt_sdf_eval(s, prec, pts, n, values + p0, stream);
    if (rc != NRT_OK) return rc;
  }
  return NRT_OK;
}

extern "C" int64_t nrt_isosurface_workspace(const nrt_lattice_t* g) {
  int rc = check_lattice(g, "nrt_isosurface_workspace");
  if (rc != NRT_OK) return rc;
  IsoWs w;
  rc = iso_layout(grid_of(g).P, nullptr, &w);
  if (rc != NRT_OK) return rc;
  return (int64_t)w.total;
}

static int iso_begin(const nrt_lattice_t* g, const float* values, float level, void* ws, size_t ws_bytes, const char* who,
                     Grid* gd, IsoWs* w) {
  int rc = check_lattice(g, who);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(isfinite(level), "%s: level is not finite", who);
  NRT_REQUIRE(values != nullptr && ws != nullptr, "%s: null values/workspace", who);
  NRT_REQUIRE(((uintptr_t)ws & 255) == 0, "%s: workspace must be 256-byte aligned", who);
  *gd = grid_of(g);
  rc = iso_layout(gd->P, ws, w);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(ws_bytes >= w->total, "%s: workspace of %zu bytes, needs %zu (nrt_isosurface_workspace)", who, ws_bytes,
              w->total);
  return NRT_OK;
}

extern "C" int nrt_isosurface_count(const nrt_lattice_t* g, const float* values, float level, void* ws, size_t ws_bytes,
                                    int64_t* counts_dev, void* stream) {
  Grid gd;
  IsoWs w;
  int rc = iso_begin(g, values, level, ws, ws_bytes, "nrt_isosurface_count", &gd, &w);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(counts_dev != nullptr, "nrt_isosurface_count: null counts");
  cudaStream_t st = (cudaStream_t)stream;
  {
    NrtProfScope _ps(TAG_ISO_COUNT, st);
    k_iso_count<<<grid_blocks(gd.P), kThreads, 0, st>>>(gd, table(), values, level, w.mask, w.vcnt, w.fcnt);
  }
  NRT_CUDA(cudaGetLastError());
  {
    NrtProfScope _ps(TAG_ISO_SCAN, st);
    size_t tb = w.temp_bytes;
    NRT_CUDA(cub::DeviceScan::ExclusiveScan(w.temp, tb, (const uint8_t*)w.vcnt, w.vbase, cuda::std::plus<int64_t>(),
                                            (int64_t)0, gd.P, st));
    tb = w.temp_bytes;
    NRT_CUDA(cub::DeviceScan::ExclusiveScan(w.temp, tb, (const uint8_t*)w.fcnt, w.fbase, cuda::std::plus<int64_t>(),
                                            (int64_t)0, gd.P, st));
    k_iso_totals<<<1, 1, 0, st>>>(w.vcnt, w.fcnt, w.vbase, w.fbase, gd.P, counts_dev);
  }
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

extern "C" int nrt_isosurface_emit(const nrt_lattice_t* g, const float* values, float level, void* ws, size_t ws_bytes,
                                   int64_t max_vertices, int64_t max_faces, float* verts, int64_t* faces, void* stream) {
  Grid gd;
  IsoWs w;
  int rc = iso_begin(g, values, level, ws, ws_bytes, "nrt_isosurface_emit", &gd, &w);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(max_vertices >= 0 && max_faces >= 0, "nrt_isosurface_emit: negative capacity");
  NRT_REQUIRE(max_vertices == 0 || verts != nullptr, "nrt_isosurface_emit: null verts");
  NRT_REQUIRE(max_faces == 0 || faces != nullptr, "nrt_isosurface_emit: null faces");
  cudaStream_t st = (cudaStream_t)stream;
  {
    NrtProfScope _ps(TAG_ISO_EMIT, st);
    k_iso_emit<<<grid_blocks(gd.P), kThreads, 0, st>>>(gd, table(), values, level, w.mask, w.vbase, w.fbase,
                                                        max_vertices, max_faces, verts, faces);
  }
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}
