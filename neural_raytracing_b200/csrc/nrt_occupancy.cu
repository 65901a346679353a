// Occupancy grid of a NeRFLE density network (nrt_occupancy_t, include/nrt_b200.h): the update (points kernel -> the plain
// forward of `first` -> one reduce kernel), the cull decision (k_occupancy_mask), and the cull + compaction that the
// gradient-free render runs in front of both tensor-core MLPs (k_occupancy_cull + CUB DeviceSelect::Flagged, called from
// render_impl in nrt_render.cu).
#include <algorithm>
#include <cmath>

#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "nrt_common.cuh"

int nrt_nerfle_pass_tc_keep(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                            const float* ts, const float* ts_per_ray, int S, const float* light_code, int light_dim,
                            const int32_t* view_of_ray, const int32_t* keep, const int32_t* rows, float* out_sigma,
                            float* out_srgb, void* workspace, size_t workspace_bytes, cudaStream_t st);

namespace {

constexpr int kThreads = 256;
size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
int blocks_for(int64_t n) { return (int)std::min<int64_t>((n + kThreads - 1) / kThreads, (int64_t)nrt_sm_count() * 32); }

// the grid as the kernels read it: inv[a] = res / (hi - lo) and h[a] = (hi - lo) / res, each computed in double and
// rounded to float once
struct OccDev {
  int res;
  float lo[3], inv[3], h[3];
  const uint32_t* bits;
};

int occ_dev(const nrt_occupancy_t* g, OccDev* d, bool need_bits, const char* who) {
  NRT_REQUIRE(g != nullptr, "%s: occupancy grid descriptor is NULL", who);
  NRT_REQUIRE(g->res >= NRT_OCC_MIN_RES && g->res <= NRT_OCC_MAX_RES, "%s: resolution %d outside [%d, %d]", who, g->res,
              NRT_OCC_MIN_RES, NRT_OCC_MAX_RES);
  for (int a = 0; a < 3; ++a) {
    NRT_REQUIRE(std::isfinite(g->bbox_min[a]) && std::isfinite(g->bbox_max[a]) && g->bbox_max[a] > g->bbox_min[a],
                "%s: the box must be finite with bbox_max > bbox_min (axis %d: [%g, %g])", who, a, (double)g->bbox_min[a],
                (double)g->bbox_max[a]);
    const double span = (double)g->bbox_max[a] - (double)g->bbox_min[a];
    d->lo[a] = g->bbox_min[a];
    d->inv[a] = (float)((double)g->res / span);
    d->h[a] = (float)(span / (double)g->res);
  }
  NRT_REQUIRE(!need_bits || g->bits != nullptr, "%s: grid bits are NULL", who);
  d->res = g->res;
  d->bits = g->bits;
  return NRT_OK;
}

// The cull decision of one sample: p = o + t d with the expression of IoNerfFirst::point (nrt_tc.cu; both translation
// units contract it the same way), cell = floor((p - lo) * inv) per axis.  A sample is culled iff every axis lands in
// [0, res) and the cell's bit is clear; outside the box and non-finite points (the comparisons fail) are kept.
__device__ __forceinline__ bool occ_culled(const OccDev& g, const float* __restrict__ ray, float t) {
  const float o[3] = {__ldg(ray), __ldg(ray + 1), __ldg(ray + 2)};
  const float d[3] = {__ldg(ray + 3), __ldg(ray + 4), __ldg(ray + 5)};
  const float p[3] = {o[0] + t * d[0], o[1] + t * d[1], o[2] + t * d[2]};
  uint32_t c[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float u = (p[a] - g.lo[a]) * g.inv[a];
    if (!(u >= 0.0f && u < (float)g.res)) return false;
    c[a] = (uint32_t)u;
  }
  const uint32_t cell = (c[0] * (uint32_t)g.res + c[1]) * (uint32_t)g.res + c[2];
  return ((__ldg(g.bits + (cell >> 5)) >> (cell & 31)) & 1u) == 0;
}

__device__ __forceinline__ float sample_t(const float* ts, const float* ts_pr, int64_t i, int s) {
  return ts_pr ? __ldg(ts_pr + i) : __ldg(ts + s);
}

// one chunk's n * S samples (m = ray * S + s): culled samples get sigma = 0 and rgb = 0 in their slots (what the render's
// compositing reads), every sample a keep flag for the compaction
__global__ void k_occupancy_cull(OccDev g, const float* __restrict__ rays, int64_t n, const float* __restrict__ ts,
                                 const float* __restrict__ ts_pr, int S, float* __restrict__ sigma, float* __restrict__ rgb,
                                 uint8_t* __restrict__ flags) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n * S; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / S;
    const int s = (int)(i - r * S);
    const bool cull = occ_culled(g, rays + r * 6, sample_t(ts, ts_pr, i, s));
    if (cull) {
      sigma[i] = 0.0f;
      rgb[3 * i] = 0.0f; rgb[3 * i + 1] = 0.0f; rgb[3 * i + 2] = 0.0f;
    }
    flags[i] = cull ? 0 : 1;
  }
}

__global__ void k_occupancy_count(const int32_t* __restrict__ rows, unsigned long long* __restrict__ samples_done) {
  atomicAdd(samples_done, (unsigned long long)*rows);
}

__global__ void k_occupancy_mask(OccDev g, const float* __restrict__ rays, int64_t R, const float* __restrict__ ts,
                                 const float* __restrict__ ts_pr, int S, uint8_t* __restrict__ keep) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < R * S; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / S;
    const int s = (int)(i - r * S);
    keep[i] = occ_culled(g, rays + r * 6, sample_t(ts, ts_pr, i, s)) ? 0 : 1;
  }
}

// update points: point q of cell c = (i, j, k) at lo + (idx + u) * h per axis, each operation rounded (no contraction);
// u = hash_u01(seed, c, 3 q + axis), or 0.5 (the cell centre) with seed 0
__global__ void k_occupancy_points(OccDev g, uint64_t seed, int ppc, int64_t c0, int64_t n_pts, float* __restrict__ pts) {
  for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < n_pts; x += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = c0 + x / ppc;
    const int q = (int)(x % ppc);
    const int64_t idx[3] = {c / ((int64_t)g.res * g.res), (c / g.res) % g.res, c % g.res};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float u = seed ? hash_u01(seed, (uint64_t)c, (uint64_t)(3 * q + a)) : 0.5f;
      pts[3 * x + a] = __fadd_rn(g.lo[a], __fmul_rn(__fadd_rn((float)idx[a], u), g.h[a]));
    }
  }
}

// density[c] = max(decay * density[c], max_q relu(sigma_raw(q))), then bit c = density[c] > threshold.  c0 is a multiple
// of 32 and every warp covers 32 consecutive cells: one ballot per bit word.
__global__ void k_occupancy_reduce(const float* __restrict__ out, int out_stride, int ppc, int64_t c0, int64_t n_cells,
                                   float decay, float threshold, float* __restrict__ density, uint32_t* __restrict__ bits) {
  const int64_t span = (n_cells + 31) / 32 * 32;
  for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < span; x += (int64_t)gridDim.x * blockDim.x) {
    const bool valid = x < n_cells;
    bool occ = false;
    if (valid) {
      float m = 0.0f;
      for (int q = 0; q < ppc; ++q) m = fmaxf(m, __ldg(out + (x * ppc + q) * out_stride));
      const float d = fmaxf(__fmul_rn(decay, density[c0 + x]), m);
      density[c0 + x] = d;
      occ = d > threshold;
    }
    const unsigned word = __ballot_sync(0xffffffffu, occ);
    if ((threadIdx.x & 31) == 0 && valid) bits[(c0 + x) >> 5] = word;
  }
}

constexpr int64_t kOccChunkPts = 1 << 19;   // update points per chunk: 6 MB of points, 136 MB of NeRFLE.first outputs
int64_t cells_per_chunk(int ppc) { return std::max<int64_t>(32, kOccChunkPts / ppc / 32 * 32); }

int select_temp_bytes(int64_t items, size_t* out) {
  size_t b = 0;
  NRT_CUDA(cub::DeviceSelect::Flagged(nullptr, b, cub::CountingInputIterator<int32_t>(0), (const uint8_t*)nullptr,
                                      (int32_t*)nullptr, (int32_t*)nullptr, (int)items, (cudaStream_t)0));
  *out = b;
  return NRT_OK;
}

}  // namespace

// ---- update ---------------------------------------------------------------------------------------------------------
extern "C" size_t nrt_occupancy_update_workspace(const nrt_mlp_t* first, int prec, int32_t res, int points_per_cell) {
  if (first == nullptr || res < NRT_OCC_MIN_RES || res > NRT_OCC_MAX_RES || points_per_cell < 1 ||
      points_per_cell > NRT_OCC_MAX_POINTS_PER_CELL)
    return 0;
  (void)prec;
  const int64_t cells = (int64_t)res * res * res;
  const int64_t pts = std::min<int64_t>(cells, cells_per_chunk(points_per_cell)) * points_per_cell;
  return align256((size_t)pts * 12) + align256((size_t)pts * first->out_size * 4);
}

extern "C" int nrt_occupancy_update(const nrt_mlp_t* first, int prec, const nrt_occupancy_t* grid, int points_per_cell,
                                    float decay, float threshold, uint64_t seed, float* density, uint32_t* bits_out,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  OccDev g;
  int rc = occ_dev(grid, &g, false, "nrt_occupancy_update");
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(first != nullptr, "nrt_occupancy_update: mlp descriptor is NULL");
  NRT_REQUIRE(points_per_cell >= 1 && points_per_cell <= NRT_OCC_MAX_POINTS_PER_CELL,
              "nrt_occupancy_update: points_per_cell = %d outside [1, %d]", points_per_cell, NRT_OCC_MAX_POINTS_PER_CELL);
  NRT_REQUIRE(decay >= 0.0f && decay <= 1.0f, "nrt_occupancy_update: decay = %g outside [0, 1]", (double)decay);
  NRT_REQUIRE(threshold >= 0.0f && std::isfinite(threshold), "nrt_occupancy_update: threshold = %g must be finite and >= 0",
              (double)threshold);
  NRT_REQUIRE(first->in_size == 3 && first->latent_size == 0 && first->out_size >= 1,
              "nrt_occupancy_update: `first` must map 3-D points to (sigma_raw, ...) without a latent input");
  NRT_REQUIRE(density != nullptr && bits_out != nullptr, "nrt_occupancy_update: null density/bits");
  const size_t need = nrt_occupancy_update_workspace(first, prec, grid->res, points_per_cell);
  NRT_REQUIRE(workspace != nullptr && workspace_bytes >= need,
              "nrt_occupancy_update: workspace of %zu bytes required, got %zu", need, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t cells = (int64_t)g.res * g.res * g.res;
  const int64_t chunk = std::min<int64_t>(cells, cells_per_chunk(points_per_cell));
  float* pts = (float*)workspace;
  float* out = (float*)((char*)workspace + align256((size_t)chunk * points_per_cell * 12));
  for (int64_t c0 = 0; c0 < cells; c0 += chunk) {
    const int64_t nc = std::min<int64_t>(chunk, cells - c0);
    const int64_t np = nc * points_per_cell;
    {
      NrtProfScope _ps(TAG_OCCUPANCY_UPDATE, st);
      k_occupancy_points<<<blocks_for(np), kThreads, 0, st>>>(g, seed, points_per_cell, c0, np, pts);
    }
    NRT_CUDA(cudaGetLastError());
    rc = nrt_mlp_forward(first, prec, NRT_OUT_NONE, pts, nullptr, np, out, nullptr, stream);
    if (rc != NRT_OK) return rc;
    {
      NrtProfScope _ps(TAG_OCCUPANCY_UPDATE, st);
      k_occupancy_reduce<<<blocks_for((nc + 31) / 32 * 32), kThreads, 0, st>>>(out, first->out_size, points_per_cell, c0, nc,
                                                                              decay, threshold, density, bits_out);
    }
    NRT_CUDA(cudaGetLastError());
  }
  return NRT_OK;
}

// ---- the cull decision alone ------------------------------------------------------------------------------------------
extern "C" int nrt_occupancy_mask(const nrt_occupancy_t* grid, const float* rays, int64_t R, const float* ts,
                                  const float* ts_per_ray, int S, uint8_t* keep, void* stream) {
  OccDev g;
  int rc = occ_dev(grid, &g, true, "nrt_occupancy_mask");
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(R >= 0 && S >= 1, "nrt_occupancy_mask: bad R = %lld / S = %d", (long long)R, S);
  NRT_REQUIRE((ts != nullptr) != (ts_per_ray != nullptr), "nrt_occupancy_mask: exactly one of ts / ts_per_ray must be given");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(rays != nullptr && keep != nullptr, "nrt_occupancy_mask: null rays/keep");
  cudaStream_t st = (cudaStream_t)stream;
  {
    NrtProfScope _ps(TAG_OCCUPANCY_CULL, st);
    k_occupancy_mask<<<blocks_for(R * S), kThreads, 0, st>>>(g, rays, R, ts, ts_per_ray, S, keep);
  }
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

// ---- the culled pass of render_impl ------------------------------------------------------------------------------------
// scratch per chunk (C rays, S = the larger pass's sample count): keep flags (1 B / sample), keep list (4 B / sample), the
// device count, CUB's selection storage
size_t nrt_occupancy_pass_workspace(int64_t C, int S) {
  size_t temp = 0;
  if (select_temp_bytes(C * S, &temp) != NRT_OK) return 0;
  return align256((size_t)C * S) + align256((size_t)C * S * 4) + align256(4) + align256(temp);
}

int nrt_occupancy_pass(const nrt_occupancy_t* grid, unsigned long long* samples_done, const nrt_mlp_t* first,
                       const nrt_mlp_t* second, int prec, const float* rays, int64_t n, const float* ts,
                       const float* ts_per_ray, int S, const float* light_code, int light_dim, const int32_t* view_of_ray,
                       float* out_sigma, float* out_srgb, void* tcws, size_t tcws_bytes, void* occws, size_t occws_bytes,
                       cudaStream_t st) {
  OccDev g;
  int rc = occ_dev(grid, &g, true, "nrt_nerfle_render_occupancy");
  if (rc != NRT_OK) return rc;
  const int64_t items = n * S;
  NRT_REQUIRE(items <= 0x7fffffff, "nrt_nerfle_render_occupancy: %lld samples in one chunk", (long long)items);
  size_t temp = 0;
  rc = select_temp_bytes(items, &temp);
  if (rc != NRT_OK) return rc;
  char* wp = (char*)occws;
  uint8_t* flags = (uint8_t*)wp; wp += align256((size_t)items);
  int32_t* keep = (int32_t*)wp; wp += align256((size_t)items * 4);
  int32_t* rows = (int32_t*)wp; wp += align256(4);
  NRT_REQUIRE((size_t)(wp - (char*)occws) + temp <= occws_bytes, "nrt_nerfle_render_occupancy: occupancy scratch too small");
  {
    NrtProfScope _ps(TAG_OCCUPANCY_CULL, st);
    k_occupancy_cull<<<blocks_for(items), kThreads, 0, st>>>(g, rays, n, ts, ts_per_ray, S, out_sigma, out_srgb, flags);
    NRT_CUDA(cudaGetLastError());
    NRT_CUDA(cub::DeviceSelect::Flagged(wp, temp, cub::CountingInputIterator<int32_t>(0), flags, keep, rows, (int)items, st));
    if (samples_done) k_occupancy_count<<<1, 1, 0, st>>>(rows, samples_done);
    NRT_CUDA(cudaGetLastError());
  }
  return nrt_nerfle_pass_tc_keep(first, second, prec, rays, n, ts, ts_per_ray, S, light_code, light_dim, view_of_ray, keep,
                                 rows, out_sigma, out_srgb, tcws, tcws_bytes, st);
}
