// nrt_nerfle_render: orchestration of the volumetric render (single pass, or
// coarse -> importance resample -> fine -> merged compositing), plus the HBM-bound
// sampling / compositing kernels of the hierarchical path.
#include <algorithm>
#include <stdlib.h>

#include "nrt_common.cuh"

int nrt_nerfle_pass_f32(const nrt_mlp_t* first, const nrt_mlp_t* second, const float* rays, int64_t R,
                        const float* ts, const float* ts_per_ray, int S, const float* light_code,
                        int light_dim, const int32_t* view_of_ray, int second_out_act, float* out_rgb,
                        float* out_sigma, float* out_srgb, cudaStream_t st);
int nrt_nerfle_pass_tc(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                       const float* ts, const float* ts_per_ray, int S, const float* light_code,
                       int light_dim, const int32_t* view_of_ray, int second_out_act, float* out_rgb,
                       float* out_sigma, float* out_srgb, void* workspace, size_t workspace_bytes,
                       cudaStream_t st, const nrt_camera_t* cam = nullptr, int64_t cam_r0 = 0);
bool nrt_nerfle_pass_tc_camera_ok(const nrt_mlp_t* first, const nrt_mlp_t* second, int light_dim);
size_t nrt_nerfle_pass_tc_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int64_t R, int S);

static int nerf_pass(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                     const float* ts, const float* ts_per_ray, int S, const float* light_code, int light_dim,
                     const int32_t* view_of_ray, float* out_rgb, float* out_sigma, float* out_srgb,
                     void* ws, size_t ws_bytes, cudaStream_t st, const nrt_camera_t* cam = nullptr, int64_t cam_r0 = 0) {
  if (prec == NRT_PREC_F32)
    return nrt_nerfle_pass_f32(first, second, rays, R, ts, ts_per_ray, S, light_code, light_dim, view_of_ray,
                               NRT_OUT_SIGMOID, out_rgb, out_sigma, out_srgb, st);
  return nrt_nerfle_pass_tc(first, second, prec, rays, R, ts, ts_per_ray, S, light_code, light_dim, view_of_ray,
                            NRT_OUT_SIGMOID, out_rgb, out_sigma, out_srgb, ws, ws_bytes, st, cam, cam_r0);
}

// Where a camera-driven frame gets its rays (SURVEY f4).  Mode 0 (default): k_camera_rays generates each chunk's rays into the
// workspace (24 B per ray) right before the chunk's first pass.  Mode 1 (nrt_set_camera_rays_mode(1), or NRT_CAMERA_RAYS=fused
// in the environment): the two tensor-core kernels compute the ray of every sample in their per-sample prologues from the
// camera (IoNerfFirst / IoNerfSecond with CAM; bit-identical rays, no ray array at all).  Measured on B200, cfg2 frame from the
// camera, alternating runs on one box: 53.6 / 54.1 / 53.9 ms (mode 0) against 54.8 / 55.8 / 55.1 ms (mode 1) -- recomputing a ray
// 64-192 times per ray in kernels whose epilogue warps are bound by the instructions they issue costs 2.5-3 %, to save 24 B of
// the 27 KB of per-ray traffic; hence mode 0 (profiles/r02i_camera_fused.md).
#include <atomic>
static std::atomic<int> g_camera_mode{-1};
static bool camera_fused_default() {
  int m = g_camera_mode.load(std::memory_order_relaxed);
  if (m < 0) {
    const char* e = getenv("NRT_CAMERA_RAYS");
    m = (e && e[0] == 'f') ? 1 : 0;
    g_camera_mode.store(m, std::memory_order_relaxed);
  }
  return m == 1;
}
extern "C" int nrt_set_camera_rays_mode(int fused) {
  NRT_REQUIRE(fused == 0 || fused == 1, "nrt_set_camera_rays_mode: 0 (prologue kernel) or 1 (inside the MLP kernels)");
  g_camera_mode.store(fused, std::memory_order_relaxed);
  return NRT_OK;
}

// ---- stratified sample distances -------------------------------------------------------------
// ts[r][s] = near + (s + u)/S * (far-near), u = hash(seed, r, s) in [0,1)  (extension; the
// reference uses the same ts for every ray, nerf.py:178).
// (32-bit arithmetic: the 64-bit splitmix of round 1 cost ~25 integer instructions per sample in kernels that should
//  be HBM-bound; oracle/port.py restates the same recipe)
__device__ __forceinline__ float hash_u01(uint64_t seed, uint64_t a, uint64_t b) {
  uint32_t h = (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x9E3779B1u);
  h = (h ^ (uint32_t)a) * 0x85EBCA77u;
  h = (h ^ (uint32_t)b) * 0xC2B2AE3Du;
  h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
  return (float)(h >> 8) * (1.0f / 16777216.0f);
}

// four consecutive samples of one ray per thread (S % 4 == 0: one 16-byte store per thread, coalesced), else one.
// seed_dev (training under CUDA graphs, nrt_nerfle_sample_hierarchical): when not NULL the seed is read from device memory
// instead of the by-value `seed`, so that a captured launch draws new jitter whenever the caller advances it.
template <int V>
__global__ void k_stratified_ts(int64_t R, int64_t r_off, int S, float t_near, float t_far, uint64_t seed,
                                const uint64_t* __restrict__ seed_dev, float* __restrict__ ts) {
  if (seed_dev) seed = *seed_dev;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int SV = S / V;
  if (i >= R * SV) return;
  const int64_t r = i / SV;
  const int s0 = (int)(i - r * SV) * V;
  const float span = t_far - t_near;
  float t[V];
#pragma unroll
  for (int k = 0; k < V; ++k) {
    const float u = seed ? hash_u01(seed, (uint64_t)(r + r_off), (uint64_t)(s0 + k)) : 0.5f;
    t[k] = t_near + ((float)(s0 + k) + u) / (float)S * span;
  }
  if (V == 4) *reinterpret_cast<float4*>(ts + r * S + s0) = make_float4(t[0], t[1], t[2], t[3]);
  else ts[r * S + s0] = t[0];
}

// ---- importance resampling (standard NeRF sample_pdf, inverse CDF over the coarse bins) ----------
// One WARP per ray (HBM-bound: 8 B per coarse sample read, 4 B per fine sample written, both coalesced): every lane
// owns a contiguous run of coarse samples; transmittance = exclusive warp-scan product, cdf = inclusive warp-scan sum
// (weights from the coarse pass with the reference's compositing formula, interior samples 1..Sc-2 as in NeRF), then
// lane j, j+32, ... binary-search the cdf in shared memory and write the fine distances.
constexpr int kPdfWarps = 4;
// exp of the compositing weights: the exact fp32 path uses the deterministic nrt_expf of nrt_detmath.h like every other
// fp32 kernel (and like the C oracle's restatement); the 16-bit path uses the SFU approximation
template <bool EXACT> __device__ __forceinline__ float exp_w(float x) { return EXACT ? nrt_expf(x) : __expf(x); }
template <bool EXACT>
__global__ void __launch_bounds__(kPdfWarps * 32)
k_sample_pdf(const float* __restrict__ sigma_c, const float* __restrict__ ts_c_shared,
             const float* __restrict__ ts_c_per_ray, int Sc, int Sf, int64_t R, int64_t r_off,
             uint64_t seed, const uint64_t* __restrict__ seed_dev, float* __restrict__ ts_f) {
  extern __shared__ float sm[];
  if (seed_dev) seed = *seed_dev;       // as in k_stratified_ts
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_t = sm + (size_t)wid * 3 * Sc;
  float* s_cdf = s_t + Sc;     // inclusive cdf over the interior samples (index = sample)
  float* s_pdf = s_cdf + Sc;
  const int per = (Sc + 31) / 32;
  for (int64_t r = (int64_t)blockIdx.x * kPdfWarps + wid; r < R; r += (int64_t)gridDim.x * kPdfWarps) {
    const float* sig = sigma_c + r * Sc;
    const float* tc = ts_c_per_ray ? ts_c_per_ray + r * Sc : ts_c_shared;
    const int e0 = lane * per, e1 = min(Sc, e0 + per);
    // alpha and the local transmittance product of this lane's run
    float prod = 1.0f;
    for (int e = e0; e < e1; ++e) {
      const float t = tc[e];
      s_t[e] = t;
      const float a = 1.0f - exp_w<EXACT>(-fmaxf(sig[e], 0.0f) * t);
      s_pdf[e] = a;                                  // alpha for now
      prod *= fmaxf(1.0f - a, 1e-10f);
    }
    float incl = prod;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl *= v;
    }
    float cp = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) cp = 1.0f;
    // un-normalised weights of the interior samples and their local sum
    float wsum = 0.0f;
    for (int e = e0; e < e1; ++e) {
      const float a = s_pdf[e];
      const float w = (e >= 1 && e <= Sc - 2) ? a * cp + 1e-5f : 0.0f;
      s_pdf[e] = w;
      wsum += w;
      cp *= fmaxf(1.0f - a, 1e-10f);
    }
    float run = wsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_up_sync(0xffffffffu, run, o);
      if (lane >= o) run += v;
    }
    const float total = __shfl_sync(0xffffffffu, run, 31);
    float c = run - wsum;                            // exclusive prefix of this lane's run
    const float inv = 1.0f / total;
    for (int e = e0; e < e1; ++e) {
      const float p = s_pdf[e] * inv;
      c += s_pdf[e];
      s_pdf[e] = p;
      s_cdf[e] = c * inv;
    }
    __syncwarp();
    float* out = ts_f + r * Sf;
    if (Sf == 128) {
      // four CONSECUTIVE fine samples per lane: u ascends, so one binary search and a linear advance find the bins, and
      // the lane writes one 16-byte vector (the strided form below spends 6 search iterations per sample and writes
      // 4-byte words; ncu round 1: issue slots 76 % busy, 10 % of the DRAM bandwidth).  1 / 128 is a power of two: the
      // multiplication equals the division bit for bit.
      float t4[4];
      int sidx = 1;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int j = 4 * lane + k;
        const float jit = seed ? hash_u01(seed ^ 0x5bd1e995u, (uint64_t)(r + r_off), (uint64_t)j) : 0.5f;
        const float u = ((float)j + jit) * (1.0f / 128.0f);
        if (k == 0) {
          int lo = 1, hi = Sc - 2;
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (u > s_cdf[mid]) lo = mid + 1; else hi = mid;
          }
          sidx = lo;
        } else {
          while (sidx < Sc - 2 && u > s_cdf[sidx]) ++sidx;
        }
        const float p = s_pdf[sidx];
        const float num = u - (s_cdf[sidx] - p);
        const float f = fminf(fmaxf(EXACT ? num / p : __fdividef(num, p), 0.0f), 1.0f);
        const float tl = 0.5f * (s_t[sidx - 1] + s_t[sidx]);
        const float th = 0.5f * (s_t[sidx] + s_t[sidx + 1]);
        t4[k] = tl + f * (th - tl);
      }
      *reinterpret_cast<float4*>(out + 4 * lane) = make_float4(t4[0], t4[1], t4[2], t4[3]);
      __syncwarp();
      continue;
    }
    for (int j = lane; j < Sf; j += 32) {
      const float jit = seed ? hash_u01(seed ^ 0x5bd1e995u, (uint64_t)(r + r_off), (uint64_t)j) : 0.5f;
      const float u = ((float)j + jit) / (float)Sf;
      // first interior sample s in [1, Sc-2] with u <= cdf[s]; the last one otherwise
      int lo = 1, hi = Sc - 2;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (u > s_cdf[mid]) lo = mid + 1; else hi = mid;
      }
      const int sidx = lo;
      const float p = s_pdf[sidx];
      const float f = fminf(fmaxf((u - (s_cdf[sidx] - p)) / p, 0.0f), 1.0f);
      const float tl = 0.5f * (s_t[sidx - 1] + s_t[sidx]);
      const float th = 0.5f * (s_t[sidx] + s_t[sidx + 1]);
      out[j] = tl + f * (th - tl);
    }
    __syncwarp();
  }
}

// ---- merged compositing over coarse + fine samples (both sorted by t), ray-major ----------
// Reads 16 B/sample (sigma + rgb) + 4 B/sample (t), writes 12 B/ray.  One warp per ray: lanes
// merge by rank, then the transmittance product is a warp scan.
template <bool EXACT>
__global__ void k_merge_composite(const float* __restrict__ sig_c, const float* __restrict__ rgb_c,
                                  const float* __restrict__ ts_c_shared, const float* __restrict__ ts_c_per_ray,
                                  int Sc, const float* __restrict__ sig_f, const float* __restrict__ rgb_f,
                                  const float* __restrict__ ts_f, int Sf, int64_t R, float* __restrict__ out) {
  extern __shared__ float sm[];
  const int warps = blockDim.x >> 5;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = Sc + Sf;
  // per warp: the two sorted distance lists (searched below: in shared memory, not through dependent global loads --
  // ncu of the round-1 kernel: long_scoreboard 12.2 warps per issue), then alpha and rgb in merged order
  float* s_tc = sm + (size_t)wid * 5 * S;
  float* s_tf = s_tc + Sc;
  float* m_a = s_tc + S;
  float* m_rgb = m_a + S;
  const int64_t r = (int64_t)blockIdx.x * warps + wid;
  if (r >= R) return;
  const float* tc = ts_c_per_ray ? ts_c_per_ray + r * Sc : ts_c_shared;
  const float* tf = Sf > 0 ? ts_f + r * Sf : nullptr;
  for (int i = lane; i < Sc; i += 32) s_tc[i] = tc[i];
  for (int j = lane; j < Sf; j += 32) s_tf[j] = tf[j];
  __syncwarp();
  // rank of each element in the merged order: coarse element i goes to i + #(fine < tc[i]),
  // fine element j to j + #(coarse <= tf[j])  (stable: coarse first on ties); alpha is computed once, here
  for (int i = lane; i < Sc; i += 32) {
    const float t = s_tc[i];
    int lo = 0, hi = Sf;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_tf[mid] < t) lo = mid + 1; else hi = mid; }
    const int p = i + lo;
    m_a[p] = 1.0f - exp_w<EXACT>(-fmaxf(sig_c[r * Sc + i], 0.0f) * t);
    m_rgb[p * 3] = rgb_c[(r * Sc + i) * 3]; m_rgb[p * 3 + 1] = rgb_c[(r * Sc + i) * 3 + 1];
    m_rgb[p * 3 + 2] = rgb_c[(r * Sc + i) * 3 + 2];
  }
  for (int j = lane; j < Sf; j += 32) {
    const float t = s_tf[j];
    int lo = 0, hi = Sc;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_tc[mid] <= t) lo = mid + 1; else hi = mid; }
    const int p = j + lo;
    m_a[p] = 1.0f - exp_w<EXACT>(-fmaxf(sig_f[r * Sf + j], 0.0f) * t);
    m_rgb[p * 3] = rgb_f[(r * Sf + j) * 3]; m_rgb[p * 3 + 1] = rgb_f[(r * Sf + j) * 3 + 1];
    m_rgb[p * 3 + 2] = rgb_f[(r * Sf + j) * 3 + 2];
  }
  __syncwarp();
  // each lane owns a contiguous run of samples; local product, then an exclusive warp scan
  const int per = (S + 31) / 32;
  const int s0 = lane * per, s1 = min(S, s0 + per);
  float prod = 1.0f;
  for (int s = s0; s < s1; ++s) prod *= fmaxf(1.0f - m_a[s], 1e-10f);
  float incl = prod;
  for (int o = 1; o < 32; o <<= 1) {
    const float v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl *= v;
  }
  float excl = __shfl_up_sync(0xffffffffu, incl, 1);
  if (lane == 0) excl = 1.0f;
  const float total = __shfl_sync(0xffffffffu, incl, 31);
  float cp = excl, acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;
  for (int s = s0; s < s1; ++s) {
    const float a = m_a[s];
    float w;
    if (s == 0) w = a * (S == 1 ? 1.0f : total);   // roll quirk: sample 0 gets the total product
    else if (s == S - 1) w = a;                      // last transmittance forced to 1
    else w = a * cp;
    acc0 += w * m_rgb[s * 3]; acc1 += w * m_rgb[s * 3 + 1]; acc2 += w * m_rgb[s * 3 + 2];
    cp *= fmaxf(1.0f - a, 1e-10f);
  }
  for (int o = 16; o > 0; o >>= 1) {
    acc0 += __shfl_down_sync(0xffffffffu, acc0, o);
    acc1 += __shfl_down_sync(0xffffffffu, acc1, o);
    acc2 += __shfl_down_sync(0xffffffffu, acc2, o);
  }
  if (lane == 0) { out[r * 3] = acc0; out[r * 3 + 1] = acc1; out[r * 3 + 2] = acc2; }
}

// ---- merged distances only (training: nrt_nerfle_sample_hierarchical), written SAMPLE-major ----------
// The same ranks as k_merge_composite (coarse first on ties), one warp per ray, but the output is ts_out [S, R_out] with
// m = s * R_out + ray, the layout of the training kernels.  A block merges kMergeTsRays rays into a shared-memory tile
// [S][kMergeTsRays + 1] and then writes every sample row as kMergeTsRays consecutive floats (coalesced across rays).  The
// padding column makes the row-wise reads of the write-out conflict-free; the per-ray column writes hit rows i + rank,
// which can be 32 apart within one warp instruction and then share a bank (rare, a few extra cycles).  With Sf = 0 the
// kernel is the transpose of the stratified distances.  Reads 4 B + writes 4 B per sample.
constexpr int kMergeTsWarps = 8, kMergeTsRays = 32;
static size_t merge_ts_smem(int S) { return ((size_t)S * (kMergeTsRays + 1) + (size_t)kMergeTsWarps * S) * sizeof(float); }
__global__ void __launch_bounds__(kMergeTsWarps * 32)
k_merge_ts(const float* __restrict__ ts_c, int Sc, const float* __restrict__ ts_f, int Sf, int64_t n, int64_t R_out,
           int64_t r_off, float* __restrict__ ts_out) {
  extern __shared__ float sm[];
  const int S = Sc + Sf;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int LD = kMergeTsRays + 1;
  float* s_out = sm;
  float* s_tc = sm + (size_t)S * LD + (size_t)wid * S;
  float* s_tf = s_tc + Sc;
  const int64_t rb = (int64_t)blockIdx.x * kMergeTsRays;
  for (int k = wid; k < kMergeTsRays; k += kMergeTsWarps) {
    const int64_t r = rb + k;
    if (r >= n) break;
    for (int i = lane; i < Sc; i += 32) s_tc[i] = ts_c[r * Sc + i];
    for (int j = lane; j < Sf; j += 32) s_tf[j] = ts_f[r * Sf + j];
    __syncwarp();
    for (int i = lane; i < Sc; i += 32) {
      const float t = s_tc[i];
      int lo = 0, hi = Sf;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_tf[mid] < t) lo = mid + 1; else hi = mid; }
      s_out[(i + lo) * LD + k] = t;
    }
    for (int j = lane; j < Sf; j += 32) {
      const float t = s_tf[j];
      int lo = 0, hi = Sc;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_tc[mid] <= t) lo = mid + 1; else hi = mid; }
      s_out[(j + lo) * LD + k] = t;
    }
    __syncwarp();
  }
  __syncthreads();
  const int nr = (int)min((int64_t)kMergeTsRays, n - rb);
  for (int e = threadIdx.x; e < S * kMergeTsRays; e += blockDim.x) {
    const int s = e / kMergeTsRays, k = e - s * kMergeTsRays;
    if (k < nr) ts_out[(int64_t)s * R_out + r_off + rb + k] = s_out[s * LD + k];
  }
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// the two sampling launches shared by the render and by nrt_nerfle_sample_hierarchical (seed_dev NULL: sampling->jitter_seed)
static int launch_stratified(int64_t n, int64_t r0, int Sc, const nrt_nerf_sampling_t* sampling, const uint64_t* seed_dev,
                             float* ts_c, cudaStream_t st) {
  NrtProfScope _ps(TAG_STRATIFIED_TS, st);
  if (Sc % 4 == 0)
    k_stratified_ts<4><<<nrt_cdiv(n * (Sc / 4), 256), 256, 0, st>>>(n, r0, Sc, sampling->t_near, sampling->t_far,
                                                                   sampling->jitter_seed, seed_dev, ts_c);
  else
    k_stratified_ts<1><<<nrt_cdiv(n * Sc, 256), 256, 0, st>>>(n, r0, Sc, sampling->t_near, sampling->t_far,
                                                             sampling->jitter_seed, seed_dev, ts_c);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

static int launch_sample_pdf(int prec, const float* sig_c, const float* ts_shared, const float* ts_pr, int Sc, int Sf,
                             int64_t n, int64_t r0, uint64_t seed, const uint64_t* seed_dev, float* ts_f, cudaStream_t st) {
  { NrtProfScope _ps(TAG_SAMPLE_PDF, st);
  const int grid = (int)std::min<int64_t>((n + kPdfWarps - 1) / kPdfWarps, (int64_t)nrt_sm_count() * 16);
  if (prec == NRT_PREC_F32)
    k_sample_pdf<true><<<grid, kPdfWarps * 32, (size_t)kPdfWarps * 3 * Sc * sizeof(float), st>>>(
        sig_c, ts_shared, ts_pr, Sc, Sf, n, r0, seed, seed_dev, ts_f);
  else
    k_sample_pdf<false><<<grid, kPdfWarps * 32, (size_t)kPdfWarps * 3 * Sc * sizeof(float), st>>>(
        sig_c, ts_shared, ts_pr, Sc, Sf, n, r0, seed, seed_dev, ts_f); }
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

// rays are rendered in chunks of this many so that the scratch (per-sample sigma / rgb / latent: ~150 B x 192 per ray)
// stays a few GB regardless of the image size (65,536-ray chunks measured 2 % slower: 3.3x the launches)
static const int64_t kRayChunk = 262144;
static size_t cam_scratch_bytes(int64_t C) { return align256((size_t)C * 24) + align256((size_t)C * 4); }

extern "C" size_t nrt_nerfle_render_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                              int64_t R, const nrt_nerf_sampling_t* sampling) {
  const int64_t C = std::min<int64_t>(R, kRayChunk);
  size_t total = 256;
  const int Sc = sampling ? sampling->n_coarse : 64, Sf = sampling ? sampling->n_fine : 0;
  const bool jitter = sampling && sampling->jitter_seed != 0;
  const bool store_c = Sf > 0 || prec != NRT_PREC_F32;    // the tensor-core pass always stores per-sample values
  total += align256((size_t)C * Sc * 4);                                              // ts_c per ray (jitter / no ts)
  (void)jitter;
  if (store_c) total += align256((size_t)C * Sc * 4) + align256((size_t)C * Sc * 12);  // sigma_c, rgb_c
  if (Sf > 0) total += align256((size_t)C * Sf * 4) * 2 + align256((size_t)C * Sf * 12);  // ts_f, sigma_f, rgb_f
  if (prec != NRT_PREC_F32) total += align256(nrt_nerfle_pass_tc_workspace(first, second, C, std::max(Sc, Sf)));
  return total;
}

int nrt_check_camera(const nrt_camera_t* cam, int64_t* total);
int nrt_camera_rays_dev(const nrt_camera_t* cam, int64_t r0, int64_t n, float* out_rays, int32_t* out_view,
                        cudaStream_t st);

// the render of R rays given either as an array (rays) or as a camera (cam: every chunk's rays are generated into the
// tail of the workspace right before its first pass; SURVEY f4).
// Per-sample mode (nrt_nerfle_render_samples): smp_sigma [R,Sc] / smp_rgb [R,Sc,3] not NULL, n_fine = 0 -- every chunk's
// pass stores its per-sample values there instead of the workspace and nothing is composited; ts_per_ray [R,Sc], when not
// NULL, gives every ray its own distances in place of ts / the stratified ones.
static int render_impl(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                       const nrt_camera_t* cam, int64_t R, const float* ts, const nrt_nerf_sampling_t* sampling,
                       const float* light_code, int light_dim, const int32_t* view_of_ray,
                       float* out_rgb, void* workspace, size_t workspace_bytes, cudaStream_t st,
                       const float* ts_per_ray = nullptr, float* smp_sigma = nullptr, float* smp_rgb = nullptr) {
  NRT_REQUIRE(R >= 0, "nrt_nerfle_render: negative R");
  if (R == 0) return NRT_OK;
  const bool samples = smp_sigma != nullptr;
  NRT_REQUIRE((rays != nullptr || cam != nullptr) && (out_rgb != nullptr || (samples && smp_rgb != nullptr)),
              "nrt_nerfle_render: null rays/out");
  NRT_REQUIRE(sampling != nullptr, "nrt_nerfle_render: sampling descriptor is NULL");
  const int Sc = sampling->n_coarse, Sf = sampling->n_fine;
  const bool jitter = sampling->jitter_seed != 0;
  NRT_REQUIRE(Sc >= 1 && Sf >= 0, "nrt_nerfle_render: bad sample counts %d/%d", Sc, Sf);
  NRT_REQUIRE(ts != nullptr || ts_per_ray != nullptr || sampling->t_far > sampling->t_near,
              "nrt_nerfle_render: need ts or t_near<t_far");
  NRT_REQUIRE(!samples || Sf == 0, "nrt_nerfle_render: per-sample outputs of a single pass only");
  NRT_REQUIRE(Sf == 0 || Sc >= 3, "hierarchical sampling needs n_coarse >= 3");
  const int64_t C = std::min<int64_t>(R, kRayChunk);
  const size_t need = nrt_nerfle_render_workspace(first, second, prec, R, sampling) + (cam ? cam_scratch_bytes(C) : 0);
  NRT_REQUIRE(workspace != nullptr && workspace_bytes >= need,
              "nrt_nerfle_render: workspace of %zu bytes required, got %zu", need, workspace_bytes);
  float* cam_rays = nullptr; int32_t* cam_view = nullptr;
  const bool fused = cam && prec != NRT_PREC_F32 && camera_fused_default() &&
                     nrt_nerfle_pass_tc_camera_ok(first, second, light_dim);
  if (cam) {
    char* tail = (char*)workspace + (need - cam_scratch_bytes(C));
    cam_rays = (float*)tail;
    if (cam->n_views > 1) cam_view = (int32_t*)(tail + align256((size_t)C * 24));
  }
  char* wp = (char*)workspace;
  auto take = [&](size_t bytes) { char* p = wp; wp += align256(bytes); return (void*)p; };
  const bool store_c = Sf > 0 || prec != NRT_PREC_F32;
  float* ts_c = (float*)take((size_t)C * Sc * 4);
  float *sig_c = nullptr, *rgb_c = nullptr, *ts_f = nullptr, *sig_f = nullptr, *rgb_f = nullptr;
  if (store_c) { sig_c = (float*)take((size_t)C * Sc * 4); rgb_c = (float*)take((size_t)C * Sc * 12); }
  if (Sf > 0) {
    ts_f = (float*)take((size_t)C * Sf * 4); sig_f = (float*)take((size_t)C * Sf * 4);
    rgb_f = (float*)take((size_t)C * Sf * 12);
  }
  void* tcws = nullptr; size_t tcws_bytes = 0;
  if (prec != NRT_PREC_F32) {
    tcws_bytes = nrt_nerfle_pass_tc_workspace(first, second, C, std::max(Sc, Sf));
    tcws = take(tcws_bytes);
  }
  const int warps = 4;
  const size_t merge_smem = (size_t)warps * 5 * (Sc + Sf) * sizeof(float);
  NRT_REQUIRE(merge_smem <= 48 * 1024, "too many samples per ray for the merge kernel");

  for (int64_t r0 = 0; r0 < R; r0 += C) {
    const int64_t n = std::min<int64_t>(C, R - r0);
    const float* c_rays = cam ? cam_rays : rays + r0 * 6;
    const int32_t* c_view = cam ? cam_view : view_of_ray ? view_of_ray + r0 : nullptr;
    // camera-fed kernels: the tensor-core pass computes the rays itself, nothing to generate
    const nrt_camera_t* kcam = (cam && fused) ? cam : nullptr;
    if (cam && !fused) {
      const int rcc = nrt_camera_rays_dev(cam, r0, n, cam_rays, cam_view, st);
      if (rcc != NRT_OK) return rcc;
    }
    float* c_out = samples ? nullptr : out_rgb + r0 * 3;
    const float* ts_shared = ts;
    const float* ts_pr = nullptr;
    if (ts_per_ray) {
      ts_shared = nullptr; ts_pr = ts_per_ray + r0 * Sc;
    } else if (jitter || ts == nullptr) {
      // per-ray (stratified) distances; without jitter this is the bin-centre grid
      const int rs = launch_stratified(n, r0, Sc, sampling, nullptr, ts_c, st);
      if (rs != NRT_OK) return rs;
      ts_shared = nullptr; ts_pr = ts_c;
    }
    int rc;
    if (samples) {
      rc = nerf_pass(first, second, prec, c_rays, n, ts_shared, ts_pr, Sc, light_code, light_dim, c_view, nullptr,
                     smp_sigma + r0 * Sc, smp_rgb + r0 * Sc * 3, tcws, tcws_bytes, st, kcam, r0);
      if (rc != NRT_OK) return rc;
      continue;
    }
    if (!store_c) {
      rc = nerf_pass(first, second, prec, c_rays, n, ts_shared, ts_pr, Sc, light_code, light_dim, c_view, c_out,
                     nullptr, nullptr, tcws, tcws_bytes, st, kcam, r0);
      if (rc != NRT_OK) return rc;
      continue;
    }
    // coarse pass keeps per-sample sigma / rgb
    rc = nerf_pass(first, second, prec, c_rays, n, ts_shared, ts_pr, Sc, light_code, light_dim, c_view, nullptr,
                   sig_c, rgb_c, tcws, tcws_bytes, st, kcam, r0);
    if (rc != NRT_OK) return rc;
    if (Sf > 0) {
      rc = launch_sample_pdf(prec, sig_c, ts_shared, ts_pr, Sc, Sf, n, r0, sampling->jitter_seed, nullptr, ts_f, st);
      if (rc != NRT_OK) return rc;
      rc = nerf_pass(first, second, prec, c_rays, n, nullptr, ts_f, Sf, light_code, light_dim, c_view, nullptr,
                     sig_f, rgb_f, tcws, tcws_bytes, st, kcam, r0);
      if (rc != NRT_OK) return rc;
    }
    { NrtProfScope _ps(TAG_MERGE_COMPOSITE, st);
    if (prec == NRT_PREC_F32)
      k_merge_composite<true><<<nrt_cdiv(n, warps), warps * 32, merge_smem, st>>>(sig_c, rgb_c, ts_shared, ts_pr, Sc, sig_f,
                                                                                  rgb_f, ts_f, Sf, n, c_out);
    else
      k_merge_composite<false><<<nrt_cdiv(n, warps), warps * 32, merge_smem, st>>>(sig_c, rgb_c, ts_shared, ts_pr, Sc, sig_f,
                                                                                   rgb_f, ts_f, Sf, n, c_out); }
    NRT_CUDA(cudaGetLastError());
  }
  return NRT_OK;
}

extern "C" int nrt_nerfle_render(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                                 int64_t R, const float* ts, const nrt_nerf_sampling_t* sampling,
                                 const float* light_code, int light_dim, const int32_t* view_of_ray,
                                 float* out_rgb, void* workspace, size_t workspace_bytes, void* stream) {
  NRT_REQUIRE(R <= 0 || rays != nullptr, "nrt_nerfle_render: null rays");
  return render_impl(first, second, prec, rays, nullptr, R, ts, sampling, light_code, light_dim, view_of_ray, out_rgb,
                     workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- hierarchical sample distances for training (extension of nerf.py:178, see nrt_b200.h) -----------------------
// The first half of render_impl: stratified coarse distances, the coarse pass keeping per-sample sigma, k_sample_pdf;
// then k_merge_ts writes the merged ascending distances sample-major.  n_fine = 0 is the render's single stratified pass:
// no coarse pass, the stratified distances are written sample-major as they are.  Chunked like the render, jitter hashed
// with the global ray index, so the distances are those the render composites over (same prec, same seed).
extern "C" size_t nrt_nerfle_sample_hierarchical_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                                           int64_t R, const nrt_nerf_sampling_t* sampling) {
  if (sampling == nullptr || R < 0) return 0;
  const int64_t C = std::min<int64_t>(R, kRayChunk);
  const int Sc = sampling->n_coarse, Sf = sampling->n_fine;
  size_t total = 256 + align256((size_t)C * Sc * 4);
  if (Sf == 0) return total;
  total += align256((size_t)C * Sc * 4) + align256((size_t)C * Sc * 12) + align256((size_t)C * Sf * 4);
  if (prec != NRT_PREC_F32) total += align256(nrt_nerfle_pass_tc_workspace(first, second, C, Sc));
  return total;
}

extern "C" int nrt_nerfle_sample_hierarchical(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                                              int64_t R, const nrt_nerf_sampling_t* sampling, const uint64_t* seed_dev,
                                              const float* light_code, int light_dim, const int32_t* view_of_ray,
                                              float* ts_out, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  NRT_REQUIRE(R >= 0, "nrt_nerfle_sample_hierarchical: negative R");
  NRT_REQUIRE(sampling != nullptr, "nrt_nerfle_sample_hierarchical: sampling descriptor is NULL");
  const int Sc = sampling->n_coarse, Sf = sampling->n_fine;
  NRT_REQUIRE(Sc >= 1 && Sf >= 0, "nrt_nerfle_sample_hierarchical: bad sample counts %d/%d", Sc, Sf);
  NRT_REQUIRE(Sf == 0 || Sc >= 3, "nrt_nerfle_sample_hierarchical: hierarchical sampling needs n_coarse >= 3");
  NRT_REQUIRE(Sc + Sf <= NRT_MAX_HIER_SAMPLES, "nrt_nerfle_sample_hierarchical: n_coarse + n_fine = %d exceeds %d",
              Sc + Sf, NRT_MAX_HIER_SAMPLES);
  NRT_REQUIRE(sampling->t_far > sampling->t_near, "nrt_nerfle_sample_hierarchical: needs t_near < t_far");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(rays != nullptr && ts_out != nullptr, "nrt_nerfle_sample_hierarchical: null rays/ts_out");
  const int64_t C = std::min<int64_t>(R, kRayChunk);
  const size_t need = nrt_nerfle_sample_hierarchical_workspace(first, second, prec, R, sampling);
  NRT_REQUIRE(workspace != nullptr && workspace_bytes >= need,
              "nrt_nerfle_sample_hierarchical: workspace of %zu bytes required, got %zu", need, workspace_bytes);
  char* wp = (char*)workspace;
  auto take = [&](size_t bytes) { char* p = wp; wp += align256(bytes); return (void*)p; };
  float* ts_c = (float*)take((size_t)C * Sc * 4);
  float *sig_c = nullptr, *rgb_c = nullptr, *ts_f = nullptr;
  if (Sf > 0) {
    sig_c = (float*)take((size_t)C * Sc * 4);
    rgb_c = (float*)take((size_t)C * Sc * 12);
    ts_f = (float*)take((size_t)C * Sf * 4);
  }
  void* tcws = nullptr; size_t tcws_bytes = 0;
  if (Sf > 0 && prec != NRT_PREC_F32) {
    tcws_bytes = nrt_nerfle_pass_tc_workspace(first, second, C, Sc);
    tcws = take(tcws_bytes);
  }
  const size_t msmem = merge_ts_smem(Sc + Sf);
  NRT_CUDA(cudaFuncSetAttribute(k_merge_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
  for (int64_t r0 = 0; r0 < R; r0 += C) {
    const int64_t n = std::min<int64_t>(C, R - r0);
    const int32_t* c_view = view_of_ray ? view_of_ray + r0 : nullptr;
    int rc = launch_stratified(n, r0, Sc, sampling, seed_dev, ts_c, st);
    if (rc != NRT_OK) return rc;
    if (Sf > 0) {
      rc = nerf_pass(first, second, prec, rays + r0 * 6, n, nullptr, ts_c, Sc, light_code, light_dim, c_view, nullptr,
                     sig_c, rgb_c, tcws, tcws_bytes, st);
      if (rc != NRT_OK) return rc;
      rc = launch_sample_pdf(prec, sig_c, nullptr, ts_c, Sc, Sf, n, r0, sampling->jitter_seed, seed_dev, ts_f, st);
      if (rc != NRT_OK) return rc;
    }
    { NrtProfScope _ps(TAG_MERGE_TS, st);
    k_merge_ts<<<nrt_cdiv(n, kMergeTsRays), kMergeTsWarps * 32, msmem, st>>>(ts_c, Sc, ts_f, Sf, n, R, r0, ts_out); }
    NRT_CUDA(cudaGetLastError());
  }
  return NRT_OK;
}

// ---- f4: the frame from a camera (main.py:57-88 for a volumetric shape as one call) ------------------------------
extern "C" size_t nrt_nerfle_render_camera_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                                     const nrt_camera_t* cam, const nrt_nerf_sampling_t* sampling) {
  int64_t R = 0;
  if (nrt_check_camera(cam, &R) != NRT_OK) return 0;
  return nrt_nerfle_render_workspace(first, second, prec, R, sampling) + cam_scratch_bytes(std::min<int64_t>(R, kRayChunk));
}

extern "C" int nrt_nerfle_render_camera(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                        const nrt_camera_t* cam, const float* ts, const nrt_nerf_sampling_t* sampling,
                                        const float* light_code, int light_dim, float* out_rgb, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  int64_t R = 0;
  const int rc = nrt_check_camera(cam, &R);
  if (rc != NRT_OK) return rc;
  return render_impl(first, second, prec, nullptr, cam, R, ts, sampling, light_code, light_dim, nullptr, out_rgb,
                     workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- the render's pass with its per-sample values as the output (what k_merge_composite would composite) ----------
extern "C" size_t nrt_nerfle_render_samples_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                                      int64_t R, int S, const nrt_camera_t* cam) {
  if (R < 0 || S < 1) return 0;
  const nrt_nerf_sampling_t samp{S, 0, 0.0f, 0.0f, 0};
  return nrt_nerfle_render_workspace(first, second, prec, R, &samp) +
         (cam ? cam_scratch_bytes(std::min<int64_t>(R, kRayChunk)) : 0);
}

extern "C" int nrt_nerfle_render_samples(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                                         const nrt_camera_t* cam, int64_t R, const float* ts, const float* ts_per_ray,
                                         int S, const float* light_code, int light_dim, const int32_t* view_of_ray,
                                         float* out_sigma, float* out_rgb, void* workspace, size_t workspace_bytes,
                                         void* stream) {
  NRT_REQUIRE(R >= 0, "nrt_nerfle_render_samples: negative R");
  NRT_REQUIRE((rays != nullptr) != (cam != nullptr), "nrt_nerfle_render_samples: exactly one of rays / cam must be given");
  if (cam) {
    int64_t Rc = 0;
    const int rc = nrt_check_camera(cam, &Rc);
    if (rc != NRT_OK) return rc;
    NRT_REQUIRE(R == Rc, "nrt_nerfle_render_samples: R = %lld but the camera has %lld rays", (long long)R, (long long)Rc);
    NRT_REQUIRE(view_of_ray == nullptr, "nrt_nerfle_render_samples: a camera gives every ray its view; view_of_ray must be NULL");
  }
  NRT_REQUIRE(S >= 1, "nrt_nerfle_render_samples: bad sample count %d", S);
  NRT_REQUIRE((ts != nullptr) != (ts_per_ray != nullptr), "nrt_nerfle_render_samples: exactly one of ts / ts_per_ray must be given");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(out_sigma != nullptr && out_rgb != nullptr, "nrt_nerfle_render_samples: null out_sigma/out_rgb");
  const nrt_nerf_sampling_t samp{S, 0, 0.0f, 0.0f, 0};
  return render_impl(first, second, prec, rays, cam, R, ts, &samp, light_code, light_dim, view_of_ray, nullptr, workspace,
                     workspace_bytes, (cudaStream_t)stream, ts_per_ray, out_sigma, out_rgb);
}

// The host-buffer entry point keeps grow-only device scratch PER DEVICE (a stream-ordered pool would hand the memory
// back at every synchronisation and re-allocate >1 GB per call); calls on the same device are serialised by the
// record's host_mu, calls on different devices are independent.
#include <mutex>
extern "C" int nrt_nerfle_render_host(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                      const float* rays_host, int64_t R, const float* ts_host, int S,
                                      const nrt_nerf_sampling_t* sampling, const float* light_code,
                                      int light_dim, float* out_rgb_host, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  NRT_REQUIRE(rays_host && out_rgb_host && sampling, "nrt_nerfle_render_host: bad arguments");
  NRT_REQUIRE(R >= 0, "nrt_nerfle_render_host: negative R");
  if (R == 0) return NRT_OK;
  void *d_rays = nullptr, *d_ts = nullptr, *d_out = nullptr, *ws = nullptr;
  NrtDeviceState* ds = nrt_device_state();
  NRT_REQUIRE(ds != nullptr, "nrt_nerfle_render_host: no current CUDA device");
  std::lock_guard<std::mutex> host_lock(ds->host_mu);
  const size_t wsb = nrt_nerfle_render_workspace(first, second, prec, R, sampling);
  int rc = nrt_host_scratch(ds, 0, (size_t)R * 24, &d_rays); if (rc != NRT_OK) return rc;
  rc = nrt_host_scratch(ds, 1, (size_t)R * 12, &d_out); if (rc != NRT_OK) return rc;
  rc = nrt_host_scratch(ds, 2, wsb, &ws); if (rc != NRT_OK) return rc;
  if (ts_host) {
    rc = nrt_host_scratch(ds, 3, (size_t)S * 4, &d_ts); if (rc != NRT_OK) return rc;
    NRT_CUDA(cudaMemcpyAsync(d_ts, ts_host, (size_t)S * 4, cudaMemcpyHostToDevice, st));
  }
  NRT_CUDA(cudaMemcpyAsync(d_rays, rays_host, (size_t)R * 24, cudaMemcpyHostToDevice, st));
  rc = nrt_nerfle_render(first, second, prec, (const float*)d_rays, R, (const float*)d_ts, sampling, light_code, light_dim,
                         nullptr, (float*)d_out, ws, wsb, st);
  if (rc != NRT_OK) return rc;
  NRT_CUDA(cudaMemcpyAsync(out_rgb_host, d_out, (size_t)R * 12, cudaMemcpyDeviceToHost, st));
  NRT_CUDA(cudaStreamSynchronize(st));
  return NRT_OK;
}

extern "C" int nrt_nerfle_render_camera_host(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                             const nrt_camera_t* cam, const float* ts_host, int S,
                                             const nrt_nerf_sampling_t* sampling, const float* light_code,
                                             int light_dim, float* out_rgb_host, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  NRT_REQUIRE(out_rgb_host && sampling, "nrt_nerfle_render_camera_host: bad arguments");
  int64_t R = 0;
  int rc = nrt_check_camera(cam, &R);
  if (rc != NRT_OK) return rc;
  if (R == 0) return NRT_OK;
  void *d_ts = nullptr, *d_out = nullptr, *ws = nullptr;
  NrtDeviceState* ds = nrt_device_state();
  NRT_REQUIRE(ds != nullptr, "nrt_nerfle_render_camera_host: no current CUDA device");
  std::lock_guard<std::mutex> host_lock(ds->host_mu);
  const size_t wsb = nrt_nerfle_render_camera_workspace(first, second, prec, cam, sampling);
  rc = nrt_host_scratch(ds, 1, (size_t)R * 12, &d_out); if (rc != NRT_OK) return rc;
  rc = nrt_host_scratch(ds, 2, wsb, &ws); if (rc != NRT_OK) return rc;
  if (ts_host) {
    rc = nrt_host_scratch(ds, 3, (size_t)S * 4, &d_ts); if (rc != NRT_OK) return rc;
    NRT_CUDA(cudaMemcpyAsync(d_ts, ts_host, (size_t)S * 4, cudaMemcpyHostToDevice, st));
  }
  rc = render_impl(first, second, prec, nullptr, cam, R, (const float*)d_ts, sampling, light_code, light_dim, nullptr,
                   (float*)d_out, ws, wsb, st);
  if (rc != NRT_OK) return rc;
  NRT_CUDA(cudaMemcpyAsync(out_rgb_host, d_out, (size_t)R * 12, cudaMemcpyDeviceToHost, st));
  NRT_CUDA(cudaStreamSynchronize(st));
  return NRT_OK;
}
