// fp32 "exact" kernels of libnrt_b200: fused SkipConnMLP forward, SphereSDF evaluation,
// persistent sphere-trace march with slot compaction, shadow march, min-along-ray scan and the
// fused NeRFLE volumetric render.  Compiled with -fmad=false: every fused multiply-add is an
// explicit nrt_fma so the arithmetic matches oracle/c/nrt_oracle.c bit for bit.
#include <algorithm>

#include "mlp_tile_f32.cuh"

namespace nrt {

// ------------------------------------------------------------------------------------------
// a2: SkipConnMLP.forward on materialised inputs (neural_blocks.py:75-86)
// ------------------------------------------------------------------------------------------
template <int H, int TM>
__global__ void __launch_bounds__(kThreads, 1)
k_mlp_fwd(MlpDev m, const float* __restrict__ x, const float* __restrict__ latent, int64_t M,
          float* __restrict__ out, float* __restrict__ acts, int out_act) {
  extern __shared__ __align__(16) float smem[];
  TileSmem s;
  carve_tile(s, smem, m.dim_p, H, m.out, TM);
  const int64_t ntiles = (M + TM - 1) / TM;
  const int lat0 = m.in_size + 2 * m.freqs;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t mb = tile * TM;
    const int valid = (int)min((int64_t)TM, M - mb);
    for (int idx = threadIdx.x; idx < TM * m.in_size; idx += kThreads) {
      const int mm = idx / m.in_size, j = idx - mm * m.in_size;
      s.enc_raw[j * TM + mm] = (mm < valid) ? x[(mb + mm) * m.in_size + j] : 0.0f;
    }
    for (int idx = threadIdx.x; idx < TM * m.latent; idx += kThreads) {
      const int mm = idx / m.latent, j = idx - mm * m.latent;
      s.enc_raw[(lat0 + j) * TM + mm] = (mm < valid) ? latent[(mb + mm) * m.latent + j] : 0.0f;
    }
    __syncthreads();
    mlp_tile_forward<H, TM>(m, s, acts, M, mb, valid);
    for (int idx = threadIdx.x; idx < TM * m.out; idx += kThreads) {
      const int mm = idx / m.out, n = idx - mm * m.out;
      if (mm < valid) out[(mb + mm) * m.out + n] = out_act_apply(out_act, s.outb[n * TM + mm]);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// a3: SphereSDF (sdfs.py:37-46) -- smooth-min of warped spheres, one thread per sample,
// spheres visited in index order (the order the oracle sums exp(-k*sd) in).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float sphere_set_smin(const SdfDev& sd, float px, float py, float pz) {
  float sum = 0.0f;
  for (int i = 0; i < sd.n; ++i) {
    const float* T = sd.tfs + i * 9;
    float q[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      // (tfs + I) applied to p, einsum "ijk,ibk->ibj" (sdfs.py:39-40)
      const float t0 = __ldg(T + j * 3 + 0) + (j == 0 ? 1.0f : 0.0f);
      const float t1 = __ldg(T + j * 3 + 1) + (j == 1 ? 1.0f : 0.0f);
      const float t2 = __ldg(T + j * 3 + 2) + (j == 2 ? 1.0f : 0.0f);
      float a = t0 * px;
      a = nrt_fma(t1, py, a);
      a = nrt_fma(t2, pz, a);
      q[j] = a - __ldg(sd.centers + i * 3 + j);
    }
    float n2 = q[0] * q[0];
    n2 = nrt_fma(q[1], q[1], n2);
    n2 = nrt_fma(q[2], q[2], n2);
    const float d = sqrtf(n2) - __ldg(sd.radii + i);
    sum = sum + nrt_expf(-32.0f * d);
  }
  // smooth_min(k=32): -log(clamp(sum, 1e-4)) / k   (utils.py:385-387)
  sum = fmaxf(sum, 1e-4f);
  return -nrt_logf(sum) / 32.0f;
}

// Evaluates the full SDF for the TM points whose coordinates sit in s.enc_raw rows 0..2.
// Result in val[TM].  sph[TM] is scratch.
template <int H, int TM>
__device__ void sdf_tile_eval(const SdfDev& sd, const TileSmem& s, float* sph, float* val) {
  const int tid = threadIdx.x;
  if (tid < TM) sph[tid] = sphere_set_smin(sd, s.enc_raw[tid], s.enc_raw[TM + tid], s.enc_raw[2 * TM + tid]);
  mlp_tile_forward<H, TM>(sd.mlp, s, nullptr, 0, 0, TM);
  if (tid < TM) val[tid] = sph[tid] + s.outb[tid];
  __syncthreads();
}

template <int H, int TM>
__global__ void __launch_bounds__(kThreads, 1)
k_sdf_eval(SdfDev sd, const float* __restrict__ p, int64_t M, float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  TileSmem s;
  float* rest = carve_tile(s, smem, sd.mlp.dim_p, H, sd.mlp.out, TM);
  float* sph = rest;
  float* val = rest + TM;
  const int64_t ntiles = (M + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t mb = tile * TM;
    const int valid = (int)min((int64_t)TM, M - mb);
    for (int idx = threadIdx.x; idx < TM * 3; idx += kThreads) {
      const int mm = idx / 3, j = idx - mm * 3;
      s.enc_raw[j * TM + mm] = (mm < valid) ? p[(mb + mm) * 3 + j] : 0.0f;
    }
    __syncthreads();
    sdf_tile_eval<H, TM>(sd, s, sph, val);
    if (threadIdx.x < valid) out[mb + threadIdx.x] = val[threadIdx.x];
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// a4 / a7: sphere-trace march (sdfs.py:111-131) and shadow march (sdfs.py:162-181).
//
// Persistent CTAs each own TM ray slots.  Rays whose trajectory has ended (hit, depth past
// max_t, or max_steps reached) write their result and free the slot; free slots are refilled
// from a global ray counter with a ballot/prefix compaction, so every MLP tile evaluation is
// spent on live rays only.  A ray's trajectory depends on nothing but its own state, hence the
// outputs equal the reference's lock-step loop exactly.
// ------------------------------------------------------------------------------------------
enum { MARCH_PRIMARY = 0, MARCH_SHADOW = 1 };

template <int H, int TM, int MODE>
__global__ void __launch_bounds__(kThreads, 1)
k_sdf_march(SdfDev sd, const float* __restrict__ rays, const float* __restrict__ max_t_per_ray,
            const uint8_t* __restrict__ active, int64_t R, float eps, int max_steps, float max_t,
            float t_start, float* __restrict__ depth, uint8_t* __restrict__ flag,
            unsigned long long* __restrict__ ray_counter, unsigned long long* __restrict__ steps_done) {
  extern __shared__ __align__(16) float smem[];
  TileSmem s;
  float* rest = carve_tile(s, smem, sd.mlp.dim_p, H, sd.mlp.out, TM);
  float* sph = rest; rest += TM;
  float* val = rest; rest += TM;
  float* so = rest; rest += 3 * TM;   // origins  [3][TM]
  float* sdir = rest; rest += 3 * TM; // dirs     [3][TM]
  float* st = rest; rest += TM;       // depth
  float* smax = rest; rest += TM;     // per-ray max_t (shadow)
  int* sray = reinterpret_cast<int*>(rest); rest += TM;   // ray id or -1 (R < 2^31 per call)
  int* sit = reinterpret_cast<int*>(rest); rest += TM;    // iterations done
  __shared__ int warp_need[TM / 32];
  __shared__ long long grab_base;
  __shared__ int n_live;
  __shared__ int exhausted;

  const int tid = threadIdx.x;
  if (tid < TM) sray[tid] = -1;
  if (tid == 0) exhausted = 0;
  unsigned long long my_steps = 0;
  __syncthreads();

  for (;;) {
    // ---- retire finished trajectories (pre-evaluation checks) ----
    if (tid < TM && sray[tid] >= 0) {
      bool done = sit[tid] >= max_steps;
      if (MODE == MARCH_PRIMARY) done = done || !(st[tid] < max_t);   // remaining &= depth < max_t
      if (done) {
        const int r = sray[tid];
        if (MODE == MARCH_PRIMARY) { depth[r] = st[tid]; flag[r] = 0; }
        else flag[r] = 1;   // never hit: `remaining` stays true => not blocked
        sray[tid] = -1;
      }
    }
    __syncthreads();
    // ---- refill free slots from the global queue ----
    if (tid < TM) {
      const bool need = (sray[tid] < 0) && !exhausted;
      const unsigned bal = __ballot_sync(0xffffffffu, need);
      if ((tid & 31) == 0) warp_need[tid >> 5] = __popc(bal);
    }
    __syncthreads();
    if (tid == 0) {
      int total = 0;
      for (int w = 0; w < TM / 32; ++w) total += warp_need[w];
      if (total > 0) {
        grab_base = (long long)atomicAdd(ray_counter, (unsigned long long)total);
        if (grab_base + total >= R) exhausted = 1;
      } else {
        grab_base = R;
      }
    }
    __syncthreads();
    if (tid < TM) {
      const bool need = (sray[tid] < 0);
      const unsigned bal = __ballot_sync(0xffffffffu, need);
      int rank = __popc(bal & ((1u << (tid & 31)) - 1u));
      for (int w = 0; w < (tid >> 5); ++w) rank += warp_need[w];
      if (need) {
        const long long r = grab_base + rank;
        if (r < R) {
          const float* rp = rays + r * 6;
          so[tid] = rp[0]; so[TM + tid] = rp[1]; so[2 * TM + tid] = rp[2];
          sdir[tid] = rp[3]; sdir[TM + tid] = rp[4]; sdir[2 * TM + tid] = rp[5];
          st[tid] = t_start;
          sit[tid] = 0;
          smax[tid] = (MODE == MARCH_SHADOW) ? max_t_per_ray[r] : max_t;
          sray[tid] = (int)r;
          if (active != nullptr && active[r] == 0) {
            // inactive rays are skipped (their shading is masked to 0 by the caller)
            if (MODE == MARCH_PRIMARY) { depth[r] = t_start; flag[r] = 0; } else flag[r] = 1;
            sray[tid] = -1;
          }
        }
      }
    }
    __syncthreads();
    if (tid == 0) n_live = 0;
    __syncthreads();
    bool evaluated = false;
    if (tid < TM) {
      const bool live = sray[tid] >= 0;
      // a freshly loaded primary ray must still pass the depth < max_t test before evaluation
      const bool eval = live && (MODE == MARCH_SHADOW || st[tid] < max_t) && sit[tid] < max_steps;
      evaluated = eval;
      const unsigned bal = __ballot_sync(0xffffffffu, live);
      if ((tid & 31) == 0 && bal) atomicAdd(&n_live, __popc(bal));
      // p = r_o + r_d * depth  (mul, then add: two roundings like the eager reference)
      const float t = st[tid];
      s.enc_raw[tid] = eval ? (so[tid] + sdir[tid] * t) : 0.0f;
      s.enc_raw[TM + tid] = eval ? (so[TM + tid] + sdir[TM + tid] * t) : 0.0f;
      s.enc_raw[2 * TM + tid] = eval ? (so[2 * TM + tid] + sdir[2 * TM + tid] * t) : 0.0f;
    }
    __syncthreads();
    if (n_live == 0) {
      if (exhausted) break;
      continue;
    }
    sdf_tile_eval<H, TM>(sd, s, sph, val);
    if (tid < TM && evaluated) {
      my_steps += 1;
      const float d = val[tid];
      const int r = sray[tid];
      if (MODE == MARCH_PRIMARY) {
        if (d <= eps) {           // hits = remaining & (dists <= eps)
          depth[r] = st[tid];     // depth is NOT advanced on the hit step
          flag[r] = 1;
          sray[tid] = -1;
        } else {
          st[tid] = st[tid] + d;
          sit[tid] += 1;
        }
      } else {
        // shadow: depth advances first (uses `remaining` from before the hit test), then
        // hits = remaining & (dists < eps); result = (depth >= max_t) | remaining
        st[tid] = st[tid] + d;
        sit[tid] += 1;
        if (d < eps) {
          flag[r] = (st[tid] >= smax[tid]) ? 1 : 0;
          sray[tid] = -1;
        }
      }
    }
    __syncthreads();
  }
  if (steps_done != nullptr) {
    for (int o = 16; o > 0; o >>= 1) my_steps += __shfl_down_sync(0xffffffffu, my_steps, o);
    if ((tid & 31) == 0 && my_steps) atomicAdd(steps_done, my_steps);
  }
}

// ------------------------------------------------------------------------------------------
// a5: SDF.throughput min-along-ray scan (sdfs.py:232-249)
// ------------------------------------------------------------------------------------------
template <int H, int TM>
__global__ void __launch_bounds__(kThreads, 1)
k_sdf_min_scan(SdfDev sd, const float* __restrict__ rays, int64_t R, double step, int n_steps,
               int32_t* __restrict__ best_idx, float* __restrict__ best_pos, float* __restrict__ min_val) {
  extern __shared__ __align__(16) float smem[];
  TileSmem s;
  float* rest = carve_tile(s, smem, sd.mlp.dim_p, H, sd.mlp.out, TM);
  float* sph = rest; rest += TM;
  float* val = rest; rest += TM;
  const int tid = threadIdx.x;
  const int64_t ntiles = (R + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t r = tile * TM + tid;
    const bool ok = tid < TM && r < R;
    float o[3] = {0, 0, 0}, d[3] = {0, 0, 0};
    if (ok) {
      const float* rp = rays + r * 6;
      o[0] = rp[0]; o[1] = rp[1]; o[2] = rp[2]; d[0] = rp[3]; d[1] = rp[4]; d[2] = rp[5];
    }
    float cur_min = 0.0f;
    int idx = 0;
    for (int j = 0; j <= n_steps; ++j) {
      // t = step*(i+1) is a python float (double) that torch rounds to fp32 when it scales d
      const float t = (float)(step * (double)j);
      if (tid < TM) {
        s.enc_raw[tid] = (j == 0) ? o[0] : (o[0] + t * d[0]);
        s.enc_raw[TM + tid] = (j == 0) ? o[1] : (o[1] + t * d[1]);
        s.enc_raw[2 * TM + tid] = (j == 0) ? o[2] : (o[2] + t * d[2]);
      }
      __syncthreads();
      sdf_tile_eval<H, TM>(sd, s, sph, val);
      if (tid < TM) {
        const float v = val[tid];
        if (j == 0) { cur_min = v; idx = 0; }
        else {
          if (v < cur_min) idx = j;          // strict <: first minimum wins
          cur_min = fminf(cur_min, v);
        }
      }
      __syncthreads();
    }
    if (ok) {
      best_idx[r] = idx;
      if (min_val) min_val[r] = cur_min;
      // best_pos = r_o + (idx.float() * fl32(step)) * d   (sdfs.py:247-248)
      const float tb = (float)idx * (float)step;
      best_pos[r * 3 + 0] = o[0] + tb * d[0];
      best_pos[r * 3 + 1] = o[1] + tb * d[1];
      best_pos[r * 3 + 2] = o[2] + tb * d[2];
    }
  }
}

// ------------------------------------------------------------------------------------------
// a18 + a19: fused NeRFLE volumetric render (nerf.py:175-214).
//   samples -> first MLP -> [latent | r_d | light] -> second MLP -> sigmoid -> compositing,
// one pass, nothing but rays in / rgb out touches HBM (or per-sample sigma/rgb in store mode).
// ------------------------------------------------------------------------------------------
struct NerfArgs {
  const float* rays;        // [R,6]
  const float* ts;          // [S] shared sample distances, or nullptr
  const float* ts_per_ray;  // [R,S] per-ray distances (hierarchical fine pass), or nullptr
  const float* light_code;  // [n_views, light_dim]
  const int32_t* view_of_ray;
  int light_dim;
  int S;
  int64_t R;
  float* out_rgb;           // [R,3]   (composite mode)
  float* out_sigma;         // [R,S]   (store mode: pre-relu density)
  float* out_srgb;          // [R,S,3] (store mode: sigmoid rgb)
  int second_out_act;       // NRT_OUT_SIGMOID for NeRFLE
};

template <int H1, int H2, int TM>
__global__ void __launch_bounds__(kThreads, 1)
k_nerfle(MlpDev m1, MlpDev m2, NerfArgs a) {
  extern __shared__ __align__(16) float smem[];
  // the two MLP contexts alias the same arena; first.outb (sigma + latent) lives outside it
  TileSmem s1, s2;
  const size_t arena1 = tile_smem_floats(m1.dim_p, H1, 0, TM);
  const size_t arena2 = tile_smem_floats(m2.dim_p, H2, m2.out, TM);
  const size_t arena = arena1 > arena2 ? arena1 : arena2;
  carve_tile(s1, smem, m1.dim_p, H1, 0, TM);
  carve_tile(s2, smem, m2.dim_p, H2, m2.out, TM);
  float* rest = smem + arena;
  s1.outb = rest; rest += m1.out * TM;
  float* s_t = rest; rest += TM;          // sample distance of each tile column
  float* s_dir = rest; rest += 3 * TM;
  float* acc_rgb = rest; rest += 3 * TM;  // running composite state per ray-in-tile
  float* acc_cp = rest; rest += TM;
  float* first_term = rest; rest += 4 * TM;  // alpha_0 and rgb_0 (needed once cp_{S-1} is known)
  int* s_ray = reinterpret_cast<int*>(rest); rest += TM;

  const int tid = threadIdx.x;
  const int S = a.S;
  // work unit = `unit` consecutive samples in ray-major order = whole rays
  const int unit = S > TM ? S : TM;
  const int rays_per_unit = unit / S;
  const int tiles_per_unit = unit / TM;
  const int64_t nunits = (a.R + rays_per_unit - 1) / rays_per_unit;
  const int rays_per_tile = TM >= S ? TM / S : 1;
  const bool store = a.out_sigma != nullptr;

  for (int64_t u = blockIdx.x; u < nunits; u += gridDim.x) {
    const int64_t ray0 = u * rays_per_unit;
    for (int tt = 0; tt < tiles_per_unit; ++tt) {
      // ---- sample generation: p = r_o + t * r_d ----
      if (tid < TM) {
        const int64_t samp = (int64_t)tt * TM + tid;  // sample index inside the unit
        const int64_t ray = ray0 + samp / S;
        const int si = (int)(samp % S);
        const bool ok = ray < a.R;
        float p0 = 0, p1 = 0, p2 = 0, t = 0, d0 = 0, d1 = 0, d2 = 0;
        if (ok) {
          const float* rp = a.rays + ray * 6;
          t = a.ts_per_ray ? a.ts_per_ray[ray * S + si] : a.ts[si];
          d0 = rp[3]; d1 = rp[4]; d2 = rp[5];
          p0 = rp[0] + t * d0; p1 = rp[1] + t * d1; p2 = rp[2] + t * d2;
        }
        s1.enc_raw[tid] = p0; s1.enc_raw[TM + tid] = p1; s1.enc_raw[2 * TM + tid] = p2;
        s_t[tid] = t; s_dir[tid] = d0; s_dir[TM + tid] = d1; s_dir[2 * TM + tid] = d2;
        s_ray[tid] = ok ? (int)(ray - ray0) : -1;
      }
      __syncthreads();
      mlp_tile_forward<H1, TM>(m1, s1, nullptr, 0, 0, TM);
      // ---- second MLP input: [latent(64) | r_d(3) | light(light_dim)]  (nerf.py:199-203) ----
      const int nlat = m1.out - 1;
      for (int idx = tid; idx < nlat * TM; idx += kThreads) s2.enc_raw[idx] = s1.outb[TM + idx];
      if (tid < TM) {
        s2.enc_raw[(nlat + 0) * TM + tid] = s_dir[tid];
        s2.enc_raw[(nlat + 1) * TM + tid] = s_dir[TM + tid];
        s2.enc_raw[(nlat + 2) * TM + tid] = s_dir[2 * TM + tid];
      }
      for (int idx = tid; idx < a.light_dim * TM; idx += kThreads) {
        const int j = idx / TM, mm = idx - j * TM;
        float v = 0.0f;
        if (s_ray[mm] >= 0) {
          const int64_t ray = ray0 + s_ray[mm];
          const int view = a.view_of_ray ? a.view_of_ray[ray] : 0;
          v = a.light_code[(int64_t)view * a.light_dim + j];
        }
        s2.enc_raw[(nlat + 3 + j) * TM + mm] = v;
      }
      __syncthreads();
      mlp_tile_forward<H2, TM>(m2, s2, nullptr, 0, 0, TM);
      // ---- epilogue ----
      if (store) {
        if (tid < TM && s_ray[tid] >= 0) {
          const int64_t samp = (ray0 + s_ray[tid]) * S + ((int64_t)tt * TM + tid) % S;
          a.out_sigma[samp] = s1.outb[tid];
          a.out_srgb[samp * 3 + 0] = out_act_apply(a.second_out_act, s2.outb[tid]);
          a.out_srgb[samp * 3 + 1] = out_act_apply(a.second_out_act, s2.outb[TM + tid]);
          a.out_srgb[samp * 3 + 2] = out_act_apply(a.second_out_act, s2.outb[2 * TM + tid]);
        }
      } else if (tid < rays_per_tile) {
        // sequential front-to-back scan, one thread per ray (cumprod order of nerf.py:208)
        const int lr = tid;                       // ray within the tile
        const int col0 = (TM >= S) ? lr * S : 0;  // first tile column of this ray
        const int ncol = (TM >= S) ? S : TM;
        const int s_base = (TM >= S) ? 0 : tt * TM;  // global sample index of column col0
        if (s_ray[col0] >= 0) {
          float cp = (s_base == 0) ? 1.0f : acc_cp[lr];
          float r = (s_base == 0) ? 0.0f : acc_rgb[lr];
          float g = (s_base == 0) ? 0.0f : acc_rgb[TM + lr];
          float b = (s_base == 0) ? 0.0f : acc_rgb[2 * TM + lr];
          for (int c = 0; c < ncol; ++c) {
            const int col = col0 + c;
            const int sidx = s_base + c;
            const float sigma = fmaxf(s1.outb[col], 0.0f);                    // relu
            const float alpha = 1.0f - nrt_expf(-sigma * s_t[col]);           // absolute t (quirk)
            const float cr = out_act_apply(a.second_out_act, s2.outb[col]);
            const float cg = out_act_apply(a.second_out_act, s2.outb[TM + col]);
            const float cb = out_act_apply(a.second_out_act, s2.outb[2 * TM + col]);
            if (sidx == 0) {
              // weight of sample 0 is alpha_0 * cp_{S-1} (roll quirk): deferred
              first_term[lr] = alpha; first_term[TM + lr] = cr;
              first_term[2 * TM + lr] = cg; first_term[3 * TM + lr] = cb;
            } else {
              // weights[s] = alpha_s * cp_{s-1}; the last sample uses 1 instead (quirk)
              const float w = alpha * ((sidx == S - 1) ? 1.0f : cp);
              r = r + w * cr; g = g + w * cg; b = b + w * cb;
            }
            cp = cp * fmaxf(1.0f - alpha, 1e-10f);
          }
          if (s_base + ncol == S) {
            const float w0 = first_term[lr] * ((S == 1) ? 1.0f : cp);
            r = r + w0 * first_term[TM + lr];
            g = g + w0 * first_term[2 * TM + lr];
            b = b + w0 * first_term[3 * TM + lr];
            const int64_t ray = ray0 + s_ray[col0];
            a.out_rgb[ray * 3 + 0] = r; a.out_rgb[ray * 3 + 1] = g; a.out_rgb[ray * 3 + 2] = b;
          } else {
            acc_cp[lr] = cp; acc_rgb[lr] = r; acc_rgb[TM + lr] = g; acc_rgb[2 * TM + lr] = b;
          }
        }
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------
// a19 standalone: compositing over materialised sample-major sigma/rgb (HBM-bound).
// One thread per ray walks the samples front to back; reads are coalesced across rays.
// ------------------------------------------------------------------------------------------
// PER_RAY: ts is [S,R] (one distance per sample, nrt_composite_forward_ts) instead of the shared [S]; the arithmetic is
// the same, so equal distances give equal bits.
template <bool PER_RAY>
__device__ __forceinline__ float comp_t(const float* __restrict__ ts, int s, int64_t R, int64_t r) {
  return PER_RAY ? __ldg(ts + (int64_t)s * R + r) : __ldg(ts + s);
}

template <bool PER_RAY>
__global__ void k_composite_fwd(const float* __restrict__ sigma_raw, const float* __restrict__ rgb,
                                const float* __restrict__ ts, int S, int64_t R, float* __restrict__ out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  float cp = 1.0f, accr = 0.f, accg = 0.f, accb = 0.f;
  float a0 = 0.f, r0 = 0.f, g0 = 0.f, b0 = 0.f;
  for (int s = 0; s < S; ++s) {
    const float sigma = fmaxf(__ldg(sigma_raw + (int64_t)s * R + r), 0.0f);
    const float alpha = 1.0f - nrt_expf(-sigma * comp_t<PER_RAY>(ts, s, R, r));
    const float* c = rgb + ((int64_t)s * R + r) * 3;
    const float cr = __ldg(c), cg = __ldg(c + 1), cb = __ldg(c + 2);
    if (s == 0) { a0 = alpha; r0 = cr; g0 = cg; b0 = cb; }
    else {
      const float w = alpha * ((s == S - 1) ? 1.0f : cp);
      accr = accr + w * cr; accg = accg + w * cg; accb = accb + w * cb;
    }
    cp = cp * fmaxf(1.0f - alpha, 1e-10f);
  }
  const float w0 = a0 * ((S == 1) ? 1.0f : cp);
  out[r * 3 + 0] = accr + w0 * r0;
  out[r * 3 + 1] = accg + w0 * g0;
  out[r * 3 + 2] = accb + w0 * b0;
}

// Backward of the above.  With a_s = 1-exp(-relu(raw_s) t_s), x_s = max(1-a_s, 1e-10),
// P_s = prod_{j<=s} x_j (P_{-1} = 1) the forward weights are
//   w_0 = a_0 P_{S-1},   w_s = a_s P_{s-1} (0 < s < S-1),   w_{S-1} = a_{S-1}.
// With D_s = <g_out, rgb_s>:  dL/da_s = D_s * {P_{S-1}, P_{s-1}, 1} and
//   dL/dx_j = P_{j-1} * (B_j + a_0 D_0 tail_j),
//   B_j = sum_{s=j+1}^{S-2} a_s D_s prod_{i=j+1}^{s-1} x_i,  tail_j = prod_{i>j} x_i,
// both built back to front without dividing by x (which may be 1e-10).  The clamp passes
// gradient where 1-a >= 1e-10 and the relu where raw > 0 (torch semantics).  g_sigma doubles
// as scratch for P_{s-1} between the forward and the backward sweep.
template <bool PER_RAY>
__global__ void k_composite_bwd(const float* __restrict__ sigma_raw, const float* __restrict__ rgb,
                                const float* __restrict__ ts, int S, int64_t R,
                                const float* __restrict__ g_out, float* __restrict__ g_sigma,
                                float* __restrict__ g_rgb) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const float go0 = g_out[r * 3], go1 = g_out[r * 3 + 1], go2 = g_out[r * 3 + 2];
  float cp = 1.0f;
  float a0 = 0.0f, D0 = 0.0f;
  for (int s = 0; s < S; ++s) {
    const int64_t off = (int64_t)s * R + r;
    g_sigma[off] = cp;  // P_{s-1}
    const float sigma = fmaxf(__ldg(sigma_raw + off), 0.0f);
    const float alpha = 1.0f - nrt_expf(-sigma * comp_t<PER_RAY>(ts, s, R, r));
    if (s == 0) {
      a0 = alpha;
      D0 = go0 * __ldg(rgb + off * 3) + go1 * __ldg(rgb + off * 3 + 1) + go2 * __ldg(rgb + off * 3 + 2);
    }
    cp = cp * fmaxf(1.0f - alpha, 1e-10f);
  }
  const float Ptot = cp;
  const float first = (S > 1) ? a0 * D0 : 0.0f;
  float B = 0.0f, tail = 1.0f;
  float nx_a = 0.0f, nx_D = 0.0f, nx_x = 1.0f;  // values of sample s+1
  for (int s = S - 1; s >= 0; --s) {
    const int64_t off = (int64_t)s * R + r;
    const float Pprev = g_sigma[off];
    const float raw = __ldg(sigma_raw + off);
    const float sigma = fmaxf(raw, 0.0f);
    const float t = comp_t<PER_RAY>(ts, s, R, r);
    const float e = nrt_expf(-sigma * t);
    const float alpha = 1.0f - e;
    const float om = 1.0f - alpha;
    const float x = fmaxf(om, 1e-10f);
    const float cr = __ldg(rgb + off * 3), cg = __ldg(rgb + off * 3 + 1), cb = __ldg(rgb + off * 3 + 2);
    const float D = go0 * cr + go1 * cg + go2 * cb;
    if (s < S - 1) {
      B = ((s + 1 <= S - 2) ? nx_a * nx_D : 0.0f) + nx_x * B;
      tail = tail * nx_x;
    }
    float wfac;  // factor multiplying a_s in w_s
    if (S == 1) wfac = 1.0f;
    else if (s == 0) wfac = Ptot;
    else if (s == S - 1) wfac = 1.0f;
    else wfac = Pprev;
    const float w = alpha * wfac;
    g_rgb[off * 3 + 0] = w * go0;
    g_rgb[off * 3 + 1] = w * go1;
    g_rgb[off * 3 + 2] = w * go2;
    const float g_x = (S > 1) ? Pprev * (B + first * tail) : 0.0f;
    float g_alpha = wfac * D;
    if (om >= 1e-10f) g_alpha = g_alpha - g_x;
    // d alpha / d sigma = t * exp(-sigma t);  relu gate
    g_sigma[off] = (raw > 0.0f) ? g_alpha * t * e : 0.0f;
    nx_a = alpha; nx_D = D; nx_x = x;
  }
}

}  // namespace nrt

// ==========================================================================================
// host side: launchers behind the C ABI (include/nrt_b200.h)
// ==========================================================================================
using namespace nrt;

#define NRT_DISPATCH_H(HV, ...)                                                          \
  switch (HV) {                                                                          \
    case 32: { constexpr int H = 32, TM = 64; __VA_ARGS__ } break;                              \
    case 64: { constexpr int H = 64, TM = 64; __VA_ARGS__ } break;                              \
    case 96: { constexpr int H = 96, TM = 64; __VA_ARGS__ } break;                              \
    case 128: { constexpr int H = 128, TM = 64; __VA_ARGS__ } break;                            \
    case 256: { constexpr int H = 256, TM = 32; __VA_ARGS__ } break;                            \
    default:                                                                             \
      nrt_set_error("unsupported hidden size %d (supported: 32, 64, 96, 128, 256)", HV); \
      return NRT_E_UNSUPPORTED;                                                          \
  }

static const size_t kMaxSmem = 227 * 1024;

template <typename K>
static int set_smem(K kernel, size_t bytes) {
  NRT_REQUIRE(bytes <= kMaxSmem, "kernel needs %zu bytes of shared memory (> %zu)", bytes, kMaxSmem);
  NRT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return NRT_OK;
}

// ray-queue counter of a persistent march launch: per device, see nrt_next_counter (nrt_capi.cu)
static int next_counter(cudaStream_t st, unsigned long long** out) { return nrt_next_counter(st, out); }

int nrt_mlp_forward_tc(const nrt_mlp_t* m, int prec, int out_act, const float* x, const float* latent,
                       int64_t M, float* out, float* acts, cudaStream_t st);  // nrt_tc.cu
int nrt_sdf_eval_tc(const nrt_sphere_sdf_t* s, int prec, const float* p, int64_t M, float* out,
                    cudaStream_t st);
int nrt_sdf_march_tc(int shadow, const nrt_sphere_sdf_t* s, int prec, const float* rays, const float* max_t_per_ray,
                     const uint8_t* active, int64_t R, float eps, int max_steps, float max_t, float t_start,
                     float* depth, uint8_t* flag, unsigned long long* counter, unsigned long long* steps_done,
                     cudaStream_t st);
int nrt_sdf_min_scan_tc(const nrt_sphere_sdf_t* s, int prec, const float* rays, int64_t R, double step, int n_steps,
                        int32_t* best_idx, float* best_pos, float* min_val, unsigned long long* counter,
                        cudaStream_t st);

extern "C" int nrt_mlp_forward(const nrt_mlp_t* m, int prec, int out_act, const float* x,
                               const float* latent, int64_t M, float* out, float* acts, void* stream) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(M >= 0, "nrt_mlp_forward: negative M");
  if (M == 0) return NRT_OK;
  NRT_REQUIRE(x != nullptr && out != nullptr, "nrt_mlp_forward: null x/out");
  NRT_REQUIRE(d.latent == 0 || latent != nullptr, "nrt_mlp_forward: latent_size=%d but latent is NULL", d.latent);
  cudaStream_t st = (cudaStream_t)stream;
  if (prec != NRT_PREC_F32) {
    return nrt_mlp_forward_tc(m, prec, out_act, x, latent, M, out, acts, st);
  }
  NRT_DISPATCH_H(d.hidden, {
    const size_t bytes = tile_smem_floats(d.dim_p, H, d.out, TM) * sizeof(float);
    rc = set_smem(k_mlp_fwd<H, TM>, bytes);
    if (rc != NRT_OK) return rc;
    const int64_t ntiles = (M + TM - 1) / TM;
    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)nrt_sm_count() * 8);
    NrtProfScope _ps(TAG_MLP_F32, st);
    k_mlp_fwd<H, TM><<<grid, kThreads, bytes, st>>>(d, x, latent, M, out, acts, out_act);
  })
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

extern "C" int nrt_sdf_eval(const nrt_sphere_sdf_t* s, int prec, const float* p, int64_t M, float* out,
                            void* stream) {
  SdfDev d;
  int rc = nrt_build_sdf_dev(s, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(M >= 0, "nrt_sdf_eval: negative M");
  if (M == 0) return NRT_OK;
  NRT_REQUIRE(p != nullptr && out != nullptr, "nrt_sdf_eval: null p/out");
  cudaStream_t st = (cudaStream_t)stream;
  if (prec != NRT_PREC_F32) return nrt_sdf_eval_tc(s, prec, p, M, out, st);
  NRT_DISPATCH_H(d.mlp.hidden, {
    const size_t bytes = (tile_smem_floats(d.mlp.dim_p, H, d.mlp.out, TM) + 2 * TM) * sizeof(float);
    rc = set_smem(k_sdf_eval<H, TM>, bytes);
    if (rc != NRT_OK) return rc;
    const int64_t ntiles = (M + TM - 1) / TM;
    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)nrt_sm_count() * 8);
    NrtProfScope _ps(TAG_SDF_EVAL_F32, st);
    k_sdf_eval<H, TM><<<grid, kThreads, bytes, st>>>(d, p, M, out);
  })
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

template <int MODE>
static int launch_march(const nrt_sphere_sdf_t* s, int prec, const float* rays, const float* max_t_per_ray,
                        const uint8_t* active, int64_t R, float eps, int max_steps, float max_t, float t_start,
                        float* depth, uint8_t* flag, unsigned long long* steps_done, cudaStream_t st) {
  SdfDev d;
  int rc = nrt_build_sdf_dev(s, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(R >= 0 && R < 2147483647LL, "march: R out of range");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(rays != nullptr && flag != nullptr && max_steps >= 0, "march: bad arguments");
  unsigned long long* counter = nullptr;
  rc = next_counter(st, &counter);
  if (rc != NRT_OK) return rc;
  if (prec != NRT_PREC_F32)
    return nrt_sdf_march_tc(MODE == MARCH_SHADOW, s, prec, rays, max_t_per_ray, active, R, eps, max_steps, max_t,
                            t_start, depth, flag, counter, steps_done, st);
  NRT_DISPATCH_H(d.mlp.hidden, {
    const size_t bytes = (tile_smem_floats(d.mlp.dim_p, H, d.mlp.out, TM) + 12 * TM) * sizeof(float);
    rc = set_smem(k_sdf_march<H, TM, MODE>, bytes);
    if (rc != NRT_OK) return rc;
    const int64_t ntiles = (R + TM - 1) / TM;
    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)nrt_sm_count());
    NrtProfScope _ps(MODE == MARCH_PRIMARY ? TAG_MARCH_F32 : TAG_SHADOW_F32, st);
    k_sdf_march<H, TM, MODE><<<grid, kThreads, bytes, st>>>(d, rays, max_t_per_ray, active, R, eps, max_steps,
                                                            max_t, t_start, depth, flag, counter, steps_done);
  })
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

extern "C" int nrt_sdf_sphere_trace(const nrt_sphere_sdf_t* s, int prec, const float* rays,
                                    const uint8_t* active, int64_t R, float epsilon, int max_steps,
                                    float max_t, float* depth, uint8_t* hit,
                                    unsigned long long* steps_done, void* stream) {
  NRT_REQUIRE(depth != nullptr || R == 0, "nrt_sdf_sphere_trace: depth is NULL");
  return launch_march<MARCH_PRIMARY>(s, prec, rays, nullptr, active, R, epsilon, max_steps, max_t, 0.0f, depth,
                                     hit, steps_done, (cudaStream_t)stream);
}

extern "C" int nrt_sdf_shadow_test(const nrt_sphere_sdf_t* s, int prec, const float* rays,
                                   const float* max_t, const uint8_t* active, int64_t R, float epsilon,
                                   int max_steps, uint8_t* not_blocked, unsigned long long* steps_done,
                                   void* stream) {
  NRT_REQUIRE(max_t != nullptr || R == 0, "nrt_sdf_shadow_test: max_t is NULL");
  // depths start at 1e2 * epsilon (python float product, then cast to fp32; sdfs.py:165-166)
  const float t0 = (float)(1e2 * (double)epsilon);
  return launch_march<MARCH_SHADOW>(s, prec, rays, max_t, active, R, epsilon, max_steps, 0.0f, t0, nullptr,
                                    not_blocked, steps_done, (cudaStream_t)stream);
}

extern "C" int nrt_sdf_min_scan(const nrt_sphere_sdf_t* s, int prec, const float* rays, int64_t R,
                                double step, int n_steps, int32_t* best_idx, float* best_pos,
                                float* min_val, void* stream) {
  SdfDev d;
  int rc = nrt_build_sdf_dev(s, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(R >= 0 && n_steps >= 0, "nrt_sdf_min_scan: bad arguments");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(rays && best_idx && best_pos, "nrt_sdf_min_scan: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (prec != NRT_PREC_F32) {
    unsigned long long* counter = nullptr;
    rc = next_counter(st, &counter);
    if (rc != NRT_OK) return rc;
    return nrt_sdf_min_scan_tc(s, prec, rays, R, step, n_steps, best_idx, best_pos, min_val, counter, st);
  }
  NRT_DISPATCH_H(d.mlp.hidden, {
    const size_t bytes = (tile_smem_floats(d.mlp.dim_p, H, d.mlp.out, TM) + 2 * TM) * sizeof(float);
    rc = set_smem(k_sdf_min_scan<H, TM>, bytes);
    if (rc != NRT_OK) return rc;
    const int64_t ntiles = (R + TM - 1) / TM;
    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)nrt_sm_count() * 4);
    NrtProfScope _ps(TAG_MIN_SCAN_F32, st);
    k_sdf_min_scan<H, TM><<<grid, kThreads, bytes, st>>>(d, rays, R, step, n_steps, best_idx, best_pos, min_val);
  })
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

extern "C" int nrt_composite_forward(const float* sigma_raw, const float* rgb, const float* ts, int S,
                                     int64_t R, float* out, void* stream) {
  NRT_REQUIRE(S >= 1 && R >= 0, "nrt_composite_forward: bad arguments");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(sigma_raw && rgb && ts && out, "nrt_composite_forward: null pointer");
  NrtProfScope _ps(TAG_COMPOSITE_FWD, (cudaStream_t)stream);
  k_composite_fwd<false><<<nrt_cdiv(R, 128), 128, 0, (cudaStream_t)stream>>>(sigma_raw, rgb, ts, S, R, out);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

extern "C" int nrt_composite_backward(const float* sigma_raw, const float* rgb, const float* ts, int S,
                                      int64_t R, const float* g_out, float* g_sigma_raw, float* g_rgb,
                                      void* stream) {
  NRT_REQUIRE(S >= 1 && R >= 0, "nrt_composite_backward: bad arguments");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(sigma_raw && rgb && ts && g_out && g_sigma_raw && g_rgb, "nrt_composite_backward: null pointer");
  NrtProfScope _ps(TAG_COMPOSITE_BWD, (cudaStream_t)stream);
  k_composite_bwd<false><<<nrt_cdiv(R, 128), 128, 0, (cudaStream_t)stream>>>(sigma_raw, rgb, ts, S, R, g_out,
                                                                             g_sigma_raw, g_rgb);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

// the same pair over per-sample distances ts [S,R] (hierarchical sampling, nrt_nerfle_sample_hierarchical)
extern "C" int nrt_composite_forward_ts(const float* sigma_raw, const float* rgb, const float* ts, int S,
                                        int64_t R, float* out, void* stream) {
  NRT_REQUIRE(S >= 1 && R >= 0, "nrt_composite_forward_ts: bad arguments");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(sigma_raw && rgb && ts && out, "nrt_composite_forward_ts: null pointer");
  NrtProfScope _ps(TAG_COMPOSITE_TS_FWD, (cudaStream_t)stream);
  k_composite_fwd<true><<<nrt_cdiv(R, 128), 128, 0, (cudaStream_t)stream>>>(sigma_raw, rgb, ts, S, R, out);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

extern "C" int nrt_composite_backward_ts(const float* sigma_raw, const float* rgb, const float* ts, int S,
                                         int64_t R, const float* g_out, float* g_sigma_raw, float* g_rgb,
                                         void* stream) {
  NRT_REQUIRE(S >= 1 && R >= 0, "nrt_composite_backward_ts: bad arguments");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(sigma_raw && rgb && ts && g_out && g_sigma_raw && g_rgb, "nrt_composite_backward_ts: null pointer");
  NrtProfScope _ps(TAG_COMPOSITE_TS_BWD, (cudaStream_t)stream);
  k_composite_bwd<true><<<nrt_cdiv(R, 128), 128, 0, (cudaStream_t)stream>>>(sigma_raw, rgb, ts, S, R, g_out,
                                                                            g_sigma_raw, g_rgb);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

// fused NeRFLE pass (fp32).  Either composites to out_rgb or stores per-sample sigma/rgb.
int nrt_nerfle_pass_f32(const nrt_mlp_t* first, const nrt_mlp_t* second, const float* rays, int64_t R,
                        const float* ts, const float* ts_per_ray, int S, const float* light_code,
                        int light_dim, const int32_t* view_of_ray, int second_out_act, float* out_rgb,
                        float* out_sigma, float* out_srgb, cudaStream_t st) {
  MlpDev m1, m2;
  int rc = nrt_build_mlp_dev(first, &m1);
  if (rc != NRT_OK) return rc;
  rc = nrt_build_mlp_dev(second, &m2);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(m1.in_size == 3 && m1.latent == 0, "NeRFLE first MLP must map xyz (in_size 3, no latent)");
  NRT_REQUIRE(m2.latent == 0 && m2.in_size == (m1.out - 1) + 3 + light_dim,
              "NeRFLE second MLP in_size %d != latent %d + 3 + light_dim %d", m2.in_size, m1.out - 1, light_dim);
  NRT_REQUIRE(m2.out == 3, "NeRFLE second MLP must output rgb");
  constexpr int TM = 64;
  NRT_REQUIRE(S >= 1 && (S % TM == 0 || TM % S == 0), "samples per ray %d must divide or be a multiple of %d", S, TM);
  NRT_REQUIRE((ts != nullptr) != (ts_per_ray != nullptr), "exactly one of ts / ts_per_ray must be given");
  NRT_REQUIRE(light_dim == 0 || light_code != nullptr, "light_code is NULL");
  if (R == 0) return NRT_OK;
  NerfArgs a;
  a.rays = rays; a.ts = ts; a.ts_per_ray = ts_per_ray; a.light_code = light_code;
  a.view_of_ray = view_of_ray; a.light_dim = light_dim; a.S = S; a.R = R;
  a.out_rgb = out_rgb; a.out_sigma = out_sigma; a.out_srgb = out_srgb; a.second_out_act = second_out_act;
  const int unit = S > TM ? S : TM;
  const int rays_per_unit = unit / S;
  const int64_t nunits = (R + rays_per_unit - 1) / rays_per_unit;
  const size_t arena1 = tile_smem_floats(m1.dim_p, m1.hidden, 0, TM);
  const size_t arena2 = tile_smem_floats(m2.dim_p, m2.hidden, m2.out, TM);
  const size_t bytes = (std::max(arena1, arena2) + (size_t)m1.out * TM + 13 * TM) * sizeof(float);
  const int grid = (int)std::min<int64_t>(nunits, (int64_t)nrt_sm_count() * 8);
#define NRT_NERF_CASE(H1, H2)                                                        \
  if (m1.hidden == H1 && m2.hidden == H2) {                                          \
    rc = set_smem(k_nerfle<H1, H2, TM>, bytes);                                      \
    if (rc != NRT_OK) return rc;                                                     \
    { NrtProfScope _ps(TAG_NERFLE_F32, st);                                          \
    k_nerfle<H1, H2, TM><<<grid, kThreads, bytes, st>>>(m1, m2, a); }                \
    NRT_CUDA(cudaGetLastError());                                                    \
    return NRT_OK;                                                                   \
  }
  NRT_NERF_CASE(128, 64)
  NRT_NERF_CASE(32, 32)
  NRT_NERF_CASE(64, 64)
#undef NRT_NERF_CASE
  nrt_set_error("unsupported NeRF hidden sizes (%d, %d); supported: (128,64), (64,64), (32,32)", m1.hidden, m2.hidden);
  return NRT_E_UNSUPPORTED;
}

