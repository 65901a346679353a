// tcgen05 / TMEM fused SkipConnMLP kernels (sm_100a): IO policies and host entry points of the gradient-free paths.
//
// k_mlp_tc (tc_core.cuh): one persistent CTA per SM keeps the weights of the network resident in shared memory
// (pre-packed fp16/bf16 UMMA tiles, one cp.async.bulk; the 333 KB SDF network streams its stage operands instead) and
// pushes 128-sample tiles through every layer with tcgen05.mma (kind::f16, M = 128, fp32 accumulators in TMEM).  The
// activations never leave the SM: the epilogue warps read the accumulator with tcgen05.ld, apply activation (the bias
// was pre-loaded into the accumulator), and write the next layer's A operand straight back into TMEM with tcgen05.st
// (the MMA reads A from TMEM, B from shared memory).  Two or three tiles are in flight per CTA (one epilogue warpgroup
// each, one MMA-issuer warp), so the tensor pipe works on one tile while the other tiles' epilogues run.
//
// What a kernel instance does with the tiles is an IO policy (this file): plain [M,in] -> [M,out] evaluation, the two
// NeRFLE render passes (points generated from rays, 16-bit latent hand-off), SDF evaluation, the batched min-along-ray
// scan, and the sphere-trace / shadow marches, where every epilogue thread runs one ray's state machine and pulls new
// rays from a global queue (compaction).
//
// Reference semantics: pytorch3d/pathtracer/neural_blocks.py:75-86, utils.py:37-40, shapes/sdfs.py:111-181, 232-249,
// shapes/nerf.py:175-214.  Fourier phases keep ~fp32 accuracy: fp32 FMAs on the CUDA cores for 3..5-D inputs, a small
// MMA with hi+lo split operands otherwise.
#include <stdlib.h>

#include "tc_core.cuh"
#include "camera_math.cuh"

namespace tc {

// ---------------------------------------------------------------------------------------------
// IO policies
// ---------------------------------------------------------------------------------------------
template <int IN, int LAT, int OUT>
struct IoPlain {   // materialised x [M,IN] (+ latent [M,LAT]) -> out [M,OUT] with output activation
  const float* x; const float* latent; float* out; int out_act;
  __device__ __forceinline__ void load(int64_t m, float* v) const {
#pragma unroll
    for (int j = 0; j < IN; ++j) v[j] = __ldg(x + m * IN + j);
#pragma unroll
    for (int j = 0; j < LAT; ++j) v[IN + j] = __ldg(latent + m * LAT + j);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
#pragma unroll
    for (int j = 0; j < OUT; ++j) {
      float v = o[j];
      if (out_act == NRT_OUT_SIGMOID) v = 1.0f / (1.0f + __expf(-v));
      else if (out_act == NRT_OUT_SOFTPLUS) v = v > 20.0f ? v : __logf(1.0f + __expf(v));
      else if (out_act == NRT_OUT_TANH) v = tanhf(v);
      out[m * OUT + j] = v;
    }
  }
};

// NeRFLE.first: samples along rays in, (sigma_raw, latent) out.  nerf.py:178-183
// The 64-d latent is handed to the second kernel as 16-bit (default: half the traffic, what the second MLP's
// hidden-layer operands round to anyway) or as fp32 (lat32: the second MLP's Fourier phases are sigma = 32 times the
// latent, so the 16-bit hand-off costs ~0.07*|latent| radians of phase error; see nerf_latent32()).  Sample m is produced and
// consumed by the thread of the same tile / lane (m / 128, m % 128), so the scratch is TILE-INTERLEAVED:
// 16-byte group g of sample m lives at ((m / 128) * G + g) * 128 + m % 128 (in 16-byte units, G groups per sample):
// one warp-wide 16-byte store or load covers 512 contiguous bytes (4 lines instead of 32).
// ray of sample m (samples-per-ray S): a shift when S is a power of two (64, 128: every script), else the 64-bit division
// (~50 integer instructions per sample in kernels whose epilogue warps are bound by their instruction count)
static inline int pow2_shift(int S) { int k = 0; while ((1 << k) < S) ++k; return (1 << k) == S ? k : -1; }
__device__ __forceinline__ int64_t ray_of(int64_t m, int S, int shift) { return shift >= 0 ? (m >> shift) : m / S; }

// CAM (SURVEY f4): the ray of a sample is not read from an array but computed from the pixel it belongs to -- ray index
// r_off + m / S of the camera's [n_views, nx, ny, bundle] block, camera_math.cuh, bit-identical to k_camera_rays -- so a
// camera-driven frame has no ray array at all (12 uniform loads of the camera matrix + ~45 arithmetic instructions per sample
// against 6 broadcast loads; measured in profiles/r02i_camera_fused.md).
struct NoCam {};
struct WithCam { nrtcam::CamDev cam; int64_t r_off; };

template <int NLAT, bool CAM = false>
struct IoNerfFirst {
  const float* rays; const float* ts; const float* ts_per_ray; int S;
  float* sigma; void* latent; int fmt; int lat32; int s_shift;
  std::conditional_t<CAM, WithCam, NoCam> c;
  // load() in two halves (k_mlp_tc, NRT_FIRST_PIPE): fetch() issues the loads of t and of the ray (the camera variant also
  // computes the ray), point() forms o + t d once they have landed
  struct Fetch { float t, o[3], d[3]; };
  __device__ __forceinline__ void fetch(int64_t m, Fetch& f) const {
    const int64_t ray = ray_of(m, S, s_shift);
    const int s = (int)(m - ray * S);
    f.t = ts_per_ray ? __ldg(ts_per_ray + m) : __ldg(ts + s);
    if constexpr (CAM) {
      int view;
      nrtcam::cam_ray(c.cam, c.r_off + ray, f.o, f.d, &view);
    } else {
      const float* r = rays + ray * 6;
#pragma unroll
      for (int j = 0; j < 3; ++j) { f.o[j] = __ldg(r + j); f.d[j] = __ldg(r + 3 + j); }
    }
  }
  __device__ __forceinline__ static void point(const Fetch& f, float* v) {
    v[0] = f.o[0] + f.t * f.d[0]; v[1] = f.o[1] + f.t * f.d[1]; v[2] = f.o[2] + f.t * f.d[2];
  }
  __device__ __forceinline__ void load(int64_t m, float* v) const {
    Fetch f;
    fetch(m, f);
    point(f, v);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
    sigma[m] = o[0];
    store_latent(m, o);
  }
  __device__ __forceinline__ void store_latent(int64_t m, const float* o) const {
    if (lat32) {
      float4* dst = reinterpret_cast<float4*>(latent) + (m >> 7) * (int64_t)(NLAT / 4 * 128) + (m & 127);
#pragma unroll
      for (int j = 0; j < NLAT / 4; ++j) dst[j * 128] = make_float4(o[1 + 4 * j], o[2 + 4 * j], o[3 + 4 * j], o[4 + 4 * j]);
      return;
    }
    uint4* dst = reinterpret_cast<uint4*>(latent) + (m >> 7) * (int64_t)(NLAT / 8 * 128) + (m & 127);
#pragma unroll
    for (int j = 0; j < NLAT / 8; ++j) {
      uint4 q;
      if (fmt == 0) {
        q.x = Elem<0>::pack(o[1 + 8 * j], o[2 + 8 * j]); q.y = Elem<0>::pack(o[3 + 8 * j], o[4 + 8 * j]);
        q.z = Elem<0>::pack(o[5 + 8 * j], o[6 + 8 * j]); q.w = Elem<0>::pack(o[7 + 8 * j], o[8 + 8 * j]);
      } else {
        q.x = Elem<1>::pack(o[1 + 8 * j], o[2 + 8 * j]); q.y = Elem<1>::pack(o[3 + 8 * j], o[4 + 8 * j]);
        q.z = Elem<1>::pack(o[5 + 8 * j], o[6 + 8 * j]); q.w = Elem<1>::pack(o[7 + 8 * j], o[8 + 8 * j]);
      }
      dst[j * 128] = q;
    }
  }
};

// NeRFLE.second: [latent | r_d | light code] in, sigmoid(rgb) out.  nerf.py:199-203
template <int NLAT, int LD, bool PACKED = false, bool CAM = false>
struct IoNerfSecond {
  const float* rays; const void* latent; const float* light_code; const int32_t* view_of_ray; int S;
  float* rgb; int fmt; int out_act; int lat32; int s_shift;
  std::conditional_t<CAM, WithCam, NoCam> c;
  // view direction and light-code row of a ray: from the ray array, or from the camera (CAM)
  __device__ __forceinline__ int dir_and_view(int64_t ray, float* d) const {
    if constexpr (CAM) {
      float o[3];
      int view;
      nrtcam::cam_ray(c.cam, c.r_off + ray, o, d, &view);
      return view;
    } else {
      const float* r = rays + ray * 6;
      d[0] = __ldg(r + 3); d[1] = __ldg(r + 4); d[2] = __ldg(r + 5);
      return view_of_ray ? __ldg(view_of_ray + ray) : 0;
    }
  }
  __device__ __forceinline__ void load(int64_t m, float* v) const {
    const int64_t ray = ray_of(m, S, s_shift);
    if (lat32) {
      const float4* src = reinterpret_cast<const float4*>(latent) + (m >> 7) * (int64_t)(NLAT / 4 * 128) + (m & 127);
#pragma unroll
      for (int j = 0; j < NLAT / 4; ++j) {
        const float4 q = __ldg(src + j * 128);
        v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
      }
    } else {
      const uint4* src = reinterpret_cast<const uint4*>(latent) + (m >> 7) * (int64_t)(NLAT / 8 * 128) + (m & 127);
#pragma unroll
      for (int j = 0; j < NLAT / 8; ++j) {
        const uint4 q = __ldg(src + j * 128);
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (fmt == 0) {
            v[8 * j + 2 * e] = Elem<0>::back((uint16_t)(w[e] & 0xffff)); v[8 * j + 2 * e + 1] = Elem<0>::back((uint16_t)(w[e] >> 16));
          } else {
            v[8 * j + 2 * e] = Elem<1>::back((uint16_t)(w[e] & 0xffff)); v[8 * j + 2 * e + 1] = Elem<1>::back((uint16_t)(w[e] >> 16));
          }
        }
      }
    }
    const int view = dir_and_view(ray, v + NLAT);
#pragma unroll
    for (int j = 0; j < LD; ++j) v[NLAT + 3 + j] = __ldg(light_code + (int64_t)view * LD + j);
  }
  // The latent arrives as 16-bit values in the kernel's own operand format: its NLAT / 2 packed pairs ARE the x_hi operand
  // of the phase GEMM and of the init / skip layers, and x_lo is zero.  load_packed hands the words through (the generic
  // path unpacks them to fp32, re-packs and computes x - x_hi = 0: ~10 instructions per pair, a tenth of the kernel's
  // instructions).  x[] receives only the view direction and the light code.
  static constexpr int kPackedPairs = PACKED ? NLAT / 2 : 0;     // PACKED: launched only with a 16-bit latent (lat32 == 0)
  __device__ __forceinline__ void load_packed(int64_t m, uint32_t* w, float* v) const {
    const int64_t ray = ray_of(m, S, s_shift);
    const uint4* src = reinterpret_cast<const uint4*>(latent) + (m >> 7) * (int64_t)(NLAT / 8 * 128) + (m & 127);
#pragma unroll
    for (int j = 0; j < NLAT / 8; ++j) {
      const uint4 q = __ldg(src + j * 128);
      w[4 * j] = q.x; w[4 * j + 1] = q.y; w[4 * j + 2] = q.z; w[4 * j + 3] = q.w;
    }
    const int view = dir_and_view(ray, v + NLAT);
#pragma unroll
    for (int j = 0; j < LD; ++j) v[NLAT + 3 + j] = __ldg(light_code + (int64_t)view * LD + j);
  }
  // load_packed in two pieces (k_mlp_tc, NRT_SECOND_PIPE): the packed latent of a whole tile is one contiguous block of
  // NLAT / 8 * 128 uint4 (copied to shared memory one tile ahead), and the 3 + LD floats of direction and light code
  __device__ __forceinline__ const uint4* packed_tile(int64_t tile) const {
    return reinterpret_cast<const uint4*>(latent) + tile * (int64_t)(NLAT / 8 * 128);
  }
  __device__ __forceinline__ void load_dir_code(int64_t m, float* v) const {
    const int view = dir_and_view(ray_of(m, S, s_shift), v);
#pragma unroll
    for (int j = 0; j < LD; ++j) v[3 + j] = __ldg(light_code + (int64_t)view * LD + j);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float v = o[j];
      if (out_act == NRT_OUT_SIGMOID) v = 1.0f / (1.0f + __expf(-v));
      else if (out_act == NRT_OUT_TANH) v = tanhf(v);
      rgb[m * 3 + j] = v;
    }
  }
};

// The occupancy-culled passes (render_impl with a grid): the kernels evaluate only the samples k_occupancy_cull kept.
// Row m of the launch is sample keep[m] (= ray * S + s within the chunk, ascending), and *rows of them exist (a device
// count, kDeviceRows): sigma and rgb go to the kept sample's own slot, the latent hand-off stays in compacted tile order,
// so the bulk copy of NRT_SECOND_PIPE reads whole tiles as before.  The keep load is one more dependent load in front of
// the ray's, issued a tile ahead with it (fetch / load_dir_code).  MMA rows are independent: a kept sample's outputs are
// the bits the full layout gives it.
template <int NLAT>
struct IoNerfFirstKeep : IoNerfFirst<NLAT> {
  const int32_t* keep; const int32_t* rows;
  static constexpr bool kDeviceRows = true;
  using Fetch = typename IoNerfFirst<NLAT>::Fetch;
  __device__ __forceinline__ void fetch(int64_t m, Fetch& f) const { IoNerfFirst<NLAT>::fetch(__ldg(keep + m), f); }
  __device__ __forceinline__ void load(int64_t m, float* v) const {
    Fetch f;
    fetch(m, f);
    IoNerfFirst<NLAT>::point(f, v);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
    this->sigma[__ldg(keep + m)] = o[0];
    this->store_latent(m, o);
  }
};
template <int NLAT, int LD>
struct IoNerfSecondKeep : IoNerfSecond<NLAT, LD, true> {
  const int32_t* keep; const int32_t* rows;
  static constexpr bool kDeviceRows = true;
  __device__ __forceinline__ int64_t ray_of_row(int64_t m) const { return ray_of(__ldg(keep + m), this->S, this->s_shift); }
  __device__ __forceinline__ void load_packed(int64_t m, uint32_t* w, float* v) const {
    const uint4* src = reinterpret_cast<const uint4*>(this->latent) + (m >> 7) * (int64_t)(NLAT / 8 * 128) + (m & 127);
#pragma unroll
    for (int j = 0; j < NLAT / 8; ++j) {
      const uint4 q = __ldg(src + j * 128);
      w[4 * j] = q.x; w[4 * j + 1] = q.y; w[4 * j + 2] = q.z; w[4 * j + 3] = q.w;
    }
    load_dir_code(m, v + NLAT);
  }
  __device__ __forceinline__ void load_dir_code(int64_t m, float* v) const {
    const int view = this->dir_and_view(ray_of_row(m), v);
#pragma unroll
    for (int j = 0; j < LD; ++j) v[3 + j] = __ldg(this->light_code + (int64_t)view * LD + j);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const { IoNerfSecond<NLAT, LD, true>::store(__ldg(keep + m), o); }
};

static long long* g_dbg_timeline = nullptr;   // development only, see tools/tc_timeline.py
static int g_dbg_timeline_tag = -1;            // stamp only the launches of this profile tag (-1: every launch)
extern "C" void nrtdbg_set_timeline(long long* dev_buf) { g_dbg_timeline = dev_buf; }
extern "C" void nrtdbg_set_timeline_tag(int tag) { g_dbg_timeline_tag = tag; }

// smooth-min of the warped spheres (sdfs.py:37-46, utils.py:385-387), fast-math version for the 16-bit path.
// The sphere parameters sit in shared memory as rows [A_j0 A_j1 A_j2 c_j] of (I + T_i) and the centre, plus the radii
// (sph_fill, once per CTA through the policies' cta_init): per sample and sphere three broadcast LDS.128 + one LDS instead
// of 13 dependent global loads in a loop that could not be unrolled.  Round 2 measured the sphere set at a quarter of the
// min-scan kernel (35.1 ms for sdf_eval against 23.5 ms for the bare MLP on 33.8 M samples).  Same operation order as
// before: values are bit-identical.  The table holds up to kSphMax = 128 spheres (nerf_synthetic.py's SphereSDF(n=2<<6); 6.5 KB
// next to the 220 KB of streamed-weight buffers); more than that take the global-memory loop.
#ifndef NRT_SPH_MAX
#define NRT_SPH_MAX 128
#endif
constexpr int kSphMax = NRT_SPH_MAX;
__device__ __forceinline__ float* sph_table() {
  __shared__ __align__(16) float tab[kSphMax * 13];
  return tab;
}
__device__ __forceinline__ void sph_fill(const SdfDev& sd) {
  if (sd.n > kSphMax) return;
  float* tab = sph_table();
  for (int e = threadIdx.x; e < sd.n * 13; e += blockDim.x) {
    const int i = e / 13, k = e - i * 13;
    float v;
    if (k == 12) v = __ldg(sd.radii + i);
    else {
      const int j = k >> 2, c = k & 3;
      v = c == 3 ? __ldg(sd.centers + i * 3 + j) : __ldg(sd.tfs + i * 9 + j * 3 + c) + (j == c ? 1.0f : 0.0f);
    }
    tab[k == 12 ? kSphMax * 12 + i : i * 12 + k] = v;
  }
}
// APPROX (shadow march, min scan: a boolean / an argmin come out): norm as d2 * rsqrt(d2) and the exponential as one
// ex2.approx on a pre-scaled argument, 2 + 2 instead of 8 + 6 instructions per sphere (sqrtf carries a Newton step and a
// slow-path branch, __expf a range check); since the end of round 2 the primary march as well (NRT_MARCH_FAST bit 1: 9.4 ->
// 8.7 ms per 262,144 rays with every golden unchanged); the point evaluation keeps the round-1 arithmetic.
template <bool APPROX = false>
__device__ __forceinline__ float sphere_smin_fast(const SdfDev& sd, float px, float py, float pz) {
  float sum = 0.0f;
  if (sd.n <= kSphMax) {
    const float4* rows = reinterpret_cast<const float4*>(sph_table());
    const float* rad = sph_table() + kSphMax * 12;
#pragma unroll 4
    for (int i = 0; i < sd.n; ++i) {
      const float4 a = rows[i * 3], b = rows[i * 3 + 1], c = rows[i * 3 + 2];
      const float q0 = fmaf(a.z, pz, fmaf(a.y, py, a.x * px)) - a.w;
      const float q1 = fmaf(b.z, pz, fmaf(b.y, py, b.x * px)) - b.w;
      const float q2 = fmaf(c.z, pz, fmaf(c.y, py, c.x * px)) - c.w;
      const float d2 = fmaf(q2, q2, fmaf(q1, q1, q0 * q0));
      if constexpr (APPROX) {
        float rs;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(fmaxf(d2, 1e-30f)));
        sum += tc::ex2_approx((rad[i] - d2 * rs) * 46.16624130844683f);     // exp(-32 (d - r)), 32 log2(e)
      } else {
        const float d = sqrtf(d2) - rad[i];
        sum += __expf(-32.0f * d);
      }
    }
    return -__logf(fmaxf(sum, 1e-4f)) * (1.0f / 32.0f);
  }
  for (int i = 0; i < sd.n; ++i) {
    const float* T = sd.tfs + i * 9;
    float q[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float t0 = __ldg(T + j * 3 + 0) + (j == 0 ? 1.0f : 0.0f);
      const float t1 = __ldg(T + j * 3 + 1) + (j == 1 ? 1.0f : 0.0f);
      const float t2 = __ldg(T + j * 3 + 2) + (j == 2 ? 1.0f : 0.0f);
      q[j] = fmaf(t2, pz, fmaf(t1, py, t0 * px)) - __ldg(sd.centers + i * 3 + j);
    }
    const float d = sqrtf(fmaf(q[2], q[2], fmaf(q[1], q[1], q[0] * q[0]))) - __ldg(sd.radii + i);
    sum += __expf(-32.0f * d);
  }
  return -__logf(fmaxf(sum, 1e-4f)) * (1.0f / 32.0f);
}

struct IoSdfEval {   // points [M,3] in, sdf value (sphere set + residual MLP) out
  static constexpr int kSplitOut = 1;
  SdfDev sd; const float* p; float* out;
  __device__ __forceinline__ void cta_init() const { sph_fill(sd); }
  __device__ __forceinline__ void load(int64_t m, float* v) const {
    v[0] = __ldg(p + m * 3); v[1] = __ldg(p + m * 3 + 1); v[2] = __ldg(p + m * 3 + 2);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
    out[m] = sphere_smin_fast(sd, __ldg(p + m * 3), __ldg(p + m * 3 + 1), __ldg(p + m * 3 + 2)) + o[0];
  }
};

// ---- iterative policies: thread = ray --------------------------------------------------------------------
// Pulls one ray index per needing lane from the global queue with ONE atomic per warp.  Returns -1 when the
// queue is exhausted.  Must be called by the whole warp.
__device__ __forceinline__ long long grab_ray(unsigned long long* counter, int64_t R, bool need) {
  const unsigned bal = __ballot_sync(0xffffffffu, need);
  if (bal == 0) return -1;
  const int lane = threadIdx.x & 31;
  unsigned long long base = 0;
  if (lane == __ffs(bal) - 1) base = atomicAdd(counter, (unsigned long long)__popc(bal));
  base = __shfl_sync(0xffffffffu, base, __ffs(bal) - 1);
  const long long r = (long long)base + __popc(bal & ((1u << lane) - 1u));
  return (need && r < R) ? r : -1;
}

enum { TC_MARCH_PRIMARY = 0, TC_MARCH_SHADOW = 1 };

// a4 / a7: sphere-trace march and shadow march on the tensor cores (sdfs.py:111-131, 162-181).  Same per-ray
// state machine as k_sdf_march (nrt_f32.cu); the SDF value comes from the 16-bit tensor-core evaluation.
template <int MODE>
struct IoMarch {
  // softplus form of the hidden layers (tc_core.cuh, SoftplusOf).  The primary march keeps the two-MUFU form: with the fp32
  // polynomial (NRT_MARCH_FAST bit 0; march 9.4 -> 9.1 ms per 262,144 rays, 8.1 ms together with bit 1) one grazing pixel of the
  // 16-basis DTU golden flips from hit to miss (36.9 instead of 94 dB on 8,192 pixels, g_spvar.init.weight cosine 0.9966 < 0.997).
  // The sphere set of the primary march takes the approximate norm / exponential of the shadow march and the scan
  // (NRT_MARCH_FAST bit 1, default): 9.4 -> 8.7 ms, every golden unchanged (hits 5,401 / 5,401, image 94.4 dB).  The shadow
  // march (a boolean comes out) takes the fp32 exponent + packed-half polynomial like the min scan.
#ifndef NRT_MARCH_FAST
#define NRT_MARCH_FAST 2
#endif
  static constexpr int kSoftplusForm = MODE == TC_MARCH_PRIMARY ? ((NRT_MARCH_FAST & 1) ? 1 : 0) : 3;
  __device__ __forceinline__ void cta_init() const { sph_fill(sd); }
  SdfDev sd;
  const float* rays; const float* max_t_per_ray; const uint8_t* active; int64_t R;
  float eps; int max_steps; float max_t; float t_start;
  float* depth; uint8_t* flag; unsigned long long* counter; unsigned long long* steps_done;
  struct State { float o[3], d[3], p[3], t, tmax; int it; long long r; bool dry; unsigned steps; };
  __device__ __forceinline__ void init(State& s) const { s.r = -1; s.dry = false; s.steps = 0; s.it = 0; s.t = 0.0f; s.tmax = 0.0f; }
  __device__ __forceinline__ bool next(State& s, float* x) const {
    for (;;) {
      if (s.r >= 0) {
        // pre-evaluation checks: max_steps reached, or (primary) `remaining &= depth < max_t`
        bool done = s.it >= max_steps;
        if (MODE == TC_MARCH_PRIMARY) done = done || !(s.t < max_t);
        if (done) {
          if (MODE == TC_MARCH_PRIMARY) { depth[s.r] = s.t; flag[s.r] = 0; }
          else flag[s.r] = 1;   // never hit: `remaining` stays true => not blocked
          s.r = -1;
        }
      }
      const bool need = s.r < 0 && !s.dry;
      if (__ballot_sync(0xffffffffu, need) == 0) break;
      const long long r = grab_ray(counter, R, need);
      if (need) {
        if (r < 0) { s.dry = true; }
        else if (active != nullptr && active[r] == 0) {
          // inactive rays are skipped (their shading is masked to 0 by the caller)
          if (MODE == TC_MARCH_PRIMARY) { depth[r] = t_start; flag[r] = 0; } else flag[r] = 1;
        } else {
          const float* rp = rays + r * 6;
          s.o[0] = __ldg(rp); s.o[1] = __ldg(rp + 1); s.o[2] = __ldg(rp + 2);
          s.d[0] = __ldg(rp + 3); s.d[1] = __ldg(rp + 4); s.d[2] = __ldg(rp + 5);
          s.t = t_start; s.it = 0; s.r = r;
          s.tmax = (MODE == TC_MARCH_SHADOW) ? __ldg(max_t_per_ray + r) : max_t;
        }
      }
    }
    if (s.r < 0) return false;
#pragma unroll
    for (int j = 0; j < 3; ++j) { s.p[j] = __fadd_rn(s.o[j], __fmul_rn(s.d[j], s.t)); x[j] = s.p[j]; }
    return true;
  }
  __device__ __forceinline__ void consume(State& s, const float* o) const {
    const float d = sphere_smin_fast<MODE != TC_MARCH_PRIMARY || ((NRT_MARCH_FAST & 2) != 0)>(sd, s.p[0], s.p[1], s.p[2]) + o[0];
    s.steps++;
    if (MODE == TC_MARCH_PRIMARY) {
      if (d <= eps) { depth[s.r] = s.t; flag[s.r] = 1; s.r = -1; }   // depth is NOT advanced on the hit step
      else { s.t += d; s.it++; }
    } else {
      s.t += d; s.it++;
      if (d < eps) { flag[s.r] = (s.t >= s.tmax) ? 1 : 0; s.r = -1; }
    }
  }
  __device__ __forceinline__ void finish(State& s) const {
    if (steps_done == nullptr) return;
    unsigned v = s.steps;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(steps_done, (unsigned long long)v);
  }
};

// a5: SDF.throughput min-along-ray scan (sdfs.py:232-249): n_steps+1 evaluations per ray, strict-< running argmin.
// The scan positions do not depend on the SDF values, so the scan is a BATCHED evaluation (sample m = ray * (n+1) + k,
// every MMA row busy whatever the ray count; the per-thread state machine of the march would serialise the n+1
// evaluations of a ray: 129 x ~25 us for a small ray batch) followed by a warp-per-ray argmin.
struct IoScanEval {
  static constexpr int kSoftplusForm = 3;   // packed-half polynomial (tc_core.cuh, SoftplusOf): the scan only picks a position
  __device__ __forceinline__ void cta_init() const { sph_fill(sd); }
  SdfDev sd;
  const float* rays; double step; int n1; float* val;
  __device__ __forceinline__ void point(int64_t m, float* p) const {
    // (a launch covers at most 262,144 rays x (n + 1) samples: 32-bit index arithmetic; the 64-bit division costs ~50
    //  integer instructions and point() runs twice per sample, in load and in store)
    const uint32_t ray = (uint32_t)m / (uint32_t)n1;
    const int k = (int)((uint32_t)m - ray * (uint32_t)n1);
    const float* rp = rays + (int64_t)ray * 6;
    const float t = (float)(step * (double)k);   // python float (double) product, rounded to fp32 when it scales d
#pragma unroll
    for (int j = 0; j < 3; ++j) p[j] = (k == 0) ? __ldg(rp + j) : __fadd_rn(__ldg(rp + j), __fmul_rn(t, __ldg(rp + 3 + j)));
  }
  __device__ __forceinline__ void load(int64_t m, float* x) const { point(m, x); }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
    float p[3];
    point(m, p);
    val[m] = sphere_smin_fast<true>(sd, p[0], p[1], p[2]) + o[0];
  }
};
__global__ void k_scan_argmin(const float* __restrict__ val, const float* __restrict__ rays, int64_t R, int n1, double step,
                              int32_t* __restrict__ best_idx, float* __restrict__ best_pos, float* __restrict__ min_val) {
  const int lane = threadIdx.x & 31;
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= R) return;
  const float* v = val + r * n1;
  float best = 3.0e38f;
  int idx = 0x7fffffff;
  for (int k = lane; k < n1; k += 32) {
    const float x = v[k];
    if (x < best) { best = x; idx = k; }        // strict <: the first minimum wins (k ascends within a lane)
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ob < best || (ob == best && oi < idx)) { best = ob; idx = oi; }
  }
  if (lane == 0) {
    best_idx[r] = idx;
    if (min_val) min_val[r] = best;
    const float tb = __fmul_rn((float)idx, (float)step);   // best_pos = r_o + (idx.float() * fl32(step)) * d  (sdfs.py:247-248)
    for (int j = 0; j < 3; ++j) best_pos[r * 3 + j] = __fadd_rn(rays[r * 6 + j], __fmul_rn(tb, rays[r * 6 + 3 + j]));
  }
}

template <class NET, class IO, int FMT, class SV = NoSave>
static int launch(const void* blob, const IO& io, int64_t M, cudaStream_t st, int tag = TAG_TC_MLP, SV sv = SV{}) {
  const size_t bytes = (size_t)SecondPipe<NET, IO, SV>::SMEM_BYTES + 256;
  auto kern = k_mlp_tc<NET, IO, FMT, SV>;
  NRT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  const int64_t ntiles = (M + 127) / 128;
  const int grid = (int)std::min<int64_t>((ntiles + NET::NSLOT - 1) / NET::NSLOT, (int64_t)nrt_sm_count());
  NrtProfScope _ps(tag, st);
  long long* dbg = g_dbg_timeline_tag < 0 || g_dbg_timeline_tag == tag ? g_dbg_timeline : nullptr;
  kern<<<grid, NET::threads(NET::WPS), bytes, st>>>(reinterpret_cast<const uint8_t*>(blob) + NET::BLOB_OFF, io, M, dbg, sv);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

// the networks instantiated on the tensor-core path (all weights must fit in 227 KB of smem)
using NetNerfFirst = Net<3, 0, 16, 128, 5, 3, 65, NRT_ACT_LEAKY_RELU>;      // NeRFLE.first   nerf.py:162-167
// NeRFLE.first's inference kernels (render pass, plain forward): with NRT_BIAS_MMA bit 2 they read the render layout, which
// nrt_mlp_pack_tc appends to the training layout (tc_core.cuh, make_render_layout); otherwise the same net as above
using NetNerfFirstR = Net<3, 0, 16, 128, 5, 3, 65, NRT_ACT_LEAKY_RELU, (NRT_BIAS_MMA & 4) != 0>;
using NetNerfSecondPT = Net<70, 0, 16, 64, 8, 3, 3, NRT_ACT_LEAKY_RELU>;    // NeRFLE.second  nerf.py:169-172
using NetNerfSecondLE = Net<115, 0, 16, 64, 8, 3, 3, NRT_ACT_LEAKY_RELU>;   // NeRFLE.second, envmap code (64+3+48)
using NetNeuralBsdf = Net<3, 0, 64, 96, 6, 3, 3, NRT_ACT_LEAKY_RELU>;       // NeuralBSDF.mlp bsdfs.py:616-621
using NetOcc = Net<5, 0, 16, 64, 8, 3, 1, NRT_ACT_LEAKY_RELU>;              // occlusion MLP  colocate.py:82-85
using NetPlainFirst = Net<3, 32, 16, 32, 5, 3, 33, NRT_ACT_LEAKY_RELU>;      // PlainNeRF.first  nerf.py:17-22 (per-image latent)
using NetPlainSecond = Net<2, 64, 16, 32, 5, 3, 3, NRT_ACT_LEAKY_RELU>;      // PlainNeRF.second nerf.py:24-28
using NetSdfShift = Net<3, 0, 32, 128, 8, 3, 1, NRT_ACT_SOFTPLUS>;         // SphereSDF.shift sdfs.py:23-31 (streamed)

template <class NET>
static bool matches(const MlpDev& d) {
  return d.in_size == NET::IN && d.latent == NET::LAT && d.freqs == NET::F && d.hidden == NET::H && d.L == NET::L &&
         d.skip == NET::SKIP && d.out == NET::OUT && d.act == NET::ACT;
}
template <class NET>
static bool matches(const nrt_mlp_t& m) {
  return m.in_size == NET::IN && m.latent_size == NET::LAT && m.freqs == NET::F && m.hidden == NET::H && m.num_layers == NET::L &&
         m.skip == NET::SKIP && m.out_size == NET::OUT && m.act == NET::ACT;
}

}  // namespace tc

using namespace tc;

static int fmt_of(int prec) { return prec == NRT_PREC_BF16 ? 1 : 0; }

extern "C" int64_t nrt_mlp_tc_blob_bytes(const nrt_mlp_t* m, int prec) {
  NRT_REQUIRE(m != nullptr, "mlp descriptor is NULL");
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "nrt_mlp_tc_blob_bytes: prec must be F16 or BF16");
  NRT_REQUIRE(m->num_layers >= 1 && m->num_layers <= NRT_MAX_LAYERS && m->hidden % 16 == 0, "unsupported MLP shape");
  if (matches<NetNerfFirst>(*m)) return (int64_t)NetNerfFirstR::BLOB_OFF + NetNerfFirstR::Y.bytes;   // + the render layout
  const Layout y = make_layout(m->in_size, m->latent_size, m->freqs, m->hidden, m->num_layers, m->skip, m->out_size);
  return (int64_t)y.bytes;
}

extern "C" int nrt_mlp_pack_tc(const nrt_mlp_t* m, int prec, void* blob_out, void* stream) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "nrt_mlp_pack_tc: prec must be F16 or BF16");
  NRT_REQUIRE(blob_out != nullptr && ((uintptr_t)blob_out & 15) == 0, "blob_out must be 16-byte aligned");
  NRT_REQUIRE(d.hidden % 16 == 0, "hidden must be a multiple of 16");
  NrtProfScope _ps(TAG_TC_PACK, (cudaStream_t)stream);
  auto pack = [&](const Layout& y, const BiasRows& br, uint8_t* dst) {
    const int grid = std::min(nrt_cdiv(pack_tc_items(y), 256), 1184);
    if (fmt_of(prec) == 0) k_pack_tc<0><<<grid, 256, 0, (cudaStream_t)stream>>>(d, y, br, dst);
    else k_pack_tc<1><<<grid, 256, 0, (cudaStream_t)stream>>>(d, y, br, dst);
  };
  pack(make_layout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out), no_bias_rows(), (uint8_t*)blob_out);
  if (NetNerfFirstR::BLOB_OFF > 0 && matches<NetNerfFirst>(d))
    pack(NetNerfFirstR::Y, NetNerfFirstR::BR, (uint8_t*)blob_out + NetNerfFirstR::BLOB_OFF);
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

template <class NET>
static int forward_plain(const nrt_mlp_t* m, int prec, int out_act, const float* x, const float* latent, int64_t M,
                         float* out, cudaStream_t st) {
  IoPlain<NET::IN, NET::LAT, NET::OUT> io{x, latent, out, out_act};
  if (fmt_of(prec) == 0) return launch<NET, decltype(io), 0>(m->params_tc, io, M, st);
  return launch<NET, decltype(io), 1>(m->params_tc, io, M, st);
}
// the same forward, also writing the post-activation layer inputs for the fused fp32 backward (training)
template <class NET>
static int forward_plain_save(const nrt_mlp_t* m, int prec, int out_act, const float* x, const float* latent, int64_t M,
                              float* out, float* acts, cudaStream_t st) {
  IoPlain<NET::IN, NET::LAT, NET::OUT> io{x, latent, out, out_act};
  SaveF32 sv{acts, M};
  if (fmt_of(prec) == 0) return launch<NET, decltype(io), 0, SaveF32>(m->params_tc, io, M, st, TAG_TC_MLP, sv);
  return launch<NET, decltype(io), 1, SaveF32>(m->params_tc, io, M, st, TAG_TC_MLP, sv);
}

int nrt_mlp_forward_tc_wide(const nrt_mlp_t* m, const MlpDev& d, int prec, int out_act, const float* x, int64_t M, float* out,
                            float* acts, cudaStream_t st, bool* handled);   // nrt_tc_wide.cu

int nrt_mlp_forward_tc(const nrt_mlp_t* m, int prec, int out_act, const float* x, const float* latent, int64_t M,
                       float* out, float* acts, cudaStream_t st) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "unknown precision %d", prec);
  NRT_REQUIRE(m->params_tc != nullptr, "mlp.params_tc is NULL: call nrt_mlp_pack_tc first");
  if (acts != nullptr) {
    // saved activations for nrt_mlp_backward on a tensor-core forward: the 256-wide networks, NeuralBSDF, occlusion MLP
    bool handled = false;
    rc = nrt_mlp_forward_tc_wide(m, d, prec, out_act, x, M, out, acts, st, &handled);
    if (handled) return rc;
    if (matches<NetNeuralBsdf>(d)) return forward_plain_save<NetNeuralBsdf>(m, prec, out_act, x, latent, M, out, acts, st);
    if (matches<NetOcc>(d)) return forward_plain_save<NetOcc>(m, prec, out_act, x, latent, M, out, acts, st);
    nrt_set_error("nrt_mlp_forward: saved activations with a 16-bit precision are produced for the 256-wide networks, "
                  "NeuralBSDF.mlp and the occlusion MLP only");
    return NRT_E_UNSUPPORTED;
  }
  if (matches<NetNerfFirst>(d)) return forward_plain<NetNerfFirstR>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetNerfSecondPT>(d)) return forward_plain<NetNerfSecondPT>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetNerfSecondLE>(d)) return forward_plain<NetNerfSecondLE>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetNeuralBsdf>(d)) return forward_plain<NetNeuralBsdf>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetOcc>(d)) return forward_plain<NetOcc>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetSdfShift>(d)) return forward_plain<NetSdfShift>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetPlainFirst>(d)) return forward_plain<NetPlainFirst>(m, prec, out_act, x, latent, M, out, st);
  if (matches<NetPlainSecond>(d)) return forward_plain<NetPlainSecond>(m, prec, out_act, x, latent, M, out, st);
  {
    bool handled = false;   // the 256-wide networks (weights streamed in K-chunks, nrt_tc_wide.cu)
    rc = nrt_mlp_forward_tc_wide(m, d, prec, out_act, x, M, out, nullptr, st, &handled);
    if (handled) return rc;
  }
  nrt_set_error("tensor-core path: MLP shape (in %d, latent %d, freqs %d, hidden %d, layers %d, out %d, act %d) is not "
                "instantiated; use NRT_PREC_F32", d.in_size, d.latent, d.freqs, d.hidden, d.L, d.out, d.act);
  return NRT_E_UNSUPPORTED;
}

int nrt_sdf_eval_tc(const nrt_sphere_sdf_t* s, int prec, const float* p, int64_t M, float* out, cudaStream_t st) {
  SdfDev d;
  int rc = nrt_build_sdf_dev(s, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "unknown precision %d", prec);
  NRT_REQUIRE(s->shift.params_tc != nullptr, "sdf.shift.params_tc is NULL: call nrt_mlp_pack_tc first");
  NRT_REQUIRE(matches<NetSdfShift>(d.mlp), "tensor-core SDF path: shift must be the 8x128 softplus MLP with 32 frequencies");
  IoSdfEval io{d, p, out};
  if (fmt_of(prec) == 0) return launch<NetSdfShift, IoSdfEval, 0>(s->shift.params_tc, io, M, st, TAG_TC_SDF_EVAL);
  return launch<NetSdfShift, IoSdfEval, 1>(s->shift.params_tc, io, M, st, TAG_TC_SDF_EVAL);
}

template <int MODE>
static int march_tc(const nrt_sphere_sdf_t* s, int prec, const float* rays, const float* max_t_per_ray,
                    const uint8_t* active, int64_t R, float eps, int max_steps, float max_t, float t_start,
                    float* depth, uint8_t* flag, unsigned long long* counter, unsigned long long* steps_done,
                    cudaStream_t st) {
  SdfDev d;
  int rc = nrt_build_sdf_dev(s, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "unknown precision %d", prec);
  NRT_REQUIRE(s->shift.params_tc != nullptr, "sdf.shift.params_tc is NULL: call nrt_mlp_pack_tc first");
  NRT_REQUIRE(matches<NetSdfShift>(d.mlp), "tensor-core SDF path: shift must be the 8x128 softplus MLP with 32 frequencies");
  IoMarch<MODE> io{d, rays, max_t_per_ray, active, R, eps, max_steps, max_t, t_start, depth, flag, counter, steps_done};
  const int tag = MODE == TC_MARCH_PRIMARY ? TAG_TC_MARCH : TAG_TC_SHADOW;
  if (fmt_of(prec) == 0) return launch<NetSdfShift, IoMarch<MODE>, 0>(s->shift.params_tc, io, R, st, tag);
  return launch<NetSdfShift, IoMarch<MODE>, 1>(s->shift.params_tc, io, R, st, tag);
}
int nrt_sdf_march_tc(int shadow, const nrt_sphere_sdf_t* s, int prec, const float* rays, const float* max_t_per_ray,
                     const uint8_t* active, int64_t R, float eps, int max_steps, float max_t, float t_start,
                     float* depth, uint8_t* flag, unsigned long long* counter, unsigned long long* steps_done,
                     cudaStream_t st) {
  if (shadow) return march_tc<TC_MARCH_SHADOW>(s, prec, rays, max_t_per_ray, active, R, eps, max_steps, max_t, t_start,
                                               depth, flag, counter, steps_done, st);
  return march_tc<TC_MARCH_PRIMARY>(s, prec, rays, max_t_per_ray, active, R, eps, max_steps, max_t, t_start, depth,
                                    flag, counter, steps_done, st);
}
int nrt_sdf_min_scan_tc(const nrt_sphere_sdf_t* s, int prec, const float* rays, int64_t R, double step, int n_steps,
                        int32_t* best_idx, float* best_pos, float* min_val, unsigned long long* counter,
                        cudaStream_t st) {
  SdfDev d;
  int rc = nrt_build_sdf_dev(s, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "unknown precision %d", prec);
  NRT_REQUIRE(s->shift.params_tc != nullptr, "sdf.shift.params_tc is NULL: call nrt_mlp_pack_tc first");
  NRT_REQUIRE(matches<NetSdfShift>(d.mlp), "tensor-core SDF path: shift must be the 8x128 softplus MLP with 32 frequencies");
  (void)counter;
  const int n1 = n_steps + 1;
  NRT_REQUIRE(n_steps >= 0 && n1 <= 8192, "tensor-core min scan: 0..8191 steps (32-bit sample index per 262,144-ray pass)");
  const int64_t kChunk = 262144;                       // rays per pass: bounds the scratch to 135 MB at n = 128
  const int64_t C = std::min<int64_t>(R, kChunk);
  // stream-ordered scratch from the device's default memory pool; without a release threshold the pool hands the
  // memory back to the OS at every synchronisation and each call pays a multi-millisecond re-allocation
  if (NrtDeviceState* ds = nrt_device_state()) {
    std::lock_guard<std::mutex> lk(ds->mu);
    if (!ds->pool_configured) {
      int dev = 0;
      cudaMemPool_t pool;
      if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = 1ull << 30;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
      ds->pool_configured = true;
    }
  }
  float* val = nullptr;
  NRT_CUDA(cudaMallocAsync((void**)&val, (size_t)C * n1 * sizeof(float), st));
  for (int64_t r0 = 0; r0 < R; r0 += kChunk) {
    const int64_t n = std::min<int64_t>(kChunk, R - r0);
    IoScanEval io{d, rays + r0 * 6, step, n1, val};
    rc = fmt_of(prec) == 0 ? launch<NetSdfShift, IoScanEval, 0>(s->shift.params_tc, io, n * n1, st, TAG_TC_MIN_SCAN)
                           : launch<NetSdfShift, IoScanEval, 1>(s->shift.params_tc, io, n * n1, st, TAG_TC_MIN_SCAN);
    if (rc != NRT_OK) break;
    NrtProfScope _ps(TAG_TC_MIN_SCAN, st);
    k_scan_argmin<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(val, rays + r0 * 6, n, n1, step, best_idx + r0, best_pos + r0 * 3,
                                                                     min_val ? min_val + r0 : nullptr);
  }
  cudaFreeAsync(val, st);
  if (rc != NRT_OK) return rc;
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

// Latent hand-off format of the RENDER path: 16-bit by default, fp32 with NRT_NERF_LATENT=f32 in the environment (read
// once).  Measured on B200 (800x800x192, profiles/r02_kernel_log.md): the second kernel reads either at the same speed,
// the first kernel is 12 % slower when it writes fp32 (32.0 vs 28.6 ms per frame).  With random-init or weight-decayed
// networks |latent| is ~0.1 and the 16-bit rounding (2e-5) is below the error the latent already carries from its own
// 16-bit GEMM (max 8e-5, tests/test_gpu_tensorcore.py); the training path always hands over fp32.
static bool nerf_latent32() {
  static const bool v = [] { const char* e = getenv("NRT_NERF_LATENT"); return e && (e[0] == 'f' || e[0] == 'F') && e[1] == '3'; }();
  return v;
}

size_t nrt_nerfle_pass_tc_workspace(const nrt_mlp_t* first, const nrt_mlp_t*, int64_t R, int S) {
  const int nlat = first->out_size - 1;
  const size_t mpad = ((size_t)R * S + 127) / 128 * 128;          // whole 128-sample tiles (tile-interleaved layout)
  return mpad * nlat * (nerf_latent32() ? 4 : 2) + 256;           // latent scratch between the two kernels
}

// whether the camera-fed kernels (IoNerfFirst / IoNerfSecond with CAM) exist for this pair of networks: the point-light net
// with the 16-bit packed latent hand-off (every script's configuration; the others take their rays from k_camera_rays)
bool nrt_nerfle_pass_tc_camera_ok(const nrt_mlp_t* first, const nrt_mlp_t* second, int light_dim) {
  MlpDev d1, d2;
  if (nrt_build_mlp_dev(first, &d1) != NRT_OK || nrt_build_mlp_dev(second, &d2) != NRT_OK) return false;
  return matches<NetNerfFirst>(d1) && matches<NetNerfSecondPT>(d2) && light_dim == 3 && !nerf_latent32();
}

int nrt_nerfle_pass_tc(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                       const float* ts, const float* ts_per_ray, int S, const float* light_code, int light_dim,
                       const int32_t* view_of_ray, int second_out_act, float* out_rgb, float* out_sigma,
                       float* out_srgb, void* workspace, size_t workspace_bytes, cudaStream_t st,
                       const nrt_camera_t* cam, int64_t cam_r0) {
  MlpDev d1, d2;
  int rc = nrt_build_mlp_dev(first, &d1);
  if (rc != NRT_OK) return rc;
  rc = nrt_build_mlp_dev(second, &d2);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(first->params_tc && second->params_tc, "params_tc is NULL: call nrt_mlp_pack_tc first");
  NRT_REQUIRE(matches<NetNerfFirst>(d1), "tensor-core NeRF path: first MLP must be NeRFLE.first (3->65, 5x128)");
  const bool pt = matches<NetNerfSecondPT>(d2) && light_dim == 3;
  const bool le = matches<NetNerfSecondLE>(d2) && light_dim == 48;
  NRT_REQUIRE(pt || le, "tensor-core NeRF path: second MLP must be NeRFLE.second (70->3 with a point light, or 115->3 with "
                        "the 48-float environment code; 8x64)");
  NRT_REQUIRE(out_rgb == nullptr && out_sigma != nullptr && out_srgb != nullptr,
              "tensor-core NeRF pass stores per-sample sigma/rgb (compositing is a separate kernel)");
  NRT_REQUIRE((ts != nullptr) != (ts_per_ray != nullptr), "exactly one of ts / ts_per_ray must be given");
  const int64_t M = R * S;
  const int lat32 = nerf_latent32() ? 1 : 0;
  NRT_REQUIRE(workspace != nullptr && workspace_bytes >= (size_t)((M + 127) / 128 * 128) * 64 * (lat32 ? 4 : 2), "workspace too small");
  void* lat = workspace;
  const int fmt = fmt_of(prec);
  const int s_shift = pow2_shift(S);
  if (cam != nullptr) {
    // rays computed inside the kernels from the camera (f4): no ray array
    NRT_REQUIRE(pt && !lat32, "camera-fed tensor-core NeRF pass: point-light net with the 16-bit latent only");
    const WithCam wc{nrtcam::make_cam_dev(cam), cam_r0};
    IoNerfFirst<64, true> io1{nullptr, ts, ts_per_ray, S, out_sigma, lat, fmt, lat32, s_shift, wc};
    rc = fmt == 0 ? launch<NetNerfFirstR, decltype(io1), 0>(first->params_tc, io1, M, st, TAG_TC_NERF_FIRST)
                  : launch<NetNerfFirstR, decltype(io1), 1>(first->params_tc, io1, M, st, TAG_TC_NERF_FIRST);
    if (rc != NRT_OK) return rc;
    IoNerfSecond<64, 3, true, true> io2{nullptr, lat, light_code, nullptr, S, out_srgb, fmt, second_out_act, lat32, s_shift, wc};
    return fmt == 0 ? launch<NetNerfSecondPT, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                    : launch<NetNerfSecondPT, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
  }
  IoNerfFirst<64> io1{rays, ts, ts_per_ray, S, out_sigma, lat, fmt, lat32, s_shift};
  rc = fmt == 0 ? launch<NetNerfFirstR, decltype(io1), 0>(first->params_tc, io1, M, st, TAG_TC_NERF_FIRST)
                : launch<NetNerfFirstR, decltype(io1), 1>(first->params_tc, io1, M, st, TAG_TC_NERF_FIRST);
  if (rc != NRT_OK) return rc;
  if (pt && !lat32) {
    IoNerfSecond<64, 3, true> io2{rays, lat, light_code, view_of_ray, S, out_srgb, fmt, second_out_act, lat32, s_shift};
    return fmt == 0 ? launch<NetNerfSecondPT, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                    : launch<NetNerfSecondPT, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
  }
  if (pt) {
    IoNerfSecond<64, 3> io2{rays, lat, light_code, view_of_ray, S, out_srgb, fmt, second_out_act, lat32, s_shift};
    return fmt == 0 ? launch<NetNerfSecondPT, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                    : launch<NetNerfSecondPT, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
  }
#ifndef NRT_LE_PACKED
#define NRT_LE_PACKED 1
#endif
  if (NRT_LE_PACKED && !lat32) {
    // environment-light net: the 16-bit latent handed through as packed operand words, like the point-light net
    IoNerfSecond<64, 48, true> io2{rays, lat, light_code, view_of_ray, S, out_srgb, fmt, second_out_act, lat32, s_shift};
    return fmt == 0 ? launch<NetNerfSecondLE, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                    : launch<NetNerfSecondLE, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
  }
  IoNerfSecond<64, 48> io2{rays, lat, light_code, view_of_ray, S, out_srgb, fmt, second_out_act, lat32, s_shift};
  return fmt == 0 ? launch<NetNerfSecondLE, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                  : launch<NetNerfSecondLE, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
}

// the pass of an occupancy-culled render (nrt_render.cu, render_impl with a grid): the same two kernels on the rows that
// k_occupancy_cull kept.  R * S is the capacity the persistent grids are sized from; *rows (device) is how many exist.
int nrt_nerfle_pass_tc_keep(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                            const float* ts, const float* ts_per_ray, int S, const float* light_code, int light_dim,
                            const int32_t* view_of_ray, const int32_t* keep, const int32_t* rows, float* out_sigma,
                            float* out_srgb, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  MlpDev d1, d2;
  int rc = nrt_build_mlp_dev(first, &d1);
  if (rc != NRT_OK) return rc;
  rc = nrt_build_mlp_dev(second, &d2);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(first->params_tc && second->params_tc, "params_tc is NULL: call nrt_mlp_pack_tc first");
  NRT_REQUIRE(matches<NetNerfFirst>(d1), "tensor-core NeRF path: first MLP must be NeRFLE.first (3->65, 5x128)");
  const bool pt = matches<NetNerfSecondPT>(d2) && light_dim == 3;
  const bool le = matches<NetNerfSecondLE>(d2) && light_dim == 48;
  NRT_REQUIRE(pt || le, "tensor-core NeRF path: second MLP must be NeRFLE.second (70->3 with a point light, or 115->3 with "
                        "the 48-float environment code; 8x64)");
  NRT_REQUIRE(rays != nullptr && keep != nullptr && rows != nullptr && out_sigma != nullptr && out_srgb != nullptr,
              "occupancy-culled NeRF pass: null rays/keep/rows/outputs");
  NRT_REQUIRE((ts != nullptr) != (ts_per_ray != nullptr), "exactly one of ts / ts_per_ray must be given");
  if (nerf_latent32()) {
    nrt_set_error("occupancy-culled NeRF pass: the 16-bit latent hand-off only (NRT_NERF_LATENT=f32 is not combined with a grid)");
    return NRT_E_UNSUPPORTED;
  }
  const int64_t M = R * S;
  NRT_REQUIRE(workspace != nullptr && workspace_bytes >= (size_t)((M + 127) / 128 * 128) * 64 * 2, "workspace too small");
  void* lat = workspace;
  const int fmt = fmt_of(prec);
  const int s_shift = pow2_shift(S);
  IoNerfFirstKeep<64> io1{{rays, ts, ts_per_ray, S, out_sigma, lat, fmt, 0, s_shift}, keep, rows};
  rc = fmt == 0 ? launch<NetNerfFirstR, decltype(io1), 0>(first->params_tc, io1, M, st, TAG_TC_NERF_FIRST)
                : launch<NetNerfFirstR, decltype(io1), 1>(first->params_tc, io1, M, st, TAG_TC_NERF_FIRST);
  if (rc != NRT_OK) return rc;
  if (pt) {
    IoNerfSecondKeep<64, 3> io2{{rays, lat, light_code, view_of_ray, S, out_srgb, fmt, NRT_OUT_SIGMOID, 0, s_shift}, keep, rows};
    return fmt == 0 ? launch<NetNerfSecondPT, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                    : launch<NetNerfSecondPT, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
  }
  IoNerfSecondKeep<64, 48> io2{{rays, lat, light_code, view_of_ray, S, out_srgb, fmt, NRT_OUT_SIGMOID, 0, s_shift}, keep, rows};
  return fmt == 0 ? launch<NetNerfSecondLE, decltype(io2), 0>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND)
                  : launch<NetNerfSecondLE, decltype(io2), 1>(second->params_tc, io2, M, st, TAG_TC_NERF_SECOND);
}
