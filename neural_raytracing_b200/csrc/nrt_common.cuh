// Shared host/device declarations for libnrt_b200 (internal; the public ABI is include/nrt_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "nrt_b200.h"
#include "nrt_detmath.h"

#define NRT_NLIN (NRT_MAX_LAYERS + 2)

// Device-side description of one SkipConnMLP with the packed-f32 offsets resolved.
struct MlpDev {
  int in_size, latent, freqs, hidden, L, skip, out, act;
  int dim_p;          // in_size + 2*freqs + latent
  int n_lin;          // L + 2
  int K[NRT_NLIN];    // fan-in of linear layer i
  int N[NRT_NLIN];    // fan-out
  int w_off[NRT_NLIN];  // float offset of W^T [K][N] in params
  int b_off[NRT_NLIN];  // float offset of bias [N]
  unsigned skip_mask;   // bit i set: hidden layer i (0-based) consumes [h | enc]
  const float* basis;   // [in_size][freqs]
  const float* params;
};

struct SdfDev {
  int n;
  const float* centers;
  const float* radii;
  const float* tfs;
  MlpDev mlp;
};

// ---- host helpers (nrt_capi.cu) -------------------------------------------------------
void nrt_set_error(const char* fmt, ...);
int nrt_check_cuda(cudaError_t e, const char* what);
#define NRT_CUDA(call)                                  \
  do {                                                  \
    int _rc = nrt_check_cuda((call), #call);            \
    if (_rc != NRT_OK) return _rc;                      \
  } while (0)
#define NRT_REQUIRE(cond, ...)      \
  do {                              \
    if (!(cond)) {                  \
      nrt_set_error(__VA_ARGS__);   \
      return NRT_E_INVALID;         \
    }                               \
  } while (0)

int nrt_build_mlp_dev(const nrt_mlp_t* m, MlpDev* out);  // validates + resolves offsets
int nrt_build_sdf_dev(const nrt_sphere_sdf_t* s, SdfDev* out);
int nrt_sm_count();   // of the current device

// Per-device state of the library (nrt_capi.cu): no process-global device pointers.
#ifdef __cplusplus
#include <mutex>
#define NRT_MAX_DEVICES 64
struct NrtDeviceState {
  static const unsigned kCounterRing = 1024;
  std::mutex mu;                       // guards the fields below
  int sm_count = 0;
  unsigned long long* counters = nullptr;   // [2 * kCounterRing]: eager ring, then graph-private slots
  unsigned counter_next = 0, capture_next = 0;
  bool pool_configured = false;
  std::mutex host_mu;                  // held by nrt_nerfle_render_host for the whole call
  void* host_ws[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t host_ws_bytes[4] = {0, 0, 0, 0};
};
NrtDeviceState* nrt_device_state();     // record of the current device (nullptr: no device)
int nrt_next_counter(cudaStream_t st, unsigned long long** out);
int nrt_host_scratch(NrtDeviceState* s, int slot, size_t bytes, void** out);
#endif

// launch accounting / optional per-kernel event timing (nrt_profile_* in the C ABI).  Tags are looked up by name; the mesh
// tags stay last, after composite_ts_bwd, so the occupancy tags sit with the other render kernels.
enum NrtTag {
  TAG_MLP_F32 = 0, TAG_SDF_EVAL_F32, TAG_MARCH_F32, TAG_SHADOW_F32, TAG_MIN_SCAN_F32, TAG_NERFLE_F32,
  TAG_COMPOSITE_FWD, TAG_COMPOSITE_BWD, TAG_TC_NERF_FIRST, TAG_TC_NERF_SECOND, TAG_TC_MLP, TAG_TC_PACK,
  TAG_STRATIFIED_TS, TAG_SAMPLE_PDF, TAG_MERGE_COMPOSITE, TAG_OCCUPANCY_CULL, TAG_OCCUPANCY_UPDATE, TAG_MLP_BWD_F32, TAG_SDF_GRAD_F32, TAG_SHADE,
  TAG_TC_SDF_EVAL, TAG_TC_MARCH, TAG_TC_SHADOW, TAG_TC_MIN_SCAN, TAG_TC_TRAIN_FWD, TAG_TC_DGRAD, TAG_TC_WGRAD, TAG_TC_MLP_WIDE,
  TAG_CAMERA_RAYS, TAG_MERGE_TS, TAG_COMPOSITE_TS_FWD, TAG_COMPOSITE_TS_BWD,
  TAG_LATTICE_POINTS, TAG_ISO_COUNT, TAG_ISO_SCAN, TAG_ISO_EMIT, TAG_COUNT
};
void nrt_prof_begin(int tag, cudaStream_t st);
void nrt_prof_end(int tag, cudaStream_t st);
struct NrtProfScope {
  int tag; cudaStream_t st;
  NrtProfScope(int t, cudaStream_t s) : tag(t), st(s) { nrt_prof_begin(tag, st); }
  ~NrtProfScope() { nrt_prof_end(tag, st); }
};

// counter hash -> uniform [0,1) with 24 bits: the jitter of the stratified and fine distances (nrt_render.cu) and of the
// occupancy grid's update points (nrt_occupancy.cu).  32-bit arithmetic: the 64-bit splitmix of round 1 cost ~25 integer
// instructions per sample in kernels that should be HBM-bound; oracle/port.py restates the same recipe.
#ifdef __CUDACC__
__device__ __forceinline__ float hash_u01(uint64_t seed, uint64_t a, uint64_t b) {
  uint32_t h = (uint32_t)seed ^ ((uint32_t)(seed >> 32) * 0x9E3779B1u);
  h = (h ^ (uint32_t)a) * 0x85EBCA77u;
  h = (h ^ (uint32_t)b) * 0xC2B2AE3Du;
  h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
  return (float)(h >> 8) * (1.0f / 16777216.0f);
}
#endif

static inline int nrt_cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
