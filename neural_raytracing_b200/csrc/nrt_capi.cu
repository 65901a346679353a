// C-ABI plumbing of libnrt_b200: error reporting, descriptor validation, device queries and
// the entry points that only orchestrate other kernels.
#include <stdarg.h>

#include <algorithm>

#include "nrt_common.cuh"

static thread_local char g_err[512] = "";

void nrt_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int nrt_check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return NRT_OK;
  nrt_set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return NRT_E_CUDA;
}

extern "C" const char* nrt_last_error(void) { return g_err; }
extern "C" int nrt_abi_version(void) { return NRT_ABI_VERSION; }

// ---- per-device state -------------------------------------------------------------------------------------------
// Everything the library keeps between calls besides thread-local error text lives here, one record per CUDA device
// (indexed by cudaGetDevice() at the time of the call), each guarded by its own mutex: the SM count, the ring of
// ray-queue counters of the persistent march kernels and the grow-only scratch of the host-buffer entry point.
#include <mutex>
static NrtDeviceState g_dev_state[NRT_MAX_DEVICES];

NrtDeviceState* nrt_device_state() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= NRT_MAX_DEVICES) return nullptr;
  return &g_dev_state[dev];
}

int nrt_sm_count() {
  NrtDeviceState* s = nrt_device_state();
  if (s == nullptr) return 148;
  std::lock_guard<std::mutex> lk(s->mu);
  if (s->sm_count > 0) return s->sm_count;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  s->sm_count = n;
  return n;
}

// One zeroed 8-byte ray-queue counter for a persistent march launch on `st`, on the CURRENT device.  Eager launches
// cycle a ring of kCounterRing slots (a slot is re-used 1,024 launches later, long after its kernel has drained on
// any stream); launches recorded into a CUDA graph take a slot from a second region that is never recycled, so that
// the address baked into the graph is private to it.
int nrt_next_counter(cudaStream_t st, unsigned long long** out) {
  NrtDeviceState* s = nrt_device_state();
  NRT_REQUIRE(s != nullptr, "no current CUDA device (or device index >= %d)", NRT_MAX_DEVICES);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  NRT_CUDA(cudaStreamIsCapturing(st, &cap));
  {
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->counters == nullptr) {
      NRT_REQUIRE(cap == cudaStreamCaptureStatusNone,
                  "the first march launch on a device cannot happen inside a CUDA-graph capture (run one eager step first)");
      NRT_CUDA(cudaMalloc(&s->counters, 2 * NrtDeviceState::kCounterRing * sizeof(unsigned long long)));
    }
    if (cap == cudaStreamCaptureStatusNone) {
      *out = s->counters + (s->counter_next++ % NrtDeviceState::kCounterRing);
    } else {
      NRT_REQUIRE(s->capture_next < NrtDeviceState::kCounterRing, "more than %u march launches captured into CUDA graphs",
                  NrtDeviceState::kCounterRing);
      *out = s->counters + NrtDeviceState::kCounterRing + s->capture_next++;
    }
  }
  NRT_CUDA(cudaMemsetAsync(*out, 0, sizeof(unsigned long long), st));
  return NRT_OK;
}

// grow-only device scratch `slot` of the current device; the caller holds s->host_mu for the duration of its use
int nrt_host_scratch(NrtDeviceState* s, int slot, size_t bytes, void** out) {
  if (s->host_ws_bytes[slot] < bytes) {
    if (s->host_ws[slot]) NRT_CUDA(cudaFree(s->host_ws[slot]));
    s->host_ws[slot] = nullptr; s->host_ws_bytes[slot] = 0;
    NRT_CUDA(cudaMalloc(&s->host_ws[slot], bytes));
    s->host_ws_bytes[slot] = bytes;
  }
  *out = s->host_ws[slot];
  return NRT_OK;
}

extern "C" int nrt_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  NRT_CUDA(cudaGetDevice(&dev));
  int n = 0, maj = 0, min = 0;
  NRT_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  NRT_CUDA(cudaDeviceGetAttribute(&maj, cudaDevAttrComputeCapabilityMajor, dev));
  NRT_CUDA(cudaDeviceGetAttribute(&min, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm_count) *sm_count = n;
  if (cc_major) *cc_major = maj;
  if (cc_minor) *cc_minor = min;
  return NRT_OK;
}

static int mlp_shape(const nrt_mlp_t* m, MlpDev* d) {
  NRT_REQUIRE(m != nullptr, "mlp descriptor is NULL");
  NRT_REQUIRE(m->in_size >= 1 && m->in_size <= 256, "mlp.in_size %d out of range", m->in_size);
  NRT_REQUIRE(m->latent_size >= 0 && m->latent_size <= 256, "mlp.latent_size %d out of range", m->latent_size);
  NRT_REQUIRE(m->freqs >= 0 && m->freqs <= 256, "mlp.freqs %d out of range", m->freqs);
  NRT_REQUIRE(m->num_layers >= 1 && m->num_layers <= NRT_MAX_LAYERS, "mlp.num_layers %d out of range [1,%d]",
              m->num_layers, NRT_MAX_LAYERS);
  NRT_REQUIRE(m->skip >= 1, "mlp.skip must be >= 1");
  NRT_REQUIRE(m->out_size >= 1 && m->out_size <= 256, "mlp.out_size %d out of range", m->out_size);
  NRT_REQUIRE(m->hidden >= 1, "mlp.hidden must be positive");
  NRT_REQUIRE(m->act == NRT_ACT_LEAKY_RELU || m->act == NRT_ACT_SOFTPLUS, "mlp.act %d unknown", m->act);
  d->in_size = m->in_size; d->latent = m->latent_size; d->freqs = m->freqs; d->hidden = m->hidden;
  d->L = m->num_layers; d->skip = m->skip; d->out = m->out_size; d->act = m->act;
  d->dim_p = m->in_size + 2 * m->freqs + m->latent_size;
  d->n_lin = m->num_layers + 2;
  d->skip_mask = 0;
  int off = 0;
  for (int li = 0; li < d->n_lin; ++li) {
    int K, N;
    if (li == 0) { K = d->dim_p; N = d->hidden; }
    else if (li == d->n_lin - 1) { K = d->hidden; N = d->out; }
    else {
      const int i = li - 1;
      const bool sk = (i % d->skip) == 0 && i != d->L - 1;   // neural_blocks.py:45-49,82
      if (sk) d->skip_mask |= (1u << i);
      K = d->hidden + (sk ? d->dim_p : 0); N = d->hidden;
    }
    d->K[li] = K; d->N[li] = N;
    d->w_off[li] = off; off += K * N;
    d->b_off[li] = off; off += N;
  }
  d->basis = m->basis; d->params = m->params;
  return off;
}

extern "C" int64_t nrt_mlp_param_count(const nrt_mlp_t* m) {
  MlpDev d;
  int n = mlp_shape(m, &d);
  return (int64_t)n;
}

int nrt_build_mlp_dev(const nrt_mlp_t* m, MlpDev* out) {
  int n = mlp_shape(m, out);
  if (n < 0) return n;
  NRT_REQUIRE(m->params != nullptr, "mlp.params is NULL");
  NRT_REQUIRE(m->freqs == 0 || m->basis != nullptr, "mlp.basis is NULL");
  NRT_REQUIRE(((uintptr_t)m->params & 15) == 0, "mlp.params must be 16-byte aligned");
  return NRT_OK;
}

int nrt_build_sdf_dev(const nrt_sphere_sdf_t* s, SdfDev* out) {
  NRT_REQUIRE(s != nullptr, "sdf descriptor is NULL");
  NRT_REQUIRE(s->n >= 1, "sdf.n must be >= 1");
  NRT_REQUIRE(s->centers && s->radii && s->tfs, "sdf sphere parameters are NULL");
  out->n = s->n; out->centers = s->centers; out->radii = s->radii; out->tfs = s->tfs;
  int rc = nrt_build_mlp_dev(&s->shift, &out->mlp);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(out->mlp.in_size == 3 && out->mlp.latent == 0 && out->mlp.out == 1,
              "sdf.shift must be a 3 -> 1 MLP without latent");
  return NRT_OK;
}

// ---- launch accounting and optional CUDA-event timing of every kernel launch ----------------
#include <vector>
static const char* kTagNames[TAG_COUNT] = {
    "mlp_fwd_f32", "sdf_eval_f32", "sdf_march_f32", "sdf_shadow_f32", "sdf_min_scan_f32", "nerfle_fused_f32",
    "composite_fwd", "composite_bwd", "mlp_tc_nerf_first", "mlp_tc_nerf_second", "mlp_tc_generic", "mlp_tc_pack",
    "stratified_ts", "sample_pdf", "merge_composite", "mlp_bwd_f32", "sdf_value_grad_f32", "shade",
    "sdf_eval_tc", "sdf_march_tc", "sdf_shadow_tc", "sdf_min_scan_tc", "mlp_tc_train_fwd", "mlp_tc_dgrad",
    "mlp_tc_wgrad", "mlp_tc_wide", "camera_rays", "merge_ts", "composite_ts_fwd", "composite_ts_bwd"};
static std::mutex g_prof_mu;
static long long g_launches[TAG_COUNT] = {0};
static bool g_prof_on = false;
struct ProfRec { cudaEvent_t a, b; int tag; };
static std::vector<ProfRec> g_prof_recs;
static std::vector<cudaEvent_t> g_prof_pool;

static cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
void nrt_prof_begin(int tag, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_launches[tag]++;
  if (!g_prof_on) return;
  ProfRec r; r.a = prof_event(); r.b = prof_event(); r.tag = tag;
  cudaEventRecord(r.a, st);
  g_prof_recs.push_back(r);
}
void nrt_prof_end(int tag, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!g_prof_on) return;
  for (size_t i = g_prof_recs.size(); i-- > 0;)
    if (g_prof_recs[i].tag == tag) { cudaEventRecord(g_prof_recs[i].b, st); break; }
}
extern "C" int nrt_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  return NRT_OK;
}
extern "C" int nrt_profile_num_tags(void) { return TAG_COUNT; }
extern "C" const char* nrt_profile_tag_name(int tag) { return (tag >= 0 && tag < TAG_COUNT) ? kTagNames[tag] : ""; }
// Synchronises the recorded events and returns, per tag, the summed device time (ms) of the launches
// recorded since the last collect and the number of launches since the last collect.  Resets both.
extern "C" int nrt_profile_collect(int n_tags, double* ms_by_tag, long long* launches_by_tag) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int t = 0; t < n_tags && t < TAG_COUNT; ++t) {
    if (ms_by_tag) ms_by_tag[t] = 0.0;
    if (launches_by_tag) { launches_by_tag[t] = g_launches[t]; }
    g_launches[t] = 0;
  }
  for (auto& r : g_prof_recs) {
    float ms = 0.0f;
    if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      if (ms_by_tag && r.tag < n_tags) ms_by_tag[r.tag] += ms;
    }
    g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b);
  }
  g_prof_recs.clear();
  return NRT_OK;
}
