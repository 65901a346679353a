/* nrt_b200.h -- C ABI of libnrt_b200.so, the B200 (sm_100a) native per-ray hot path of
 * prashantraina/neural_raytracing.
 *
 * The reference has NO native/FFI boundary on this path: it is eager PyTorch
 * (SURVEY.md section 8b).  The boundary a maintainer binds is therefore the set of
 * Python call sites listed next to each entry point below; INTEGRATION.md shows the
 * ctypes / torch.library stub for each.  Conventions:
 *
 *   - plain C: pointers + sizes, no torch types.  Every pointer is a DEVICE pointer
 *     (fp32 unless stated) except `nrt_*_host` entry points, which take HOST buffers and do
 *     the H2D/D2H copies themselves (used for the end-to-end benchmark leg).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  All work
 *     is enqueued on it; no entry point synchronises the host unless documented.
 *   - return value: 0 on success, a negative NRT_E_* code otherwise;
 *     nrt_last_error() returns a human readable message for the calling thread.
 *   - no CPU fallback exists: without a CUDA device every compute entry point returns
 *     NRT_E_CUDA.
 *
 * Layouts
 *   rays      [R,6]  (origin xyz, direction xyz), row-major, as the reference's
 *                    rays[N,W,H,B,6] flattened (cameras.py:53, renderer/cameras.py:575).
 *   MLP weights: one flat fp32 blob per SkipConnMLP ("packed f32"), see nrt_mlp_t.
 */
#ifndef NRT_B200_H_
#define NRT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRT_ABI_VERSION 1

/* error codes */
#define NRT_OK 0
#define NRT_E_INVALID (-1)  /* bad argument / unsupported shape */
#define NRT_E_CUDA (-2)     /* CUDA runtime error (message has the cudaError string) */
#define NRT_E_UNSUPPORTED (-3)

/* hidden activation (neural_blocks.py:26 default leaky_relu; sdfs.py:29 softplus) */
#define NRT_ACT_LEAKY_RELU 0
#define NRT_ACT_SOFTPLUS 1
/* output activation applied by the caller sites (bsdfs.py:536,635; scene.py:315;
 * nerf.py:203,60) -- fused into the epilogue */
#define NRT_OUT_NONE 0
#define NRT_OUT_SIGMOID 1
#define NRT_OUT_SOFTPLUS 2
#define NRT_OUT_TANH 3

/* arithmetic mode of the MLP contraction */
#define NRT_PREC_F32 0  /* fp32 FMA, fixed k-sequential order: bit-exact vs oracle/c */
#define NRT_PREC_F16 1  /* tcgen05 kind::f16, fp16 operands, fp32 accumulate in TMEM   */
#define NRT_PREC_BF16 2 /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM   */

#define NRT_MAX_LAYERS 20

/* One SkipConnMLP (pytorch3d/pathtracer/neural_blocks.py:12-86).
 *
 * dim_p = in_size + 2*freqs + latent_size.  Linear layers in evaluation order:
 *   index 0          init   : K = dim_p,                       N = hidden
 *   index 1..L       layers : K = hidden (+dim_p if (i%skip)==0 && i!=L-1), N = hidden
 *   index L+1        out    : K = hidden,                      N = out_size
 * `params` is the packed-f32 blob: for each linear layer in that order, W^T stored
 * row-major as [K][N] (so element (k,n) = torch weight[n][k]) followed by bias[N].
 * For skip layers k runs over [hidden activations | encoding] exactly as
 * torch.cat([x, init], -1) does (neural_blocks.py:83).
 * `basis` is basis_p [in_size][freqs] row-major (utils.py:33-36).
 * `params_tc` is the optional tensor-core blob produced by nrt_mlp_pack_tc (NULL when
 * only NRT_PREC_F32 is used). */
typedef struct nrt_mlp {
  int32_t in_size;
  int32_t latent_size;
  int32_t freqs;
  int32_t hidden;
  int32_t num_layers;
  int32_t skip;
  int32_t out_size;
  int32_t act;
  const float* basis;
  const float* params;
  const void* params_tc;
} nrt_mlp_t;

/* SphereSDF (pytorch3d/pathtracer/shapes/sdfs.py:16-46): smooth-min (k=32, clamp 1e-4,
 * utils.py:385-387) of n affine-warped spheres plus the residual MLP `shift`. */
typedef struct nrt_sphere_sdf {
  int32_t n;
  const float* centers; /* [n,3]   */
  const float* radii;   /* [n]     */
  const float* tfs;     /* [n,3,3] (identity is added inside, sdfs.py:39) */
  nrt_mlp_t shift;
} nrt_sphere_sdf_t;

/* ---- library ------------------------------------------------------------------------ */
int nrt_abi_version(void);
const char* nrt_last_error(void);
/* number of SMs / compute capability of the current device; NRT_E_CUDA if none. */
int nrt_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- launch accounting / per-kernel timing (used by bench.py for `roofline` and `gpu_launches`) -- */
/* When enabled every kernel launch of the library is bracketed by CUDA events on its stream. */
int nrt_profile_enable(int on);
int nrt_profile_num_tags(void);
const char* nrt_profile_tag_name(int tag);
/* per tag: summed device ms of the launches recorded since the last collect (needs enable) and the
 * number of launches since the last collect (always counted).  Synchronises the events; resets. */
int nrt_profile_collect(int n_tags, double* ms_by_tag, long long* launches_by_tag);

/* ---- packed parameter sizes --------------------------------------------------------- */
/* number of floats in the packed-f32 blob of `m` (pointers in m may be NULL). */
int64_t nrt_mlp_param_count(const nrt_mlp_t* m);
/* bytes of the tensor-core blob for `prec` (NRT_PREC_F16 / NRT_PREC_BF16). */
int64_t nrt_mlp_tc_blob_bytes(const nrt_mlp_t* m, int prec);
/* builds the tensor-core blob (UMMA canonical K-major fp16/bf16 tiles + fp32 biases) from
 * m->params on the device. */
int nrt_mlp_pack_tc(const nrt_mlp_t* m, int prec, void* blob_out, void* stream);

/* ---- a2: SkipConnMLP.forward (neural_blocks.py:75-86; fourier2 utils.py:37-40) ---- */
/* x [M,in_size], latent [M,latent_size] or NULL, out [M,out_size].  out_act is applied to
 * the result.  If `acts` is non-NULL it receives the post-activation layer inputs needed by
 * nrt_mlp_backward ([M, hidden*(num_layers+1)] floats). */
int nrt_mlp_forward(const nrt_mlp_t* m, int prec, int out_act, const float* x,
                    const float* latent, int64_t M, float* out, float* acts, void* stream);
/* reverse mode of the above.  g_out [M,out_size] is the gradient w.r.t. the *activated*
 * output `out` (which must be passed back); params_nk holds the same weights in nn.Linear's
 * native layout (per layer W [N][K], evaluation order, no biases) so the data-gradient GEMM
 * streams rows over n; g_params (packed-f32 layout, ACCUMULATED into with atomics: zero it
 * first); g_x [M,in_size] / g_latent [M,latent] may be NULL. */
int nrt_mlp_backward(const nrt_mlp_t* m, int out_act, const float* x, const float* latent,
                     int64_t M, const float* out, const float* acts, const float* g_out,
                     const float* params_nk, float* g_params, float* g_x, float* g_latent,
                     void* stream);

/* ---- a2 (training): SkipConnMLP forward + backward on the tensor cores ---------------- */
/* What torch.autograd does for neural_blocks.py:75-86 in the reference's training loops (nerfle.py:113-116,
 * training_utils.py:211-260), as three tcgen05 kernels: a forward that saves its activations as 16-bit tiles,
 * the fused data-gradient chain, and the weight-gradient kernel.  prec = NRT_PREC_F16 (default; gradients are
 * loss-scaled on the device by a power of two taken from max|g_out|) or NRT_PREC_BF16; fp32 accumulation.
 * Instantiated for NeRFLE.first (3->65, 5x128), NeRFLE.second (70 / 115 -> 3, 8x64), NeuralBSDF.mlp (3->3, 6x96), the
 * occlusion MLP (5->1, 8x64), SphereSDF.shift (3->1, 8x128 softplus; no g_x) and the 256-wide nets (sp_var_fn 4 / 8 / 16
 * bases, LightField; streamed weights).
 *   workspace: nrt_mlp_train_tc_workspace_bytes(m, M) bytes, 256-byte aligned, must stay untouched between the
 *              forward and the backward call of the same batch;
 *   m->params_tc: the nrt_mlp_pack_tc blob of the same prec;
 *   dgrad_blob: transposed weights, nrt_mlp_pack_tc_dgrad (need_x = 1 adds the rows needed for g_x);
 *   out [M,out_size]: the ACTIVATED output of the forward; g_out: gradient w.r.t. it;
 *   g_params: packed-f32 layout, ACCUMULATED into (zero it first); g_x [M,in_size] or NULL. */
int64_t nrt_mlp_train_tc_workspace_bytes(const nrt_mlp_t* m, int64_t M);
int64_t nrt_mlp_tc_dgrad_blob_bytes(const nrt_mlp_t* m, int need_x);
int nrt_mlp_pack_tc_dgrad(const nrt_mlp_t* m, int prec, int need_x, void* blob_out, void* stream);
int nrt_mlp_forward_train_tc(const nrt_mlp_t* m, int prec, int out_act, const float* x, int64_t M, float* out,
                             void* workspace, size_t workspace_bytes, void* stream);
int nrt_mlp_backward_tc(const nrt_mlp_t* m, int prec, int out_act, int64_t M, const float* out, const float* g_out,
                        const void* dgrad_blob, void* workspace, size_t workspace_bytes, float* g_params,
                        float* g_x, void* stream);

/* ---- a18 (training): both NeRFLE MLPs of nerf.py:175-214 under autograd, fused --------------------------------- */
/* Forward: rays [R,6], ts [S] (the shared sample distances), light_code [n_views, light_dim] (3: point-light location,
 * 48: environment code), view_of_ray [R] or NULL -> sigma [S,R] (pre-relu density) and rgb [S,R,3] (sigmoid), both
 * SAMPLE-major like the reference, ready for nrt_composite_forward/backward.  The 64-d latent goes from the first to
 * the second MLP through `latent` (ceil(S*R/128)*128*64 floats, 16-byte aligned; fp32 so that the second MLP's Fourier phases,
 * sigma = 32 times its inputs, keep fp32 accuracy through a hi+lo split of the phase GEMM).
 * ws_first / ws_second: nrt_mlp_train_tc_workspace_bytes(first|second, S*R) bytes each, kept until the backward.
 * Backward: g_sigma [S,R], g_rgb [S,R,3] (from nrt_composite_backward) -> g_params_first / g_params_second (packed-f32
 * layout, ACCUMULATED into: zero them first); g_latent_scratch: ceil(S*R/128)*128*64 floats of scratch. */
int nrt_nerfle_train_forward(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                             int64_t R, const float* ts, int S, const float* light_code, int light_dim,
                             const int32_t* view_of_ray, float* sigma, float* rgb, float* latent,
                             void* ws_first, size_t ws_first_bytes, void* ws_second, size_t ws_second_bytes,
                             void* stream);
/* The same forward with per-sample distances ts [S,R] (sample m = s * R + ray at distance ts[m]), e.g. the merged
 * coarse + fine distances of nrt_nerfle_sample_hierarchical.  Extension: the reference uses one shared ts (nerf.py:178).
 * The backward is nrt_nerfle_train_backward unchanged (it needs no distances). */
int nrt_nerfle_train_forward_ts(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                                int64_t R, const float* ts, int S, const float* light_code, int light_dim,
                                const int32_t* view_of_ray, float* sigma, float* rgb, float* latent,
                                void* ws_first, size_t ws_first_bytes, void* ws_second, size_t ws_second_bytes,
                                void* stream);
int nrt_nerfle_train_backward(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, int64_t R, int S,
                              int light_dim, const float* rgb, const float* g_sigma, const float* g_rgb,
                              const void* dgrad_blob_first, const void* dgrad_blob_second, void* ws_first,
                              void* ws_second, float* g_latent_scratch, float* g_params_first,
                              float* g_params_second, void* stream);

/* ---- a3: SphereSDF.forward (sdfs.py:41-46) ------------------------------------------- */
int nrt_sdf_eval(const nrt_sphere_sdf_t* s, int prec, const float* p, int64_t M, float* out,
                 void* stream);
/* a6: value and analytic d(sdf)/dp (replaces SDF.autograd_diff, sdfs.py:184-197). */
int nrt_sdf_value_grad(const nrt_sphere_sdf_t* s, const float* p, int64_t M, float* value,
                       float* grad, void* stream);
/* a6 + a22 (training): the sphere set of SphereSDF alone (sdfs.py:37-45 without `shift`): value [K] and its gradient
 * grad [K,3] = d value / d p (grad may be NULL), and the reverse pass of both outputs into centers [n,3] / radii [n] /
 * tfs [n,3,3] (g_* ACCUMULATED into: zero them first; g_value [K] or NULL, g_grad [K,3] or NULL).  Replaces the torch
 * expression + autograd.grad(create_graph=True) + double backward of SDF.autograd_diff (sdfs.py:184-197) for this part
 * of the SDF; p carries no gradient. */
int nrt_sphere_set_forward(int n, const float* centers, const float* radii, const float* tfs, const float* p, int64_t K,
                           float* value, float* grad, void* stream);
int nrt_sphere_set_backward(int n, const float* centers, const float* radii, const float* tfs, const float* p, int64_t K,
                            const float* g_value, const float* g_grad, float* g_centers, float* g_radii, float* g_tfs,
                            void* stream);
/* a6 + a22 (training): the same forward-mode evaluation for a bare SkipConnMLP with in_size 3 (SphereSDF.shift),
 * keeping what the reverse pass needs, and that reverse pass.  Together they replace the create_graph autograd of
 * SDF.autograd_diff (sdfs.py:184-197) and the double backward that loss.backward() runs through it for
 * eikonal_loss (utils.py:294) and the shading normals (sdfs.py:156-159).
 *   forward : p [M,3] -> value [M,out], jac [M,out,3] = d value / d p;  acts (optional) receives the post-activation
 *             states of the four-column network, [(num_layers+1)*hidden][4*M] floats.
 *   backward: g_value [M,out], g_jac [M,out,3] -> g_params (packed-f32 layout, ACCUMULATED into: zero it first).
 *             params_nk as for nrt_mlp_backward.  p carries no gradient (the march is no_grad in the reference). */
int nrt_mlp_value_jac_forward(const nrt_mlp_t* m, const float* p, int64_t M, float* value, float* jac,
                              float* acts, void* stream);
int nrt_mlp_value_jac_backward(const nrt_mlp_t* m, const float* p, int64_t M, const float* acts,
                               const float* g_value, const float* g_jac, const float* params_nk,
                               float* g_params, void* stream);
/* The same pair on the tensor cores (tcgen05, 16-bit operands, fp32 accumulation), for SphereSDF.shift (3 -> 1, 8 x 128,
 * softplus, 32 frequencies; sdfs.py:23-31): four rows per point (value, d/dp_0..2) through the streamed-weight forward
 * with the coupled activation a_v = softplus(z_v), a_t = sigmoid(z_v) z_t, saved as 16-bit tiles; the reverse pass is
 * a dgrad chain with g_z_v = s g_a_v + (1 - s) sum_t g_a_t a_t, g_z_t = s g_a_t and the shared weight-gradient kernel.
 *   K points; p [K,3] -> value [K], jac [K,3];  workspace: nrt_mlp_value_jac_tc_workspace_bytes(m, K) bytes, 256-byte
 *   aligned, untouched between the two calls;  m->params_tc / dgrad_blob (need_x = 0): as for nrt_mlp_forward_train_tc;
 *   g_value [K] or NULL, g_jac [K,3] -> g_params (packed-f32 layout, ACCUMULATED into). */
int64_t nrt_mlp_value_jac_tc_workspace_bytes(const nrt_mlp_t* m, int64_t K);
int nrt_mlp_value_jac_forward_tc(const nrt_mlp_t* m, int prec, const float* p, int64_t K, float* value, float* jac,
                                 void* workspace, size_t workspace_bytes, void* stream);
int nrt_mlp_value_jac_backward_tc(const nrt_mlp_t* m, int prec, int64_t K, const float* g_value, const float* g_jac,
                                  const void* dgrad_blob, void* workspace, size_t workspace_bytes, float* g_params,
                                  void* stream);

/* ---- a4: SDF.intersect march loop (sdfs.py:111-131) ---------------------------------- */
/* depth [R] (final `depths`), hit [R] uint8 (`out_active`).  `active` (optional, [R]
 * uint8) lets the caller skip rays whose result it will mask anyway (skipped rays report
 * depth 0 / hit 0, resp. not_blocked 1).  steps_done (optional, device
 * uint64) accumulates the number of SDF samples actually evaluated (compaction skips
 * finished rays; the reference evaluates R*max_steps). */
int nrt_sdf_sphere_trace(const nrt_sphere_sdf_t* s, int prec, const float* rays,
                         const uint8_t* active, int64_t R, float epsilon, int max_steps,
                         float max_t, float* depth, uint8_t* hit,
                         unsigned long long* steps_done, void* stream);
/* ---- a7: SDF.intersect_test shadow march (sdfs.py:162-181) -------------------------- */
/* max_t [R] per ray; not_blocked [R] uint8. */
int nrt_sdf_shadow_test(const nrt_sphere_sdf_t* s, int prec, const float* rays,
                        const float* max_t, const uint8_t* active, int64_t R, float epsilon,
                        int max_steps, uint8_t* not_blocked, unsigned long long* steps_done,
                        void* stream);
/* ---- a5: SDF.throughput min-along-ray scan (sdfs.py:232-249) ------------------------- */
/* Scans t_i = fl32(step*(i)) for i = 0..n_steps (step given in double like the python
 * float), strict-< running argmin.  Outputs best_idx [R] int32, best_pos [R,3]
 * (= o + fl32(fl32(idx)*fl32(step)) * d, sdfs.py:247-248) and min_val [R]. */
int nrt_sdf_min_scan(const nrt_sphere_sdf_t* s, int prec, const float* rays, int64_t R,
                     double step, int n_steps, int32_t* best_idx, float* best_pos,
                     float* min_val, void* stream);

/* ---- a19: NeRF alpha compositing (nerf.py:206-213 / :66-74) -------------------------- */
/* Sample-major like the reference: sigma_raw [S,R] (pre-relu density), rgb [S,R,3],
 * ts [S]; out [R,3].  Replicates the reference quirks: alpha from absolute t, the
 * roll-by-one, and the last sample's transmittance forced to 1. */
int nrt_composite_forward(const float* sigma_raw, const float* rgb, const float* ts, int S,
                          int64_t R, float* out, void* stream);
int nrt_composite_backward(const float* sigma_raw, const float* rgb, const float* ts, int S,
                           int64_t R, const float* g_out, float* g_sigma_raw, float* g_rgb,
                           void* stream);
/* The same pair with per-sample distances ts [S,R] (sample s of ray r at ts[s*R + r]; the hierarchical samples of
 * nrt_nerfle_sample_hierarchical), keeping every quirk above (nerf.py:205-213): alpha from the absolute t, the
 * roll-by-one that gives sample 0 the total transmittance, the last transmittance forced to 1, and a backward built
 * from suffix recurrences without dividing by the clamped 1 - alpha.  With ts[s*R + r] = ts_shared[s] the results
 * equal nrt_composite_forward / _backward bit for bit. */
int nrt_composite_forward_ts(const float* sigma_raw, const float* rgb, const float* ts, int S,
                             int64_t R, float* out, void* stream);
int nrt_composite_backward_ts(const float* sigma_raw, const float* rgb, const float* ts, int S,
                              int64_t R, const float* g_out, float* g_sigma_raw, float* g_rgb,
                              void* stream);

/* ---- a18: NeRFLE.forward fused volumetric render (nerf.py:175-214) ------------------- */
/* rays [R,6]; ts [S] sample distances (the reference uses linspace(0, 2+U*0.1, 64));
 * light_code [n_views, light_dim] with light_dim = second.in_size - 64 - 3 (3 = light
 * location, nerf.py:197; 48 = envmap code, :184-195); view_of_ray [R] int32 selects the
 * row (NULL = row 0 for all).  out rgb [R,3].  Optional stratified/hierarchical sampling
 * is selected through nrt_nerf_sampling_t (extension; not in the reference). */
typedef struct nrt_nerf_sampling {
  int32_t n_coarse;     /* S for the first pass                                      */
  int32_t n_fine;       /* 0 = reference behaviour (single pass, shared ts)          */
  float t_near, t_far;  /* used when ts == NULL                                      */
  uint64_t jitter_seed; /* 0 = no stratified jitter                                  */
} nrt_nerf_sampling_t;
int nrt_nerfle_render(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                      const float* rays, int64_t R, const float* ts,
                      const nrt_nerf_sampling_t* sampling, const float* light_code,
                      int light_dim, const int32_t* view_of_ray, float* out_rgb,
                      void* workspace, size_t workspace_bytes, void* stream);
size_t nrt_nerfle_render_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                   int64_t R, const nrt_nerf_sampling_t* sampling);
/* Hierarchical sample distances for TRAINING on what nrt_nerfle_render renders (extension of nerf.py:178, which uses
 * one shared uniform ts; the render's hierarchical mode is pinned by oracle/port.py): the first half of that render --
 * stratified coarse distances in [t_near, t_far), the coarse pass keeping per-sample sigma (at `prec`), inverse-CDF
 * resampling of n_fine distances -- then the coarse and fine lists merged in ascending order (coarse first on ties, as
 * the render's merged compositing orders them) into ts_out [n_coarse + n_fine, R], SAMPLE-major (m = s * R + ray, the
 * layout of nrt_nerfle_train_forward_ts and nrt_composite_forward_ts).  n_fine = 0 is the render's single stratified
 * pass: ts_out is the stratified distances, no coarse pass runs.  Needs n_coarse >= 1 (>= 3 when n_fine > 0),
 * n_coarse + n_fine <= NRT_MAX_HIER_SAMPLES and t_near < t_far.
 * seed_dev: a device uint64 read by the kernels in place of sampling->jitter_seed (NULL: use jitter_seed), so that a
 * CUDA-graph replay draws new jitter after the caller advanced it; 0 means no jitter (bin centres, u = 0.5).
 * Jitter is hashed with the ray's index in the call, so equal seeds give the distances of nrt_nerfle_render.
 * workspace: nrt_nerfle_sample_hierarchical_workspace bytes (256-byte aligned). */
#define NRT_MAX_HIER_SAMPLES 512
size_t nrt_nerfle_sample_hierarchical_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                                int64_t R, const nrt_nerf_sampling_t* sampling);
int nrt_nerfle_sample_hierarchical(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays,
                                   int64_t R, const nrt_nerf_sampling_t* sampling, const uint64_t* seed_dev,
                                   const float* light_code, int light_dim, const int32_t* view_of_ray,
                                   float* ts_out, void* workspace, size_t workspace_bytes, void* stream);
/* Host-buffer variant: copies rays H2D, renders, copies rgb D2H, synchronises. */
int nrt_nerfle_render_host(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                           const float* rays_host, int64_t R, const float* ts_host, int S,
                           const nrt_nerf_sampling_t* sampling, const float* light_code,
                           int light_dim, float* out_rgb_host, void* stream);

/* ---- a21 / f4: ray generators on the device, and the camera-driven whole-frame render ------------------------------
 * Pixel -> ray [origin(3) | unit direction(3)] for the three cameras the scripts use:
 *   NRT_CAM_NERF  NeRFCamera.sample_positions            pathtracer/cameras/cameras.py:23-54
 *   NRT_CAM_DTU   DTUCamera.sample_positions (+ lift)    pathtracer/cameras/cameras.py:132-147, 156-192
 *   NRT_CAM_FOV   FoVPerspectiveCameras.sample_positions renderer/cameras.py:539-575
 * The rays of one call form the reference's [n_views, nx, ny, bundle, 6] block: ray
 * r = ((view * nx + i) * ny + j) * bundle + b looks through pixel position (u, v) = (y0 + j, x0 + i), which is how
 * pathtrace lays out a tile (main.py:67-74: positions = stack([grid_y, grid_x])).  `positions`, when not NULL, replaces
 * that grid with explicit pixel positions [nx * ny * pos_per_pixel, 2] (the caller's jittered samples; pos_per_pixel is 1
 * or `bundle`); otherwise `jitter` > 0 perturbs the grid by (U - 0.5) * jitter with the library's counter hash (the
 * reference draws the same perturbation from torch's generator, cameras.py:35-37 / renderer/cameras.py:553-556).
 * All matrices are fp32 DEVICE pointers, so no host synchronisation is needed to render from a camera that lives on the GPU. */
#define NRT_CAM_NERF 0
#define NRT_CAM_DTU 1
#define NRT_CAM_FOV 2
typedef struct nrt_camera {
  int32_t kind;             /* NRT_CAM_*                                                                              */
  int32_t n_views;
  const float* a;           /* NERF: cam_to_world; DTU: pose; FOV: inverse of the full projection matrix (row vectors)   */
  const float* b;           /* DTU: intrinsics; FOV: camera centres [n_views,3] (row stride 3); NERF: unused (NULL)      */
  int32_t a_view_stride, a_row_stride;   /* in floats: 16 / 4 for [n,4,4], 12 / 4 for [n,3,4]                          */
  int32_t b_view_stride, b_row_stride;
  float focal;              /* NERF                                                                                  */
  float size;               /* the `size` pixel positions are normalised by (all three)                              */
  int32_t x0, y0, nx, ny;   /* pixel window                                                                          */
  int32_t bundle;           /* rays per pixel (NERF: 1)                                                              */
  int32_t pos_per_pixel;    /* rows of `positions` per pixel: 1 or bundle                                            */
  const float* positions;   /* optional explicit pixel positions, see above                                          */
  float jitter;             /* window-grid jitter amplitude in pixels (0 = pixel positions as they are)              */
  uint64_t jitter_seed;
} nrt_camera_t;
/* Rays r0 .. r0 + n - 1 of the block -> out_rays [n,6]; out_view [n] int32 = view of each ray, or NULL. */
int nrt_camera_rays(const nrt_camera_t* cam, int64_t r0, int64_t n, float* out_rays, int32_t* out_view,
                    void* stream);
/* f4: nrt_nerfle_render with the rays generated on the device inside the call (per 262,144-ray chunk, into the
 * workspace): replaces pathtrace's Python tile loop + sample_positions + integrator call for a volumetric shape
 * (main.py:57-88) by one library call per frame.  R = n_views * nx * ny * bundle; light_code row = the ray's view.
 * out_rgb [R,3] in the block order above, i.e. already the reference's [n_views, nx, ny(, bundle), 3] image. */
size_t nrt_nerfle_render_camera_workspace(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                          const nrt_camera_t* cam, const nrt_nerf_sampling_t* sampling);
int nrt_nerfle_render_camera(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                             const nrt_camera_t* cam, const float* ts, const nrt_nerf_sampling_t* sampling,
                             const float* light_code, int light_dim, float* out_rgb, void* workspace,
                             size_t workspace_bytes, void* stream);
/* Where nrt_nerfle_render_camera takes the rays of the 16-bit (tensor-core) passes from: 0 (default) = k_camera_rays writes each
 * chunk's rays into the workspace before the chunk's first pass; 1 = the MLP kernels compute every sample's ray from the camera
 * in their prologues (no ray array; bit-identical image; measured 2.5-3 % slower on B200, see DESIGN.md section 8).  Process-wide. */
int nrt_set_camera_rays_mode(int fused);
/* Host-image variant: nothing but the camera goes in, the image comes back to (pinned) host memory; synchronises. */
int nrt_nerfle_render_camera_host(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec,
                                  const nrt_camera_t* cam, const float* ts_host, int S,
                                  const nrt_nerf_sampling_t* sampling, const float* light_code, int light_dim,
                                  float* out_rgb_host, void* stream);

/* ---- a8/a9/a12/a14/a15/a16: shading glue as fused elementwise kernels ---------------- */
/* coordinate_system + to_local(-r_d) (interaction.py:9-27,38-41; sdfs.py:158-159).
 * normals [R,3] -> frame [R,3,3] (columns s,t,n as torch.stack(dim=-1)), wi [R,3]. */
int nrt_shading_frame(const float* normals, const float* rays, int64_t R, float* frame,
                      float* wi, void* stream);
/* to_local(frame, v) for arbitrary v [R,3]. */
int nrt_to_local(const float* frame, const float* v, int64_t R, float* out, void* stream);
/* param_rusin2 (utils.py:233-258): a = first argument (`wo` in the source, called with
 * it.wi), b = second. out [R,3]. */
int nrt_param_rusin2(const float* a, const float* b, int64_t R, float* out, void* stream);

/* ---- a8-a16 fused: the shading glue of Direct.sample (integrators/integrators.py:156-206) on the K COMPACTED hit rays,
 *      forward and backward, as three elementwise stages around the MLP evaluations (SURVEY 8b(8) `shade_direct`).
 *      All arrays are fp32 device pointers of K rows; gradients of per-hit inputs are OVERWRITTEN, gradients of shared
 *      parameters (g_amp, g_coef, g_sig_color, g_refl, g_cond_*) are ACCUMULATED into (zero them first). ------------ */
#define NRT_MAX_BSDFS 16
#define NRT_LIGHT_POINT 0   /* PointLights.sample_direction  lights/lights.py:89-110 */
#define NRT_LIGHT_FIELD 1   /* LightField.sample_direction   lights/lights.py:175-195 */
typedef struct nrt_light {
  int32_t mode;               /* NRT_LIGHT_POINT | NRT_LIGHT_FIELD */
  int32_t n_views;            /* point lights: rows of location / amp */
  const float* location;      /* [n_views,3] */
  const float* amp;           /* [n_views,3] = scale * normalize(intensity)              (lights.py:104) */
  const float* coef;          /* [3] const, linear, square, each already clamp(min=1e-6)  (lights.py:105-107) */
  const int32_t* view_of_hit; /* [K] row of location / amp per hit, or NULL (one view) */
  const float* v;             /* light field: MLP output at the hit points [K,3]          (lights.py:181) */
  const float* sig_color;     /* light field: sigmoid(color) [3]                          (lights.py:193) */
} nrt_light_t;
#define NRT_BSDF_NEURAL 0     /* NeuralBSDF.eval_and_pdf   bsdf/bsdfs.py:634-637 */
#define NRT_BSDF_DIFFUSE 1    /* Diffuse.eval_and_pdf      bsdf/bsdfs.py:108-118 */
#define NRT_BSDF_CONDUCTOR 2  /* Conductor.eval_and_pdf    bsdf/bsdfs.py:364-388 */
typedef struct nrt_blend {
  int32_t nb;                    /* children of ComposeSpatialVarying (bsdfs.py:482-540), <= NRT_MAX_BSDFS */
  int32_t kind[NRT_MAX_BSDFS];   /* NRT_BSDF_* per child, in the order of the sp_var logits */
  int32_t neural_act;            /* NeuralBSDF.act: 0 sigmoid, 1 softplus, 2 identity */
  int32_t diffuse_pre;           /* Diffuse.preproc: 0 identity, 1 x / pi, 2 softplus, 3 sigmoid */
} nrt_blend_t;
/* sdfs.py:152-159, interaction.py:9-41: raw_n [K,3] (d sdf / d p at the hits), p_hit [K,3], rays_hit [K,6] ->
 * n = normalize(raw_n, 1e-6), p_off = p_hit + eps5 * n, wi = to_local(frame(n), -r_d), frame [K,3,3] (or NULL). */
int nrt_shade_geom_forward(const float* raw_n, const float* p_hit, const float* rays_hit, int64_t K, float eps5,
                           float* n, float* p_off, float* wi, float* frame, void* stream);
/* g_n / g_p_off / g_wi (any may be NULL) -> g_raw_n [K,3]. */
int nrt_shade_geom_backward(const float* raw_n, const float* rays_hit, int64_t K, float eps5, const float* g_n,
                            const float* g_p_off, const float* g_wi, float* g_raw_n, void* stream);
/* lights.py:89-110 | 175-195, interaction.py:38-41, utils.py:233-258, 490-494: the light sample at every hit ->
 * d [K,3] world direction to the light, dist [K] (distance | light-field magnitude), wo = to_local(frame(n), d),
 * rusin = param_rusin2(wi, wo), e [K,3] emitter spectrum (before occlusion), elaz [K,2] = dir_to_elev_azim(d) or NULL. */
int nrt_shade_light_forward(const nrt_light_t* light, const float* n, const float* wi, const float* p_off, int64_t K,
                            float* d, float* dist, float* wo, float* rusin, float* e, float* elaz, void* stream);
/* g_wo / g_rusin / g_e / g_elaz (any may be NULL) -> g_n, g_wi, g_pv [K,3] (w.r.t. p_off for point lights, w.r.t. v for
 * the light field), and the reduced g_amp [n_views,3], g_coef [3] (point lights) or g_sig_color [3] (light field). */
int nrt_shade_light_backward(const nrt_light_t* light, const float* n, const float* wi, const float* p_off, int64_t K,
                             const float* g_wo, const float* g_rusin, const float* g_e, const float* g_elaz, float* g_n,
                             float* g_wi, float* g_pv, float* g_amp, float* g_coef, float* g_sig_color, void* stream);
/* bsdfs.py:515-536 + integrators.py:183-187: out [K,3] = (sum_b sigmoid(logits_b) * spectrum_b) * e * inv_samples with
 * logits [K,nb] (sp_var MLP output), neural_raw [n_neural,K,3] (NeuralBSDF MLP outputs before `act`), refl
 * [n_diffuse,3], cond_spec [3] = act(specular), cond_eta [1] = softplus(eta), e = emitter spectrum incl. occlusion. */
int nrt_shade_blend_forward(const nrt_blend_t* cfg, const float* logits, const float* neural_raw, const float* wi,
                            const float* wo, const float* e, const float* refl, const float* cond_spec,
                            const float* cond_eta, float inv_samples, int64_t K, float* out, void* stream);
int nrt_shade_blend_backward(const nrt_blend_t* cfg, const float* logits, const float* neural_raw, const float* wi,
                             const float* wo, const float* e, const float* refl, const float* cond_spec,
                             const float* cond_eta, float inv_samples, int64_t K, const float* g_out, float* g_logits,
                             float* g_neural, float* g_wi, float* g_wo, float* g_e, float* g_refl, float* g_cond_spec,
                             float* g_cond_eta, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NRT_B200_H_ */
