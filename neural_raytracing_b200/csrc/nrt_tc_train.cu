// Tensor-core TRAINING path of the fused SkipConnMLP (sm_100a): forward that saves its activations, the fused
// data-gradient chain and the weight-gradient kernel.  fp16 operands by default (the forward's rounding decides
// which leaky_relu kinks flip, and fp16 is 8x finer than bf16), fp32 accumulation in TMEM; the gradients are
// loss-scaled by a power of two derived from max|g_out| on the device so that they stay in fp16's normal range,
// and un-scaled when the weight gradients leave TMEM.  NRT_PREC_BF16 selects bf16 operands (scale still applied).
//
//   forward  (k_mlp_tc<.., SaveTiles>, tc_core.cuh): as inference, plus per 128-sample tile the activations a_l
//            (l = 0..L), the raw and the activated encoding as UMMA-canonical MN-major tiles (MN = feature,
//            K = sample; 16-byte vector stores per thread).
//   dgrad    (k_mlp_dgrad_tc): g_out -> dZ_L -> ... -> dZ_0 (-> dEnc -> g_x) with the TRANSPOSED weights resident
//            in shared memory; dZ_l never leaves the SM on its way to the next layer (TMEM operand), and is
//            saved once as a tile for the weight gradients.
//   wgrad    (k_mlp_wgrad_tc): per linear layer dW^T = dZ^T . [input | 1]: both operands are saved tiles pulled
//            into shared memory with one bulk copy each (2-stage ring), K' = samples, the accumulator
//            [N_out x (K_in + 16)] stays in TMEM over the CTA's whole sample range and is flushed once with
//            coalesced float atomics.  The "1" row of the activation tiles makes the bias gradient one more
//            accumulator column.
//
// Reference semantics: what torch.autograd computes for neural_blocks.py:75-86 (+ utils.py:37-40 for g_x).
#include "tc_train.cuh"

namespace tc {

template <int FMT>
__global__ void k_pack_dgrad(MlpDev m, Layout y, DLayout d, int needx, uint8_t* __restrict__ blob) {
  uint16_t* w = reinterpret_cast<uint16_t*>(blob);
  const int L = m.L, h = m.hidden;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < d.w_elems; idx += gridDim.x * blockDim.x) {
    int o = 0;
    while (o + 1 < d.n_ops && idx >= d.op_off[o + 1]) ++o;
    const int e = idx - d.op_off[o];
    const int N = d.opN[o];
    const int chunk = e / (N * 8), rem = e - chunk * (N * 8);
    const int n = rem / 8, k = chunk * 8 + (rem & 7);
    float v = 0.0f;
    if (o == 0) {
      if (k < m.out) v = m.params[m.w_off[m.n_lin - 1] + n * m.out + k];
    } else if (o <= L) {
      const int li = 1 + (L - o);
      if (n < h) v = m.params[m.w_off[li] + n * h + k];
      else { const int r = enc_ref_index(y, m.in_size, n - h); if (r >= 0) v = m.params[m.w_off[li] + (h + r) * h + k]; }
    } else if (o == L + 1) {
      const int r = enc_ref_index(y, m.in_size, n);
      if (r >= 0) v = m.params[m.w_off[0] + r * h + k];
    } else {
      if (n < m.in_size && k < m.freqs) v = m.basis[n * m.freqs + k];
    }
    (void)needx;
    w[idx] = Elem<FMT>::cvt(v);
  }
}

// ---------------------------------------------------------------------------------------------
// dgrad chain
// ---------------------------------------------------------------------------------------------
template <class NET, bool NEEDX>
struct DNet {
  static constexpr DLayout DY = make_dlayout(NET::IN, NET::LAT, NET::F, NET::H, NET::L, NET::SKIP, NET::OUT, NEEDX);
  static constexpr int H = NET::H, L = NET::L, KE = NET::KE, XR = NET::XR, FP = NET::FP, NOP = NET::NOP;
  static constexpr int MC = imax(H, NEEDX ? XR : 0);          // main fp32 accumulator columns
  static constexpr int EC = NEEDX ? KE : 0;                   // dEnc accumulator columns
  static constexpr int AC = imax(H, imax(NOP, FP)) / 2;       // 16-bit A operand columns
  static constexpr int COLS = MC + EC + AC;
  static constexpr int NSLOT = (2 * COLS <= 512) ? 2 : 1;
  static constexpr int STAGES = DY.n_ops;
  static constexpr int first_skip_op() {   // backward-order index of the first op that adds into dEnc (-1: none)
    for (int o = 1; o <= L; ++o) if (is_skip(L - o, NET::SKIP, L)) return o;
    return -1;
  }
  static constexpr int FIRST_E = first_skip_op();
  static_assert(COLS <= 512, "dgrad tile does not fit in TMEM");
  // split inputs ([x_hi | x_lo | x_hi | 0] in the raw-x segment): both halves see the same weight rows, so the gradient
  // w.r.t. x is the one of the x_hi columns (columns 0 .. IN-1, the only ones the final store reads)
  static_assert(!NEEDX || NET::LAT == 0, "input gradients: no latent");
  static_assert(NET::ACT == NRT_ACT_LEAKY_RELU, "tensor-core backward: leaky_relu networks");
  static_assert(DY.bytes + 1024 <= 227 * 1024, "transposed weights do not fit in shared memory");
};

template <class NET, class DN, int FMT, int ST>
__device__ __forceinline__ void issue_dstage(uint32_t sW_addr, uint32_t dM, uint32_t dE, uint32_t aA, uint64_t* done_bar) {
  constexpr DLayout D = DN::DY;
  constexpr int L = NET::L, H = NET::H;
  constexpr uint32_t N = (uint32_t)D.opN[ST];
  constexpr int kch = D.opK[ST] / 16;
  constexpr uint32_t lbo = N * 16;
  constexpr bool has_enc = (ST >= 1 && ST <= L) && (N > (uint32_t)H);   // skip layer with NEEDX
  constexpr bool to_e = (ST == L + 1);                                   // init layer: accumulate into dEnc
  constexpr uint32_t n_main = has_enc ? (uint32_t)H : N;
  constexpr uint32_t idesc_main = (1u << 4) | ((uint32_t)FMT << 7) | ((uint32_t)FMT << 10) | ((n_main >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  constexpr uint32_t n_enc = has_enc ? (N - (uint32_t)H) : 16u;
  constexpr uint32_t idesc_enc = (1u << 4) | ((uint32_t)FMT << 7) | ((uint32_t)FMT << 10) | ((n_enc >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  if (elect_one()) {
    const uint64_t bd0 = make_desc(sW_addr + (uint32_t)D.op_off[ST] * 2, lbo, 128);
#pragma unroll
    for (int kc = 0; kc < kch; ++kc) {
      const uint64_t bd = bd0 + (uint64_t)((kc * 2 * lbo) >> 4);
      if constexpr (to_e) {
        mma_ts(dE, aA + kc * 8, bd, idesc_main, (DN::FIRST_E >= 0 || kc > 0) ? 1u : 0u);
      } else {
        mma_ts(dM, aA + kc * 8, bd, idesc_main, kc > 0 ? 1u : 0u);
        if constexpr (has_enc)
          mma_ts(dE, aA + kc * 8, bd + (uint64_t)((H * 16) >> 4), idesc_enc, (ST != DN::FIRST_E || kc > 0) ? 1u : 0u);
      }
    }
    tc_commit(done_bar);
  }
  __syncwarp();
}
template <class NET, class DN, int FMT, int ST = 0>
__device__ __forceinline__ void issue_dstage_dyn(int st, uint32_t sW_addr, uint32_t dM, uint32_t dE, uint32_t aA, uint64_t* done_bar) {
  if constexpr (ST < DN::STAGES) {
    if (st == ST) issue_dstage<NET, DN, FMT, ST>(sW_addr, dM, dE, aA, done_bar);
    else issue_dstage_dyn<NET, DN, FMT, ST + 1>(st, sW_addr, dM, dE, aA, done_bar);
  }
}

template <class NET, class DN, class IO, int FMT>
__global__ void __launch_bounds__(kEpiThreads * 2 + 32 * DN::NSLOT, 1)
k_mlp_dgrad_tc(const uint8_t* __restrict__ blob, IO io, int64_t M, TrainWs ws) {
  using E = Elem<FMT>;
  constexpr DLayout D = DN::DY;
  constexpr int H = NET::H, L = NET::L, IN = NET::IN, F = NET::F, KE = NET::KE, NOP = NET::NOP, XR = NET::XR;
  constexpr int NSLOT = DN::NSLOT;
  constexpr bool NEEDX = DN::EC > 0;
  constexpr int NC = H / 32;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_w;
  __shared__ __align__(8) uint64_t bar_ready[2];
  __shared__ __align__(8) uint64_t bar_done[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int mma_id = warp - 8;                 // >= 0: MMA-issuing warp, one per tile slot (as in k_mlp_tc)
  const bool is_mma_warp = mma_id == 0;        // the one that owns the TMEM allocation and the weight load
  const int64_t ntiles = (M + 127) / 128;
  if (tid == 0) {
    mbar_init(&bar_w, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&bar_ready[s], kEpiThreads); mbar_init(&bar_done[s], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (is_mma_warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    if ((tid & 31) == 0) {
      mbar_expect_tx(&bar_w, (uint32_t)D.bytes);
      for (uint32_t off = 0; off < (uint32_t)D.bytes; off += 32768u)
        bulk_g2s(smem + off, blob + off, min(32768u, (uint32_t)D.bytes - off), &bar_w);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  mbar_wait(&bar_w, 0);

  if (mma_id >= 0) {
    // each MMA warp blocks on the `ready` barrier of its own slot and issues that slot's stages
    const uint32_t sW_addr = smem_u32(smem);
    const int slot = mma_id;
    if (slot < NSLOT) {
      const uint32_t base = tmem + slot * DN::COLS;
      uint32_t n_ready = 0;
      for (int64_t tile = (int64_t)blockIdx.x * NSLOT + slot; tile < ntiles; tile += (int64_t)gridDim.x * NSLOT) {
        for (int st = 0; st < DN::STAGES; ++st) {
          mbar_wait(&bar_ready[slot], n_ready & 1);
          n_ready++;
          tc_fence_after();
          issue_dstage_dyn<NET, DN, FMT>(st, sW_addr, base, base + DN::MC, base + DN::MC + DN::EC, &bar_done[slot]);
        }
      }
    }
  } else {
    const int slot = warp >> 2;
    const int lane_row = tid & 127;
    if (slot < NSLOT) {
      const uint32_t lane_off = ((uint32_t)((warp & 3) * 32)) << 16;
      const uint32_t base = tmem + slot * DN::COLS + lane_off;
      const uint32_t dM = base, dE = base + DN::MC, aA = base + DN::MC + DN::EC;
      uint32_t n_done = 0;
      const int64_t mpad = ntiles * 128;
      for (int64_t t0 = (int64_t)blockIdx.x * NSLOT; t0 < ntiles; t0 += (int64_t)gridDim.x * NSLOT) {
        const int64_t tile = t0 + slot;
        if (tile >= ntiles) break;
        const int64_t m = tile * 128 + lane_row;
        const bool valid = m < M;
        // ---- g_out -> A operand of the output layer's transposed GEMM (+ saved as a tile for wgrad) ----
        {
          float g[NET::OUT];
          if (valid) io.load_g(m, g);
          else {
#pragma unroll
            for (int j = 0; j < NET::OUT; ++j) g[j] = 0.0f;
          }
          uint32_t pk[NOP / 2];
#pragma unroll
          for (int j = 0; j < NOP / 2; ++j)
            pk[j] = E::pack(2 * j < NET::OUT ? g[2 * j] : 0.0f, 2 * j + 1 < NET::OUT ? g[2 * j + 1] : 0.0f);
          tmem_store<NOP / 2>(aA, pk);
          save_cols<NOP / 2>(tile_row_ptr(ws.gout, tile, NOP, lane_row), 0, pk);
          tc_wait_st();
          tc_fence_before();
          mbar_arrive(&bar_ready[slot]);
        }
        // ---- dA_l -> dZ_l = dA_l * act'(z_l), l = L .. 0 ----
#pragma unroll 1
        for (int i = 0; i <= L; ++i) {
          const int l = L - i;
          // leaky_relu'(z_l): the sign bits of a_l, written by the forward as one word per 32 features (coalesced over
          // the samples); loaded before the wait so that the latency hides under the layer's MMA
          uint32_t mask[NC];
#pragma unroll
          for (int c = 0; c < NC; ++c) mask[c] = __ldg(ws.masks + ((int64_t)(l * NC + c)) * mpad + m);
          mbar_wait(&bar_done[slot], n_done & 1); n_done++;
          tc_fence_after();
          uint16_t* zrow = tile_row_ptr(ws.dz, (int64_t)l * ntiles + tile, H, lane_row);
          uint32_t buf[2][32];
          TmemIO<32>::ld(dM, buf[0]);
          tc_wait_ld();
#pragma unroll
          for (int c = 0; c < NC; ++c) {
            if (c + 1 < NC) TmemIO<32>::ld(dM + 32 * (c + 1), buf[(c + 1) & 1]);
            uint32_t pk[16];
            dconvert32<FMT>(buf[c & 1], mask[c], pk);
            TmemIO<16>::st(aA + 16 * c, pk);
            save_cols<16>(zrow, 32 * c, pk);
            if (c + 1 < NC) tc_wait_ld();
          }
          if constexpr (NEEDX) {
            if (i == L) {
              // dEnc so far = sum over skip layers of d act(enc): through act' (sign of the raw encoding) in place
              const uint16_t* er = tile_row_ptr(ws.enc_raw, tile, KE + kTileRowsExtra, lane_row);
#pragma unroll
              for (int c = 0; c < KE / 16; ++c) {
                uint32_t e[16];
                TmemIO<16>::ld(dE + 16 * c, e);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  const uint16_t r = er[tile_elem(16 * c + j)];
                  if (DN::FIRST_E < 0) e[j] = 0u;
                  else if (r & 0x8000u) e[j] = __float_as_uint(0.01f * __uint_as_float(e[j]));
                }
                TmemIO<16>::st(dE + 16 * c, e);
              }
            }
          }
          if (i < L || NEEDX) {
            tc_wait_st();
            tc_fence_before();
            mbar_arrive(&bar_ready[slot]);
          } else {
            tc_fence_before();
          }
        }
        if constexpr (NEEDX) {
          const uint16_t* er = tile_row_ptr(ws.enc_raw, tile, KE + kTileRowsExtra, lane_row);
          // ---- dEnc complete (init layer added): q_f = cos_f * dsin_f - sin_f * dcos_f -> A operand of the basis GEMM ----
          {
            mbar_wait(&bar_done[slot], n_done & 1); n_done++;
            tc_fence_after();
            uint32_t ds[F], dc[F];
            tmem_load<F>(dE + XR, ds);
            tmem_load<F>(dE + XR + F, dc);
            tc_wait_ld();
            uint32_t q[NET::FP / 2];
#pragma unroll
            for (int j = 0; j < F / 2; ++j) {
              float qq[2];
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const int f = 2 * j + e;
                const float sn = E::back(er[tile_elem(XR + f)]), cs = E::back(er[tile_elem(XR + F + f)]);
                qq[e] = cs * __uint_as_float(ds[f]) - sn * __uint_as_float(dc[f]);
              }
              q[j] = E::pack(qq[0], qq[1]);
            }
            tmem_store<NET::FP / 2>(aA, q);
            tc_wait_st();
            tc_fence_before();
            mbar_arrive(&bar_ready[slot]);
          }
          // ---- g_x = dEnc[x] + q . basis^T ----
          {
            mbar_wait(&bar_done[slot], n_done & 1); n_done++;
            tc_fence_after();
            constexpr int XC = (IN + 7) / 8 * 8;
#pragma unroll
            for (int c = 0; c < XC / 8; ++c) {
              uint32_t a[8], b[8];
              TmemIO<8>::ld(dE + 8 * c, a);
              TmemIO<8>::ld(dM + 8 * c, b);
              tc_wait_ld();
              if (valid) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                  if (8 * c + j < IN) io.store_gx1(m, 8 * c + j, __uint_as_float(a[j]) + __uint_as_float(b[j]));
              }
            }
            tc_fence_before();
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (is_mma_warp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

using NetNerfFirst = Net<3, 0, 16, 128, 5, 3, 65, NRT_ACT_LEAKY_RELU>;
using NetNerfSecondPT = Net<70, 0, 16, 64, 8, 3, 3, NRT_ACT_LEAKY_RELU>;
using NetNerfSecondLE = Net<115, 0, 16, 64, 8, 3, 3, NRT_ACT_LEAKY_RELU>;
using NetNeuralBsdf = Net<3, 0, 64, 96, 6, 3, 3, NRT_ACT_LEAKY_RELU>;       // NeuralBSDF.mlp bsdfs.py:616-621
using NetOcc = Net<5, 0, 16, 64, 8, 3, 1, NRT_ACT_LEAKY_RELU>;              // occlusion MLP  colocate.py:82-85

template <class NET>
static bool matches(const MlpDev& d) {
  return d.in_size == NET::IN && d.latent == NET::LAT && d.freqs == NET::F && d.hidden == NET::H && d.L == NET::L &&
         d.skip == NET::SKIP && d.out == NET::OUT && d.act == NET::ACT;
}

template <class NET, int FMT, class IO>
static int train_forward_io(const nrt_mlp_t* m, const IO& io, int64_t M, const TrainWs& ws, cudaStream_t st);

template <class NET, int FMT>
static int train_forward(const nrt_mlp_t* m, int out_act, const float* x, int64_t M, float* out, const TrainWs& ws, cudaStream_t st) {
  IoTrainFwd<NET::IN, NET::OUT> io{x, out, out_act};
  return train_forward_io<NET, FMT>(m, io, M, ws, st);
}

template <class NET, int FMT, class IO>
static int train_forward_io(const nrt_mlp_t* m, const IO& io, int64_t M, const TrainWs& ws, cudaStream_t st) {
  SaveTiles sv{ws.acts, ws.enc_raw, ws.enc_act, ws.masks, ws.ntiles};
  const size_t bytes = (size_t)NET::SMEM_BYTES + 256;
  auto kern = k_mlp_tc<NET, IO, FMT, SaveTiles>;
  NRT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  const int grid = (int)std::min<int64_t>((ws.ntiles + NET::NSLOT - 1) / NET::NSLOT, (int64_t)nrt_sm_count());
  {
    NrtProfScope _ps(TAG_TC_TRAIN_FWD, st);
    kern<<<grid, NET::threads(NET::WPS), bytes, st>>>(reinterpret_cast<const uint8_t*>(m->params_tc), io, M, nullptr, sv);
  }
  NRT_CUDA(cudaGetLastError());
  NRT_CUDA(cudaGetLastError());
  return NRT_OK;
}

template <class NET, bool NEEDX, int FMT, class IO>
static int train_backward_io(const nrt_mlp_t* m, const MlpDev& d, IO io, int64_t M, const void* dblob, const TrainWs& ws,
                             float* g_params, cudaStream_t st);

template <class NET, bool NEEDX, int FMT>
static int train_backward(const nrt_mlp_t* m, const MlpDev& d, int out_act, int64_t M, const float* out, const float* g_out,
                          const void* dblob, const TrainWs& ws, float* g_params, float* g_x, cudaStream_t st) {
  IoGrad<NET::IN, NET::OUT> io{out, g_out, g_x, out_act, ws.scale};
  return train_backward_io<NET, NEEDX, FMT>(m, d, io, M, dblob, ws, g_params, st);
}

// IO: g_pre(m, j) (gradient w.r.t. the pre-activation output, un-scaled), load_g(m, g) (scaled by scale[1]),
// store_gx1(m, j, v) (NEEDX; must un-scale by scale[2]); the member `scale` is set here.
template <class NET, bool NEEDX, int FMT, class IO>
static int train_backward_io(const nrt_mlp_t* m, const MlpDev& d, IO io, int64_t M, const void* dblob, const TrainWs& ws,
                             float* g_params, cudaStream_t st) {
  using DN = DNet<NET, NEEDX>;
  io.scale = ws.scale;
  {
    NrtProfScope _ps(TAG_TC_DGRAD, st);
    NRT_CUDA(cudaMemsetAsync(ws.scale, 0, 16, st));
    k_grad_absmax<IO, NET::OUT><<<(int)std::min<int64_t>((M * NET::OUT + 255) / 256, 148 * 8), 256, 0, st>>>(io, M, ws.scale);
    k_grad_scale<<<1, 1, 0, st>>>(ws.scale);
    NRT_CUDA(cudaGetLastError());
  }
  {
    const size_t bytes = (size_t)DN::DY.bytes + 256;
    auto kern = k_mlp_dgrad_tc<NET, DN, IO, FMT>;
    NRT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    const int grid = (int)std::min<int64_t>((ws.ntiles + DN::NSLOT - 1) / DN::NSLOT, (int64_t)nrt_sm_count());
    NrtProfScope _ps(TAG_TC_DGRAD, st);
    kern<<<grid, kEpiThreads * 2 + 32 * DN::NSLOT, bytes, st>>>(reinterpret_cast<const uint8_t*>(dblob), io, M, ws);
    NRT_CUDA(cudaGetLastError());
  }
  (void)m;
  return launch_wgrad_std<NET, FMT>(d, ws, g_params, st);
}

// ---------------------------------------------------------------------------------------------
// NeRFLE (nerf.py:175-214) training through both MLPs without materialising their inputs / outputs in fp32:
// samples are indexed sample-major like the reference (m = s * R + ray), so sigma [S,R] and rgb [S,R,3] feed the
// compositing kernels directly; the 64-d latent travels between the two MLPs as fp32 (the second MLP splits it into
// hi + lo operands for its Fourier-phase GEMM), and so does its gradient on the way back.
// ---------------------------------------------------------------------------------------------
// PER_SAMPLE: ts [S,R] holds one distance per sample (t = ts[m], hierarchical sampling) instead of the shared ts [S]
template <bool PER_SAMPLE>
struct IoNerfTrainFirst {
  const float* rays; const float* ts; int64_t R; float* sigma; float* latent;
  __device__ __forceinline__ void load(int64_t m, float* v) const {
    const int64_t s = m / R, ray = m - s * R;
    const float t = __ldg(ts + (PER_SAMPLE ? m : s));
    const float* r = rays + ray * 6;
    v[0] = __ldg(r) + t * __ldg(r + 3); v[1] = __ldg(r + 1) + t * __ldg(r + 4); v[2] = __ldg(r + 2) + t * __ldg(r + 5);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
    sigma[m] = o[0];
    // tile-interleaved scratch (see IoNerfFirst, nrt_tc.cu): warp-wide 16-byte stores cover 512 contiguous bytes
    float4* dst = reinterpret_cast<float4*>(latent) + (m >> 7) * (int64_t)(16 * 128) + (m & 127);
#pragma unroll
    for (int j = 0; j < 16; ++j) dst[j * 128] = make_float4(o[1 + 4 * j], o[2 + 4 * j], o[3 + 4 * j], o[4 + 4 * j]);
  }
};
template <int LD>
struct IoNerfTrainSecond {
  const float* rays; const float* latent; const float* light_code; const int32_t* view_of_ray; int64_t R; float* rgb;
  __device__ __forceinline__ void load(int64_t m, float* v) const {
    const int64_t s = m / R, ray = m - s * R;
    const float4* src = reinterpret_cast<const float4*>(latent) + (m >> 7) * (int64_t)(16 * 128) + (m & 127);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float4 q = __ldg(src + j * 128);
      v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
    }
    const float* r = rays + ray * 6;
    v[64] = __ldg(r + 3); v[65] = __ldg(r + 4); v[66] = __ldg(r + 5);
    const int view = view_of_ray ? __ldg(view_of_ray + ray) : 0;
#pragma unroll
    for (int j = 0; j < LD; ++j) v[67 + j] = __ldg(light_code + (int64_t)view * LD + j);
  }
  __device__ __forceinline__ void store(int64_t m, const float* o) const {
#pragma unroll
    for (int j = 0; j < 3; ++j) rgb[m * 3 + j] = 1.0f / (1.0f + __expf(-o[j]));     // nerf.py:203
  }
};
struct IoNerfGradSecond {      // g w.r.t. sigmoid(rgb) in, g w.r.t. the latent out
  const float* rgb; const float* g_rgb; float* g_latent; const float* scale;
  __device__ __forceinline__ float g_pre(int64_t m, int j) const {
    const float y = __ldg(rgb + m * 3 + j);
    return __ldg(g_rgb + m * 3 + j) * y * (1.0f - y);
  }
  __device__ __forceinline__ void load_g(int64_t m, float* g) const {
    const float S = scale[1];
#pragma unroll
    for (int j = 0; j < 3; ++j) g[j] = g_pre(m, j) * S;
  }
  // g_latent scratch is tile-interleaved too: element j of sample m at ((m / 128) * 64 + j) * 128 + m % 128 (coalesced
  // scalar stores here, coalesced scalar loads in IoNerfGradFirst)
  __device__ __forceinline__ void store_gx1(int64_t m, int j, float v) const {
    if (j < 64) g_latent[((m >> 7) * 64 + j) * 128 + (m & 127)] = v * scale[2];
  }
};
struct IoNerfGradFirst {       // [g_sigma | g_latent] in
  static constexpr bool kColMajor = true;
  const float* g_sigma; const float* g_latent; const float* scale;
  __device__ __forceinline__ float g_pre(int64_t m, int j) const {
    return j == 0 ? __ldg(g_sigma + m) : __ldg(g_latent + ((m >> 7) * 64 + (j - 1)) * 128 + (m & 127));
  }
  __device__ __forceinline__ void load_g(int64_t m, float* g) const {
    const float S = scale[1];
    g[0] = __ldg(g_sigma + m) * S;
    const float* src = g_latent + (m >> 7) * (int64_t)(64 * 128) + (m & 127);
#pragma unroll
    for (int j = 0; j < 64; ++j) g[1 + j] = __ldg(src + j * 128) * S;
  }
  __device__ __forceinline__ void store_gx1(int64_t, int, float) const {}
};

}  // namespace tc

using namespace tc;

// the 256-wide networks (streamed weights): nrt_tc_train_wide.cu
int nrt_train_wide_id(const MlpDev& d);
int64_t nrt_train_wide_dgrad_blob_bytes(const MlpDev& d, bool need_x);
int nrt_train_wide_pack_dgrad(const MlpDev& d, int prec, bool need_x, void* blob_out, cudaStream_t st);
int nrt_train_wide_forward(const nrt_mlp_t* m, const MlpDev& d, int prec, int out_act, const float* x, int64_t M, float* out,
                           const TrainWs& ws, cudaStream_t st);
int nrt_train_wide_backward(const MlpDev& d, int prec, int out_act, int64_t M, const float* out, const float* g_out,
                            const void* dblob, const TrainWs& ws, float* g_params, float* g_x, cudaStream_t st);

// SphereSDF.shift (softplus, streamed weights): nrt_tc_train_sdf.cu
bool nrt_train_is_sdf(const MlpDev& d);
int64_t nrt_train_sdf_dgrad_tail_bytes(const MlpDev& d);
int nrt_train_sdf_pack_tail(const MlpDev& d, void* tail, cudaStream_t st);
int nrt_train_sdf_forward(const nrt_mlp_t* m, int prec, int out_act, const float* x, int64_t M, float* out, const TrainWs& ws,
                          cudaStream_t st);
int nrt_train_sdf_backward(const MlpDev& d, int prec, int out_act, int64_t M, const float* out, const float* g_out,
                           const void* dblob, const TrainWs& ws, float* g_params, cudaStream_t st);

// which networks the training path instantiates, and whether their input gradient is available
static int train_net_id(const MlpDev& d) {
  if (matches<NetNerfFirst>(d)) return 1;
  if (matches<NetNerfSecondPT>(d)) return 2;
  if (matches<NetNerfSecondLE>(d)) return 3;
  if (matches<NetNeuralBsdf>(d)) return 4;
  if (matches<NetOcc>(d)) return 5;
  return 0;
}

extern "C" int64_t nrt_mlp_train_tc_workspace_bytes(const nrt_mlp_t* m, int64_t M) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(train_net_id(d) != 0 || nrt_train_wide_id(d) != 0 || nrt_train_is_sdf(d), "tensor-core training path: this MLP shape is not instantiated");
  const Layout y = make_layout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out);
  return (int64_t)carve_ws(y, d.hidden, d.L, M, nullptr).bytes;
}

extern "C" int64_t nrt_mlp_tc_dgrad_blob_bytes(const nrt_mlp_t* m, int need_x) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  if (nrt_train_wide_id(d) != 0) return nrt_train_wide_dgrad_blob_bytes(d, need_x != 0);
  return (int64_t)make_dlayout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out, need_x != 0).bytes +
         (nrt_train_is_sdf(d) ? nrt_train_sdf_dgrad_tail_bytes(d) : 0);
}

extern "C" int nrt_mlp_pack_tc_dgrad(const nrt_mlp_t* m, int prec, int need_x, void* blob_out, void* stream) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(blob_out != nullptr && ((uintptr_t)blob_out & 15) == 0, "blob_out must be 16-byte aligned");
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "nrt_mlp_pack_tc_dgrad: prec must be F16 or BF16");
  if (nrt_train_wide_id(d) != 0) return nrt_train_wide_pack_dgrad(d, prec, need_x != 0, blob_out, (cudaStream_t)stream);
  const Layout y = make_layout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out);
  const DLayout dl = make_dlayout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out, need_x != 0);
  NrtProfScope _ps(TAG_TC_PACK, (cudaStream_t)stream);
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "nrt_mlp_pack_tc_dgrad: prec must be F16 or BF16");
  const int grid = std::min(nrt_cdiv(dl.w_elems, 256), 1184);
  if (prec == NRT_PREC_F16) k_pack_dgrad<0><<<grid, 256, 0, (cudaStream_t)stream>>>(d, y, dl, need_x, (uint8_t*)blob_out);
  else k_pack_dgrad<1><<<grid, 256, 0, (cudaStream_t)stream>>>(d, y, dl, need_x, (uint8_t*)blob_out);
  NRT_CUDA(cudaGetLastError());
  if (nrt_train_is_sdf(d)) return nrt_train_sdf_pack_tail(d, (uint8_t*)blob_out + dl.bytes, (cudaStream_t)stream);
  return NRT_OK;
}

extern "C" int nrt_mlp_forward_train_tc(const nrt_mlp_t* m, int prec, int out_act, const float* x, int64_t M, float* out,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(M >= 0, "negative M");
  if (M == 0) return NRT_OK;
  NRT_REQUIRE(x && out && workspace, "nrt_mlp_forward_train_tc: null pointer");
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "tensor-core training path: prec must be F16 or BF16");
  NRT_REQUIRE(m->params_tc != nullptr, "mlp.params_tc is NULL: call nrt_mlp_pack_tc (same prec) first");
  const Layout y = make_layout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out);
  const TrainWs ws = carve_ws(y, d.hidden, d.L, M, workspace);
  NRT_REQUIRE(workspace_bytes >= ws.bytes && ((uintptr_t)workspace & 255) == 0, "training workspace too small or not 256-byte aligned");
  if (nrt_train_wide_id(d) != 0) return nrt_train_wide_forward(m, d, prec, out_act, x, M, out, ws, (cudaStream_t)stream);
  if (nrt_train_is_sdf(d)) return nrt_train_sdf_forward(m, prec, out_act, x, M, out, ws, (cudaStream_t)stream);
  switch (train_net_id(d)) {
    case 1:
      if (prec == NRT_PREC_F16) return train_forward<NetNerfFirst, 0>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
      return train_forward<NetNerfFirst, 1>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
    case 2:
      if (prec == NRT_PREC_F16) return train_forward<NetNerfSecondPT, 0>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
      return train_forward<NetNerfSecondPT, 1>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
    case 3:
      if (prec == NRT_PREC_F16) return train_forward<NetNerfSecondLE, 0>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
      return train_forward<NetNerfSecondLE, 1>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
    case 4:
      if (prec == NRT_PREC_F16) return train_forward<NetNeuralBsdf, 0>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
      return train_forward<NetNeuralBsdf, 1>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
    case 5:
      if (prec == NRT_PREC_F16) return train_forward<NetOcc, 0>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
      return train_forward<NetOcc, 1>(m, out_act, x, M, out, ws, (cudaStream_t)stream);
  }
  nrt_set_error("tensor-core training path: this MLP shape is not instantiated (NeRFLE.first / NeRFLE.second PT and LE are)");
  return NRT_E_UNSUPPORTED;
}

extern "C" int nrt_mlp_backward_tc(const nrt_mlp_t* m, int prec, int out_act, int64_t M, const float* out, const float* g_out,
                                   const void* dgrad_blob, void* workspace, size_t workspace_bytes, float* g_params,
                                   float* g_x, void* stream) {
  MlpDev d;
  int rc = nrt_build_mlp_dev(m, &d);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(M >= 0, "negative M");
  if (M == 0) return NRT_OK;
  NRT_REQUIRE(out && g_out && dgrad_blob && workspace && g_params, "nrt_mlp_backward_tc: null pointer");
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "tensor-core training path: prec must be F16 or BF16");
  const bool f16 = prec == NRT_PREC_F16;
  const Layout y = make_layout(d.in_size, d.latent, d.freqs, d.hidden, d.L, d.skip, d.out);
  const TrainWs ws = carve_ws(y, d.hidden, d.L, M, workspace);
  NRT_REQUIRE(workspace_bytes >= ws.bytes, "training workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  if (nrt_train_wide_id(d) != 0) return nrt_train_wide_backward(d, prec, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
  if (nrt_train_is_sdf(d)) {
    NRT_REQUIRE(g_x == nullptr, "tensor-core training path: SphereSDF.shift has no input gradient (its points come out of a no_grad march)");
    return nrt_train_sdf_backward(d, prec, out_act, M, out, g_out, dgrad_blob, ws, g_params, st);
  }
  switch (train_net_id(d)) {
    case 1:
      NRT_REQUIRE(g_x == nullptr, "NeRFLE.first on the tensor-core path has no input gradient (split-precision inputs)");
      if (f16) return train_backward<NetNerfFirst, false, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
      return train_backward<NetNerfFirst, false, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
    case 2:
      if (g_x) {
        if (f16) return train_backward<NetNerfSecondPT, true, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
        return train_backward<NetNerfSecondPT, true, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
      }
      if (f16) return train_backward<NetNerfSecondPT, false, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
      return train_backward<NetNerfSecondPT, false, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
    case 3:
      if (g_x) {
        if (f16) return train_backward<NetNerfSecondLE, true, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
        return train_backward<NetNerfSecondLE, true, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
      }
      if (f16) return train_backward<NetNerfSecondLE, false, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
      return train_backward<NetNerfSecondLE, false, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
    case 4:
      if (g_x) {
        if (f16) return train_backward<NetNeuralBsdf, true, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
        return train_backward<NetNeuralBsdf, true, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
      }
      if (f16) return train_backward<NetNeuralBsdf, false, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
      return train_backward<NetNeuralBsdf, false, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
    case 5:
      if (g_x) {
        if (f16) return train_backward<NetOcc, true, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
        return train_backward<NetOcc, true, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, g_x, st);
      }
      if (f16) return train_backward<NetOcc, false, 0>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
      return train_backward<NetOcc, false, 1>(m, d, out_act, M, out, g_out, dgrad_blob, ws, g_params, nullptr, st);
  }
  nrt_set_error("tensor-core training path: this MLP shape is not instantiated");
  return NRT_E_UNSUPPORTED;
}

// ---- NeRFLE fused training entry points ----------------------------------------------------------------------
static int nerfle_train_nets(const nrt_mlp_t* first, const nrt_mlp_t* second, int light_dim, MlpDev* d1, MlpDev* d2, int* id2) {
  int rc = nrt_build_mlp_dev(first, d1);
  if (rc != NRT_OK) return rc;
  rc = nrt_build_mlp_dev(second, d2);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(train_net_id(*d1) == 1, "NeRFLE training path: first MLP must be NeRFLE.first (3->65, 5x128)");
  *id2 = train_net_id(*d2);
  NRT_REQUIRE((*id2 == 2 && light_dim == 3) || (*id2 == 3 && light_dim == 48),
              "NeRFLE training path: second MLP must be NeRFLE.second with a point light (70 inputs) or the 48-float environment code (115)");
  return NRT_OK;
}

template <bool PER_SAMPLE>
static int nerfle_train_forward_impl(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                                     const float* ts, int S, const float* light_code, int light_dim,
                                     const int32_t* view_of_ray, float* sigma, float* rgb, float* latent,
                                     void* ws_first, size_t ws_first_bytes, void* ws_second, size_t ws_second_bytes,
                                     cudaStream_t st) {
  MlpDev d1, d2;
  int id2 = 0;
  int rc = nerfle_train_nets(first, second, light_dim, &d1, &d2, &id2);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "tensor-core training path: prec must be F16 or BF16");
  NRT_REQUIRE(R >= 0 && S >= 1, "nrt_nerfle_train_forward: bad arguments");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(rays && ts && light_code && sigma && rgb && latent && ws_first && ws_second, "nrt_nerfle_train_forward: null pointer");
  NRT_REQUIRE(first->params_tc && second->params_tc, "params_tc is NULL: call nrt_mlp_pack_tc (same prec) first");
  NRT_REQUIRE(((uintptr_t)latent & 15) == 0, "latent must be 16-byte aligned");
  const int64_t M = R * S;
  const Layout y1 = make_layout(d1.in_size, d1.latent, d1.freqs, d1.hidden, d1.L, d1.skip, d1.out);
  const Layout y2 = make_layout(d2.in_size, d2.latent, d2.freqs, d2.hidden, d2.L, d2.skip, d2.out);
  const TrainWs w1 = carve_ws(y1, d1.hidden, d1.L, M, ws_first), w2 = carve_ws(y2, d2.hidden, d2.L, M, ws_second);
  NRT_REQUIRE(ws_first_bytes >= w1.bytes && ws_second_bytes >= w2.bytes, "training workspace too small");
  const int fmt = prec == NRT_PREC_BF16 ? 1 : 0;
  IoNerfTrainFirst<PER_SAMPLE> io1{rays, ts, R, sigma, latent};
  rc = fmt == 0 ? train_forward_io<NetNerfFirst, 0>(first, io1, M, w1, st) : train_forward_io<NetNerfFirst, 1>(first, io1, M, w1, st);
  if (rc != NRT_OK) return rc;
  if (id2 == 2) {
    IoNerfTrainSecond<3> io2{rays, latent, light_code, view_of_ray, R, rgb};
    return fmt == 0 ? train_forward_io<NetNerfSecondPT, 0>(second, io2, M, w2, st) : train_forward_io<NetNerfSecondPT, 1>(second, io2, M, w2, st);
  }
  IoNerfTrainSecond<48> io2{rays, latent, light_code, view_of_ray, R, rgb};
  return fmt == 0 ? train_forward_io<NetNerfSecondLE, 0>(second, io2, M, w2, st) : train_forward_io<NetNerfSecondLE, 1>(second, io2, M, w2, st);
}

extern "C" int nrt_nerfle_train_forward(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                                        const float* ts, int S, const float* light_code, int light_dim,
                                        const int32_t* view_of_ray, float* sigma, float* rgb, float* latent,
                                        void* ws_first, size_t ws_first_bytes, void* ws_second, size_t ws_second_bytes,
                                        void* stream) {
  return nerfle_train_forward_impl<false>(first, second, prec, rays, R, ts, S, light_code, light_dim, view_of_ray, sigma, rgb,
                                          latent, ws_first, ws_first_bytes, ws_second, ws_second_bytes, (cudaStream_t)stream);
}

extern "C" int nrt_nerfle_train_forward_ts(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, const float* rays, int64_t R,
                                           const float* ts, int S, const float* light_code, int light_dim,
                                           const int32_t* view_of_ray, float* sigma, float* rgb, float* latent,
                                           void* ws_first, size_t ws_first_bytes, void* ws_second, size_t ws_second_bytes,
                                           void* stream) {
  return nerfle_train_forward_impl<true>(first, second, prec, rays, R, ts, S, light_code, light_dim, view_of_ray, sigma, rgb,
                                         latent, ws_first, ws_first_bytes, ws_second, ws_second_bytes, (cudaStream_t)stream);
}

extern "C" int nrt_nerfle_train_backward(const nrt_mlp_t* first, const nrt_mlp_t* second, int prec, int64_t R, int S,
                                         int light_dim, const float* rgb, const float* g_sigma, const float* g_rgb,
                                         const void* dgrad_blob_first, const void* dgrad_blob_second, void* ws_first,
                                         void* ws_second, float* g_latent_scratch, float* g_params_first,
                                         float* g_params_second, void* stream) {
  MlpDev d1, d2;
  int id2 = 0;
  int rc = nerfle_train_nets(first, second, light_dim, &d1, &d2, &id2);
  if (rc != NRT_OK) return rc;
  NRT_REQUIRE(prec == NRT_PREC_F16 || prec == NRT_PREC_BF16, "tensor-core training path: prec must be F16 or BF16");
  if (R == 0) return NRT_OK;
  NRT_REQUIRE(rgb && g_sigma && g_rgb && dgrad_blob_first && dgrad_blob_second && ws_first && ws_second && g_latent_scratch &&
              g_params_first && g_params_second, "nrt_nerfle_train_backward: null pointer");
  const int64_t M = R * S;
  const Layout y1 = make_layout(d1.in_size, d1.latent, d1.freqs, d1.hidden, d1.L, d1.skip, d1.out);
  const Layout y2 = make_layout(d2.in_size, d2.latent, d2.freqs, d2.hidden, d2.L, d2.skip, d2.out);
  const TrainWs w1 = carve_ws(y1, d1.hidden, d1.L, M, ws_first), w2 = carve_ws(y2, d2.hidden, d2.L, M, ws_second);
  cudaStream_t st = (cudaStream_t)stream;
  const bool f16 = prec == NRT_PREC_F16;
  IoNerfGradSecond g2{rgb, g_rgb, g_latent_scratch, nullptr};
  if (id2 == 2) rc = f16 ? train_backward_io<NetNerfSecondPT, true, 0>(second, d2, g2, M, dgrad_blob_second, w2, g_params_second, st)
                         : train_backward_io<NetNerfSecondPT, true, 1>(second, d2, g2, M, dgrad_blob_second, w2, g_params_second, st);
  else rc = f16 ? train_backward_io<NetNerfSecondLE, true, 0>(second, d2, g2, M, dgrad_blob_second, w2, g_params_second, st)
                : train_backward_io<NetNerfSecondLE, true, 1>(second, d2, g2, M, dgrad_blob_second, w2, g_params_second, st);
  if (rc != NRT_OK) return rc;
  IoNerfGradFirst g1{g_sigma, g_latent_scratch, nullptr};
  return f16 ? train_backward_io<NetNerfFirst, false, 0>(first, d1, g1, M, dgrad_blob_first, w1, g_params_first, st)
             : train_backward_io<NetNerfFirst, false, 1>(first, d1, g1, M, dgrad_blob_first, w1, g_params_first, st);
}
