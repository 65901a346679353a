// tcgen05 / TMEM building blocks shared by the forward kernels (nrt_tc.cu) and the training kernels
// (nrt_tc_train.cu): blob layout, PTX wrappers, TMEM load/store helpers, the compile-time network description
// and the fused forward kernel template k_mlp_tc.  Internal header of libnrt_b200.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <type_traits>

#include "nrt_common.cuh"

namespace tc {

// ---------------------------------------------------------------------------------------------
// blob layout, shared by the pack kernel (runtime) and the MMA kernels (compile time)
// ---------------------------------------------------------------------------------------------
constexpr int kMaxOps = NRT_MAX_LAYERS + 3;

struct Layout {
  int split, XR, KRAW, KE, KX, KPH, FP, NOP;
  int n_ops;            // encB, init, layers[0..L-1], out
  int opN[kMaxOps], opK[kMaxOps];
  int op_off[kMaxOps];  // in 16-bit elements
  int w_elems;
  int bias_off[kMaxOps];  // float offset inside the bias area (ops 1..n_ops-1)
  int bias_floats;        // floats of the fp32 area: biases, then the two optional tables below
  int wout_f32_off;       // [H][4] fp32 output weights (out <= 4: the output layer runs in the last epilogue), or -1
  int basis_f32_off;      // [in][FP] fp32 Fourier basis (split-precision inputs: phases on the CUDA cores), or -1
  int bytes;              // everything above, then the bias K-chunks if there are any (bk_off below)
};
// where the biases of a render layout (make_render_layout) are; -1 = none (every other layout).  Kept out of Layout, whose
// size shapes the stack frame of every k_mlp_tc instance.
struct BiasRows {
  int row;                // K index in the x segment of the encoding of the three rows b_hi, b_mid, b_lo (init / skip layers)
  int bk8_off[kMaxOps];   // 16-bit element offset of the op's 8-deep bias chunk (before the weights)
};

__host__ __device__ constexpr int c16(int x) { return (x + 15) / 16 * 16; }
__host__ __device__ constexpr int imax(int a, int b) { return a > b ? a : b; }
__host__ __device__ constexpr bool is_skip(int i, int skip, int L) { return (i % skip) == 0 && i != L - 1; }

// shared memory that k_mlp_tc may fill with a resident blob (larger blobs are streamed stage by stage)
constexpr int kSmemBudget = 227 * 1024 - 2048;

// NRT_BIAS_MMA: the biases of the MMA layers (init + hidden) ride the layer's MMA as one more K-chunk instead of being
// pre-loaded into the accumulator by the previous epilogue (LDS + tcgen05.st + wait::st on every stage's critical chain).
// The blob then carries, after the fp32 area, one 16-deep B chunk per such layer: row 0 = b_hi, row 1 = b_mid, row 2 = b_lo
// (b = b_hi + b_mid + b_lo in the 16-bit operand format), rows 3..15 zero; k_mlp_tc multiplies it by a constant A chunk
// [1, 1, 1, 0, ...] held once per CTA in TMEM.  Nothing before the chunks moves, so every kernel that reads the blob
// without them (training forward, the SDF / wide kernels) sees the same offsets.  Laid out for nets with hidden width <= 64
// (a stage's MMAs are ~160 cycles, shorter than the preload chain they replace), a tensor-core phase GEMM (in > 5) and a
// fused output layer (out <= 4: no bias chunk of width NOP), while the resident blob still fits: among the instantiated
// nets this is NeRFLE.second (point and environment light).  NeRFLE.first (221 KB of 225) would not fit its 7 chunks;
// its inference kernels read a layout of their own instead (make_render_layout).
// The switch is a bit set: bit 0 the bias K-chunks, bit 1 the skipped zero x_lo chunks of the phase GEMM (k_mlp_tc, ZLO),
// bit 2 the render layout of NeRFLE.first (nrt_tc.cu); 0 builds the kernels without any of them.
#ifndef NRT_BIAS_MMA
#define NRT_BIAS_MMA 7
#endif

__host__ __device__ constexpr Layout make_layout(int in, int lat, int f, int h, int L, int skip, int out) {
  Layout y{};
  // raw-x segment: [x_hi | x_lo] (split) or [x]; padded to 16 K-elements so that every later
  // segment (sin, cos, latent) starts on an 8-column TMEM boundary.  The same 16-aligned segment
  // doubles as the A tile of the phase GEMM ([x_hi | x_lo | x_hi] when split).
  y.split = in <= 5 ? 1 : 0;
  y.XR = c16(in * (y.split ? 2 : 1));
  y.KRAW = y.XR + 2 * f + lat;
  y.KE = c16(y.KRAW);
  y.KX = y.XR;
  // K of the phase GEMM (op 0).  Inputs that are not split column-wise (in > 5) get their Fourier phases from a
  // hi+lo split MMA: x.B ~= x_hi.B_hi + x_lo.B_hi + x_hi.B_lo, K = 3*XR (A chunks: x_hi, x_lo, x_hi again; B chunks:
  // B_hi, B_hi, B_lo), so that sin / cos arguments of tens to hundreds of radians keep ~fp32 accuracy.
  y.KPH = y.split ? y.KX : 3 * y.XR;
  y.FP = c16(f);
  y.NOP = c16(out);
  y.n_ops = L + 3;
  int off = 0, boff = 0;
  for (int o = 0; o < y.n_ops; ++o) {
    int N = 0, K = 0;
    if (o == 0) { N = y.FP; K = y.KPH; }
    else if (o == 1) { N = h; K = y.KE; }
    else if (o == y.n_ops - 1) { N = y.NOP; K = h; }
    else { N = h; K = h + (is_skip(o - 2, skip, L) ? y.KE : 0); }
    y.opN[o] = N; y.opK[o] = K; y.op_off[o] = off; off += N * K;
    y.bias_off[o] = boff;
    if (o >= 1) boff += N;
  }
  y.w_elems = off;
  y.wout_f32_off = -1;
  y.basis_f32_off = -1;
  if (out <= 4) { y.wout_f32_off = boff; boff += h * 4; }
  if (y.split) { y.basis_f32_off = boff; boff += in * y.FP; }
  y.bias_floats = boff;
  y.bytes = off * 2 + boff * 4;
  if ((NRT_BIAS_MMA & 1) && h <= 64 && !y.split && out <= 4) {
    const int bytes = (y.bytes + 127) / 128 * 128 + (y.n_ops - 2) * h * 16 * 2;    // ops 1 .. n_ops-2, each N = h
    if (bytes <= kSmemBudget) y.bytes = bytes;
  }
  return y;
}
// byte offset of the bias K-chunks (128-byte aligned after the fp32 area), or -1 when the blob has none
__host__ __device__ constexpr int bk_off(const Layout& y) {
  const int end = y.w_elems * 2 + y.bias_floats * 4;
  return y.bytes > end ? (end + 127) / 128 * 128 : -1;
}
// Render layout (NRT_BIAS_MMA bit 2; NeRFLE.first, whose training layout leaves 5 KB of shared memory free): every bias
// rides an MMA that k_mlp_tc issues, so the layout has no fp32 biases, only the Fourier basis.
//  * init and skip layers: the x segment of the encoding is [x_hi | x_lo | x_hi | 0 ...] (raw) and [act_hi | act_lo | 0 ...]
//    (activated); the kernel writes the constant 1 into its columns bias_row .. bias_row+2 = 3*in .. 3*in+2 in both, and
//    the three weight rows there hold b_hi, b_mid, b_lo.  The bias enters through MMAs that are issued anyway.
//  * the other layers: an 8-deep B chunk, rows b_hi, b_mid, b_lo, 0 ..., times the constant A chunk [1, 1, 1, 0, ...].
//    Only the k = 0..7 core-matrix group is stored; the MMA still reads a k = 8..15 group at +LBO = 16*N bytes, which
//    meets zeros of the A chunk and may be any finite 16-bit data.  The chunks sit in front of the weights, the output
//    layer's (the narrowest) first, so each of those windows lies on the next chunk or on the weights.
// The weights follow unchanged (op_off shifted by the chunks).
__host__ __device__ constexpr BiasRows no_bias_rows() {
  BiasRows b{};
  b.row = -1;
  for (int o = 0; o < kMaxOps; ++o) b.bk8_off[o] = -1;
  return b;
}
__host__ __device__ constexpr BiasRows render_bias_rows(int in, int lat, int f, int h, int L, int skip, int out) {
  const Layout y = make_layout(in, lat, f, h, L, skip, out);
  BiasRows b = no_bias_rows();
  b.row = 3 * in;
  int c = 0;
  b.bk8_off[y.n_ops - 1] = c; c += 8 * y.opN[y.n_ops - 1];
  for (int o = 2; o < y.n_ops - 1; ++o)
    if (!is_skip(o - 2, skip, L)) { b.bk8_off[o] = c; c += 8 * y.opN[o]; }
  return b;
}
__host__ __device__ constexpr Layout make_render_layout(int in, int lat, int f, int h, int L, int skip, int out) {
  Layout y = make_layout(in, lat, f, h, L, skip, out);
  const BiasRows b = render_bias_rows(in, lat, f, h, L, skip, out);
  int c = 0;   // 16-bit elements of the chunks
  for (int o = 0; o < y.n_ops; ++o) c += b.bk8_off[o] >= 0 ? 8 * y.opN[o] : 0;
  for (int o = 0; o < y.n_ops; ++o) { y.op_off[o] += c; y.bias_off[o] = -1; }
  y.w_elems += c;
  y.wout_f32_off = -1;
  y.basis_f32_off = 0;
  y.bias_floats = in * y.FP;
  y.bytes = y.w_elems * 2 + y.bias_floats * 4;
  return y;
}
// what k_mlp_tc relies on in a render layout: split inputs with room for the three bias rows in the x segment, an output
// layer on the tensor cores, and every 8-deep chunk's k = 8..15 window inside 16-bit chunk or weight data
__host__ __device__ constexpr bool render_layout_ok(const Layout& y, const BiasRows& b) {
  if (!y.split || b.row + 3 > y.XR || y.wout_f32_off >= 0) return false;
  for (int o = 0; o < y.n_ops; ++o)
    if (b.bk8_off[o] >= 0 && (b.bk8_off[o] + 16 * y.opN[o] > y.w_elems || b.bk8_off[o] + 8 * y.opN[o] > y.op_off[0])) return false;
  return true;
}

// maps a K index of the tensor-core encoding layout to the reference encoding index (-1: padding)
__host__ __device__ inline int enc_ref_index(const Layout& y, int in, int k) {
  if (k >= y.KRAW) return -1;
  if (k >= y.XR) return k - y.XR + in;        // sin | cos | latent follow the padded x segment
  if (k < in) return k;                        // x (hi part)
  if (y.split && k < 2 * in) return k - in;    // x_lo columns reuse the x weights
  return -1;                                   // padding (and the third copy of x_hi used by the phase GEMM)
}

template <int FMT> struct Elem;   // FMT 0: fp16, 1: bf16 (= tcgen05 a/b_format)
template <> struct Elem<0> {
  static __device__ __forceinline__ uint16_t cvt(float v) { return __half_as_ushort(__float2half_rn(v)); }
  static __device__ __forceinline__ float back(uint16_t u) { return __half2float(__ushort_as_half(u)); }
  static __device__ __forceinline__ uint32_t pack(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
};
template <> struct Elem<1> {
  static __device__ __forceinline__ uint16_t cvt(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
  static __device__ __forceinline__ float back(uint16_t u) { return __bfloat162float(__ushort_as_bfloat16(u)); }
  static __device__ __forceinline__ uint32_t pack(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
};

// ---------------------------------------------------------------------------------------------
// pack kernel: packed-f32 parameters -> UMMA canonical (no-swizzle, K-major) 16-bit tiles + biases
// element (n,k) of an [N x K] operand lives at ((k/8)*N + n)*8 + k%8
// ---------------------------------------------------------------------------------------------
// elements k_pack_tc writes: 16-bit weights, fp32 area, 16-bit bias K-chunks
__host__ __device__ constexpr int pack_tc_items(const Layout& y) {
  return y.w_elems + y.bias_floats + (bk_off(y) >= 0 ? (y.n_ops - 2) * y.opN[1] * 16 : 0);
}
// term t (0: b_hi, 1: b_mid, 2: b_lo) of a bias b = b_hi + b_mid + b_lo in the 16-bit operand format: each term is the
// rounding of what the previous ones left over
template <int FMT>
__device__ __forceinline__ float bias_term(float b, int t) {
  float v = 0.0f;
  for (int i = 0; i <= t; ++i) { v = Elem<FMT>::back(Elem<FMT>::cvt(b)); b -= v; }
  return v;
}
template <int FMT>
__global__ void k_pack_tc(MlpDev m, Layout y, BiasRows br, uint8_t* __restrict__ blob) {
  uint16_t* w = reinterpret_cast<uint16_t*>(blob);
  float* bias = reinterpret_cast<float*>(blob + (size_t)y.w_elems * 2);
  const int total = pack_tc_items(y);
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    if (idx >= y.w_elems + y.bias_floats) {
      // bias K-chunk of op o = 1 + e / (N*16), N = hidden: element (n, k) at (k/8)*N*8 + n*8 + k%8; rows k = 0, 1, 2 hold
      // b_hi, b_mid, b_lo
      const int e = idx - y.w_elems - y.bias_floats, N = y.opN[1];
      const int o = 1 + e / (N * 16), r = e - (o - 1) * (N * 16);
      const int kg = r / (N * 8), rem = r - kg * (N * 8), n = rem / 8, k = kg * 8 + (rem & 7);
      const float v = (k < 3 && n < m.N[o - 1]) ? bias_term<FMT>(m.params[m.b_off[o - 1] + n], k) : 0.0f;
      reinterpret_cast<uint16_t*>(blob + bk_off(y))[e] = Elem<FMT>::cvt(v);
      continue;
    }
    if (idx < y.op_off[0]) {
      // 8-deep bias chunk of the render layout: element (n, k < 8) at n*8 + k
      int o = 0;
      while (br.bk8_off[o] < 0 || idx < br.bk8_off[o] || idx >= br.bk8_off[o] + 8 * y.opN[o]) ++o;
      const int e = idx - br.bk8_off[o], n = e >> 3, k = e & 7;
      w[idx] = Elem<FMT>::cvt((k < 3 && n < m.N[o - 1]) ? bias_term<FMT>(m.params[m.b_off[o - 1] + n], k) : 0.0f);
      continue;
    }
    if (idx >= y.w_elems) {
      int b = idx - y.w_elems;
      if (y.basis_f32_off >= 0 && b >= y.basis_f32_off) {
        const int e = b - y.basis_f32_off, j = e / y.FP, f = e - j * y.FP;
        bias[b] = f < m.freqs ? m.basis[j * m.freqs + f] : 0.0f;
        continue;
      }
      if (y.wout_f32_off >= 0 && b >= y.wout_f32_off) {
        const int e = b - y.wout_f32_off, k = e >> 2, j = e & 3;
        bias[b] = j < m.out ? m.params[m.w_off[m.n_lin - 1] + k * m.out + j] : 0.0f;
        continue;
      }
      // biases: ops 1..n_ops-1
      int o = 1;
      while (o + 1 < y.n_ops && b >= y.bias_off[o + 1]) ++o;
      const int n = b - y.bias_off[o];
      const int li = o - 1;
      bias[b] = (n < m.N[li]) ? m.params[m.b_off[li] + n] : 0.0f;
      continue;
    }
    int o = 0;
    while (o + 1 < y.n_ops && idx >= y.op_off[o + 1]) ++o;
    const int e = idx - y.op_off[o];
    const int N = y.opN[o];
    const int chunk = e / (N * 8), rem = e - chunk * (N * 8);
    const int n = rem / 8, k = chunk * 8 + (rem & 7);
    float v = 0.0f;
    if (o == 0) {
      if (n < m.freqs) {
        if (y.split) {
          const int seg = k / m.in_size, j = k - seg * m.in_size;
          if (seg < 3) {
            const float bv = m.basis[j * m.freqs + n];
            const float hi = Elem<FMT>::back(Elem<FMT>::cvt(bv));
            v = (seg < 2) ? hi : (bv - hi);
          }
        } else {
          // hi+lo phase GEMM: K segments [B_hi | B_hi | B_lo], each XR wide
          const int seg = k / y.XR, j = k - seg * y.XR;
          if (j < m.in_size) {
            const float bv = m.basis[j * m.freqs + n];
            const float hi = Elem<FMT>::back(Elem<FMT>::cvt(bv));
            v = (seg < 2) ? hi : (bv - hi);
          }
        }
      }
    } else if (o == y.n_ops - 1) {
      if (n < m.out) v = m.params[m.w_off[m.n_lin - 1] + k * m.out + n];
    } else {
      const int li = o - 1;
      int kref;
      if (o == 1) kref = enc_ref_index(y, m.in_size, k);
      else if (k < m.hidden) kref = k;
      else { const int r = enc_ref_index(y, m.in_size, k - m.hidden); kref = r < 0 ? -1 : m.hidden + r; }
      if (kref >= 0) v = m.params[m.w_off[li] + kref * m.hidden + n];
      // render layout: the bias rows in the padding of the encoding's x segment (init and skip layers)
      const int ke = o == 1 ? k : k - m.hidden;
      if (br.row >= 0 && ke >= br.row && ke < br.row + 3) v = bias_term<FMT>(m.params[m.b_off[li] + n], ke - br.row);
    }
    w[idx] = Elem<FMT>::cvt(v);
  }
}

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// NRT_TRYWAIT_HINT (ns, 0 = none): suspend-time hint of mbarrier.try_wait.  Without it a waiting warp's try_wait returns after
// a short implementation-defined time and the loop re-issues it (ncu source page of NeRFLE.second: SYNCS + BRA + YIELD of the
// wait loops = 18 % of all warp instructions executed, ~7 polls per wait).
#ifndef NRT_TRYWAIT_HINT
#define NRT_TRYWAIT_HINT 0
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t ok = 0;
  while (!ok) {
#if NRT_TRYWAIT_HINT > 0
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(a), "r"(parity), "r"((uint32_t)NRT_TRYWAIT_HINT) : "memory");
#else
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(a), "r"(parity) : "memory");
#endif
  }
}
// non-blocking phase test (all lanes of the warp call it; the result is warp-uniform)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (sm_100); no swizzle; base offset 0
  return d;
}
// D[tmem] (+)= A[tmem] * B[smem]^T, M = 128, K = 16
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n"
               ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}

// tcgen05.ld / st, shape 32x32b: thread i of the warp <-> TMEM lane (32*(warp%4) + i), N columns
template <int N> struct TmemIO;
#define NRT_R4(a, i) "=r"(a[i]), "=r"(a[i + 1]), "=r"(a[i + 2]), "=r"(a[i + 3])
#define NRT_W4(a, i) "r"(a[i]), "r"(a[i + 1]), "r"(a[i + 2]), "r"(a[i + 3])
template <> struct TmemIO<1> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(t));
  }
  static __device__ __forceinline__ void st(uint32_t t, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(t), "r"(r[0]) : "memory");
  }
};
template <> struct TmemIO<2> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(t));
  }
  static __device__ __forceinline__ void st(uint32_t t, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(t), "r"(r[0]), "r"(r[1]) : "memory");
  }
};
template <> struct TmemIO<4> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : NRT_R4(r, 0) : "r"(t));
  }
  static __device__ __forceinline__ void st(uint32_t t, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(t), NRT_W4(r, 0) : "memory");
  }
};
template <> struct TmemIO<8> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : NRT_R4(r, 0), NRT_R4(r, 4) : "r"(t));
  }
  static __device__ __forceinline__ void st(uint32_t t, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(t), NRT_W4(r, 0), NRT_W4(r, 4) : "memory");
  }
};
template <> struct TmemIO<16> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : NRT_R4(r, 0), NRT_R4(r, 4), NRT_R4(r, 8), NRT_R4(r, 12) : "r"(t));
  }
  static __device__ __forceinline__ void st(uint32_t t, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(t), NRT_W4(r, 0), NRT_W4(r, 4), NRT_W4(r, 8), NRT_W4(r, 12) : "memory");
  }
};
template <> struct TmemIO<32> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : NRT_R4(r, 0), NRT_R4(r, 4), NRT_R4(r, 8), NRT_R4(r, 12), NRT_R4(r, 16), NRT_R4(r, 20), NRT_R4(r, 24), NRT_R4(r, 28)
                 : "r"(t));
  }
};
#define NRT_R16(a, i) NRT_R4(a, i), NRT_R4(a, i + 4), NRT_R4(a, i + 8), NRT_R4(a, i + 12)
#define NRT_W16(a, i) NRT_W4(a, i), NRT_W4(a, i + 4), NRT_W4(a, i + 8), NRT_W4(a, i + 12)
template <> struct TmemIO<64> {
  static __device__ __forceinline__ void ld(uint32_t t, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,"
                 "%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,"
                 "%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
                 : NRT_R16(r, 0), NRT_R16(r, 16), NRT_R16(r, 32), NRT_R16(r, 48) : "r"(t));
  }
};
// x32 store lives outside TmemIO<32> (which only loads)
__device__ __forceinline__ void tmem_st32(uint32_t t, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
               "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
               ::"r"(t), NRT_W16(r, 0), NRT_W16(r, 16) : "memory");
}
// store NP packed 32-bit columns starting at column address t (compile-time decomposition)
template <int NP>
__device__ __forceinline__ void tmem_store(uint32_t t, const uint32_t* r) {
  if constexpr (NP >= 32) { tmem_st32(t, r); tmem_store<NP - 32>(t + 32, r + 32); }
  else if constexpr (NP >= 16) { TmemIO<16>::st(t, r); tmem_store<NP - 16>(t + 16, r + 16); }
  else if constexpr (NP >= 8) { TmemIO<8>::st(t, r); tmem_store<NP - 8>(t + 8, r + 8); }
  else if constexpr (NP >= 4) { TmemIO<4>::st(t, r); tmem_store<NP - 4>(t + 4, r + 4); }
  else if constexpr (NP >= 2) { TmemIO<2>::st(t, r); tmem_store<NP - 2>(t + 2, r + 2); }
  else if constexpr (NP == 1) { TmemIO<1>::st(t, r); }
}
template <int NP>
__device__ __forceinline__ void tmem_load(uint32_t t, uint32_t* r) {
  if constexpr (NP >= 64) { TmemIO<64>::ld(t, r); tmem_load<NP - 64>(t + 64, r + 64); }
  else if constexpr (NP >= 32) { TmemIO<32>::ld(t, r); tmem_load<NP - 32>(t + 32, r + 32); }
  else if constexpr (NP >= 16) { TmemIO<16>::ld(t, r); tmem_load<NP - 16>(t + 16, r + 16); }
  else if constexpr (NP >= 8) { TmemIO<8>::ld(t, r); tmem_load<NP - 8>(t + 8, r + 8); }
  else if constexpr (NP >= 4) { TmemIO<4>::ld(t, r); tmem_load<NP - 4>(t + 4, r + 4); }
  else if constexpr (NP >= 2) { TmemIO<2>::ld(t, r); tmem_load<NP - 2>(t + 2, r + 2); }
  else if constexpr (NP == 1) { TmemIO<1>::ld(t, r); }
}

// Softplus forms.  Generic code (act_fast, convert32, the training kernels): NRT_SOFTPLUS_POLY, default 0 = two MUFU
// (ex2 + lg2); 1 = ex2 + degree-4 polynomial of log1p on the FMA pipe (fp32); 2 = everything on packed halves.
// The hidden-layer conversion of the inference kernel k_mlp_tc (convert_row_pipe) takes its form from the IO policy
// (SoftplusOf<IO>): 0 = two MUFU, chunked conversion (the primary sphere-trace march), 1 = fp32 polynomial (default:
// point evaluation), 3 = exponent in fp32, polynomial + max on packed halves (the min scan of SDF.throughput, which only
// picks a position, and the shadow march, which returns a boolean).
// Measured on B200 with one form for all three kernels (262,144 rays: march / shadow march / min scan, ms):
// two MUFU 10.6 / 15.1 / 34.2, form 1: 9.5 / 14.1 / 32.1, form 3: 8.5 / 12.2 / 27.8; median depth error of the march
// vs the exact kernels 0.9e-5 / 1.2e-5 / 1.6e-5, but with form 3 only 97.4 % (< 99 %) of the 64x64 colocate depths stay
// within 2e-3 of the reference (tests/test_gpu_configs.py), hence form 1 where depths are produced.
#ifndef NRT_SOFTPLUS_POLY
#define NRT_SOFTPLUS_POLY 0
#endif
template <class T, class = void> struct SoftplusOf { static constexpr int value = 1; };
template <class T> struct SoftplusOf<T, std::void_t<decltype(T::kSoftplusForm)>> { static constexpr int value = T::kSoftplusForm; };
// fast activations for the 16-bit path (results are rounded to 16 bits anyway)
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
template <int ACT>
__device__ __forceinline__ float act_fast(float x) {
  if constexpr (ACT == NRT_ACT_SOFTPLUS) {
    // branch-free softplus: max(x,0) + log(1 + exp(-|x|)); beyond torch's threshold (20) the log term is < 3e-9,
    // i.e. the result is x like F.softplus.  Two MUFU ops, no divergence (a `x > 20 ? x : ...` form compiles to a
    // per-element branch that cost ~100 cycles per element).  NRT_SOFTPLUS_POLY: the log term as u * q(u), u = exp(-|x|),
    // q a degree-3 minimax polynomial (|error| <= 7.1e-5, a quarter of an fp16 ulp of the result): one MUFU.
#if NRT_SOFTPLUS_POLY
    const float u = ex2_approx(-1.4426950408889634f * fabsf(x));
    float q = fmaf(-5.875710231e-02f, u, 2.256856408e-01f);
    q = fmaf(q, u, -4.713012532e-01f);
    q = fmaf(q, u, 9.974489612e-01f);
    return fmaf(q, u, fmaxf(x, 0.0f));
#else
    return fmaf(0.6931471805599453f, lg2_approx(1.0f + ex2_approx(-1.4426950408889634f * fabsf(x))), fmaxf(x, 0.0f));
#endif
  } else {
    return fmaxf(x, 0.01f * x);
  }
}
// act(a), act(b) rounded to the operand format and packed; the leaky ReLU runs on the packed pair
template <int ACT, int FMT>
__device__ __forceinline__ uint32_t act_pack(float a, float b) {
  if constexpr (ACT == NRT_ACT_SOFTPLUS) {
    return Elem<FMT>::pack(act_fast<ACT>(a), act_fast<ACT>(b));
  } else if constexpr (FMT == 0) {
    const __half2 h = __floats2half2_rn(a, b);
    const __half2 r = __hmax2(h, __hmul2(h, __floats2half2_rn(0.01f, 0.01f)));
    return *reinterpret_cast<const uint32_t*>(&r);
  } else {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const __nv_bfloat162 r = __hmax2(h, __hmul2(h, __floats2bfloat162_rn(0.01f, 0.01f)));
    return *reinterpret_cast<const uint32_t*>(&r);
  }
}
// 32 accumulator columns -> act -> 16 packed operand columns.  Written structure-of-arrays over groups of 8
// elements so that every step is 8 independent instructions: a single epilogue warp has its SM sub-partition
// (almost) to itself, so the conversion runs at the speed of its dependent chains unless the ILP is explicit
// (the straight per-pair loop over a whole 128-column row measured ~4 cycles per instruction).
template <int ACT, int FMT>
__device__ __forceinline__ void convert32(const uint32_t* __restrict__ acc, uint32_t* __restrict__ pk) {
  if constexpr (ACT == NRT_ACT_SOFTPLUS) {
#if NRT_SOFTPLUS_POLY == 2
    if constexpr (FMT == 0) {
      // packed-half form: one F2FP per pair up front, exponent argument / polynomial / max on half2 (half the issue
      // slots of the fp32 form), MUFU.EX2.F16 per element
      const __half2 kL = __floats2half2_rn(-1.4426950408889634f, -1.4426950408889634f);
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        __half2 x[8], u[8], q[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = __floats2half2_rn(__uint_as_float(acc[16 * g + 2 * i]), __uint_as_float(acc[16 * g + 2 * i + 1]));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 t = __hmul2(__habs2(x[i]), kL);
          uint32_t tu = *reinterpret_cast<const uint32_t*>(&t), uu;
          asm("ex2.approx.f16x2 %0, %1;" : "=r"(uu) : "r"(tu));
          u[i] = *reinterpret_cast<__half2*>(&uu);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) q[i] = __hfma2(__floats2half2_rn(-5.875710231e-02f, -5.875710231e-02f), u[i], __floats2half2_rn(2.256856408e-01f, 2.256856408e-01f));
#pragma unroll
        for (int i = 0; i < 8; ++i) q[i] = __hfma2(q[i], u[i], __floats2half2_rn(-4.713012532e-01f, -4.713012532e-01f));
#pragma unroll
        for (int i = 0; i < 8; ++i) q[i] = __hfma2(q[i], u[i], __floats2half2_rn(9.974489612e-01f, 9.974489612e-01f));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 r = __hfma2(q[i], u[i], __hmax2(x[i], __floats2half2_rn(0.0f, 0.0f)));
          pk[8 * g + i] = *reinterpret_cast<const uint32_t*>(&r);
        }
      }
      return;
    }
#endif
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float x[8], u[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = __uint_as_float(acc[8 * g + i]);
#pragma unroll
      for (int i = 0; i < 8; ++i) u[i] = ex2_approx(-1.4426950408889634f * fabsf(x[i]));
#if NRT_SOFTPLUS_POLY
      // log1p(u) = u * q(u) on (0,1]: degree-4 minimax polynomial without constant term (max error 7.1e-5, a quarter of
      // an fp16 ulp of the result where it matters) on the FMA pipe instead of a second MUFU; max(x,0) is the addend
      // of the last FMA.  ncu shows the XU pipe (MUFU + F2FP) 60-77 % busy with the two-MUFU form.
      float q[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) q[i] = fmaf(-5.875710231e-02f, u[i], 2.256856408e-01f);
#pragma unroll
      for (int i = 0; i < 8; ++i) q[i] = fmaf(q[i], u[i], -4.713012532e-01f);
#pragma unroll
      for (int i = 0; i < 8; ++i) q[i] = fmaf(q[i], u[i], 9.974489612e-01f);
#pragma unroll
      for (int i = 0; i < 8; ++i) u[i] = fmaf(q[i], u[i], fmaxf(x[i], 0.0f));
#else
#pragma unroll
      for (int i = 0; i < 8; ++i) u[i] = lg2_approx(1.0f + u[i]);
#pragma unroll
      for (int i = 0; i < 8; ++i) u[i] = fmaf(0.6931471805599453f, u[i], fmaxf(x[i], 0.0f));
#endif
#pragma unroll
      for (int i = 0; i < 4; ++i) pk[4 * g + i] = Elem<FMT>::pack(u[2 * i], u[2 * i + 1]);
    }
  } else {
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      uint32_t h[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) h[i] = Elem<FMT>::pack(__uint_as_float(acc[16 * g + 2 * i]), __uint_as_float(acc[16 * g + 2 * i + 1]));
      if constexpr (FMT == 0) {
        __half2 m[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) m[i] = __hmul2(*reinterpret_cast<__half2*>(&h[i]), __floats2half2_rn(0.01f, 0.01f));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 r = __hmax2(*reinterpret_cast<__half2*>(&h[i]), m[i]);
          pk[8 * g + i] = *reinterpret_cast<const uint32_t*>(&r);
        }
      } else {
        __nv_bfloat162 m[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) m[i] = __hmul2(*reinterpret_cast<__nv_bfloat162*>(&h[i]), __floats2bfloat162_rn(0.01f, 0.01f));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&h[i]), m[i]);
          pk[8 * g + i] = *reinterpret_cast<const uint32_t*>(&r);
        }
      }
    }
  }
}
// ---- saved-activation tiles (training) -------------------------------------------------------------------
// A saved tensor [M x F] is stored as one block per 128-sample tile in the UMMA canonical MN-major (no swizzle)
// layout with MN = feature, K = sample: 8x8 core matrices whose rows are 8 consecutive FEATURES (16 bytes) of one
// sample, 8 samples per core matrix, feature groups 128 bytes apart, sample groups FR*16 bytes apart:
//     element (feature f, sample s) of a tile with FR rows  ->  ((s/8)*(FR/8) + f/8)*64 + (s%8)*8 + f%8.
// The epilogue thread that owns sample s therefore writes its row with 16-byte vector stores (8 lanes = 128
// contiguous bytes), and the weight-gradient kernel pulls a whole tile into shared memory with one bulk copy and
// feeds it to tcgen05.mma as is (K' = samples, a_major = b_major = MN).  Activation tiles carry 16 extra rows;
// row F is the constant 1 (its product with dZ is the bias gradient), rows F+1..F+15 are never written nor used.
constexpr int kTileRowsExtra = 16;
struct NoSave { static constexpr bool kOn = false; static constexpr bool kF32 = false; };
// fp32 activations for the fused fp32 backward (nrt_mlp_backward): acts[(l * H + k) * M + m]
struct SaveF32 { static constexpr bool kOn = false; static constexpr bool kF32 = true; float* acts; int64_t M; };
struct SaveTiles {
  static constexpr bool kOn = true;
  static constexpr bool kF32 = false;
  uint16_t* acts;      // [L+1][ntiles] tiles of (H+16) x 128: a_l = act(z) feeding hidden layer l (l = L: output layer)
  uint16_t* enc_raw;   // [ntiles] tiles of (KE+16) x 128: the encoding as the init layer sees it
  uint16_t* enc_act;   // [ntiles] tiles of (KE+16) x 128: act(encoding) as the skip layers see it
  uint32_t* masks;     // [L+1][H/32][ntiles*128]: sign bits of a_l (what leaky_relu' needs), one word per 32 features
  int64_t ntiles;
};
// sign bits of 16 packed 16-bit pairs (32 features) -> one word, bit j = sign of feature j
__device__ __forceinline__ uint32_t sign_mask32(const uint32_t* pk) {
  uint32_t w = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    // high bytes of the four halves of two registers -> one register; keep the sign bits; gather them into a nibble
    const uint32_t b = __byte_perm(pk[2 * q], pk[2 * q + 1], 0x7531) & 0x80808080u;
    w |= ((b * 0x00204081u) >> 28) << (4 * q);
  }
  return w;
}
// thread-private view of one tile: pointer to (feature 0, this thread's sample)
__device__ __forceinline__ uint16_t* tile_row_ptr(uint16_t* tiles, int64_t tile, int FR, int s) {
  return tiles + tile * (int64_t)(FR * 128) + (s >> 3) * (FR * 8) + (s & 7) * 8;
}
__device__ __forceinline__ int tile_elem(int f) { return (f >> 3) * 64 + (f & 7); }   // offset of feature f in a row view
// stores NP packed pairs = features col0 .. col0+2NP-1 of this thread's sample (col0 % 8 == 0, NP % 4 == 0)
template <int NP>
__device__ __forceinline__ void save_cols(uint16_t* row, int col0, const uint32_t* pk) {
  static_assert(NP % 4 == 0, "whole 8-feature groups");
#pragma unroll
  for (int g = 0; g < NP / 4; ++g)
    *reinterpret_cast<uint4*>(row + ((col0 >> 3) + g) * 64) = make_uint4(pk[4 * g], pk[4 * g + 1], pk[4 * g + 2], pk[4 * g + 3]);
}
template <int FMT> __device__ __forceinline__ uint16_t one16() { return FMT == 0 ? (uint16_t)0x3C00 : (uint16_t)0x3F80; }

// One accumulator row (H fp32 columns at dD) -> activated 16-bit operand columns at aU, in 32-column chunks:
// the tcgen05.ld of chunk c+1 is in flight while chunk c is converted (64 + 16 live registers instead of 192).
// (H here is the number of columns THIS thread converts: the whole layer, or one half of it in the 8-warp variant;
//  dD / aU already point at the thread's first column, col0 is that column's index for the saved tile)
template <int ACT, int FMT, int H, bool SAVE = false>
__device__ __forceinline__ void convert_row(uint32_t dD, uint32_t aU, uint16_t* save_row = nullptr, int col0 = 0,
                                            int one_col = -1, uint32_t* mask_ptr = nullptr, int64_t mask_stride = 0) {
  static_assert(H % 32 == 0, "hidden width must be a multiple of 32");
  constexpr int NC = H / 32;
  uint32_t buf[2][32];
  TmemIO<32>::ld(dD, buf[0]);
  tc_wait_ld();
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (c + 1 < NC) TmemIO<32>::ld(dD + 32 * (c + 1), buf[(c + 1) & 1]);
    uint32_t pk[16];
    convert32<ACT, FMT>(buf[c & 1], pk);
    TmemIO<16>::st(aU + 16 * c, pk);
    if constexpr (SAVE) {
      save_cols<16>(save_row, col0 + 32 * c, pk);
      mask_ptr[(int64_t)(col0 / 32 + c) * mask_stride] = sign_mask32(pk);
    }
    if (c + 1 < NC) tc_wait_ld();
  }
  if constexpr (SAVE) { if (one_col >= 0) save_row[tile_elem(one_col)] = one16<FMT>(); }
}

// Softplus rows (NRT_SOFTPLUS_FULLROW): the WHOLE accumulator row goes into registers first.  The accumulator is
// then free, so `pre` (next layer's bias: LDS + tcgen05.st) runs under the conversion instead of after it, and the
// four 32-column conversions form one basic block without tcgen05.wait::ld in between: the MUFU pipe of a warp that has
// its SM sub-partition to itself stays busy across the chunk boundaries (timeline of the chunked form: 2,050 cycles per
// row for 1,024 cycles of MUFU, the pipeline drains at every wait).
template <int ACT, int FMT, int H, class PRE>
__device__ __forceinline__ void convert_row_full(uint32_t dD, uint32_t aU, PRE pre) {
  static_assert(H % 32 == 0, "hidden width must be a multiple of 32");
  constexpr int NC = H / 32;
  uint32_t acc[H];
  tmem_load<H>(dD, acc);
  tc_wait_ld();
  pre();
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    uint32_t pk[16];
    convert32<ACT, FMT>(acc + 32 * c, pk);
    TmemIO<16>::st(aU + 16 * c, pk);
  }
}

// Softplus rows, software pipelined (NRT_SOFTPLUS_PIPE): 16-column chunks, the exponentials (MUFU, one per 8 cycles
// and sub-partition) of chunk k+1 are issued between the polynomial FMAs of chunk k, while chunk k+2 is being loaded.
// A lone warp otherwise alternates between a MUFU-bound phase with idle issue slots and an FMA phase with an idle
// MUFU pipe (timeline: 1,950 cycles per 128-column row for ~1,050 cycles of either).  `pre` (next layer's bias into the
// accumulator) runs as soon as the last chunk has been read.
template <int FMT, int H, int FORM, class PRE>
__device__ __forceinline__ void convert_row_pipe(uint32_t dD, uint32_t aU, PRE pre, long long* t_dbg = nullptr) {
  static_assert(H % 16 == 0 && H >= 48, "pipelined softplus conversion: at least three 16-column chunks");
  constexpr int NC = H / 16;
  uint32_t xb[3][16];
  float u[2][16];
  TmemIO<16>::ld(dD, xb[0]);
  TmemIO<16>::ld(dD + 16, xb[1]);
  tc_wait_ld();
#pragma unroll
  for (int i = 0; i < 16; ++i) u[0][i] = ex2_approx(-1.4426950408889634f * fabsf(__uint_as_float(xb[0][i])));
#ifdef NRT_DBG_CONV
  if (t_dbg) t_dbg[0] = clock64();
#endif
#pragma unroll
  for (int k = 0; k < NC; ++k) {
    if (k + 2 < NC) TmemIO<16>::ld(dD + 16 * (k + 2), xb[(k + 2) % 3]);
    uint32_t pk[8];
    if constexpr (FORM == 3 && FMT == 0) {
      // exponent argument and MUFU in fp32 (accurate for large |x|), then u and x packed: polynomial and max on half2
      // (11 instead of 15 instructions per pair; the result is rounded twice: ~1 fp16 ulp instead of 0.5)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (k + 1 < NC) {
          u[(k + 1) & 1][2 * i] = ex2_approx(-1.4426950408889634f * fabsf(__uint_as_float(xb[(k + 1) % 3][2 * i])));
          u[(k + 1) & 1][2 * i + 1] = ex2_approx(-1.4426950408889634f * fabsf(__uint_as_float(xb[(k + 1) % 3][2 * i + 1])));
        }
        const __half2 uu = __floats2half2_rn(u[k & 1][2 * i], u[k & 1][2 * i + 1]);
        // max(x, 0) of the pair in the conversion itself (cvt.rn.relu: one instruction instead of F2FP + HMNMX2; the
        // epilogue warp is bound by its instruction count)
        uint32_t rx;
        asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(rx) : "f"(__uint_as_float(xb[k % 3][2 * i + 1])), "f"(__uint_as_float(xb[k % 3][2 * i])));
        __half2 q = __hfma2(__floats2half2_rn(-5.875710231e-02f, -5.875710231e-02f), uu, __floats2half2_rn(2.256856408e-01f, 2.256856408e-01f));
        q = __hfma2(q, uu, __floats2half2_rn(-4.713012532e-01f, -4.713012532e-01f));
        q = __hfma2(q, uu, __floats2half2_rn(9.974489612e-01f, 9.974489612e-01f));
        const __half2 r = __hfma2(q, uu, *reinterpret_cast<const __half2*>(&rx));
        pk[i] = *reinterpret_cast<const uint32_t*>(&r);
      }
    } else {
    float r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (k + 1 < NC) u[(k + 1) & 1][i] = ex2_approx(-1.4426950408889634f * fabsf(__uint_as_float(xb[(k + 1) % 3][i])));
      const float uu = u[k & 1][i], xx = __uint_as_float(xb[k % 3][i]);
      // log1p(u) = u * q(u), q of degree 4: |error| <= 9.9e-6 (the fp16 rounding of the result is >= 6e-5 for results
      // above 0.125); with degree 3 (7.1e-5) the DTU step's most position-sensitive gradient (sp_var_fn.init.weight,
      // sigma = 128) drops from cosine 0.9975 to 0.9964 against the reference: more rays stop one march step apart
      float q = fmaf(3.215182172e-02f, uu, -1.360436010e-01f);
      q = fmaf(q, uu, 2.894552203e-01f);
      q = fmaf(q, uu, -4.919007447e-01f);
      q = fmaf(q, uu, 9.994943976e-01f);
      r[i] = fmaf(q, uu, fmaxf(xx, 0.0f));
      if (i & 1) pk[i >> 1] = Elem<FMT>::pack(r[i - 1], r[i]);
    }
    }
    TmemIO<8>::st(aU + 8 * k, pk);
    if (k + 2 < NC) tc_wait_ld();
#ifdef NRT_DBG_CONV
    if (t_dbg && k + 3 == NC) t_dbg[1] = clock64();
#endif
    if (k + 3 == NC) pre();   // every accumulator column has been read
  }
}

// K-split variant (see Net::KSPLIT): whole row into registers, `pre()` (bias of the next layer into the now free
// accumulator, in-place encoding activation), first half -> arrive on bar_a, second half -> arrive on bar_b.
template <int ACT, int FMT, int H, class PRE>
__device__ __forceinline__ void convert_row_split(uint32_t dD, uint32_t aU, uint64_t* bar_a, uint64_t* bar_b, PRE pre,
                                                  long long* t_loaded = nullptr, long long* t_a = nullptr) {
  static_assert(H % 64 == 0, "two halves of whole 32-column chunks");
  constexpr int NC = H / 32;
  uint32_t acc[H];
  tmem_load<H>(dD, acc);
  tc_wait_ld();
  if (t_loaded) *t_loaded = clock64();
  pre();
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    uint32_t pk[16];
    convert32<ACT, FMT>(acc + 32 * c, pk);
    TmemIO<16>::st(aU + 16 * c, pk);
    if (c == NC / 2 - 1) {
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(bar_a);
      if (t_a) *t_a = clock64();
      // keep the compiler from hoisting the second half's conversion above the arrive (volatile asm statements
      // stay in order; the conversion is register-only code and would otherwise be scheduled first)
#pragma unroll
      for (int i = H / 2; i < H; ++i) asm volatile("" : "+r"(acc[i]));
    }
  }
  tc_wait_st();
  tc_fence_before();
  mbar_arrive(bar_b);
}

// Last hidden layer of a network with a tiny output layer: act(accumulator row) . W_out (fp32, [H][4] in shared
// memory, broadcast reads) accumulated on the fly; o[] must hold the output bias on entry.
template <int ACT, int FMT, int H, int OUT, bool SAVE, bool POLY = (NRT_SOFTPLUS_POLY != 0)>
__device__ __forceinline__ void convert_row_out(uint32_t dD, const float* __restrict__ wout, float* __restrict__ o,
                                                uint16_t* save_row = nullptr, uint32_t* mask_ptr = nullptr,
                                                int64_t mask_stride = 0) {
  static_assert(H % 32 == 0 && OUT <= 4, "fused output layer");
  constexpr int NC = H / 32;
  uint32_t buf[2][32];
  TmemIO<32>::ld(dD, buf[0]);
  tc_wait_ld();
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (c + 1 < NC) TmemIO<32>::ld(dD + 32 * (c + 1), buf[(c + 1) & 1]);
    uint32_t pk[16];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float a[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = __uint_as_float(buf[c & 1][8 * g + i]);
      if constexpr (ACT == NRT_ACT_SOFTPLUS) {
        float u[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) u[i] = ex2_approx(-1.4426950408889634f * fabsf(a[i]));
        if constexpr (POLY) {
          float q[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) q[i] = fmaf(-5.875710231e-02f, u[i], 2.256856408e-01f);
#pragma unroll
          for (int i = 0; i < 8; ++i) q[i] = fmaf(q[i], u[i], -4.713012532e-01f);
#pragma unroll
          for (int i = 0; i < 8; ++i) q[i] = fmaf(q[i], u[i], 9.974489612e-01f);
#pragma unroll
          for (int i = 0; i < 8; ++i) a[i] = fmaf(q[i], u[i], fmaxf(a[i], 0.0f));
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) u[i] = lg2_approx(1.0f + u[i]);
#pragma unroll
          for (int i = 0; i < 8; ++i) a[i] = fmaf(0.6931471805599453f, u[i], fmaxf(a[i], 0.0f));
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = fmaxf(a[i], 0.01f * a[i]);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 w = *reinterpret_cast<const float4*>(wout + (32 * c + 8 * g + i) * 4);
        o[0] = fmaf(a[i], w.x, o[0]);
        if constexpr (OUT > 1) o[1] = fmaf(a[i], w.y, o[1]);
        if constexpr (OUT > 2) o[2] = fmaf(a[i], w.z, o[2]);
        if constexpr (OUT > 3) o[3] = fmaf(a[i], w.w, o[3]);
      }
      if constexpr (SAVE) {
#pragma unroll
        for (int i = 0; i < 4; ++i) pk[4 * g + i] = Elem<FMT>::pack(a[2 * i], a[2 * i + 1]);
      }
    }
    if constexpr (SAVE) {
      save_cols<16>(save_row, 32 * c, pk);
      mask_ptr[(int64_t)c * mask_stride] = sign_mask32(pk);
    }
    if (c + 1 < NC) tc_wait_ld();
  }
  if constexpr (SAVE) save_row[tile_elem(H)] = one16<FMT>();
}

// Training forward with a tensor-core forward and the fused fp32 backward (256-wide nets, NeuralBSDF, occlusion MLP):
// the forward kernel also writes the post-activation layer inputs in the layout of
// the fused fp32 backward (nrt_mlp_backward: acts[(l * H + k) * M + m], fp32) -- the values the next layer's operand
// actually holds (rounded to the operand format), so the backward differentiates the forward that ran.  For fixed k
// the 32 lanes of a warp write 32 consecutive samples: coalesced 128-byte stores.
template <int ACT, int FMT, int H>
__device__ __forceinline__ void convert_row_savef32(uint32_t dD, uint32_t aU, float* __restrict__ acts, int64_t stride) {
  constexpr int NC = H / 32;
  uint32_t buf[2][32];
  TmemIO<32>::ld(dD, buf[0]);
  tc_wait_ld();
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (c + 1 < NC) TmemIO<32>::ld(dD + 32 * (c + 1), buf[(c + 1) & 1]);
    uint32_t pk[16];
    convert32<ACT, FMT>(buf[c & 1], pk);
    TmemIO<16>::st(aU + 16 * c, pk);
    if (acts != nullptr) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        acts[(int64_t)(32 * c + 2 * i) * stride] = Elem<FMT>::back((uint16_t)(pk[i] & 0xffffu));
        acts[(int64_t)(32 * c + 2 * i + 1) * stride] = Elem<FMT>::back((uint16_t)(pk[i] >> 16));
      }
    }
    if (c + 1 < NC) tc_wait_ld();
  }
}
// last hidden layer with the fused (out <= 4) output layer: activations stay fp32 here, and are saved as such
template <int ACT, int FMT, int H, int OUT>
__device__ __forceinline__ void convert_row_out_savef32(uint32_t dD, const float* __restrict__ wout, float* __restrict__ o,
                                                        float* __restrict__ acts, int64_t stride) {
  constexpr int NC = H / 32;
  uint32_t buf[2][32];
  TmemIO<32>::ld(dD, buf[0]);
  tc_wait_ld();
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (c + 1 < NC) TmemIO<32>::ld(dD + 32 * (c + 1), buf[(c + 1) & 1]);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float z = __uint_as_float(buf[c & 1][i]);
      const float a = act_fast<ACT>(z);
      const float4 w = *reinterpret_cast<const float4*>(wout + (32 * c + i) * 4);
      o[0] = fmaf(a, w.x, o[0]);
      if constexpr (OUT > 1) o[1] = fmaf(a, w.y, o[1]);
      if constexpr (OUT > 2) o[2] = fmaf(a, w.z, o[2]);
      if constexpr (OUT > 3) o[3] = fmaf(a, w.w, o[3]);
      if (acts != nullptr) acts[(int64_t)(32 * c + i) * stride] = a;
    }
    if (c + 1 < NC) tc_wait_ld();
  }
}

// leaky_relu on a packed 16-bit pair
template <int FMT>
__device__ __forceinline__ uint32_t leaky_packed(uint32_t v) {
  if constexpr (FMT == 0) {
    const __half2 h = *reinterpret_cast<const __half2*>(&v);
    const __half2 r = __hmax2(h, __hmul2(h, __floats2half2_rn(0.01f, 0.01f)));
    return *reinterpret_cast<const uint32_t*>(&r);
  } else {
    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&v);
    const __nv_bfloat162 r = __hmax2(h, __hmul2(h, __floats2bfloat162_rn(0.01f, 0.01f)));
    return *reinterpret_cast<const uint32_t*>(&r);
  }
}

// D[lane][0..N) = bias[0..N): the next layer's MMA then only accumulates (no bias add in its epilogue)
template <int N>
__device__ __forceinline__ void preload_bias(uint32_t dD, const float* __restrict__ bias) {
  static_assert(N % 8 == 0, "bias pieces are multiples of 8 columns");
  uint32_t r[N];
#pragma unroll
  for (int j = 0; j < N / 4; ++j) {
    const float4 b = *reinterpret_cast<const float4*>(bias + 4 * j);
    r[4 * j] = __float_as_uint(b.x); r[4 * j + 1] = __float_as_uint(b.y);
    r[4 * j + 2] = __float_as_uint(b.z); r[4 * j + 3] = __float_as_uint(b.w);
  }
  tmem_store<N>(dD, r);
}
__device__ __forceinline__ void sincos_fast(float x, float* s, float* c) {
  // two-constant reduction by 2*pi, then MUFU sin/cos on [-pi, pi]
  const float k = rintf(x * 0.15915494309189535f);
  float r = fmaf(-k, 6.2831854820251465f, x);
  r = fmaf(-k, -1.7484555314695172e-07f, r);
  *s = __sinf(r);
  *c = __cosf(r);
}

// ---------------------------------------------------------------------------------------------
// compile-time network description
// ---------------------------------------------------------------------------------------------
// RENDER: the net reads the render layout (make_render_layout), which the pack appends to the training layout in the same
// blob at BLOB_OFF; inference kernels only (k_mlp_tc without saved activations).
template <int IN_, int LAT_, int F_, int H_, int L_, int SKIP_, int OUT_, int ACT_, bool RENDER = false>
struct Net {
  static constexpr int IN = IN_, LAT = LAT_, F = F_, H = H_, L = L_, SKIP = SKIP_, OUT = OUT_, ACT = ACT_;
  static constexpr Layout Y = RENDER ? make_render_layout(IN, LAT, F, H, L, SKIP, OUT) : make_layout(IN, LAT, F, H, L, SKIP, OUT);
  static constexpr int BLOB_OFF = RENDER ? (make_layout(IN, LAT, F, H, L, SKIP, OUT).bytes + 127) / 128 * 128 : 0;
  static constexpr BiasRows BR = RENDER ? render_bias_rows(IN, LAT, F, H, L, SKIP, OUT) : no_bias_rows();
  static constexpr bool BIAS_ROWS = RENDER;
  static constexpr bool SPLIT = Y.split != 0;
  static constexpr int XR = Y.XR, KE = Y.KE, KX = Y.KX, KPH = Y.KPH, FP = Y.FP, NOP = Y.NOP, KRAW = Y.KRAW;
  static constexpr int DC = imax(H, imax(NOP, FP));       // fp32 accumulator columns
  // TMEM plan per tile slot.  Standard: accumulator | union region (phase-GEMM operand -> raw encoding -> hidden
  // activations) | act(encoding).  In-place plan: the raw encoding is written into the encoding region, read there by
  // the init layer's MMA, and converted to act(encoding) IN PLACE by the first hidden epilogue (nothing reads the raw
  // encoding after the init layer); the union region then only holds the phase operand / hidden activations.  It is
  // used when it buys another tile slot (NeRFLE.second: 176 -> 160 columns = three tiles in flight).
  static constexpr int EC = KE / 2;                       // (act) encoding region
  static constexpr int UC_STD = imax(H, imax(KE, KX)) / 2;
  static constexpr int UC_INP = imax(H, KX) / 2;
  static constexpr int kMaxSlots = 3;
  static constexpr int slots_of(int cols) { return 512 / cols < kMaxSlots ? 512 / cols : kMaxSlots; }
  static constexpr bool INPLACE = (ACT == NRT_ACT_LEAKY_RELU) && LAT == 0 &&
                                  slots_of(DC + UC_INP + EC) > slots_of(DC + UC_STD + EC);
  static constexpr int UC = INPLACE ? UC_INP : UC_STD;
  static constexpr int COLS = DC + UC + EC;
  static constexpr int NSLOT = slots_of(COLS);
  static constexpr int NWG = NSLOT < 2 ? 2 : NSLOT;       // epilogue warpgroups launched
  static constexpr int STAGES = L + 3;                    // encode, init, L layers, out
  // Two of those stages need no tensor core and cost a full MMA -> commit -> wait round trip each:
  //  * split-precision inputs (in <= 5): the Fourier phases are in*F FMAs per sample -> computed in fp32 by the
  //    epilogue thread that owns the sample, together with sin / cos, BEFORE the first MMA (stage 0 disappears);
  //  * out <= 4: the output layer is H*out FMAs per sample -> accumulated in fp32 while the last hidden
  //    activations are produced (the last stage disappears, and that layer no longer rounds to 16 bits).
  // warps per tile slot.  8 = two warps per TMEM lane quarter, each converting half of the columns of a hidden layer
  // (k_mlp_tc implements both).  Measured on B200 the 8-warp variant is SLOWER (NeRFLE.first +6 %, .second +25 %,
  // SDF march +15 %): the epilogue is bound by the throughput of the conversion pipes of the SM sub-partition
  // (F2FP.PACK_AB ~4 cycles, HMUL2 / HMNMX2 2 cycles per warp instruction: ~512 cycles per 128x128 tile layer),
  // not by the latency of one warp's dependent chain, and 17 warps cap the kernel at 96 registers per thread.
#ifndef NRT_SOFTPLUS_WPS
#define NRT_SOFTPLUS_WPS 4
#endif
  static constexpr int WPS = ACT == NRT_ACT_SOFTPLUS ? NRT_SOFTPLUS_WPS : 4;
  // K-split early start (k_mlp_tc): a hidden epilogue pulls the WHOLE accumulator row into registers first (the
  // accumulator is then free: bias in), converts the first half of the columns, arrives on `ready_a`, converts the
  // second half, arrives on `ready`.  The MMA warp issues the K-chunks of the first half (and the encoding chunks of
  // a skip layer) on `ready_a`, i.e. UNDER the conversion of the second half, and only the remaining chunks after
  // `ready`: the per-layer dependency chain  MMA -> epilogue -> MMA  loses about half a layer of tensor time.
#ifndef NRT_KSPLIT
#define NRT_KSPLIT 0
#endif
  static constexpr bool KSPLIT = NRT_KSPLIT != 0 && H % 64 == 0 && H <= 128;
  static constexpr bool ENC_CUDA = Y.basis_f32_off >= 0;
  static constexpr bool FUSE_OUT = Y.wout_f32_off >= 0;
  static constexpr int FIRST_STAGE = ENC_CUDA ? 1 : 0;
  static constexpr int END_STAGE = FUSE_OUT ? STAGES - 1 : STAGES;   // one past the last MMA stage
  static constexpr bool FITS_TMEM = COLS <= 512;          // asserted by k_mlp_tc (the wide kernel has its own plan)
  static_assert(XR % 16 == 0 && F % 16 == 0 && LAT % 16 == 0 && KRAW == KE, "encoding segments must be multiples of 16");
  static_assert(!SPLIT || 3 * IN <= 16, "split encoding needs 3*in <= 16");
  static_assert(H % 16 == 0 && H <= 256, "hidden must be a multiple of 16");
  // Weights that do not fit in shared memory are STREAMED: each tile slot owns two stage buffers and the MMA warp
  // prefetches the next stage's operand (cp.async.bulk from L2) while the current stage computes.
  static constexpr bool STREAM = Y.bytes > kSmemBudget;
  // Bias K-chunks (NRT_BIAS_MMA, see make_layout and make_render_layout): the constant A chunk [1, 1, 1, 0, ...] takes 8
  // TMEM columns after the slots (NeRFLE.second: 3 x 160 + 8 = 488 of 512 point light, 2 x 208 + 8 = 424 environment
  // light; NeRFLE.first: 2 x 216 + 8 = 440)
  static constexpr int ONES_COL = NSLOT * COLS;
  static constexpr int BK_OFF = bk_off(Y);
  static constexpr bool BIAS_MMA = (BK_OFF >= 0 && !STREAM && FUSE_OUT && ONES_COL + 8 <= 512) || RENDER;
  static_assert(!RENDER || (Y.bytes <= kSmemBudget && ONES_COL + 8 <= 512 && render_layout_ok(Y, BR)),
                "render layout: resident in shared memory, room for the constant A chunk in TMEM, bias rows and chunks in place");
  // One MMA-issuing warp per tile slot for the networks with resident weights (NRT_MMA_WARP_PER_SLOT=0: always a
  // single warp that serves the slots in ready order).  Measured on B200: NeRFLE.first 32.3 -> 30.7 ms, .second
  // 32.2 -> 24.3 ms per 800x800x192 frame; the weight-streaming softplus SDF net is SFU-bound in its epilogue and
  // is 7 % FASTER with the single warp (march 10.6 vs 11.3 ms), so it keeps one.
#ifndef NRT_MMA_WARP_PER_SLOT
#define NRT_MMA_WARP_PER_SLOT 1
#endif
#ifndef NRT_MMA_WARP_PER_SLOT_STREAM
#define NRT_MMA_WARP_PER_SLOT_STREAM 0
#endif
  // Self-issue (NRT_SELF_ISSUE, the streamed softplus net): NO MMA warp.  The first epilogue warp of each tile slot
  // waits for its slot's `ready` barrier after its own arrive (it would only wait for `done` otherwise) and issues the
  // stage itself, under a CTA-wide lock so that the two slots' tcgen05.mma batches do not interleave.  8 (16) warps
  // instead of 9 (17): two (four) warps per SM sub-partition and therefore 255 (128) registers per thread instead of
  // 168 (96) -- ptxas caps at 16 K registers / warps of the fullest sub-partition.
#ifndef NRT_SELF_ISSUE
#define NRT_SELF_ISSUE 0
#endif
  static constexpr bool SELF = NRT_SELF_ISSUE != 0 && STREAM && ACT == NRT_ACT_SOFTPLUS && ENC_CUDA && FUSE_OUT && NSLOT == 2;
  static constexpr int NMMA = SELF ? 0 : ((STREAM ? NRT_MMA_WARP_PER_SLOT_STREAM != 0 : NRT_MMA_WARP_PER_SLOT != 0) ? NSLOT : 1);
  static constexpr int threads(int wps) { return NWG * wps * 32 + 32 * NMMA; }
  static constexpr int max_op_bytes() {
    int m = 0;
    for (int o = 0; o < Y.n_ops; ++o) m = imax(m, Y.opN[o] * Y.opK[o] * 2);
    return m;
  }
  static constexpr int MAXOP = max_op_bytes();
  static constexpr int BIAS_BYTES = Y.bias_floats * 4;
  static constexpr int SMEM_BYTES = STREAM ? NSLOT * 2 * MAXOP + BIAS_BYTES : Y.bytes;
  static constexpr bool FITS_SMEM = SMEM_BYTES <= kSmemBudget;
};

constexpr int kEpiThreads = 128;

// Issues the MMAs of stage ST of one tile slot.  Called by the WHOLE MMA warp (convergent); one elected lane
// issues.  (Issuing from a divergent single lane makes the compiler wrap every UTCHMMA in an
// ELECT / R2UR / BRA.U.ANY serialisation loop: ~135 cycles per MMA instead of ~72, see profiles/.)
// PART 0: the whole stage; 1: first half of the hidden K-chunks + the encoding chunks, no commit (K-split, on
// `ready_a`); 2: second half of the hidden K-chunks + commit (on `ready`).
// BMMA: stages >= 1 start with the layer's bias K-chunk (NET::BIAS_MMA), which overwrites the accumulator.
// ZLO: leading 16-column chunks of the x_lo segment of the phase GEMM that are identically zero (a latent handed over
// already in the operand format has x_lo = 0); they are not issued.
template <class NET, int FMT, int ST, int PART = 0, bool BMMA = false, int ZLO = 0>
__device__ __forceinline__ void issue_stage(uint32_t b_addr, uint32_t dD, uint32_t aU, uint32_t aE, uint64_t* done_bar) {
  constexpr Layout Y = NET::Y;
  constexpr uint32_t N = (uint32_t)Y.opN[ST];
  constexpr uint32_t idesc = (1u << 4) | ((uint32_t)FMT << 7) | ((uint32_t)FMT << 10) | ((N >> 3) << 17) |
                             ((uint32_t)(128 >> 4) << 24);
  constexpr uint32_t lbo = N * 16, sbo = 128;
  constexpr int kch = Y.opK[ST] / 16;
  // K chunks taken from U: the hidden part of a hidden layer; everything for the other stages, except that the
  // in-place plan keeps the (raw) encoding in the encoding region for the init layer
  constexpr int k_u = (ST >= 2 && ST < NET::STAGES - 1) ? NET::H / 16 : ((NET::INPLACE && ST == 1) ? 0 : kch);
  if (elect_one()) {
    // resident weights: b_addr is the base of the weight area and the operand offset is a compile-time constant;
    // streamed weights: b_addr is the stage buffer
    const uint64_t bd0 = make_desc(NET::STREAM ? b_addr : b_addr + (uint32_t)Y.op_off[ST] * 2u, lbo, sbo);
    // render layout: the init and skip layers take their bias from the encoding's bias rows, so their first MMA starts
    // from zero; the other layers start with their 8-deep bias chunk
    constexpr bool kBiasChunk = BMMA && !NET::BIAS_ROWS && ST > 0 && ST < NET::END_STAGE;
    constexpr bool kBiasChunk8 = BMMA && NET::BIAS_ROWS && NET::BR.bk8_off[ST] >= 0;
    constexpr bool kFromZero = ST == 0 || (BMMA && NET::BIAS_ROWS && NET::BR.bk8_off[ST] < 0);
    if constexpr (kBiasChunk) {
      static_assert(NET::BIAS_MMA && N == (uint32_t)NET::H, "bias K-chunks: hidden-width MMA layers of a resident blob");
      mma_ts(dD, (uint32_t)NET::ONES_COL, make_desc(b_addr + (uint32_t)NET::BK_OFF + (uint32_t)(ST - 1) * N * 32u, lbo, sbo), idesc, 0u);
    }
    if constexpr (kBiasChunk8) {
      static_assert(!NET::STREAM, "bias chunks of a resident blob");
      mma_ts(dD, (uint32_t)NET::ONES_COL, make_desc(b_addr + (uint32_t)NET::BR.bk8_off[ST] * 2u, lbo, sbo), idesc, 0u);
    }
#pragma unroll
    for (int kc = 0; kc < kch; ++kc) {
      if (PART == 1 && kc >= k_u / 2 && kc < k_u) continue;
      if (PART == 2 && (kc < k_u / 2 || kc >= k_u)) continue;
      uint32_t a;
      if constexpr (ST == 0) {
        // hi+lo phase GEMM (K = 3*XR): chunks [x_hi | x_lo | x_hi] against [B_hi | B_hi | B_lo].  x_hi sits where the
        // raw encoding keeps it (in-place plan: the encoding region, else the union region), x_lo in the other one
        // (free until the epilogue of this stage has run).
        constexpr int xch = NET::XR / 16;
        static_assert(ZLO < xch, "the chunk with the non-latent x_lo columns stays");
        if (kc >= xch && kc < xch + ZLO) continue;
        const uint32_t hi = NET::INPLACE ? aE : aU, lo = NET::INPLACE ? aU : aE;
        a = (kc >= xch && kc < 2 * xch) ? (lo + (kc - xch) * 8) : (hi + (kc % xch) * 8);
      } else {
        a = (kc < k_u) ? (aU + kc * 8) : (aE + (kc - k_u) * 8);
      }
      // the phase GEMM (stage 0) starts from zero, and so do the layers with bias rows; every other layer's accumulator
      // holds its bias already: pre-loaded by the previous epilogue, or written by the bias chunk above
      mma_ts(dD, a, bd0 + (uint64_t)((kc * 2 * lbo) >> 4), idesc, (!kFromZero || kc > 0) ? 1u : 0u);
    }
    if (PART != 1) tc_commit(done_bar);
  }
  __syncwarp();
}
// runtime stage -> compile-time stage through a jump table (a linear if-chain cost up to ~150 cycles of taken
// branches per stage on the single issuing warp, which serves every tile slot)
template <class NET, int FMT, int PART = 0, bool BMMA = false, int ZLO = 0>
__device__ __forceinline__ void issue_stage_dyn(int st, uint32_t b_addr, uint32_t dD, uint32_t aU, uint32_t aE,
                                                uint64_t* done_bar) {
#define NRT_STAGE_CASE(S) case S: if constexpr (S < NET::STAGES && (PART == 0 || S >= 2)) issue_stage<NET, FMT, S, PART, BMMA, ZLO>(b_addr, dD, aU, aE, done_bar); break;
  switch (st) {
    NRT_STAGE_CASE(0) NRT_STAGE_CASE(1) NRT_STAGE_CASE(2) NRT_STAGE_CASE(3) NRT_STAGE_CASE(4) NRT_STAGE_CASE(5)
    NRT_STAGE_CASE(6) NRT_STAGE_CASE(7) NRT_STAGE_CASE(8) NRT_STAGE_CASE(9) NRT_STAGE_CASE(10) NRT_STAGE_CASE(11)
    NRT_STAGE_CASE(12) NRT_STAGE_CASE(13) NRT_STAGE_CASE(14) NRT_STAGE_CASE(15) NRT_STAGE_CASE(16) NRT_STAGE_CASE(17)
    NRT_STAGE_CASE(18) NRT_STAGE_CASE(19) NRT_STAGE_CASE(20) NRT_STAGE_CASE(21) NRT_STAGE_CASE(22)
    default: break;
  }
#undef NRT_STAGE_CASE
}
// bulk copy of one stage operand (<= 32 KB pieces) from the blob into a stage buffer; completes on `bar`
__device__ __forceinline__ void stream_op(uint8_t* dst, const uint8_t* src, uint32_t bytes, uint64_t* bar) {
  mbar_expect_tx(bar, bytes);
  for (uint32_t off = 0; off < bytes; off += 32768u) bulk_g2s(dst + off, src + off, min(32768u, bytes - off), bar);
}

// IO policy concepts.
//   tile policy:       struct IO { __device__ void load(int64_t m, float* x /*IN+LAT*/) const;
//                                  __device__ void store(int64_t m, const float* o /*OUT, bias added*/) const; };
//     sample m of the flat batch <-> row m % 128 of tile m / 128; tiles are dealt round-robin to the CTAs.
//   iterative policy:  struct IO { struct State; void init(State&); bool next(State&, float* x); void consume(State&, const float* o);
//                                  void finish(State&); };
//     every epilogue thread owns one *trajectory* (a marching ray): next() retires a finished trajectory, pulls a
//     new one from a global queue (warp-aggregated atomic) and produces the next evaluation point; consume()
//     takes the network output.  The tile slot keeps cycling while any of its 128 threads is live, so every MMA
//     row is (up to the queue tail) spent on a live ray: this is the compaction of the sphere-trace march.
template <class T, class = void> struct PackedPairsOf { static constexpr int value = 0; };
template <class T> struct PackedPairsOf<T, std::void_t<decltype(T::kPackedPairs)>> { static constexpr int value = T::kPackedPairs; };
// tile policies whose load() is a dependent global load followed by arithmetic can split it into fetch() (issue the loads
// into a `Fetch` record) and point() (the arithmetic); k_mlp_tc with NRT_FIRST_PIPE fetches one tile ahead
template <class T, class D, class = void> struct FetchOf { using type = D; };
template <class T, class D> struct FetchOf<T, D, std::void_t<typename T::Fetch>> { using type = typename T::Fetch; };
template <class T, class = void> struct HasCtaInit : std::false_type {};
template <class T> struct HasCtaInit<T, std::void_t<decltype(&T::cta_init)>> : std::true_type {};
template <class T, class = void> struct IsIterative : std::false_type {};
template <class T> struct IsIterative<T, std::void_t<typename T::State>> : std::true_type {};
struct NoState {};
template <class T, class = void> struct StateOf { using type = NoState; };
template <class T> struct StateOf<T, std::void_t<typename T::State>> { using type = typename T::State; };

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ptxas rounds the block size of __launch_bounds__ up to a multiple of 128 threads when it derives the register cap:
// the 288-thread kernels (8 epilogue warps + 1 MMA warp) get 168 registers, as if they had 384 threads.
// NRT_MAXNREG replaces the launch bound by an explicit __maxnreg__ = 64 K registers / threads (the two cannot be combined).
#ifdef NRT_MAXNREG
#define NRT_KMLP_BOUNDS(T) __maxnreg__(((65536 / (T)) / 8 * 8) > 255 ? 255 : ((65536 / (T)) / 8 * 8))
#else
#define NRT_KMLP_BOUNDS(T) __launch_bounds__(T, 1)
#endif
template <class NET, class IO, int FMT, class SV = NoSave, int WPS = NET::WPS>
__global__ void NRT_KMLP_BOUNDS(NET::threads(WPS))
k_mlp_tc(const uint8_t* __restrict__ blob, IO io, int64_t M, long long* __restrict__ dbg, SV sv = SV{}) {
  constexpr int EPI = WPS * 32;                 // epilogue threads per tile slot
  static_assert(NET::FITS_TMEM, "network does not fit in TMEM");
  static_assert(NET::FITS_SMEM, "stage buffers do not fit in shared memory");
  // dbg (development only, tools/tc_timeline.py): clock64 stamps of CTA 0 for a few tile iterations
  constexpr int kDbgIt0 = 4, kDbgIts = 4;
  auto stamp = [&](int it, int st, int slot, int k) {
    if (dbg != nullptr && slot < 2 && blockIdx.x == 0 && it >= kDbgIt0 && it < kDbgIt0 + kDbgIts)
      dbg[(((it - kDbgIt0) * NET::STAGES + st) * 2 + slot) * 8 + k] = clock64();
  };
  using E = Elem<FMT>;
  constexpr Layout Y = NET::Y;
  constexpr int H = NET::H, IN = NET::IN, LAT = NET::LAT, F = NET::F, L = NET::L;
  constexpr int NSLOT = NET::NSLOT;
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr bool STREAM = NET::STREAM;
  uint16_t* sW = reinterpret_cast<uint16_t*>(smem);
  const float* sBias = reinterpret_cast<const float*>(smem + (STREAM ? (size_t)NSLOT * 2 * NET::MAXOP : (size_t)Y.w_elems * 2));
  __shared__ __align__(8) uint64_t bar_w;
  __shared__ __align__(8) uint64_t bar_wfull[3][2];   // streaming: stage buffer b of slot s has landed
  __shared__ uint32_t s_opoff[NET::STAGES], s_opbytes[NET::STAGES];
  __shared__ __align__(8) uint64_t bar_ready[3];
  __shared__ __align__(8) uint64_t bar_ready_a[3];    // K-split: first half of the activations is in place
  __shared__ __align__(8) uint64_t bar_done[3];
  // K-split early start: not with the 8-warp epilogue, not while saving activation tiles (training forward)
  constexpr bool KSPLIT = NET::KSPLIT && WPS == 4 && !SV::kOn && !SV::kF32;
#ifndef NRT_SOFTPLUS_FULLROW
#define NRT_SOFTPLUS_FULLROW 0
#endif
#ifndef NRT_SOFTPLUS_PIPE
#define NRT_SOFTPLUS_PIPE 1
#endif
  constexpr bool kPipeRow = NRT_SOFTPLUS_PIPE != 0 && SoftplusOf<IO>::value != 0 && NET::ACT == NRT_ACT_SOFTPLUS && !KSPLIT &&
                            !SV::kOn && !SV::kF32;
  constexpr bool kFullRow = NRT_SOFTPLUS_FULLROW != 0 && !kPipeRow && NET::ACT == NRT_ACT_SOFTPLUS && !KSPLIT && !SV::kOn && !SV::kF32;
  __shared__ uint32_t tmem_base_s;
  __shared__ uint32_t s_bias[NET::STAGES];
  constexpr bool ITER = IsIterative<IO>::value;
  // bias K-chunks instead of the epilogue's bias preload (not in the training forward, which keeps the preload)
  constexpr bool BMMA = NET::BIAS_MMA && !KSPLIT && WPS == 4 && !SV::kOn && !SV::kF32;
  static_assert(BMMA || !NET::BIAS_ROWS, "the render layout has no fp32 biases to pre-load");
  // leading input pairs that the IO policy can hand over already packed in the operand format (IoNerfSecond); their x_lo
  // is zero, so the phase GEMM skips the ZLO x_lo chunks that hold nothing else
  constexpr int kPP = (!ITER && !NET::SPLIT && !SV::kOn && !SV::kF32 && LAT == 0 && NET::ACT == NRT_ACT_LEAKY_RELU) ? PackedPairsOf<IO>::value : 0;
  constexpr int ZLO = (NRT_BIAS_MMA & 2) ? 2 * kPP / 16 : 0;
  // NRT_FIRST_PIPE (NeRFLE.first's inference kernels, i.e. the render layout): the tile boundary leaves the per-slot chain.
  // The next tile's inputs are fetched right after this tile's encoding was handed to the MMA warp, its encoding is
  // computed while the output layer runs, and on the output `done` the epilogue reads the accumulator, stores that
  // encoding and arrives on `ready` before it writes this tile's outputs: the next tile's init layer runs under the stores.
#ifndef NRT_FIRST_PIPE
#define NRT_FIRST_PIPE 1
#endif
  constexpr bool PIPE = NRT_FIRST_PIPE != 0 && NET::BIAS_ROWS && !ITER;
  static_assert(!PIPE || (BMMA && NET::SPLIT && NET::ENC_CUDA && !NET::FUSE_OUT && !NET::INPLACE && LAT == 0 && WPS == 4),
                "NRT_FIRST_PIPE: NeRFLE.first's render layout (split fp32 encoding, bias rows, an MMA output layer)");
  __shared__ volatile uint32_t s_slot_live[3];   // iterative policies: 0 once the slot's queue has run dry
  __shared__ uint32_t s_warp_live[3][4];

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  constexpr bool SELF = NET::SELF;
  const int mma_id = SELF ? -1 : warp - NET::NWG * WPS;   // >= 0: MMA-issuing warp
  const bool is_mma_warp = SELF ? warp == 0 : mma_id == 0;   // the one that also owns TMEM allocation and the weight load
  __shared__ uint32_t s_issue_lock;                  // self-issue: one slot's MMA batch at a time
  const int64_t ntiles = (M + 127) / 128;
  // IO policies that keep per-CTA tables in shared memory (the sphere set of the SDF policies) fill them here; the
  // __syncthreads() below publishes them
  if constexpr (HasCtaInit<IO>::value) io.cta_init();
  if (tid < NET::STAGES) {
    s_bias[tid] = (uint32_t)Y.bias_off[tid];
    s_opoff[tid] = (uint32_t)Y.op_off[tid] * 2;
    s_opbytes[tid] = (uint32_t)(Y.opN[tid] * Y.opK[tid] * 2);
  }

  if (tid == 0) {
    s_slot_live[0] = 1; s_slot_live[1] = 1; s_slot_live[2] = 1;
    s_issue_lock = 0;
    mbar_init(&bar_w, 1);
    for (int s = 0; s < 3; ++s) {
      mbar_init(&bar_ready[s], EPI); mbar_init(&bar_done[s], 1); mbar_init(&bar_ready_a[s], EPI);
      mbar_init(&bar_wfull[s][0], 1); mbar_init(&bar_wfull[s][1], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (is_mma_warp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    if ((tid & 31) == 0) {
      if (STREAM) {
        // only the biases are resident; stage operands are streamed by the MMA loop
        mbar_expect_tx(&bar_w, (uint32_t)NET::BIAS_BYTES);
        bulk_g2s(smem + (size_t)NSLOT * 2 * NET::MAXOP, blob + (size_t)Y.w_elems * 2, (uint32_t)NET::BIAS_BYTES, &bar_w);
      } else {
        // all weights + biases: global (L2) -> shared, once per CTA
        mbar_expect_tx(&bar_w, (uint32_t)Y.bytes);
        constexpr uint32_t kChunk = 32768;
        for (uint32_t off = 0; off < (uint32_t)Y.bytes; off += kChunk) {
          const uint32_t n = min(kChunk, (uint32_t)Y.bytes - off);
          bulk_g2s(smem + off, blob + off, n, &bar_w);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // The whole TMEM (512 columns) is allocated, so the base address is lane 0 / column 0.  Treating it as the
  // compile-time constant 0 lets every tcgen05.mma operand of a (slot, stage) pair be an immediate: otherwise the
  // base comes out of shared memory into a vector register and costs ~7 R2UR moves in front of every stage.
  if (tmem_base_s != 0u) __trap();
  constexpr uint32_t tmem = 0u;
  if constexpr (BMMA) {
    // the constant A chunk of the bias K-chunks, K elements [1, 1, 1, 0, ...] in every lane, shared read-only by all
    // slots: warp w writes lane quarter w, before any MMA can read it
    if (warp < 4) {
      const uint32_t one = (uint32_t)one16<FMT>();
      const uint32_t r[8] = {one | (one << 16), one, 0u, 0u, 0u, 0u, 0u, 0u};
      TmemIO<8>::st(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)NET::ONES_COL, r);
      tc_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  mbar_wait(&bar_w, 0);

  if (mma_id >= 0) {
    // ===================== MMA issuer(s) =====================
    // The whole warp runs this loop convergently (one elected lane issues).  With one MMA warp per tile slot
    // (NET::NMMA == NSLOT) every warp blocks on its own slot's `ready` barrier: a slot is served as soon as its
    // epilogue arrives, instead of after the other slots' stages (a single warp needs 50-60 cycles per tcgen05.mma
    // it issues, 300-700 per stage, and served the slots round robin).  With a single MMA warp the slots are polled
    // and served in whatever order they become ready.  Either way the tiles drift into anti-phase: the tensor pipe
    // works on one tile while the other tile's epilogue (or prologue / output store) runs.
    constexpr int NMMA = NET::NMMA;
    constexpr bool OWN = NMMA == NSLOT;      // this warp serves exactly one slot: blocking waits
    auto mine = [&](int slot) { return slot % (NMMA > 0 ? NMMA : 1) == mma_id; };
    // Single warp, two slots (NRT_MMA_ALTERNATE): the slots are served strictly in turn with a BLOCKING wait on the
    // slot whose turn it is.  The polling loop (mbarrier test + nanosleep) saw an arrive 120-580 cycles late (350 on
    // average, 10 % of a stage); a slot can only arrive once per stage it is served, so alternation costs nothing in
    // the steady state and keeps the two tiles in anti-phase (one in its MMAs while the other converts).
#ifndef NRT_MMA_ALTERNATE
#define NRT_MMA_ALTERNATE 0
#endif
    constexpr bool ALT = NRT_MMA_ALTERNATE != 0 && !OWN && NSLOT == 2 && !KSPLIT;
    int turn = 0;
    bool live[3];
    auto is_ready = [&](int slot, uint64_t* bar, uint32_t parity) {
      if constexpr (OWN) { mbar_wait(bar, parity); return true; }
      else if constexpr (ALT) {
        if (slot != turn && live[turn]) return false;
        mbar_wait(bar, parity);
        turn = slot ^ 1;
        return true;
      }
      else return mbar_test(bar, parity);
    };
    const uint32_t sW_addr = smem_u32(sW);
    int st[3] = {NET::FIRST_STAGE, NET::FIRST_STAGE, NET::FIRST_STAGE};
    uint32_t n_ready[3] = {0, 0, 0};
    uint32_t n_ready_a[3] = {0, 0, 0};
    bool half_issued[3] = {false, false, false};
    int64_t tile[3] = {(int64_t)blockIdx.x * NSLOT, (int64_t)blockIdx.x * NSLOT + 1, (int64_t)blockIdx.x * NSLOT + 2};
    live[0] = mine(0) && (ITER || tile[0] < ntiles);
    live[1] = NSLOT > 1 && mine(1) && (ITER || tile[1] < ntiles);
    live[2] = NSLOT > 2 && mine(2) && (ITER || tile[2] < ntiles);
    int it_dbg[3] = {0, 0, 0};
    uint32_t n_issued[3] = {0, 0, 0};   // streaming: stages issued per slot (selects the stage buffer)
    if (STREAM) {
#pragma unroll
      for (int slot = 0; slot < NSLOT; ++slot)
        if (live[slot] && elect_one())
          stream_op(smem + (size_t)(slot * 2) * NET::MAXOP, blob + s_opoff[NET::FIRST_STAGE], s_opbytes[NET::FIRST_STAGE],
                    &bar_wfull[slot][0]);
      __syncwarp();
    }
    while (live[0] || live[1] || live[2]) {
      bool progressed = false;
#pragma unroll
      for (int slot = 0; slot < NSLOT; ++slot) {
        if (!live[slot]) continue;
        if constexpr (KSPLIT) {
          if (st[slot] >= 2 && !half_issued[slot]) {
            // first half of a hidden stage's operand is in place: issue its K-chunks under the rest of the epilogue
            if (!is_ready(slot, &bar_ready_a[slot], n_ready_a[slot] & 1)) continue;
            progressed = true;
            n_ready_a[slot]++;
            half_issued[slot] = true;
            tc_fence_after();
            const uint32_t base = tmem + slot * NET::COLS;
            uint32_t b_addr = sW_addr;
            if (STREAM) {
              const uint32_t b = n_issued[slot] & 1;
              mbar_wait(&bar_wfull[slot][b], (n_issued[slot] >> 1) & 1);
              b_addr = sW_addr + (uint32_t)((slot * 2 + b) * NET::MAXOP);
            }
            if ((tid & 31) == 0) stamp(it_dbg[slot], st[slot], slot, 0);
            issue_stage_dyn<NET, FMT, 1>(st[slot], b_addr, base, base + NET::DC, base + NET::DC + NET::UC, &bar_done[slot]);
            continue;
          }
        }
        if (!is_ready(slot, &bar_ready[slot], n_ready[slot] & 1)) continue;
        progressed = true;
        n_ready[slot]++;
        tc_fence_after();
        if constexpr (ITER) {
          if (st[slot] == NET::FIRST_STAGE && s_slot_live[slot] == 0) {
            // the slot's epilogue found no live trajectory and the queue is empty: retire the slot (after draining
            // the operand prefetch that was issued for the iteration that will not happen)
            live[slot] = false;
            if (STREAM) mbar_wait(&bar_wfull[slot][n_issued[slot] & 1], (n_issued[slot] >> 1) & 1);
            continue;
          }
        }
        if ((tid & 31) == 0) stamp(it_dbg[slot], st[slot], slot, 1);
        const uint32_t base = tmem + slot * NET::COLS;
        uint32_t b_addr = sW_addr;
        if (STREAM) {
          const uint32_t b = n_issued[slot] & 1;
          mbar_wait(&bar_wfull[slot][b], (n_issued[slot] >> 1) & 1);
          b_addr = sW_addr + (uint32_t)((slot * 2 + b) * NET::MAXOP);
          if ((tid & 31) == 0) stamp(it_dbg[slot], st[slot], slot, 0);   // streamed operand has landed
        }
        if (KSPLIT && half_issued[slot]) {
          half_issued[slot] = false;
          issue_stage_dyn<NET, FMT, 2>(st[slot], b_addr, base, base + NET::DC, base + NET::DC + NET::UC, &bar_done[slot]);
        } else {
          issue_stage_dyn<NET, FMT, 0, BMMA, ZLO>(st[slot], b_addr, base, base + NET::DC, base + NET::DC + NET::UC, &bar_done[slot]);
        }
        if ((tid & 31) == 0) stamp(it_dbg[slot], st[slot], slot, 2);
        if (++st[slot] == NET::END_STAGE) {
          st[slot] = NET::FIRST_STAGE;
          it_dbg[slot]++;
          if constexpr (!ITER) {
            tile[slot] += (int64_t)gridDim.x * NSLOT;
            live[slot] = tile[slot] < ntiles;
          }
        }
        if (STREAM) {
          // prefetch the operand of this slot's next stage into its other buffer.  That buffer held the operand
          // of the previous stage, whose MMAs completed before the epilogue that made this stage ready.
          n_issued[slot]++;
          if (live[slot] && elect_one()) {
            const uint32_t nb = n_issued[slot] & 1;
            stream_op(smem + (size_t)(slot * 2 + nb) * NET::MAXOP, blob + s_opoff[st[slot]], s_opbytes[st[slot]],
                      &bar_wfull[slot][nb]);
          }
          __syncwarp();
        }
      }
      // (a back-off here -- the warp shares its SM sub-partition with two epilogue warps -- measured 1 % slower than
      //  plain polling for the streamed SDF net: min scan 28.1 vs 27.8 ms)
#ifndef NRT_MMA_POLL_SLEEP_NS
#define NRT_MMA_POLL_SLEEP_NS 0
#endif
      if (NRT_MMA_POLL_SLEEP_NS > 0 && !progressed) __nanosleep(NRT_MMA_POLL_SLEEP_NS);
    }
  } else {
    // ===================== epilogue warpgroups (one per tile slot) =====================
    const int slot = warp / WPS;
    // 8-warp variant: warps q and q+4 of a slot share TMEM lane quarter q; `half` selects the columns a warp converts.
    // Half 0 ("primary") also owns the sample: input load / encoding / output; half 1 only helps in the hidden layers.
    const int half = (WPS == 8) ? ((warp >> 2) & 1) : 0;
    const bool primary = half == 0;
    const int lane_row = (warp & 3) * 32 + (tid & 31);   // TMEM lane == row of the tile == sample
    constexpr int HW = (WPS == 8) ? H / 2 : H;            // hidden columns converted per thread
    if (slot < NSLOT) {
      const uint32_t lane_off = ((uint32_t)((warp & 3) * 32)) << 16;
      const uint32_t base = tmem + slot * NET::COLS + lane_off;
      const uint32_t dD = base, aU = base + NET::DC, aE = base + NET::DC + NET::UC;
      uint32_t n_done = 0;
      int it_dbg = 0;
#ifndef NRT_DBG_LANE
#define NRT_DBG_LANE 0
#endif
      auto estamp = [&](int st, int k) { if (lane_row == NRT_DBG_LANE) stamp(it_dbg, st, slot, k); };
      typename StateOf<IO>::type state;
      if constexpr (ITER) io.init(state);
      // ---- self-issue: the slot's first warp is its MMA issuer ----
      const bool leader = SELF && (warp % WPS) == 0;
      int st_mma = NET::FIRST_STAGE;
      uint32_t n_ready_l = 0, n_issued_l = 0;
      const uint32_t sW_addr_l = smem_u32(sW);
      if constexpr (SELF) {
        if (leader) {
          if (elect_one())
            stream_op(smem + (size_t)(slot * 2) * NET::MAXOP, blob + s_opoff[NET::FIRST_STAGE], s_opbytes[NET::FIRST_STAGE],
                      &bar_wfull[slot][0]);
          __syncwarp();
        }
      }
      // called by every warp of the slot right after its arrive on `ready`; only the leader does anything
      auto self_issue = [&]() {
        if constexpr (SELF) {
          if (leader) {
            mbar_wait(&bar_ready[slot], n_ready_l & 1); n_ready_l++;
            const uint32_t b = n_issued_l & 1;
            mbar_wait(&bar_wfull[slot][b], (n_issued_l >> 1) & 1);
            if ((tid & 31) == 0) {
              while (atomicCAS(&s_issue_lock, 0u, 1u) != 0u) __nanosleep(64);
            }
            __syncwarp();
            tc_fence_after();
            if ((tid & 31) == 0) stamp(it_dbg, st_mma, slot, 1);
            const uint32_t base0 = tmem + slot * NET::COLS;
            issue_stage_dyn<NET, FMT>(st_mma, sW_addr_l + (uint32_t)((slot * 2 + b) * NET::MAXOP), base0, base0 + NET::DC,
                                      base0 + NET::DC + NET::UC, &bar_done[slot]);
            if ((tid & 31) == 0) {
              stamp(it_dbg, st_mma, slot, 2);
              __threadfence_block();
              atomicExch(&s_issue_lock, 0u);
            }
            if (++st_mma == NET::END_STAGE) st_mma = NET::FIRST_STAGE;
            n_issued_l++;
            // prefetch the operand of the slot's next stage (possibly of an iteration that never happens: drained at
            // exit).  The other buffer held the previous stage's operand, whose MMAs completed before the epilogue
            // that made this stage ready.
            if (elect_one()) {
              const uint32_t nb = n_issued_l & 1;
              stream_op(smem + (size_t)(slot * 2 + nb) * NET::MAXOP, blob + s_opoff[st_mma], s_opbytes[st_mma], &bar_wfull[slot][nb]);
            }
            __syncwarp();
          }
        }
      };
      auto self_drain = [&]() {
        if constexpr (SELF) {
          if (leader) mbar_wait(&bar_wfull[slot][n_issued_l & 1], (n_issued_l >> 1) & 1);
        }
      };
#ifndef NRT_SLOT_STAGGER
#define NRT_SLOT_STAGGER 900
#endif
      if (NRT_SLOT_STAGGER > 0 && slot > 0) {
        // start the slots out of phase (cycles per slot index): slots that reach their MMA stages together interleave
        // in the in-order tensor pipe and then run their epilogues together as well (measured: 57.3 -> 56.4 ms/frame)
        const long long t_start = clock64();
        while (clock64() - t_start < (long long)slot * NRT_SLOT_STAGGER) {}
      }
      // development (NRT_DBG_BOUNDARY, tools/tc_timeline_nerf.py --first): the tile boundary in row 0 of the stamps --
      // 3 output `done` seen, 4 outputs stored, 5 inputs in registers, 6 encoding stored, 7 `ready` arrived for the init layer
#ifdef NRT_DBG_BOUNDARY
      auto bstamp = [&](int it, int k) { if (lane_row == NRT_DBG_LANE) stamp(it, 0, slot, k); };
      auto bstamp_dep = [&](int it, int k, float v) { if (lane_row == NRT_DBG_LANE && __float_as_uint(v) != 0xffffffffu) stamp(it, 0, slot, k); };
#else
      auto bstamp = [&](int, int) {};
      auto bstamp_dep = [&](int, int, float) {};
#endif
      // ---- NRT_FIRST_PIPE: a tile's inputs fetched one tile ahead, its encoding computed in registers ----
      struct Inputs { float v[IN + LAT]; };
      using Pre = typename FetchOf<IO, Inputs>::type;
      struct Enc { uint32_t ax[NET::KX / 2], ex[NET::XR / 2], sr[F / 2], cr[F / 2], sa[F / 2], ca[F / 2]; };
      const int64_t tstride = (int64_t)gridDim.x * NSLOT;
      Pre pre;                 // inputs of the slot's next tile (rows m >= M: not fetched, pre_ok false)
      bool pre_ok = false;
      auto fetch = [&](int64_t mm) {
        if constexpr (PIPE) {
          pre_ok = mm < M;    // (also false past the last tile: mm >= ntiles * 128 >= M)
          if (pre_ok) {
            if constexpr (std::is_same_v<Pre, Inputs>) io.load(mm, pre.v);
            else io.fetch(mm, pre);
          }
        }
      };
      auto inputs = [&](float* xi) {
        if (PIPE && pre_ok) {
          if constexpr (std::is_same_v<Pre, Inputs>) {
#pragma unroll
            for (int j = 0; j < IN; ++j) xi[j] = pre.v[j];
          } else io.point(pre, xi);
        } else {
#pragma unroll
          for (int j = 0; j < IN; ++j) xi[j] = 0.0f;
        }
      };
      // stages 0 and 1 of the loop below (the SPLIT, BIAS_ROWS and ENC_CUDA branches), the same operations in the same order
      auto encode = [&](const float* xi, Enc& e) {
        if constexpr (PIPE) {
        uint16_t v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0;
        uint16_t a[2 * IN];
#pragma unroll
        for (int j = 0; j < IN; ++j) {
          const uint16_t hi = E::cvt(xi[j]);
          const uint16_t lo = E::cvt(xi[j] - E::back(hi));
          v[j] = hi; v[IN + j] = lo; v[2 * IN + j] = hi;
          const float ax_ = act_fast<NET::ACT>(xi[j]);
          const uint16_t ahi = E::cvt(ax_);
          a[j] = ahi; a[IN + j] = E::cvt(ax_ - E::back(ahi));
        }
#pragma unroll
        for (int t = 0; t < 3; ++t) v[NET::BR.row + t] = one16<FMT>();
#pragma unroll
        for (int j = 0; j < NET::XR / 2; ++j) e.ex[j] = 0;
#pragma unroll
        for (int j = 0; j < NET::KX / 2; ++j) e.ax[j] = (uint32_t)v[2 * j] | ((uint32_t)v[2 * j + 1] << 16);
#pragma unroll
        for (int j = 0; j < IN; ++j) e.ex[j] = (uint32_t)a[2 * j] | ((uint32_t)a[2 * j + 1] << 16);
#pragma unroll
        for (int t = 0; t < 3; ++t) e.ex[(NET::BR.row + t) / 2] |= (uint32_t)one16<FMT>() << (16 * ((NET::BR.row + t) & 1));
        const float* sB = sBias + Y.basis_f32_off;
        uint32_t ph[F];
#pragma unroll
        for (int f = 0; f < F; ++f) {
          float p = xi[0] * sB[f];
#pragma unroll
          for (int j = 1; j < IN; ++j) p = fmaf(xi[j], sB[j * NET::FP + f], p);
          ph[f] = __float_as_uint(p);
        }
#pragma unroll
        for (int j = 0; j < F / 2; ++j) {
          float s0, c0, s1, c1;
          sincos_fast(__uint_as_float(ph[2 * j]), &s0, &c0);
          sincos_fast(__uint_as_float(ph[2 * j + 1]), &s1, &c1);
          e.sr[j] = E::pack(s0, s1); e.cr[j] = E::pack(c0, c1);
          e.sa[j] = E::pack(act_fast<NET::ACT>(s0), act_fast<NET::ACT>(s1));
          e.ca[j] = E::pack(act_fast<NET::ACT>(c0), act_fast<NET::ACT>(c1));
        }
        }
      };
      auto enc_store = [&](const Enc& e) {
        tmem_store<NET::KX / 2>(aU, e.ax);
        tmem_store<NET::XR / 2>(aE, e.ex);
        tmem_store<F / 2>(aU + NET::XR / 2, e.sr);
        tmem_store<F / 2>(aU + NET::XR / 2 + F / 2, e.cr);
        tmem_store<F / 2>(aE + NET::XR / 2, e.sa);
        tmem_store<F / 2>(aE + NET::XR / 2 + F / 2, e.ca);
      };
      if constexpr (PIPE) {
        // the slot's first tile: fetched, encoded and handed to the MMA warp here; later tiles in the previous tile's
        // output stage
        const int64_t tile = (int64_t)blockIdx.x * NSLOT + slot;
        if (tile < ntiles) {
          fetch(tile * 128 + lane_row);
          float xi[IN];
          inputs(xi);
          Enc e;
          encode(xi, e);
          enc_store(e);
          tc_wait_st();
          tc_fence_before();
          mbar_arrive(&bar_ready[slot]);
          fetch((tile + tstride) * 128 + lane_row);
        }
      }
      for (int64_t t0 = (int64_t)blockIdx.x * NSLOT;; t0 += (int64_t)gridDim.x * NSLOT, ++it_dbg) {
        int64_t m = 0;
        bool valid;
        float x[IN + LAT];
        uint32_t pw[kPP > 0 ? kPP : 1];
        if constexpr (ITER) {
          valid = primary ? io.next(state, x) : false;
          const unsigned bal = __ballot_sync(0xffffffffu, valid);
          if (primary && (tid & 31) == 0) s_warp_live[slot][warp & 3] = bal;
          named_bar_sync(1 + slot, EPI);
          const bool any = (s_warp_live[slot][0] | s_warp_live[slot][1] | s_warp_live[slot][2] | s_warp_live[slot][3]) != 0;
          if (!any) {
            if (lane_row == 0) s_slot_live[slot] = 0;
            mbar_arrive(&bar_ready[slot]);   // release: the MMA warp reads s_slot_live after its acquire
            self_drain();
            break;
          }
        } else {
          const int64_t tile = t0 + slot;
          if (tile >= ntiles) { self_drain(); break; }
          m = tile * 128 + lane_row;
          valid = m < M;
          if constexpr (PIPE) {
            // the tile's encoding is in TMEM already
          } else if constexpr (kPP > 0) {
            if (valid && primary) io.load_packed(m, pw, x);
          } else {
            if (valid && primary) io.load(m, x);
            if (valid) bstamp_dep(it_dbg, 5, x[0]);
          }
        }
        if constexpr (PIPE) {
        } else if (!primary) {
          // the helper half has no work before the first hidden layer: keep in phase with the barriers only
          if constexpr (!NET::ENC_CUDA) {
            mbar_arrive(&bar_ready[slot]);
            mbar_wait(&bar_done[slot], n_done & 1); n_done++;
          }
          mbar_arrive(&bar_ready[slot]);
          self_issue();
        } else {
        // ---- stage 0: inputs -> encode-GEMM A operand (+ x / latent parts of enc_raw, enc_act) ----
        uint32_t ex[NET::XR / 2];     // act(x): stored in stage 1 when the hi+lo phase GEMM borrows its place for x_lo
        {
          if (!valid) {
#pragma unroll
            for (int j = 0; j < IN + LAT; ++j) x[j] = 0.0f;
          }
          uint32_t ax[NET::KX / 2];
#pragma unroll
          for (int j = 0; j < NET::KX / 2; ++j) { ax[j] = 0; ex[j] = 0; }
          if constexpr (NET::SPLIT) {
            uint16_t v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = 0;
            uint16_t a[2 * IN];
#pragma unroll
            for (int j = 0; j < IN; ++j) {
              const uint16_t hi = E::cvt(x[j]);
              const uint16_t lo = E::cvt(x[j] - E::back(hi));
              v[j] = hi; v[IN + j] = lo; v[2 * IN + j] = hi;
              const float ax_ = act_fast<NET::ACT>(x[j]);
              const uint16_t ahi = E::cvt(ax_);
              a[j] = ahi; a[IN + j] = E::cvt(ax_ - E::back(ahi));
            }
            // render layout: the constant-1 columns that the bias rows of the init and skip layers multiply
            if constexpr (NET::BIAS_ROWS) {
#pragma unroll
              for (int t = 0; t < 3; ++t) v[NET::BR.row + t] = one16<FMT>();
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) ax[j] = (uint32_t)v[2 * j] | ((uint32_t)v[2 * j + 1] << 16);
#pragma unroll
            for (int j = 0; j < IN; ++j) ex[j] = (uint32_t)a[2 * j] | ((uint32_t)a[2 * j + 1] << 16);
            if constexpr (NET::BIAS_ROWS) {
#pragma unroll
              for (int t = 0; t < 3; ++t) ex[(NET::BR.row + t) / 2] |= (uint32_t)one16<FMT>() << (16 * ((NET::BR.row + t) & 1));
            }
            tmem_store<NET::KX / 2>(aU, ax);
            if constexpr (NET::INPLACE) tmem_store<NET::XR / 2>(aE, ax);   // raw x part; activated in place later
            else tmem_store<NET::XR / 2>(aE, ex);
          } else {
            // x_hi (what the init / skip layers see) and x_lo = x - x_hi (second operand of the hi+lo phase GEMM)
            uint32_t lx[NET::XR / 2];
#pragma unroll
            for (int j = 0; j < NET::XR / 2; ++j) lx[j] = 0;
#pragma unroll
            for (int j = 0; j < (IN + 1) / 2; ++j) {
              if (kPP > 0 && j < kPP) {
                ax[j] = valid ? pw[j] : 0u;      // x_hi as stored; x_lo = 0 (lx stays zero); NET::INPLACE: act(x) is made in place later
                if constexpr (!NET::INPLACE) ex[j] = leaky_packed<FMT>(ax[j]);
                continue;
              }
              const float xa = x[2 * j], xb = (2 * j + 1 < IN) ? x[2 * j + 1 < IN ? 2 * j + 1 : 0] : 0.0f;   // odd in: zero pad
              ax[j] = E::pack(xa, xb);
              const float ha = E::back((uint16_t)(ax[j] & 0xffffu)), hb = E::back((uint16_t)(ax[j] >> 16));
              lx[j] = E::pack(xa - ha, xb - hb);
              ex[j] = E::pack(act_fast<NET::ACT>(xa), (2 * j + 1 < IN) ? act_fast<NET::ACT>(xb) : 0.0f);
            }
            // in-place plan: x_hi into the encoding region (its final place), x_lo into the union region;
            // otherwise x_hi into the union region (its final place) and x_lo TEMPORARILY into the encoding region:
            // act(x) is stored there in stage 1, once the phase GEMM has read x_lo
            if constexpr (NET::INPLACE) { tmem_store<NET::XR / 2>(aE, ax); tmem_store<NET::XR / 2>(aU, lx); }
            else { tmem_store<NET::XR / 2>(aU, ax); tmem_store<NET::XR / 2>(aE, lx); }
          }
          if constexpr (SV::kOn) {
            static_assert(!ITER, "activation tiles are saved by the tile policies only");
            uint16_t* rr = tile_row_ptr(sv.enc_raw, m >> 7, NET::KE + kTileRowsExtra, lane_row);
            uint16_t* ra = tile_row_ptr(sv.enc_act, m >> 7, NET::KE + kTileRowsExtra, lane_row);
            save_cols<NET::KX / 2>(rr, 0, ax);
            if constexpr (!NET::INPLACE) save_cols<NET::XR / 2>(ra, 0, ex);
            rr[tile_elem(NET::KE)] = one16<FMT>();
            ra[tile_elem(NET::KE)] = one16<FMT>();
          }
          if constexpr (LAT > 0) {
            // latent part of the encoding (raw and activated); sits after sin/cos
            uint32_t lr[LAT / 2], la[LAT / 2];
#pragma unroll
            for (int j = 0; j < LAT / 2; ++j) {
              lr[j] = E::pack(x[IN + 2 * j], x[IN + 2 * j + 1]);
              la[j] = E::pack(act_fast<NET::ACT>(x[IN + 2 * j]), act_fast<NET::ACT>(x[IN + 2 * j + 1]));
            }
            tmem_store<LAT / 2>(aU + (NET::XR + 2 * F) / 2, lr);
            tmem_store<LAT / 2>(aE + (NET::XR + 2 * F) / 2, la);
            if constexpr (SV::kOn) {
              save_cols<LAT / 2>(tile_row_ptr(sv.enc_raw, m >> 7, NET::KE + kTileRowsExtra, lane_row), NET::XR + 2 * F, lr);
              save_cols<LAT / 2>(tile_row_ptr(sv.enc_act, m >> 7, NET::KE + kTileRowsExtra, lane_row), NET::XR + 2 * F, la);
            }
          }
          if constexpr (!NET::ENC_CUDA) {
            tc_wait_st();
            tc_fence_before();
            mbar_arrive(&bar_ready[slot]);
          }
        }
        // ---- stage 1: phases -> sin / cos -> rest of enc_raw / enc_act ----
        {
          uint32_t ph[F];
          if constexpr (NET::ENC_CUDA) {
            // phases x.B in fp32 on the CUDA cores (in*F FMAs), no MMA round trip; the accumulator is free (the
            // previous tile's output was read), so the init layer's bias goes in right away
            const float* sB = sBias + Y.basis_f32_off;
#pragma unroll
            for (int f = 0; f < F; ++f) {
              float p = x[0] * sB[f];
#pragma unroll
              for (int j = 1; j < IN; ++j) p = fmaf(x[j], sB[j * NET::FP + f], p);
              ph[f] = __float_as_uint(p);
            }
          } else {
            mbar_wait(&bar_done[slot], n_done & 1); n_done++;
            tc_fence_after();
            tmem_load<F>(dD, ph);
            tc_wait_ld();
            // the phase GEMM has read x_lo: act(x) takes its place in the encoding region
            if constexpr (!NET::INPLACE) tmem_store<NET::XR / 2>(aE, ex);
          }
          if constexpr (!BMMA) preload_bias<H>(dD, sBias + s_bias[1]);
          uint32_t sr[F / 2], cr[F / 2], sa[F / 2], ca[F / 2];
#pragma unroll
          for (int j = 0; j < F / 2; ++j) {
            float s0, c0, s1, c1;
            sincos_fast(__uint_as_float(ph[2 * j]), &s0, &c0);
            sincos_fast(__uint_as_float(ph[2 * j + 1]), &s1, &c1);
            sr[j] = E::pack(s0, s1); cr[j] = E::pack(c0, c1);
            sa[j] = E::pack(act_fast<NET::ACT>(s0), act_fast<NET::ACT>(s1));
            ca[j] = E::pack(act_fast<NET::ACT>(c0), act_fast<NET::ACT>(c1));
          }
          if constexpr (NET::INPLACE) {
            tmem_store<F / 2>(aE + NET::XR / 2, sr);
            tmem_store<F / 2>(aE + NET::XR / 2 + F / 2, cr);
          } else {
            tmem_store<F / 2>(aU + NET::XR / 2, sr);
            tmem_store<F / 2>(aU + NET::XR / 2 + F / 2, cr);
            tmem_store<F / 2>(aE + NET::XR / 2, sa);
            tmem_store<F / 2>(aE + NET::XR / 2 + F / 2, ca);
          }
          if constexpr (SV::kOn) {
            uint16_t* rr = tile_row_ptr(sv.enc_raw, m >> 7, NET::KE + kTileRowsExtra, lane_row);
            uint16_t* ra = tile_row_ptr(sv.enc_act, m >> 7, NET::KE + kTileRowsExtra, lane_row);
            save_cols<F / 2>(rr, NET::XR, sr);
            save_cols<F / 2>(rr, NET::XR + F, cr);
            if constexpr (!NET::INPLACE) {
              save_cols<F / 2>(ra, NET::XR, sa);
              save_cols<F / 2>(ra, NET::XR + F, ca);
            }
          }
          // (the raw-x segment keeps the phase-GEMM tile [x_hi | x_lo | x_hi | 0]; the init / skip weights
          //  of the third copy and of the padding are zero, see enc_ref_index)
          tc_wait_st();
          bstamp(it_dbg, 6);
          tc_fence_before();
          mbar_arrive(&bar_ready[slot]);
          bstamp(it_dbg, 7);
          self_issue();
        }
        }   // primary
        // ---- stages 2 .. L+1: hidden activations ----
        constexpr int NHID = NET::FUSE_OUT ? L : L + 1;   // epilogues that feed another MMA stage
#pragma unroll 1
        for (int st = 0; st < NHID; ++st) {
          estamp(2 + st, 3);
          mbar_wait(&bar_done[slot], n_done & 1); n_done++;
          tc_fence_after();
          estamp(2 + st, 4);
          if constexpr (!KSPLIT) estamp(2 + st, 5);
          const int coff = half * HW;     // this thread's first hidden column
          // everything that must be in place before the next stage's MMAs: the bias of the layer that consumes
          // these activations (into the accumulator, free once its row has been read) and, for the in-place plan,
          // the activated encoding
          auto pre = [&]() {
            if constexpr (NET::INPLACE) {
              if (st == 0 && primary) {
                // the init layer has consumed the raw encoding: turn it into act(encoding) for the skip layers
                static_assert(NET::KE % 16 == 0, "encoding width");
#pragma unroll
                for (int c = 0; c < NET::EC / 8; ++c) {
                  uint32_t e[8];
                  TmemIO<8>::ld(aE + 8 * c, e);
                  tc_wait_ld();
#pragma unroll
                  for (int j = 0; j < 8; ++j) e[j] = leaky_packed<FMT>(e[j]);
                  TmemIO<8>::st(aE + 8 * c, e);
                  if constexpr (SV::kOn)
                    save_cols<8>(tile_row_ptr(sv.enc_act, m >> 7, NET::KE + kTileRowsExtra, lane_row), 16 * c, e);
                }
              }
            }
            if constexpr (BMMA) {
              // the next stage's bias K-chunk overwrites the accumulator
            } else if (st < L) preload_bias<HW>(dD + coff, sBias + s_bias[2 + st] + coff);
            else {
              // output-layer bias: every half writes only the accumulator columns it has just read
              // (one warp per lane quarter: the primary writes all of them, also those beyond the hidden width -- an
              //  output wider than the hidden layers, PlainNeRF.first 32 -> 33)
              constexpr int N0 = (WPS != 8 || NET::NOP < HW) ? NET::NOP : HW, N1 = (WPS == 8 && NET::NOP > HW) ? NET::NOP - HW : 0;
              if (primary) preload_bias<N0>(dD, sBias + s_bias[NET::STAGES - 1]);
              else if constexpr (N1 > 0) preload_bias<N1>(dD + HW, sBias + s_bias[NET::STAGES - 1] + HW);
            }
          };
          if constexpr (KSPLIT) {
            // (one convergent call: the tcgen05 instructions inside are .sync.aligned; only lane_row 0 gets stamp slots)
            long long* d = nullptr;
            if (dbg != nullptr && lane_row == 0 && slot < 2 && blockIdx.x == 0 && it_dbg >= kDbgIt0 && it_dbg < kDbgIt0 + kDbgIts)
              d = dbg + (((it_dbg - kDbgIt0) * NET::STAGES + 2 + st) * 2 + slot) * 8;
            convert_row_split<NET::ACT, FMT, HW>(dD, aU, &bar_ready_a[slot], &bar_ready[slot], pre, d ? d + 5 : nullptr,
                                                 d ? d + 6 : nullptr);
            estamp(2 + st, 7);
          } else {
          if constexpr (SV::kOn)
            convert_row<NET::ACT, FMT, HW, true>(dD + coff, aU + coff / 2,
                tile_row_ptr(sv.acts, (int64_t)st * sv.ntiles + (m >> 7), H + kTileRowsExtra, lane_row), coff, primary ? H : -1,
                sv.masks + (int64_t)st * (H / 32) * (sv.ntiles * 128) + m, sv.ntiles * 128);
          else if constexpr (SV::kF32)
            convert_row_savef32<NET::ACT, FMT, HW>(dD + coff, aU + coff / 2,
                                                   valid ? sv.acts + ((int64_t)st * H) * sv.M + m : nullptr, sv.M);
          else if constexpr (kPipeRow) {
            long long* d = nullptr;
#ifdef NRT_DBG_CONV
            // development: stamps 3 / 4 of the stage row are reused for "first exponentials issued" / "all columns read"
            if (dbg != nullptr && lane_row == NRT_DBG_LANE && slot < 2 && blockIdx.x == 0 && it_dbg >= kDbgIt0 && it_dbg < kDbgIt0 + kDbgIts)
              d = dbg + (((it_dbg - kDbgIt0) * NET::STAGES + 2 + st) * 2 + slot) * 8 + 3;
#endif
            convert_row_pipe<FMT, HW, SoftplusOf<IO>::value>(dD + coff, aU + coff / 2, pre, d);
          }
          else if constexpr (kFullRow)
            convert_row_full<NET::ACT, FMT, HW>(dD + coff, aU + coff / 2, pre);
          else
            convert_row<NET::ACT, FMT, HW>(dD + coff, aU + coff / 2);
          // done after the conversion so the accumulator registers are dead and all LDS.128 can be in flight
          if constexpr (!(kFullRow || kPipeRow) || SV::kOn || SV::kF32) pre();
          estamp(2 + st, 6);
          tc_wait_st();
          tc_fence_before();
          mbar_arrive(&bar_ready[slot]);
          estamp(2 + st, 7);
          self_issue();
          }
        }
        // ---- NRT_FIRST_PIPE: the next tile's encoding, under the output layer's MMAs ----
        const bool has_next = PIPE && t0 + slot + tstride < ntiles;
        Enc en;
        if constexpr (PIPE) {
          if (has_next) {
            float xi[IN];
            inputs(xi);
            bstamp_dep(it_dbg + 1, 5, xi[0]);
            encode(xi, en);
          }
        }
        // ---- output layer ----
        if (!primary) {
          mbar_wait(&bar_done[slot], n_done & 1); n_done++;
          tc_fence_after();
          tc_fence_before();
        } else if constexpr (NET::FUSE_OUT) {
          // last hidden activations and the (tiny) output layer in one pass, fp32 on the CUDA cores
          mbar_wait(&bar_done[slot], n_done & 1); n_done++;
          tc_fence_after();
          float o[NET::OUT];
#pragma unroll
          for (int j = 0; j < NET::OUT; ++j) o[j] = sBias[s_bias[NET::STAGES - 1] + j];
          if constexpr (SV::kOn)
            convert_row_out<NET::ACT, FMT, H, NET::OUT, true>(dD, sBias + Y.wout_f32_off, o,
                tile_row_ptr(sv.acts, (int64_t)L * sv.ntiles + (m >> 7), H + kTileRowsExtra, lane_row),
                sv.masks + (int64_t)L * (H / 32) * (sv.ntiles * 128) + m, sv.ntiles * 128);
          else if constexpr (SV::kF32)
            convert_row_out_savef32<NET::ACT, FMT, H, NET::OUT>(dD, sBias + Y.wout_f32_off, o,
                                                                  valid ? sv.acts + ((int64_t)L * H) * sv.M + m : nullptr, sv.M);
          else
            convert_row_out<NET::ACT, FMT, H, NET::OUT, false, kPipeRow || (NRT_SOFTPLUS_POLY != 0)>(dD, sBias + Y.wout_f32_off, o);
          if constexpr (ITER) { if (valid) io.consume(state, o); }
          else { if (valid) io.store(m, o); }
          tc_fence_before();
        } else {
          mbar_wait(&bar_done[slot], n_done & 1); n_done++;
          tc_fence_after();
          constexpr int OC = (NET::OUT + 7) / 8 * 8;
          uint32_t acc[OC];
          bstamp(it_dbg, 3);
          tmem_load<OC>(dD, acc);
          if constexpr (PIPE) {
            // the output MMAs have read the last hidden activations: the next tile's encoding goes into the union and
            // encoding regions, and once the accumulator is in registers its init layer may overwrite it
            if (has_next) enc_store(en);
            tc_wait_ld();
            if (has_next) {
              tc_wait_st();
              bstamp(it_dbg + 1, 6);
              tc_fence_before();
              mbar_arrive(&bar_ready[slot]);
              bstamp(it_dbg + 1, 7);
              fetch((t0 + slot + 2 * tstride) * 128 + lane_row);
            }
          } else {
            tc_wait_ld();
          }
          float o[NET::OUT];   // bias already accumulated (pre-loaded into the accumulator)
#pragma unroll
          for (int j = 0; j < NET::OUT; ++j) o[j] = __uint_as_float(acc[j]);
          if constexpr (ITER) { if (valid) io.consume(state, o); }
          else { if (valid) io.store(m, o); }
          bstamp(it_dbg, 4);
          // the accumulator / operand regions of this slot may now be reused by the next tile
          tc_fence_before();
        }
      }
      if constexpr (ITER) { if (primary) io.finish(state); }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (is_mma_warp) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}


}  // namespace tc
