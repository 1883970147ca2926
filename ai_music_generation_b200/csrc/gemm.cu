// bf16 GEMM for sm_100a: C[M,N] = sum_k A[m,k] * B[n,k], fp32 accumulation in TMEM.
//
// Covers every nn.Linear of the reference's hot path (nanoGPT/model.py:56,75,88,90,186) in its three
// autograd roles, selected by operand majorness instead of materialised transposes:
//   forward  Y  = X  * W^T        A = X  (K-major)   B = W  (K-major)
//   dgrad    dX = dY * W          A = dY (K-major)   B = W  (MN-major: W is [k_contract, n_out] row-major)
//   wgrad    dW = dY^T * X        A = dY (MN-major)  B = X  (MN-major), fp32 reduction into the grad arena
//
// Structure (one CTA per SM, persistent over output tiles):
//   warp 0      TMA producer   cp.async.bulk.tensor 2D, 128B swizzle, STAGES-deep mbarrier ring
//   warp 1      MMA issuer     one thread issues tcgen05.mma.cta_group::1.kind::f16 (128 x BN x 16)
//   warps 2..9  epilogue       tcgen05.ld TMEM -> registers -> fused epilogue -> global
// The accumulator is double-buffered in TMEM (2 x BN columns) so the epilogue of tile i overlaps the
// main loop of tile i+1.
#include "common.h"
#include "dropout.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace abcgpt {

unsigned long long* g_gemm_stats = nullptr;  // debug only: set through abcgpt_debug_gemm_stats

namespace {

__device__ __forceinline__ long long globaltimer_ns() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kNumEpiWarps = 16;   // four per scheduler: the epilogue arithmetic is dependency-latency bound (ncu: `wait` stalls,
                                   // IPC 0.15 with two warps per scheduler), so it needs thread-level parallelism, not fewer instructions
constexpr int kNumThreads = 64 + 32 * kNumEpiWarps;  // 1 producer warp + 1 MMA warp + the epilogue warps
// Warp roles.  The two issuing warps take the HIGHEST warp ids of the CTA: the scheduler arbitrates highest-warp-id-first among
// eligible warps (B300_MICROARCH "arbiter priority"), and with ids 0 / 1 the TMA and MMA issuers — a few dozen instructions per
// k-block on the critical path of the tensor pipe — queued behind the four epilogue warps of their scheduler whenever those
// were in their arithmetic phase.
constexpr int kProdWarp = kNumEpiWarps, kMmaWarp = kNumEpiWarps + 1, kEpiWarp0 = 0;

struct GemmParams {
  int M, N, K;
  int num_m_blk, num_n_blk, num_k_blk;
  int splits, kb_per_split;
  void* c;
  long long ldc;
  void* c2;
  long long ldc2;
  const void* aux;
  long long ldaux;
  const float* bias;
  int act_tanh;  // GELU / DGELU epilogues: 0 = exact erf (nn.GELU()), 1 = tanh form (HF "gelu_new", TunesFormer's GPT-2 blocks)
  int wide;  // 1: every epilogue pointer / leading dimension is 32-byte aligned -> 256-bit global accesses
  DropCfg drop;  // RESID epilogue only: dropout on the Linear output before the residual add (model.py:75-76,91)
  long long head_stride;  // BF16 epilogue: != 0 -> column c of a row goes to (c / 64) * head_stride + c % 64 (head-major KV cache)
  int half_from, half_extra;  // pair kernel: tiles >= half_from are processed as two 256 x 128 half tiles (work items
                              // half_from + 2 j, + 2 j + 1 of tile half_from + j): see "Half tiles" above gemm2_kernel
  unsigned long long* stats;  // optional debug counters (cycles): [0] producer empty-wait, [1] mma full-wait,
                              // [2] mma tmem-empty wait, [3] epilogue tmem-full wait, [4] epilogue busy, [5] cta total
};

template <int BN>
struct Cfg {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN >= 256) ? 4 : (BN >= 192 ? 5 : (BN >= 128 ? 6 : 8));
  static constexpr int TMEM_COLS = (2 * BN <= 128) ? 128 : ((2 * BN <= 256) ? 256 : 512);
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256 /*barriers*/ + 1024 /*alignment slack*/;
};

// ---- GELU (exact-erf form of nn.GELU(), model.py:83) ---------------------------------------------------
// Evaluated on the packed fp32x2 FMA pipe for two columns at a time with ONE MUFU per element.
//   Phi(-t)   = 0.5 erfc(t / sqrt 2)         = 2^(t (a2 t + a1)) P6(t)      t = min(|x|, 6.5)
//   gelu'(-t) = Phi(-t) - t phi(t)           = 2^(t (a2 t + b1)) Q5(t)
// i.e. a Gaussian times e^(-b t) (the linear term absorbs most of the Mills ratio's decay) times a short polynomial, fitted for
// minimal ABSOLUTE error of the product on [0, 6.5] (Lawson-weighted least squares, tools/fit_gelu.py): |dPhi| < 1.5e-7 in fp32 arithmetic (the class of erff itself, and of the Abramowitz-Stegun 7.1.26 form
// this replaces), |d gelu'| < 2.8e-6 (the derivative only multiplies a bf16 gradient).  Beyond 6.5 the clamp leaves
// Phi(-t) < 5e-11.  Then gelu(x) = x/2 + |x| (1/2 - Phi(-|x|)) and gelu'(x) = 1/2 + sign(x) (1/2 - gelu'(-|x|)).
// Why: the A-S form needs a reciprocal AND an exponential per element (4 MUFU per column pair); at 16 MUFU lanes per SM the
// 128 x 256 elements of a CTA's output tile cost 4096 cycles of MUFU issue against the 6144 cycles of a K = 768 main loop, and
// the GELU / GELU' epilogues were the bottleneck of their GEMMs (accumulator-empty waits of 25-40 % on the MMA issuer,
// tools/gemm_stats.py).  Here: 15-16 FMA-pipe instructions + 2 MUFU per pair.
constexpr float kGeluClamp = 6.5f;
__device__ __forceinline__ float2 f2u(uint32_t a, uint32_t b) { return make_float2(__uint_as_float(a), __uint_as_float(b)); }
__device__ __forceinline__ float2 ex2_2(float2 a) {
  float2 e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(a.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(a.y));
  return e;
}
#define ABCGPT_C2(c) make_float2(c, c)
// Phi(-t), t >= 0 already clamped
__device__ __forceinline__ float2 gelu_q2(float2 t) {
  const float2 arg = __fmul2_rn(t, __ffma2_rn(t, ABCGPT_C2(-0.72134752044448170f), ABCGPT_C2(-1.3849872392534049f)));  // -(t^2/2 + 0.96 t) log2 e
  const float2 e = ex2_2(arg);
  float2 acc = ABCGPT_C2(2.6089192608e-04f);
  acc = __ffma2_rn(acc, t, ABCGPT_C2(-9.7434194520e-04f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(8.2275534932e-03f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(-2.7531754286e-03f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(9.7337472177e-02f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(8.1064425089e-02f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(4.9999990985e-01f));
  return __fmul2_rn(acc, e);
}
__device__ __forceinline__ float2 gelu_fwd2(float2 x) {
  const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
  const float2 t = make_float2(fminf(ax.x, kGeluClamp), fminf(ax.y, kGeluClamp));
  const float2 d = __ffma2_rn(gelu_q2(t), ABCGPT_C2(-1.0f), ABCGPT_C2(0.5f));  // 1/2 - Phi(-|x|) >= 0
  return __ffma2_rn(d, ax, __fmul2_rn(x, ABCGPT_C2(0.5f)));
}
__device__ __forceinline__ float2 gelu_bwd2(float2 x) {
  const float2 t = make_float2(fminf(fabsf(x.x), kGeluClamp), fminf(fabsf(x.y), kGeluClamp));
  const float2 arg = __fmul2_rn(t, __ffma2_rn(t, ABCGPT_C2(-0.72134752044448170f), ABCGPT_C2(-0.75020142126226098f)));  // -(t^2/2 + 0.52 t) log2 e
  const float2 e = ex2_2(arg);
  float2 acc = ABCGPT_C2(-3.6013674782e-03f);
  acc = __ffma2_rn(acc, t, ABCGPT_C2(4.0705955963e-03f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(-9.5264921960e-02f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(-9.8502707031e-02f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(-5.3775135947e-01f));
  acc = __ffma2_rn(acc, t, ABCGPT_C2(4.9999814610e-01f));
  const float2 d = __ffma2_rn(__fmul2_rn(acc, e), ABCGPT_C2(-1.0f), ABCGPT_C2(0.5f));  // 1/2 - gelu'(-|x|)
  // 1/2 + sign(x) d: flip d's sign where x is negative
  const float dx = __uint_as_float(__float_as_uint(d.x) ^ (__float_as_uint(x.x) & 0x80000000u));
  const float dy = __uint_as_float(__float_as_uint(d.y) ^ (__float_as_uint(x.y) & 0x80000000u));
  return __fadd2_rn(make_float2(dx, dy), ABCGPT_C2(0.5f));
}

// tanh form: gelu_new(x) = 0.5 x (1 + tanh(k (x + 0.044715 x^3))), k = sqrt(2/pi)   (tunesformer/utils.py: HF GPT2 activation)
__device__ __forceinline__ float2 gelu_tanh_t2(float2 x, float2& inner_deriv) {
  const float2 xx = __fmul2_rn(x, x);
  const float2 u = __fmul2_rn(x, __ffma2_rn(xx, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f)));
  inner_deriv = __ffma2_rn(xx, make_float2(0.1070322243f, 0.1070322243f), make_float2(0.7978845608f, 0.7978845608f));
  float2 t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(u.x));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(u.y));
  return t;
}
__device__ __forceinline__ float2 gelu_tanh_fwd2(float2 x) {
  float2 du;
  const float2 t = gelu_tanh_t2(x, du);
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(hx, t, hx);
}
__device__ __forceinline__ float2 gelu_tanh_bwd2(float2 x) {
  float2 du;
  const float2 t = gelu_tanh_t2(x, du);
  // 0.5 (1 + t) + 0.5 x (1 - t^2) du
  const float2 omt2 = __ffma2_rn(t, make_float2(-t.x, -t.y), make_float2(1.0f, 1.0f));
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  const float2 a = __ffma2_rn(t, make_float2(0.5f, 0.5f), make_float2(0.5f, 0.5f));
  return __ffma2_rn(__fmul2_rn(hx, omt2), du, a);
}

// ---- epilogues: one thread owns 32 consecutive columns of one output row -------------------------------
// Auxiliary inputs (the fp32 residual for RESID, the bf16 pre-activation for DGELU) do not depend on the
// accumulator, so they are fetched BEFORE the thread blocks on the accumulator barrier: their DRAM latency hides
// behind the main loop instead of adding to the epilogue.
template <int EPI>
struct AuxChunk {
  // RESID: 32 fp32 = 4 x 32 B; DGELU: 32 bf16 = 2 x 32 B
  static constexpr int N = (EPI == ABCGPT_EPI_RESID) ? 4 : ((EPI == ABCGPT_EPI_DGELU) ? 2 : 1);
  ptx::u32x8 v[N];
};

template <int EPI>
__device__ __forceinline__ void load_aux(AuxChunk<EPI>& a, const GemmParams& p, int row, int col0) {
  if constexpr (EPI == ABCGPT_EPI_RESID || EPI == ABCGPT_EPI_DGELU) {
    constexpr int EB = (EPI == ABCGPT_EPI_RESID) ? 4 : 2;  // element bytes
    constexpr int PER = 32 / EB;                            // elements per 32-byte group
    const char* base = reinterpret_cast<const char*>(p.aux) + (static_cast<long long>(row) * p.ldaux + col0) * EB;
#pragma unroll
    for (int j = 0; j < AuxChunk<EPI>::N; ++j) {
      const int c = col0 + j * PER;
      if (row < p.M && c + PER <= p.N && p.wide) {
        a.v[j] = ptx::ldg256(base + 32 * j);
      } else {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint4 t = make_uint4(0u, 0u, 0u, 0u);
          if (row < p.M && c + h * (PER / 2) < p.N) t = __ldg(reinterpret_cast<const uint4*>(base + 32 * j + 16 * h));
          a.v[j].v[4 * h + 0] = t.x; a.v[j].v[4 * h + 1] = t.y; a.v[j].v[4 * h + 2] = t.z; a.v[j].v[4 * h + 3] = t.w;
        }
      }
    }
  }
}

// store 16 bf16 columns (8 packed words) starting at column 16*j of the chunk; ncols is a multiple of 8
__device__ __forceinline__ void store_bf16x16(__nv_bfloat16* c, int j, int ncols, bool wide, const uint32_t* pk) {
  if (16 * j + 16 <= ncols && wide) {
    ptx::stg256(c + 16 * j, pk[0], pk[1], pk[2], pk[3], pk[4], pk[5], pk[6], pk[7]);
  } else {
    if (16 * j < ncols) reinterpret_cast<uint4*>(c + 16 * j)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    if (16 * j + 8 < ncols) reinterpret_cast<uint4*>(c + 16 * j)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
  }
}

template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, int row, int col0, uint32_t (&r)[32],
                                               const AuxChunk<EPI>& aux) {
  if (row >= p.M || col0 >= p.N) return;
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
  if (p.bias != nullptr) {
    if (col0 + 32 <= p.N && (reinterpret_cast<uintptr_t>(p.bias + col0) & 15) == 0) {
      // every thread of the warp reads the same 32 columns: eight broadcast 128-bit loads instead of 32 scalar ones
      const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (col0 + i < p.N) v[i] += __ldg(p.bias + col0 + i);
    }
  }
  const int ncols = min(32, p.N - col0);  // multiple of 8 (host-checked)

  if constexpr (EPI == ABCGPT_EPI_BF16 || EPI == ABCGPT_EPI_GELU || EPI == ABCGPT_EPI_DGELU) {
    __nv_bfloat16* c = reinterpret_cast<__nv_bfloat16*>(p.c) + static_cast<long long>(row) * p.ldc +
                       (p.head_stride ? (col0 >> 6) * p.head_stride + (col0 & 63) : col0);
    uint32_t pk[16];
    if constexpr (EPI == ABCGPT_EPI_DGELU) {
      // dH = bf16(acc) * gelu'(h): the reference's gelu_backward sees the bf16 dgrad output and the bf16 h
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const uint32_t hw = aux.v[i >> 3].v[i & 7];
        const uint32_t db = ptx::pack_bf16x2(v[2 * i], v[2 * i + 1]);
        const float2 hx = make_float2(ptx::bf16lo(hw), ptx::bf16hi(hw));
        const float2 d = __fmul2_rn(make_float2(ptx::bf16lo(db), ptx::bf16hi(db)), p.act_tanh ? gelu_tanh_bwd2(hx) : gelu_bwd2(hx));
        pk[i] = ptx::pack_bf16x2(d.x, d.y);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) pk[i] = ptx::pack_bf16x2(v[2 * i], v[2 * i + 1]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) store_bf16x16(c, j, ncols, p.wide, pk + 8 * j);
    if constexpr (EPI == ABCGPT_EPI_GELU) {
      __nv_bfloat16* g = reinterpret_cast<__nv_bfloat16*>(p.c2) + static_cast<long long>(row) * p.ldc2 + col0;
      uint32_t gk[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float2 hx = make_float2(ptx::bf16lo(pk[i]), ptx::bf16hi(pk[i]));  // GELU of the bf16 h
        const float2 a = p.act_tanh ? gelu_tanh_fwd2(hx) : gelu_fwd2(hx);
        gk[i] = ptx::pack_bf16x2(a.x, a.y);
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) store_bf16x16(g, j, ncols, p.wide, gk + 8 * j);
    }
  } else if constexpr (EPI == ABCGPT_EPI_RESID) {
    // x_out(fp32) = x_in(fp32) + bf16(acc): the reference adds the bf16 Linear output into the fp32 stream
    float* xout = reinterpret_cast<float*>(p.c) + static_cast<long long>(row) * p.ldc + col0;
    const uint32_t drop_rk = drop_row_key(p.drop.key, static_cast<uint32_t>(row));
#pragma unroll
    for (int j = 0; j < 4; ++j) {  // 8 columns per 32-byte group
      if (8 * j < ncols) {
        uint32_t o[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t b = ptx::pack_bf16x2(v[8 * j + 2 * q], v[8 * j + 2 * q + 1]);
          float y0 = ptx::bf16lo(b), y1 = ptx::bf16hi(b);
          if (p.drop.thr16 != 0) {  // bf16 dropout like nn.Dropout on the bf16 Linear output: scale, round, or zero
            const uint32_t bits = drop_pair_bits(drop_rk, static_cast<uint32_t>(col0 + 8 * j + 2 * q) >> 1);
            y0 = drop_keep_lo(bits, p.drop.thr16) ? ptx::bf16_round(y0 * p.drop.inv_keep) : 0.f;
            y1 = drop_keep_hi(bits, p.drop.thr16) ? ptx::bf16_round(y1 * p.drop.inv_keep) : 0.f;
          }
          o[2 * q] = __float_as_uint(__uint_as_float(aux.v[j].v[2 * q]) + y0);
          o[2 * q + 1] = __float_as_uint(__uint_as_float(aux.v[j].v[2 * q + 1]) + y1);
        }
        if (p.wide) {
          ptx::stg256(xout + 8 * j, o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7]);
        } else {
          reinterpret_cast<uint4*>(xout + 8 * j)[0] = make_uint4(o[0], o[1], o[2], o[3]);
          reinterpret_cast<uint4*>(xout + 8 * j)[1] = make_uint4(o[4], o[5], o[6], o[7]);
        }
      }
    }
  } else if constexpr (EPI == ABCGPT_EPI_F32_RED) {
    float* c = reinterpret_cast<float*>(p.c) + static_cast<long long>(row) * p.ldc + col0;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (4 * j < ncols) ptx::red_add_v4(c + 4 * j, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  } else {  // ABCGPT_EPI_F32
    float4* c = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.c) + static_cast<long long>(row) * p.ldc + col0);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (4 * j < ncols) c[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  }
}

// fp32 accumulator words (+ bias) -> packed bf16 pairs, 16 registers per 32 columns (TMA-store epilogues of the pair kernel).
// (A variant that packed BOTH chunks of a tile before any arithmetic, to hand the accumulator back earlier, measured slower:
// c_fc + GELU 0.163 vs 0.155 ms — 64 live accumulator registers leave the 96-register budget of an 18-warp CTA no room.)
__device__ __forceinline__ void pack_chunk(const GemmParams& p, int col0, const uint32_t (&r)[32], uint32_t (&pk)[16]) {
  if (p.bias != nullptr && col0 < p.N) {
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
    if (col0 + 32 <= p.N && (reinterpret_cast<uintptr_t>(p.bias + col0) & 15) == 0) {
      const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (col0 + i < p.N) v[i] += __ldg(p.bias + col0 + i);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) pk[i] = ptx::pack_bf16x2(v[2 * i], v[2 * i + 1]);
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) pk[i] = ptx::pack_bf16x2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
  }
}

// write 32 consecutive bf16 columns (16 packed words = 64 bytes) of row r of a [32 rows x 64 B] SWIZZLE_64B staging chunk:
// 16-byte unit j of row r lives at unit j ^ ((r >> 1) & 3) (address bits [4,6) ^= bits [7,9)); eight consecutive lanes
// cover all 32 banks, so the four 128-bit stores are conflict-free
__device__ __forceinline__ void st_stage_bf16(uint32_t buf, int r, const uint32_t* pk) {
  const uint32_t base = buf + r * 64;
  const int x = (r >> 1) & 3;
#pragma unroll
  for (int q = 0; q < 4; ++q)
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + ((q ^ x) << 4)), "r"(pk[4 * q]), "r"(pk[4 * q + 1]),
                 "r"(pk[4 * q + 2]), "r"(pk[4 * q + 3])
                 : "memory");
}

__device__ __forceinline__ void timed_wait(uint64_t* bar, uint32_t parity, int tag, unsigned long long* stats, int slot,
                                           long long& acc) {
  if (stats == nullptr) {
    ptx::mbar_wait(bar, parity, tag);
  } else {
    const long long t0 = clock64();
    ptx::mbar_wait(bar, parity, tag);
    acc += clock64() - t0;
  }
}

template <int BN, bool A_MN, bool B_MN, int EPI>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty = full + C::STAGES;
  uint64_t* tfull = empty + C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = ptx::uniform(threadIdx.x >> 5);  // provably warp-uniform: the issuer loops below stay on the uniform datapath
  const int lane = threadIdx.x & 31;

  if (warp == kProdWarp && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int s = 0; s < C::STAGES; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], kNumEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    ptx::tmem_alloc(tmem_slot, C::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();               // everything above touched only this CTA's shared memory / TMEM

  const int total_work = p.num_m_blk * p.num_n_blk * p.splits;
  const long long t_start = p.stats ? clock64() : 0;
  long long w0 = 0, w1 = 0;

  if (warp == kProdWarp) {
    // ===================== TMA producer =====================
    {
      const bool issue = ptx::elect_one();  // whole warp runs the loop, one elected lane issues (uniform operands)
      int stage = 0;
      uint32_t phase = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        const int split = w % p.splits;
        const int tile = w / p.splits;
        const int m_blk = tile / p.num_n_blk;
        const int n_blk = tile % p.num_n_blk;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.num_k_blk, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          timed_wait(&empty[stage], phase ^ 1, 1, p.stats, 0, w0);
          if (issue) ptx::mbar_expect_tx(&full[stage], C::STAGE_BYTES);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          if constexpr (!A_MN) {
            if (issue) ptx::tma_load_2d(sa, &tmA, &full[stage], kb * BK, m_blk * BM);
          } else {
#pragma unroll
            for (int a = 0; a < BM / 64; ++a)
              if (issue) ptx::tma_load_2d(sa + a * (BK * 128), &tmA, &full[stage], m_blk * BM + a * 64, kb * BK);
          }
          if constexpr (!B_MN) {
            if (issue) ptx::tma_load_2d(sb, &tmB, &full[stage], kb * BK, n_blk * BN);
          } else {
#pragma unroll
            for (int b = 0; b < BN / 64; ++b)
              if (issue) ptx::tma_load_2d(sb + b * (BK * 128), &tmB, &full[stage], n_blk * BN + b * 64, kb * BK);
          }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      if (issue && p.stats) atomicAdd(&p.stats[0], static_cast<unsigned long long>(w0));
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer =====================
    {
      // the whole warp runs the loop (uniform operands, see ptx::elect_one); one elected lane issues
      const bool issue = ptx::elect_one();
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x, ++it) {
        const int split = w % p.splits;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.num_k_blk, kb0 + p.kb_per_split);
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        timed_wait(&tempty[as], aphase ^ 1, 2, p.stats, 2, w1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          timed_wait(&full[stage], phase, 3, p.stats, 1, w0);
          ptx::tc_fence_after();
          const uint32_t a_base = ptx::smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t b_base = a_base + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // K-major SW128: 16 bf16 of K = 32 bytes inside the 128-byte swizzle row; SBO = 8 rows * 128 B.
            // MN-major SW128: 16 K-rows = 2048 B; LBO = one 64-wide MN atom (BK rows * 128 B), SBO = 1024 B.
            const uint64_t adesc = A_MN ? ptx::umma_smem_desc(a_base + k * 2048, BK * 128, 1024)
                                        : ptx::umma_smem_desc(a_base + k * 32, 0, 1024);
            const uint64_t bdesc = B_MN ? ptx::umma_smem_desc(b_base + k * 2048, BK * 128, 1024)
                                        : ptx::umma_smem_desc(b_base + k * 32, 0, 1024);
            if (issue) ptx::umma_ss(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if (issue) ptx::umma_commit(&empty[stage]);  // frees the smem slot once these MMAs have read it
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (issue) ptx::umma_commit(&tfull[as]);  // accumulator complete
      }
      if (issue && p.stats) {
        atomicAdd(&p.stats[1], static_cast<unsigned long long>(w0));
        atomicAdd(&p.stats[2], static_cast<unsigned long long>(w1));
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps =====================
    const int quarter = warp & 3;          // TMEM lanes [32*quarter, 32*quarter+32) are visible to this warp
    const int half = (warp - kEpiWarp0) >> 2;      // which quarter of the BN columns
    constexpr int COLS_PER_WARP = BN / (kNumEpiWarps / 4);
    int it = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x, ++it) {
      const int tile = w / p.splits;
      const int m_blk = tile / p.num_n_blk;
      const int n_blk = tile % p.num_n_blk;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      const int row = m_blk * BM + quarter * 32 + lane;
      const int col_base = n_blk * BN + half * COLS_PER_WARP;
      constexpr int NCH = COLS_PER_WARP / 32;
      AuxChunk<EPI> aux[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) load_aux<EPI>(aux[c], p, row, col_base + c * 32);
      timed_wait(&tfull[as], aphase, 4, p.stats, 3, w0);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + as * BN + half * COLS_PER_WARP;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        uint32_t r[32];
        ptx::tmem_ld32(taddr + c * 32, r);
        ptx::tmem_ld_wait();
        epilogue_chunk<EPI>(p, row, col_base + c * 32, r, aux[c]);
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[as]);
    }
    if (p.stats && warp == kEpiWarp0 && lane == 0) {
      atomicAdd(&p.stats[3], static_cast<unsigned long long>(w0));
      atomicAdd(&p.stats[5], static_cast<unsigned long long>(clock64() - t_start));
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) ptx::tmem_dealloc(tmem_base, C::TMEM_COLS);
}

template <int BN, bool A_MN, bool B_MN, int EPI>
int launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, int grid, cudaStream_t stream) {
  using C = Cfg<BN>;
  auto kern = gemm_kernel<BN, A_MN, B_MN, EPI>;
  static bool configured = false;  // per instantiation; benign race (idempotent)
  if (!configured) {
    ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    configured = true;
  }
  launch_k(kern, dim3(grid), dim3(kNumThreads), C::SMEM_BYTES, stream, tmA, tmB, p);
  return launch_status("gemm_kernel");
}

template <int BN, bool A_MN, bool B_MN>
int dispatch_epi(int epi, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, int grid,
                 cudaStream_t stream) {
  switch (epi) {
    case ABCGPT_EPI_BF16: return launch<BN, A_MN, B_MN, ABCGPT_EPI_BF16>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_GELU: return launch<BN, A_MN, B_MN, ABCGPT_EPI_GELU>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_RESID: return launch<BN, A_MN, B_MN, ABCGPT_EPI_RESID>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_DGELU: return launch<BN, A_MN, B_MN, ABCGPT_EPI_DGELU>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_F32_RED: return launch<BN, A_MN, B_MN, ABCGPT_EPI_F32_RED>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_F32: return launch<BN, A_MN, B_MN, ABCGPT_EPI_F32>(tmA, tmB, p, grid, stream);
  }
  return fail(-1, "unknown GEMM epilogue %d", epi);
}

template <int BN>
int dispatch_major(int a_mn, int b_mn, int epi, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p,
                   int grid, cudaStream_t stream) {
  if (!a_mn && !b_mn) return dispatch_epi<BN, false, false>(epi, tmA, tmB, p, grid, stream);
  if (!a_mn && b_mn) return dispatch_epi<BN, false, true>(epi, tmA, tmB, p, grid, stream);
  if (a_mn && b_mn) return dispatch_epi<BN, true, true>(epi, tmA, tmB, p, grid, stream);
  return fail(-1, "GEMM operand combination A=MN-major,B=K-major is not instantiated");
}


// =====================================================================================================================
// CTA-pair variant (cta_group::2): two CTAs of a cluster compute one 256 x 256 output tile.  Each CTA stages its own
// 128 rows of A and its own 128 rows (half of N) of B, so per-CTA operand traffic from L2 drops from 48 KB to 32 KB per
// 64-deep k-block and the ring gets 6 stages; the leader CTA issues tcgen05.mma.cta_group::2 (M = 256), which reads
// both CTAs' shared memory and writes both CTAs' TMEM.  Barrier protocol:
//   full[s]    (leader)  1 arrival (leader's expect_tx for BOTH CTAs' bytes) + complete_tx from both CTAs' TMA
//   empty[s]   (each)    tcgen05.commit multicast to both CTAs
//   tfull[a]   (each)    tcgen05.commit multicast to both CTAs
//   tempty[a]  (leader)  2 x 8 epilogue warps (the peer's arrive remotely)
// =====================================================================================================================
struct Cfg2 {
  static constexpr int BN = 256;
  static constexpr int A_BYTES = BM * BK * 2;         // 128 rows of A per CTA
  static constexpr int B_BYTES = (BN / 2) * BK * 2;   // 128 of the 256 B rows per CTA
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int TMEM_COLS = 512;
};
// TMA-store epilogues (TS): every epilogue warp owns TWO staging buffers of one 32-row x 32-column bf16 chunk each (2 KB,
// SWIZZLE_64B): one per output stream for the GELU epilogue (h and gelu(h)), alternating by chunk for the single-stream ones.
// Every tensor store is its own bulk group and a buffer is rewritten after cp.async.bulk.wait_group.read 1, i.e. the store that
// read it last has had one whole other store's worth of arithmetic to drain (with one buffer and wait_group.read 0 the warps
// spent 14 % of their time in that wait, ncu source view).  The staging area costs one operand stage (5 instead of 6).
template <int EPI, bool TS>
struct Cfg2S {
  static constexpr int NOUT = !TS ? 0 : (EPI == ABCGPT_EPI_GELU ? 2 : 1);
  static constexpr int STG_WARP = TS ? 4096 : 0;
  static constexpr int STG_BYTES = kNumEpiWarps * STG_WARP;
  static constexpr int STAGES = TS ? 5 : 6;
  static constexpr int RING_BYTES = STAGES * Cfg2::STAGE_BYTES;
  static constexpr int SMEM_BYTES = RING_BYTES + STG_BYTES + 512 + 1024;
  static_assert(SMEM_BYTES <= 232448, "pair GEMM: shared memory budget");
};

// 18 warps: ptxas caps the kernel at 96 registers per thread, and that IS the hardware limit (registers are allocated per warp
// in units of 512: 112 per thread rounds to 4096 per warp, x 18 > 65 536 — a __maxnreg__(112) build fails to launch).
template <bool A_MN, bool B_MN, int EPI, bool TS>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmC2, const GemmParams p) {
  struct C : Cfg2, Cfg2S<EPI, TS> {};
  constexpr int BN = C::BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint8_t* ctrl = smem + C::RING_BYTES + C::STG_BYTES;   // operand ring | epilogue staging (TS) | barriers
  uint64_t* full = reinterpret_cast<uint64_t*>(ctrl);
  uint64_t* empty = full + C::STAGES;
  uint64_t* tfull = empty + C::STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = ptx::uniform(threadIdx.x >> 5);  // provably warp-uniform: the issuer loops below stay on the uniform datapath
  const int lane = threadIdx.x & 31;
  const uint32_t crank = ptx::cluster_ctarank();  // rank in the cluster
  const uint32_t rank = crank & 1;                // CTA within its pair
  const uint32_t pr = crank >> 1;                 // pair within the cluster
  const bool leader = rank == 0;
  // debug timeline (p.stats, tools/gemm_timeline.py), nanoseconds of %globaltimer over all CTAs: [8] min kernel entry, [9] max
  // "prologue done", [10] min / [11] max "first operand stage landed", [12] max "last MMA committed", [13] max "epilogue
  // done", [14] max kernel exit, [15] min "prologue done"
  if (p.stats && threadIdx.x == 0) atomicMin(&p.stats[8], static_cast<unsigned long long>(globaltimer_ns()));

  if (warp == kProdWarp && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    if constexpr (TS) {
      ptx::prefetch_tmap(&tmC);
      if constexpr (C::NOUT == 2) ptx::prefetch_tmap(&tmC2);
    }
    for (int s = 0; s < C::STAGES; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], 2 * kNumEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    ptx::tmem_alloc_2sm(tmem_slot, C::TMEM_COLS);
    ptx::tmem_relinquish_2sm();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // barrier inits + TMEM allocations of BOTH CTAs are visible before anything is signalled
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();               // everything above touched only this CTA's shared memory / TMEM
  long long g_start = 0;
  if (p.stats && threadIdx.x == 0) {
    const unsigned long long t = static_cast<unsigned long long>(globaltimer_ns());
    atomicMax(&p.stats[9], t);
    atomicMin(&p.stats[15], t);
  }
  if (p.stats) g_start = globaltimer_ns();

  const int m_units = (p.num_m_blk + 1) / 2;
  // Half tiles: with T tiles on P pairs the static schedule takes ceil(T / P) rounds; when the last round would hold r <= P / 2
  // tiles (GPT-2-small's N = 768 layers at 32 k tokens: 384 tiles on 74 pairs = 5.19 -> 6 rounds, 13 % of the GEMM idle), those r
  // tiles are issued as 2 r work items of 256 x 128 (MMA N = 128: the same operand boxes are loaded and the first 64 B rows /
  // columns of each CTA used, half the MMA time, column groups 2 and 3 of the epilogue idle): the last round costs half a tile.
  const int total_work = m_units * p.num_n_blk * p.splits + p.half_extra;
  const int pair_id = blockIdx.x / 2;       // cluster index
  const long long t_start = p.stats ? clock64() : 0;
  long long w0 = 0, w1 = 0;
  const int num_pairs = gridDim.x / 2;
  // static round-robin: iteration `it` of a pair processes work item pair_id + it * num_pairs

  if (warp == kProdWarp) {
    // ===================== TMA producer (both CTAs) =====================
    {
      const bool issue = ptx::elect_one();  // whole warp runs the loop, one elected lane issues (uniform operands)
      int stage = 0;
      uint32_t phase = 0;
      for (int w = pair_id; w < total_work; w += num_pairs) {
        const int split = w % p.splits;
        const bool is_half = w >= p.half_from;   // (half tiles only with splits == 1: w is the tile index below half_from)
        const int tile = is_half ? p.half_from + ((w - p.half_from) >> 1) : w / p.splits;
        const int m_unit = tile / p.num_n_blk;
        const int m0 = m_unit * 256 + static_cast<int>(rank) * 128;
        const int n0 = (tile % p.num_n_blk) * BN + (is_half ? ((w - p.half_from) & 1) * (BN / 2) + static_cast<int>(rank) * (BN / 4)
                                                             : static_cast<int>(rank) * (BN / 2));
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.num_k_blk, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          timed_wait(&empty[stage], phase ^ 1, 41, p.stats, 0, w0);
          const uint32_t full_leader = ptx::mapa(ptx::smem_u32(&full[stage]), crank & ~1u);  // own pair's leader
          if (leader && issue) ptx::mbar_expect_tx(&full[stage], 2 * C::STAGE_BYTES);
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          uint8_t* sb = sa + C::A_BYTES;
          if constexpr (!A_MN) {
            if (issue) ptx::tma_load_2d_2sm(sa, &tmA, full_leader, kb * BK, m0);
          } else {
#pragma unroll
            for (int a = 0; a < 2; ++a) if (issue) ptx::tma_load_2d_2sm(sa + a * (BK * 128), &tmA, full_leader, m0 + a * 64, kb * BK);
          }
          if constexpr (!B_MN) {
            if (issue) ptx::tma_load_2d_2sm(sb, &tmB, full_leader, kb * BK, n0);
          } else {
#pragma unroll
            for (int b = 0; b < 2; ++b) if (issue) ptx::tma_load_2d_2sm(sb + b * (BK * 128), &tmB, full_leader, n0 + b * 64, kb * BK);
          }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      if (issue && p.stats) atomicAdd(&p.stats[0], static_cast<unsigned long long>(w0));
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      // the whole warp runs the loop (uniform operands, see ptx::elect_one); one elected lane issues
      const bool issue = ptx::elect_one();
      constexpr uint32_t idesc_full = ptx::umma_idesc_bf16(256, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      constexpr uint32_t idesc_half = ptx::umma_idesc_bf16(256, BN / 2, A_MN ? 1 : 0, B_MN ? 1 : 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0, w = pair_id; w < total_work; ++it, w += num_pairs) {
        const uint32_t idesc = w >= p.half_from ? idesc_half : idesc_full;
        const int split = w % p.splits;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.num_k_blk, kb0 + p.kb_per_split);
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        timed_wait(&tempty[as], aphase ^ 1, 42, p.stats, 2, w1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          timed_wait(&full[stage], phase, 43, p.stats, 1, w0);
          ptx::tc_fence_after();
          if (p.stats && it == 0 && kb == kb0 && issue) {
            const unsigned long long t = static_cast<unsigned long long>(globaltimer_ns());
            atomicMin(&p.stats[10], t);
            atomicMax(&p.stats[11], t);
          }
          const uint32_t a_base = ptx::smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t b_base = a_base + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t adesc = A_MN ? ptx::umma_smem_desc(a_base + k * 2048, BK * 128, 1024)
                                        : ptx::umma_smem_desc(a_base + k * 32, 0, 1024);
            const uint64_t bdesc = B_MN ? ptx::umma_smem_desc(b_base + k * 2048, BK * 128, 1024)
                                        : ptx::umma_smem_desc(b_base + k * 32, 0, 1024);
            if (issue) ptx::umma_ss_2sm(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if (issue) ptx::umma_commit_2sm(&empty[stage], 0x3);
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (issue) ptx::umma_commit_2sm(&tfull[as], static_cast<uint16_t>(0x3u << (2 * pr)));
      }
      if (issue && p.stats) {
        atomicAdd(&p.stats[1], static_cast<unsigned long long>(w0));
        atomicAdd(&p.stats[2], static_cast<unsigned long long>(w1));
        atomicMax(&p.stats[12], static_cast<unsigned long long>(globaltimer_ns()));
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (both CTAs, own 128 rows) =====================
    const int quarter = warp & 3;
    const int half = (warp - kEpiWarp0) >> 2;      // which quarter of the BN columns
    constexpr int COLS_PER_WARP = BN / (kNumEpiWarps / 4);
    for (int it = 0, w = pair_id; w < total_work; ++it, w += num_pairs) {
      const bool is_half = w >= p.half_from;
      const int tile = is_half ? p.half_from + ((w - p.half_from) >> 1) : w / p.splits;
      const int m_unit = tile / p.num_n_blk;
      const int m0 = m_unit * 256 + static_cast<int>(rank) * 128;
      const int n_blk = tile % p.num_n_blk;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      const int row = m0 + quarter * 32 + lane;
      // half tile: accumulator columns [0, BN / 2) hold output columns n_blk BN + (w & 1) BN / 2 + ...; the warps of column
      // groups 2 and 3 have nothing to store (their column base is pushed past N: every store / load below clips itself)
      const int col_base = !is_half ? n_blk * BN + half * COLS_PER_WARP
                                    : (2 * half < kNumEpiWarps / 4 ? n_blk * BN + ((w - p.half_from) & 1) * (BN / 2) + half * COLS_PER_WARP
                                                                   : p.N + 32);
      constexpr int NCH = COLS_PER_WARP / 32;
      // auxiliary operands are requested before the accumulator wait (their DRAM latency hides behind the main loop)
      AuxChunk<EPI> aux[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) load_aux<EPI>(aux[c], p, row, col_base + c * 32);
      timed_wait(&tfull[as], aphase, 44, p.stats, 3, w0);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + as * BN + half * COLS_PER_WARP;
      if constexpr (TS) {
        // bf16 outputs leave through shared memory and the TMA engine: the thread writes the 64 bytes of its row into the
        // warp's swizzled staging chunk (conflict-free 128-bit stores), one lane issues a 2 KB tensor store per stream.  The
        // LSU sees 4 wavefronts per 512 bytes instead of the 16 of row-per-thread st.global.v8, nobody holds registers while
        // a store queue drains, rows >= M / columns >= N are clipped by the tensor map, and the accumulator goes back to the
        // MMA issuer as soon as the tile's LAST chunk is in registers (its arithmetic overlaps the next-but-one main loop).
        const int row0 = m0 + quarter * 32;
        const uint32_t stg = ptx::smem_u32(smem + C::RING_BYTES) + static_cast<uint32_t>(warp - kEpiWarp0) * C::STG_WARP;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int col0 = col_base + c * 32;
          uint32_t r[32];
          ptx::tmem_ld32(taddr + c * 32, r);
          ptx::tmem_ld_wait();
          if (c == NCH - 1) {
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tempty[as]), crank & ~1u));
          }
          if (row0 >= p.M || col0 >= p.N) continue;   // warp-uniform: the whole chunk lies outside the matrix
          if constexpr (EPI == ABCGPT_EPI_F32_RED) {
            // split-K / accumulating weight gradient: the 32 x 32 fp32 chunk leaves as two [32 rows x 64 B] staging halves, each
            // added into the gradient by ONE tensor reduction (whole 64-byte row pieces per L2 operation) instead of 32 x 8
            // row-per-thread red.global.add.v4 (16 bytes per L2 atomic, 32 different lines per warp instruction): the exposed
            // reduction of a pair's last tile was ~10 us of every wgrad launch (tools/gemm_timeline.py)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const uint32_t buf = stg + hh * 2048;
              if (lane == 0) ptx::tma_store_wait_read<1>();
              __syncwarp();
              st_stage_bf16(buf, lane, r + 16 * hh);
              ptx::fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0 && col0 + 16 * hh < p.N) {
                ptx::tma_reduce_add_2d_s(&tmC, buf, col0 + 16 * hh, row0);
                ptx::tma_store_commit();
              }
            }
            continue;
          }
          uint32_t pk[16];
          if constexpr (EPI == ABCGPT_EPI_DGELU) {
            // dH = acc * gelu'(h), one rounding.  (The reference's gelu_backward sees the dgrad output already rounded to bf16;
            // multiplying the fp32 accumulator skips that intermediate rounding — closer to the fp32 gradient, and three
            // instructions per column pair less in an epilogue that is the bottleneck of its GEMM.)
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const uint32_t hw = aux[c].v[i >> 3].v[i & 7];
              const float2 hx = make_float2(ptx::bf16lo(hw), ptx::bf16hi(hw));
              const float2 d = __fmul2_rn(f2u(r[2 * i], r[2 * i + 1]), p.act_tanh ? gelu_tanh_bwd2(hx) : gelu_bwd2(hx));
              pk[i] = ptx::pack_bf16x2(d.x, d.y);
            }
          } else {
            pack_chunk(p, col0, r, pk);
          }
          const uint32_t buf0 = (EPI == ABCGPT_EPI_GELU) ? stg : stg + (c & 1) * 2048;
          if (lane == 0) ptx::tma_store_wait_read<1>();   // the store that last read this buffer has drained (see Cfg2S)
          __syncwarp();
          st_stage_bf16(buf0, lane, pk);
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_2d_s(&tmC, buf0, col0, row0);
            ptx::tma_store_commit();
          }
          if constexpr (EPI == ABCGPT_EPI_GELU) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float2 hx = make_float2(ptx::bf16lo(pk[i]), ptx::bf16hi(pk[i]));  // GELU of the bf16 h
              const float2 a = p.act_tanh ? gelu_tanh_fwd2(hx) : gelu_fwd2(hx);
              pk[i] = ptx::pack_bf16x2(a.x, a.y);
            }
            if (lane == 0) ptx::tma_store_wait_read<1>();
            __syncwarp();
            st_stage_bf16(stg + 2048, lane, pk);
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              ptx::tma_store_2d_s(&tmC2, stg + 2048, col0, row0);
              ptx::tma_store_commit();
            }
          }
        }
      } else {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          uint32_t r[32];
          ptx::tmem_ld32(taddr + c * 32, r);
          ptx::tmem_ld_wait();
          epilogue_chunk<EPI>(p, row, col_base + c * 32, r, aux[c]);
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&tempty[as]), crank & ~1u));
      }
    }
    if constexpr (TS) {
      if (lane == 0) ptx::tma_store_wait<0>();   // shared memory must outlive the engine's reads
      __syncwarp();
    }
    if (p.stats && warp == kEpiWarp0 && lane == 0) {
      atomicAdd(&p.stats[3], static_cast<unsigned long long>(w0));
      atomicAdd(&p.stats[5], static_cast<unsigned long long>(clock64() - t_start));
    }
    if (p.stats && lane == 0) atomicMax(&p.stats[13], static_cast<unsigned long long>(globaltimer_ns()));
    if (p.stats && warp == kEpiWarp0 && lane == 0 && blockIdx.x == 0) {  // SM clock of this launch = [6] cycles / [7] ns (CTA 0)
      p.stats[6] = static_cast<unsigned long long>(clock64() - t_start);
      p.stats[7] = static_cast<unsigned long long>(globaltimer_ns() - g_start);
    }
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == kMmaWarp) ptx::tmem_dealloc_2sm(tmem_base, C::TMEM_COLS);
  if (p.stats && threadIdx.x == 0) atomicMax(&p.stats[14], static_cast<unsigned long long>(globaltimer_ns()));
}

// Persistent launch with a cluster dimension attribute.  `units` = work items (one per cluster); the grid is the number of
// clusters that can be co-resident (queried once per instantiation) or fewer.
template <bool A_MN, bool B_MN, int EPI, bool TS>
int launch2c(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmC2, const GemmParams& p,
             long long units, cudaStream_t stream) {
  auto kern = gemm2_kernel<A_MN, B_MN, EPI, TS>;
  constexpr int CL = 2;
  constexpr int kSmem = Cfg2S<EPI, TS>::SMEM_BYTES;
  static int max_clusters = 0;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // see launch_k (common.h)
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = kSmem;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (max_clusters == 0) {
    ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    cfg.gridDim = dim3(CL * (sm_count() / CL));
    int n = 0;
    ABCGPT_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    max_clusters = n > 0 ? n : 1;
  }
  const long long clusters = units < max_clusters ? units : max_clusters;
  cfg.gridDim = dim3(static_cast<unsigned>(CL * clusters));
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  ABCGPT_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmC, tmC2, p));
  return launch_status("gemm2_kernel");
}

// TMA-store epilogue for the bf16-output roles of the pair kernel (plain, GELU, GELU'): needs 16-byte aligned outputs with
// 16-byte pitches (what cuTensorMapEncodeTiled accepts) and the plain row-major output layout (no head-major KV cache);
// other outputs keep the row-per-thread st.global epilogue.
// MEASURED (cfg3 shapes, isolated): c_fc + GELU 0.155 -> 0.140 ms, dgrad + GELU' 0.171 -> 0.166 ms, plain bf16 outputs equal; the
// MMA issuer's wait for an accumulator buffer went from 23-36 % to 1 % of the GELU GEMM (tools/gemm_stats.py).  The fp32 RESID
// epilogue was tried the same way (one 4 KB SWIZZLE_128B chunk per warp) and measured SLOWER (0.082 vs 0.080 ms at K = 768): that
// kernel waits for its residual LOADS, not its stores, so it keeps the st.global path.
template <bool A_MN, bool B_MN, int EPI>
int launch2(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, long long units, cudaStream_t stream) {
  CUtensorMap tmC = {}, tmC2 = {};
  if constexpr (EPI == ABCGPT_EPI_BF16 || EPI == ABCGPT_EPI_GELU || EPI == ABCGPT_EPI_DGELU) {
    auto ok16 = [](const void* ptr, long long ld) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && ((ld * 2) & 15) == 0; };
    bool ts = p.head_stride == 0 && ok16(p.c, p.ldc);
    if (EPI == ABCGPT_EPI_GELU) ts = ts && ok16(p.c2, p.ldc2);
    if (ts) {
      int rc = encode_tmap_2d_sw(&tmC, p.c, 2, static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.ldc) * 2, 32, 32, 64);
      if (rc) return rc;
      if (EPI == ABCGPT_EPI_GELU) {
        rc = encode_tmap_2d_sw(&tmC2, p.c2, 2, static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.ldc2) * 2, 32, 32, 64);
        if (rc) return rc;
      }
      return launch2c<A_MN, B_MN, EPI, true>(tmA, tmB, tmC, tmC2, p, units, stream);
    }
  }
  if constexpr (EPI == ABCGPT_EPI_F32_RED) {
    // weight gradients: TMA tile reductions (cp.reduce.async.bulk.tensor .add) instead of per-thread red.global (see the
    // epilogue); outputs that are not 16-byte aligned keep red.global
    if ((reinterpret_cast<uintptr_t>(p.c) & 15) == 0 && ((p.ldc * 4) & 15) == 0) {
      const int rc = encode_tmap_2d_sw(&tmC, p.c, 4, static_cast<uint64_t>(p.N), static_cast<uint64_t>(p.M), static_cast<uint64_t>(p.ldc) * 4, 16, 32, 64);
      if (rc) return rc;
      return launch2c<A_MN, B_MN, EPI, true>(tmA, tmB, tmC, tmC2, p, units, stream);
    }
  }
  return launch2c<A_MN, B_MN, EPI, false>(tmA, tmB, tmC, tmC2, p, units, stream);
}

template <bool A_MN, bool B_MN>
int dispatch_epi2(int epi, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p, long long grid, cudaStream_t stream) {
  switch (epi) {
    case ABCGPT_EPI_BF16: return launch2<A_MN, B_MN, ABCGPT_EPI_BF16>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_GELU: return launch2<A_MN, B_MN, ABCGPT_EPI_GELU>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_RESID: return launch2<A_MN, B_MN, ABCGPT_EPI_RESID>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_DGELU: return launch2<A_MN, B_MN, ABCGPT_EPI_DGELU>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_F32_RED: return launch2<A_MN, B_MN, ABCGPT_EPI_F32_RED>(tmA, tmB, p, grid, stream);
    case ABCGPT_EPI_F32: return launch2<A_MN, B_MN, ABCGPT_EPI_F32>(tmA, tmB, p, grid, stream);
  }
  return fail(-1, "unknown GEMM epilogue %d", epi);
}

int dispatch_major2(int a_mn, int b_mn, int epi, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmParams& p,
                    long long grid, cudaStream_t stream) {
  if (!a_mn && !b_mn) return dispatch_epi2<false, false>(epi, tmA, tmB, p, grid, stream);
  if (!a_mn && b_mn) return dispatch_epi2<false, true>(epi, tmA, tmB, p, grid, stream);
  if (a_mn && b_mn) return dispatch_epi2<true, true>(epi, tmA, tmB, p, grid, stream);
  return fail(-1, "GEMM operand combination A=MN-major,B=K-major is not instantiated");
}

}  // namespace

int gemm_bf16(const void* a, int a_mn, long long lda, const void* b, int b_mn, long long ldb, int M, int N, int K,
              int epi, void* c, long long ldc, void* c2, long long ldc2, const void* aux, long long ldaux,
              const float* bias, int bn_hint, int splits_hint, float drop_p, uint32_t drop_key, cudaStream_t stream) {

  const int act_tanh = (epi & ABCGPT_ACT_TANH) ? 1 : 0;
  epi &= ~ABCGPT_ACT_TANH;
  ABCGPT_CHECK_ARG(!act_tanh || epi == ABCGPT_EPI_GELU || epi == ABCGPT_EPI_DGELU, "gemm: ABCGPT_ACT_TANH only modifies the GELU / DGELU epilogues");
  ABCGPT_CHECK_ARG(M > 0 && N > 0 && K > 0, "gemm: M,N,K must be positive (got %d,%d,%d)", M, N, K);
  ABCGPT_CHECK_ARG(N % 8 == 0, "gemm: N must be a multiple of 8 (pad the output; got %d)", N);
  ABCGPT_CHECK_ARG(c != nullptr, "gemm: null output");
  ABCGPT_CHECK_ARG(drop_p == 0.f || (epi == ABCGPT_EPI_RESID && drop_p > 0.f && drop_p < 1.f),
                   "gemm: dropout is fused into the RESID epilogue only (0 <= p < 1)");
  ABCGPT_CHECK_ARG(epi != ABCGPT_EPI_GELU || c2 != nullptr, "gemm: GELU epilogue needs the second output");
  ABCGPT_CHECK_ARG(epi != ABCGPT_EPI_DGELU || bias == nullptr, "gemm: the GELU' epilogue (a dgrad) takes no bias");
  ABCGPT_CHECK_ARG((epi != ABCGPT_EPI_RESID && epi != ABCGPT_EPI_DGELU) || aux != nullptr,
                   "gemm: epilogue %d needs the aux input", epi);

  // Tile choice.  bn_hint: 0 = auto, 128 / 256 = one CTA per 128 x bn tile, 512 = CTA pair per 256 x 256 tile.
  const int sms = sm_count();
  const int num_m_blk = (M + BM - 1) / BM;
  const int num_k_blk = (K + BK - 1) / BK;
  int bn = bn_hint;
  if (bn == 0) {
    // CTA pairs halve the B-operand traffic per SM (the single-CTA kernel is starved by L2->SM operand delivery);
    // they need N > 128 to be worth a 256-wide tile.
    if (N > 128) {
      bn = 512;
      // ... unless the problem is not 256-aligned: at the baby GPT's N = 384 a pair tile grid is a quarter padding (and 128 tiles on
      // 74 pairs take two full rounds), where 128 x 128 single-CTA tiles waste nothing.  Cost in units of one pair-tile main loop;
      // the single-CTA kernel pays ~15 % for its doubled operand traffic per FLOP.  MEASURED (tools/gemm_tile_sweep.py, 16384 tokens
      // x 384): mlp.c_proj + residual 35.3 -> 31.3 us, dgrad attn.c_proj 14.4 -> 13.1, wgrad c_attn 23.3 -> 21.1, wgrad c_fc 27.3 ->
      // 25.1 us; every 256-aligned shape (GPT-2-small, the hierarchical model) keeps the pair kernel.
      const long long tp = static_cast<long long>((M + 255) / 256) * ((N + 255) / 256);
      const long long t1 = static_cast<long long>((M + 127) / 128) * ((N + 127) / 128);
      if (epi == ABCGPT_EPI_F32_RED) {
        // split-K balances the rounds whatever the tile: what differs is the padded output area (tokens = K here)
        if (M >= 256 && K >= 4096 && 1.15 * static_cast<double>(t1) < 0.95 * 4.0 * static_cast<double>(tp)) bn = 128;
      } else if (M >= 4096) {
        const long long P = sms / 2, r = tp % P;
        const double rounds_pair = static_cast<double>(tp / P) + (r == 0 ? 0.0 : ((tp > P && 2 * r <= P) ? 0.5 : 1.0));
        const double rounds_128 = static_cast<double>((t1 + sms - 1) / sms) * 0.5 * 1.15;
        if (rounds_128 < 0.95 * rounds_pair) bn = 128;
      }
    } else {
      bn = 128;
    }
  }
  ABCGPT_CHECK_ARG(bn == 128 || bn == 256 || bn == 512, "gemm: unsupported tile hint %d", bn);
  const bool pair = bn == 512;
  const int tile_n = pair ? 256 : bn;
  const int num_n_blk = (N + tile_n - 1) / tile_n;
  const int num_m_units = pair ? (num_m_blk + 1) / 2 : num_m_blk;  // schedulable row blocks
  const int units = pair ? sms / 2 : sms;                           // schedulable CTAs / CTA pairs

  int splits = 1;
  if (epi == ABCGPT_EPI_F32_RED) {
    // split-K so that the persistent schedule's last wave is full: minimise rounds(s) * (k-blocks per split + a fixed
    // per-work-item cost for the reduction epilogue)
    const long long tiles = static_cast<long long>(num_m_units) * num_n_blk;
    if (splits_hint > 0) {
      splits = splits_hint;
    } else {
      long long best = -1;
      for (int sp = 1; sp <= 64 && sp <= num_k_blk; ++sp) {
        const long long rounds = (tiles * sp + units - 1) / units;
        const long long cost = rounds * ((num_k_blk + sp - 1) / sp + 6);
        if (best < 0 || cost < best) {
          best = cost;
          splits = sp;
        }
      }
    }
    if (splits > num_k_blk) splits = num_k_blk;
    if (splits < 1) splits = 1;
  }
  const int kb_per_split = (num_k_blk + splits - 1) / splits;
  splits = (num_k_blk + kb_per_split - 1) / kb_per_split;

  CUtensorMap tmA, tmB;
  int rc;
  if (!a_mn)
    rc = encode_tmap_2d(&tmA, a, 2, K, M, lda * 2, BK, BM, true);
  else
    rc = encode_tmap_2d(&tmA, a, 2, M, K, lda * 2, 64, BK, true);
  if (rc) return rc;
  if (!b_mn)
    rc = encode_tmap_2d(&tmB, b, 2, K, N, ldb * 2, BK, pair ? 128 : bn, true);
  else
    rc = encode_tmap_2d(&tmB, b, 2, N, K, ldb * 2, 64, BK, true);
  if (rc) return rc;

  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.num_m_blk = num_m_blk; p.num_n_blk = num_n_blk; p.num_k_blk = num_k_blk;
  p.splits = splits; p.kb_per_split = kb_per_split;
  p.c = c; p.ldc = ldc; p.c2 = c2; p.ldc2 = ldc2; p.aux = aux; p.ldaux = ldaux; p.bias = bias; p.act_tanh = act_tanh; p.head_stride = (epi == ABCGPT_EPI_BF16 && c2 == nullptr) ? ldc2 : 0; p.stats = g_gemm_stats; p.drop = make_drop(drop_p, drop_key);
  {
    const bool f32_out = (epi == ABCGPT_EPI_RESID || epi == ABCGPT_EPI_F32 || epi == ABCGPT_EPI_F32_RED);
    const long long cb = f32_out ? 4 : 2, ab = (epi == ABCGPT_EPI_RESID) ? 4 : 2;
    bool ok = (reinterpret_cast<uintptr_t>(c) % 32 == 0) && ((ldc * cb) % 32 == 0);
    if (c2) ok = ok && (reinterpret_cast<uintptr_t>(c2) % 32 == 0) && ((ldc2 * 2) % 32 == 0);
    if (aux) ok = ok && (reinterpret_cast<uintptr_t>(aux) % 32 == 0) && ((ldaux * ab) % 32 == 0);
    p.wide = ok ? 1 : 0;
  }

  long long total = static_cast<long long>(num_m_units) * num_n_blk * splits;
  p.half_from = 0x7fffffff;
  p.half_extra = 0;
  if (pair && splits == 1 && epi != ABCGPT_EPI_F32_RED) {
    // half tiles for a short last round of the static schedule (see gemm2_kernel)
    const long long r = total % units;
    if (total > units && r > 0 && 2 * r <= units && total + r < 0x7fffffff) {
      p.half_from = static_cast<int>(total - r);
      p.half_extra = static_cast<int>(r);
      total += r;
    }
  }
  if (pair) return dispatch_major2(a_mn, b_mn, epi, tmA, tmB, p, total, stream);
  const int grid = static_cast<int>(total < sms ? total : sms);
  if (bn == 256) return dispatch_major<256>(a_mn, b_mn, epi, tmA, tmB, p, grid, stream);
  return dispatch_major<128>(a_mn, b_mn, epi, tmA, tmB, p, grid, stream);
}

}  // namespace abcgpt
