// Shared device helpers of the attention kernels (csrc/attn.cu: one CTA per 128-row tile; csrc/attn_pair.cu: CTA pairs on
// cta_group::2 MMAs): constants, the per-chunk softmax / dS arithmetic, tile-class logic for the causal mask, packing of
// short sequences, the static persistent schedule.  Everything lives in an anonymous namespace per translation unit.
#pragma once
#include "common.h"
#include "dropout.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace abcgpt {
namespace {

constexpr int HS = 64;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kScale = 0.125f;  // 1/sqrt(64)
constexpr float kSl2 = kScale * kLog2e;
// softmax scale 1/sqrt(D) of the supported head sizes (csrc/attn_hd.cu: D = 32, 128); D = 64 gives exactly kScale / kSl2, so
// the head-size-64 kernels compile to the same code as before the head size became a template parameter
__host__ __device__ constexpr float scale_of(int D) { return D == 32 ? 0.17677669529663687f : (D == 128 ? 0.08838834764831845f : kScale); }
__host__ __device__ constexpr float sl2_of(int D) { return D == HS ? kSl2 : scale_of(D) * kLog2e; }
constexpr int kThreads = 192;  // warp 0 TMA, warp 1 MMA, warps 2..5 one thread per tile row

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// K-major SW128 operand: rows x 64 bf16 slab, 16-column K step k16
__device__ __forceinline__ uint64_t desc_k(uint32_t slab_addr, int k16) {
  return ptx::umma_smem_desc(slab_addr + k16 * 32, 0, 1024);
}
// MN-major SW128 operand over a [k rows x 64] slab (64 contiguous MN elements per row), K step of 16 rows
__device__ __forceinline__ uint64_t desc_mn(uint32_t slab_addr, int k16) {
  return ptx::umma_smem_desc(slab_addr + k16 * 2048, 8192, 1024);
}


__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float2 f2(uint32_t a, uint32_t b) { return make_float2(__uint_as_float(a), __uint_as_float(b)); }

// Per-chunk mask classes (a chunk = 32 consecutive score columns seen by one warp = 32 consecutive rows).  Row and
// column ranges are both 32-aligned, so a chunk is either entirely visible, entirely masked, or the diagonal one.
constexpr int kFull = 0, kDiag = 1, kMasked = 2;

// forward pass 1: row max of one chunk
template <int MODE>
__device__ __forceinline__ float fwd_chunk_max(uint32_t taddr, int lane) {
  if (MODE == kMasked) return -1e30f;
  uint32_t v[32];
  ptx::tmem_ld32(taddr, v);
  ptx::tmem_ld_wait();
  float m0 = -1e30f, m1 = -1e30f, m2 = -1e30f, m3 = -1e30f;
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    float a = __uint_as_float(v[i]), b = __uint_as_float(v[i + 1]), c = __uint_as_float(v[i + 2]), d = __uint_as_float(v[i + 3]);
    if (MODE == kDiag) {
      a = (i <= lane) ? a : -1e30f;
      b = (i + 1 <= lane) ? b : -1e30f;
      c = (i + 2 <= lane) ? c : -1e30f;
      d = (i + 3 <= lane) ? d : -1e30f;
    }
    m0 = fmaxf(m0, a); m1 = fmaxf(m1, b); m2 = fmaxf(m2, c); m3 = fmaxf(m3, d);
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}

// prmt.b32 with a selector whose nibbles have bit 3 set replicates the SIGN of the chosen byte: 0xBB99 turns bits 15 / 31
// into a bf16x2 AND mask, 0x9999 / 0xBBBB into fp32 masks for the even / odd column of a pair (csrc/dropout.cuh)
__device__ __forceinline__ uint32_t prmt_sign(uint32_t x, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(x), "r"(0u), "r"(sel));
  return d;
}

// backward (dQ kernel): dS = P * (dP*scale - delta*scale) for one chunk; row statistics are per thread
template <int MODE, bool DROP, int D = HS>
__device__ __forceinline__ void dq_chunk(uint32_t taddr_s, uint32_t taddr_dp, int lane, float neg_lse2, float neg_delta8,
                                         uint32_t* pk, const DropCfg& dcfg, uint32_t drop_rk, int kv0) {
  if (MODE == kMasked) {
#pragma unroll
    for (int i = 0; i < 16; ++i) pk[i] = 0u;
    return;
  }
  uint32_t s[32], dp[32];
  ptx::tmem_ld32(taddr_s, s);
  ptx::tmem_ld32(taddr_dp, dp);
  ptx::tmem_ld_wait();
  const float2 sl = make_float2(sl2_of(D), sl2_of(D)), nl = make_float2(neg_lse2, neg_lse2);
  const float scv = DROP ? scale_of(D) * dcfg.inv_keep : scale_of(D);  // dP = (dO V^T) o mask / (1-p): the factor rides on the scale
  const float2 sc = make_float2(scv, scv), nd = make_float2(neg_delta8, neg_delta8);
  const uint32_t drop_b = drop_row_key2(drop_rk);
  const uint32_t drop_s = drop_rk + (static_cast<uint32_t>(kv0) >> 1) * kDropWeyl;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float2 t = __ffma2_rn(f2(s[2 * i], s[2 * i + 1]), sl, nl);
    const float2 p = make_float2(ex2(t.x), ex2(t.y));
    float2 dpe = f2(dp[2 * i], dp[2 * i + 1]);
    if (DROP) {
      const uint32_t u = attn_drop_signs(attn_drop_fold(drop_s + static_cast<uint32_t>(i) * kDropWeyl, drop_b), dcfg.k15);
      dpe.x = __uint_as_float(dp[2 * i] & prmt_sign(u, 0x9999u));
      dpe.y = __uint_as_float(dp[2 * i + 1] & prmt_sign(u, 0xBBBBu));
    }
    const float2 u = __ffma2_rn(dpe, sc, nd);
    float2 d = __fmul2_rn(p, u);
    if (MODE == kDiag) {  // keep column <= row
      d.x = (2 * i <= lane) ? d.x : 0.f;
      d.y = (2 * i + 1 <= lane) ? d.y : 0.f;
    }
    pk[i] = ptx::pack_bf16x2(d.x, d.y);
  }
}

// backward (dK/dV kernel): P^T and dS^T for one chunk; statistics are per COLUMN (query), read from shared memory.
// MODE kDiag here is the general path: keep iff (q >= kv) && (q < T).
template <int MODE, bool DROP, int D = HS>
__device__ __forceinline__ void dkv_chunk(uint32_t taddr_s, uint32_t taddr_dp, uint32_t st_lse2, uint32_t st_delta8,
                                          int q_base, int kv_t, int T, uint32_t* pk_p, uint32_t* pk_ds, const DropCfg& dcfg,
                                          uint32_t st_rowkey, int kv_real) {
  if (MODE == kMasked) {
#pragma unroll
    for (int i = 0; i < 16; ++i) { pk_p[i] = 0u; pk_ds[i] = 0u; }
    return;
  }
  uint32_t s[32], dp[32];
  ptx::tmem_ld32(taddr_s, s);
  ptx::tmem_ld32(taddr_dp, dp);
  ptx::tmem_ld_wait();
  const float scv = DROP ? scale_of(D) * dcfg.inv_keep : scale_of(D);  // the 1/(1-p) of dP rides on the scale, that of dV on its epilogue
  const float2 sl = make_float2(sl2_of(D), sl2_of(D)), sc = make_float2(scv, scv);
  // the mask row is the QUERY (a column here), so every element needs its own hash: lane (kv & 1) of pair kv >> 1
  const uint32_t drop_off = (static_cast<uint32_t>(kv_real) >> 1) * kDropWeyl;  // kv_real: key position in its real sequence
  const uint32_t drop_sel = (kv_t & 1) ? 0xBBBBu : 0x9999u;
#pragma unroll
  for (int i4 = 0; i4 < 8; ++i4) {
    const float4 l4 = lds128(st_lse2 + 16 * i4);     // already negated: -lse*log2e   (ld.shared, broadcast)
    const float4 d4 = lds128(st_delta8 + 16 * i4);   // already negated: -delta*scale
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = 2 * i4 + h;  // pair index: columns 2i, 2i+1
      const float2 nl = h == 0 ? make_float2(l4.x, l4.y) : make_float2(l4.z, l4.w);
      const float2 nd = h == 0 ? make_float2(d4.x, d4.y) : make_float2(d4.z, d4.w);
      const float2 t = __ffma2_rn(f2(s[2 * i], s[2 * i + 1]), sl, nl);
      float2 p = make_float2(ex2(t.x), ex2(t.y));
      float2 dpe = f2(dp[2 * i], dp[2 * i + 1]);
      float2 pd = p;  // the (dropped) probabilities that multiply dO in dV
      if (DROP) {
        uint32_t rk0, rk1;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(rk0), "=r"(rk1) : "r"(st_rowkey + 8 * i));
        const uint32_t m0 = prmt_sign(attn_drop_signs(attn_drop_fold(rk0 + drop_off, drop_row_key2(rk0)), dcfg.k15), drop_sel);
        const uint32_t m1 = prmt_sign(attn_drop_signs(attn_drop_fold(rk1 + drop_off, drop_row_key2(rk1)), dcfg.k15), drop_sel);
        pd.x = __uint_as_float(__float_as_uint(p.x) & m0);
        pd.y = __uint_as_float(__float_as_uint(p.y) & m1);
        dpe.x = __uint_as_float(dp[2 * i] & m0);
        dpe.y = __uint_as_float(dp[2 * i + 1] & m1);
      }
      const float2 u = __ffma2_rn(dpe, sc, nd);
      float2 d = __fmul2_rn(p, u);
      if (MODE == kDiag) {
        const int q0 = q_base + 2 * i;
        const bool k0 = (q0 >= kv_t) && (q0 < T), k1 = (q0 + 1 >= kv_t) && (q0 + 1 < T);
        pd.x = k0 ? pd.x : 0.f; d.x = k0 ? d.x : 0.f;
        pd.y = k1 ? pd.y : 0.f; d.y = k1 ? d.y : 0.f;
      }
      pk_p[i] = ptx::pack_bf16x2(pd.x, pd.y);
      pk_ds[i] = ptx::pack_bf16x2(d.x, d.y);
    }
  }
}

constexpr float kRescaleThreshold = 64.0f;  // log2 units

// Short sequences (T = 32 or 64: the character level of the hierarchical model) are packed 128 / T to a 128-row tile: the
// kernels see B*T/128 "virtual" sequences of 128 rows and mask block-diagonally (seq_shift = log2 of the real length;
// kNoPack = not packed).  Row statistics (LSE, delta) and the dropout row counters keep the canonical [B, H, T] indexing of
// the real sequences, so packing is invisible outside the kernels.
constexpr int kNoPack = 30;
__device__ __forceinline__ long long stat_idx(int b, int h, int t, int H, int T, int seq_shift) {
  if (seq_shift >= kNoPack) return (static_cast<long long>(b) * H + h) * T + t;
  const int per = T >> seq_shift;
  return (((static_cast<long long>(b) * per + (t >> seq_shift)) * H + h) << seq_shift) + (t & ((1 << seq_shift) - 1));
}
// c0, r0: first column / row of two 32-wide blocks; both lie in the same real sequence?
__device__ __forceinline__ bool same_seq(int c0, int r0, int seq_shift) { return (c0 >> seq_shift) == (r0 >> seq_shift); }
// key position inside its real sequence (the dropout mask's column counter)
__device__ __forceinline__ int real_col(int c, int seq_shift) { return c & ((1 << seq_shift) - 1); }

// p = 2^(s*sl2 - m_ref) for one 32-column chunk, also tracks the raw row max; MODE as for the other chunk helpers
// DROP: attention dropout (SDPA dropout_p, model.py:64): the row sum uses the undropped probabilities, the P fed to P V is
// masked and scaled by 1/(1-p); mask bit = f(site key, row (b,h,q), key position), regenerated in the backward kernels.
template <int MODE, bool DROP, int D = HS>
__device__ __forceinline__ void fwd_chunk(uint32_t taddr, int lane, float neg_m, float& tmax, float& rowsum, uint32_t* pk,
                                          const DropCfg& dcfg, uint32_t drop_rk, int kv0) {
  if (MODE == kMasked) {
#pragma unroll
    for (int i = 0; i < 16; ++i) pk[i] = 0u;
    return;
  }
  uint32_t v[32];
  ptx::tmem_ld32(taddr, v);
  ptx::tmem_ld_wait();
  const float2 sl = make_float2(sl2_of(D), sl2_of(D)), nm = make_float2(neg_m, neg_m);
  float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
  float m0 = tmax, m1 = -1e30f;
  const uint32_t drop_b = drop_row_key2(drop_rk);
  const uint32_t drop_s = drop_rk + (static_cast<uint32_t>(kv0) >> 1) * kDropWeyl;
#pragma unroll
  for (int i = 0; i < 16; i += 2) {
    float s0 = __uint_as_float(v[2 * i]), s1 = __uint_as_float(v[2 * i + 1]);
    float s2 = __uint_as_float(v[2 * i + 2]), s3 = __uint_as_float(v[2 * i + 3]);
    if (MODE == kDiag) {
      s0 = (2 * i <= lane) ? s0 : -1e30f;
      s1 = (2 * i + 1 <= lane) ? s1 : -1e30f;
      s2 = (2 * i + 2 <= lane) ? s2 : -1e30f;
      s3 = (2 * i + 3 <= lane) ? s3 : -1e30f;
    }
    m0 = fmaxf(m0, fmaxf(s0, s1));
    m1 = fmaxf(m1, fmaxf(s2, s3));
    const float2 t0 = __ffma2_rn(make_float2(s0, s1), sl, nm);
    const float2 t1 = __ffma2_rn(make_float2(s2, s3), sl, nm);
    float2 p0 = make_float2(ex2(t0.x), ex2(t0.y));  // masked entries: 2^(-huge) = 0
    float2 p1 = make_float2(ex2(t1.x), ex2(t1.y));
    acc0 = __fadd2_rn(acc0, p0);
    acc1 = __fadd2_rn(acc1, p1);
    pk[i] = ptx::pack_bf16x2(p0.x, p0.y);
    pk[i + 1] = ptx::pack_bf16x2(p1.x, p1.y);
    if (DROP) {  // AND mask on the packed pair; the 1/(1-p) factor is applied to O in the item epilogue
      const uint32_t u0 = attn_drop_signs(attn_drop_fold(drop_s + static_cast<uint32_t>(i) * kDropWeyl, drop_b), dcfg.k15);
      const uint32_t u1 = attn_drop_signs(attn_drop_fold(drop_s + static_cast<uint32_t>(i + 1) * kDropWeyl, drop_b), dcfg.k15);
      pk[i] &= prmt_sign(u0, 0xBB99u);
      pk[i + 1] &= prmt_sign(u1, 0xBB99u);
    }
  }
  tmax = fmaxf(m0, m1);
  rowsum += (acc0.x + acc0.y) + (acc1.x + acc1.y);
}

template <bool DROP, int D = HS>
__device__ __forceinline__ void fwd_tile(uint32_t tm_s, int lane, int cls0, int cls1, float neg_m, float& tmax, float& rowsum,
                                         uint32_t* pk, const DropCfg& dcfg, uint32_t drop_rk, int kv_tile0, int seq_shift) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const int cls = c == 0 ? cls0 : cls1;
    const int kv0 = real_col(kv_tile0 + c * 32, seq_shift);
    if (cls == kFull) fwd_chunk<kFull, DROP, D>(tm_s + c * 32, lane, neg_m, tmax, rowsum, pk + c * 16, dcfg, drop_rk, kv0);
    else if (cls == kDiag) fwd_chunk<kDiag, DROP, D>(tm_s + c * 32, lane, neg_m, tmax, rowsum, pk + c * 16, dcfg, drop_rk, kv0);
    else fwd_chunk<kMasked, DROP, D>(tm_s + c * 32, lane, neg_m, tmax, rowsum, pk + c * 16, dcfg, drop_rk, kv0);
  }
}

// Item decode without integer division.  Every role of every persistent kernel turns an item number into (tile, batch*head)
// and (batch, head) at each item boundary; `x / d` with a run-time d compiles to a ~25-instruction dependent chain through
// I2F / MUFU.RCP (~150 cycles), and the compute warps ran four to six of them back to back on the critical path of an item's
// first step (~1000 cycles per item in the step traces).  d is fixed per launch: the host passes m = floor(2^32 / d) + 1 and
// the device takes the high word of x * m, exact for x * d < 2^32 (checked by the host: it falls back to m = 0 = plain '/').
struct FastDiv {
  uint32_t d, m;
};
__host__ inline FastDiv make_fastdiv(uint32_t d, uint64_t max_x) {
  FastDiv f;
  f.d = d;
  f.m = (d > 1 && max_x * d < (1ull << 32)) ? static_cast<uint32_t>((1ull << 32) / d) + 1u : 0u;
  return f;
}
__device__ __forceinline__ int fdiv(int x, const FastDiv& f) {
  if (f.m == 0u) return f.d == 1u ? x : x / static_cast<int>(f.d);
  return static_cast<int>(__umulhi(static_cast<uint32_t>(x), f.m));
}
__device__ __forceinline__ int fmodi(int x, const FastDiv& f) { return x - fdiv(x, f) * static_cast<int>(f.d); }
__device__ __forceinline__ void fdivmod(int x, const FastDiv& f, int& q, int& r) {
  q = fdiv(x, f);
  r = x - q * static_cast<int>(f.d);
}

// ======================================================================================================
// persistent scheduling
// ======================================================================================================
// All three tensor-core kernels are PERSISTENT: a fixed grid (one or two CTAs per SM) walks a static list of work
// items, one item = one (128-row tile, batch*head) pair.  Measured before (one CTA per item): every CTA paid ~2.3-3.6 us
// of un-overlapped prologue / epilogue plus ~1.5 us of launch gap against ~5 us of useful steps.  Now the producer,
// MMA and compute roles each run their own loop over the item list with free-running step counters, so the loads and
// score MMAs of the next item start while the current item's accumulators are still being drained.
// Items are numbered heaviest tile first (all batch*heads of the heaviest tile, then the next one, ...) and dealt to
// the CTAs in boustrophedon passes: a static schedule whose per-CTA load differs by <= 1-2 % at the cfg3 shape.
__device__ __forceinline__ int sched_item(int k, int nitems) {
  const int G = gridDim.x, c = blockIdx.x;
  const int i = k * G + ((k & 1) ? G - 1 - c : c);
  return i < nitems ? i : -1;
}


}  // namespace
}  // namespace abcgpt
