// Causal flash attention for head sizes D = 32 and 128 (csrc/attn.cu is the tuned head-size-64 family), forward, backward
// and single-token decode.  Same arithmetic, mask, dropout counters and statistics layout as attn.cu, and the same roles per
// CTA: warp 0 issues the TMA loads, warp 1 the tcgen05 MMAs (whole warp in the loop, one elected lane issues), warps 2..5 own
// one 128-row tile row per thread and do the softmax / dS arithmetic (the chunk helpers of attn_helpers.cuh with the scale of D).
// q | k | v are read straight out of the packed [B*T, 3C] buffer through TMA column offsets, out / dqkv are written in place.
//
// One CTA per (128-row tile, batch*head) item, heaviest tiles first (no persistent schedule, no CTA pairs: those are the
// head-size-64 tuning).  Inside an item the loads run through a ring, the score tiles are double-buffered in tensor memory and
// the accumulators (O, dQ, dK / dV) stay in tensor memory across the item.
//
// Operand layouts.  D = 128: a 256-byte row is two 64-column SWIZZLE_128B slabs stored one after the other (two TMA boxes),
// a K step of 16 columns selects the slab and the 32-byte offset in it; as an MN-major B operand (N = 128) the second slab is
// the next 64-wide MN atom (leading byte offset = one slab).  D = 32: 64-byte rows, SWIZZLE_64B tensor maps and descriptors.
//
// Budgets (B200: 228 KB shared memory, 512 tensor-memory columns per SM):
//   forward   tensor memory: S 2 x 64 + O D columns -> 256-column allocation, two CTAs per SM.  D = 128: Q 32 KB + a two-stage
//             K/V ring of 32 KB per stage = 96 KB per CTA; D = 32: Q 8 KB + four stages of 8 KB.
//   dQ        S | dP 2 x 128 + dQ D columns -> 512, one CTA per SM; Q, dO tiles + a K/V ring (D = 128: 3 stages, 160 KB).
//   dK / dV   S^T | dP^T 2 x 128 + dV, dK 2 x D columns -> 512 (exactly full at D = 128); K, V tiles + a Q/dO ring.
#include "attn_helpers.cuh"

namespace abcgpt {
namespace {

template <int D>
struct HdLayout {
  static_assert(D == 32 || D == 128, "attn_hd.cu: head sizes 32 and 128");
  static constexpr int SLAB_COLS = D == 32 ? 32 : 64;  // columns of one swizzled slab (= one TMA box)
  static constexpr int NSLAB = D / SLAB_COLS;
  static constexpr int ROWB = SLAB_COLS * 2;           // bytes per slab row = swizzle width
  static constexpr int T128 = 128 * D * 2;             // bytes of a 128-row tile
  static constexpr int T64 = 64 * D * 2;               // bytes of a 64-row tile
};

// K-major operand (rows = M or N, columns = the contraction over D) of a `rows`-row tile, K step kk of 16 columns
template <int D>
__device__ __forceinline__ uint64_t desc_kmaj(uint32_t tile, int rows, int kk) {
  if constexpr (D == 32) return ptx::umma_smem_desc_lt(tile + kk * 32, 16, 512, 4);   // SW64: 8-row groups 512 bytes apart
  else return desc_k(tile + (kk >> 2) * rows * 128, kk & 3);
}
// MN-major B operand over a [64 k-rows x D] tile (N = D contiguous), K step of 16 rows
template <int D>
__device__ __forceinline__ uint64_t desc_nmaj(uint32_t tile, int k16) {
  if constexpr (D == 32) return ptx::umma_smem_desc_lt(tile + k16 * 1024, 512, 512, 4);
  else return desc_mn(tile, k16);   // leading byte offset 8192 = the second 64-column slab of the 64-row tile
}

// TMA loads of one tile: NSLAB boxes of [rows x SLAB_COLS] at global column `col`
template <int D>
__device__ __forceinline__ void load_tile(uint8_t* dst, const CUtensorMap* tm, uint64_t* bar, int col, int row, int rows) {
  using L = HdLayout<D>;
#pragma unroll
  for (int s = 0; s < L::NSLAB; ++s) ptx::tma_load_2d(dst + s * rows * L::ROWB, tm, bar, col + s * L::SLAB_COLS, row);
}

__device__ __forceinline__ uint8_t* align1024(uint8_t* p) {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~static_cast<uintptr_t>(1023));
}

// 32 fp32 accumulator columns of one row -> 32 bf16 at o (times `mul`)
__device__ __forceinline__ void store_row32(__nv_bfloat16* o, const uint32_t (&v)[32], float mul) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint4 w;
    w.x = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 0]) * mul, __uint_as_float(v[8 * q + 1]) * mul);
    w.y = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 2]) * mul, __uint_as_float(v[8 * q + 3]) * mul);
    w.z = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 4]) * mul, __uint_as_float(v[8 * q + 5]) * mul);
    w.w = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 6]) * mul, __uint_as_float(v[8 * q + 7]) * mul);
    reinterpret_cast<uint4*>(o)[q] = w;
  }
}

// ======================================================================================================
// forward
// ======================================================================================================
template <int D>
struct FwdHdSmem {
  using L = HdLayout<D>;
  static constexpr int RING = D == 128 ? 2 : 4;
  static constexpr int Q = 0;
  static constexpr int KV = L::T128;                 // RING stages x (K 64 x D | V 64 x D)
  static constexpr int STAGE = 2 * L::T64;
  static constexpr int BAR = KV + RING * STAGE;
  static constexpr int TOTAL = BAR + 256 + 1024;
};

template <int D, bool DROP>
__global__ void __launch_bounds__(kThreads, 2)
attn_fwd_hd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                   __nv_bfloat16* __restrict__ out, float* __restrict__ lse, int T, int H, int C, const DropCfg dcfg) {
  using L = HdLayout<D>;
  using S = FwdHdSmem<D>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::BAR);
  uint64_t* q_full = bars;                  // [1]
  uint64_t* kv_full = bars + 1;             // [RING]
  uint64_t* kv_empty = kv_full + S::RING;   // [RING]
  uint64_t* s_full = kv_empty + S::RING;    // [2]
  uint64_t* p_full = s_full + 2;            // [2]
  uint64_t* p_empty = p_full + 2;           // [2]
  uint64_t* o_full = p_empty + 2;           // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 1);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nqt = (T + 127) / 128;
  const int bh = blockIdx.x, qt = nqt - 1 - static_cast<int>(blockIdx.y);   // heaviest query tiles first
  const int b = bh / H, h = bh % H;
  const int num_kv = (min(T, qt * 128 + 128) + 63) / 64;   // 64-row K/V tiles up to the diagonal

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ);
    ptx::prefetch_tmap(&tmKV);
    ptx::mbar_init(q_full, 1);
    ptx::mbar_init(o_full, 1);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&p_full[s], 128);
      ptx::mbar_init(&p_empty[s], 1);
    }
    for (int s = 0; s < S::RING; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], 1);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 256);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);   // S buffers at columns [0, 64) and [64, 128); O at [128, 128 + D)
  const uint32_t tm_O = tmem_base + 128;
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();

  if (warp == 0) {
    const bool issue = ptx::elect_one();
    if (issue) {
      ptx::mbar_expect_tx(q_full, L::T128);
      load_tile<D>(smem + S::Q, &tmQ, q_full, h * D, b * T + qt * 128, 128);
    }
    for (int j = 0; j < num_kv; ++j) {
      const int st = j % S::RING;
      ptx::mbar_wait(&kv_empty[st], ((j / S::RING) & 1) ^ 1, 40);
      uint8_t* dst = smem + S::KV + st * S::STAGE;
      if (issue) {
        ptx::mbar_expect_tx(&kv_full[st], S::STAGE);
        load_tile<D>(dst, &tmKV, &kv_full[st], C + h * D, b * T + j * 64, 64);
        load_tile<D>(dst + L::T64, &tmKV, &kv_full[st], 2 * C + h * D, b * T + j * 64, 64);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    const bool leader = ptx::elect_one();
    constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t idesc_o = ptx::umma_idesc_bf16(128, D, 0, 1);
    const uint32_t sQ = ptx::smem_u32(smem + S::Q), sKV = ptx::smem_u32(smem + S::KV);
    // S_{j+1} = Q K_{j+1}^T is issued before O += P_j V_j, so the tensor core computes the next scores while the softmax
    // threads work on this tile; the tensor pipe runs in issue order, so S_{j+2} cannot overwrite P_j before P_j V_j read it
    auto issue_s = [&](int j) {
      const int st = j % S::RING;
      ptx::mbar_wait(&kv_full[st], (j / S::RING) & 1, 41);
      ptx::tc_fence_after();
      const uint32_t sK = sKV + st * S::STAGE;
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        if (leader) ptx::umma_ss(tmem_base + (j & 1) * 64, desc_kmaj<D>(sQ, 128, kk), desc_kmaj<D>(sK, 64, kk), idesc_s, kk > 0);
      if (leader) ptx::umma_commit(&s_full[j & 1]);
    };
    ptx::mbar_wait(q_full, 0, 42);
    issue_s(0);
    for (int j = 0; j < num_kv; ++j) {
      if (j + 1 < num_kv) issue_s(j + 1);
      ptx::mbar_wait(&p_full[j & 1], (j >> 1) & 1, 43);
      ptx::tc_fence_after();
      const int st = j % S::RING;
      const uint32_t sV = sKV + st * S::STAGE + L::T64;
      const uint32_t tP = tmem_base + (j & 1) * 64;   // bf16 P (32 packed columns) written over the consumed S tile
#pragma unroll
      for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ts(tm_O, tP + 8 * k, desc_nmaj<D>(sV, k), idesc_o, (j > 0 || k > 0));
      if (leader) ptx::umma_commit(&kv_empty[st]);
      if (leader) ptx::umma_commit(&p_empty[j & 1]);
    }
    if (leader) ptx::umma_commit(o_full);
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;                                    // row inside the tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const int r0 = qt * 128 + quarter * 32;                               // first query row of this warp
    const uint32_t drop_rk = DROP ? drop_row_key(dcfg.key, static_cast<uint32_t>((static_cast<long long>(bh) * T) + qt * 128 + r)) : 0u;
    float m_ref = 0.f, l = 0.f;
    bool have_ref = false;
    for (int j = 0; j < num_kv; ++j) {
      const int bsel = j & 1;
      const uint32_t tm_s = tmem_base + lane_off + bsel * 64;
      const int c0 = j * 64, c1 = j * 64 + 32;
      const int cls0 = (c0 + 31 <= r0) ? kFull : ((c0 > r0 + 31) ? kMasked : kDiag);
      const int cls1 = (c1 + 31 <= r0) ? kFull : ((c1 > r0 + 31) ? kMasked : kDiag);
      ptx::mbar_wait(&s_full[bsel], (j >> 1) & 1, 44);
      ptx::tc_fence_after();
      uint32_t pk[32];
      float tmax = -1e30f, rowsum = 0.f;
      if (!have_ref && (cls0 != kMasked || cls1 != kMasked)) {
        // first visible tile: the reference exponent is its true row max (see attn.cu: lazy in-TMEM rescale)
        have_ref = true;
        const float mx0 = cls0 == kFull ? fwd_chunk_max<kFull>(tm_s, lane) : (cls0 == kDiag ? fwd_chunk_max<kDiag>(tm_s, lane) : -1e30f);
        const float mx1 = cls1 == kFull ? fwd_chunk_max<kFull>(tm_s + 32, lane) : (cls1 == kDiag ? fwd_chunk_max<kDiag>(tm_s + 32, lane) : -1e30f);
        tmax = fmaxf(mx0, mx1);
        m_ref = tmax * sl2_of(D);
        fwd_tile<DROP, D>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, kNoPack);
      } else {
        fwd_tile<DROP, D>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, kNoPack);
        const bool need = tmax * sl2_of(D) - m_ref > kRescaleThreshold;
        if (__any_sync(0xffffffffu, need)) {
          // rare: raise the reference, rescale the O accumulator in TMEM, recompute this tile's P
          const float m_new = need ? tmax * sl2_of(D) : m_ref;
          const float alpha = ex2(m_ref - m_new);
          ptx::mbar_wait(&p_empty[(j - 1) & 1], ((j - 1) >> 1) & 1, 45);  // every earlier P V product has landed in O
          ptx::tc_fence_after();
#pragma unroll
          for (int c = 0; c < D / 32; ++c) {
            uint32_t o[32];
            ptx::tmem_ld32(tm_O + lane_off + c * 32, o);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            ptx::tmem_st32(tm_O + lane_off + c * 32, o);
          }
          ptx::tmem_st_wait();
          l *= alpha;
          m_ref = m_new;
          tmax = -1e30f;
          rowsum = 0.f;
          fwd_tile<DROP, D>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, kNoPack);
        }
      }
      l += rowsum;
      ptx::tmem_st16(tm_s, pk);
      ptx::tmem_st16(tm_s + 16, pk + 16);
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&p_full[bsel]);
    }
    // epilogue: O / l -> bf16, LSE
    ptx::mbar_wait(o_full, 0, 46);
    ptx::tc_fence_after();
    const int t = qt * 128 + r;
    const float inv = (DROP ? dcfg.inv_keep : 1.0f) / l;
    __nv_bfloat16* o = out + static_cast<long long>(b * T + t) * C + h * D;
#pragma unroll
    for (int c = 0; c < D / 32; ++c) {
      uint32_t v[32];
      ptx::tmem_ld32(tm_O + lane_off + c * 32, v);
      ptx::tmem_ld_wait();
      if (t < T) store_row32(o + c * 32, v, inv);
    }
    if (t < T) lse[static_cast<long long>(bh) * T + t] = (m_ref + log2f(l)) * kLn2;
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 256);
}

// ======================================================================================================
// backward: delta = rowsum(dO * O) per (token, head)
// ======================================================================================================
// one warp per token row, a lane reads 16-byte units (8 columns): D / 8 lanes cover one head (4 at D = 32, 16 at D = 128)
template <int D>
__global__ void __launch_bounds__(256)
attn_delta_hd_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout, float* __restrict__ delta,
                     int B, int T, int H, int C) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  constexpr int LPH = D / 8;   // lanes per head
  const int lane = threadIdx.x & 31;
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= static_cast<long long>(B) * T) return;
  const int b = static_cast<int>(row / T), t = static_cast<int>(row % T);
  const uint4* orow = reinterpret_cast<const uint4*>(o + row * C);
  const uint4* drow = reinterpret_cast<const uint4*>(dout + row * C);
  const int units = C / 8;   // H * LPH, a multiple of 4
  for (int u = lane; u < ((units + 31) & ~31); u += 32) {
    float s = 0.f;
    if (u < units) {
      const uint4 a = __ldg(orow + u), d = __ldg(drow + u);
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) s += ptx::bf16lo(aw[e]) * ptx::bf16lo(dw[e]) + ptx::bf16hi(aw[e]) * ptx::bf16hi(dw[e]);
    }
#pragma unroll
    for (int off = LPH / 2; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if ((lane & (LPH - 1)) == 0 && u < units) delta[(static_cast<long long>(b) * H + u / LPH) * T + t] = s;
  }
}

// ======================================================================================================
// backward: dQ   (item = 128 query rows; K/V in 64-row tiles:  S, dP -> dS -> dQ += dS K, accumulated in TMEM)
// ======================================================================================================
template <int D>
struct DqHdSmem {
  using L = HdLayout<D>;
  static constexpr int RING = D == 128 ? 3 : 4;
  static constexpr int Q = 0;
  static constexpr int DO = L::T128;
  static constexpr int KV = 2 * L::T128;            // RING stages x (K 64 x D | V 64 x D)
  static constexpr int STAGE = 2 * L::T64;
  static constexpr int BAR = KV + RING * STAGE;
  static constexpr int TOTAL = BAR + 256 + 1024;
};

template <int D, bool DROP>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dq_hd_kernel(const __grid_constant__ CUtensorMap tmQKV128, const __grid_constant__ CUtensorMap tmQKV64,
                      const __grid_constant__ CUtensorMap tmDO128, const float* __restrict__ lse, const float* __restrict__ delta,
                      __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, const DropCfg dcfg) {
  using L = HdLayout<D>;
  using S = DqHdSmem<D>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::BAR);
  uint64_t* qdo_full = bars;                 // [1]
  uint64_t* kv_full = bars + 1;              // [RING]
  uint64_t* kv_empty = kv_full + S::RING;    // [RING]
  uint64_t* s_full = kv_empty + S::RING;     // [2]
  uint64_t* ds_full = s_full + 2;            // [2]
  uint64_t* acc_full = ds_full + 2;          // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nqt = (T + 127) / 128;
  const int bh = blockIdx.x, qt = nqt - 1 - static_cast<int>(blockIdx.y);
  const int b = bh / H, h = bh % H;
  const int num_kv = (min(T, qt * 128 + 128) + 63) / 64;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQKV128);
    ptx::prefetch_tmap(&tmQKV64);
    ptx::prefetch_tmap(&tmDO128);
    ptx::mbar_init(qdo_full, 1);
    ptx::mbar_init(acc_full, 1);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&ds_full[s], 128);
    }
    for (int s = 0; s < S::RING; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], 1);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);   // score buffer s: S at 128 s, dP at 128 s + 64; dQ at [256, 256 + D)
  const uint32_t tm_dQ = tmem_base + 256;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();

  if (warp == 0) {
    const bool issue = ptx::elect_one();
    if (issue) {
      const int row0 = b * T + qt * 128;
      ptx::mbar_expect_tx(qdo_full, 2 * L::T128);
      load_tile<D>(smem + S::Q, &tmQKV128, qdo_full, h * D, row0, 128);
      load_tile<D>(smem + S::DO, &tmDO128, qdo_full, h * D, row0, 128);
    }
    for (int j = 0; j < num_kv; ++j) {
      const int st = j % S::RING;
      ptx::mbar_wait(&kv_empty[st], ((j / S::RING) & 1) ^ 1, 50);
      uint8_t* dst = smem + S::KV + st * S::STAGE;
      if (issue) {
        ptx::mbar_expect_tx(&kv_full[st], S::STAGE);
        load_tile<D>(dst, &tmQKV64, &kv_full[st], C + h * D, b * T + j * 64, 64);
        load_tile<D>(dst + L::T64, &tmQKV64, &kv_full[st], 2 * C + h * D, b * T + j * 64, 64);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    const bool leader = ptx::elect_one();
    constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t idesc_dq = ptx::umma_idesc_bf16(128, D, 0, 1);
    const uint32_t sQ = ptx::smem_u32(smem + S::Q), sDO = ptx::smem_u32(smem + S::DO), sKV = ptx::smem_u32(smem + S::KV);
    // S_j = Q K_j^T and dP_j = dO V_j^T into score buffer j & 1; issued one tile ahead of dQ += dS_{j} K_j
    auto issue_s = [&](int j) {
      const int st = j % S::RING;
      ptx::mbar_wait(&kv_full[st], (j / S::RING) & 1, 51);
      ptx::tc_fence_after();
      const uint32_t sK = sKV + st * S::STAGE, sV = sK + L::T64;
      const uint32_t tS = tmem_base + (j & 1) * 128;
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        if (leader) ptx::umma_ss(tS, desc_kmaj<D>(sQ, 128, kk), desc_kmaj<D>(sK, 64, kk), idesc_s, kk > 0);
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        if (leader) ptx::umma_ss(tS + 64, desc_kmaj<D>(sDO, 128, kk), desc_kmaj<D>(sV, 64, kk), idesc_s, kk > 0);
      if (leader) ptx::umma_commit(&s_full[j & 1]);
    };
    ptx::mbar_wait(qdo_full, 0, 52);
    issue_s(0);
    for (int j = 0; j < num_kv; ++j) {
      if (j + 1 < num_kv) issue_s(j + 1);
      ptx::mbar_wait(&ds_full[j & 1], (j >> 1) & 1, 53);
      ptx::tc_fence_after();
      const int st = j % S::RING;
      const uint32_t sK = sKV + st * S::STAGE;
      const uint32_t tA = tmem_base + (j & 1) * 128;   // dS (bf16 pairs, 32 columns) over the consumed scores
#pragma unroll
      for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ts(tm_dQ, tA + 8 * k, desc_nmaj<D>(sK, k), idesc_dq, (j > 0 || k > 0));
      if (leader) ptx::umma_commit(&kv_empty[st]);
    }
    if (leader) ptx::umma_commit(acc_full);
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const int r0 = qt * 128 + quarter * 32;
    const int t = qt * 128 + r;
    const long long sidx = static_cast<long long>(bh) * T + t;
    const float neg_l = t < T ? -__ldg(lse + sidx) * kLog2e : 0.f;
    const float neg_d = t < T ? -__ldg(delta + sidx) * scale_of(D) : 0.f;
    const uint32_t drop_rk = DROP ? drop_row_key(dcfg.key, static_cast<uint32_t>(sidx)) : 0u;
    for (int j = 0; j < num_kv; ++j) {
      ptx::mbar_wait(&s_full[j & 1], (j >> 1) & 1, 54);
      ptx::tc_fence_after();
      const uint32_t tbuf = tmem_base + lane_off + (j & 1) * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = j * 64 + c * 32;
        const uint32_t ta_s = tbuf + c * 32, ta_dp = ta_s + 64;
        uint32_t pk[16];
        if (c0 > r0 + 31) dq_chunk<kMasked, DROP, D>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, c0);
        else if (c0 + 31 <= r0) dq_chunk<kFull, DROP, D>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, c0);
        else dq_chunk<kDiag, DROP, D>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, c0);
        ptx::tmem_st16(tbuf + c * 16, pk);   // dS chunk c over score columns this thread has consumed
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&ds_full[j & 1]);
    }
    ptx::mbar_wait(acc_full, 0, 55);
    ptx::tc_fence_after();
    __nv_bfloat16* o = dqkv + static_cast<long long>(b * T + t) * (3 * C) + h * D;
#pragma unroll
    for (int c = 0; c < D / 32; ++c) {
      uint32_t v[32];
      ptx::tmem_ld32(tm_dQ + lane_off + c * 32, v);
      ptx::tmem_ld_wait();
      if (t < T) store_row32(o + c * 32, v, 1.f);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 512);
}

// ======================================================================================================
// backward: dK / dV   (item = 128 key rows; Q/dO in 64-row tiles from the diagonal on:  S^T, dP^T -> P^T, dS^T ->
//                      dV += P^T dO, dK += dS^T Q, accumulated in TMEM)
// ======================================================================================================
template <int D>
struct DkvHdSmem {
  using L = HdLayout<D>;
  static constexpr int RING = D == 128 ? 3 : 4;
  static constexpr int K = 0;
  static constexpr int V = L::T128;
  static constexpr int QDO = 2 * L::T128;           // RING stages x (Q 64 x D | dO 64 x D)
  static constexpr int STAGE = 2 * L::T64;
  static constexpr int STAT = QDO + RING * STAGE;   // 2 step parities x (-lse2[64] | -delta8[64] | dropout row key[64])
  static constexpr int BAR = STAT + 1536;
  static constexpr int TOTAL = BAR + 256 + 1024;
};

template <int D, bool DROP>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dkv_hd_kernel(const __grid_constant__ CUtensorMap tmQKV128, const __grid_constant__ CUtensorMap tmQKV64,
                       const __grid_constant__ CUtensorMap tmDO64, const float* __restrict__ lse, const float* __restrict__ delta,
                       __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, const DropCfg dcfg) {
  using L = HdLayout<D>;
  using S = DkvHdSmem<D>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align1024(smem_raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::BAR);
  uint64_t* kv_full = bars;                   // [1]
  uint64_t* qdo_full = bars + 1;              // [RING]
  uint64_t* qdo_empty = qdo_full + S::RING;   // [RING]
  uint64_t* s_full = qdo_empty + S::RING;     // [2]
  uint64_t* pds_full = s_full + 2;            // [2]
  uint64_t* acc_full = pds_full + 2;          // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  float* stat = reinterpret_cast<float*>(smem + S::STAT);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nkt = (T + 127) / 128, nq64 = (T + 63) / 64;
  const int bh = blockIdx.x, kt = static_cast<int>(blockIdx.y);   // key tile 0 sees every query tile: heaviest first
  (void)nkt;
  const int b = bh / H, h = bh % H;
  const int i0 = kt * 2, nsteps = nq64 - i0;   // 64-row query tiles from the diagonal on

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQKV128);
    ptx::prefetch_tmap(&tmQKV64);
    ptx::prefetch_tmap(&tmDO64);
    ptx::mbar_init(kv_full, 1);
    ptx::mbar_init(acc_full, 1);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&pds_full[s], 128);
    }
    for (int s = 0; s < S::RING; ++s) {
      ptx::mbar_init(&qdo_full[s], 1);
      ptx::mbar_init(&qdo_empty[s], 1);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);   // score buffer s: S^T at 128 s, dP^T at 128 s + 64; dV at 256, dK at 256 + D
  const uint32_t tm_dV = tmem_base + 256, tm_dK = tm_dV + D;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();

  if (warp == 0) {
    const bool issue = ptx::elect_one();
    if (issue) {
      ptx::mbar_expect_tx(kv_full, 2 * L::T128);
      load_tile<D>(smem + S::K, &tmQKV128, kv_full, C + h * D, b * T + kt * 128, 128);
      load_tile<D>(smem + S::V, &tmQKV128, kv_full, 2 * C + h * D, b * T + kt * 128, 128);
    }
    for (int n = 0; n < nsteps; ++n) {
      const int st = n % S::RING;
      ptx::mbar_wait(&qdo_empty[st], ((n / S::RING) & 1) ^ 1, 60);
      uint8_t* dst = smem + S::QDO + st * S::STAGE;
      if (issue) {
        ptx::mbar_expect_tx(&qdo_full[st], S::STAGE);
        load_tile<D>(dst, &tmQKV64, &qdo_full[st], h * D, b * T + (i0 + n) * 64, 64);
        load_tile<D>(dst + L::T64, &tmDO64, &qdo_full[st], h * D, b * T + (i0 + n) * 64, 64);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    const bool leader = ptx::elect_one();
    constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t idesc_g = ptx::umma_idesc_bf16(128, D, 0, 1);
    const uint32_t sK = ptx::smem_u32(smem + S::K), sV = ptx::smem_u32(smem + S::V), sQDO = ptx::smem_u32(smem + S::QDO);
    auto issue_s = [&](int n) {
      const int st = n % S::RING;
      ptx::mbar_wait(&qdo_full[st], (n / S::RING) & 1, 61);
      ptx::tc_fence_after();
      const uint32_t sQ = sQDO + st * S::STAGE, sDO = sQ + L::T64;
      const uint32_t tS = tmem_base + (n & 1) * 128;
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        if (leader) ptx::umma_ss(tS, desc_kmaj<D>(sK, 128, kk), desc_kmaj<D>(sQ, 64, kk), idesc_s, kk > 0);
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        if (leader) ptx::umma_ss(tS + 64, desc_kmaj<D>(sV, 128, kk), desc_kmaj<D>(sDO, 64, kk), idesc_s, kk > 0);
      if (leader) ptx::umma_commit(&s_full[n & 1]);
    };
    ptx::mbar_wait(kv_full, 0, 62);
    issue_s(0);
    for (int n = 0; n < nsteps; ++n) {
      if (n + 1 < nsteps) issue_s(n + 1);
      ptx::mbar_wait(&pds_full[n & 1], (n >> 1) & 1, 63);
      ptx::tc_fence_after();
      const int st = n % S::RING;
      const uint32_t sQ = sQDO + st * S::STAGE, sDO = sQ + L::T64;
      const uint32_t tP = tmem_base + (n & 1) * 128, tDS = tP + 64;   // bf16 pairs written over the consumed scores
#pragma unroll
      for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ts(tm_dV, tP + 8 * k, desc_nmaj<D>(sDO, k), idesc_g, (n > 0 || k > 0));
#pragma unroll
      for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ts(tm_dK, tDS + 8 * k, desc_nmaj<D>(sQ, k), idesc_g, (n > 0 || k > 0));
      if (leader) ptx::umma_commit(&qdo_empty[st]);
    }
    if (leader) ptx::umma_commit(acc_full);
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const int tid = (warp - 2) * 32 + lane;   // 0..127
    const int r = quarter * 32 + lane;        // key row inside the tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const int kv_t = kt * 128 + r, r0 = kt * 128 + quarter * 32;
    const float* stat_src = (tid < 64 ? lse : delta) + static_cast<long long>(bh) * T;
    const float stat_coef = tid < 64 ? -kLog2e : -scale_of(D);
    for (int n = 0; n < nsteps; ++n) {
      const int q0 = (i0 + n) * 64;
      // column (query) statistics of this step into shared memory: two buffers by step parity; a buffer is rewritten two steps
      // later, after a barrier that follows every read of it
      float* st = stat + (n & 1) * 192;
      const int qi = q0 + (tid & 63);
      st[tid] = qi < T ? __ldg(stat_src + qi) * stat_coef : 0.f;
      if (DROP && tid < 64) st[128 + tid] = __uint_as_float(drop_row_key(dcfg.key, static_cast<uint32_t>(static_cast<long long>(bh) * T + qi)));
      ptx::bar_sync(1, 128);
      ptx::mbar_wait(&s_full[n & 1], (n >> 1) & 1, 64);
      ptx::tc_fence_after();
      const uint32_t tbuf = tmem_base + lane_off + (n & 1) * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = q0 + c * 32;
        const uint32_t ta_s = tbuf + c * 32, ta_dp = ta_s + 64;
        const uint32_t l2 = ptx::smem_u32(st) + c * 128, d8 = l2 + 256, rkeys = l2 + 512;
        uint32_t pk_p[16], pk_ds[16];
        if (c0 + 31 < r0 || c0 >= T) dkv_chunk<kMasked, DROP, D>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kv_t);
        else if (c0 > r0 && c0 + 31 < T) dkv_chunk<kFull, DROP, D>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kv_t);
        else dkv_chunk<kDiag, DROP, D>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kv_t);
        // P^T / dS^T chunk c (32 query columns = 16 packed words each) over score columns already consumed
        ptx::tmem_st16(tbuf + c * 16, pk_p);
        ptx::tmem_st16(tbuf + 64 + c * 16, pk_ds);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&pds_full[n & 1]);
    }
    ptx::mbar_wait(acc_full, 0, 65);
    ptx::tc_fence_after();
    __nv_bfloat16* orow = dqkv + static_cast<long long>(b * T + kv_t) * (3 * C) + h * D;
#pragma unroll
    for (int c = 0; c < D / 32; ++c) {
      uint32_t v[32];
      ptx::tmem_ld32(tm_dV + lane_off + c * 32, v);   // dV = (P o mask)^T dO / (1-p)
      ptx::tmem_ld_wait();
      if (kv_t < T) store_row32(orow + 2 * C + c * 32, v, DROP ? dcfg.inv_keep : 1.f);
      ptx::tmem_ld32(tm_dK + lane_off + c * 32, v);
      ptx::tmem_ld_wait();
      if (kv_t < T) store_row32(orow + C + c * 32, v, 1.f);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 512);
}

// ======================================================================================================
// single-token decode: append k, v of position t to the head-major cache, attend over cache rows [0, t]
// ======================================================================================================
__device__ __forceinline__ uint4 ld_v4(const void* p) {   // plain (coherent) load: the block itself wrote row t of the cache
  uint4 v;
  asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint2 ld_v2(const void* p) {
  uint2 v;
  asm volatile("ld.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ld_u32(const void* p) {
  uint32_t v;
  asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// One block of 128 threads per (batch, head); HBM-bound (K and V of the sequence are read once).  qkv_row: bf16 [B, 3C], the
// c_attn output of position t; cache: bf16 [B, 2H, Tmax, D] (k heads | v heads), so the rows of one (b, h) are contiguous.
template <int D>
__global__ void __launch_bounds__(128)
attn_decode_hd_kernel(const __nv_bfloat16* __restrict__ qkv_row, __nv_bfloat16* cache, __nv_bfloat16* __restrict__ out, int Tmax,
                      int t, int H) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  extern __shared__ float prob[];   // [t + 1]
  __shared__ float q[D];
  __shared__ float red[4];
  __shared__ float part[4][D];
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = H * D, n_keys = t + 1;
  const long long head = static_cast<long long>(Tmax) * D;
  __nv_bfloat16* kc = cache + (static_cast<long long>(b) * 2 * H + h) * head;
  __nv_bfloat16* vc = kc + H * head;
  const __nv_bfloat16* row = qkv_row + static_cast<long long>(b) * 3 * C + h * D;
  if (tid < D / 8) reinterpret_cast<uint4*>(kc + static_cast<long long>(t) * D)[tid] = reinterpret_cast<const uint4*>(row + C)[tid];
  else if (tid < D / 4) reinterpret_cast<uint4*>(vc + static_cast<long long>(t) * D)[tid - D / 8] = reinterpret_cast<const uint4*>(row + 2 * C)[tid - D / 8];
  if (tid < D) q[tid] = __bfloat162float(row[tid]) * scale_of(D);
  __syncthreads();
  float mx = -INFINITY;
  {
    // scores: D / 8 lanes share a key (16 bytes each), whole rows per group of lanes, U loads in flight per lane
    constexpr int LPK = D / 8, KPI = 32 / LPK, U = D == 128 ? 8 : 4;
    const int sub = lane % LPK, grp = lane / LPK;
    float qr[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) qr[e] = q[sub * 8 + e];
    const __nv_bfloat16* kb = kc + sub * 8;
    for (int k0 = warp * KPI * U; k0 < n_keys; k0 += 4 * KPI * U) {
      uint4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int k = k0 + u * KPI + grp;
        v[u] = k < n_keys ? ld_v4(kb + static_cast<long long>(k) * D) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
        float sc = 0.f;
#pragma unroll
        for (int e = 0; e < 4; ++e) sc += qr[2 * e] * ptx::bf16lo(w[e]) + qr[2 * e + 1] * ptx::bf16hi(w[e]);
#pragma unroll
        for (int off = 1; off < LPK; off <<= 1) sc += __shfl_xor_sync(0xffffffffu, sc, off);
        const int k = k0 + u * KPI + grp;
        if (k < n_keys) {
          if (sub == 0) prob[k] = sc;
          mx = fmaxf(mx, sc);
        }
      }
    }
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  __syncthreads();
  float sum = 0.f;
  for (int k = tid; k < n_keys; k += 128) {
    const float e = __expf(prob[k] - mx);
    prob[k] = e;
    sum += e;
  }
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  const float inv = 1.0f / ((red[0] + red[1]) + (red[2] + red[3]));
  // out[d] = sum_k p_k V[k][d] with P rounded to bf16 like the flash kernels.  A row is D / 2 words: LPR lanes read WPL
  // adjacent words each, RPI rows per warp instruction, eight rows in flight per lane
  constexpr int LPR = D / 2 < 32 ? D / 2 : 32, WPL = D / 2 / LPR, RPI = 32 / LPR, STEP = 4 * RPI;
  const int cw = lane % LPR, rsub = lane / LPR;
  const uint32_t* vb = reinterpret_cast<const uint32_t*>(vc) + cw * WPL;
  float acc[2 * WPL];
#pragma unroll
  for (int i = 0; i < 2 * WPL; ++i) acc[i] = 0.f;
  auto fma_row = [&](const uint32_t* w, float p) {
#pragma unroll
    for (int i = 0; i < WPL; ++i) {
      acc[2 * i] += p * ptx::bf16lo(w[i]);
      acc[2 * i + 1] += p * ptx::bf16hi(w[i]);
    }
  };
  auto load_row = [&](int k, uint32_t* w) {
    const uint32_t* p = vb + static_cast<long long>(k) * (D / 2);
    if constexpr (WPL == 2) {
      const uint2 x = ld_v2(p);
      w[0] = x.x;
      w[1] = x.y;
    } else {
      w[0] = ld_u32(p);
    }
  };
  int k = warp * RPI + rsub;
  for (; k + 7 * STEP < n_keys; k += 8 * STEP) {
    uint32_t w[8][WPL];
#pragma unroll
    for (int u = 0; u < 8; ++u) load_row(k + u * STEP, w[u]);
#pragma unroll
    for (int u = 0; u < 8; ++u) fma_row(w[u], ptx::bf16_round(prob[k + u * STEP] * inv));
  }
  for (; k < n_keys; k += STEP) {
    uint32_t w[WPL];
    load_row(k, w);
    fma_row(w, ptx::bf16_round(prob[k] * inv));
  }
#pragma unroll
  for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
    for (int i = 0; i < 2 * WPL; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], off);
  if (rsub == 0) {
#pragma unroll
    for (int i = 0; i < 2 * WPL; ++i) part[warp][cw * 2 * WPL + i] = acc[i];
  }
  __syncthreads();
  if (tid < D) {
    const float o = (part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid]);
    out[static_cast<long long>(b) * C + h * D + tid] = __float2bfloat16_rn(o);
  }
}

// ======================================================================================================
// host side
// ======================================================================================================
template <typename K>
int prepare(K kern, int bytes) {
  ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return 0;
}

int check_hd(const char* who, int B, int T, int H, int D) {
  ABCGPT_CHECK_ARG(D == 32 || D == 128, "%s: head size %d is not supported (supported head sizes: 32, 64, 128)", who, D);
  ABCGPT_CHECK_ARG(B > 0 && T > 0 && H > 0, "%s: bad shape B=%d T=%d H=%d", who, B, T, H);
  ABCGPT_CHECK_ARG(static_cast<long long>(B) * H < (1ll << 31) - 1, "%s: too many batch*head items", who);
  ABCGPT_CHECK_ARG((T + 127) / 128 <= 65535, "%s: sequence too long", who);
  return 0;
}

// [rows x 3C] or [rows x C] bf16 operand, boxes of [box_rows x SLAB_COLS] with the swizzle of D
template <int D>
int tmap_hd(CUtensorMap* tm, const void* p, uint64_t cols, uint64_t rows, int box_rows) {
  using L = HdLayout<D>;
  return encode_tmap_2d_sw(tm, p, 2, cols, rows, cols * 2, L::SLAB_COLS, box_rows, L::ROWB);
}

template <int D>
int fwd_hd(const void* qkv, void* out, float* lse, int B, int T, int H, const DropCfg& dcfg, cudaStream_t stream) {
  using S = FwdHdSmem<D>;
  const int C = H * D;
  const uint64_t rows = static_cast<uint64_t>(B) * T;
  CUtensorMap tmQ, tmKV;
  int rc;
  if ((rc = tmap_hd<D>(&tmQ, qkv, 3ull * C, rows, 128))) return rc;
  if ((rc = tmap_hd<D>(&tmKV, qkv, 3ull * C, rows, 64))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = prepare(attn_fwd_hd_kernel<D, false>, S::TOTAL))) return rc;
    if ((rc = prepare(attn_fwd_hd_kernel<D, true>, S::TOTAL))) return rc;
    done = true;
  }
  const dim3 grid(B * H, (T + 127) / 128);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  if (dcfg.thr16 == 0) launch_k(attn_fwd_hd_kernel<D, false>, grid, dim3(kThreads), S::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, dcfg);
  else launch_k(attn_fwd_hd_kernel<D, true>, grid, dim3(kThreads), S::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, dcfg);
  return launch_status("attn_fwd_hd_kernel");
}

template <int D>
int bwd_hd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, int B, int T, int H,
           const DropCfg& dcfg, cudaStream_t stream) {
  using Sq = DqHdSmem<D>;
  using Skv = DkvHdSmem<D>;
  const int C = H * D;
  const uint64_t rows = static_cast<uint64_t>(B) * T;
  CUtensorMap tmQKV128, tmQKV64, tmDO128, tmDO64;
  int rc;
  if ((rc = tmap_hd<D>(&tmQKV128, qkv, 3ull * C, rows, 128))) return rc;
  if ((rc = tmap_hd<D>(&tmQKV64, qkv, 3ull * C, rows, 64))) return rc;
  if ((rc = tmap_hd<D>(&tmDO128, dout, static_cast<uint64_t>(C), rows, 128))) return rc;
  if ((rc = tmap_hd<D>(&tmDO64, dout, static_cast<uint64_t>(C), rows, 64))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = prepare(attn_bwd_dq_hd_kernel<D, false>, Sq::TOTAL))) return rc;
    if ((rc = prepare(attn_bwd_dq_hd_kernel<D, true>, Sq::TOTAL))) return rc;
    if ((rc = prepare(attn_bwd_dkv_hd_kernel<D, false>, Skv::TOTAL))) return rc;
    if ((rc = prepare(attn_bwd_dkv_hd_kernel<D, true>, Skv::TOTAL))) return rc;
    done = true;
  }
  launch_k(attn_delta_hd_kernel<D>, dim3(static_cast<unsigned>((rows + 7) / 8)), dim3(256), 0, stream,
           reinterpret_cast<const __nv_bfloat16*>(out), reinterpret_cast<const __nv_bfloat16*>(dout), delta, B, T, H, C);
  if ((rc = launch_status("attn_delta_hd_kernel"))) return rc;
  const dim3 grid(B * H, (T + 127) / 128);
  __nv_bfloat16* g = reinterpret_cast<__nv_bfloat16*>(dqkv);
  if (dcfg.thr16 == 0) {
    launch_k(attn_bwd_dkv_hd_kernel<D, false>, grid, dim3(kThreads), Skv::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, g, T, H, C, dcfg);
    if ((rc = launch_status("attn_bwd_dkv_hd_kernel"))) return rc;
    launch_k(attn_bwd_dq_hd_kernel<D, false>, grid, dim3(kThreads), Sq::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, g, T, H, C, dcfg);
  } else {
    launch_k(attn_bwd_dkv_hd_kernel<D, true>, grid, dim3(kThreads), Skv::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, g, T, H, C, dcfg);
    if ((rc = launch_status("attn_bwd_dkv_hd_kernel"))) return rc;
    launch_k(attn_bwd_dq_hd_kernel<D, true>, grid, dim3(kThreads), Sq::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, g, T, H, C, dcfg);
  }
  return launch_status("attn_bwd_dq_hd_kernel");
}

template <int D>
int decode_hd(const void* qkv_row, void* cache, void* out, int B, int Tmax, int t, int H, cudaStream_t stream) {
  const size_t smem = static_cast<size_t>(t + 1) * sizeof(float);
  if (smem > 48 * 1024) {
    static bool done = false;
    if (!done) {
      ABCGPT_CUDA(cudaFuncSetAttribute(attn_decode_hd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      done = true;
    }
  }
  launch_k(attn_decode_hd_kernel<D>, dim3(B * H), dim3(128), smem, stream, reinterpret_cast<const __nv_bfloat16*>(qkv_row),
           reinterpret_cast<__nv_bfloat16*>(cache), reinterpret_cast<__nv_bfloat16*>(out), Tmax, t, H);
  return launch_status("attn_decode_hd_kernel");
}

}  // namespace

int attn_fwd_hd(const void* qkv, void* out, float* lse, int B, int T, int H, int D, float drop_p, uint32_t drop_key,
                cudaStream_t stream) {
  int rc = check_hd("attn_fwd_hd", B, T, H, D);
  if (rc) return rc;
  ABCGPT_CHECK_ARG(qkv && out && lse, "attn_fwd_hd: null pointer");
  ABCGPT_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f, "attn_fwd_hd: dropout p must be in [0, 1)");
  const DropCfg dcfg = make_drop(drop_p, drop_key);
  return D == 32 ? fwd_hd<32>(qkv, out, lse, B, T, H, dcfg, stream) : fwd_hd<128>(qkv, out, lse, B, T, H, dcfg, stream);
}

int attn_bwd_hd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, int B, int T,
                int H, int D, float drop_p, uint32_t drop_key, cudaStream_t stream) {
  int rc = check_hd("attn_bwd_hd", B, T, H, D);
  if (rc) return rc;
  ABCGPT_CHECK_ARG(qkv && out && dout && lse && delta && dqkv, "attn_bwd_hd: null pointer");
  ABCGPT_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f, "attn_bwd_hd: dropout p must be in [0, 1)");
  const DropCfg dcfg = make_drop(drop_p, drop_key);
  return D == 32 ? bwd_hd<32>(qkv, out, dout, lse, delta, dqkv, B, T, H, dcfg, stream)
                 : bwd_hd<128>(qkv, out, dout, lse, delta, dqkv, B, T, H, dcfg, stream);
}

int attn_decode_hd(const void* qkv_row, void* cache, void* out, int B, int Tmax, int t, int H, int D, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(D == 32 || D == 128,
                   "attn_decode_hd: head size %d is not supported (supported head sizes: 32, 128; head size 64 decodes through "
                   "abcgpt_attn_decode)", D);
  ABCGPT_CHECK_ARG(qkv_row && cache && out && B > 0 && H > 0 && t >= 0 && t < Tmax, "attn_decode_hd: bad arguments");
  ABCGPT_CHECK_ARG(static_cast<size_t>(t + 1) * 4 <= 200 * 1024, "attn_decode_hd: context too long for the probability buffer");
  return D == 32 ? decode_hd<32>(qkv_row, cache, out, B, Tmax, t, H, stream) : decode_hd<128>(qkv_row, cache, out, B, Tmax, t, H, stream);
}

}  // namespace abcgpt
