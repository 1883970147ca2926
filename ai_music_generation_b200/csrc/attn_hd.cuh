// Templated causal flash attention kernels (forward, delta, dQ, dK / dV) of csrc/attn_hd.cu (dense batches, head sizes 32 and
// 128; csrc/attn.cu is the tuned head-size-64 family) and csrc/attn_varlen.cu (packed sequences of arbitrary lengths, head sizes
// 32, 64 and 128).  Same arithmetic, mask, dropout counters and statistics layout as attn.cu, and the same roles per CTA: warp 0
// issues the TMA loads, warp 1 the tcgen05 MMAs (whole warp in the loop, one elected lane issues), warps 2..5 own one 128-row
// tile row per thread and do the softmax / dS arithmetic (the chunk helpers of attn_helpers.cuh with the scale of D).
// q | k | v are read straight out of the packed [rows, 3C] buffer through TMA column offsets, out / dqkv are written in place.
//
// One CTA per (128-row tile, sequence*head) item, heaviest tiles first (no persistent schedule, no CTA pairs: those are the
// head-size-64 tuning).  Inside an item the loads run through a ring, the score tiles are double-buffered in tensor memory and
// the accumulators (O, dQ, dK / dV) stay in tensor memory across the item.  VL selects how an item finds its sequence
// (HdItem): dense, blockIdx.x = b * H + h over B sequences of T rows; varlen, blockIdx.x = s * H + h over the rows
// [cu_seqlens[s], cu_seqlens[s+1]), statistics [H, total_rows].  Tiles may cover rows past the sequence end (the next sequence
// or, past the buffer, TMA zero fill): the causal mask already excludes every key past a query, query rows past the end are
// never stored, and the dK / dV kernel masks query columns past the end, so no value of a neighbouring row reaches a result.
//
// Operand layouts.  D = 128: a 256-byte row is two 64-column SWIZZLE_128B slabs stored one after the other (two TMA boxes),
// a K step of 16 columns selects the slab and the 32-byte offset in it; as an MN-major B operand (N = 128) the second slab is
// the next 64-wide MN atom (leading byte offset = one slab).  D = 64: one slab.  D = 32: 64-byte rows, SWIZZLE_64B tensor maps
// and descriptors.
//
// Budgets (B200: 228 KB shared memory, 512 tensor-memory columns per SM):
//   forward   tensor memory: S 2 x 64 + O D columns -> 256-column allocation, two CTAs per SM.  D = 128: Q 32 KB + a two-stage
//             K/V ring of 32 KB per stage = 96 KB per CTA; D = 64: Q 16 KB + four stages of 16 KB; D = 32: Q 8 KB + four
//             stages of 8 KB.
//   dQ        S | dP 2 x 128 + dQ D columns -> 512, one CTA per SM; Q, dO tiles + a K/V ring (D = 128: 3 stages, 160 KB).
//   dK / dV   S^T | dP^T 2 x 128 + dV, dK 2 x D columns -> 512 (exactly full at D = 128); K, V tiles + a Q/dO ring.
#pragma once
#include "attn_helpers.cuh"

namespace abcgpt {
namespace {

template <int D>
struct HdLayout {
  static_assert(D == 32 || D == 64 || D == 128, "attn_hd.cuh: head sizes 32, 64 and 128");
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

// The sequence of one CTA: T rows starting at packed row row0, head h, statistics (lse / delta / dropout row counter) of its
// row t at stat0 + t, and the 128-row tile of this CTA (fwd / dQ: query tiles, last first; dK / dV: key tiles, first first).
struct HdItem {
  int T, h, row0, tile;
  long long stat0;
};
struct VarlenSeqs {
  const int32_t* cu;   // [n_seqs + 1] row offsets
  int total;           // rows of the packed buffer (= cu[n_seqs]): the statistics stride of a head
};
// false: the grid (sized by the longest sequence) has no tile of this sequence at blockIdx.y; the whole CTA returns
template <bool VL>
__device__ __forceinline__ bool hd_item(HdItem& it, int T, int H, const VarlenSeqs& vs, bool last_first) {
  const int x = static_cast<int>(blockIdx.x);
  it.h = x % H;
  if constexpr (VL) {
    ptx::pdl_wait();   // the sequence table may be written by the preceding kernel
    const int s = x / H;
    const int r0 = vs.cu[s];
    it.T = vs.cu[s + 1] - r0;
    it.row0 = r0;
    it.stat0 = static_cast<long long>(it.h) * vs.total + r0;
  } else {
    it.T = T;
    it.row0 = (x / H) * T;
    it.stat0 = static_cast<long long>(x) * T;
  }
  const int ntiles = (it.T + 127) / 128;
  if (VL && static_cast<int>(blockIdx.y) >= ntiles) return false;   // a dense grid has exactly ntiles rows
  it.tile = last_first ? ntiles - 1 - static_cast<int>(blockIdx.y) : static_cast<int>(blockIdx.y);
  return true;
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

template <int D, bool DROP, bool VL = false>
__global__ void __launch_bounds__(kThreads, 2)
attn_fwd_hd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                   __nv_bfloat16* __restrict__ out, float* __restrict__ lse, int T, int H, int C, const DropCfg dcfg,
                   const VarlenSeqs vs) {
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
  HdItem it;
  if (!hd_item<VL>(it, T, H, vs, true)) return;   // heaviest query tiles first
  T = it.T;
  const int qt = it.tile, h = it.h, row0 = it.row0;
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
      load_tile<D>(smem + S::Q, &tmQ, q_full, h * D, row0 + qt * 128, 128);
    }
    for (int j = 0; j < num_kv; ++j) {
      const int st = j % S::RING;
      ptx::mbar_wait(&kv_empty[st], ((j / S::RING) & 1) ^ 1, 40);
      uint8_t* dst = smem + S::KV + st * S::STAGE;
      if (issue) {
        ptx::mbar_expect_tx(&kv_full[st], S::STAGE);
        load_tile<D>(dst, &tmKV, &kv_full[st], C + h * D, row0 + j * 64, 64);
        load_tile<D>(dst + L::T64, &tmKV, &kv_full[st], 2 * C + h * D, row0 + j * 64, 64);
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
    const uint32_t drop_rk = DROP ? drop_row_key(dcfg.key, static_cast<uint32_t>(it.stat0 + qt * 128 + r)) : 0u;
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
    __nv_bfloat16* o = out + static_cast<long long>(row0 + t) * C + h * D;
#pragma unroll
    for (int c = 0; c < D / 32; ++c) {
      uint32_t v[32];
      ptx::tmem_ld32(tm_O + lane_off + c * 32, v);
      ptx::tmem_ld_wait();
      if (t < T) store_row32(o + c * 32, v, inv);
    }
    if (t < T) lse[it.stat0 + t] = (m_ref + log2f(l)) * kLn2;
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

template <int D, bool DROP, bool VL = false>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dq_hd_kernel(const __grid_constant__ CUtensorMap tmQKV128, const __grid_constant__ CUtensorMap tmQKV64,
                      const __grid_constant__ CUtensorMap tmDO128, const float* __restrict__ lse, const float* __restrict__ delta,
                      __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, const DropCfg dcfg, const VarlenSeqs vs) {
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
  HdItem it;
  if (!hd_item<VL>(it, T, H, vs, true)) return;
  T = it.T;
  const int qt = it.tile, h = it.h, row0 = it.row0;
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
      const int q_row = row0 + qt * 128;
      ptx::mbar_expect_tx(qdo_full, 2 * L::T128);
      load_tile<D>(smem + S::Q, &tmQKV128, qdo_full, h * D, q_row, 128);
      load_tile<D>(smem + S::DO, &tmDO128, qdo_full, h * D, q_row, 128);
    }
    for (int j = 0; j < num_kv; ++j) {
      const int st = j % S::RING;
      ptx::mbar_wait(&kv_empty[st], ((j / S::RING) & 1) ^ 1, 50);
      uint8_t* dst = smem + S::KV + st * S::STAGE;
      if (issue) {
        ptx::mbar_expect_tx(&kv_full[st], S::STAGE);
        load_tile<D>(dst, &tmQKV64, &kv_full[st], C + h * D, row0 + j * 64, 64);
        load_tile<D>(dst + L::T64, &tmQKV64, &kv_full[st], 2 * C + h * D, row0 + j * 64, 64);
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
    const long long sidx = it.stat0 + t;
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
    __nv_bfloat16* o = dqkv + static_cast<long long>(row0 + t) * (3 * C) + h * D;
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

template <int D, bool DROP, bool VL = false>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_dkv_hd_kernel(const __grid_constant__ CUtensorMap tmQKV128, const __grid_constant__ CUtensorMap tmQKV64,
                       const __grid_constant__ CUtensorMap tmDO64, const float* __restrict__ lse, const float* __restrict__ delta,
                       __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, const DropCfg dcfg, const VarlenSeqs vs) {
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
  HdItem it;
  if (!hd_item<VL>(it, T, H, vs, false)) return;   // key tile 0 sees every query tile: heaviest first
  T = it.T;
  const int kt = it.tile, h = it.h, row0 = it.row0;
  const int nq64 = (T + 63) / 64;
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
      load_tile<D>(smem + S::K, &tmQKV128, kv_full, C + h * D, row0 + kt * 128, 128);
      load_tile<D>(smem + S::V, &tmQKV128, kv_full, 2 * C + h * D, row0 + kt * 128, 128);
    }
    for (int n = 0; n < nsteps; ++n) {
      const int st = n % S::RING;
      ptx::mbar_wait(&qdo_empty[st], ((n / S::RING) & 1) ^ 1, 60);
      uint8_t* dst = smem + S::QDO + st * S::STAGE;
      if (issue) {
        ptx::mbar_expect_tx(&qdo_full[st], S::STAGE);
        load_tile<D>(dst, &tmQKV64, &qdo_full[st], h * D, row0 + (i0 + n) * 64, 64);
        load_tile<D>(dst + L::T64, &tmDO64, &qdo_full[st], h * D, row0 + (i0 + n) * 64, 64);
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
    const float* stat_src = (tid < 64 ? lse : delta) + it.stat0;
    const float stat_coef = tid < 64 ? -kLog2e : -scale_of(D);
    for (int n = 0; n < nsteps; ++n) {
      const int q0 = (i0 + n) * 64;
      // column (query) statistics of this step into shared memory: two buffers by step parity; a buffer is rewritten two steps
      // later, after a barrier that follows every read of it
      float* st = stat + (n & 1) * 192;
      const int qi = q0 + (tid & 63);
      st[tid] = qi < T ? __ldg(stat_src + qi) * stat_coef : 0.f;
      if (DROP && tid < 64) st[128 + tid] = __uint_as_float(drop_row_key(dcfg.key, static_cast<uint32_t>(it.stat0 + qi)));
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
    __nv_bfloat16* orow = dqkv + static_cast<long long>(row0 + kv_t) * (3 * C) + h * D;
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

}  // namespace
}  // namespace abcgpt
