// Causal flash attention, forward and backward, head size 64, on tcgen05 tensor cores with TMEM accumulators.
// Replaces F.scaled_dot_product_attention(q, k, v, is_causal=True) at nanoGPT/model.py:64 together with the head
// split / merge copies at model.py:56-59,72: the kernels read q|k|v straight out of the packed c_attn output
// [B*T, 3C] through one TMA tensor map (column offset selects q/k/v and the head) and write [B*T, C] directly.
//
// Work item = (128-row tile, batch*head); all three kernels are persistent over a static item schedule.
//   attn_fwd_kernel       item = 128 query rows; K/V streamed in 64-row tiles
//                         S = Q K^T (UMMA 128x64x64) -> TMEM -> softmax, one thread per query row -> bf16 P back into
//                         TMEM -> O += P V (UMMA, A operand from TMEM) accumulated in TMEM -> registers at item end
//   attn_bwd_dq_kernel    item = 128 query rows, K/V in 64-row tiles:   S, dP -> dS -> dQ += dS K   (TMEM acc)
//   attn_bwd_dkv_kernel   item = 128 key rows,  Q/dO in 64-row tiles:  S^T, dP^T -> P^T, dS^T -> dV += P^T dO,
//                         dK += dS^T Q (TMEM acc).  Two kernels instead of atomics on dQ: deterministic gradients.
// The forward runs two CTAs per SM so that one CTA's softmax (MUFU-bound) overlaps the other's MMAs.
#include "attn_helpers.cuh"

namespace abcgpt {

// csrc/attn_pair.cu: the same backward on CTA pairs (cta_group::2 MMAs) for unpacked sequences of >= 512 positions
int attn_bwd_pair(const void* qkv, const void* dout, const float* lse, const float* delta, void* dqkv, int B, int T, int H,
                  const DropCfg& dcfg, cudaStream_t stream);
// csrc/attn_fwd3.cu: the forward with three CTAs per SM (single-buffered S / O in 128 tensor-memory columns)
int attn_fwd3(const CUtensorMap& tmQ, const CUtensorMap& tmKV, void* out, float* lse, int T, int H, int C, int BH, int nitems,
              const DropCfg& dcfg, int seq_shift, uint32_t fBH_d, uint32_t fBH_m, uint32_t fH_d, uint32_t fH_m, cudaStream_t stream);

namespace {

// ======================================================================================================
// forward
// ======================================================================================================
// 128 query rows per item, K/V streamed in 64-row tiles through a ring.  The score tile S (128 x 64 fp32) is
// double-buffered in TMEM so the tensor core computes S_{j+1} while the softmax threads work on S_j; the bf16 P tile is
// written back over the consumed S tile and read by the P V MMA straight from TMEM; O accumulates in TMEM across all
// tiles of an item (two O buffers: the epilogue of item i overlaps the MMAs of item i+1).  Accumulating O in TMEM
// needs a per-row reference exponent that is NOT the running max: m_ref is the true max of the first tile and is
// only raised (with an in-TMEM rescale of O) when a later tile exceeds it by more than 2^64 -- exact in floating
// point, because a common power-of-two factor cancels in O / l.
constexpr int kFwdRing = 4;
struct FwdSmem {
  static constexpr int Q = 0;                       // 2 items x (128 x 64 bf16)
  static constexpr int KV = 32768;                  // kFwdRing stages x (K 64x64 | V 64x64)
  static constexpr int BAR = KV + kFwdRing * 16384;
  static constexpr int TOTAL = BAR + 256 + 1024;
};

// Four compute warps, one per 32-row quarter of the tile (a warp can only reach the tensor-memory lanes of its own quarter): a
// thread owns one row and all 64 columns of every step.  With both resident CTAs in their softmax phase the SM runs 2 x 8192
// exponentials per ~1300-cycle step = 12.6 per clock of the MUFU's 16, with its issue slots ~60 % busy: the kernel sits on both
// limits, so neither more warps per row nor trading MUFU for FMA instructions moves it (DESIGN.md §4.2 records both attempts).
template <bool DROP>
__global__ void __launch_bounds__(kThreads, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                __nv_bfloat16* __restrict__ out, float* __restrict__ lse, int T, int H, int C, int BH, int nitems,
                const DropCfg dcfg, int seq_shift, const FastDiv fBH, const FastDiv fH) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + FwdSmem::BAR);
  uint64_t* q_full = bars + 0;                   // [2]
  uint64_t* q_empty = bars + 2;                  // [2]
  uint64_t* kv_full = bars + 4;                  // [kFwdRing]
  uint64_t* kv_empty = kv_full + kFwdRing;       // [kFwdRing]
  uint64_t* s_full = kv_empty + kFwdRing;        // [2]
  uint64_t* p_full = s_full + 2;                 // [2]
  uint64_t* p_empty = p_full + 2;                // [2]
  uint64_t* o_full = p_empty + 2;                // [2]
  uint64_t* o_free = o_full + 2;                 // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_free + 2);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nqt = (T + 127) / 128;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ);
    ptx::prefetch_tmap(&tmKV);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&q_full[s], 1);
      ptx::mbar_init(&q_empty[s], 1);
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&p_full[s], 128);
      ptx::mbar_init(&p_empty[s], 1);
      ptx::mbar_init(&o_full[s], 1);
      ptx::mbar_init(&o_free[s], 128);
    }
    for (int s = 0; s < kFwdRing; ++s) {
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
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);  // S buffers at columns [0,64) and [64,128); O buffers at [128,192) and [192,256)
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();               // everything above touched only this CTA's shared memory / TMEM

  // number of 64-row K/V tiles of an item
  auto tiles_of = [&](int it) {
    const int qt = nqt - 1 - fdiv(it, fBH);
    return (min(T, qt * 128 + 128) + 63) / 64;
  };

  if (warp == 0) {
    {
      const bool issue = ptx::elect_one();  // whole warp runs the loop, one elected lane issues (uniform operands)
      int gt = 0;
      for (int item_k = 0;; ++item_k) {
        const int it = sched_item(item_k, nitems);
        if (it < 0) break;
        const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
        const int num_kv = tiles_of(it);
        const int qb = item_k & 1;
        ptx::mbar_wait(&q_empty[qb], ((item_k >> 1) & 1) ^ 1, 10);
        if (issue) ptx::mbar_expect_tx(&q_full[qb], 16384);
        if (issue) ptx::tma_load_2d(smem + FwdSmem::Q + qb * 16384, &tmQ, &q_full[qb], h * HS, b * T + qt * 128);
        for (int j = 0; j < num_kv; ++j, ++gt) {
          const int st = gt % kFwdRing;
          ptx::mbar_wait(&kv_empty[st], ((gt / kFwdRing) & 1) ^ 1, 11);
          if (issue) ptx::mbar_expect_tx(&kv_full[st], 16384);
          uint8_t* dst = smem + FwdSmem::KV + st * 16384;
          if (issue) ptx::tma_load_2d(dst, &tmKV, &kv_full[st], C + h * HS, b * T + j * 64);
          if (issue) ptx::tma_load_2d(dst + 8192, &tmKV, &kv_full[st], 2 * C + h * HS, b * T + j * 64);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    {
      const bool leader = ptx::elect_one();  // the whole warp runs this loop (uniform operands); one elected lane issues
      constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
      constexpr uint32_t idesc_o = ptx::umma_idesc_bf16(128, 64, 0, 1);
      const uint32_t sQ = ptx::smem_u32(smem + FwdSmem::Q);
      const uint32_t sKV = ptx::smem_u32(smem + FwdSmem::KV);
      // two cursors over the same (item, tile) sequence: the S = Q K^T issue runs one tile ahead of the P V issue, across
      // item boundaries, so the tensor core computes S of the next tile while the softmax threads work on this one
      int s_k = 0, s_it = sched_item(0, nitems), s_j = 0, s_n = s_it >= 0 ? tiles_of(s_it) : 0, s_gt = 0;
      int p_k = 0, p_it = s_it, p_j = 0, p_n = s_n, p_gt = 0;
      auto issue_s = [&]() {
        if (s_j == 0) ptx::mbar_wait(&q_full[s_k & 1], (s_k >> 1) & 1, 12);
        ptx::mbar_wait(&kv_full[s_gt % kFwdRing], (s_gt / kFwdRing) & 1, 13);
        ptx::tc_fence_after();
        const uint32_t sQi = sQ + (s_k & 1) * 16384, sK = sKV + (s_gt % kFwdRing) * 16384;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ss(tmem_base + (s_gt & 1) * 64, desc_k(sQi, k), desc_k(sK, k), idesc_s, k > 0);
        if (leader) ptx::umma_commit(&s_full[s_gt & 1]);
        if (leader && (s_j == s_n - 1)) ptx::umma_commit(&q_empty[s_k & 1]);  // last S of the item: its Q tile may be overwritten
        ++s_j;
        ++s_gt;
        if (s_j == s_n) {
          ++s_k;
          s_it = sched_item(s_k, nitems);
          s_j = 0;
          s_n = s_it >= 0 ? tiles_of(s_it) : 0;
        }
      };
      if (s_it >= 0) issue_s();
      while (p_it >= 0) {
        if (s_it >= 0) issue_s();
        if (p_j == 0 && p_k >= 2) ptx::mbar_wait(&o_free[p_k & 1], ((p_k >> 1) - 1) & 1, 14);  // item p_k-2 has been drained
        ptx::mbar_wait(&p_full[p_gt & 1], (p_gt >> 1) & 1, 15);
        ptx::tc_fence_after();
        const uint32_t sV = sKV + (p_gt % kFwdRing) * 16384 + 8192;
        const uint32_t tP = tmem_base + (p_gt & 1) * 64;  // bf16 P (32 packed columns) written over the consumed S tile
        const uint32_t tO = tmem_base + 128 + (p_k & 1) * 64;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ts(tO, tP + 8 * k, desc_mn(sV, k), idesc_o, (p_j > 0 || k > 0));
        if (leader) ptx::umma_commit(&kv_empty[p_gt % kFwdRing]);
        if (leader) ptx::umma_commit(&p_empty[p_gt & 1]);
        if (leader && (p_j == p_n - 1)) ptx::umma_commit(&o_full[p_k & 1]);
        ++p_j;
        ++p_gt;
        if (p_j == p_n) {
          ++p_k;
          p_it = sched_item(p_k, nitems);
          p_j = 0;
          p_n = p_it >= 0 ? tiles_of(p_it) : 0;
        }
      }
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;  // row inside the tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    // item epilogue: O / l -> bf16, LSE.  The O buffer is released as soon as it sits in registers.  It runs AFTER the
    // first tile of the following item: by then the last P V of this item has completed (no stall on o_full) and the
    // tensor core already has the next S tiles to chew on.
    auto epilogue = [&](int k, int it, float l, float m_ref) {
      const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
      const uint32_t tm_O = tmem_base + 128 + (k & 1) * 64;
      ptx::mbar_wait(&o_full[k & 1], (k >> 1) & 1, 20);
      ptx::tc_fence_after();
      uint32_t v0[32], v1[32];
      ptx::tmem_ld32(tm_O + lane_off, v0);
      ptx::tmem_ld32(tm_O + lane_off + 32, v1);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&o_free[k & 1]);
      const int t = qt * 128 + r;
      if (t < T) {
        const float inv = (DROP ? dcfg.inv_keep : 1.0f) / l;
        __nv_bfloat16* o = out + static_cast<long long>(b * T + t) * C + h * HS;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 w;
          w.x = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 0]) * inv, __uint_as_float(v0[8 * q + 1]) * inv);
          w.y = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 2]) * inv, __uint_as_float(v0[8 * q + 3]) * inv);
          w.z = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 4]) * inv, __uint_as_float(v0[8 * q + 5]) * inv);
          w.w = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 6]) * inv, __uint_as_float(v0[8 * q + 7]) * inv);
          reinterpret_cast<uint4*>(o)[q] = w;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 w;
          w.x = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 0]) * inv, __uint_as_float(v1[8 * q + 1]) * inv);
          w.y = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 2]) * inv, __uint_as_float(v1[8 * q + 3]) * inv);
          w.z = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 4]) * inv, __uint_as_float(v1[8 * q + 5]) * inv);
          w.w = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 6]) * inv, __uint_as_float(v1[8 * q + 7]) * inv);
          reinterpret_cast<uint4*>(o)[4 + q] = w;
        }
        lse[stat_idx(b, h, t, H, T, seq_shift)] = (m_ref + log2f(l)) * kLn2;
      }
    };
    auto chunk_max = [&](int cls, uint32_t taddr) -> float {
      if (cls == kFull) return fwd_chunk_max<kFull>(taddr, lane);
      if (cls == kDiag) return fwd_chunk_max<kDiag>(taddr, lane);
      return -1e30f;
    };
    bool pend = false;
    int pend_k = 0, pend_it = 0;
    float pend_l = 1.f, pend_m = 0.f;
    int gt = 0;
    for (int item_k = 0;; ++item_k) {
      const int it = sched_item(item_k, nitems);
      if (it < 0) break;
      const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH);
      const int num_kv = tiles_of(it);
      const uint32_t tm_O = tmem_base + 128 + (item_k & 1) * 64;
      const int r0 = qt * 128 + quarter * 32;  // first query row of this warp (relative to the sequence)
      float m_ref = 0.f, l = 0.f;
      bool have_ref = false;  // the reference exponent comes from the first tile that has a visible key for this warp
      const uint32_t drop_rk =
          DROP ? drop_row_key(dcfg.key, static_cast<uint32_t>(stat_idx(fdiv(bh, fH), fmodi(bh, fH), qt * 128 + r, H, T, seq_shift))) : 0u;
      for (int j = 0; j < num_kv; ++j, ++gt) {
        const int bsel = gt & 1;
        const uint32_t tm_s = tmem_base + lane_off + bsel * 64;
        // chunk classes of this warp's rows for key columns [64j, 64j+32) and [64j+32, 64j+64)
        const int c0 = j * 64, c1 = j * 64 + 32;
        const int cls0 = !same_seq(c0, r0, seq_shift) ? kMasked : ((c0 + 31 <= r0) ? kFull : ((c0 > r0 + 31) ? kMasked : kDiag));
        const int cls1 = !same_seq(c1, r0, seq_shift) ? kMasked : ((c1 + 31 <= r0) ? kFull : ((c1 > r0 + 31) ? kMasked : kDiag));
        ptx::mbar_wait(&s_full[bsel], (gt >> 1) & 1, 17);
        ptx::tc_fence_after();
        uint32_t pk[32];
        float tmax = -1e30f, rowsum = 0.f;
        if (!have_ref && (cls0 != kMasked || cls1 != kMasked)) {
          have_ref = true;
          // first tile (with packed short sequences: the first tile of this warp's own sequence): the reference exponent
          // is its true row max (cheap max-only pass, then the exp pass)
          tmax = fmaxf(chunk_max(cls0, tm_s), chunk_max(cls1, tm_s + 32));
          m_ref = tmax * kSl2;
          fwd_tile<DROP>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, seq_shift);
        } else {
          fwd_tile<DROP>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, seq_shift);
          const bool need = tmax * kSl2 - m_ref > kRescaleThreshold;
          if (__any_sync(0xffffffffu, need)) {
            // rare: raise the reference, rescale the O accumulator in TMEM, recompute this tile's P
            const float m_new = need ? tmax * kSl2 : m_ref;
            const float alpha = ex2(m_ref - m_new);
            ptx::mbar_wait(&p_empty[(gt - 1) & 1], ((gt - 1) >> 1) & 1, 19);  // every earlier P V product has landed in O
            ptx::tc_fence_after();
#pragma unroll
            for (int c = 0; c < 2; ++c) {
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
            fwd_tile<DROP>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, seq_shift);
          }
        }
        l += rowsum;
        // P (64 key columns = 32 packed words) overwrites the first half of this tile's S buffer; the tensor pipe runs in
        // issue order, so S_{j+2} cannot overwrite it before P V of this tile has consumed it
        ptx::tmem_st16(tm_s, pk);
        ptx::tmem_st16(tm_s + 16, pk + 16);
        ptx::tmem_st_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(&p_full[bsel]);
        if (pend) {
          epilogue(pend_k, pend_it, pend_l, pend_m);
          pend = false;
        }
      }
      // this item's epilogue is deferred until after the first tile of the next item (see below)
      pend = true;
      pend_k = item_k;
      pend_it = it;
      pend_l = l;
      pend_m = m_ref;
    }
    if (pend) epilogue(pend_k, pend_it, pend_l, pend_m);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 256);
}

// ======================================================================================================
// backward: delta = rowsum(dO * O) per (token, head)
// ======================================================================================================
__global__ void __launch_bounds__(256)
attn_delta_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ dout, float* __restrict__ delta,
                  int B, int T, int H, int C, int seq_shift) {
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();
  // one warp per token row; a lane reads 16-byte units (8 columns), 8 lanes cover one head (64 columns): 128-bit loads,
  // three shuffles per head group instead of five per head
  const int lane = threadIdx.x & 31;
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= static_cast<long long>(B) * T) return;
  const int b = static_cast<int>(row / T), t = static_cast<int>(row % T);
  const uint4* orow = reinterpret_cast<const uint4*>(o + row * C);
  const uint4* drow = reinterpret_cast<const uint4*>(dout + row * C);
  const int units = C / 8;  // H * 8
  for (int u = lane; u < ((units + 31) & ~31); u += 32) {
    float s = 0.f;
    if (u < units) {
      const uint4 a = __ldg(orow + u), d = __ldg(drow + u);
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, dw[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) s += ptx::bf16lo(aw[e]) * ptx::bf16lo(dw[e]) + ptx::bf16hi(aw[e]) * ptx::bf16hi(dw[e]);
    }
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    if ((lane & 7) == 0 && u < units) delta[stat_idx(b, u >> 3, t, H, T, seq_shift)] = s;
  }
}

// ======================================================================================================
// backward: dQ and dK/dV
// ======================================================================================================
// Both backward kernels run ONE persistent CTA per SM with two compute groups of 128 threads.  The score tiles S and dP
// (128 x 64 fp32 each) are triple-buffered in TMEM and consecutive steps alternate between the groups: while group 0
// turns S/dP of step j into dS, the tensor core already produces S/dP of step j+1 for group 1, and the accumulating
// MMAs (dQ, or dV and dK) of finished steps interleave in between.  Step counters run freely across items, so the
// producer and the score MMAs are already working on the next item while this item's accumulators are drained.
constexpr int kSBuf = 3;          // S/dP score buffers in TMEM: two are being consumed by the two groups, one is being produced
constexpr int kRing = 6;          // K/V (dQ kernel) or Q/dO (dK/dV kernel) tiles in flight: TMA latency >> one step
constexpr int kBwdThreads = 352;  // warp 0 TMA, warp 1 score MMAs, warps 2..5 group 0, warps 6..9 group 1, warp 10 accumulating MMAs

struct DqSmem {
  static constexpr int QDO = 0;       // 2 items x (Q 128x64 | dO 128x64)
  static constexpr int KV = 65536;    // kRing stages x (K 64x64 | V 64x64)
  static constexpr int BAR = KV + kRing * 16384;  // dS never touches shared memory: it is written back into TMEM
  static constexpr int TOTAL = BAR + 512 + 1024;
};

template <bool DROP>
__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQKV128, const __grid_constant__ CUtensorMap tmQKV64,
                   const __grid_constant__ CUtensorMap tmDO128, const float* __restrict__ lse,
                   const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, int BH,
                   int nitems, const DropCfg dcfg, int seq_shift, const FastDiv fBH, const FastDiv fH) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + DqSmem::BAR);
  uint64_t* qdo_full = bars + 0;                // [2]
  uint64_t* qdo_empty = bars + 2;               // [2]
  uint64_t* kv_full = bars + 4;                 // [kRing]
  uint64_t* kv_empty = kv_full + kRing;         // [kRing]
  uint64_t* s_full = kv_empty + kRing;          // [kSBuf]
  uint64_t* s_free = s_full + kSBuf;            // [kSBuf] committed after the dQ MMA that read dS out of this buffer
  uint64_t* ds_full = s_free + kSBuf;           // [kSBuf] one per score buffer (NOT per group: a group may finish two steps
                                                //         while the dQ issuer waits for acc_free; a parity wait tolerates one phase)
  uint64_t* acc_full = ds_full + kSBuf;         // [2] dQ accumulator of an item complete
  uint64_t* acc_free = acc_full + 2;            // [2] ... and drained into registers by all 256 compute threads
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_free + 2);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nqt = (T + 127) / 128;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQKV128);
    ptx::prefetch_tmap(&tmQKV64);
    ptx::prefetch_tmap(&tmDO128);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&qdo_full[s], 1);
      ptx::mbar_init(&qdo_empty[s], 1);
      ptx::mbar_init(&acc_full[s], 1);
      ptx::mbar_init(&acc_free[s], 256);
    }
    for (int s = 0; s < kRing; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], 1);
    }
    for (int s = 0; s < kSBuf; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&s_free[s], 1);
      ptx::mbar_init(&ds_full[s], 128);
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
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();               // everything above touched only this CTA's shared memory / TMEM
  const uint32_t tm_dQ = tmem_base + 128 * kSBuf;  // score buffer b: S at 128 b, dP at 128 b + 64; dQ buffers at 384, 448

  // number of 64-row K/V tiles of an item (item -> query tile nqt-1-rank: heaviest first)
  auto tiles_of = [&](int it) {
    const int qt = nqt - 1 - fdiv(it, fBH);
    return (min(T, qt * 128 + 128) + 63) / 64;
  };

  if (warp == 0) {
    {
      const bool issue = ptx::elect_one();  // whole warp runs the loop, one elected lane issues (uniform operands)
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_item(k, nitems);
        if (it < 0) break;
        const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
        const int num_kv = tiles_of(it), row0 = b * T + qt * 128;
        const int qb = k & 1;
        ptx::mbar_wait(&qdo_empty[qb], ((k >> 1) & 1) ^ 1, 20);
        if (issue) ptx::mbar_expect_tx(&qdo_full[qb], 32768);
        if (issue) ptx::tma_load_2d(smem + DqSmem::QDO + qb * 32768, &tmQKV128, &qdo_full[qb], h * HS, row0);
        if (issue) ptx::tma_load_2d(smem + DqSmem::QDO + qb * 32768 + 16384, &tmDO128, &qdo_full[qb], h * HS, row0);
        for (int j = 0; j < num_kv; ++j, ++gs) {
          const int st = gs % kRing;
          ptx::mbar_wait(&kv_empty[st], ((gs / kRing) & 1) ^ 1, 21);
          if (issue) ptx::mbar_expect_tx(&kv_full[st], 16384);
          uint8_t* dst = smem + DqSmem::KV + st * 16384;
          if (issue) ptx::tma_load_2d(dst, &tmQKV64, &kv_full[st], C + h * HS, b * T + j * 64);
          if (issue) ptx::tma_load_2d(dst + 8192, &tmQKV64, &kv_full[st], 2 * C + h * HS, b * T + j * 64);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---- score MMAs: S_j = Q K_j^T, dP_j = dO V_j^T into TMEM score buffer gs % kSBuf (one issuing thread per MMA
    // family: a single thread issuing all twelve MMAs of a step plus its barrier traffic was the bottleneck)
    {
      const bool leader = ptx::elect_one();  // the whole warp runs this loop (uniform operands); one elected lane issues
      constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
      const uint64_t dQDO0 = desc_k(ptx::smem_u32(smem + DqSmem::QDO), 0);
      const uint64_t dKV0 = desc_k(ptx::smem_u32(smem + DqSmem::KV), 0);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_item(k, nitems);
        if (it < 0) break;
        const int num_kv = tiles_of(it);
        const uint64_t dQ0 = dQDO0 + static_cast<uint64_t>((k & 1) * (32768 >> 4)), dDO0 = dQ0 + (16384 >> 4);
        ptx::mbar_wait(&qdo_full[k & 1], (k >> 1) & 1, 22);
        for (int j = 0; j < num_kv; ++j, ++gs) {
          ptx::mbar_wait(&kv_full[gs % kRing], (gs / kRing) & 1, 23);
          if (gs >= kSBuf) ptx::mbar_wait(&s_free[gs % kSBuf], ((gs / kSBuf) - 1) & 1, 24);  // the dQ MMA of step gs-3 has read its dS
          ptx::tc_fence_after();
          const uint64_t dK = dKV0 + static_cast<uint64_t>((gs % kRing) * (16384 >> 4)), dV = dK + (8192 >> 4);
          const uint32_t tS = tmem_base + (gs % kSBuf) * 128;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss(tS, dQ0 + 2 * kk, dK + 2 * kk, idesc_s, kk > 0);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss(tS + 64, dDO0 + 2 * kk, dV + 2 * kk, idesc_s, kk > 0);
          if (leader) ptx::umma_commit(&s_full[gs % kSBuf]);
        }
        if (leader) ptx::umma_commit(&qdo_empty[k & 1]);  // all score MMAs of the item done: its Q / dO tiles may be overwritten
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    // ---- accumulating MMAs: dQ += dS_j K_j  (dQ accumulator double-buffered by item parity)
    {
      const bool leader = ptx::elect_one();  // the whole warp runs this loop (uniform operands); one elected lane issues
      constexpr uint32_t idesc_dq = ptx::umma_idesc_bf16(128, 64, 0, 1);
      const uint64_t dKmn0 = desc_mn(ptx::smem_u32(smem + DqSmem::KV), 0);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_item(k, nitems);
        if (it < 0) break;
        const int num_kv = tiles_of(it);
        const uint32_t tAcc = tm_dQ + (k & 1) * 64;
        if (k >= 2) {
          ptx::mbar_wait(&acc_free[k & 1], ((k >> 1) - 1) & 1, 25);
          ptx::tc_fence_after();
        }
        for (int j = 0; j < num_kv; ++j, ++gs) {
          ptx::mbar_wait(&ds_full[gs % kSBuf], (gs / kSBuf) & 1, 26);
          ptx::tc_fence_after();
          // A = dS (bf16 pairs, 32 columns) sits in the first columns of this step's score buffer
          const uint32_t tA = tmem_base + (gs % kSBuf) * 128;
          const uint64_t dK = dKmn0 + static_cast<uint64_t>((gs % kRing) * (16384 >> 4));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ts(tAcc, tA + 8 * kk, dK + (2048 >> 4) * kk, idesc_dq, (j > 0 || kk > 0));
          if (leader) ptx::umma_commit(&kv_empty[gs % kRing]);  // S_j / dP_j (other issuer) completed before ds_full could complete
          if (leader) ptx::umma_commit(&s_free[gs % kSBuf]);    // the score buffer (now holding dS) may be overwritten
        }
        if (leader) ptx::umma_commit(&acc_full[k & 1]);
      }
    }
    __syncwarp();
  } else {
    const int g = (warp - 2) >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    // per-item row statistics of this thread's query row: RAW values prefetched one item ahead (the scaling happens at
    // the point of use, otherwise the multiply sits right behind the load and the warp eats the global-load latency)
    auto load_stats = [&](int k, float& raw_l, float& raw_d) {
      raw_l = 0.f;
      raw_d = 0.f;
      const int it = sched_item(k, nitems);
      if (it < 0) return;
      const int t = (nqt - 1 - fdiv(it, fBH)) * 128 + r;
      if (t < T) {
        const int bh = fmodi(it, fBH);
        const long long idx = stat_idx(fdiv(bh, fH), fmodi(bh, fH), t, H, T, seq_shift);
        raw_l = __ldg(lse + idx);
        raw_d = __ldg(delta + idx);
      }
    };
    // item epilogue: group g writes columns [32 g, 32 g + 32) of dQ; the accumulator is released once it is in registers
    auto epilogue = [&](int k) {
      const int it = sched_item(k, nitems);
      const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
      const int t = qt * 128 + r;
      ptx::mbar_wait(&acc_full[k & 1], (k >> 1) & 1, 27);
      ptx::tc_fence_after();
      uint32_t v[32];
      ptx::tmem_ld32(tm_dQ + (k & 1) * 64 + lane_off + g * 32, v);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&acc_free[k & 1]);
      if (t < T) {
        __nv_bfloat16* o = dqkv + static_cast<long long>(b * T + t) * (3 * C) + h * HS + g * 32;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 w;
          w.x = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 0]), __uint_as_float(v[8 * q + 1]));
          w.y = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3]));
          w.z = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5]));
          w.w = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7]));
          reinterpret_cast<uint4*>(o)[q] = w;
        }
      }
    };
    // cursor over this group's steps: item pass c_k, step c_n inside the item, global step c_base + c_n (parity == g)
    int c_k = 0, c_it = sched_item(0, nitems), c_n = g, c_base = 0, c_nq = c_it >= 0 ? tiles_of(c_it) : 0;
    auto normalize = [&]() {
      while (c_it >= 0 && c_n >= c_nq) {
        c_n -= c_nq;
        c_base += c_nq;
        ++c_k;
        c_it = sched_item(c_k, nitems);
        c_nq = c_it >= 0 ? tiles_of(c_it) : 0;
      }
    };
    normalize();
    int ep_k = 0, stat_k = -1, nxt_k = c_k;
    int r0 = 0;
    uint32_t drop_rk = 0;
    float neg_l = 0.f, neg_d = 0.f, nxt_l, nxt_d;
    load_stats(c_k, nxt_l, nxt_d);
    while (c_it >= 0) {
      if (stat_k != c_k) {  // first own step in a new item: decode it once, take its row statistics, prefetch the next item's
        if (nxt_k != c_k) load_stats(c_k, nxt_l, nxt_d);  // (prefetch guessed another item: never at the shapes in use)
        neg_l = -nxt_l * kLog2e;
        neg_d = -nxt_d * kScale;
        const int qt = nqt - 1 - fdiv(c_it, fBH), bh = fmodi(c_it, fBH);
        r0 = qt * 128 + quarter * 32;
        if (DROP) drop_rk = drop_row_key(dcfg.key, static_cast<uint32_t>(stat_idx(fdiv(bh, fH), fmodi(bh, fH), qt * 128 + r, H, T, seq_shift)));
        stat_k = c_k;
        // the next item this group touches is c_k + 1 unless that item has a single step owned by the other group
        int nk = c_k + 1;
        {
          const int nit = sched_item(nk, nitems);
          if (nit >= 0 && tiles_of(nit) == 1 && ((c_base + c_nq) & 1) != g) ++nk;
        }
        load_stats(nk, nxt_l, nxt_d);
        nxt_k = nk;
      }
      const int gs = c_base + c_n;
      ptx::mbar_wait(&s_full[gs % kSBuf], (gs / kSBuf) & 1, 28);
      ptx::tc_fence_after();
      const uint32_t tbuf = tmem_base + lane_off + (gs % kSBuf) * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = c_n * 64 + c * 32;
        const uint32_t ta_s = tbuf + c * 32, ta_dp = ta_s + 64;
        uint32_t pk[16];
        const int cr = real_col(c0, seq_shift);
        if (c0 > r0 + 31 || !same_seq(c0, r0, seq_shift)) dq_chunk<kMasked, DROP>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, cr);
        else if (c0 + 31 <= r0) dq_chunk<kFull, DROP>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, cr);
        else dq_chunk<kDiag, DROP>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, cr);
        // dS chunk c (32 key columns = 16 packed words) overwrites score columns that this thread has already consumed
        ptx::tmem_st16(tbuf + c * 16, pk);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&ds_full[gs % kSBuf]);
      // earlier items are drained AFTER this group's first step in a later item: by then their last MMAs (which wait for
      // the other group's final step) have completed, so the drain does not stall the step pipeline
      while (ep_k < c_k) epilogue(ep_k++);
      c_n += 2;
      normalize();
    }
    // items not yet drained (c_k is now one past the last item of this CTA)
    while (ep_k < c_k) epilogue(ep_k++);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 512);
}

struct DkvSmem {
  static constexpr int KV = 0;         // 2 items x (K 128x64 | V 128x64)
  static constexpr int QDO = 65536;    // kRing stages x (Q 64x64 | dO 64x64)
  // P^T and dS^T never touch shared memory: they are written back into TMEM and consumed as the A operand from there
  static constexpr int STAT = QDO + kRing * 16384;  // 2 groups x 2 buffers x (-lse2[64] | -delta8[64] | dropout row key[64])
  static constexpr int BAR = STAT + 3072;
  static constexpr int TOTAL = BAR + 512 + 1024;
};

template <bool DROP>
__global__ void __launch_bounds__(kBwdThreads, 1)
attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap tmQKV128, const __grid_constant__ CUtensorMap tmQKV64,
                    const __grid_constant__ CUtensorMap tmDO64, const float* __restrict__ lse,
                    const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, int BH,
                    int nitems, const DropCfg dcfg, int seq_shift, const FastDiv fBH, const FastDiv fH) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + DkvSmem::BAR);
  uint64_t* kv_full = bars + 0;                 // [2]
  uint64_t* kv_empty = bars + 2;                // [2]
  uint64_t* qdo_full = bars + 4;                // [kRing]
  uint64_t* qdo_empty = qdo_full + kRing;       // [kRing]
  uint64_t* s_full = qdo_empty + kRing;         // [kSBuf]
  uint64_t* s_free = s_full + kSBuf;            // [kSBuf] committed after the dV / dK MMAs that read P^T / dS^T out of the buffer
  uint64_t* pds_full = s_free + kSBuf;          // [kSBuf] one per score buffer (see the dQ kernel)
  uint64_t* acc_full = pds_full + kSBuf;        // dV / dK accumulators of an item complete
  uint64_t* acc_free = acc_full + 1;            // ... and drained into registers by all 256 compute threads
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_free + 1);
  float* stat = reinterpret_cast<float*>(smem + DkvSmem::STAT);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nq64 = (T + 63) / 64;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQKV128);
    ptx::prefetch_tmap(&tmQKV64);
    ptx::prefetch_tmap(&tmDO64);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], 1);
    }
    for (int s = 0; s < kRing; ++s) {
      ptx::mbar_init(&qdo_full[s], 1);
      ptx::mbar_init(&qdo_empty[s], 1);
    }
    for (int s = 0; s < kSBuf; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&s_free[s], 1);
      ptx::mbar_init(&pds_full[s], 128);
    }
    ptx::mbar_init(acc_full, 1);
    ptx::mbar_init(acc_free, 256);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();               // everything above touched only this CTA's shared memory / TMEM
  const uint32_t tm_dV = tmem_base + 128 * kSBuf, tm_dK = tm_dV + 64;  // score buffer b: S^T at 128 b, dP^T at 128 b + 64

  // item -> key tile kt = rank (tile 0 sees every query tile: heaviest first); steps = 64-row query tiles from 2 kt on
  auto steps_of = [&](int it) { return nq64 - fdiv(it, fBH) * 2; };

  if (warp == 0) {
    {
      const bool issue = ptx::elect_one();  // whole warp runs the loop, one elected lane issues (uniform operands)
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_item(k, nitems);
        if (it < 0) break;
        const int kt = fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
        const int i0 = kt * 2, nq = steps_of(it);
        const int kb = k & 1;
        ptx::mbar_wait(&kv_empty[kb], ((k >> 1) & 1) ^ 1, 30);
        if (issue) ptx::mbar_expect_tx(&kv_full[kb], 32768);
        if (issue) ptx::tma_load_2d(smem + DkvSmem::KV + kb * 32768, &tmQKV128, &kv_full[kb], C + h * HS, b * T + kt * 128);
        if (issue) ptx::tma_load_2d(smem + DkvSmem::KV + kb * 32768 + 16384, &tmQKV128, &kv_full[kb], 2 * C + h * HS, b * T + kt * 128);
        for (int n = 0; n < nq; ++n, ++gs) {
          const int st = gs % kRing;
          ptx::mbar_wait(&qdo_empty[st], ((gs / kRing) & 1) ^ 1, 31);
          if (issue) ptx::mbar_expect_tx(&qdo_full[st], 16384);
          uint8_t* dst = smem + DkvSmem::QDO + st * 16384;
          if (issue) ptx::tma_load_2d(dst, &tmQKV64, &qdo_full[st], h * HS, b * T + (i0 + n) * 64);
          if (issue) ptx::tma_load_2d(dst + 8192, &tmDO64, &qdo_full[st], h * HS, b * T + (i0 + n) * 64);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---- score MMAs: S^T_n = K Q_n^T, dP^T_n = V dO_n^T into TMEM score buffer gs % kSBuf
    {
      const bool leader = ptx::elect_one();  // the whole warp runs this loop (uniform operands); one elected lane issues
      constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
      const uint64_t dKV0 = desc_k(ptx::smem_u32(smem + DkvSmem::KV), 0);
      const uint64_t dQDO0 = desc_k(ptx::smem_u32(smem + DkvSmem::QDO), 0);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_item(k, nitems);
        if (it < 0) break;
        const int nq = steps_of(it);
        const uint64_t dK0 = dKV0 + static_cast<uint64_t>((k & 1) * (32768 >> 4)), dV0 = dK0 + (16384 >> 4);
        ptx::mbar_wait(&kv_full[k & 1], (k >> 1) & 1, 32);
        for (int n = 0; n < nq; ++n, ++gs) {
          ptx::mbar_wait(&qdo_full[gs % kRing], (gs / kRing) & 1, 33);
          if (gs >= kSBuf) ptx::mbar_wait(&s_free[gs % kSBuf], ((gs / kSBuf) - 1) & 1, 34);  // dV / dK of step gs-3 have read it
          ptx::tc_fence_after();
          const uint64_t dQ = dQDO0 + static_cast<uint64_t>((gs % kRing) * (16384 >> 4)), dDO = dQ + (8192 >> 4);
          const uint32_t tS = tmem_base + (gs % kSBuf) * 128;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss(tS, dK0 + 2 * kk, dQ + 2 * kk, idesc_s, kk > 0);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss(tS + 64, dV0 + 2 * kk, dDO + 2 * kk, idesc_s, kk > 0);
          if (leader) ptx::umma_commit(&s_full[gs % kSBuf]);
        }
        if (leader) ptx::umma_commit(&kv_empty[k & 1]);  // all score MMAs of the item done: its K / V tiles may be overwritten
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    // ---- accumulating MMAs: dV += P^T_n dO_n, dK += dS^T_n Q_n
    {
      const bool leader = ptx::elect_one();  // the whole warp runs this loop (uniform operands); one elected lane issues
      constexpr uint32_t idesc_g = ptx::umma_idesc_bf16(128, 64, 0, 1);
      const uint64_t dQmn0 = desc_mn(ptx::smem_u32(smem + DkvSmem::QDO), 0);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_item(k, nitems);
        if (it < 0) break;
        const int nq = steps_of(it);
        if (k >= 1) {  // the previous item's dV / dK have been read out of TMEM
          ptx::mbar_wait(acc_free, (k - 1) & 1, 35);
          ptx::tc_fence_after();
        }
        for (int n = 0; n < nq; ++n, ++gs) {
          ptx::mbar_wait(&pds_full[gs % kSBuf], (gs / kSBuf) & 1, 36);
          ptx::tc_fence_after();
          const uint32_t tP = tmem_base + (gs % kSBuf) * 128, tDS = tP + 64;  // bf16 pairs written over the consumed scores
          const uint64_t dQ = dQmn0 + static_cast<uint64_t>((gs % kRing) * (16384 >> 4)), dDO = dQ + (8192 >> 4);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ts(tm_dV, tP + 8 * kk, dDO + (2048 >> 4) * kk, idesc_g, (n > 0 || kk > 0));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ts(tm_dK, tDS + 8 * kk, dQ + (2048 >> 4) * kk, idesc_g, (n > 0 || kk > 0));
          if (leader) ptx::umma_commit(&qdo_empty[gs % kRing]);
          if (leader) ptx::umma_commit(&s_free[gs % kSBuf]);
        }
        if (leader) ptx::umma_commit(acc_full);
      }
    }
    __syncwarp();
  } else {
    const int g = (warp - 2) >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;      // key row inside the tile
    const int tid = (warp - 2 - 4 * g) * 32 + lane;  // 0..127 within the group
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    // per-step column statistics (lse for threads 0..63, delta for threads 64..127 of the group): the RAW value of the
    // next own step is loaded one step ahead and scaled only when it is stored to shared memory, so the global-load
    // latency hides behind a whole step of arithmetic
    const float* stat_src = tid < 64 ? lse : delta;
    const float stat_coef = tid < 64 ? -kLog2e : -kScale;
    int ls_it = -2, ls_q = 0, ls_bh = 0;  // item decode cached across steps: two integer divisions per item, not per step
    const float* ls_row = stat_src;
    auto load_stat = [&](int it, int n) {
      float v = 0.f;
      if (it >= 0) {
        if (it != ls_it) {
          ls_it = it;
          ls_q = (fdiv(it, fBH)) * 128 + (tid & 63);
          ls_bh = fmodi(it, fBH);
          ls_row = stat_src + static_cast<long long>(ls_bh) * T;
        }
        const int qi = ls_q + n * 64;
        if (qi < T) v = __ldg(seq_shift >= kNoPack ? ls_row + qi : stat_src + stat_idx(fdiv(ls_bh, fH), fmodi(ls_bh, fH), qi, H, T, seq_shift));
      }
      return v;
    };
    // item epilogue: group 0 writes dV, group 1 writes dK; the accumulators are released once they sit in registers
    auto epilogue = [&](int k) {
      const int it = sched_item(k, nitems);
      const int kt = fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
      const int kv_t = kt * 128 + r;
      ptx::mbar_wait(acc_full, k & 1, 37);
      ptx::tc_fence_after();
      const uint32_t tm = (g == 0 ? tm_dV : tm_dK) + lane_off;
      uint32_t v0[32], v1[32];
      ptx::tmem_ld32(tm, v0);
      ptx::tmem_ld32(tm + 32, v1);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(acc_free);
      if (DROP && g == 0) {  // dV = (P o mask)^T dO / (1-p)
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          v0[i] = __float_as_uint(__uint_as_float(v0[i]) * dcfg.inv_keep);
          v1[i] = __float_as_uint(__uint_as_float(v1[i]) * dcfg.inv_keep);
        }
      }
      if (kv_t < T) {
        __nv_bfloat16* o = dqkv + static_cast<long long>(b * T + kv_t) * (3 * C) + (g == 0 ? 2 * C : C) + h * HS;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 w;
          w.x = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 0]), __uint_as_float(v0[8 * q + 1]));
          w.y = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 2]), __uint_as_float(v0[8 * q + 3]));
          w.z = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 4]), __uint_as_float(v0[8 * q + 5]));
          w.w = ptx::pack_bf16x2(__uint_as_float(v0[8 * q + 6]), __uint_as_float(v0[8 * q + 7]));
          reinterpret_cast<uint4*>(o)[q] = w;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 w;
          w.x = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 0]), __uint_as_float(v1[8 * q + 1]));
          w.y = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 2]), __uint_as_float(v1[8 * q + 3]));
          w.z = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 4]), __uint_as_float(v1[8 * q + 5]));
          w.w = ptx::pack_bf16x2(__uint_as_float(v1[8 * q + 6]), __uint_as_float(v1[8 * q + 7]));
          reinterpret_cast<uint4*>(o)[4 + q] = w;
        }
      }
    };
    // cursor over this group's steps (global step parity == g) and a look-ahead cursor one own step further
    int c_k = 0, c_it = sched_item(0, nitems), c_n = g, c_base = 0, c_nq = c_it >= 0 ? steps_of(c_it) : 0;
    auto normalize = [&](int& k, int& it, int& n, int& base, int& nq) {
      while (it >= 0 && n >= nq) {
        n -= nq;
        base += nq;
        ++k;
        it = sched_item(k, nitems);
        nq = it >= 0 ? steps_of(it) : 0;
      }
    };
    normalize(c_k, c_it, c_n, c_base, c_nq);
    int a_k = c_k, a_it = c_it, a_n = c_n + 2, a_base = c_base, a_nq = c_nq;
    normalize(a_k, a_it, a_n, a_base, a_nq);
    float raw_cur = load_stat(c_it, c_n);
    int ep_k = 0, use = 0, dec_k = -1;
    int kt = 0, bh = 0;
    while (c_it >= 0) {
      if (dec_k != c_k) {  // decode the item once
        kt = fdiv(c_it, fBH);
        bh = fmodi(c_it, fBH);
        dec_k = c_k;
      }
      const int kv_t = kt * 128 + r;
      const int r0 = kt * 128 + quarter * 32;
      const int q0 = (kt * 2 + c_n) * 64;
      const int gs = c_base + c_n;
      float* st_lse = stat + (g * 2 + (use & 1)) * 192;
      st_lse[tid] = raw_cur * stat_coef;
      if (DROP && tid < 64)
        st_lse[128 + tid] = __uint_as_float(
            drop_row_key(dcfg.key, static_cast<uint32_t>(stat_idx(fdiv(bh, fH), fmodi(bh, fH), q0 + tid, H, T, seq_shift))));
      raw_cur = load_stat(a_it, a_n);  // next own step: consumed at the top of the next iteration
      ptx::bar_sync(1 + g, 128);
      ptx::mbar_wait(&s_full[gs % kSBuf], (gs / kSBuf) & 1, 38);
      ptx::tc_fence_after();
      const uint32_t tbuf = tmem_base + lane_off + (gs % kSBuf) * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = q0 + c * 32;
        const uint32_t ta_s = tbuf + c * 32, ta_dp = ta_s + 64;
        const uint32_t l2 = ptx::smem_u32(st_lse) + c * 128, d8 = l2 + 256, rkeys = l2 + 512;
        uint32_t pk_p[16], pk_ds[16];
        const int kvr = real_col(kv_t, seq_shift);
        if (c0 + 31 < r0 || c0 >= T || !same_seq(c0, r0, seq_shift)) dkv_chunk<kMasked, DROP>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kvr);
        else if (c0 > r0 && c0 + 31 < T) dkv_chunk<kFull, DROP>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kvr);
        else dkv_chunk<kDiag, DROP>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kvr);
        // P^T / dS^T chunk c (32 query columns = 16 packed words each) overwrite score columns already consumed
        ptx::tmem_st16(tbuf + c * 16, pk_p);
        ptx::tmem_st16(tbuf + 64 + c * 16, pk_ds);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(&pds_full[gs % kSBuf]);
      ++use;
      // earlier items are drained AFTER this group's first step in a later item (their last MMAs wait for the other
      // group's final step; by now they have completed): the drain does not stall the step pipeline
      while (ep_k < c_k) epilogue(ep_k++);
      c_k = a_k; c_it = a_it; c_n = a_n; c_base = a_base; c_nq = a_nq;
      a_n += 2;
      normalize(a_k, a_it, a_n, a_base, a_nq);
    }
    while (ep_k < c_k) epilogue(ep_k++);  // c_k is now one past the last item of this CTA
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 512);
}

template <typename K>
int set_smem(K kern, int bytes) {
  ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  // two CTAs per SM need the full shared-memory carve-out
  ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return 0;
}

// sequences of 32 or 64 positions are packed to 128-row virtual sequences when the batch fills whole tiles (see kNoPack)
int pack_short(int& B, int& T) {
  if ((T == 32 || T == 64) && (static_cast<long long>(B) * T) % 128 == 0) {
    const int shift = T == 32 ? 5 : 6;
    B = static_cast<int>(static_cast<long long>(B) * T / 128);
    T = 128;
    return shift;
  }
  return kNoPack;
}

int check_shape(const char* who, int B, int T, int H) {
  ABCGPT_CHECK_ARG(B > 0 && T > 0 && H > 0, "%s: bad shape B=%d T=%d H=%d", who, B, T, H);
  ABCGPT_CHECK_ARG(static_cast<long long>(B) * H * ((T + 127) / 128) < (1ll << 30), "%s: too many (tile, batch*head) items", who);
  return 0;
}

}  // namespace

int attn_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, float drop_p, uint32_t drop_key,
             cudaStream_t stream) {
  int rc = check_shape("attn_fwd", B, T, H);
  if (rc) return rc;
  ABCGPT_CHECK_ARG(qkv && out && lse, "attn_fwd: null pointer");
  ABCGPT_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f, "attn_fwd: dropout p must be in [0, 1)");
  const int C = H * HS;
  const DropCfg dcfg = make_drop(drop_p, drop_key);
  const int seq_shift = pack_short(B, T);
  CUtensorMap tmQ, tmKV;
  if ((rc = encode_tmap_2d(&tmQ, qkv, 2, 3ull * C, static_cast<uint64_t>(B) * T, 3ull * C * 2, 64, 128, true))) return rc;
  if ((rc = encode_tmap_2d(&tmKV, qkv, 2, 3ull * C, static_cast<uint64_t>(B) * T, 3ull * C * 2, 64, 64, true))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = set_smem(attn_fwd_kernel<false>, FwdSmem::TOTAL))) return rc;
    if ((rc = set_smem(attn_fwd_kernel<true>, FwdSmem::TOTAL))) return rc;
    done = true;
  }
  const int BH = B * H, nitems = ((T + 127) / 128) * BH;
  const FastDiv fBH = make_fastdiv(static_cast<uint32_t>(BH), static_cast<uint64_t>(nitems)), fH = make_fastdiv(static_cast<uint32_t>(H), BH);
  const int grid = nitems < 2 * sm_count() ? nitems : 2 * sm_count();  // persistent: two CTAs per SM
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  // Three CTAs per SM with single-buffered S / O (csrc/attn_fwd3.cu) for sequences of >= 256 positions: 0.110 vs 0.120 ms per
  // layer at cfg3, 0.0196 vs 0.0205 ms at cfg2; packed short sequences (T = 32: 0.279 vs 0.273 ms at the cfg4 character level)
  // keep the two-CTA kernel.
  if (seq_shift == kNoPack && T >= 256)
    return attn_fwd3(tmQ, tmKV, out, lse, T, H, C, BH, nitems, dcfg, seq_shift, fBH.d, fBH.m, fH.d, fH.m, stream);
  if (dcfg.thr16 == 0)
    launch_k(attn_fwd_kernel<false>, dim3(grid), dim3(kThreads), FwdSmem::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, BH, nitems, dcfg,
             seq_shift, fBH, fH);
  else
    launch_k(attn_fwd_kernel<true>, dim3(grid), dim3(kThreads), FwdSmem::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, BH, nitems, dcfg,
             seq_shift, fBH, fH);
  return launch_status("attn_fwd_kernel");
}

int attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, int B,
             int T, int H, float drop_p, uint32_t drop_key, cudaStream_t stream) {
  int rc = check_shape("attn_bwd", B, T, H);
  if (rc) return rc;
  ABCGPT_CHECK_ARG(qkv && out && dout && lse && delta && dqkv, "attn_bwd: null pointer");
  ABCGPT_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f, "attn_bwd: dropout p must be in [0, 1)");
  const int C = H * HS;
  const DropCfg dcfg = make_drop(drop_p, drop_key);
  const int seq_shift = pack_short(B, T);
  const uint64_t rows = static_cast<uint64_t>(B) * T;
  CUtensorMap tmQKV128, tmQKV64, tmDO128, tmDO64;
  if ((rc = encode_tmap_2d(&tmQKV128, qkv, 2, 3ull * C, rows, 3ull * C * 2, 64, 128, true))) return rc;
  if ((rc = encode_tmap_2d(&tmQKV64, qkv, 2, 3ull * C, rows, 3ull * C * 2, 64, 64, true))) return rc;
  if ((rc = encode_tmap_2d(&tmDO128, dout, 2, static_cast<uint64_t>(C), rows, static_cast<uint64_t>(C) * 2, 64, 128, true))) return rc;
  if ((rc = encode_tmap_2d(&tmDO64, dout, 2, static_cast<uint64_t>(C), rows, static_cast<uint64_t>(C) * 2, 64, 64, true))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = set_smem(attn_bwd_dq_kernel<false>, DqSmem::TOTAL))) return rc;
    if ((rc = set_smem(attn_bwd_dq_kernel<true>, DqSmem::TOTAL))) return rc;
    if ((rc = set_smem(attn_bwd_dkv_kernel<false>, DkvSmem::TOTAL))) return rc;
    if ((rc = set_smem(attn_bwd_dkv_kernel<true>, DkvSmem::TOTAL))) return rc;
    done = true;
  }
  {
    const long long nrows = static_cast<long long>(B) * T;
    attn_delta_kernel<<<static_cast<int>((nrows + 7) / 8), 256, 0, stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(out), reinterpret_cast<const __nv_bfloat16*>(dout), delta, B, T, H, C, seq_shift);
    if ((rc = launch_status("attn_delta_kernel"))) return rc;
  }
  // CTA-pair kernels (csrc/attn_pair.cu) for sequences of >= 512 positions (at T = 256 a pair item has only 4 steps and the
  // single-CTA kernels are 10 % faster: 0.057 vs 0.063 ms at cfg2).
  if (seq_shift == kNoPack && T >= 512)
    return attn_bwd_pair(qkv, dout, lse, delta, dqkv, B, T, H, dcfg, stream);
  const int BH = B * H, nitems = ((T + 127) / 128) * BH;
  const FastDiv fBH = make_fastdiv(static_cast<uint32_t>(BH), static_cast<uint64_t>(nitems)), fH = make_fastdiv(static_cast<uint32_t>(H), BH);
  const int grid = nitems < sm_count() ? nitems : sm_count();  // persistent: one CTA per SM
  __nv_bfloat16* dq = reinterpret_cast<__nv_bfloat16*>(dqkv);
  if (dcfg.thr16 == 0) {
    launch_k(attn_bwd_dkv_kernel<false>, dim3(grid), dim3(kBwdThreads), DkvSmem::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, dq, T, H, C,
                                                                              BH, nitems, dcfg, seq_shift, fBH, fH);
    if ((rc = launch_status("attn_bwd_dkv_kernel"))) return rc;
    launch_k(attn_bwd_dq_kernel<false>, dim3(grid), dim3(kBwdThreads), DqSmem::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, dq, T, H, C,
                                                                            BH, nitems, dcfg, seq_shift, fBH, fH);
  } else {
    launch_k(attn_bwd_dkv_kernel<true>, dim3(grid), dim3(kBwdThreads), DkvSmem::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, dq, T, H, C,
                                                                             BH, nitems, dcfg, seq_shift, fBH, fH);
    if ((rc = launch_status("attn_bwd_dkv_kernel"))) return rc;
    launch_k(attn_bwd_dq_kernel<true>, dim3(grid), dim3(kBwdThreads), DqSmem::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, dq, T, H, C,
                                                                           BH, nitems, dcfg, seq_shift, fBH, fH);
  }
  return launch_status("attn_bwd_dq_kernel");
}

}  // namespace abcgpt
