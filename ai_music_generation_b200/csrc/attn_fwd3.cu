// Causal flash-attention forward, THREE CTAs per SM (head size 64) — an alternative schedule of csrc/attn.cu's forward kernel.
//
// Why.  A forward step (128 query rows x 64 keys) of the two-CTA kernel is ~1640 cycles of one CTA, of which ~1170 are the softmax
// (64 MUFU instructions per warp at the ~18 cycles each that two warps sharing a scheduler's MUFU get) and ~470-650 are latencies
// in which that CTA issues no MUFU work at all: the hand-over of P, the wait for the next S, tensor-memory round trips, loop
// bookkeeping (tools/attn_trace.py).  Measured this round: the time does not move when the per-thread work is halved (eight
// compute warps), nor when MUFU work is traded for FMA work (1/8, 1/4, 1/2 of the exponentials as polynomials), and the clean
// MUFU benchmark (tools/mufu2_bench.py) shows ONE warp per scheduler can saturate the unit (15.6 of 16 results per clock): the
// SM simply has too few independent instruction streams — with two CTAs both are regularly inside their gaps at once and the
// MUFU idles (62 % busy in steady state, 43 % over the kernel).  More resident CTAs is the cheap way to more streams, and what
// stops a third CTA is tensor memory: 2 x 64 columns of double-buffered S plus 2 x 64 of double-buffered O = 256 of 512.
//
// Here a CTA owns 128 columns: ONE S buffer and ONE O buffer.  The price is a longer chain inside the CTA — S_{j+1} can only be
// issued behind P_j V (the tensor pipe runs in order, so it overwrites P_j after the product has consumed it), and the O
// epilogue of an item runs at the item's end instead of behind the next item's first step — paid for by the other two CTAs
// filling those gaps.  Shared memory: Q double-buffered (2 x 16 KB) + a two-stage K|V ring (2 x 16 KB) = 64 KB per CTA.
// Everything a softmax thread computes is the code of the two-CTA kernel (csrc/attn_helpers.cuh), including dropout, packed
// short sequences and the lazy in-TMEM rescale.
// MEASURED (cfg3: 32 x 12 heads x 1024, per layer): 0.110 ms against 0.120 ms for the two-CTA kernel (465 vs 430 TFLOP/s of causal
// FLOPs) — the first change of the round that moved this kernel.
#include "attn_helpers.cuh"

namespace abcgpt {
namespace {

constexpr int kRing3 = 2;
struct Fwd3Smem {
  static constexpr int QB = 2;                       // Q buffers
  static constexpr int Q = 0;                        // QB items x (128 x 64 bf16)
  static constexpr int KV = QB * 16384;              // kRing3 stages x (K 64x64 | V 64x64)
  static constexpr int BAR = KV + kRing3 * 16384;
  static constexpr int TOTAL = BAR + 256 + 1024;
};

template <bool DROP>
__global__ void __launch_bounds__(kThreads, 3)
attn_fwd3_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                 __nv_bfloat16* __restrict__ out, float* __restrict__ lse, int T, int H, int C, int BH, int nitems,
                 const DropCfg dcfg, int seq_shift, const FastDiv fBH, const FastDiv fH) {
  using SM = Fwd3Smem;
  constexpr int QB = SM::QB;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::BAR);
  uint64_t* q_full = bars + 0;                  // [2]
  uint64_t* q_empty = bars + 2;                 // [2]
  uint64_t* kv_full = bars + 4;                 // [kRing3]
  uint64_t* kv_empty = kv_full + kRing3;        // [kRing3]
  uint64_t* s_full = kv_empty + kRing3;         // S_g complete            (phase g & 1)
  uint64_t* p_full = s_full + 1;                // P_g written, 128 arrivals
  uint64_t* pv_done = p_full + 1;               // P_g V landed in O
  uint64_t* o_full = pv_done + 1;               // item k's O complete     (phase k & 1)
  uint64_t* o_free = o_full + 1;                // item k's O drained, 128 arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_free + 1);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int nqt = (T + 127) / 128;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ);
    ptx::prefetch_tmap(&tmKV);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&q_full[s], 1);
      ptx::mbar_init(&q_empty[s], 1);
    }
    for (int s = 0; s < kRing3; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], 1);
    }
    ptx::mbar_init(s_full, 1);
    ptx::mbar_init(p_full, 128);
    ptx::mbar_init(pv_done, 1);
    ptx::mbar_init(o_full, 1);
    ptx::mbar_init(o_free, 128);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 128);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);  // S at columns [0, 64), O at [64, 128)
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();

  auto tiles_of = [&](int it) {
    const int qt = nqt - 1 - fdiv(it, fBH);
    return (min(T, qt * 128 + 128) + 63) / 64;
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    const bool issue = ptx::elect_one();
    int gt = 0;
    for (int item_k = 0;; ++item_k) {
      const int it = sched_item(item_k, nitems);
      if (it < 0) break;
      const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
      const int num_kv = tiles_of(it);
      const int qb = item_k % QB;
      ptx::mbar_wait(&q_empty[qb], ((item_k / QB) & 1) ^ 1, 30);
      if (issue) ptx::mbar_expect_tx(&q_full[qb], 16384);
      if (issue) ptx::tma_load_2d(smem + SM::Q + qb * 16384, &tmQ, &q_full[qb], h * HS, b * T + qt * 128);
      for (int j = 0; j < num_kv; ++j, ++gt) {
        const int st = gt % kRing3;
        ptx::mbar_wait(&kv_empty[st], ((gt / kRing3) & 1) ^ 1, 31);
        if (issue) ptx::mbar_expect_tx(&kv_full[st], 16384);
        uint8_t* dst = smem + SM::KV + st * 16384;
        if (issue) ptx::tma_load_2d(dst, &tmKV, &kv_full[st], C + h * HS, b * T + j * 64);
        if (issue) ptx::tma_load_2d(dst + 8192, &tmKV, &kv_full[st], 2 * C + h * HS, b * T + j * 64);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer: S_g, then (behind the softmax) P_g V, strictly alternating =====================
    const bool leader = ptx::elect_one();
    constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t idesc_o = ptx::umma_idesc_bf16(128, 64, 0, 1);
    const uint32_t sQ = ptx::smem_u32(smem + SM::Q);
    const uint32_t sKV = ptx::smem_u32(smem + SM::KV);
    const uint32_t tS = tmem_base, tO = tmem_base + 64;
    int gt = 0;
    for (int item_k = 0;; ++item_k) {
      const int it = sched_item(item_k, nitems);
      if (it < 0) break;
      const int num_kv = tiles_of(it);
      ptx::mbar_wait(&q_full[item_k % QB], (item_k / QB) & 1, 32);
      for (int j = 0; j < num_kv; ++j, ++gt) {
        const int st = gt % kRing3;
        ptx::mbar_wait(&kv_full[st], (gt / kRing3) & 1, 33);
        ptx::tc_fence_after();
        const uint32_t sQi = sQ + (item_k % QB) * 16384, sK = sKV + st * 16384, sV = sK + 8192;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ss(tS, desc_k(sQi, k), desc_k(sK, k), idesc_s, k > 0);
        if (leader) ptx::umma_commit(s_full);
        if (leader && j == num_kv - 1) ptx::umma_commit(&q_empty[item_k % QB]);  // last S of the item: its Q tile may be overwritten
        if (j == 0 && item_k >= 1) ptx::mbar_wait(o_free, (item_k - 1) & 1, 34);  // the previous item's O sits in registers
        ptx::mbar_wait(p_full, gt & 1, 35);
        ptx::tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k) if (leader) ptx::umma_ts(tO, tS + 8 * k, desc_mn(sV, k), idesc_o, (j > 0 || k > 0));
        if (leader) ptx::umma_commit(&kv_empty[st]);
        if (leader) ptx::umma_commit(pv_done);
        if (leader && j == num_kv - 1) ptx::umma_commit(o_full);
      }
    }
    __syncwarp();
  } else {
    // ===================== softmax / epilogue: one thread per query row =====================
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t tm_s = tmem_base + lane_off, tm_O = tmem_base + 64 + lane_off;
    int gt = 0;
    for (int item_k = 0;; ++item_k) {
      const int it = sched_item(item_k, nitems);
      if (it < 0) break;
      const int qt = nqt - 1 - fdiv(it, fBH), bh = fmodi(it, fBH), b = fdiv(bh, fH), h = fmodi(bh, fH);
      const int num_kv = tiles_of(it);
      const int r0 = qt * 128 + quarter * 32;
      float m_ref = 0.f, l = 0.f;
      bool have_ref = false;
      const uint32_t drop_rk = DROP ? drop_row_key(dcfg.key, static_cast<uint32_t>(stat_idx(b, h, qt * 128 + r, H, T, seq_shift))) : 0u;
      for (int j = 0; j < num_kv; ++j, ++gt) {
        const int c0 = j * 64, c1 = j * 64 + 32;
        const int cls0 = !same_seq(c0, r0, seq_shift) ? kMasked : ((c0 + 31 <= r0) ? kFull : ((c0 > r0 + 31) ? kMasked : kDiag));
        const int cls1 = !same_seq(c1, r0, seq_shift) ? kMasked : ((c1 + 31 <= r0) ? kFull : ((c1 > r0 + 31) ? kMasked : kDiag));
        ptx::mbar_wait(s_full, gt & 1, 36);
        ptx::tc_fence_after();
        uint32_t pk[32];
        float tmax = -1e30f, rowsum = 0.f;
        if (!have_ref && (cls0 != kMasked || cls1 != kMasked)) {
          have_ref = true;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int cls = c == 0 ? cls0 : cls1;
            if (cls == kFull) tmax = fmaxf(tmax, fwd_chunk_max<kFull>(tm_s + c * 32, lane));
            else if (cls == kDiag) tmax = fmaxf(tmax, fwd_chunk_max<kDiag>(tm_s + c * 32, lane));
          }
          m_ref = tmax * kSl2;
          fwd_tile<DROP>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, seq_shift);
        } else {
          fwd_tile<DROP>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, seq_shift);
          const bool need = tmax * kSl2 - m_ref > kRescaleThreshold;
          if (__any_sync(0xffffffffu, need)) {
            // rare: raise the reference, rescale the O accumulator in TMEM, recompute this tile's P
            const float m_new = need ? tmax * kSl2 : m_ref;
            const float alpha = ex2(m_ref - m_new);
            if (j > 0) {  // every earlier P V product of the item has landed in O (j == 0: nothing accumulated yet)
              ptx::mbar_wait(pv_done, (gt - 1) & 1, 37);
              ptx::tc_fence_after();
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                uint32_t o[32];
                ptx::tmem_ld32(tm_O + c * 32, o);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                ptx::tmem_st32(tm_O + c * 32, o);
              }
              ptx::tmem_st_wait();
            }
            l *= alpha;
            m_ref = m_new;
            tmax = -1e30f;
            rowsum = 0.f;
            fwd_tile<DROP>(tm_s, lane, cls0, cls1, -m_ref, tmax, rowsum, pk, dcfg, drop_rk, j * 64, seq_shift);
          }
        }
        l += rowsum;
        ptx::tmem_st16(tm_s, pk);
        ptx::tmem_st16(tm_s + 16, pk + 16);
        ptx::tmem_st_wait();
        ptx::tc_fence_before();
        ptx::mbar_arrive(p_full);
      }
      // item epilogue: O / l -> bf16, LSE; the O buffer is released as soon as it sits in registers
      ptx::mbar_wait(o_full, item_k & 1, 38);
      ptx::tc_fence_after();
      uint32_t v0[32], v1[32];
      ptx::tmem_ld32(tm_O, v0);
      ptx::tmem_ld32(tm_O + 32, v1);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(o_free);
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
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 128);
}

}  // namespace

// Three-CTA-per-SM schedule of the attention forward; same contract as the launch inside attn_fwd (csrc/attn.cu), which
// dispatches here.
int attn_fwd3(const CUtensorMap& tmQ, const CUtensorMap& tmKV, void* out, float* lse, int T, int H, int C, int BH, int nitems,
              const DropCfg& dcfg, int seq_shift, uint32_t fBH_d, uint32_t fBH_m, uint32_t fH_d, uint32_t fH_m, cudaStream_t stream) {
  const FastDiv fBH{fBH_d, fBH_m}, fH{fH_d, fH_m};   // FastDiv lives in each translation unit's anonymous namespace
  static bool done = false;
  if (!done) {
    ABCGPT_CUDA(cudaFuncSetAttribute(attn_fwd3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Fwd3Smem::TOTAL));
    ABCGPT_CUDA(cudaFuncSetAttribute(attn_fwd3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Fwd3Smem::TOTAL));
    done = true;
  }
  const int grid = nitems < 3 * sm_count() ? nitems : 3 * sm_count();  // persistent: three CTAs per SM
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  if (dcfg.thr16 == 0)
    launch_k(attn_fwd3_kernel<false>, dim3(grid), dim3(kThreads), Fwd3Smem::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, BH, nitems, dcfg,
             seq_shift, fBH, fH);
  else
    launch_k(attn_fwd3_kernel<true>, dim3(grid), dim3(kThreads), Fwd3Smem::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, BH, nitems, dcfg,
             seq_shift, fBH, fH);
  return launch_status("attn_fwd3_kernel");
}

}  // namespace abcgpt
