// Causal flash-attention backward on CTA PAIRS (tcgen05.mma.cta_group::2), head size 64 — the kernels behind
// abcgpt_attn_bwd for sequences of at least 256 positions (nanoGPT/model.py:64 backward; the single-CTA kernels of csrc/attn.cu
// keep serving short and packed sequences).
//
// Why pairs: every MMA of a head-size-64 attention step has N = 64, and a single-CTA 128x64x16 tcgen05.mma costs 74 cycles for
// 32 cycles of math whatever the operand source, while the pair form 256x64x16 costs 43 cycles for BOTH CTAs' rows
// (tools/mma_bench.py): 3.4x the MMA throughput per unit of attention work.  The single-CTA backward kernels sat on that issue
// floor (1184 + 888 tensor-pipe cycles per 128x64 block over the two kernels).
//
// One cluster of two CTAs works on TWO adjacent 128-row tiles of one (batch, head) in lockstep and streams the other operand
// in 64-row tiles that both CTAs share:
//   attn_bwd_dkv2_kernel  pair item = key tiles (2p, 2p+1); streams Q / dO tiles.  Per step, M = 256 keys:
//        S^T  = K  Q^T      A = K  (own 128 rows, smem)   B = Q  rows  [32r, 32r+32) of the 64-row tile, K-major
//        dP^T = V  dO^T     A = V                         B = dO rows  (same split)
//        dV  += P^T  dO     A = P^T  (own TMEM)           B = dO columns [32r, 32r+32): 64 x 32 slab, MN-major, 64-byte swizzle
//        dK  += dS^T Q      A = dS^T (own TMEM)           B = Q  columns (same split)
//   attn_bwd_dq2_kernel   pair item = query tiles (2p, 2p+1); streams K / V tiles.  Per step, M = 256 queries:
//        S  = Q  K^T, dP = dO V^T   (B = K / V row halves),     dQ += dS K   (A = dS in TMEM, B = K column halves)
// B of a cta_group::2 MMA is split by N between the CTAs, so each CTA stages HALF of every streamed tile (in the two layouts
// the two MMA families need): the L2 -> shared-memory traffic per unit of work is half of the single-CTA kernels'.
// The leader CTA (cluster rank 0) issues every MMA; barrier protocol as in the pair GEMM (csrc/gemm.cu): "full" barriers live
// in the leader and collect the TMA bytes of both CTAs, "written / drained" barriers in the leader collect one arrival per
// compute warp of both CTAs (remote mbarrier.arrive), every tcgen05.commit is multicast to the CTAs that wait for it.
// Everything a compute thread does (statistics, masks, dropout, exp2, packing, TMEM write-back, epilogues) is the code of the
// single-CTA kernels (csrc/attn_helpers.cuh); a tile that lies entirely above the diagonal for one CTA of the pair (the first
// two query steps of the upper key tile, the last two key steps of the lower query tile) takes the "masked" chunk class there.
#include "attn_helpers.cuh"

namespace abcgpt {
namespace {

constexpr int kSBuf = 3;          // S/dP score buffers in TMEM (as in csrc/attn.cu)
constexpr int kRing = 6;          // streamed tiles in flight
// Thread layout: warp 0 TMA, warp 1 score MMAs, warps 2 .. 4 NG + 1 compute, warp 4 NG + 2 accumulating MMAs.  The compute
// warps form NG STEP GROUPS of four (one warp per tensor-memory lane quarter): group g owns the steps gs with gs % NG == g, and a
// thread owns one row and all 64 columns of each of its steps.  The dK/dV kernel alternates two groups over the three score
// buffers (the issuer runs one step ahead).  The dQ kernel gives every score buffer its own group: a third independent
// instruction stream per SM for the latency gaps of the other two (the forward gains from a third resident CTA for the same
// reason, csrc/attn_fwd3.cu).  More warps per step do not pay: with eight compute warps the steady state already runs at
// 80-90 % of the MUFU (ex2) rate, and splitting a step's columns over more warps only adds per-step barrier traffic.  In the dQ
// kernel each group idles ~60 % of its cycle (3 x 1050 cycles per own step against ~1250 of arithmetic): the score / accumulate
// MMA chain and its operand re-reads (Q and dO, 4 KB each per MMA, are the shared-memory-bound A operands of eight of the
// twelve MMAs of a step) are the next thing to look at.
template <int NG> struct PairCfg {
  static constexpr int kCompWarps = 4 * NG;
  static constexpr int kAccWarp = 2 + kCompWarps;
  static constexpr int kThreads = (kAccWarp + 1) * 32;
};
using DkvCfg = PairCfg<2>;   // 352 threads
using DqCfg = PairCfg<3>;    // 480 threads

// static schedule over PAIR items: pair c of G walks items c, 2G-1-c, 2G+c, ... (heaviest first, boustrophedon)
__device__ __forceinline__ int sched_pair_item(int k, int nitems) {
  const int G = gridDim.x >> 1, c = blockIdx.x >> 1;
  const int i = k * G + ((k & 1) ? G - 1 - c : c);
  return i < nitems ? i : -1;
}
// MN-major B operand, column half of a 64-row tile: [64 k-rows x 32 n] slab with 64-byte rows and SWIZZLE_64B; one MMA
// (K = 16) covers 16 rows = 1024 bytes, 8-row groups are 512 bytes apart, the 32 columns are one MN atom
__device__ __forceinline__ uint64_t desc_mn64(uint32_t slab_addr, int k16) {
  return ptx::umma_smem_desc_lt(slab_addr + k16 * 1024, 512, 512, 4);
}
// one arrival per warp on a barrier of the pair's leader CTA, after every lane's tensor-memory traffic has completed
__device__ __forceinline__ void warp_arrive_leader(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(bar), 0));
}

// ======================================================================================================
// dK / dV
// ======================================================================================================
struct Dkv2Smem {
  static constexpr int KV = 0;         // 2 items x (K 128x64 | V 128x64), this CTA's key tile
  static constexpr int QDO = 65536;    // kRing stages x (Q rows-half 32x64 | dO rows-half | Q cols-half 64x32 | dO cols-half)
  static constexpr int STAT = QDO + kRing * 16384;  // 2 groups x 2 buffers x (-lse2[64] | -delta8[64] | dropout row key[64])
  static constexpr int BAR = STAT + 3072;
  static constexpr int TOTAL = BAR + 512 + 1024;
};

template <bool DROP>
__global__ void __launch_bounds__(DkvCfg::kThreads, 1)
attn_bwd_dkv2_kernel(const __grid_constant__ CUtensorMap tmKV128, const __grid_constant__ CUtensorMap tmQ32,
                     const __grid_constant__ CUtensorMap tmDO32, const __grid_constant__ CUtensorMap tmQc,
                     const __grid_constant__ CUtensorMap tmDOc, const float* __restrict__ lse, const float* __restrict__ delta,
                     __nv_bfloat16* __restrict__ dqkv, int T, int H, int C, int BH, int nitems, const DropCfg dcfg,
                     const FastDiv fBH, const FastDiv fH) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Dkv2Smem::BAR);
  uint64_t* kv_full = bars + 0;                 // [2]      leader: TMA bytes of both CTAs
  uint64_t* kv_empty = bars + 2;                // [2]      each CTA: multicast commit
  uint64_t* qdo_full = bars + 4;                // [kRing]  leader
  uint64_t* qdo_empty = qdo_full + kRing;       // [kRing]  each CTA
  uint64_t* s_full = qdo_empty + kRing;         // [kSBuf]  each CTA
  uint64_t* s_free = s_full + kSBuf;            // [kSBuf]  leader
  uint64_t* pds_full = s_free + kSBuf;          // [kSBuf]  leader: 8 warps x 2 CTAs
  uint64_t* acc_full = pds_full + kSBuf;        //          each CTA
  uint64_t* acc_free = acc_full + 1;            //          leader: 16 warps x 2 CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_free + 1);
  float* stat = reinterpret_cast<float*>(smem + Dkv2Smem::STAT);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int rank = static_cast<int>(ptx::cluster_ctarank());
  const bool leader_cta = rank == 0;
  const int nq64 = (T + 63) / 64;
  constexpr int seq_shift = kNoPack;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmKV128);
    ptx::prefetch_tmap(&tmQ32);
    ptx::prefetch_tmap(&tmDO32);
    ptx::prefetch_tmap(&tmQc);
    ptx::prefetch_tmap(&tmDOc);
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
      ptx::mbar_init(&pds_full[s], 2 * 4);
    }
    ptx::mbar_init(acc_full, 1);
    ptx::mbar_init(acc_free, 2 * DkvCfg::kCompWarps);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, 512);
    ptx::tmem_relinquish_2sm();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // barrier inits + TMEM allocations of BOTH CTAs are visible before anything is signalled
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const uint32_t tm_dV = tmem_base + 128 * kSBuf, tm_dK = tm_dV + 64;  // score buffer b: S^T at 128 b, dP^T at 128 b + 64

  // pair item -> key tiles (2 p, 2 p + 1), p = it / BH (pair 0 sees every query tile: heaviest first); steps = 64-row query
  // tiles from the first key of the pair on
  auto steps_of = [&](int it) { return nq64 - fdiv(it, fBH) * 4; };

  if (warp == 0) {
    {
      const bool issue = ptx::elect_one();  // whole warp runs the loop, one elected lane issues (uniform operands)
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_pair_item(k, nitems);
        if (it < 0) break;
        int p, bh, b, h;
        fdivmod(it, fBH, p, bh);
        fdivmod(bh, fH, b, h);
        const int kt = 2 * p + rank, i0 = 4 * p, nq = nq64 - 4 * p;
        const int kb = k & 1;
        ptx::mbar_wait(&kv_empty[kb], ((k >> 1) & 1) ^ 1, 60);
        const uint32_t kvf = ptx::mapa(ptx::smem_u32(&kv_full[kb]), 0);
        if (leader_cta && issue) ptx::mbar_expect_tx(&kv_full[kb], 2 * 32768);
        if (issue) ptx::tma_load_2d_2sm(smem + Dkv2Smem::KV + kb * 32768, &tmKV128, kvf, C + h * HS, b * T + kt * 128);
        if (issue) ptx::tma_load_2d_2sm(smem + Dkv2Smem::KV + kb * 32768 + 16384, &tmKV128, kvf, 2 * C + h * HS, b * T + kt * 128);
        for (int n = 0; n < nq; ++n, ++gs) {
          const int st = gs % kRing;
          ptx::mbar_wait(&qdo_empty[st], ((gs / kRing) & 1) ^ 1, 61);
          const uint32_t qf = ptx::mapa(ptx::smem_u32(&qdo_full[st]), 0);
          if (leader_cta && issue) ptx::mbar_expect_tx(&qdo_full[st], 2 * 16384);
          uint8_t* dst = smem + Dkv2Smem::QDO + st * 16384;
          const int row = b * T + (i0 + n) * 64;
          if (issue) ptx::tma_load_2d_2sm(dst, &tmQ32, qf, h * HS, row + 32 * rank);
          if (issue) ptx::tma_load_2d_2sm(dst + 4096, &tmDO32, qf, h * HS, row + 32 * rank);
          if (issue) ptx::tma_load_2d_2sm(dst + 8192, &tmQc, qf, h * HS + 32 * rank, row);
          if (issue) ptx::tma_load_2d_2sm(dst + 12288, &tmDOc, qf, h * HS + 32 * rank, row);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---- score MMAs (leader CTA): S^T_n = K Q_n^T, dP^T_n = V dO_n^T for both key tiles into score buffer gs % kSBuf
    if (leader_cta) {
      const bool leader = ptx::elect_one();
      constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(256, 64, 0, 0);
      const uint64_t dKV0 = desc_k(ptx::smem_u32(smem + Dkv2Smem::KV), 0);
      const uint64_t dQDO0 = desc_k(ptx::smem_u32(smem + Dkv2Smem::QDO), 0);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_pair_item(k, nitems);
        if (it < 0) break;
        const int nq = steps_of(it);
        const uint64_t dK0 = dKV0 + static_cast<uint64_t>((k & 1) * (32768 >> 4)), dV0 = dK0 + (16384 >> 4);
        ptx::mbar_wait(&kv_full[k & 1], (k >> 1) & 1, 62);
        for (int n = 0; n < nq; ++n, ++gs) {
          ptx::mbar_wait(&qdo_full[gs % kRing], (gs / kRing) & 1, 63);
          if (gs >= kSBuf) ptx::mbar_wait(&s_free[gs % kSBuf], ((gs / kSBuf) - 1) & 1, 64);  // dV / dK of step gs-3 have read it
          ptx::tc_fence_after();
          const uint64_t dQ = dQDO0 + static_cast<uint64_t>((gs % kRing) * (16384 >> 4)), dDO = dQ + (4096 >> 4);
          const uint32_t tS = tmem_base + (gs % kSBuf) * 128;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss_2sm(tS, dK0 + 2 * kk, dQ + 2 * kk, idesc_s, kk > 0);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss_2sm(tS + 64, dV0 + 2 * kk, dDO + 2 * kk, idesc_s, kk > 0);
          if (leader) ptx::umma_commit_2sm(&s_full[gs % kSBuf], 0x3);
        }
        if (leader) ptx::umma_commit_2sm(&kv_empty[k & 1], 0x3);  // all score MMAs of the item done: K / V may be overwritten
      }
    }
    __syncwarp();
  } else if (warp == DkvCfg::kAccWarp) {
    // ---- accumulating MMAs (leader CTA): dV += P^T_n dO_n, dK += dS^T_n Q_n
    if (leader_cta) {
      const bool leader = ptx::elect_one();
      constexpr uint32_t idesc_g = ptx::umma_idesc_bf16(256, 64, 0, 1);
      const uint32_t sQDO = ptx::smem_u32(smem + Dkv2Smem::QDO);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_pair_item(k, nitems);
        if (it < 0) break;
        const int nq = steps_of(it);
        if (k >= 1) {  // the previous item's dV / dK have been read out of BOTH CTAs' tensor memory
          ptx::mbar_wait(acc_free, (k - 1) & 1, 65);
          ptx::tc_fence_after();
        }
        for (int n = 0; n < nq; ++n, ++gs) {
          ptx::mbar_wait(&pds_full[gs % kSBuf], (gs / kSBuf) & 1, 66);
          ptx::tc_fence_after();
          const uint32_t tP = tmem_base + (gs % kSBuf) * 128, tDS = tP + 64;  // bf16 pairs written over consumed scores (see below)
          const uint64_t dQc = desc_mn64(sQDO + (gs % kRing) * 16384 + 8192, 0), dDOc = dQc + (4096 >> 4);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)  // queries [16 kk, 16 kk + 16): 8 packed words at column (kk / 2) * 32 + (kk % 2) * 8
            if (leader) ptx::umma_ts_2sm(tm_dV, tP + (kk >> 1) * 32 + (kk & 1) * 8, dDOc + (1024 >> 4) * kk, idesc_g, (n > 0 || kk > 0));
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            if (leader) ptx::umma_ts_2sm(tm_dK, tDS + (kk >> 1) * 32 + (kk & 1) * 8, dQc + (1024 >> 4) * kk, idesc_g, (n > 0 || kk > 0));
          if (leader) ptx::umma_commit_2sm(&qdo_empty[gs % kRing], 0x3);
          if (leader) ptx::umma_commit_2sm(&s_free[gs % kSBuf], 0x1);
        }
        if (leader) ptx::umma_commit_2sm(acc_full, 0x3);
      }
    }
    __syncwarp();
  } else {
    const int cw = warp - 2;                // 0 .. 7
    const int sg = cw / 4;                  // step group: owns the steps of parity sg
    const int quarter = warp & 3;           // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;      // key row inside this CTA's tile
    const int tid = (cw % 4) * 32 + lane;   // 0 .. 127 within the step group
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    // per-step column statistics: threads 0..63 of the step group stage -lse*log2e and the dropout row keys, 64..127
    // -delta*scale, of the step's 64 queries; the RAW value of the next own step is loaded one step ahead
    const int stat_role = tid >> 6;         // 0: lse and dropout row keys, 1: delta
    const float* stat_src = stat_role == 0 ? lse : delta;
    const float stat_coef = stat_role == 0 ? -kLog2e : -kScale;
    int ls_it = -2, ls_q = 0;
    const float* ls_row = stat_src;
    auto load_stat = [&](int it, int n) {
      float v = 0.f;
      if (it >= 0) {
        if (it != ls_it) {
          int p_, bh_;
          fdivmod(it, fBH, p_, bh_);
          ls_it = it;
          ls_q = p_ * 256 + (tid & 63);
          ls_row = stat_src + static_cast<long long>(bh_) * T;
        }
        const int qi = ls_q + n * 64;
        if (qi < T) v = __ldg(ls_row + qi);
      }
      return v;
    };
    // item epilogue: step group 0 writes dV, step group 1 dK; each thread the 64 columns of its key row
    auto epilogue = [&](int k) {
      const int it = sched_pair_item(k, nitems);
      int p_, bh_, b, h;
      fdivmod(it, fBH, p_, bh_);
      fdivmod(bh_, fH, b, h);
      const int kv_t = (2 * p_ + rank) * 128 + r;
      ptx::mbar_wait(acc_full, k & 1, 67);
      ptx::tc_fence_after();
      uint32_t v[2][32];
#pragma unroll
      for (int c = 0; c < 2; ++c) ptx::tmem_ld32((sg == 0 ? tm_dV : tm_dK) + lane_off + c * 32, v[c]);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      warp_arrive_leader(acc_free, lane);
      if (kv_t < T) {
        const float sc = (DROP && sg == 0) ? dcfg.inv_keep : 1.0f;  // dV = (P o mask)^T dO / (1-p)
        __nv_bfloat16* o = dqkv + static_cast<long long>(b * T + kv_t) * (3 * C) + (sg == 0 ? 2 * C : C) + h * HS;
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 w;
            w.x = ptx::pack_bf16x2(__uint_as_float(v[c][8 * q + 0]) * sc, __uint_as_float(v[c][8 * q + 1]) * sc);
            w.y = ptx::pack_bf16x2(__uint_as_float(v[c][8 * q + 2]) * sc, __uint_as_float(v[c][8 * q + 3]) * sc);
            w.z = ptx::pack_bf16x2(__uint_as_float(v[c][8 * q + 4]) * sc, __uint_as_float(v[c][8 * q + 5]) * sc);
            w.w = ptx::pack_bf16x2(__uint_as_float(v[c][8 * q + 6]) * sc, __uint_as_float(v[c][8 * q + 7]) * sc);
            reinterpret_cast<uint4*>(o)[4 * c + q] = w;
          }
      }
    };
    // cursor over this step group's steps (global step parity == sg) and a look-ahead cursor one own step further
    int c_k = 0, c_it = sched_pair_item(0, nitems), c_n = sg, c_base = 0, c_nq = c_it >= 0 ? steps_of(c_it) : 0;
    auto normalize = [&](int& k, int& it, int& n, int& base, int& nq) {
      while (it >= 0 && n >= nq) {
        n -= nq;
        base += nq;
        ++k;
        it = sched_pair_item(k, nitems);
        nq = it >= 0 ? steps_of(it) : 0;
      }
    };
    normalize(c_k, c_it, c_n, c_base, c_nq);
    int a_k = c_k, a_it = c_it, a_n = c_n + 2, a_base = c_base, a_nq = c_nq;
    normalize(a_k, a_it, a_n, a_base, a_nq);
    float raw_cur = load_stat(c_it, c_n);
    int ep_k = 0, use = 0, dec_k = -1;
    int p = 0, bh = 0, hb = 0, hh = 0;
    while (c_it >= 0) {
      if (dec_k != c_k) {  // decode the item once
        fdivmod(c_it, fBH, p, bh);
        if (DROP) fdivmod(bh, fH, hb, hh);
        dec_k = c_k;
      }
      const int kt = 2 * p + rank;
      const int kv_t = kt * 128 + r;
      const int r0 = kt * 128 + quarter * 32;
      const int q0 = (4 * p + c_n) * 64;
      const int gs = c_base + c_n;
      float* st_lse = stat + (sg * 2 + (use & 1)) * 192;
      st_lse[tid] = raw_cur * stat_coef;
      if (DROP && stat_role == 0)
        st_lse[128 + (tid & 63)] = __uint_as_float(drop_row_key(dcfg.key, static_cast<uint32_t>(stat_idx(hb, hh, q0 + (tid & 63), H, T, seq_shift))));
      raw_cur = load_stat(a_it, a_n);  // next own step: consumed at the top of the next iteration
      ptx::bar_sync(1 + sg, 128);
      ptx::mbar_wait(&s_full[gs % kSBuf], (gs / kSBuf) & 1, 68);
      ptx::tc_fence_after();
      const uint32_t tbuf = tmem_base + lane_off + (gs % kSBuf) * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = q0 + c * 32;
        const uint32_t ta_s = tbuf + c * 32, ta_dp = ta_s + 64;
        const uint32_t l2 = ptx::smem_u32(st_lse) + c * 128, d8 = l2 + 256, rkeys = l2 + 512;
        uint32_t pk_p[16], pk_ds[16];
        if (c0 + 31 < r0 || c0 >= T) dkv_chunk<kMasked, DROP>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kv_t);
        else if (c0 > r0 && c0 + 31 < T) dkv_chunk<kFull, DROP>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kv_t);
        else dkv_chunk<kDiag, DROP>(ta_s, ta_dp, l2, d8, c0, kv_t, T, pk_p, pk_ds, dcfg, rkeys, kv_t);
        // P^T / dS^T of column half c (16 packed words each) go over the score columns that were just consumed: S^T columns
        // [32 c, 32 c + 16) and dP^T columns [64 + 32 c, ...) — never into the other half's inputs.  The A operand of the
        // accumulating MMAs is two runs of 16 words 32 columns apart.
        ptx::tmem_st16(tbuf + c * 32, pk_p);
        ptx::tmem_st16(tbuf + 64 + c * 32, pk_ds);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      warp_arrive_leader(&pds_full[gs % kSBuf], lane);
      ++use;
      // earlier items are drained AFTER this group's first step in a later item (their last MMAs have completed by now)
      while (ep_k < c_k) epilogue(ep_k++);
      c_k = a_k; c_it = a_it; c_n = a_n; c_base = a_base; c_nq = a_nq;
      a_n += 2;
      normalize(a_k, a_it, a_n, a_base, a_nq);
    }
    while (ep_k < c_k) epilogue(ep_k++);  // c_k is now one past the last item of this pair
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // the peer may still be arriving on this CTA's barriers / reading its shared memory
  if (warp == 1) ptx::tmem_dealloc_2sm(tmem_base, 512);
}

// ======================================================================================================
// dQ
// ======================================================================================================
struct Dq2Smem {
  static constexpr int QDO = 0;       // 2 items x (Q 128x64 | dO 128x64), this CTA's query tile
  static constexpr int KV = 65536;    // kRing stages x (K rows-half 32x64 | V rows-half 32x64 | K cols-half 64x32 | unused)
  static constexpr int BAR = KV + kRing * 16384;
  static constexpr int TOTAL = BAR + 512 + 1024;
};

template <bool DROP>
__global__ void __launch_bounds__(DqCfg::kThreads, 1)
attn_bwd_dq2_kernel(const __grid_constant__ CUtensorMap tmQ128, const __grid_constant__ CUtensorMap tmDO128,
                    const __grid_constant__ CUtensorMap tmKV32, const __grid_constant__ CUtensorMap tmKc,
                    const float* __restrict__ lse, const float* __restrict__ delta, __nv_bfloat16* __restrict__ dqkv, int T,
                    int H, int C, int BH, int nitems, const DropCfg dcfg, const FastDiv fBH, const FastDiv fH) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Dq2Smem::BAR);
  uint64_t* qdo_full = bars + 0;                // [2]      leader
  uint64_t* qdo_empty = bars + 2;               // [2]      each CTA
  uint64_t* kv_full = bars + 4;                 // [kRing]  leader
  uint64_t* kv_empty = kv_full + kRing;         // [kRing]  each CTA
  uint64_t* s_full = kv_empty + kRing;          // [kSBuf]  each CTA
  uint64_t* s_free = s_full + kSBuf;            // [kSBuf]  leader
  uint64_t* ds_full = s_free + kSBuf;           // [kSBuf]  leader: 8 warps x 2 CTAs
  uint64_t* acc_full = ds_full + kSBuf;         // [2]      each CTA
  uint64_t* acc_free = acc_full + 2;            // [2]      leader: 16 warps x 2 CTAs
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_free + 2);

  const int warp = ptx::uniform(threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int rank = static_cast<int>(ptx::cluster_ctarank());
  const bool leader_cta = rank == 0;
  const int npt = (T + 255) / 256;   // query tile pairs per sequence
  constexpr int seq_shift = kNoPack;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ128);
    ptx::prefetch_tmap(&tmDO128);
    ptx::prefetch_tmap(&tmKV32);
    ptx::prefetch_tmap(&tmKc);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&qdo_full[s], 1);
      ptx::mbar_init(&qdo_empty[s], 1);
      ptx::mbar_init(&acc_full[s], 1);
      ptx::mbar_init(&acc_free[s], 2 * DqCfg::kCompWarps);
    }
    for (int s = 0; s < kRing; ++s) {
      ptx::mbar_init(&kv_full[s], 1);
      ptx::mbar_init(&kv_empty[s], 1);
    }
    for (int s = 0; s < kSBuf; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&s_free[s], 1);
      ptx::mbar_init(&ds_full[s], 2 * 4);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, 512);
    ptx::tmem_relinquish_2sm();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::uniform(*tmem_slot);
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const uint32_t tm_dQ = tmem_base + 128 * kSBuf;  // score buffer b: S at 128 b, dP at 128 b + 64; dQ buffers at 384, 448

  // pair item -> query tiles (2 p, 2 p + 1), p = npt - 1 - it / BH (heaviest first); steps = 64-row key tiles up to the
  // last key the upper query tile sees
  auto tiles_of = [&](int it) {
    const int p = npt - 1 - fdiv(it, fBH);
    return (min(T, p * 256 + 256) + 63) / 64;
  };

  if (warp == 0) {
    {
      const bool issue = ptx::elect_one();
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_pair_item(k, nitems);
        if (it < 0) break;
        int pr, bh, b, h;
        fdivmod(it, fBH, pr, bh);
        fdivmod(bh, fH, b, h);
        const int p = npt - 1 - pr;
        const int num_kv = (min(T, p * 256 + 256) + 63) / 64, row0 = b * T + (2 * p + rank) * 128;
        const int qb = k & 1;
        ptx::mbar_wait(&qdo_empty[qb], ((k >> 1) & 1) ^ 1, 70);
        const uint32_t qf = ptx::mapa(ptx::smem_u32(&qdo_full[qb]), 0);
        if (leader_cta && issue) ptx::mbar_expect_tx(&qdo_full[qb], 2 * 32768);
        if (issue) ptx::tma_load_2d_2sm(smem + Dq2Smem::QDO + qb * 32768, &tmQ128, qf, h * HS, row0);
        if (issue) ptx::tma_load_2d_2sm(smem + Dq2Smem::QDO + qb * 32768 + 16384, &tmDO128, qf, h * HS, row0);
        for (int j = 0; j < num_kv; ++j, ++gs) {
          const int st = gs % kRing;
          ptx::mbar_wait(&kv_empty[st], ((gs / kRing) & 1) ^ 1, 71);
          const uint32_t kf = ptx::mapa(ptx::smem_u32(&kv_full[st]), 0);
          if (leader_cta && issue) ptx::mbar_expect_tx(&kv_full[st], 2 * 12288);
          uint8_t* dst = smem + Dq2Smem::KV + st * 16384;
          const int row = b * T + j * 64;
          if (issue) ptx::tma_load_2d_2sm(dst, &tmKV32, kf, C + h * HS, row + 32 * rank);
          if (issue) ptx::tma_load_2d_2sm(dst + 4096, &tmKV32, kf, 2 * C + h * HS, row + 32 * rank);
          if (issue) ptx::tma_load_2d_2sm(dst + 8192, &tmKc, kf, C + h * HS + 32 * rank, row);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---- score MMAs (leader CTA): S_j = Q K_j^T, dP_j = dO V_j^T for both query tiles
    if (leader_cta) {
      const bool leader = ptx::elect_one();
      constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(256, 64, 0, 0);
      const uint64_t dQDO0 = desc_k(ptx::smem_u32(smem + Dq2Smem::QDO), 0);
      const uint64_t dKV0 = desc_k(ptx::smem_u32(smem + Dq2Smem::KV), 0);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_pair_item(k, nitems);
        if (it < 0) break;
        const int num_kv = tiles_of(it);
        const uint64_t dQ0 = dQDO0 + static_cast<uint64_t>((k & 1) * (32768 >> 4)), dDO0 = dQ0 + (16384 >> 4);
        ptx::mbar_wait(&qdo_full[k & 1], (k >> 1) & 1, 72);
        for (int j = 0; j < num_kv; ++j, ++gs) {
          ptx::mbar_wait(&kv_full[gs % kRing], (gs / kRing) & 1, 73);
          if (gs >= kSBuf) ptx::mbar_wait(&s_free[gs % kSBuf], ((gs / kSBuf) - 1) & 1, 74);  // the dQ MMA of step gs-3 has read its dS
          ptx::tc_fence_after();
          const uint64_t dK = dKV0 + static_cast<uint64_t>((gs % kRing) * (16384 >> 4)), dV = dK + (4096 >> 4);
          const uint32_t tS = tmem_base + (gs % kSBuf) * 128;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss_2sm(tS, dQ0 + 2 * kk, dK + 2 * kk, idesc_s, kk > 0);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) if (leader) ptx::umma_ss_2sm(tS + 64, dDO0 + 2 * kk, dV + 2 * kk, idesc_s, kk > 0);
          if (leader) ptx::umma_commit_2sm(&s_full[gs % kSBuf], 0x3);
        }
        if (leader) ptx::umma_commit_2sm(&qdo_empty[k & 1], 0x3);  // all score MMAs of the item done: Q / dO may be overwritten
      }
    }
    __syncwarp();
  } else if (warp == DqCfg::kAccWarp) {
    // ---- accumulating MMAs (leader CTA): dQ += dS_j K_j (accumulator double-buffered by item parity)
    if (leader_cta) {
      const bool leader = ptx::elect_one();
      constexpr uint32_t idesc_dq = ptx::umma_idesc_bf16(256, 64, 0, 1);
      const uint32_t sKV = ptx::smem_u32(smem + Dq2Smem::KV);
      int gs = 0;
      for (int k = 0;; ++k) {
        const int it = sched_pair_item(k, nitems);
        if (it < 0) break;
        const int num_kv = tiles_of(it);
        const uint32_t tAcc = tm_dQ + (k & 1) * 64;
        if (k >= 2) {
          ptx::mbar_wait(&acc_free[k & 1], ((k >> 1) - 1) & 1, 75);
          ptx::tc_fence_after();
        }
        for (int j = 0; j < num_kv; ++j, ++gs) {
          ptx::mbar_wait(&ds_full[gs % kSBuf], (gs / kSBuf) & 1, 76);
          ptx::tc_fence_after();
          const uint32_t tA = tmem_base + (gs % kSBuf) * 128;  // dS as bf16 pairs: 16 words per column half, over the S columns it consumed
          const uint64_t dKc = desc_mn64(sKV + (gs % kRing) * 16384 + 8192, 0);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)  // keys [16 kk, 16 kk + 16): 8 packed words at column (kk / 2) * 32 + (kk % 2) * 8
            if (leader) ptx::umma_ts_2sm(tAcc, tA + (kk >> 1) * 32 + (kk & 1) * 8, dKc + (1024 >> 4) * kk, idesc_dq, (j > 0 || kk > 0));
          if (leader) ptx::umma_commit_2sm(&kv_empty[gs % kRing], 0x3);  // S_j / dP_j completed before ds_full could complete
          if (leader) ptx::umma_commit_2sm(&s_free[gs % kSBuf], 0x1);
        }
        if (leader) ptx::umma_commit_2sm(&acc_full[k & 1], 0x3);
      }
    }
    __syncwarp();
  } else {
    const int cw = warp - 2;                // 0 .. 11
    const int sg = cw / 4;                  // step group: owns the steps gs with gs % 3 == sg
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    auto load_stats = [&](int k, float& raw_l, float& raw_d) {
      raw_l = 0.f;
      raw_d = 0.f;
      const int it = sched_pair_item(k, nitems);
      if (it < 0) return;
      int pr, bh;
      fdivmod(it, fBH, pr, bh);
      const int t = (2 * (npt - 1 - pr) + rank) * 128 + r;
      if (t < T) {
        const long long idx = static_cast<long long>(bh) * T + t;
        raw_l = __ldg(lse + idx);
        raw_d = __ldg(delta + idx);
      }
    };
    // item epilogue: each step group writes 16-column granules of its row of this CTA's dQ tile: group 0 granules 0 and 1,
    // groups 1 and 2 one each
    auto epilogue = [&](int k) {
      const int it = sched_pair_item(k, nitems);
      int pr, bh, b, h;
      fdivmod(it, fBH, pr, bh);
      fdivmod(bh, fH, b, h);
      const int qt = 2 * (npt - 1 - pr) + rank;
      const int t = qt * 128 + r;
      const int colq = sg == 0 ? 0 : sg + 1;   // first granule
      const int nq = sg == 0 ? 2 : 1;          // granules
      ptx::mbar_wait(&acc_full[k & 1], (k >> 1) & 1, 77);
      ptx::tc_fence_after();
      uint32_t v[32];
#pragma unroll
      for (int c = 0; c < 2; ++c)
        if (c < nq) ptx::tmem_ld16(tm_dQ + (k & 1) * 64 + lane_off + (colq + c) * 16, *reinterpret_cast<uint32_t(*)[16]>(v + 16 * c));
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      warp_arrive_leader(&acc_free[k & 1], lane);
      if (t < T) {
        __nv_bfloat16* o = dqkv + static_cast<long long>(b * T + t) * (3 * C) + h * HS + colq * 16;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (q >= 2 * nq) break;
          uint4 w;
          w.x = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 0]), __uint_as_float(v[8 * q + 1]));
          w.y = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3]));
          w.z = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5]));
          w.w = ptx::pack_bf16x2(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7]));
          reinterpret_cast<uint4*>(o)[q] = w;
        }
      }
    };
    // cursor over this step group's steps: item pass c_k, step c_n inside the item, global step c_base + c_n (== sg mod 3)
    int c_k = 0, c_it = sched_pair_item(0, nitems), c_n = sg, c_base = 0, c_nq = c_it >= 0 ? tiles_of(c_it) : 0;
    auto normalize = [&]() {
      while (c_it >= 0 && c_n >= c_nq) {
        c_n -= c_nq;
        c_base += c_nq;
        ++c_k;
        c_it = sched_pair_item(c_k, nitems);
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
        if (nxt_k != c_k) load_stats(c_k, nxt_l, nxt_d);
        neg_l = -nxt_l * kLog2e;
        neg_d = -nxt_d * kScale;
        int pr, bh;
        fdivmod(c_it, fBH, pr, bh);
        const int qt = 2 * (npt - 1 - pr) + rank;
        r0 = qt * 128 + quarter * 32;
        if (DROP) {
          int hb, hh;
          fdivmod(bh, fH, hb, hh);
          drop_rk = drop_row_key(dcfg.key, static_cast<uint32_t>(stat_idx(hb, hh, qt * 128 + r, H, T, seq_shift)));
        }
        stat_k = c_k;
        // items have at least four steps (T >= 256), so every group owns a step of every item: the next one is c_k + 1
        load_stats(c_k + 1, nxt_l, nxt_d);
        nxt_k = c_k + 1;
      }
      const int gs = c_base + c_n;
      ptx::mbar_wait(&s_full[gs % kSBuf], (gs / kSBuf) & 1, 78);
      ptx::tc_fence_after();
      const uint32_t tbuf = tmem_base + lane_off + (gs % kSBuf) * 128;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = c_n * 64 + c * 32;
        const uint32_t ta_s = tbuf + c * 32, ta_dp = ta_s + 64;
        uint32_t pk[16];
        if (c0 > r0 + 31) dq_chunk<kMasked, DROP>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, c0);
        else if (c0 + 31 <= r0) dq_chunk<kFull, DROP>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, c0);
        else dq_chunk<kDiag, DROP>(ta_s, ta_dp, lane, neg_l, neg_d, pk, dcfg, drop_rk, c0);
        // dS of column half c (16 packed words) overwrites S columns [32 c, 32 c + 16): columns that were just consumed
        ptx::tmem_st16(tbuf + c * 32, pk);
      }
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      warp_arrive_leader(&ds_full[gs % kSBuf], lane);
      while (ep_k < c_k) epilogue(ep_k++);
      c_n += 3;
      normalize();
    }
    while (ep_k < c_k) epilogue(ep_k++);
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) ptx::tmem_dealloc_2sm(tmem_base, 512);
}

template <typename K>
int set_smem(K kern, int bytes) {
  ABCGPT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return 0;
}

template <typename... P, typename... A>
cudaError_t launch_pair(void (*kern)(P...), int grid, int threads, size_t smem, cudaStream_t stream, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(static_cast<unsigned>(threads));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<P>(args)...);
}

}  // namespace

// dK/dV and dQ of causal attention on CTA pairs.  Preconditions (checked by the caller, attn_bwd in csrc/attn.cu): T >= 256, no
// short-sequence packing; `delta` already holds rowsum(dO o O).
int attn_bwd_pair(const void* qkv, const void* dout, const float* lse, const float* delta, void* dqkv, int B, int T, int H,
                  const DropCfg& dcfg, cudaStream_t stream) {
  const int C = H * HS;
  const uint64_t rows = static_cast<uint64_t>(B) * T;
  const uint64_t pitch_qkv = 3ull * C * 2, pitch_do = static_cast<uint64_t>(C) * 2;
  CUtensorMap tmQKV128, tmQKV32, tmQKVc, tmDO128, tmDO32, tmDOc;
  int rc;
  if ((rc = encode_tmap_2d(&tmQKV128, qkv, 2, 3ull * C, rows, pitch_qkv, 64, 128, true))) return rc;
  if ((rc = encode_tmap_2d(&tmQKV32, qkv, 2, 3ull * C, rows, pitch_qkv, 64, 32, true))) return rc;
  if ((rc = encode_tmap_2d_sw(&tmQKVc, qkv, 2, 3ull * C, rows, pitch_qkv, 32, 64, 64))) return rc;
  if ((rc = encode_tmap_2d(&tmDO128, dout, 2, static_cast<uint64_t>(C), rows, pitch_do, 64, 128, true))) return rc;
  if ((rc = encode_tmap_2d(&tmDO32, dout, 2, static_cast<uint64_t>(C), rows, pitch_do, 64, 32, true))) return rc;
  if ((rc = encode_tmap_2d_sw(&tmDOc, dout, 2, static_cast<uint64_t>(C), rows, pitch_do, 32, 64, 64))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = set_smem(attn_bwd_dq2_kernel<false>, Dq2Smem::TOTAL))) return rc;
    if ((rc = set_smem(attn_bwd_dq2_kernel<true>, Dq2Smem::TOTAL))) return rc;
    if ((rc = set_smem(attn_bwd_dkv2_kernel<false>, Dkv2Smem::TOTAL))) return rc;
    if ((rc = set_smem(attn_bwd_dkv2_kernel<true>, Dkv2Smem::TOTAL))) return rc;
    done = true;
  }
  const int BH = B * H, nitems = ((T + 255) / 256) * BH;
  const FastDiv fBH = make_fastdiv(static_cast<uint32_t>(BH), static_cast<uint64_t>(nitems)), fH = make_fastdiv(static_cast<uint32_t>(H), BH);
  const int pairs = sm_count() / 2;
  const int grid = 2 * (nitems < pairs ? nitems : pairs);  // persistent: one CTA per SM, SMs paired into clusters
  __nv_bfloat16* dq = reinterpret_cast<__nv_bfloat16*>(dqkv);
  if (dcfg.thr16 == 0) {
    ABCGPT_CUDA(launch_pair(attn_bwd_dkv2_kernel<false>, grid, DkvCfg::kThreads, Dkv2Smem::TOTAL, stream, tmQKV128, tmQKV32, tmDO32, tmQKVc,
                            tmDOc, lse, delta, dq, T, H, C, BH, nitems, dcfg, fBH, fH));
    ABCGPT_CUDA(launch_pair(attn_bwd_dq2_kernel<false>, grid, DqCfg::kThreads, Dq2Smem::TOTAL, stream, tmQKV128, tmDO128, tmQKV32, tmQKVc,
                            lse, delta, dq, T, H, C, BH, nitems, dcfg, fBH, fH));
  } else {
    ABCGPT_CUDA(launch_pair(attn_bwd_dkv2_kernel<true>, grid, DkvCfg::kThreads, Dkv2Smem::TOTAL, stream, tmQKV128, tmQKV32, tmDO32, tmQKVc,
                            tmDOc, lse, delta, dq, T, H, C, BH, nitems, dcfg, fBH, fH));
    ABCGPT_CUDA(launch_pair(attn_bwd_dq2_kernel<true>, grid, DqCfg::kThreads, Dq2Smem::TOTAL, stream, tmQKV128, tmDO128, tmQKV32, tmQKVc,
                            lse, delta, dq, T, H, C, BH, nitems, dcfg, fBH, fH));
  }
  return launch_status("attn_bwd pair kernels");
}

}  // namespace abcgpt
