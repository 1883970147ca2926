// Sampling head of GPT.generate (nanoGPT/model.py:316-328): logits / temperature, optional top-k crop, softmax, one
// multinomial draw per sequence — fused into ONE launch that writes the next token straight into the token column the
// following decode step reads, so sample.py's defaults (temperature 0.8, top_k 200; nanoGPT/sample.py:33-36) never leave the
// C ABI and the whole decode step stays a replayable launch list.
//
//   reference                                       here (one CTA per sequence, the row lives in shared memory)
//   logits = logits[:, -1, :] / temperature         x_i = bf16(float(l_i) / temperature)   (the reference's logits are bf16
//                                                   under autocast, and bf16_tensor / python_float rounds back to bf16)
//   v, _ = torch.topk(logits, min(top_k, V))        kth = exact k-th largest x (MSB-first radix select on order-preserving keys)
//   logits[logits < v[:, [-1]]] = -inf              keep x_i >= kth   (ties at the threshold are all kept, as in the reference)
//   probs = F.softmax(logits, dim=-1)               p_i = exp(x_i - max) in fp32 (autocast runs softmax in fp32)
//   idx_next = torch.multinomial(probs, 1)          inverse CDF: smallest i with cumsum(p)_i > u * sum(p)
// u is one Philox4x32-10 draw per (seed, sequence, decode position): a pure function of its counters, so a replayed launch
// list needs no generator state, and tests/oracle can regenerate the very same uniform on the host (oracle: philox_uniform).
// The stream of random numbers is NOT torch's (torch.multinomial draws per-category exponentials): parity with the reference
// is distributional (chi-square in tests/test_sampling_gpu.py) and exact given u (every sampled token is checked against the
// CDF interval that u falls into).
//
// Two implementations of that one contract, chosen from V alone (sample_topk below):
//   V <= 56 320   sample_topk_kernel: one CTA per row, the row as fp32 in shared memory (V * 4 bytes <= 220 KB).
//   V <= 786 432  sample_topk_cluster_kernel: one cluster of 8 CTAs per row, each CTA holding a contiguous slice of x as
//                 bf16 (x is a bf16 value, so nothing is lost) in up to 192 KB of shared memory; cross-CTA steps read the
//                 peers' shared memory (distributed shared memory) between cluster barriers.  Large vocabularies such as
//                 the 98 465 whitespace tokens of the irishman corpus take this path.
#include "common.h"
#include "kernels.h"
#include "ptx.cuh"

#include <climits>
#include <cuda_bf16.h>

namespace abcgpt {
namespace {

constexpr int kSampleThreads = 128;

__device__ __forceinline__ uint32_t philox_uniform_bits(uint64_t seed, uint32_t row, uint64_t counter) {
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
  uint32_t c0 = row, c1 = static_cast<uint32_t>(counter), c2 = static_cast<uint32_t>(counter >> 32), c3 = 0x5A17u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c0;
}

// order-preserving map float -> uint32 (larger float <=> larger key)
__device__ __forceinline__ uint32_t order_key(float x) {
  const uint32_t b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ int block_sum_int(int v, int* scratch) {
  v = __reduce_add_sync(0xffffffffu, v);
  __syncthreads();  // scratch reuse
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  int t = 0;
#pragma unroll
  for (int w = 0; w < kSampleThreads / 32; ++w) t += scratch[w];
  return t;
}

__global__ void __launch_bounds__(kSampleThreads)
sample_topk_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, int V, float temperature, int top_k,
                   const unsigned long long* __restrict__ seed, long long counter, int64_t* __restrict__ out,
                   long long out_stride) {
  extern __shared__ float xs[];  // [V]
  __shared__ float red_f[kSampleThreads / 32];
  __shared__ int red_i[kSampleThreads / 32];
  __shared__ int red_idx[kSampleThreads / 32];
  __shared__ int chosen;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int row = blockIdx.x;
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl;

  // ---- x = bf16(l / temperature); row max and its first index
  float mx = -INFINITY;
  int mi = 0x7fffffff;
  for (int i = tid; i < V; i += kSampleThreads) {
    const float x = __bfloat162float(__float2bfloat16_rn(__fdiv_rn(__bfloat162float(lr[i]), temperature)));
    xs[i] = x;
    if (x > mx) { mx = x; mi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > mx || (om == mx && oi < mi)) { mx = om; mi = oi; }
  }
  if (lane == 0) { red_f[warp] = mx; red_idx[warp] = mi; }
  __syncthreads();
  mx = red_f[0];
  mi = red_idx[0];
#pragma unroll
  for (int w = 1; w < kSampleThreads / 32; ++w)
    if (red_f[w] > mx || (red_f[w] == mx && red_idx[w] < mi)) { mx = red_f[w]; mi = red_idx[w]; }
  if (tid == 0) chosen = mi;  // fall-back if rounding leaves the target at the very end of the CDF

  // ---- k-th largest value (exact): build its key bit by bit, counting how many keys are >= the candidate
  uint32_t thr_key = 0u;  // everything passes
  if (top_k > 0 && top_k < V) {
    uint32_t prefix = 0u;
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = prefix | (1u << bit);
      int c = 0;
      for (int i = tid; i < V; i += kSampleThreads) c += (order_key(xs[i]) >= cand) ? 1 : 0;
      if (block_sum_int(c, red_i) >= top_k) prefix = cand;
    }
    thr_key = prefix;
  }

  // ---- softmax numerators over a contiguous chunk per thread (so that a prefix over threads is a prefix over tokens)
  const int chunk = (V + kSampleThreads - 1) / kSampleThreads;
  const int i0 = min(V, tid * chunk), i1 = min(V, i0 + chunk);
  float local = 0.f;
  for (int i = i0; i < i1; ++i) {
    const float x = xs[i];
    const float p = (order_key(x) >= thr_key) ? __expf(x - mx) : 0.f;
    xs[i] = p;  // only this thread touches [i0, i1)
    local += p;
  }
  // inclusive scan of `local` over the block
  float incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  __syncthreads();  // red_f reuse
  if (lane == 31) red_f[warp] = incl;
  __syncthreads();
  float warp_off = 0.f, total = 0.f;
#pragma unroll
  for (int w = 0; w < kSampleThreads / 32; ++w) {
    if (w < warp) warp_off += red_f[w];
    total += red_f[w];
  }
  const float excl = warp_off + incl - local;

  const uint32_t bits = philox_uniform_bits(*seed, static_cast<uint32_t>(row), static_cast<uint64_t>(counter));
  const float u = static_cast<float>(bits >> 8) * (1.0f / 16777216.0f);  // [0, 1)
  const float target = u * total;
  if (local > 0.f && target >= excl && target < excl + local) {
    float acc = excl;
    int pick = -1, last_pos = -1;
    for (int i = i0; i < i1; ++i) {
      const float p = xs[i];
      if (p > 0.f) {
        last_pos = i;
        acc += p;
        if (acc > target) { pick = i; break; }
      }
    }
    chosen = pick >= 0 ? pick : last_pos;  // exactly one thread's interval contains the target
  }
  __syncthreads();
  if (tid == 0) out[static_cast<long long>(row) * out_stride] = chosen;
}

// ---- large vocabularies: one cluster per row ---------------------------------------------------------------------------
// Steps (every cross-CTA combination runs in rank order, so a (logits, seed, row, counter) gives the same token every run):
//   load     16-byte loads of the CTA's slice, x stored as bf16 bits; slice max and first index; when cropping, a 256-bin
//            histogram of the high byte of x's 16-bit order key                                          | cluster barrier 1
//   max      every CTA combines the 8 (max, index) pairs; the k-th largest key's high byte is the bin where the suffix count
//            of the summed histograms reaches k
//   low byte histogram of the low key byte over the keys with that high byte                         | cluster barrier 2
//            -> exact k-th largest key, ties at it all kept
//   draw     contiguous chunk of p = exp(x - max) per thread, CTA scan, exclusive prefix of the 8 CTA totals | barrier 3
//            the thread whose interval holds u * total walks its chunk and min-reduces its pick into rank 0
//   exit     cluster barrier 4 (no CTA leaves while a peer may still read its shared memory); rank 0 writes the token, or
//            the row maximum's first index when rounding left the target in no interval
constexpr int kClusterCtas = 8;                                // portable cluster size
constexpr int kClusterThreads = 256;                           // one histogram bin per thread
constexpr int kClusterWarps = kClusterThreads / 32;
constexpr int kClusterSliceMax = 96 * 1024;                    // bf16 values per CTA: 192 KB of shared memory
constexpr int kClusterMaxV = kClusterCtas * kClusterSliceMax;  // 786 432 (include/abcgpt.h)

// 16-bit order-preserving key of a bf16 bit pattern (larger value <=> larger key)
__device__ __forceinline__ uint32_t order_key16(uint32_t b) { return (b & 0x8000u) ? (~b & 0xffffu) : (b | 0x8000u); }

// bits of x = bf16(l / temperature); -0 is stored as +0 so that equal values have equal keys (the reference compares values)
__device__ __forceinline__ uint32_t scaled_bits(__nv_bfloat16 l, float temperature) {
  const uint32_t b = __bfloat16_as_ushort(__float2bfloat16_rn(__fdiv_rn(__bfloat162float(l), temperature)));
  return b == 0x8000u ? 0u : b;
}

__device__ __forceinline__ float bits_to_float(uint32_t b) { return __uint_as_float(b << 16); }

// Sums the 256-bin histograms `hist` of the cluster's CTAs and returns, in every thread, the bin b that holds the k-th
// largest key: count(bins > b) < k <= count(bins >= b).  *k becomes the rank of that key inside bin b.
__device__ __forceinline__ uint32_t cluster_select_bin(const uint32_t* hist, int* k, int* scan_w, int* sel) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t bin = 255 - tid;  // descending bins: a prefix over threads is a suffix over bins
  const uint32_t addr = ptx::smem_u32(hist + bin);
  int c = 0;
#pragma unroll
  for (int r = 0; r < kClusterCtas; ++r) c += static_cast<int>(ptx::ld_shared_cluster_u32(ptx::mapa(addr, r)));
  int incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) scan_w[warp] = incl;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kClusterWarps; ++w)
    if (w < warp) incl += scan_w[w];
  const int kk = *k;  // incl = count(bins >= bin)
  if (incl >= kk && incl - c < kk) {
    sel[0] = static_cast<int>(bin);
    sel[1] = kk - (incl - c);
  }
  __syncthreads();
  *k = sel[1];
  return static_cast<uint32_t>(sel[0]);
}

__global__ void __launch_bounds__(kClusterThreads)
sample_topk_cluster_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, int V, int slice, float temperature,
                           int top_k, const unsigned long long* __restrict__ seed, long long counter,
                           int64_t* __restrict__ out, long long out_stride) {
  static_assert(kClusterThreads == 256, "one histogram bin per thread");
  extern __shared__ __align__(16) uint16_t xb[];  // [slice] bits of x
  __shared__ uint32_t hist_hi[256], hist_lo[256];
  __shared__ float red_f[kClusterWarps], cta_f[kClusterCtas];
  __shared__ int red_i[kClusterWarps], scan_w[kClusterWarps], cta_i[kClusterCtas], sel[2];
  __shared__ float slice_max, slice_sum;  // read by the peers
  __shared__ int slice_arg;
  __shared__ int chosen;  // rank 0: smallest pick of the cluster
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rank = static_cast<int>(ptx::cluster_ctarank());
  const int row = blockIdx.x / kClusterCtas;
  const int base = rank * slice;
  const int n = max(0, min(slice, V - base));
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl + base;
  const bool crop = top_k > 0 && top_k < V;

  hist_hi[tid] = 0u;
  hist_lo[tid] = 0u;
  if (tid == 0) chosen = INT_MAX;
  __syncthreads();

  // ---- load: x into shared memory, slice max and its first index, high-byte histogram
  float mx = -INFINITY;
  int mi = INT_MAX;  // every thread visits its indices in increasing order, so a strict > keeps the first maximum
  const int n8 = (reinterpret_cast<uintptr_t>(lr) & 15u) == 0 ? n / 8 : 0;
  for (int v = tid; v < n8; v += kClusterThreads) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(lr) + v);
    const __nv_bfloat16* l8 = reinterpret_cast<const __nv_bfloat16*>(&raw);
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t b = scaled_bits(l8[j], temperature);
      const float x = bits_to_float(b);
      if (x > mx) { mx = x; mi = v * 8 + j; }
      if (crop) atomicAdd(&hist_hi[order_key16(b) >> 8], 1u);
      if (j & 1) w[j >> 1] |= b << 16; else w[j >> 1] = b;
    }
    reinterpret_cast<uint4*>(xb)[v] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  for (int i = n8 * 8 + tid; i < n; i += kClusterThreads) {
    const uint32_t b = scaled_bits(lr[i], temperature);
    const float x = bits_to_float(b);
    xb[i] = static_cast<uint16_t>(b);
    if (x > mx) { mx = x; mi = i; }
    if (crop) atomicAdd(&hist_hi[order_key16(b) >> 8], 1u);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > mx || (om == mx && oi < mi)) { mx = om; mi = oi; }
  }
  if (lane == 0) { red_f[warp] = mx; red_i[warp] = mi; }
  __syncthreads();
  if (tid == 0) {
#pragma unroll
    for (int w = 1; w < kClusterWarps; ++w)
      if (red_f[w] > mx || (red_f[w] == mx && red_i[w] < mi)) { mx = red_f[w]; mi = red_i[w]; }
    slice_max = mx;
    slice_arg = mi == INT_MAX ? INT_MAX : base + mi;
  }
  ptx::cluster_sync_all();  // 1

  // ---- row max and its first index: the slices in rank order hold increasing indices
  if (tid < kClusterCtas) {
    cta_f[tid] = __uint_as_float(ptx::ld_shared_cluster_u32(ptx::mapa(ptx::smem_u32(&slice_max), tid)));
    cta_i[tid] = static_cast<int>(ptx::ld_shared_cluster_u32(ptx::mapa(ptx::smem_u32(&slice_arg), tid)));
  }
  __syncthreads();
  mx = cta_f[0];
  mi = cta_i[0];
#pragma unroll
  for (int r = 1; r < kClusterCtas; ++r)
    if (cta_f[r] > mx) { mx = cta_f[r]; mi = cta_i[r]; }

  // ---- exact k-th largest key: high byte from the summed histograms, then the low byte among the keys with that high byte
  uint32_t thr_key = 0u;  // everything passes
  if (crop) {
    int k = top_k;
    const uint32_t hi = cluster_select_bin(hist_hi, &k, scan_w, sel);
    for (int v = tid; v * 8 < n; v += kClusterThreads) {
      const uint4 q = reinterpret_cast<const uint4*>(xb)[v];
      const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t key = order_key16((w[j >> 1] >> (16 * (j & 1))) & 0xffffu);
        if (v * 8 + j < n && (key >> 8) == hi) atomicAdd(&hist_lo[key & 0xffu], 1u);
      }
    }
    ptx::cluster_sync_all();  // 2
    thr_key = (hi << 8) | cluster_select_bin(hist_lo, &k, scan_w, sel);
  }

  // ---- softmax numerators over a contiguous chunk per thread (a prefix over threads and ranks is a prefix over tokens)
  const int chunk = (n + kClusterThreads - 1) / kClusterThreads;
  const int i0 = min(n, tid * chunk), i1 = min(n, i0 + chunk);
  float local = 0.f;
  for (int i = i0; i < i1; ++i) {
    const uint32_t b = xb[i];
    local += (order_key16(b) >= thr_key) ? __expf(bits_to_float(b) - mx) : 0.f;
  }
  float incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) red_f[warp] = incl;  // red_f was last read before cluster barrier 1
  __syncthreads();
  float warp_off = 0.f, cta_total = 0.f;
#pragma unroll
  for (int w = 0; w < kClusterWarps; ++w) {
    if (w < warp) warp_off += red_f[w];
    cta_total += red_f[w];
  }
  if (tid == 0) slice_sum = cta_total;
  ptx::cluster_sync_all();  // 3
  if (tid < kClusterCtas)
    cta_f[tid] = __uint_as_float(ptx::ld_shared_cluster_u32(ptx::mapa(ptx::smem_u32(&slice_sum), tid)));
  __syncthreads();
  float cta_off = 0.f, total = 0.f;
#pragma unroll
  for (int r = 0; r < kClusterCtas; ++r) {
    if (r < rank) cta_off += cta_f[r];
    total += cta_f[r];
  }
  const float excl = cta_off + (warp_off + incl - local);

  const uint32_t bits = philox_uniform_bits(*seed, static_cast<uint32_t>(row), static_cast<uint64_t>(counter));
  const float u = static_cast<float>(bits >> 8) * (1.0f / 16777216.0f);  // [0, 1)
  const float target = u * total;
  if (local > 0.f && target >= excl && target < excl + local) {
    float acc = excl;
    int pick = -1, last_pos = -1;
    for (int i = i0; i < i1; ++i) {
      const uint32_t b = xb[i];
      const float p = (order_key16(b) >= thr_key) ? __expf(bits_to_float(b) - mx) : 0.f;
      if (p > 0.f) {
        last_pos = i;
        acc += p;
        if (acc > target) { pick = i; break; }
      }
    }
    // rounding may let two neighbouring intervals overlap: the smallest pick wins, whatever the order of arrival
    ptx::red_min_shared_cluster_s32(ptx::mapa(ptx::smem_u32(&chosen), 0), base + (pick >= 0 ? pick : last_pos));
  }
  ptx::cluster_sync_all();  // 4
  if (rank == 0 && tid == 0) out[static_cast<long long>(row) * out_stride] = chosen != INT_MAX ? chosen : mi;
}

int sample_topk_cluster(const __nv_bfloat16* logits, long long ldl, int V, float temperature, int top_k,
                        const unsigned long long* seed, long long counter, int64_t* out, long long out_stride, int B,
                        cudaStream_t stream) {
  ABCGPT_CHECK_ARG(V <= kClusterMaxV, "sample_topk: vocabulary of %d is above the sampler's bound of %d tokens", V,
                   kClusterMaxV);
  ABCGPT_CHECK_ARG(B <= INT_MAX / kClusterCtas, "sample_topk: %d rows do not fit one grid", B);
  const int slice = ((V + kClusterCtas - 1) / kClusterCtas + 7) / 8 * 8;  // a multiple of 8: 16-byte aligned slices
  static bool configured = false;
  if (!configured) {
    ABCGPT_CUDA(cudaFuncSetAttribute(sample_topk_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     kClusterSliceMax * static_cast<int>(sizeof(uint16_t))));
    configured = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(B) * kClusterCtas);
  cfg.blockDim = dim3(kClusterThreads);
  cfg.dynamicSmemBytes = static_cast<size_t>(slice) * sizeof(uint16_t);
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = kClusterCtas;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  ABCGPT_CUDA(cudaLaunchKernelEx(&cfg, sample_topk_cluster_kernel, logits, ldl, V, slice, temperature, top_k, seed, counter,
                                 out, out_stride));
  return launch_status("sample_topk_cluster_kernel");
}

// ---- nucleus / top-k / temperature head of the TunesFormer character decoder ------------------------------------------
// The reference draws each character with the `samplings` package (tunesformer/utils.py:247-250), restated on the host by
// top_p_filter / top_k_filter / temperature_draw in tunesformer.py.  One CTA per row, V <= 1024 (the character vocabulary
// is 128), everything in shared memory:
//   softmax  p = softmax(float(l)) in fp32
//   rank     every token's position in the order (p descending, lower index first), as numpy's stable argsort(-p)
//   nucleus  keep ranks 0 .. r* where r* is the first rank whose running sum (in rank order) reaches top_p; all if none does
//   top-k    keep ranks < top_k (exactly k tokens, ties by lower index; unlike sample_topk_kernel, which keeps ties)
//   draw     temperature <= 0 or a single kept token with p > 0: the rank-0 token (first maximal index); otherwise weights
//            (p / p_max)^(1 / temperature) on the kept tokens, inverse CDF in token order with one Philox uniform
// The renormalisations of the restatement are divisions by one constant per step: they change no order and no cut point
// (the nucleus cut is taken on the raw p, whose sum is 1), so they are left out.
constexpr int kTopPThreads = 128;
constexpr int kTopPMaxV = 1024;  // include/abcgpt.h
constexpr int kTopPWarps = kTopPThreads / 32;

__device__ __forceinline__ float tp_block_max(float v, float* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();  // scratch reuse
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = scratch[0];
#pragma unroll
  for (int w = 1; w < kTopPWarps; ++w) t = fmaxf(t, scratch[w]);
  return t;
}

// sum in a fixed order (butterfly inside the warp, warps in order): the same inputs give the same bits in every thread
__device__ __forceinline__ float tp_block_sum(float v, float* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < kTopPWarps; ++w) t += scratch[w];
  return t;
}

__device__ __forceinline__ int tp_block_min(int v, int* scratch) {
  v = __reduce_min_sync(0xffffffffu, v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  int t = scratch[0];
#pragma unroll
  for (int w = 1; w < kTopPWarps; ++w) t = min(t, scratch[w]);
  return t;
}

// exclusive prefix of one value per thread over the block (threads in order); *total = the block sum
__device__ __forceinline__ float tp_block_excl_scan(float v, float* scratch, float* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  __syncthreads();
  if (lane == 31) scratch[warp] = incl;
  __syncthreads();
  float off = 0.f, tot = 0.f;
#pragma unroll
  for (int w = 0; w < kTopPWarps; ++w) {
    if (w < warp) off += scratch[w];
    tot += scratch[w];
  }
  *total = tot;
  return off + incl - v;
}

__global__ void __launch_bounds__(kTopPThreads)
sample_top_p_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, int V, float top_p, int top_k, float temperature,
                    const unsigned long long* __restrict__ seed, const long long* __restrict__ counter_base, long long counter,
                    const int64_t* __restrict__ row_id, int64_t* __restrict__ out, long long out_stride) {
  __shared__ float p[kTopPMaxV];      // softmax in token order, then the weights of the draw
  __shared__ float sp[kTopPMaxV];     // softmax in rank order
  __shared__ short tok[kTopPMaxV];    // token at each rank
  __shared__ short rk[kTopPMaxV];     // rank of each token
  __shared__ float red_f[kTopPWarps];
  __shared__ int red_i[kTopPWarps];
  const int tid = threadIdx.x, row = blockIdx.x;
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl;

  // ---- p = softmax(float(l))
  float mx = -INFINITY;
  for (int i = tid; i < V; i += kTopPThreads) {
    const float x = __bfloat162float(lr[i]);
    p[i] = x;
    mx = fmaxf(mx, x);
  }
  mx = tp_block_max(mx, red_f);
  float s = 0.f;
  for (int i = tid; i < V; i += kTopPThreads) {
    const float e = expf(p[i] - mx);
    p[i] = e;
    s += e;
  }
  const float z = tp_block_sum(s, red_f);
  for (int i = tid; i < V; i += kTopPThreads) p[i] = __fdiv_rn(p[i], z);
  __syncthreads();

  // ---- rank of every token: (p descending, index ascending)
  for (int i = tid; i < V; i += kTopPThreads) {
    const float pi = p[i];
    int r = 0;
    for (int j = 0; j < V; ++j) {
      const float pj = p[j];  // the same address in every lane: a broadcast
      r += (pj > pi || (pj == pi && j < i)) ? 1 : 0;
    }
    sp[r] = pi;
    tok[r] = static_cast<short>(i);
    rk[i] = static_cast<short>(r);
  }
  __syncthreads();

  // ---- nucleus, then top-k: the kept tokens are the ranks [0, n_keep)
  const int chunk = (V + kTopPThreads - 1) / kTopPThreads;  // contiguous per thread: a prefix over threads is a prefix of V
  const int c0 = min(V, tid * chunk), c1 = min(V, c0 + chunk);
  int n_keep = V;
  if (top_p < 1.f) {
    float local = 0.f;
    for (int r = c0; r < c1; ++r) local += sp[r];
    float total;
    float acc = tp_block_excl_scan(local, red_f, &total);
    int first = INT_MAX;
    for (int r = c0; r < c1; ++r) {
      acc += sp[r];
      if (acc >= top_p) { first = r; break; }
    }
    first = tp_block_min(first, red_i);  // the first rank at which the running sum reaches top_p
    n_keep = first == INT_MAX ? V : first + 1;
  }
  if (top_k > 0 && top_k < n_keep) n_keep = top_k;

  // ---- greedy: temperature <= 0, or one kept token with p > 0 (zeros sort last)
  if (temperature <= 0.f || n_keep == 1 || !(sp[1] > 0.f)) {
    if (tid == 0) out[static_cast<long long>(row) * out_stride] = tok[0];
    return;
  }

  // ---- weights (p / p_max)^(1 / temperature) on the kept tokens, one inverse-CDF draw in token order
  const float inv_t = 1.f / temperature, ptop = sp[0];
  float local = 0.f;
  for (int i = c0; i < c1; ++i) {
    const float w = (rk[i] < n_keep && p[i] > 0.f) ? powf(__fdiv_rn(p[i], ptop), inv_t) : 0.f;
    p[i] = w;  // only this thread touches [c0, c1) from here on
    local += w;
  }
  float total;
  const float excl = tp_block_excl_scan(local, red_f, &total);
  const long long rid = row_id != nullptr ? row_id[row] : row;
  const uint32_t bits = philox_uniform_bits(*seed, static_cast<uint32_t>(rid), static_cast<uint64_t>(*counter_base + counter));
  const float u = static_cast<float>(bits >> 8) * (1.0f / 16777216.0f);  // [0, 1)
  const float target = u * total;
  int pick = INT_MAX, last = -1;
  float acc = excl;
  for (int i = c0; i < c1; ++i) {
    const float w = p[i];
    if (w > 0.f) {
      last = i;
      acc += w;
      if (pick == INT_MAX && acc > target && target >= excl) pick = i;
    }
  }
  // rounding may let two neighbouring chunks both claim the target (the smallest wins) or neither (the last kept token)
  pick = tp_block_min(pick, red_i);
  last = -tp_block_min(-last, red_i);
  if (tid == 0) out[static_cast<long long>(row) * out_stride] = pick != INT_MAX ? pick : last;
}

}  // namespace

int sample_top_p(const void* logits, long long ldl, int V, float top_p, int top_k, float temperature, const void* seed,
                 const void* counter_base, long long counter, const int64_t* row_id, int64_t* out, long long out_stride, int B,
                 cudaStream_t stream) {
  ABCGPT_CHECK_ARG(logits && out && seed && counter_base && B > 0, "sample_top_p: bad arguments");
  ABCGPT_CHECK_ARG(V >= 1 && V <= kTopPMaxV, "sample_top_p: vocabulary of %d tokens is outside [1, %d]", V, kTopPMaxV);
  ABCGPT_CHECK_ARG(ldl >= V, "sample_top_p: row stride %lld is below V = %d", ldl, V);
  sample_top_p_kernel<<<B, kTopPThreads, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, V, top_p, top_k,
                                                      temperature, reinterpret_cast<const unsigned long long*>(seed),
                                                      reinterpret_cast<const long long*>(counter_base), counter, row_id, out,
                                                      out_stride);
  return launch_status("sample_top_p_kernel");
}

int sample_topk(const void* logits, long long ldl, int V, float temperature, int top_k, const void* seed, long long counter,
                int64_t* out, long long out_stride, int B, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(logits && out && seed && V > 0 && B > 0, "sample_topk: bad arguments");
  ABCGPT_CHECK_ARG(temperature > 0.f, "sample_topk: temperature must be positive (got %g)", static_cast<double>(temperature));
  const size_t smem = static_cast<size_t>(V) * sizeof(float);
  if (smem > 220 * 1024)  // the row does not fit one CTA's shared memory
    return sample_topk_cluster(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, V, temperature, top_k,
                               reinterpret_cast<const unsigned long long*>(seed), counter, out, out_stride, B, stream);
  static bool configured = false;
  if (!configured && smem > 48 * 1024) {
    ABCGPT_CUDA(cudaFuncSetAttribute(sample_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    configured = true;
  }
  sample_topk_kernel<<<B, kSampleThreads, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, V, temperature,
                                                          top_k, reinterpret_cast<const unsigned long long*>(seed), counter, out,
                                                          out_stride);
  return launch_status("sample_topk_kernel");
}

}  // namespace abcgpt
