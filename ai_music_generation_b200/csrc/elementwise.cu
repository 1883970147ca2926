// HBM-bound kernels of the step that are not LayerNorm: embedding gather / scatter, fused softmax
// cross-entropy for the small ABC vocabulary, gradient sum-of-squares, fused clip + AdamW (+ bf16 weight
// shadow), casts and the greedy sampling head.  All global traffic is 128-bit where alignment allows.
#include "common.h"
#include "dropout.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace abcgpt {
namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// scale-or-zero the four columns [4*c4, 4*c4+4) of `row` according to the dropout mask of this site
__device__ __forceinline__ void drop4(float4& v, const DropCfg& d, uint32_t row, int c4) {
  if (d.thr16 == 0) return;
  const uint32_t rk = drop_row_key(d.key, row);
  const uint32_t b0 = drop_pair_bits(rk, 2 * c4), b1 = drop_pair_bits(rk, 2 * c4 + 1);
  v.x = drop_keep_lo(b0, d.thr16) ? v.x * d.inv_keep : 0.f;
  v.y = drop_keep_hi(b0, d.thr16) ? v.y * d.inv_keep : 0.f;
  v.z = drop_keep_lo(b1, d.thr16) ? v.z * d.inv_keep : 0.f;
  v.w = drop_keep_hi(b1, d.thr16) ? v.w * d.inv_keep : 0.f;
}

// ---- embedding (model.py:177-179) ----------------------------------------------------------------------
__global__ void embed_fwd_kernel(const int64_t* __restrict__ idx, const float4* __restrict__ wte,
                                 const float4* __restrict__ wpe, float4* __restrict__ x, long long total, int T,
                                 int C4, int V, DropCfg drop) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / C4;
    const int c = static_cast<int>(i - m * C4);
    long long tok = __ldg(idx + m);
    tok = tok < 0 ? 0 : (tok >= V ? V - 1 : tok);
    const int t = static_cast<int>(m % T);
    const float4 a = __ldg(wte + tok * C4 + c);
    const float4 b = __ldg(wpe + static_cast<long long>(t) * C4 + c);
    float4 o = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    drop4(o, drop, static_cast<uint32_t>(m), c);
    x[i] = o;
  }
}

// dwpe[t,:] += sum_b dx[b,t,:]: one thread per (t, 4 columns) loops over a slice of the batch.  With long sequences one
// slice covers the whole batch (deterministic read-modify-write); short sequences with huge batches (the character level
// of the hierarchical model: T = 32, B ~ 8000) have too few (t, column) pairs to fill the GPU, so the batch is cut into
// gridDim.y slices that add their partial sums with vector reductions.
__global__ void embed_bwd_wpe_kernel(const float4* __restrict__ dx, float4* __restrict__ dwpe, int B, int T, int C4,
                                     int per_slice, DropCfg drop) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= static_cast<long long>(T) * C4) return;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
  const long long stride = static_cast<long long>(T) * C4;
  const int b0 = blockIdx.y * per_slice, b1 = min(B, b0 + per_slice);
  const uint32_t trow = static_cast<uint32_t>(i / C4);
  const int c = static_cast<int>(i % C4);
  int b = b0;
  for (; b + 1 < b1; b += 2) {  // two independent chains
    float4 v = __ldg(dx + b * stride + i), w = __ldg(dx + (b + 1) * stride + i);
    drop4(v, drop, static_cast<uint32_t>(b * T) + trow, c);
    drop4(w, drop, static_cast<uint32_t>((b + 1) * T) + trow, c);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    acc2.x += w.x; acc2.y += w.y; acc2.z += w.z; acc2.w += w.w;
  }
  if (b < b1) {
    float4 v = __ldg(dx + b * stride + i);
    drop4(v, drop, static_cast<uint32_t>(b * T) + trow, c);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  acc.x += acc2.x; acc.y += acc2.y; acc.z += acc2.z; acc.w += acc2.w;
  if (gridDim.y == 1) {
    float4 o = dwpe[i];
    o.x += acc.x; o.y += acc.y; o.z += acc.z; o.w += acc.w;
    dwpe[i] = o;
  } else {
    ptx::red_add_v4(reinterpret_cast<float*>(dwpe + i), acc.x, acc.y, acc.z, acc.w);
  }
}
// batch slices for the kernel above: enough blocks for ~8 per SM, at least 16 sequences per slice
static void wpe_slices(int B, long long n, int* slices, int* per_slice) {
  const long long blocks_x = (n + 127) / 128;
  long long want = (8ll * sm_count() + blocks_x - 1) / blocks_x;
  if (want > B / 16) want = B / 16;
  if (want < 1) want = 1;
  *per_slice = static_cast<int>((B + want - 1) / want);
  *slices = (B + *per_slice - 1) / *per_slice;
}

// dwte[idx[m],:] += dx[m,:].  The ABC vocabulary has ~95 rows, so thousands of tokens collide on each row:
// every block first accumulates ROWS_PER_BLOCK tokens x 128 columns into a shared-memory table (shared
// atomics), then flushes the touched vocabulary rows with vector reductions.  For large vocabularies
// (table does not fit) it falls back to direct global vector reductions.
constexpr int kWteCols = 128;
__global__ void __launch_bounds__(256)
embed_bwd_wte_smem_kernel(const int64_t* __restrict__ idx, const float* __restrict__ dx, float* __restrict__ dwte,
                          int M, int C, int V, int rows_per_block, DropCfg drop) {
  extern __shared__ float table[];  // [V][kWteCols]
  const int col0 = blockIdx.y * kWteCols;
  const int ncols = min(kWteCols, C - col0);
  for (int i = threadIdx.x; i < V * kWteCols; i += blockDim.x) table[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int m0 = blockIdx.x * rows_per_block;
  const int m1 = min(M, m0 + rows_per_block);
  for (int m = m0 + warp; m < m1; m += nwarps) {
    long long tok = __ldg(idx + m);
    if (tok < 0 || tok >= V) continue;
    const int c = lane * 4;
    if (c < ncols) {
      float4 v = __ldg(reinterpret_cast<const float4*>(dx + static_cast<long long>(m) * C + col0 + c));
      drop4(v, drop, static_cast<uint32_t>(m), (col0 + c) >> 2);
      float* t = table + tok * kWteCols + c;
      atomicAdd(t + 0, v.x); atomicAdd(t + 1, v.y); atomicAdd(t + 2, v.z); atomicAdd(t + 3, v.w);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < V * (kWteCols / 4); i += blockDim.x) {
    const int r = i / (kWteCols / 4), c = (i % (kWteCols / 4)) * 4;
    if (c < ncols) {
      const float* t = table + r * kWteCols + c;
      if (t[0] != 0.f || t[1] != 0.f || t[2] != 0.f || t[3] != 0.f)
        ptx::red_add_v4(dwte + static_cast<long long>(r) * C + col0 + c, t[0], t[1], t[2], t[3]);
    }
  }
}
__global__ void embed_bwd_wte_direct_kernel(const int64_t* __restrict__ idx, const float4* __restrict__ dx,
                                            float* __restrict__ dwte, long long total, int C4, int V, DropCfg drop) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / C4;
    const int c = static_cast<int>(i - m * C4);
    const long long tok = __ldg(idx + m);
    if (tok < 0 || tok >= V) continue;
    float4 v = __ldg(dx + i);
    drop4(v, drop, static_cast<uint32_t>(m), c);
    ptx::red_add_v4(dwte + (tok * C4 + c) * 4, v.x, v.y, v.z, v.w);
  }
}

// ---- fused softmax cross-entropy (model.py:187) ------------------------------------------------------------
// one warp per row; logits are bf16 (the autocast lm_head output), the softmax runs in fp32 like
// F.cross_entropy under autocast.
__global__ void __launch_bounds__(256)
ce_fwd_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, const int64_t* __restrict__ targets,
              float* __restrict__ row_loss, int M, int V) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const long long tgt = __ldg(targets + row);
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl;
  float mx = -INFINITY;
  for (int c = lane; c < V; c += 32) mx = fmaxf(mx, __bfloat162float(lr[c]));
  mx = warp_max(mx);
  float s = 0.f;
  for (int c = lane; c < V; c += 32) s += __expf(__bfloat162float(lr[c]) - mx);
  s = warp_sum(s);
  if (lane == 0) {
    float l = 0.f;
    if (tgt >= 0 && tgt < V) l = (mx + __logf(s)) - __bfloat162float(lr[tgt]);
    row_loss[row] = l;
  }
}

__global__ void __launch_bounds__(1024)
ce_finalize_kernel(const float* __restrict__ row_loss, const int64_t* __restrict__ targets, int M,
                   float* __restrict__ sum_count, float* __restrict__ loss) {
  __shared__ float ssum[32];
  __shared__ float scnt[32];
  float s = 0.f, n = 0.f;
  // fixed assignment of rows to threads => bitwise reproducible loss
  for (int i = threadIdx.x; i < M; i += blockDim.x) {
    const long long t = __ldg(targets + i);
    if (t >= 0) {
      s += row_loss[i];
      n += 1.f;
    }
  }
  s = warp_sum(s);
  n = warp_sum(n);
  if ((threadIdx.x & 31) == 0) {
    ssum[threadIdx.x >> 5] = s;
    scnt[threadIdx.x >> 5] = n;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    s = ssum[threadIdx.x];
    n = scnt[threadIdx.x];
    s = warp_sum(s);
    n = warp_sum(n);
    if (threadIdx.x == 0) {
      sum_count[0] = s;
      sum_count[1] = n;
      if (loss) loss[0] = s / n;  // all-ignored batch -> nan, like F.cross_entropy
    }
  }
}

__global__ void __launch_bounds__(256)
ce_bwd_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, const int64_t* __restrict__ targets,
              const float* __restrict__ sum_count, const float* __restrict__ grad_loss,
              __nv_bfloat16* __restrict__ dlogits, int M, int V) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const long long tgt = __ldg(targets + row);
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl;
  __nv_bfloat16* dr = dlogits + static_cast<long long>(row) * ldl;
  const bool valid = tgt >= 0 && tgt < V;
  const float scale = valid ? __ldg(grad_loss) / __ldg(sum_count + 1) : 0.f;
  float mx = -INFINITY;
  for (int c = lane; c < V; c += 32) mx = fmaxf(mx, __bfloat162float(lr[c]));
  mx = warp_max(mx);
  float s = 0.f;
  for (int c = lane; c < V; c += 32) s += __expf(__bfloat162float(lr[c]) - mx);
  s = warp_sum(s);
  const float inv = 1.0f / s;
  for (int c = lane; c < static_cast<int>(ldl); c += 32) {
    float g = 0.f;
    if (c < V && valid) {
      const float p = __expf(__bfloat162float(lr[c]) - mx) * inv;
      g = (p - (c == tgt ? 1.f : 0.f)) * scale;
    }
    dr[c] = __float2bfloat16_rn(g);
  }
}

// ---- gradient norm, clip + AdamW (train.py:350-354; torch.optim.AdamW single-tensor formulas) -----------------
// Deterministic two-stage reduction (fixed grid, fixed order): every data-parallel rank must derive the SAME clip
// coefficient from the same all-reduced gradients, or the replicas drift apart bit by bit.
constexpr int kSumsqBlocks = 1024;
__global__ void __launch_bounds__(512) sumsq_kernel(const float* __restrict__ g, long long n, float* __restrict__ partial) {
  __shared__ float sh[16];
  float s = 0.f;
  const long long n4 = n >> 2;
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(g4 + i);
    s += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const float v = g[(n4 << 2) + threadIdx.x];
    s += v * v;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
    s = warp_sum(s);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
  }
}
__global__ void __launch_bounds__(1024) sumsq_final_kernel(const float* __restrict__ partial, int nparts, float* __restrict__ out) {
  __shared__ float sh[32];
  float s = threadIdx.x < nparts ? partial[threadIdx.x] : 0.f;
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = sh[threadIdx.x];
    s = warp_sum(s);
    if (threadIdx.x == 0) out[0] += s;
  }
}

struct AdamArgs {
  float lr, beta1, beta2, eps, wd, step_size, inv_bc2_sqrt, max_norm;
};

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, const AdamArgs& a, float gscale) {
  g *= gscale;
  p *= (1.0f - a.lr * a.wd);
  m = m + (1.0f - a.beta1) * (g - m);                 // lerp(m, g, 1-beta1)
  v = a.beta2 * v + (1.0f - a.beta2) * g * g;
  const float denom = sqrtf(v) * a.inv_bc2_sqrt + a.eps;
  p -= a.step_size * (m / denom);
}

__global__ void __launch_bounds__(512)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
             __nv_bfloat16* __restrict__ shadow, long long n, AdamArgs a, const float* __restrict__ sumsq) {
  float gscale = 1.0f;
  if (sumsq != nullptr) {
    const float norm = sqrtf(__ldg(sumsq));
    gscale = fminf(1.0f, a.max_norm / (norm + 1e-6f));
  }
  const long long n4 = n >> 2;
  float4* p4 = reinterpret_cast<float4*>(p);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* m4 = reinterpret_cast<float4*>(m);
  float4* v4 = reinterpret_cast<float4*>(v);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 pp = p4[i], mm = m4[i], vv = v4[i];
    const float4 gg = __ldg(g4 + i);
    adam_one(pp.x, gg.x, mm.x, vv.x, a, gscale);
    adam_one(pp.y, gg.y, mm.y, vv.y, a, gscale);
    adam_one(pp.z, gg.z, mm.z, vv.z, a, gscale);
    adam_one(pp.w, gg.w, mm.w, vv.w, a, gscale);
    p4[i] = pp; m4[i] = mm; v4[i] = vv;
    if (shadow) reinterpret_cast<uint2*>(shadow)[i] = make_uint2(ptx::pack_bf16x2(pp.x, pp.y), ptx::pack_bf16x2(pp.z, pp.w));
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const long long i = (n4 << 2) + threadIdx.x;
    float pp = p[i], mm = m[i], vv = v[i];
    adam_one(pp, g[i], mm, vv, a, gscale);
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (shadow) shadow[i] = __float2bfloat16_rn(pp);
  }
}

__global__ void __launch_bounds__(512) cast_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n) {
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    reinterpret_cast<uint2*>(y)[i] = make_uint2(ptx::pack_bf16x2(v.x, v.y), ptx::pack_bf16x2(v.z, v.w));
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const long long i = (n4 << 2) + threadIdx.x;
    y[i] = __float2bfloat16_rn(x[i]);
  }
}


// ---- bias gradient: out[n] += sum_m dy[m,n]  (bf16 in, fp32 accumulate; only used when config.bias=True) ----
__global__ void __launch_bounds__(256)
colsum_kernel(const __nv_bfloat16* __restrict__ dy, long long ld, int M, int N, int rows_per_block,
              float* __restrict__ out) {
  __shared__ float sh[8][64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = blockIdx.x * 64 + lane * 2;
  const int m0 = blockIdx.y * rows_per_block, m1 = min(M, m0 + rows_per_block);
  float a0 = 0.f, a1 = 0.f;
  if (col < N) {
    for (int m = m0 + warp; m < m1; m += 8) {
      const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(dy + static_cast<long long>(m) * ld + col));
      a0 += ptx::bf16lo(v);
      a1 += ptx::bf16hi(v);
    }
  }
  sh[warp][lane * 2] = a0;
  sh[warp][lane * 2 + 1] = a1;
  __syncthreads();
  if (threadIdx.x < 64) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sh[w][threadIdx.x];
    const int c = blockIdx.x * 64 + threadIdx.x;
    if (c < N) atomicAdd(out + c, s);
  }
}

// wide form (N % 8 == 0, 16-byte aligned rows): a lane owns 8 consecutive columns (one 128-bit load per row), a warp 256 columns,
// four rows in flight per thread — 64 bytes per thread outstanding instead of 4 (the narrow kernel ran at 4.3 TB/s on the
// TunesFormer-shaped step's 11 GB of bias-gradient reads)
__global__ void __launch_bounds__(256)
colsum8_kernel(const __nv_bfloat16* __restrict__ dy, long long ld, int M, int N, int rows_per_block, float* __restrict__ out) {
  __shared__ float sh[8][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + lane * 8;
  const int m0 = blockIdx.y * rows_per_block, m1 = min(M, m0 + rows_per_block);
  float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (col < N) {
    const __nv_bfloat16* p = dy + col;
    int m = m0 + warp;
    for (; m + 24 < m1; m += 32) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const uint4*>(p + static_cast<long long>(m + 8 * u) * ld));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        a[0] += ptx::bf16lo(v[u].x); a[1] += ptx::bf16hi(v[u].x); a[2] += ptx::bf16lo(v[u].y); a[3] += ptx::bf16hi(v[u].y);
        a[4] += ptx::bf16lo(v[u].z); a[5] += ptx::bf16hi(v[u].z); a[6] += ptx::bf16lo(v[u].w); a[7] += ptx::bf16hi(v[u].w);
      }
    }
    for (; m < m1; m += 8) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(p + static_cast<long long>(m) * ld));
      a[0] += ptx::bf16lo(v.x); a[1] += ptx::bf16hi(v.x); a[2] += ptx::bf16lo(v.y); a[3] += ptx::bf16hi(v.y);
      a[4] += ptx::bf16lo(v.z); a[5] += ptx::bf16hi(v.z); a[6] += ptx::bf16lo(v.w); a[7] += ptx::bf16hi(v.w);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) sh[warp][lane * 8 + i] = a[i];
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += sh[w][threadIdx.x];
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < N) atomicAdd(out + c, s);
}

// ---- single-token decode attention over a KV cache (generate(), model.py:305-330, with the O(T^2)-per-token context
// recompute of the reference replaced by a cache) --------------------------------------------------------------------
// cache: bf16 [B, Tmax, 3C] holding the c_attn output (q | k | v) of every position decoded so far; the query is the
// row at position n_keys-1.  One block per (batch, head); HBM-bound (K and V of the sequence are read once).
__global__ void __launch_bounds__(128)
attn_decode_kernel(const __nv_bfloat16* __restrict__ cache, __nv_bfloat16* __restrict__ out, int Tmax, int n_keys, int H,
                   int C) {
  ptx::pdl_launch_dependents();  // programmatic dependent launch: see launch_k (common.h)
  ptx::pdl_wait();
  extern __shared__ float prob[];  // [n_keys]
  __shared__ float q[64];
  __shared__ float red[4];
  __shared__ float part[4][64];
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // head-major cache [B, 3H, Tmax, 64] (q heads | k heads | v heads): the K and V rows of one (b, h) are contiguous, so both
  // phases stream whole DRAM pages instead of 128-byte pieces 4.6 KB apart
  const long long head = static_cast<long long>(Tmax) * 64;
  const __nv_bfloat16* base = cache + static_cast<long long>(b) * 3 * H * head;
  if (tid < 64) q[tid] = __bfloat162float(base[h * head + static_cast<long long>(n_keys - 1) * 64 + tid]) * 0.125f;
  __syncthreads();
  float mx = -INFINITY;
  {
    // scores: eight lanes share a key (16 bytes = 8 head dimensions each), so one warp instruction reads four whole 128-byte
    // K rows; 16 keys in flight per warp.  (One thread per key read 16 bytes from 32 different lines per instruction: the
    // L1 tag stage, one line per clock, capped that at ~4.5 TB/s chip-wide.)
    const int sub = lane & 7, grp = lane >> 3;
    float qr[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) qr[e] = q[sub * 8 + e];
    const __nv_bfloat16* kbase = base + (H + h) * head + sub * 8;
    for (int k0 = warp * 16; k0 < n_keys; k0 += 64) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = k0 + u * 4 + grp;
        v[u] = k < n_keys ? __ldg(reinterpret_cast<const uint4*>(kbase + static_cast<long long>(k) * 64)) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
        float sc = 0.f;
#pragma unroll
        for (int e = 0; e < 4; ++e) sc += qr[2 * e] * ptx::bf16lo(w[e]) + qr[2 * e + 1] * ptx::bf16hi(w[e]);
        sc += __shfl_xor_sync(0xffffffffu, sc, 1);
        sc += __shfl_xor_sync(0xffffffffu, sc, 2);
        sc += __shfl_xor_sync(0xffffffffu, sc, 4);
        const int k = k0 + u * 4 + grp;
        if (k < n_keys) {
          if (sub == 0) prob[k] = sc;
          mx = fmaxf(mx, sc);
        }
      }
    }
  }
  mx = warp_max(mx);
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
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  const float inv = 1.0f / ((red[0] + red[1]) + (red[2] + red[3]));
  // out[d] = sum_k p_k V[k][d]: the flash kernels round P to bf16 before the second matmul; mirror that.  Each warp takes
  // every fourth key, a lane two adjacent columns (one 128 B row segment per warp instruction), four keys in flight per warp.
  const uint32_t* vbase = reinterpret_cast<const uint32_t*>(base + (2 * H + h) * head) + lane;
  const long long vstride = 32;  // row stride in 32-bit words
  float a0 = 0.f, a1 = 0.f, c0 = 0.f, c1 = 0.f;
  int k = warp;
  // eight keys in flight per warp: with four (24 KB per SM at 12 resident blocks) this phase was latency-bound, below the
  // ~35 KB per SM that HBM latency x bandwidth asks for
  for (; k + 28 < n_keys; k += 32) {
    uint32_t v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __ldg(vbase + (k + 4 * u) * vstride);
#pragma unroll
    for (int u = 0; u < 8; u += 2) {
      const float p0 = ptx::bf16_round(prob[k + 4 * u] * inv), p1 = ptx::bf16_round(prob[k + 4 * u + 4] * inv);
      a0 += p0 * ptx::bf16lo(v[u]); a1 += p0 * ptx::bf16hi(v[u]);
      c0 += p1 * ptx::bf16lo(v[u + 1]); c1 += p1 * ptx::bf16hi(v[u + 1]);
    }
  }
  for (; k + 12 < n_keys; k += 16) {
    const uint32_t v0 = __ldg(vbase + k * vstride), v1 = __ldg(vbase + (k + 4) * vstride);
    const uint32_t v2 = __ldg(vbase + (k + 8) * vstride), v3 = __ldg(vbase + (k + 12) * vstride);
    const float p0 = ptx::bf16_round(prob[k] * inv), p1 = ptx::bf16_round(prob[k + 4] * inv);
    const float p2 = ptx::bf16_round(prob[k + 8] * inv), p3 = ptx::bf16_round(prob[k + 12] * inv);
    a0 += p0 * ptx::bf16lo(v0); a1 += p0 * ptx::bf16hi(v0);
    c0 += p1 * ptx::bf16lo(v1); c1 += p1 * ptx::bf16hi(v1);
    a0 += p2 * ptx::bf16lo(v2); a1 += p2 * ptx::bf16hi(v2);
    c0 += p3 * ptx::bf16lo(v3); c1 += p3 * ptx::bf16hi(v3);
  }
  for (; k < n_keys; k += 4) {
    const uint32_t v0 = __ldg(vbase + k * vstride);
    const float p0 = ptx::bf16_round(prob[k] * inv);
    a0 += p0 * ptx::bf16lo(v0); a1 += p0 * ptx::bf16hi(v0);
  }
  part[warp][2 * lane] = a0 + c0;
  part[warp][2 * lane + 1] = a1 + c1;
  __syncthreads();
  if (tid < 64)
    out[static_cast<long long>(b) * C + h * 64 + tid] =
        __float2bfloat16_rn((part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid]));
}


// ---- device-resident token stream (get_batch, train.py:122-144): x[b,:] = data[ix[b] : ix[b]+T], y[b,:] = data[ix[b]+1 : ...+T+1]
// The whole uint16 (or uint32) corpus lives in HBM (IrishMAN char-level: 61 M tokens = 122 MB); one launch widens B
// random windows to the int64 ids the model consumes, replacing B host slices + astype + pin + two H2D copies per batch.
template <typename TokT>
__global__ void __launch_bounds__(256)
sample_batch_kernel(const TokT* __restrict__ data, const int64_t* __restrict__ ix, int64_t* __restrict__ x,
                    int64_t* __restrict__ y, int B, int T) {
  const long long total = static_cast<long long>(B) * T;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / T), t = static_cast<int>(i - static_cast<long long>(b) * T);
    const long long o = __ldg(ix + b) + t;
    const TokT a = __ldg(data + o), c = __ldg(data + o + 1);
    x[i] = static_cast<int64_t>(a);
    y[i] = static_cast<int64_t>(c);
  }
}

// ---- greedy head (model.py:316-328 with top_k=1) -----------------------------------------------------------
__global__ void __launch_bounds__(256)
argmax_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, int V, int64_t* __restrict__ out,
              long long out_stride, int B) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B) return;
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int c = lane; c < V; c += 32) {
    const float x = __bfloat162float(lr[c]);
    if (x > best) { best = x; bi = c; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (lane == 0) out[static_cast<long long>(row) * out_stride] = bi;
}

inline int grid_for(long long work_items, int threads, int waves = 8) {
  long long g = (work_items + threads - 1) / threads;
  const long long cap = static_cast<long long>(sm_count()) * waves;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}


// ---- hierarchical (TunesFormer-shaped) decoders: embeddings that come from another network ----------------------------
// x[m,:] = e[m,:] + wpe[m % T,:]   (HF GPT2Model(inputs_embeds=...), tunesformer/utils.py:102-106)
__global__ void add_pos_kernel(const float4* __restrict__ e, const float4* __restrict__ wpe, float4* __restrict__ x,
                               long long total, int T, int C4) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / C4;
    const int c = static_cast<int>(i - m * C4);
    const float4 a = __ldg(e + i);
    const float4 b = __ldg(wpe + (m % T) * C4 + c);
    x[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}
// x[b,0,:] = first[b,:] + wpe[0,:]: the char-level decoder's first input embedding is the encoded patch
// (tunesformer/utils.py:146-150)
__global__ void set_first_pos_kernel(const float4* __restrict__ first, const float4* __restrict__ wpe, float4* __restrict__ x,
                                     int B, int T, int C4) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= static_cast<long long>(B) * C4) return;
  const long long b = i / C4;
  const int c = static_cast<int>(i - b * C4);
  const float4 a = __ldg(first + i), p = __ldg(wpe + c);
  x[b * T * C4 + c] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
}
// one-hot rows for the patch embedding Linear(S * V -> C) (tunesformer/utils.py:102-104): out[m, s * V + tok[m,s]] = 1
__global__ void onehot_bf16_kernel(const int64_t* __restrict__ tok, __nv_bfloat16* __restrict__ out, long long total, int S,
                                   int V) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  long long t = __ldg(tok + i);
  t = t < 0 ? 0 : (t >= V ? V - 1 : t);
  const long long m = i / S;
  const int s = static_cast<int>(i - m * S);
  out[(m * S + s) * V + t] = __float2bfloat16(1.0f);
}

// ---- packed sequences (TunesFormer training on tunes of different lengths) ------------------------------------------------
// sequence of packed row m: the s with cu[s] <= m < cu[s+1] (cu ascending, cu[0] = 0)
__device__ __forceinline__ int seq_of_row(const int32_t* __restrict__ cu, int n_seqs, int m) {
  int lo = 0, hi = n_seqs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(cu + mid) <= m) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}
// x[m,:] = e[m,:] + wpe[m - cu[seq(m)],:]: positions restart at every sequence; one block per row
__global__ void __launch_bounds__(128)
add_pos_varlen_kernel(const float4* __restrict__ e, const float4* __restrict__ wpe, float4* __restrict__ x,
                      const int32_t* __restrict__ cu, int n_seqs, int C4) {
  const int m = blockIdx.x;
  const int t = m - __ldg(cu + seq_of_row(cu, n_seqs, m));
  const long long row = static_cast<long long>(m) * C4;
  for (int c = threadIdx.x; c < C4; c += blockDim.x) {
    const float4 a = __ldg(e + row + c);
    const float4 b = __ldg(wpe + static_cast<long long>(t) * C4 + c);
    x[row + c] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
  }
}
// dwpe[t,:] += sum over s with len_s > t of dx[cu[s] + t,:]: one thread per (t, 4 columns), sequences summed in index order
// (no atomics: the position gradient is bitwise reproducible)
__global__ void __launch_bounds__(128)
pos_bwd_varlen_kernel(const float4* __restrict__ dx, float4* __restrict__ dwpe, const int32_t* __restrict__ cu, int n_seqs, int C4) {
  const int t = blockIdx.x;
  const int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= C4) return;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int r0 = __ldg(cu);
  for (int s = 0; s < n_seqs; ++s) {
    const int r1 = __ldg(cu + s + 1);
    if (t < r1 - r0) {
      const float4 v = __ldg(dx + static_cast<long long>(r0 + t) * C4 + c);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    r0 = r1;
  }
  float4* o = dwpe + static_cast<long long>(t) * C4 + c;
  const float4 p = *o;
  *o = make_float4(p.x + acc.x, p.y + acc.y, p.z + acc.z, p.w + acc.w);
}
// w[m] = 1 / (n_groups * valid rows of group(m)) for a valid target, else 0 (one block: shared-memory integer counts)
__global__ void __launch_bounds__(1024)
ce_group_weights_kernel(const int64_t* __restrict__ targets, const int32_t* __restrict__ row_group, int n_groups, int M, int V,
                        float* __restrict__ w) {
  extern __shared__ int cnt[];
  for (int g = threadIdx.x; g < n_groups; g += blockDim.x) cnt[g] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < M; i += blockDim.x) {
    const long long t = __ldg(targets + i);
    const int g = __ldg(row_group + i);
    if (t >= 0 && t < V && g >= 0 && g < n_groups) atomicAdd(&cnt[g], 1);
  }
  __syncthreads();
  const float ng = static_cast<float>(n_groups);
  for (int i = threadIdx.x; i < M; i += blockDim.x) {
    const long long t = __ldg(targets + i);
    const int g = __ldg(row_group + i);
    w[i] = (t >= 0 && t < V && g >= 0 && g < n_groups) ? 1.0f / (ng * static_cast<float>(cnt[g])) : 0.f;
  }
}
// loss[0] = sum_m w[m] * row_loss[m]; fixed assignment of rows to threads => bitwise reproducible
__global__ void __launch_bounds__(1024)
ce_finalize_weighted_kernel(const float* __restrict__ row_loss, const float* __restrict__ w, int M, float* __restrict__ loss) {
  __shared__ float ssum[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < M; i += blockDim.x) s += __ldg(w + i) * row_loss[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) ssum[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = warp_sum(ssum[threadIdx.x]);
    if (threadIdx.x == 0) loss[0] = s;
  }
}
// dlogits = (softmax - onehot) * grad_loss * w[m]; zero for ignored rows and the padding columns V..ldl
__global__ void __launch_bounds__(256)
ce_bwd_weighted_kernel(const __nv_bfloat16* __restrict__ logits, long long ldl, const int64_t* __restrict__ targets,
                       const float* __restrict__ w, const float* __restrict__ grad_loss, __nv_bfloat16* __restrict__ dlogits,
                       int M, int V) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const long long tgt = __ldg(targets + row);
  const __nv_bfloat16* lr = logits + static_cast<long long>(row) * ldl;
  __nv_bfloat16* dr = dlogits + static_cast<long long>(row) * ldl;
  const bool valid = tgt >= 0 && tgt < V;
  const float scale = valid ? __ldg(grad_loss) * __ldg(w + row) : 0.f;
  float mx = -INFINITY;
  for (int c = lane; c < V; c += 32) mx = fmaxf(mx, __bfloat162float(lr[c]));
  mx = warp_max(mx);
  float s = 0.f;
  for (int c = lane; c < V; c += 32) s += __expf(__bfloat162float(lr[c]) - mx);
  s = warp_sum(s);
  const float inv = 1.0f / s;
  for (int c = lane; c < static_cast<int>(ldl); c += 32) {
    float g = 0.f;
    if (c < V && valid) {
      const float p = __expf(__bfloat162float(lr[c]) - mx) * inv;
      g = (p - (c == tgt ? 1.f : 0.f)) * scale;
    }
    dr[c] = __float2bfloat16_rn(g);
  }
}

}  // namespace

int embed_fwd(const int64_t* idx, const float* wte, const float* wpe, float* x, int M, int T, int C, int V, float drop_p,
              uint32_t drop_key, cudaStream_t stream) {
  const DropCfg drop = make_drop(drop_p, drop_key);
  ABCGPT_CHECK_ARG(idx && wte && wpe && x, "embed_fwd: null pointer");
  ABCGPT_CHECK_ARG(M > 0 && T > 0 && C % 4 == 0 && V > 0, "embed_fwd: bad shape M=%d T=%d C=%d V=%d", M, T, C, V);
  const long long total = static_cast<long long>(M) * (C / 4);
  embed_fwd_kernel<<<grid_for(total, 256), 256, 0, stream>>>(idx, reinterpret_cast<const float4*>(wte),
                                                             reinterpret_cast<const float4*>(wpe),
                                                             reinterpret_cast<float4*>(x), total, T, C / 4, V, drop);
  return launch_status("embed_fwd_kernel");
}

int embed_bwd(const int64_t* idx, const float* dx, float* dwte, float* dwpe, int M, int T, int C, int V, float drop_p,
              uint32_t drop_key, cudaStream_t stream) {
  const DropCfg drop = make_drop(drop_p, drop_key);
  ABCGPT_CHECK_ARG(idx && dx && dwte && dwpe, "embed_bwd: null pointer");
  ABCGPT_CHECK_ARG(M > 0 && T > 0 && M % T == 0 && C % 4 == 0 && V > 0, "embed_bwd: bad shape M=%d T=%d C=%d V=%d", M, T, C, V);
  const int C4 = C / 4;
  {
    const long long n = static_cast<long long>(T) * C4;
    int slices, per_slice;
    wpe_slices(M / T, n, &slices, &per_slice);
    embed_bwd_wpe_kernel<<<dim3(static_cast<unsigned>((n + 127) / 128), slices), 128, 0, stream>>>(
        reinterpret_cast<const float4*>(dx), reinterpret_cast<float4*>(dwpe), M / T, T, C4, per_slice, drop);
    int rc = launch_status("embed_bwd_wpe_kernel");
    if (rc) return rc;
  }
  const size_t table_bytes = static_cast<size_t>(V) * kWteCols * sizeof(float);
  if (table_bytes <= 96 * 1024) {
    static bool done = false;
    if (!done) {
      ABCGPT_CUDA(cudaFuncSetAttribute(embed_bwd_wte_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      done = true;
    }
    const int rows_per_block = 512;
    dim3 grid((M + rows_per_block - 1) / rows_per_block, (C + kWteCols - 1) / kWteCols);
    embed_bwd_wte_smem_kernel<<<grid, 256, table_bytes, stream>>>(idx, dx, dwte, M, C, V, rows_per_block, drop);
    return launch_status("embed_bwd_wte_smem_kernel");
  }
  const long long total = static_cast<long long>(M) * C4;
  embed_bwd_wte_direct_kernel<<<grid_for(total, 256), 256, 0, stream>>>(idx, reinterpret_cast<const float4*>(dx), dwte,
                                                                        total, C4, V, drop);
  return launch_status("embed_bwd_wte_direct_kernel");
}

int add_pos(const float* e, const float* wpe, float* x, int M, int T, int C, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(e && wpe && x && M > 0 && T > 0 && C % 4 == 0, "add_pos: bad arguments");
  const long long total = static_cast<long long>(M) * (C / 4);
  add_pos_kernel<<<grid_for(total, 256), 256, 0, stream>>>(reinterpret_cast<const float4*>(e), reinterpret_cast<const float4*>(wpe),
                                                           reinterpret_cast<float4*>(x), total, T, C / 4);
  return launch_status("add_pos_kernel");
}
int set_first_pos(const float* first, const float* wpe, float* x, int B, int T, int C, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(first && wpe && x && B > 0 && T > 0 && C % 4 == 0, "set_first_pos: bad arguments");
  const long long total = static_cast<long long>(B) * (C / 4);
  set_first_pos_kernel<<<static_cast<int>((total + 255) / 256), 256, 0, stream>>>(
      reinterpret_cast<const float4*>(first), reinterpret_cast<const float4*>(wpe), reinterpret_cast<float4*>(x), B, T, C / 4);
  return launch_status("set_first_pos_kernel");
}
int pos_bwd(const float* dx, float* dwpe, int M, int T, int C, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(dx && dwpe && M > 0 && T > 0 && M % T == 0 && C % 4 == 0, "pos_bwd: bad arguments");
  const long long n = static_cast<long long>(T) * (C / 4);
  int slices, per_slice;
  wpe_slices(M / T, n, &slices, &per_slice);
  embed_bwd_wpe_kernel<<<dim3(static_cast<unsigned>((n + 127) / 128), slices), 128, 0, stream>>>(
      reinterpret_cast<const float4*>(dx), reinterpret_cast<float4*>(dwpe), M / T, T, C / 4, per_slice, make_drop(0.f, 0));
  return launch_status("embed_bwd_wpe_kernel");
}
int onehot_bf16(const int64_t* tok, void* out, int M, int S, int V, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(tok && out && M > 0 && S > 0 && V > 0, "onehot_bf16: bad arguments");
  const long long total = static_cast<long long>(M) * S;
  ABCGPT_CUDA(cudaMemsetAsync(out, 0, static_cast<size_t>(total) * V * 2, stream));
  onehot_bf16_kernel<<<static_cast<int>((total + 255) / 256), 256, 0, stream>>>(tok, reinterpret_cast<__nv_bfloat16*>(out), total, S, V);
  return launch_status("onehot_bf16_kernel");
}

int ce_fwd(const void* logits, long long ldl, const int64_t* targets, float* row_loss, int M, int V,
           cudaStream_t stream) {
  ABCGPT_CHECK_ARG(logits && targets && row_loss && M > 0 && V > 0 && ldl >= V, "ce_fwd: bad arguments");
  ce_fwd_kernel<<<(M + 7) / 8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, targets, row_loss,
                                                 M, V);
  return launch_status("ce_fwd_kernel");
}
int ce_finalize(const float* row_loss, const int64_t* targets, int M, float* loss_sum_count, float* loss,
                cudaStream_t stream) {
  ABCGPT_CHECK_ARG(row_loss && targets && loss_sum_count && M > 0, "ce_finalize: bad arguments");
  ce_finalize_kernel<<<1, 1024, 0, stream>>>(row_loss, targets, M, loss_sum_count, loss);
  return launch_status("ce_finalize_kernel");
}
int ce_bwd(const void* logits, long long ldl, const int64_t* targets, const float* loss_sum_count,
           const float* grad_loss, void* dlogits, int M, int V, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(logits && targets && loss_sum_count && grad_loss && dlogits && M > 0 && V > 0 && ldl >= V,
                   "ce_bwd: bad arguments");
  ce_bwd_kernel<<<(M + 7) / 8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, targets,
                                                 loss_sum_count, grad_loss, reinterpret_cast<__nv_bfloat16*>(dlogits), M,
                                                 V);
  return launch_status("ce_bwd_kernel");
}

int add_pos_varlen(const float* e, const float* wpe, float* x, const int32_t* cu_seqlens, int n_seqs, int total_rows, int C,
                   cudaStream_t stream) {
  ABCGPT_CHECK_ARG(e && wpe && x && cu_seqlens && n_seqs > 0 && total_rows > 0 && C % 4 == 0, "add_pos_varlen: bad arguments");
  add_pos_varlen_kernel<<<total_rows, 128, 0, stream>>>(reinterpret_cast<const float4*>(e), reinterpret_cast<const float4*>(wpe),
                                                       reinterpret_cast<float4*>(x), cu_seqlens, n_seqs, C / 4);
  return launch_status("add_pos_varlen_kernel");
}
int pos_bwd_varlen(const float* dx, float* dwpe, const int32_t* cu_seqlens, int n_seqs, int max_len, int C, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(dx && dwpe && cu_seqlens && n_seqs > 0 && max_len > 0 && C % 4 == 0, "pos_bwd_varlen: bad arguments");
  const int C4 = C / 4;
  pos_bwd_varlen_kernel<<<dim3(max_len, (C4 + 127) / 128), 128, 0, stream>>>(reinterpret_cast<const float4*>(dx),
                                                                              reinterpret_cast<float4*>(dwpe), cu_seqlens, n_seqs, C4);
  return launch_status("pos_bwd_varlen_kernel");
}
int ce_group_weights(const int64_t* targets, const int32_t* row_group, int n_groups, int M, int V, float* w, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(targets && row_group && w && M > 0 && V > 0, "ce_group_weights: bad arguments");
  ABCGPT_CHECK_ARG(n_groups > 0 && n_groups <= kMaxCeGroups, "ce_group_weights: n_groups must lie in [1, %d] (got %d)", kMaxCeGroups,
                   n_groups);
  ce_group_weights_kernel<<<1, 1024, n_groups * sizeof(int), stream>>>(targets, row_group, n_groups, M, V, w);
  return launch_status("ce_group_weights_kernel");
}
int ce_finalize_weighted(const float* row_loss, const float* weights, int M, float* loss, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(row_loss && weights && loss && M > 0, "ce_finalize_weighted: bad arguments");
  ce_finalize_weighted_kernel<<<1, 1024, 0, stream>>>(row_loss, weights, M, loss);
  return launch_status("ce_finalize_weighted_kernel");
}
int ce_bwd_weighted(const void* logits, long long ldl, const int64_t* targets, const float* weights, const float* grad_loss,
                    void* dlogits, int M, int V, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(logits && targets && weights && grad_loss && dlogits && M > 0 && V > 0 && ldl >= V, "ce_bwd_weighted: bad arguments");
  ce_bwd_weighted_kernel<<<(M + 7) / 8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, targets, weights,
                                                          grad_loss, reinterpret_cast<__nv_bfloat16*>(dlogits), M, V);
  return launch_status("ce_bwd_weighted_kernel");
}

int sumsq(const float* g, long long n, float* out, float* workspace, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(g && out && workspace && n > 0, "sumsq: bad arguments");
  ABCGPT_CHECK_ARG((reinterpret_cast<uintptr_t>(g) & 15) == 0, "sumsq: pointer must be 16-byte aligned");
  sumsq_kernel<<<kSumsqBlocks, 512, 0, stream>>>(g, n, workspace);
  int rc = launch_status("sumsq_kernel");
  if (rc) return rc;
  sumsq_final_kernel<<<1, 1024, 0, stream>>>(workspace, kSumsqBlocks, out);
  return launch_status("sumsq_final_kernel");
}

int adamw(float* p, const float* g, float* m, float* v, void* shadow_bf16, long long n, float lr, float beta1,
          float beta2, float eps, float weight_decay, int step, const float* sumsq_ptr, float max_norm,
          cudaStream_t stream) {
  ABCGPT_CHECK_ARG(p && g && m && v && n > 0 && step >= 1, "adamw: bad arguments");
  ABCGPT_CHECK_ARG(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15) == 0 && (reinterpret_cast<uintptr_t>(shadow_bf16) & 7) == 0,
                   "adamw: arenas must be 16-byte aligned");
  AdamArgs a;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.wd = weight_decay; a.max_norm = max_norm;
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), step);
  const double bc2 = 1.0 - pow(static_cast<double>(beta2), step);
  a.step_size = static_cast<float>(static_cast<double>(lr) / bc1);
  a.inv_bc2_sqrt = static_cast<float>(1.0 / sqrt(bc2));
  adamw_kernel<<<grid_for(n / 4 + 1, 512, 4), 512, 0, stream>>>(p, g, m, v, reinterpret_cast<__nv_bfloat16*>(shadow_bf16),
                                                                n, a, sumsq_ptr);
  return launch_status("adamw_kernel");
}

int cast_f32_to_bf16(const float* x, void* y, long long n, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(x && y && n > 0, "cast: bad arguments");
  ABCGPT_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 7) == 0,
                   "cast: pointers must be 16/8-byte aligned");
  cast_kernel<<<grid_for(n / 4 + 1, 512, 4), 512, 0, stream>>>(x, reinterpret_cast<__nv_bfloat16*>(y), n);
  return launch_status("cast_kernel");
}

int attn_decode(const void* cache, void* out, int B, int Tmax, int n_keys, int H, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(cache && out && B > 0 && H > 0 && n_keys > 0 && n_keys <= Tmax, "attn_decode: bad arguments");
  ABCGPT_CHECK_ARG(static_cast<size_t>(n_keys) * 4 <= 200 * 1024, "attn_decode: context too long for the probability buffer");
  const size_t smem = static_cast<size_t>(n_keys) * sizeof(float);
  if (smem > 48 * 1024) {
    static bool done = false;
    if (!done) {
      ABCGPT_CUDA(cudaFuncSetAttribute(attn_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      done = true;
    }
  }
  launch_k(attn_decode_kernel, dim3(B * H), dim3(128), smem, stream, reinterpret_cast<const __nv_bfloat16*>(cache),
                                                   reinterpret_cast<__nv_bfloat16*>(out), Tmax, n_keys, H, H * 64);
  return launch_status("attn_decode_kernel");
}

int sample_batch(const void* data, int token_bytes, long long n_tokens, const int64_t* ix, int64_t* x, int64_t* y, int B, int T,
                 cudaStream_t stream) {
  ABCGPT_CHECK_ARG(data && ix && x && y && B > 0 && T > 0 && n_tokens > T, "sample_batch: bad arguments");
  ABCGPT_CHECK_ARG(token_bytes == 2 || token_bytes == 4, "sample_batch: tokens must be uint16 or uint32");
  const long long total = static_cast<long long>(B) * T;
  if (token_bytes == 2)
    sample_batch_kernel<uint16_t><<<grid_for(total, 256), 256, 0, stream>>>(reinterpret_cast<const uint16_t*>(data), ix, x, y, B, T);
  else
    sample_batch_kernel<uint32_t><<<grid_for(total, 256), 256, 0, stream>>>(reinterpret_cast<const uint32_t*>(data), ix, x, y, B, T);
  return launch_status("sample_batch_kernel");
}

int colsum_bf16(const void* dy, long long ld, int M, int N, float* out, cudaStream_t stream) {
  ABCGPT_CHECK_ARG(dy && out && M > 0 && N > 0 && N % 2 == 0 && ld % 2 == 0, "colsum: bad arguments");
  const int rows_per_block = 1024;
  if (N % 8 == 0 && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0) {
    dim3 grid8((N + 255) / 256, (M + rows_per_block - 1) / rows_per_block);
    colsum8_kernel<<<grid8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(dy), ld, M, N, rows_per_block, out);
    return launch_status("colsum8_kernel");
  }
  dim3 grid((N + 63) / 64, (M + rows_per_block - 1) / rows_per_block);
  colsum_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(dy), ld, M, N, rows_per_block, out);
  return launch_status("colsum_kernel");
}

int argmax_rows(const void* logits, long long ldl, int V, int64_t* out, long long out_stride, int B,
                cudaStream_t stream) {
  ABCGPT_CHECK_ARG(logits && out && V > 0 && B > 0, "argmax: bad arguments");
  argmax_kernel<<<(B + 7) / 8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(logits), ldl, V, out, out_stride, B);
  return launch_status("argmax_kernel");
}

}  // namespace abcgpt
