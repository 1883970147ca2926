// Head sizes 32 and 128 over dense batches (abcgpt_attn_fwd_hd / abcgpt_attn_bwd_hd: the host side of the flash kernels of
// attn_hd.cuh) and their single-token decode (abcgpt_attn_decode_hd).
#include "attn_hd.cuh"

namespace abcgpt {
namespace {

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
  if (dcfg.thr16 == 0) launch_k(attn_fwd_hd_kernel<D, false>, grid, dim3(kThreads), S::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, dcfg, VarlenSeqs{});
  else launch_k(attn_fwd_hd_kernel<D, true>, grid, dim3(kThreads), S::TOTAL, stream, tmQ, tmKV, o, lse, T, H, C, dcfg, VarlenSeqs{});
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
    launch_k(attn_bwd_dkv_hd_kernel<D, false>, grid, dim3(kThreads), Skv::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, g, T, H, C, dcfg, VarlenSeqs{});
    if ((rc = launch_status("attn_bwd_dkv_hd_kernel"))) return rc;
    launch_k(attn_bwd_dq_hd_kernel<D, false>, grid, dim3(kThreads), Sq::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, g, T, H, C, dcfg, VarlenSeqs{});
  } else {
    launch_k(attn_bwd_dkv_hd_kernel<D, true>, grid, dim3(kThreads), Skv::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, g, T, H, C, dcfg, VarlenSeqs{});
    if ((rc = launch_status("attn_bwd_dkv_hd_kernel"))) return rc;
    launch_k(attn_bwd_dq_hd_kernel<D, true>, grid, dim3(kThreads), Sq::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, g, T, H, C, dcfg, VarlenSeqs{});
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
