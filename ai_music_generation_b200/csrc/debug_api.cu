// Debug / micro-benchmark entry points (include/abcgpt_debug.h).  NOT part of the product library: build.py links this file
// and microbench.cu only into libabcgpt_debug.so, which the scripts under tools/ load explicitly.
#include "common.h"
#include "kernels.h"
#include "../../include/abcgpt_debug.h"

namespace abcgpt {
extern unsigned long long* g_gemm_stats;
int tmem_ld_bench(long long*, int, int, int, cudaStream_t);
int mma_bench(long long*, int, int, int, cudaStream_t);
int mma2_bench(long long*, int, int, cudaStream_t);
int pair_probe(const void*, const void*, float*, int, cudaStream_t);
int mufu_bench(long long*, float*, int, int, int, cudaStream_t);
int tmem_mma_bench(long long*, int, int, int, int, int, int, cudaStream_t);
int mufu2_bench(long long*, float*, int, int, int, cudaStream_t);
}  // namespace abcgpt

#define S(stream) reinterpret_cast<cudaStream_t>(stream)

extern "C" {

/* debug: device pointer to 8 uint64 cycle counters filled by subsequent GEMM launches (NULL disables) */
int abcgpt_debug_gemm_stats(void* device_counters) {
  abcgpt::g_gemm_stats = reinterpret_cast<unsigned long long*>(device_counters);
  return 0;
}

/* debug: cycles of `iters` x (inflight x tcgen05.ld 32x32b.x32 + wait) on nwarps warps of one CTA; out[warp] */
int abcgpt_debug_tmem_ld_bench(void* out, int iters, int nwarps, int inflight, void* stream) {
  return abcgpt::tmem_ld_bench(reinterpret_cast<long long*>(out), iters, nwarps, inflight, S(stream));
}

/* debug: cycles of 4 x iters tcgen05.mma 128 x n x 16 (mode: A 0 smem K-major / 1 smem MN-major / 2 TMEM; +4 B MN-major) */
int abcgpt_debug_mma_bench(void* out, int iters, int n, int mode, void* stream) {
  if (mode < 0) return abcgpt::mma2_bench(reinterpret_cast<long long*>(out), iters, n, S(stream));  /* CTA pair, 256 x n x 16 */
  return abcgpt::mma_bench(reinterpret_cast<long long*>(out), iters, n, mode, S(stream));
}

/* debug: D[256,64] fp32 = A[256,64] bf16 x B[64,64] bf16 through one CTA-pair MMA chain (operand-format probe, tools/pair_probe.py) */
int abcgpt_debug_pair_probe(const void* a, const void* b, void* d, int mode, void* stream) {
  return abcgpt::pair_probe(a, b, reinterpret_cast<float*>(d), mode, S(stream));
}

/* debug: cycles of iters x 16 independent ex2 (mode 0), fma + ex2 (1) or an FMA-pipe exp2 (2) per thread, `warps` warps of one CTA; out[warp] */
int abcgpt_debug_mufu_bench(void* out, void* sink, int iters, int warps, int mode, void* stream) {
  return abcgpt::mufu_bench(reinterpret_cast<long long*>(out), reinterpret_cast<float*>(sink), iters, warps, mode, S(stream));
}

/* debug: tcgen05.ld cost while warp 1 issues 4 x mma_iters tcgen05.mma 128 x mma_n x 16 (mma_iters = 0: idle tensor core);
 * out[0] = MMA chain cycles, out[2 + w] = cycles of `iters` x (inflight x ld (x16: 32x32b.x16, else .x32) + wait) on load warp w */
int abcgpt_debug_tmem_mma_bench(void* out, int iters, int nwarps, int x16, int inflight, int mma_n, int mma_iters, void* stream) {
  return abcgpt::tmem_mma_bench(reinterpret_cast<long long*>(out), iters, nwarps, x16, inflight, mma_n, mma_iters, S(stream));
}

/* debug: MUFU.EX2 rate by operand format, compile-time modes (csrc/microbench.cu mufu2_bench_kernel); out[warp] = cycles */
int abcgpt_debug_mufu2_bench(void* out, void* sink, int iters, int warps, int mode, void* stream) {
  return abcgpt::mufu2_bench(reinterpret_cast<long long*>(out), reinterpret_cast<float*>(sink), iters, warps, mode, S(stream));
}

}  // extern "C"
