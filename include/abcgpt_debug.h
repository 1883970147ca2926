/*
 * libabcgpt_debug — instrumentation and hardware micro-benchmarks used by the scripts under tools/ (tools/gemm_stats.py,
 * tools/gemm_timeline.py, tools/mma_bench.py, tools/tmem_bench.py).  These entry points are NOT in
 * the product library libabcgpt.so: `python -m ai_music_generation_b200.build --debug` links them (csrc/debug_api.cu,
 * csrc/microbench.cu) together with the product objects into libabcgpt_debug.so.
 */
#ifndef ABCGPT_DEBUG_H_
#define ABCGPT_DEBUG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Debug aid: device pointer to 16 uint64 counters accumulated by subsequent GEMM launches (NULL disables): cycles
 * [0] producer empty-wait [1] MMA full-wait [2] MMA tmem-empty wait [3] epilogue tmem-full wait [5] CTA total; pair kernel
 * only, %globaltimer nanoseconds over all CTAs (the caller presets the min slots to ~0): [8] min kernel entry, [9] max / [15] min
 * prologue done, [10] min / [11] max first operand stage landed, [12] max last MMA committed, [13] max epilogue done, [14] max exit. */
int abcgpt_debug_gemm_stats(void* device_counters);
int abcgpt_debug_mma_bench(void* out, int iters, int n, int mode, void* stream);
int abcgpt_debug_tmem_ld_bench(void* out, int iters, int nwarps, int inflight, void* stream);
/* Operand-format probe of the CTA-pair MMA: d[256,64] fp32 = a[256,64] bf16 x B; mode bit 0: b is B^T [n][k] (K-major halves) instead
 * of B [k][n] (MN-major column halves, 64-byte swizzle); bit 1: A is staged through tensor memory. */
/* MUFU.EX2 rate: cycles of iters x 16 independent ex2 per thread (mode 0), fma + ex2 (1), FMA-pipe-only exp2 (2); out[warp] */
int abcgpt_debug_mufu_bench(void* out, void* sink, int iters, int warps, int mode, void* stream);
/* tcgen05.ld under tensor-core load: see csrc/microbench.cu (tools/tmem_mma_bench.py) */
int abcgpt_debug_tmem_mma_bench(void* out, int iters, int nwarps, int x16, int inflight, int mma_n, int mma_iters, void* stream);
/* MUFU.EX2 rate by operand format (f32, f16x2, bf16x2, the fp32 softmax pattern, the packed-f16 alternative); tools/mufu2_bench.py */
int abcgpt_debug_mufu2_bench(void* out, void* sink, int iters, int warps, int mode, void* stream);
int abcgpt_debug_pair_probe(const void* a, const void* b, void* d, int mode, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ABCGPT_DEBUG_H_ */
