// extern "C" surface of libabcgpt (declared in include/abcgpt.h).  Plain pointers and sizes only; no torch
// types, no exceptions across the boundary.
#include "common.h"
#include "kernels.h"
#include <string.h>

using namespace abcgpt;

#define S(stream) reinterpret_cast<cudaStream_t>(stream)

extern "C" {

int abcgpt_version(void) { return ABCGPT_VERSION; }
const char* abcgpt_last_error(void) { return last_error_buf(); }

int abcgpt_gemm_bf16(const void* a, int a_mn_major, int64_t lda, const void* b, int b_mn_major, int64_t ldb, int M,
                     int N, int K, int epilogue, void* c, int64_t ldc, void* c2, int64_t ldc2, const void* aux,
                     int64_t ldaux, const float* bias, int tile_n, int splits, float dropout_p, uint32_t dropout_key,
                     void* stream) {
  return gemm_bf16(a, a_mn_major, lda, b, b_mn_major, ldb, M, N, K, epilogue, c, ldc, c2, ldc2, aux, ldaux, bias,
                   tile_n, splits, dropout_p, dropout_key, S(stream));
}

int abcgpt_embed_fwd(const int64_t* idx, const float* wte, const float* wpe, float* x, int M, int T, int C, int V,
                     float dropout_p, uint32_t dropout_key, void* stream) {
  return embed_fwd(idx, wte, wpe, x, M, T, C, V, dropout_p, dropout_key, S(stream));
}
int abcgpt_embed_bwd(const int64_t* idx, const float* dx, float* dwte, float* dwpe, int M, int T, int C, int V,
                     float dropout_p, uint32_t dropout_key, void* stream) {
  return embed_bwd(idx, dx, dwte, dwpe, M, T, C, V, dropout_p, dropout_key, S(stream));
}

/* hierarchical (TunesFormer-shaped) decoders: embeddings supplied by another network, one-hot patch rows */
int abcgpt_add_pos(const float* e, const float* wpe, float* x, int M, int T, int C, void* stream) {
  return add_pos(e, wpe, x, M, T, C, S(stream));
}
int abcgpt_set_first_pos(const float* first, const float* wpe, float* x, int B, int T, int C, void* stream) {
  return set_first_pos(first, wpe, x, B, T, C, S(stream));
}
int abcgpt_pos_bwd(const float* dx, float* dwpe, int M, int T, int C, void* stream) {
  return pos_bwd(dx, dwpe, M, T, C, S(stream));
}
int abcgpt_onehot_bf16(const int64_t* tok, void* out, int M, int S_, int V, void* stream) {
  return onehot_bf16(tok, out, M, S_, V, S(stream));
}

int abcgpt_layernorm_fwd(const float* x, const float* weight, const float* bias, void* y_bf16, float* y_f32,
                         float* mean, float* rstd, int M, int C, void* stream) {
  return layernorm_fwd(x, weight, bias, y_bf16, y_f32, mean, rstd, M, C, S(stream));
}
int abcgpt_layernorm_fwd_resid(const float* x_in, const void* branch_bf16, float* x_out, const float* weight, const float* bias,
                               void* y_bf16, float* mean, float* rstd, int M, int C, float dropout_p, uint32_t dropout_key,
                               void* stream) {
  return layernorm_fwd_resid(x_in, branch_bf16, x_out, weight, bias, y_bf16, mean, rstd, M, C, dropout_p, dropout_key, S(stream));
}
int abcgpt_layernorm_bwd(const void* dy_bf16, const float* x, const float* weight, const float* mean,
                         const float* rstd, const float* dresid_in, float* dx_out, void* dx_bf16, float* dweight,
                         float* dbias, int M, int C, float dropout_p, uint32_t dropout_key, void* stream) {
  return layernorm_bwd(dy_bf16, x, weight, mean, rstd, dresid_in, dx_out, dx_bf16, dweight, dbias, M, C, dropout_p,
                       dropout_key, S(stream));
}

int abcgpt_attn_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, float dropout_p, uint32_t dropout_key,
                    void* stream) {
  return attn_fwd(qkv, out, lse, B, T, H, dropout_p, dropout_key, S(stream));
}
int abcgpt_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv,
                    int B, int T, int H, float dropout_p, uint32_t dropout_key, void* stream) {
  return attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, dropout_p, dropout_key, S(stream));
}
int abcgpt_attn_fwd_hd(const void* qkv, void* out, float* lse, int B, int T, int H, int head_size, float dropout_p,
                       uint32_t dropout_key, void* stream) {
  if (head_size == 64) return abcgpt_attn_fwd(qkv, out, lse, B, T, H, dropout_p, dropout_key, stream);
  return attn_fwd_hd(qkv, out, lse, B, T, H, head_size, dropout_p, dropout_key, S(stream));
}
int abcgpt_attn_bwd_hd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, int B,
                       int T, int H, int head_size, float dropout_p, uint32_t dropout_key, void* stream) {
  if (head_size == 64) return abcgpt_attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, dropout_p, dropout_key, stream);
  return attn_bwd_hd(qkv, out, dout, lse, delta, dqkv, B, T, H, head_size, dropout_p, dropout_key, S(stream));
}

int abcgpt_ce_fwd(const void* logits, int64_t ldl, const int64_t* targets, float* row_loss, int M, int V,
                  void* stream) {
  return ce_fwd(logits, ldl, targets, row_loss, M, V, S(stream));
}
int abcgpt_ce_finalize(const float* row_loss, const int64_t* targets, int M, float* loss_sum_count, float* loss,
                       void* stream) {
  return ce_finalize(row_loss, targets, M, loss_sum_count, loss, S(stream));
}
int abcgpt_ce_bwd(const void* logits, int64_t ldl, const int64_t* targets, const float* loss_sum_count,
                  const float* grad_loss, void* dlogits, int M, int V, void* stream) {
  return ce_bwd(logits, ldl, targets, loss_sum_count, grad_loss, dlogits, M, V, S(stream));
}

int abcgpt_sumsq(const float* g, int64_t n, float* out, float* workspace, void* stream) {
  return sumsq(g, n, out, workspace, S(stream));
}
int abcgpt_adamw(float* p, const float* g, float* m, float* v, void* shadow_bf16, int64_t n, float lr, float beta1,
                 float beta2, float eps, float weight_decay, int step, const float* sumsq_ptr, float max_norm,
                 void* stream) {
  return adamw(p, g, m, v, shadow_bf16, n, lr, beta1, beta2, eps, weight_decay, step, sumsq_ptr, max_norm, S(stream));
}
int abcgpt_cast_f32_to_bf16(const float* x, void* y_bf16, int64_t n, void* stream) {
  return cast_f32_to_bf16(x, y_bf16, n, S(stream));
}
int abcgpt_attn_decode(const void* cache, void* out, int B, int Tmax, int n_keys, int H, void* stream) {
  return attn_decode(cache, out, B, Tmax, n_keys, H, S(stream));
}
int abcgpt_attn_decode_hd(const void* qkv_row, void* cache, void* out, int B, int Tmax, int t, int H, int head_size,
                          void* stream) {
  return attn_decode_hd(qkv_row, cache, out, B, Tmax, t, H, head_size, S(stream));
}
int abcgpt_sample_batch(const void* data, int token_bytes, int64_t n_tokens, const int64_t* ix, int64_t* x, int64_t* y, int B,
                        int T, void* stream) {
  return sample_batch(data, token_bytes, n_tokens, ix, x, y, B, T, S(stream));
}
int abcgpt_colsum_bf16(const void* dy, int64_t ld, int M, int N, float* out, void* stream) {
  return colsum_bf16(dy, ld, M, N, out, S(stream));
}
int abcgpt_argmax(const void* logits, int64_t ldl, int V, int64_t* out, int64_t out_stride, int B, void* stream) {
  return argmax_rows(logits, ldl, V, out, out_stride, B, S(stream));
}
int abcgpt_sample_topk(const void* logits, int64_t ldl, int V, float temperature, int top_k, const void* seed,
                       int64_t counter, int64_t* out, int64_t out_stride, int B, void* stream) {
  return sample_topk(logits, ldl, V, temperature, top_k, seed, counter, out, out_stride, B, S(stream));
}
int abcgpt_sample_top_p(const void* logits, int64_t ldl, int V, float top_p, int top_k, float temperature, const void* seed,
                        const void* counter_base, int64_t counter, const int64_t* row_id, int64_t* out, int64_t out_stride, int B,
                        void* stream) {
  return sample_top_p(logits, ldl, V, top_p, top_k, temperature, seed, counter_base, counter, row_id, out, out_stride, B,
                      S(stream));
}

/*
 * Replay of a recorded launch list with position-affine arguments (the decode loop of GPT.generate is launch-bound: ~90
 * launches per generated token, ~10 us of Python / ctypes each).  prog: per call [function id, nargs, (value, delta) x nargs];
 * every argument is passed as value + k * delta; pointers and integers as int64, floats as the bit pattern of a double.
 */
static inline float abcgpt_word_f(int64_t w) {
  double d;
  memcpy(&d, &w, sizeof(d));
  return static_cast<float>(d);
}
#define P_(i) reinterpret_cast<void*>(a[i])
#define CP_(T, i) reinterpret_cast<const T*>(a[i])
#define MP_(T, i) reinterpret_cast<T*>(a[i])
#define I_(i) static_cast<int>(a[i])
int abcgpt_replay(const int64_t* prog, int64_t n_words, int64_t k) {
  int64_t i = 0;
  while (i < n_words) {
    const int64_t fn = prog[i], nargs = prog[i + 1];
    if (nargs < 0 || nargs > 24 || i + 2 + 2 * nargs > n_words) return fail(-1, "abcgpt_replay: malformed program at word %lld", (long long)i);
    int64_t a[24];
    for (int64_t j = 0; j < nargs; ++j) a[j] = prog[i + 2 + 2 * j] + k * prog[i + 3 + 2 * j];
    i += 2 + 2 * nargs;
    int rc = 0;
    switch (fn) {
      case ABCGPT_FN_GEMM:
        if (nargs != 22) return fail(-1, "abcgpt_replay: gemm takes 22 arguments");
        rc = abcgpt_gemm_bf16(P_(0), I_(1), a[2], P_(3), I_(4), a[5], I_(6), I_(7), I_(8), I_(9), P_(10), a[11], P_(12), a[13], P_(14),
                              a[15], CP_(float, 16), I_(17), I_(18), abcgpt_word_f(a[19]), static_cast<uint32_t>(a[20]), P_(21));
        break;
      case ABCGPT_FN_EMBED_FWD:
        if (nargs != 11) return fail(-1, "abcgpt_replay: embed_fwd takes 11 arguments");
        rc = abcgpt_embed_fwd(CP_(int64_t, 0), CP_(float, 1), CP_(float, 2), MP_(float, 3), I_(4), I_(5), I_(6), I_(7),
                              abcgpt_word_f(a[8]), static_cast<uint32_t>(a[9]), P_(10));
        break;
      case ABCGPT_FN_LAYERNORM_FWD:
        if (nargs != 10) return fail(-1, "abcgpt_replay: layernorm_fwd takes 10 arguments");
        rc = abcgpt_layernorm_fwd(CP_(float, 0), CP_(float, 1), CP_(float, 2), P_(3), MP_(float, 4), MP_(float, 5), MP_(float, 6), I_(7),
                                  I_(8), P_(9));
        break;
      case ABCGPT_FN_ATTN_DECODE:
        if (nargs != 7) return fail(-1, "abcgpt_replay: attn_decode takes 7 arguments");
        rc = abcgpt_attn_decode(P_(0), P_(1), I_(2), I_(3), I_(4), I_(5), P_(6));
        break;
      case ABCGPT_FN_ARGMAX:
        if (nargs != 7) return fail(-1, "abcgpt_replay: argmax takes 7 arguments");
        rc = abcgpt_argmax(P_(0), a[1], I_(2), MP_(int64_t, 3), a[4], I_(5), P_(6));
        break;
      case ABCGPT_FN_ATTN_DECODE_HD:
        if (nargs != 9) return fail(-1, "abcgpt_replay: attn_decode_hd takes 9 arguments");
        rc = abcgpt_attn_decode_hd(CP_(void, 0), P_(1), P_(2), I_(3), I_(4), I_(5), I_(6), I_(7), P_(8));
        break;
      case ABCGPT_FN_SAMPLE_TOPK:
        if (nargs != 11) return fail(-1, "abcgpt_replay: sample_topk takes 11 arguments");
        rc = abcgpt_sample_topk(P_(0), a[1], I_(2), abcgpt_word_f(a[3]), I_(4), P_(5), a[6], MP_(int64_t, 7), a[8], I_(9), P_(10));
        break;
      case ABCGPT_FN_SAMPLE_TOP_P:
        if (nargs != 14) return fail(-1, "abcgpt_replay: sample_top_p takes 14 arguments");
        rc = abcgpt_sample_top_p(P_(0), a[1], I_(2), abcgpt_word_f(a[3]), I_(4), abcgpt_word_f(a[5]), P_(6), P_(7), a[8],
                                 CP_(int64_t, 9), MP_(int64_t, 10), a[11], I_(12), P_(13));
        break;
      default:
        return fail(-1, "abcgpt_replay: unknown function id %lld", (long long)fn);
    }
    if (rc) return rc;
  }
  return 0;
}
#undef P_
#undef CP_
#undef MP_
#undef I_

/* Programmatic dependent launch for subsequent launches of this process (GEMM, attention, LayerNorm, decode attention):
 * the next kernel's CTAs become resident and run their prologue while the previous kernel drains.  Pays on chains of small
 * kernels (a decoded token); default off. */
int abcgpt_set_pdl(int on) {
  abcgpt::set_pdl(on != 0);
  return 0;
}

/* Cross-stream ordering for launch plans that run independent kernels on a second stream (the weight-gradient GEMMs of the
 * backward, ai_music_generation_b200/model.py): `abcgpt_event_record(slot, stream)` marks the work enqueued on `stream` so far,
 * `abcgpt_event_wait(slot, stream)` makes `stream` wait (on the device) for the most recent mark of `slot`.  Slots are small
 * integers owned by the caller; the events live per device inside the library (created on first use, no timing). */
namespace {
constexpr int kEventSlots = 1024, kEventDevs = 16;
cudaEvent_t g_events[kEventDevs][kEventSlots];
bool g_event_made[kEventDevs][kEventSlots];
int event_of(int slot, cudaEvent_t* ev) {
  int dev = 0;
  ABCGPT_CUDA(cudaGetDevice(&dev));
  if (slot < 0 || slot >= kEventSlots || dev < 0 || dev >= kEventDevs) return fail(-1, "event slot %d / device %d out of range", slot, dev);
  if (!g_event_made[dev][slot]) {
    ABCGPT_CUDA(cudaEventCreateWithFlags(&g_events[dev][slot], cudaEventDisableTiming));
    g_event_made[dev][slot] = true;
  }
  *ev = g_events[dev][slot];
  return 0;
}
}  // namespace
int abcgpt_event_record(int slot, void* stream) {
  cudaEvent_t ev;
  if (int rc = event_of(slot, &ev)) return rc;
  ABCGPT_CUDA(cudaEventRecord(ev, S(stream)));
  return 0;
}
int abcgpt_event_wait(int slot, void* stream) {
  cudaEvent_t ev;
  if (int rc = event_of(slot, &ev)) return rc;
  ABCGPT_CUDA(cudaStreamWaitEvent(S(stream), ev, 0));
  return 0;
}

/* Data-parallel gradient exchange over NVLink-switch multicast memory, fused with the clip norm (csrc/nvls.cu) */
int abcgpt_nvls_allreduce_sumsq(void* grad_multicast, int64_t n, int rank, int world, float scale, void* partials_multicast,
                                int blocks_per_rank, int threads_per_block, void* stream) {
  return nvls_allreduce_sumsq(grad_multicast, n, rank, world, scale, partials_multicast, blocks_per_rank, threads_per_block, S(stream));
}
int abcgpt_sumsq_partials(const float* partials, int nparts, float* out, void* stream) {
  return sumsq_partials(partials, nparts, out, S(stream));
}

/* Ticket-based tile scheduler of the CTA-pair GEMM for the launches that follow (0 = static round-robin, the default): resident
 * pairs absorb the tiles of pairs that share their SM with another stream's kernel — with the gradient exchange running in a few
 * small CTAs beside the backward a static schedule waits for the slowest SM (+13..48 % per GEMM, tools/coresidency_probe.py), the
 * dynamic one loses 3-7 %. */
int abcgpt_set_dynamic_tiles(int on) {
  abcgpt::set_dynamic_tiles(on != 0);
  return 0;
}

}  // extern "C"
