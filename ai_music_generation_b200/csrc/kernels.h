// Internal C++ entry points (one per kernel family); api.cu exposes them through the C ABI in include/abcgpt.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/abcgpt.h"

namespace abcgpt {

int gemm_bf16(const void* a, int a_mn, long long lda, const void* b, int b_mn, long long ldb, int M, int N, int K,
              int epi, void* c, long long ldc, void* c2, long long ldc2, const void* aux, long long ldaux,
              const float* bias, int bn_hint, int splits_hint, float drop_p, uint32_t drop_key, cudaStream_t stream);

int embed_fwd(const int64_t* idx, const float* wte, const float* wpe, float* x, int M, int T, int C, int V, float drop_p,
              uint32_t drop_key, cudaStream_t stream);
int embed_bwd(const int64_t* idx, const float* dx, float* dwte, float* dwpe, int M, int T, int C, int V, float drop_p,
              uint32_t drop_key, cudaStream_t stream);

int add_pos(const float* e, const float* wpe, float* x, int M, int T, int C, cudaStream_t stream);
int set_first_pos(const float* first, const float* wpe, float* x, int B, int T, int C, cudaStream_t stream);
int pos_bwd(const float* dx, float* dwpe, int M, int T, int C, cudaStream_t stream);
int onehot_bf16(const int64_t* tok, void* out, int M, int S, int V, cudaStream_t stream);
// packed sequences: cu_seqlens int32 [n_seqs + 1] row offsets
int add_pos_varlen(const float* e, const float* wpe, float* x, const int32_t* cu_seqlens, int n_seqs, int total_rows, int C,
                   cudaStream_t stream);
int pos_bwd_varlen(const float* dx, float* dwpe, const int32_t* cu_seqlens, int n_seqs, int max_len, int C, cudaStream_t stream);

int layernorm_fwd(const float* x, const float* weight, const float* bias, void* y_bf16, float* y_f32, float* mean,
                  float* rstd, int M, int C, cudaStream_t stream);
int layernorm_fwd_resid(const float* x_in, const void* branch_bf16, float* x_out, const float* weight, const float* bias,
                        void* y_bf16, float* mean, float* rstd, int M, int C, float drop_p, uint32_t drop_key,
                        cudaStream_t stream);
int layernorm_bwd(const void* dy_bf16, const float* x, const float* weight, const float* mean, const float* rstd,
                  const float* dresid_in, float* dx_out, void* dx_bf16, float* dweight, float* dbias, int M, int C,
                  float drop_p, uint32_t drop_key, cudaStream_t stream);

int attn_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, float drop_p, uint32_t drop_key,
             cudaStream_t stream);
int attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, int B,
             int T, int H, float drop_p, uint32_t drop_key, cudaStream_t stream);
// csrc/attn_hd.cu: head sizes 32 and 128
int attn_fwd_hd(const void* qkv, void* out, float* lse, int B, int T, int H, int D, float drop_p, uint32_t drop_key,
                cudaStream_t stream);
int attn_bwd_hd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, int B, int T,
                int H, int D, float drop_p, uint32_t drop_key, cudaStream_t stream);
int attn_decode_hd(const void* qkv_row, void* cache, void* out, int B, int Tmax, int t, int H, int D, cudaStream_t stream);
// csrc/attn_varlen.cu: packed sequences, head sizes 32, 64 and 128
int attn_varlen_fwd(const void* qkv, void* out, float* lse, const int32_t* cu_seqlens, int n_seqs, int max_len, int total_rows,
                    int H, int D, float drop_p, uint32_t drop_key, cudaStream_t stream);
int attn_varlen_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv,
                    const int32_t* cu_seqlens, int n_seqs, int max_len, int total_rows, int H, int D, float drop_p,
                    uint32_t drop_key, cudaStream_t stream);

int ce_fwd(const void* logits, long long ldl, const int64_t* targets, float* row_loss, int M, int V,
           cudaStream_t stream);
int ce_finalize(const float* row_loss, const int64_t* targets, int M, float* loss_sum_count, float* loss,
                cudaStream_t stream);
int ce_bwd(const void* logits, long long ldl, const int64_t* targets, const float* loss_sum_count,
           const float* grad_loss, void* dlogits, int M, int V, cudaStream_t stream);
constexpr int kMaxCeGroups = 12288;   // ce_group_weights: one int counter per group in 48 KB of shared memory
int ce_group_weights(const int64_t* targets, const int32_t* row_group, int n_groups, int M, int V, float* w, cudaStream_t stream);
int ce_finalize_weighted(const float* row_loss, const float* weights, int M, float* loss, cudaStream_t stream);
int ce_bwd_weighted(const void* logits, long long ldl, const int64_t* targets, const float* weights, const float* grad_loss,
                    void* dlogits, int M, int V, cudaStream_t stream);

int sumsq(const float* g, long long n, float* out, float* workspace, cudaStream_t stream);
int adamw(float* p, const float* g, float* m, float* v, void* shadow_bf16, long long n, float lr, float beta1,
          float beta2, float eps, float weight_decay, int step, const float* sumsq, float max_norm,
          cudaStream_t stream);
int cast_f32_to_bf16(const float* x, void* y, long long n, cudaStream_t stream);
int attn_decode(const void* cache, void* out, int B, int Tmax, int n_keys, int H, cudaStream_t stream);
int sample_batch(const void* data, int token_bytes, long long n_tokens, const int64_t* ix, int64_t* x, int64_t* y, int B, int T,
                 cudaStream_t stream);
int nvls_allreduce_sumsq(void* grad_mc, long long n, int rank, int world, float scale, void* partials_mc, int blocks_per_rank,
                         int threads, cudaStream_t stream);
int sumsq_partials(const float* partials, int nparts, float* out, cudaStream_t stream);
int colsum_bf16(const void* dy, long long ld, int M, int N, float* out, cudaStream_t stream);
int argmax_rows(const void* logits, long long ldl, int V, int64_t* out, long long out_stride, int B,
                cudaStream_t stream);
int sample_topk(const void* logits, long long ldl, int V, float temperature, int top_k, const void* seed, long long counter,
                int64_t* out, long long out_stride, int B, cudaStream_t stream);
int sample_top_p(const void* logits, long long ldl, int V, float top_p, int top_k, float temperature, const void* seed,
                 const void* counter_base, long long counter, const int64_t* row_id, int64_t* out, long long out_stride, int B,
                 cudaStream_t stream);
int sample_top_p_cluster(const void* logits, long long ldl, int V, float top_p, int top_k, float temperature, const void* seed,
                         const void* counter_base, long long counter, const int64_t* row_id, int64_t* out, long long out_stride,
                         int B, cudaStream_t stream);

}  // namespace abcgpt
