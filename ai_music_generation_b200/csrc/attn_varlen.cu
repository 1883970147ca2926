// Causal attention over packed sequences of arbitrary lengths (abcgpt_attn_varlen_fwd / abcgpt_attn_varlen_bwd): sequence s is
// the rows [cu_seqlens[s], cu_seqlens[s+1]) of the qkv / out / dqkv buffers; attention is causal inside it and never crosses
// into another.  The kernels are the templated flash kernels of attn_hd.cuh, instantiated for head sizes 32, 64 and 128 with
// the varlen item decode (HdItem): grid (n_seqs * H, ceil(max_len / 128)); CTA (s * H + h, y) takes query tile ntiles(s)-1-y
// (forward, dQ) or key tile y (dK / dV) of sequence s and returns at once when s has no such tile.  The host sizes the grid
// from n_seqs and max_len alone and never reads the sequence table, so a launch needs no host synchronisation and its
// arguments do not depend on how the rows are split.  lse / delta: fp32 [H, total_rows].
#include "attn_hd.cuh"

namespace abcgpt {
namespace {

int check_varlen(const char* who, const int32_t* cu_seqlens, int n_seqs, int max_len, int total_rows, int H, int D,
                 float drop_p) {
  ABCGPT_CHECK_ARG(D == 32 || D == 64 || D == 128, "%s: head size %d is not supported (supported head sizes: 32, 64, 128)", who, D);
  ABCGPT_CHECK_ARG(drop_p == 0.f, "%s: attention dropout over packed sequences is not implemented (dropout_p must be 0)", who);
  ABCGPT_CHECK_ARG(cu_seqlens != nullptr, "%s: null sequence table", who);
  ABCGPT_CHECK_ARG(n_seqs > 0 && max_len > 0 && total_rows > 0 && H > 0, "%s: bad shape n_seqs=%d max_len=%d total_rows=%d H=%d",
                   who, n_seqs, max_len, total_rows, H);
  ABCGPT_CHECK_ARG(static_cast<long long>(n_seqs) * H < (1ll << 31) - 1, "%s: too many sequence*head items", who);
  ABCGPT_CHECK_ARG((max_len + 127) / 128 <= 65535, "%s: sequence too long", who);
  return 0;
}

template <int D>
int fwd_varlen(const void* qkv, void* out, float* lse, const VarlenSeqs& vs, int n_seqs, int max_len, int H, cudaStream_t stream) {
  using S = FwdHdSmem<D>;
  const int C = H * D;
  CUtensorMap tmQ, tmKV;
  int rc;
  if ((rc = tmap_hd<D>(&tmQ, qkv, 3ull * C, static_cast<uint64_t>(vs.total), 128))) return rc;
  if ((rc = tmap_hd<D>(&tmKV, qkv, 3ull * C, static_cast<uint64_t>(vs.total), 64))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = prepare(attn_fwd_hd_kernel<D, false, true>, S::TOTAL))) return rc;
    done = true;
  }
  const dim3 grid(n_seqs * H, (max_len + 127) / 128);
  launch_k(attn_fwd_hd_kernel<D, false, true>, grid, dim3(kThreads), S::TOTAL, stream, tmQ, tmKV,
           reinterpret_cast<__nv_bfloat16*>(out), lse, 0, H, C, make_drop(0.f, 0), vs);
  return launch_status("attn_fwd_hd_kernel (varlen)");
}

template <int D>
int bwd_varlen(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv, const VarlenSeqs& vs,
               int n_seqs, int max_len, int H, cudaStream_t stream) {
  using Sq = DqHdSmem<D>;
  using Skv = DkvHdSmem<D>;
  const int C = H * D;
  const uint64_t rows = static_cast<uint64_t>(vs.total);
  CUtensorMap tmQKV128, tmQKV64, tmDO128, tmDO64;
  int rc;
  if ((rc = tmap_hd<D>(&tmQKV128, qkv, 3ull * C, rows, 128))) return rc;
  if ((rc = tmap_hd<D>(&tmQKV64, qkv, 3ull * C, rows, 64))) return rc;
  if ((rc = tmap_hd<D>(&tmDO128, dout, static_cast<uint64_t>(C), rows, 128))) return rc;
  if ((rc = tmap_hd<D>(&tmDO64, dout, static_cast<uint64_t>(C), rows, 64))) return rc;
  static bool done = false;
  if (!done) {
    if ((rc = prepare(attn_bwd_dq_hd_kernel<D, false, true>, Sq::TOTAL))) return rc;
    if ((rc = prepare(attn_bwd_dkv_hd_kernel<D, false, true>, Skv::TOTAL))) return rc;
    done = true;
  }
  // delta [H, total_rows] is the dense [B = 1, H, T = total_rows] layout
  launch_k(attn_delta_hd_kernel<D>, dim3(static_cast<unsigned>((rows + 7) / 8)), dim3(256), 0, stream,
           reinterpret_cast<const __nv_bfloat16*>(out), reinterpret_cast<const __nv_bfloat16*>(dout), delta, 1, vs.total, H, C);
  if ((rc = launch_status("attn_delta_hd_kernel (varlen)"))) return rc;
  const dim3 grid(n_seqs * H, (max_len + 127) / 128);
  const DropCfg nodrop = make_drop(0.f, 0);
  __nv_bfloat16* g = reinterpret_cast<__nv_bfloat16*>(dqkv);
  launch_k(attn_bwd_dkv_hd_kernel<D, false, true>, grid, dim3(kThreads), Skv::TOTAL, stream, tmQKV128, tmQKV64, tmDO64, lse, delta, g,
           0, H, C, nodrop, vs);
  if ((rc = launch_status("attn_bwd_dkv_hd_kernel (varlen)"))) return rc;
  launch_k(attn_bwd_dq_hd_kernel<D, false, true>, grid, dim3(kThreads), Sq::TOTAL, stream, tmQKV128, tmQKV64, tmDO128, lse, delta, g,
           0, H, C, nodrop, vs);
  return launch_status("attn_bwd_dq_hd_kernel (varlen)");
}

}  // namespace

int attn_varlen_fwd(const void* qkv, void* out, float* lse, const int32_t* cu_seqlens, int n_seqs, int max_len, int total_rows,
                    int H, int D, float drop_p, uint32_t drop_key, cudaStream_t stream) {
  (void)drop_key;
  int rc = check_varlen("attn_varlen_fwd", cu_seqlens, n_seqs, max_len, total_rows, H, D, drop_p);
  if (rc) return rc;
  ABCGPT_CHECK_ARG(qkv && out && lse, "attn_varlen_fwd: null pointer");
  const VarlenSeqs vs{cu_seqlens, total_rows};
  if (D == 32) return fwd_varlen<32>(qkv, out, lse, vs, n_seqs, max_len, H, stream);
  if (D == 64) return fwd_varlen<64>(qkv, out, lse, vs, n_seqs, max_len, H, stream);
  return fwd_varlen<128>(qkv, out, lse, vs, n_seqs, max_len, H, stream);
}

int attn_varlen_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv,
                    const int32_t* cu_seqlens, int n_seqs, int max_len, int total_rows, int H, int D, float drop_p,
                    uint32_t drop_key, cudaStream_t stream) {
  (void)drop_key;
  int rc = check_varlen("attn_varlen_bwd", cu_seqlens, n_seqs, max_len, total_rows, H, D, drop_p);
  if (rc) return rc;
  ABCGPT_CHECK_ARG(qkv && out && dout && lse && delta && dqkv, "attn_varlen_bwd: null pointer");
  const VarlenSeqs vs{cu_seqlens, total_rows};
  if (D == 32) return bwd_varlen<32>(qkv, out, dout, lse, delta, dqkv, vs, n_seqs, max_len, H, stream);
  if (D == 64) return bwd_varlen<64>(qkv, out, dout, lse, delta, dqkv, vs, n_seqs, max_len, H, stream);
  return bwd_varlen<128>(qkv, out, dout, lse, delta, dqkv, vs, n_seqs, max_len, H, stream);
}

}  // namespace abcgpt
