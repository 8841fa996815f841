// rpx_kernels.cuh — launchers of the non-GEMM kernels (defined in rpx_attention.cu,
// rpx_elementwise.cu, rpx_simtopk.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace rpx {

// ---- rpx_attention.cu
// qkv [T, 3*heads*d_kv] bf16 packed tokens; out [T, heads*d_kv] bf16;
// bias_lut [heads][2*max_distance+1] fp32, entry (delta + max_distance), delta = key - query clamped.
// Throughput: t5_attention_tc_kernel (128-query CTAs, any length).  Latency: t5_attention_short_kernel
// (32-query CTAs, max_len <= 1024, bias table within the shared-memory opt-in), RPX_ERR_UNSUPPORTED outside
// that range.  Auto: the latency kernel where it can run, the throughput kernel otherwise.
enum class AttnKernel { Throughput, Latency, Auto };
int launch_t5_attention(const __nv_bfloat16* qkv, __nv_bfloat16* out, const int32_t* cu_seqlens,
                        const float* bias_lut, int n_tokens, int n_seqs, int max_len, int n_heads, int d_kv,
                        int max_distance, cudaStream_t stream, AttnKernel kernel);
// Whether the throughput kernel (the one every length can use) holds the bias table of `max_distance`.
bool t5_attention_bias_fits(int max_distance);

// ---- rpx_elementwise.cu
// ByT5 tokenisation of packed byte strings into packed token ids (byte + 3, EOS = 1 last,
// truncated to max_seq_len including EOS).  cu_bytes / cu_tokens are [n_seqs + 1] device arrays.
int launch_tokenize_bytes(const uint8_t* bytes, const int64_t* cu_bytes, const int32_t* cu_tokens,
                          int32_t* ids, int n_seqs, int n_tokens, cudaStream_t stream);
// Padded [B, L] int64 ids -> packed ids using cu_tokens (first len_b ids of each row).
int launch_pack_ids(const int64_t* ids, const int32_t* cu_tokens, int32_t* packed, int batch, int seq_len,
                    int n_tokens, int vocab, int32_t* bad_flag, cudaStream_t stream);
// lens[b] = sum(mask[b, :]); flag |= 1 if the mask is not a prefix of ones or a row is empty.
int launch_mask_lengths(const int64_t* mask, int32_t* lens, int32_t* bad_flag, int batch, int seq_len,
                        cudaStream_t stream);
// h32[t] = table[ids[t]] (fp32), h16 = bf16(h32), ss[0][t] = sum h32^2, ss[1..n_parts)[t] = 0.
int launch_embed(const int32_t* ids, const float* table, float* h32, __nv_bfloat16* h16, float* ss,
                 int ss_stride, int n_parts, int n_tokens, int d_model, cudaStream_t stream);
// Final RMSNorm + masked mean-pool + L2 normalise (retrieval/model.py:108-114):
//   out[s] = normalize( (1/len_s) * sum_t  w .* h32[t] * rs[t] )
int launch_pool_normalize(const float* h32, const float* ss, int ss_stride, int n_parts, const float* ln_w,
                          const int32_t* cu_tokens, void* out, int out_dtype, int n_seqs, int d_model,
                          float eps, cudaStream_t stream, float* group_scratch = nullptr, int max_len = 0);

// Weight packing (rpx_encoder_create): dst[n, k] = bf16(src[n, k] * scale[k]) (scale may be null),
// rows written at dst_row0 + (n / blk) * blk_stride + (n % blk)  (FFN interleave when blk_stride != blk).
int launch_pack_weight(const float* src, const float* scale, __nv_bfloat16* dst, int n_rows, int n_cols,
                       int dst_row0, int blk, int blk_stride, cudaStream_t stream);

// ---- top-k paths (rpx_simtopk.cu: tcgen05, rpx_smallq.cu: HBM streaming, rpx_exact.cu: exact fp64)
struct IndexState;
struct ExactBound;
// One similarity + top-k request (all pointers are device pointers).
struct TopkCall {
  const __nv_bfloat16* Q;   // [nq, d]
  int nq;
  const __nv_bfloat16* E;   // [n, d]
  int64_t n;
  int d, k;
  const uint32_t* mask;     // optional access bitmask [nq][mask_stride]
  int64_t mask_stride;
  float* out_scores;        // [nq, k]
  double* out_scores64;     // optional [nq, k]
  int64_t* out_idx;         // [nq, k]
  int32_t* out_count;       // optional [nq]
  int64_t* out_packed;      // optional [nq, k, 2]: (fp64 score bits, index) — the all-gather payload
  int64_t idx_offset;
  IndexState* state;        // device state of the index handle
  uint32_t* flagged;        // [nq] guard scratch
  ExactBound* bounds;       // [nq] guard scratch
  cudaStream_t st;
};
// re-score set size for k results (k + margin; the guard covers what the margin does not)
inline int topk_n_res(int k) { return k + (k / 8 > 12 ? k / 8 : 12); }
constexpr int kFastPathMaxK = 200;   // larger k goes through the exact path

int launch_row_norm_max(const __nv_bfloat16* E, int64_t n, int d, IndexState* state, cudaStream_t st);
size_t exact_cand_bytes(int64_t n);
int launch_exact_topk(const TopkCall& c, void* cand_ws, bool all_queries);
bool smallq_supported(int nq, int k, int d);
size_t smallq_workspace_bytes(int num_sms);
int launch_smallq_topk(const TopkCall& c, void* ws, int n_res);
size_t mma_topk_workspace_bytes(int nq, int k, int d, int num_sms);
int run_mma_topk(const TopkCall& c, void* ws, size_t ws_bytes);
// k-way merge of per-shard results; `packed`: one [n_parts, nq, k, 2] (score bits, index) buffer.
int launch_topk_merge(const double* d_scores64, const int64_t* d_idx_or_packed, bool packed, int n_parts, int nq, int k,
                      float* d_out_scores, double* d_out_scores64, int64_t* d_out_idx, int32_t* d_out_count,
                      cudaStream_t st);

}  // namespace rpx
