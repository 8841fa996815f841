/* rpx.h — C ABI of the B200-native premise-retrieval engine (librpx.so).
 *
 * The reference (lean-dojo/ReProver) has NO plugin / operator / FFI interface for
 * this path: its seam is the Python attribute surface of `PremiseRetriever`
 * (retrieval/model.py:29) and `Corpus.get_nearest_premises` (common.py:299).  Each
 * entry point below therefore cites the reference Python call it replaces; the
 * Python shim `reprover_b200.retriever.B200PremiseRetriever` re-creates the
 * reference surface on top of these calls (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers / integers, no torch types, no C++ exceptions.
 *   - Every function returning `int` returns RPX_OK (0) or an RPX_ERR_* code; the
 *     message is available from rpx_last_error() (thread-local).
 *   - `d_` parameters are DEVICE pointers, `h_` parameters are HOST pointers.  The
 *     caller owns every buffer; the library borrows them for the duration of the
 *     stream-ordered work it enqueues and never frees them.  The only memory the
 *     library uses beyond its arguments is the explicit workspace / packed-weight
 *     buffers whose sizes it reports.
 *   - `stream` is a cudaStream_t passed as void*.  All work is enqueued on it;
 *     functions return without synchronising unless stated.
 *   - Handles are not thread-safe per handle; distinct handles are independent.
 *   - sm_100a (B200) only.  There is no CPU or other-GPU fallback: calling a
 *     compute entry point without such a device fails with RPX_ERR_CUDA /
 *     RPX_ERR_UNSUPPORTED.
 */
#ifndef RPX_H_
#define RPX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RPX_VERSION 200 /* 0.2.0 */

enum {
  RPX_OK = 0,
  RPX_ERR_INVALID = 1,     /* bad argument */
  RPX_ERR_CUDA = 2,        /* a CUDA runtime / driver call failed */
  RPX_ERR_UNSUPPORTED = 3, /* valid request outside what the engine implements */
  RPX_ERR_WORKSPACE = 4,   /* workspace / packed buffer too small */
  RPX_ERR_MASK = 5         /* attention_mask is not a right-padded prefix mask */
};

enum { RPX_DTYPE_BF16 = 0, RPX_DTYPE_F32 = 1 };

/* Last error message of the calling thread ("" if none). */
const char* rpx_last_error(void);
int rpx_version(void);
/* RPX_OK iff the current CUDA device is compute capability 10.x. */
int rpx_device_check(void);

/* ------------------------------------------------------------------------- encoder
 * Replaces the HF `T5EncoderModel` forward that `PremiseRetriever._encode`
 * (retrieval/model.py:92-114) calls at :101-105, plus the masked mean-pool and
 * F.normalize at :108-114.  Architecture constants come from the checkpoint's
 * config.json (HF T5Config; ByT5-small values in SURVEY.md §8).
 */
typedef struct {
  int32_t vocab_size;       /* 384  */
  int32_t d_model;          /* 1472 */
  int32_t d_kv;             /* 64   */
  int32_t d_ff;             /* 3584 */
  int32_t num_layers;       /* 12   */
  int32_t num_heads;        /* 6    */
  int32_t rel_buckets;      /* 32   */
  int32_t rel_max_distance; /* 128  */
  float ln_eps;             /* 1e-6 */
} rpx_t5_config;

/* Raw HF weights, fp32, row-major, DEVICE pointers.  The per-layer members are
 * HOST arrays of `num_layers` device pointers.  Safetensors key for each member
 * is given on the right (i = layer). */
typedef struct {
  const float* d_shared;         /* shared.weight                                   [vocab, d_model]   */
  const float* d_rel_bias;       /* encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight [buckets, heads] */
  const float* d_final_ln;       /* encoder.final_layer_norm.weight                 [d_model]          */
  const float* const* h_q;       /* encoder.block.i.layer.0.SelfAttention.q.weight  [heads*d_kv, d_model] */
  const float* const* h_k;       /* ...k.weight                                                         */
  const float* const* h_v;       /* ...v.weight                                                         */
  const float* const* h_o;       /* ...o.weight                                     [d_model, heads*d_kv] */
  const float* const* h_ln0;     /* encoder.block.i.layer.0.layer_norm.weight       [d_model]          */
  const float* const* h_wi0;     /* encoder.block.i.layer.1.DenseReluDense.wi_0.weight [d_ff, d_model]  */
  const float* const* h_wi1;     /* ...wi_1.weight                                                      */
  const float* const* h_wo;      /* ...wo.weight                                    [d_model, d_ff]    */
  const float* const* h_ln1;     /* encoder.block.i.layer.1.layer_norm.weight       [d_model]          */
} rpx_t5_weights;

typedef struct rpx_encoder rpx_encoder; /* opaque */

/* Bytes of device memory the packed (bf16, RMSNorm-folded, FFN-interleaved)
 * weight image needs; the caller allocates it and keeps it alive while the
 * handle lives. */
size_t rpx_encoder_packed_bytes(const rpx_t5_config* cfg);

/* Builds the packed weight image on `stream` and returns a handle.
 * Mirrors `PremiseRetriever.load_hf` (retrieval/model.py:52-66) for the encoder
 * part: fp32 checkpoint -> bf16 compute copy. */
int rpx_encoder_create(const rpx_t5_config* cfg, const rpx_t5_weights* w, void* d_packed,
                       size_t packed_bytes, void* stream, rpx_encoder** out);
int rpx_encoder_destroy(rpx_encoder* enc);

/* Workspace needed to encode up to `max_tokens` packed tokens in `max_seqs`
 * sequences in one call. */
size_t rpx_encoder_workspace_bytes(const rpx_encoder* enc, int64_t max_tokens, int64_t max_seqs);

/* Tokenise + encode + pool + normalise `n_seqs` byte strings.
 * Replaces, per batch, the tokenizer call at retrieval/model.py:199-205 (ByT5:
 * id = byte + 3, EOS = 1 appended, truncation to max_seq_len INCLUDING the EOS;
 * HF tokenization_byt5.py:195-208) followed by `_encode` (:92-114).
 *   d_bytes     concatenated UTF-8 bytes of all sequences (device)
 *   h_offsets   n_seqs + 1 byte offsets into d_bytes (HOST; the host needs the
 *               lengths to size the launch)
 *   d_out       [n_seqs, d_model] unit-norm rows, RPX_DTYPE_BF16 or RPX_DTYPE_F32
 * If h_offsets is page-locked memory it must stay valid until `stream` reaches this call.
 * Strings must not contain ByT5 special-token literals ("</s>", "<pad>", "<unk>",
 * "<extra_id_N>"); callers route those through rpx_encode_ids (the Python shim does). */
int rpx_encode_bytes(rpx_encoder* enc, const uint8_t* d_bytes, const int64_t* h_offsets,
                     int32_t n_seqs, int32_t max_seq_len, void* d_out, int32_t out_dtype,
                     void* d_workspace, size_t workspace_bytes, void* stream);

/* Exact `_encode(input_ids, attention_mask)` signature (retrieval/model.py:92-94):
 * int64 [B, L] ids and mask on the device.  The mask must be a right-padded
 * prefix mask with at least one token per row (what the reference tokenizer call
 * produces); anything else returns RPX_ERR_MASK.  Synchronises `stream` once
 * (row lengths are read back to size the launch). */
int rpx_encode_ids(rpx_encoder* enc, const int64_t* d_input_ids, const int64_t* d_attention_mask,
                   int32_t batch, int32_t seq_len, void* d_out, int32_t out_dtype,
                   void* d_workspace, size_t workspace_bytes, void* stream);

/* Latency path: encode calls with at most `max_tokens` packed tokens (0 = never, the default) run on
 * kernels shaped for ONE proof state — the reference's per-state call (`retrieve`,
 * retrieval/model.py:348-357) — instead of the 256 x 256 pair tiles that are sized for re-indexing: narrow
 * 1-CTA GEMM tiles (64 or 128 tokens x 64 columns, 128 x 128 for the gated FFN-up) that spread the state's work
 * over 70-140 SMs, attention on 32-query CTAs whose four softmax warps share the key range, pooling as
 * per-group partial rows, everything chained by programmatic dependent launch.  Results agree with the
 * throughput path to a few 1e-4 on unit-norm embeddings (the RMSNorm statistics are summed in another
 * grouping, which flips the odd bf16 rounding of an intermediate), not bit for bit, so a caller that needs
 * re-indexing's bits leaves it off; within the latency path a sequence's embedding does not depend on what
 * else is in the call. */
int rpx_encoder_set_latency_tokens(rpx_encoder* enc, int32_t max_tokens);

/* T5 bidirectional relative-position bucket of `relative_position` = key - query
 * (HF modeling_t5.py:189-234).  Pure host function (no GPU needed); exported so the
 * CPU test-suite can pin the table the attention kernel uses against the HF code. */
int32_t rpx_t5_relative_bucket(int32_t relative_position, int32_t num_buckets, int32_t max_distance);

/* Debug / parity hook: when non-NULL, every encode call also writes the fp32
 * residual stream after the embedding and after each block to
 * d_hidden[(slab * max_tokens + t) * d_model ...] (num_layers + 1 slabs of max_tokens rows;
 * the call's packed tokens fill the first T rows of each).  An encode call with more than
 * `max_tokens` packed tokens returns RPX_ERR_WORKSPACE while the hook is set. */
int rpx_encoder_set_debug_hidden(rpx_encoder* enc, float* d_hidden, int64_t max_tokens);

/* Per-kernel-class device timing (CUDA events on the launch stream).  Classes:
 * 0 embed, 1 qkv gemm, 2 attention, 3 o-proj gemm, 4 ffn-up gemm, 5 ffn-down gemm, 6 pool. */
#define RPX_N_KERNEL_CLASSES 7
int rpx_encoder_set_profiling(rpx_encoder* enc, int32_t enable);
/* Synchronises the recorded events; adds elapsed ms / launch counts since the
 * last read into ms[RPX_N_KERNEL_CLASSES], launches[RPX_N_KERNEL_CLASSES]. */
int rpx_encoder_read_profile(rpx_encoder* enc, float* h_ms, int64_t* h_launches);

/* --------------------------------------------------------------- similarity + top-k
 * Replaces the matmul + argsort half of `Corpus.get_nearest_premises`
 * (common.py:307-308) and the first-k walk at :316-322:
 *     S = Q E^T ; per query the k best rows of E, best first.
 * Ordering contract (deterministic refinement of the reference's unspecified
 * argsort tie order): score descending, then index ascending, where `score` is
 * the canonical fp64 dot product of the bf16 operands (oracle/rpx_oracle.c:
 * rpx_oracle_dot64).  out_scores are that value rounded to fp32.
 *
 * Exactness.  The fast paths rank by an fp32 score (tensor-core or FMA accumulation)
 * and re-score a superset of the answer in fp64.  A per-query guard compares the k-th
 * re-scored entry with the best fp32 score any row outside the re-scored set can have;
 * when the gap is inside the accumulation error bound (c(d) * ||q|| * max_i ||e_i||)
 * the query is recomputed by an exact fp64 pass over all admissible rows.  The result is
 * therefore the contract's answer on any input (near-duplicate rows included); only the
 * time depends on the data.
 *
 * rpx_index — a handle on a [n, d] bf16 matrix (what the reference keeps in
 * `self.corpus_embeddings`, retrieval/model.py:190, 363-366; d % 64 == 0).  Creating it
 * runs the one pass that depends only on the matrix (row-norm bound of the guard).  The
 * caller owns the matrix and the `rpx_index_state_bytes()` bytes of device state it hands in;
 * both must outlive the handle, and the handle must be re-created after the matrix changes.
 * One call at a time per handle (the device state holds the call's counters).
 */
typedef struct rpx_index rpx_index; /* opaque */
size_t rpx_index_state_bytes(void);
int rpx_index_create(const void* d_E, int64_t n, int32_t d, void* d_state, void* stream, rpx_index** out);
int rpx_index_destroy(rpx_index* ix);
/* Diagnostics (synchronises `stream`): the row-norm bound, the largest |fp32 - fp64| score difference
 * and the largest epsilon any guard has seen, and how many queries took the exact pass. */
int rpx_index_stats(rpx_index* ix, void* stream, float* h_norm_max, float* h_max_err, float* h_max_eps,
                    int64_t* h_n_exact);

/* Path selection flags of rpx_index_topk (0 = automatic: streaming kernel for nq <= 2, tcgen05
 * kernel otherwise, exact pass for k > 200).  The forcing flags exist for parity tests. */
enum { RPX_TOPK_AUTO = 0, RPX_TOPK_FORCE_MMA = 1, RPX_TOPK_FORCE_STREAM = 2, RPX_TOPK_FORCE_EXACT = 4 };

/*   d_Q [nq, d] bf16; 1 <= k <= 1024 (k <= 200 on the fast paths).
 *   d_access_mask  optional bitmask, row q = mask_stride_words uint32 words, bit
 *                  (i & 31) of word i >> 5 set <=> premise i is accessible to query q
 *                  (the `p in accessible_premises` test, common.py:313-318).
 *   d_out_count    optional [nq]: number of valid results (< k when fewer than k
 *                  candidates exist; the tail is idx = -1, score = -inf).
 *   d_out_scores64 optional [nq, k] fp64 scores.
 *   d_out_packed   optional [nq, k, 2] int64: (fp64 score bits, index) records — the
 *                  payload of the multi-GPU all-gather (rpx_topk_merge_packed).
 *   idx_offset     added to every output index (row offset of this shard).
 */
size_t rpx_index_topk_workspace_bytes(int64_t n, int32_t d, int32_t nq, int32_t k);
int rpx_index_topk(rpx_index* ix, const void* d_Q, int32_t nq, int32_t k, const uint32_t* d_access_mask,
                   int64_t mask_stride_words, float* d_out_scores, double* d_out_scores64, int64_t* d_out_idx,
                   int32_t* d_out_count, int64_t* d_out_packed, int64_t idx_offset, int32_t flags,
                   void* d_workspace, size_t workspace_bytes, void* stream);

/* One-shot form without a handle: same result, but the row-norm pass over E runs on every call
 * (one extra read of the matrix).  Use rpx_index_* when the same matrix is queried repeatedly. */
size_t rpx_sim_topk_workspace_bytes(int64_t n, int32_t d, int32_t nq, int32_t k);
int rpx_sim_topk(const void* d_Q, int32_t nq, const void* d_E, int64_t n, int32_t d, int32_t k,
                 const uint32_t* d_access_mask, int64_t mask_stride_words, float* d_out_scores,
                 double* d_out_scores64, int64_t* d_out_idx, int32_t* d_out_count,
                 int64_t idx_offset, void* d_workspace, size_t workspace_bytes, void* stream);

/* k-way merge of per-shard results after the all-gather (SURVEY.md §8e):
 * inputs [n_parts, nq, k] (fp64 scores, int64 global indices; each [part, query] row sorted under
 * the ordering contract with its empty slots, idx < 0, at the end — exactly what the top-k calls
 * emit), outputs the global top-k per query under the same ordering contract.
 * The _packed form takes the gathered `d_out_packed` records, [n_parts, nq, k, 2] int64. */
int rpx_topk_merge(const double* d_scores64, const int64_t* d_idx, int32_t n_parts, int32_t nq,
                   int32_t k, float* d_out_scores, double* d_out_scores64, int64_t* d_out_idx,
                   int32_t* d_out_count, void* stream);
int rpx_topk_merge_packed(const int64_t* d_packed, int32_t n_parts, int32_t nq, int32_t k,
                          float* d_out_scores, double* d_out_scores64, int64_t* d_out_idx,
                          int32_t* d_out_count, void* stream);

/* ------------------------------------------------------------------- test utilities
 * Debug timeline: while `d_stamps` (device, n_slots x 8 uint64) is set, every launch of the 1-CTA GEMM
 * kernel takes the next slot and its CTA 0 records %globaltimer at: kernel entry, prologue done,
 * producer past the dependency wait, first operand stage landed, last MMA committed, accumulator seen by
 * the epilogue, epilogue done, kernel exit.  NULL switches it off.  Not thread-safe; tooling only. */
int rpx_debug_set_timeline(unsigned long long* d_stamps, int32_t n_slots);

/*
 * Plain tcgen05 GEMM used by the parity tests of the contraction core:
 * C[M, N] (fp32, ldc = N) = A[M, K] * B[N, K]^T, bf16 inputs; K % 64 == 0, N % 32 == 0. */
int rpx_gemm_bf16_f32(const void* d_A, const void* d_B, float* d_C, int32_t M, int32_t N,
                      int32_t K, void* stream);
/* Same contract through the 2-CTA (cta_group::2, 256 x 256 tile) form of the core. */
int rpx_gemm2_bf16_f32(const void* d_A, const void* d_B, float* d_C, int32_t M, int32_t N,
                       int32_t K, void* stream);

/*
 * The encoder's T5 self-attention on caller-provided operands, for parity tests of the kernels:
 *   d_qkv        [T, 3 * n_heads * 64] bf16 packed tokens, q | k | v (head h at columns h*64 of each third)
 *   d_out        [T, n_heads * 64] bf16; rows [cu[s], cu[s+1]) of each sequence are written, no others
 *   d_cu_seqlens / h_cu_seqlens  the same n_seqs + 1 token offsets on the device and on the host;
 *                cu[0] = 0, every sequence non-empty, T = cu[n_seqs]
 *   d_bias_lut   [n_heads][2 * rel_max_distance + 1] fp32, entry clamp(key - query, +-R) + R
 *   kernel       0 = throughput kernel (any length), 1 = latency kernel (RPX_ERR_UNSUPPORTED when a
 *                sequence is longer than 1024 tokens or the bias table does not fit its shared memory)
 * out = softmax(q k^T + bias) v per sequence and head (no 1/sqrt(d) scaling, as in T5). */
int rpx_t5_attention_bf16(const void* d_qkv, void* d_out, const int32_t* d_cu_seqlens,
                          const int32_t* h_cu_seqlens, int32_t n_seqs, int32_t n_heads,
                          const float* d_bias_lut, int32_t rel_max_distance, int32_t kernel, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RPX_H_ */
