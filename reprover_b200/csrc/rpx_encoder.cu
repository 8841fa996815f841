// rpx_encoder.cu — the ByT5 / T5 encoder forward (+ pool + normalise) on packed tokens.
//
// Replaces `PremiseRetriever._encode` (reference retrieval/model.py:92-114) and the HF
// `T5Stack` it calls (modeling_t5.py:637-792): per layer
//     h += O( attn( RMSNorm(h) ) )                      modeling_t5.py:366-375
//     h += wo( gelu_new(wi_0 n) * (wi_1 n) ), n = RMSNorm(h)   :146-150, :115-131
// then final RMSNorm, masked mean over tokens, L2 normalise.
//
// Data layout in HBM (T = packed tokens of the call, D = d_model):
//     h32  [T, D] fp32   residual stream (master copy)
//     h16  [T, D] bf16   same values, GEMM A operand
//     qkv  [T, 3*H*64] bf16,  attn [T, H*64] bf16,  ffn [T, d_ff] bf16
//     ssA / ssB [n_parts][T] fp32  per-row partial sums of h32^2, one per n-tile of the GEMM that
//                             produced h32 (6 for d_model = 1472) -> RMSNorm row scale
// RMSNorm never runs as its own kernel: its weight vector is folded into the next
// GEMM's B operand when the weights are packed, and the row scale rsqrt(mean(h^2)+eps)
// is applied to the fp32 accumulator in that GEMM's epilogue (rpx_gemm.cuh RowScale).
#include <math.h>

#include <new>
#include <vector>

#include "rpx_gemm_launch.cuh"
#include "rpx_kernels.cuh"

namespace rpx {

namespace {

constexpr int kBlockN = 256;

#ifndef RPX_GEMM_2CTA
#define RPX_GEMM_2CTA 1
#endif
// The encoder's GEMMs: 2-CTA (cta_group::2) tiles by default, the 1-CTA kernel with -DRPX_GEMM_2CTA=0.
template <class Epi>
int encoder_gemm(const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K,
                 const typename Epi::Params& ep, cudaStream_t st) {
#if RPX_GEMM_2CTA
  return launch_gemm2<Epi>(A, lda, B, ldb, M, N, K, ep, st);
#else
  return launch_gemm<kBlockN, Epi>(A, lda, B, ldb, M, N, K, ep, st);
#endif
}

// Residual-update GEMMs (attention output projection, FFN down projection).  With the 2-CTA kernel
// the residual stream moves through TMA (EpiResidualTma: RPX_RES_RING boxes per warp, which leaves
// room for RPX_RES_STAGES operand stages); -DRPX_RES_TMA=0 or a model too narrow for the ring's
// look-ahead uses the register epilogue.
#ifndef RPX_RES_TMA
#define RPX_RES_TMA (RPX_GEMM_2CTA && RPX_EPI_WARPS == 4)
#endif
// The TMA epilogue pays for its ring with operand stages (4 instead of 6), which costs a
// tensor-bound GEMM more than the epilogue gains: it is used while the MMA time of a tile
// (~0.43 us per 64 of K) is below the ~7 us the tile's 320 KB of residual traffic need, i.e. for
// the attention output projection (K = 384: 57.6 -> 38.5 ms per 4096-premise step) but not for the
// FFN down projection (K = 3584: 99.8 ms with the register epilogue, 114 ms with this one).
#ifndef RPX_RES_TMA_MAX_K
#define RPX_RES_TMA_MAX_K 1024
#endif
#ifndef RPX_RES_RING
#define RPX_RES_RING 4
#endif
#ifndef RPX_RES_STAGES
#define RPX_RES_STAGES 4
#endif
using EpiResTma = EpiResidualTma<RPX_RES_RING>;

struct ResidualMaps {
  bool use_tma = false;
  CUtensorMap h32, h16;
};

// Narrowest n-tile of the 2-CTA kernel for an N-column output (see n_tile_range).
inline int min_tile_cols(int N) {
  const int tiles_n = ceil_div(N, kBlockN);
  return 32 * (ceil_div(N, 32) / tiles_n);
}

int make_residual_maps(ResidualMaps* m, float* h32, __nv_bfloat16* h16, int T, int D) {
  m->use_tma = false;
#if RPX_RES_TMA
  if (D % 32 == 0 && min_tile_cols(D) >= 32 * (RPX_RES_RING - 1)) {
    RPX_TRY(make_tmap_2d(&m->h32, 4, h32, (uint64_t)T, (uint64_t)D, (uint64_t)D, 32, 32, 128));
    RPX_TRY(make_tmap_2d(&m->h16, 2, h16, (uint64_t)T, (uint64_t)D, (uint64_t)D, 32, 32, 64));
    m->use_tma = true;
  }
#endif
  return RPX_OK;
}

// h32 += A @ B^T, h16 = bf16(h32), ss = partial sums of h32^2 per n-tile.
int residual_gemm(const ResidualMaps& maps, const void* A, int64_t lda, const void* B, int64_t ldb, int T, int D,
                  int K, float* h32, __nv_bfloat16* h16, float* ss, cudaStream_t st) {
#if RPX_RES_TMA
  if (maps.use_tma && K <= RPX_RES_TMA_MAX_K) {
    EpiResTma::Params ep;
    ep.tm_h32 = maps.h32;
    ep.tm_h16 = maps.h16;
    ep.ss_out = ss;
    ep.ss_stride = T;
    return launch_gemm2<EpiResTma, RPX_RES_STAGES>(A, lda, B, ldb, T, D, K, ep, st);
  }
#endif
  EpiResidual::Params ep{h32, h16, D, ss, T};
  return encoder_gemm<EpiResidual>(A, lda, B, ldb, T, D, K, ep, st);
}

struct LayerW {
  const __nv_bfloat16* qkv;  // [3*inner, D]   (ln0 folded)
  const __nv_bfloat16* o;    // [D, inner]
  const __nv_bfloat16* wi;   // [2*d_ff, D]    (ln1 folded; wi_0 / wi_1 interleaved in 128-row blocks)
  const __nv_bfloat16* wo;   // [D, d_ff]
};

struct ProfRec {
  int cls;
  cudaEvent_t a, b;
};

}  // namespace

}  // namespace rpx

// T5 relative-position bucket, bidirectional (HF modeling_t5.py:189-234), float32 math
// like the reference implementation.  Host function, exported for the CPU parity test.
extern "C" int32_t rpx_t5_relative_bucket(int32_t relative_position, int32_t num_buckets, int32_t max_distance) {
  int nb = num_buckets / 2;
  int ret = relative_position > 0 ? nb : 0;
  int n = relative_position < 0 ? -relative_position : relative_position;
  const int max_exact = nb / 2;
  if (n < max_exact) return ret + n;
  float v = logf((float)n / (float)max_exact) / (float)log((double)max_distance / (double)max_exact) *
            (float)(nb - max_exact);
  int large = max_exact + (int)v;
  if (large > nb - 1) large = nb - 1;
  return ret + large;
}

struct rpx_encoder {
  rpx_t5_config cfg;
  int inner = 0;
  int n_parts = 0;      // RMSNorm partial sums per row on the throughput path: one per 256-wide n-tile
  int n_parts_lat = 0;  // ... on the latency path: one per 32-column chunk
  int latency_tokens = 0;  // calls with at most this many packed tokens take the latency path (0: never)
  size_t layer_bytes = 0;  // packed weights of one layer (qkv | o | wi | wo, contiguous from LayerW::qkv)
  const float* emb = nullptr;
  const float* final_ln = nullptr;
  const float* bias_lut = nullptr;
  std::vector<rpx::LayerW> layers;
  float* debug_hidden = nullptr;
  int64_t debug_tokens = 0;  // capacity of debug_hidden in tokens (the slab stride)
  bool profiling = false;
  std::vector<rpx::ProfRec> prof_pending;
  std::vector<cudaEvent_t> event_pool;
  float prof_ms[RPX_N_KERNEL_CLASSES] = {0};
  int64_t prof_launches[RPX_N_KERNEL_CLASSES] = {0};
  std::vector<int32_t> h_cu_tokens;
  std::vector<int32_t> h_lens;
};

namespace rpx {

namespace {

struct PackedLayout {
  size_t emb, final_ln, bias_lut, bucket_tmp, layer0, layer_stride, qkv, o, wi, wo, total;
};

PackedLayout packed_layout(const rpx_t5_config& c) {
  PackedLayout L{};
  const size_t D = c.d_model, inner = (size_t)c.num_heads * c.d_kv, F = c.d_ff;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  L.emb = take((size_t)c.vocab_size * D * 4);
  L.final_ln = take(D * 4);
  L.bias_lut = take((size_t)c.num_heads * (2 * c.rel_max_distance + 1) * 4);
  L.bucket_tmp = take((size_t)(2 * c.rel_max_distance + 1) * 4);
  L.layer0 = off;
  L.qkv = 0;
  size_t lo = 0;
  auto ltake = [&](size_t bytes) {
    size_t o = lo;
    lo = align_up(lo + bytes, 256);
    return o;
  };
  L.qkv = ltake(3 * inner * D * 2);
  L.o = ltake(D * inner * 2);
  L.wi = ltake(2 * F * D * 2);
  L.wo = ltake(D * F * 2);
  L.layer_stride = lo;
  L.total = L.layer0 + lo * (size_t)c.num_layers;
  return L;
}

int validate_cfg(const rpx_t5_config* c) {
  RPX_REQUIRE(c != nullptr, RPX_ERR_INVALID, "config is null");
  RPX_REQUIRE(c->d_kv == 64, RPX_ERR_UNSUPPORTED, "d_kv=%d: only 64 is implemented", c->d_kv);
  RPX_REQUIRE(c->d_model % 64 == 0 && c->d_model > 0, RPX_ERR_UNSUPPORTED, "d_model=%d must be a multiple of 64", c->d_model);
  RPX_REQUIRE(c->d_ff % 128 == 0 && c->d_ff > 0, RPX_ERR_UNSUPPORTED, "d_ff=%d must be a multiple of 128", c->d_ff);
  RPX_REQUIRE(c->num_heads > 0 && c->num_layers > 0 && c->vocab_size > 0, RPX_ERR_INVALID, "bad config");
  RPX_REQUIRE(c->rel_buckets >= 4 && c->rel_buckets % 4 == 0 && c->rel_max_distance >= c->rel_buckets / 4 &&
                  c->rel_max_distance <= 2048,
              RPX_ERR_UNSUPPORTED, "unsupported relative attention config (%d buckets, max distance %d)",
              c->rel_buckets, c->rel_max_distance);
  RPX_REQUIRE(t5_attention_bias_fits(c->rel_max_distance), RPX_ERR_UNSUPPORTED,
              "rel_max_distance=%d: the attention kernel's shared memory does not hold that bias table",
              c->rel_max_distance);
  return RPX_OK;
}

__global__ void bias_lut_kernel(const float* __restrict__ rel_bias, const int32_t* __restrict__ buckets,
                                float* __restrict__ lut, int n_heads, int width) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_heads * width) return;
  const int h = i / width, j = i % width;
  lut[i] = rel_bias[buckets[j] * n_heads + h];
}

struct Workspace {
  int32_t* cu_tokens;
  int64_t* cu_bytes;
  int32_t* ids;
  int32_t* lens;
  int32_t* flag;
  float* h32;
  __nv_bfloat16* h16;
  __nv_bfloat16* qkv;
  __nv_bfloat16* attn;
  __nv_bfloat16* ffn;
  float* ssA;
  float* ssB;
  size_t total;
};

Workspace carve(const rpx_encoder* e, uint8_t* base, int64_t T, int64_t S) {
  Workspace w{};
  const size_t D = e->cfg.d_model, inner = e->inner, F = e->cfg.d_ff;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* p = base ? base + off : nullptr;
    off = align_up(off + bytes, 256);
    return p;
  };
  w.cu_tokens = (int32_t*)take((S + 1) * 4);
  w.cu_bytes = (int64_t*)take((S + 1) * 8);
  w.lens = (int32_t*)take((S + 1) * 4);
  w.flag = (int32_t*)take(256);
  w.ids = (int32_t*)take(T * 4);
  w.h32 = (float*)take(T * D * 4);
  w.h16 = (__nv_bfloat16*)take(T * D * 2);
  w.qkv = (__nv_bfloat16*)take(T * 3 * inner * 2);
  w.attn = (__nv_bfloat16*)take(T * inner * 2);
  w.ffn = (__nv_bfloat16*)take(T * F * 2);
  const size_t parts = e->n_parts > e->n_parts_lat ? e->n_parts : e->n_parts_lat;
  w.ssA = (float*)take(parts * T * 4);
  w.ssB = (float*)take(parts * T * 4);
  w.total = off;
  return w;
}

struct Prof {
  rpx_encoder* e;
  cudaStream_t st;
  int cls;
  cudaEvent_t a = nullptr, b = nullptr;
  Prof(rpx_encoder* e_, cudaStream_t st_, int cls_) : e(e_), st(st_), cls(cls_) {
    if (!e->profiling) return;
    a = get();
    b = get();
    cudaEventRecord(a, st);
  }
  ~Prof() {
    if (!e->profiling) return;
    cudaEventRecord(b, st);
    e->prof_pending.push_back({cls, a, b});
  }
  cudaEvent_t get() {
    if (!e->event_pool.empty()) {
      cudaEvent_t ev = e->event_pool.back();
      e->event_pool.pop_back();
      return ev;
    }
    cudaEvent_t ev;
    cudaEventCreate(&ev);
    return ev;
  }
};

// ---------------------------------------------------------------------------------------------
// Latency path: one proof state per call (`retrieve`, retrieval/model.py:348-357, encodes ONE context).
// With T of a few hundred tokens the 256 x 256 pair tiles of the throughput path leave most of the GPU
// idle (QKV: 5 tiles, O / FFN-down: 6 tiles on 74 pairs) and every GEMM is bound by the latency of
// streaming its operands through a handful of SMs.  Here the same contraction core runs narrow 1-CTA tiles:
//   up to 384 tokens   QKV, O-proj, FFN-down on 64-ROW tiles (tcgen05.mma M = 64) x 64 columns with a 12-deep
//                      ring of 16 KB stages: 72 / 92 CTAs for a 200-token state, 138 at 384 tokens (one wave);
//                      a narrow GEMM's time is its k-blocks times the round trip of the operand ring divided by
//                      the ring depth, and half-empty 128-row tiles would cost their full intake
//   beyond             128 x 64 tiles, 8-deep ring (the 64-row tiles would need a second wave: 512 tokens 0.99
//                      vs 0.59 ms)
//   FFN-up             128 x 128 tiles = 64 gated hidden units (128 x 64 = 32 units up to 128 tokens), B tile in
//                      two boxes (gate rows, linear rows)
// K is never split, so every output element is accumulated over k in the same order whatever the tile, and
// the residual epilogues write their RMSNorm partial sums per 32-column chunk (n_parts_lat of them) whatever
// the tile: a state's embedding does not depend on what it was batched with.
constexpr int kLatBlockN = 64;
constexpr int kLatStages = 8;
constexpr int kLatSmallM = 64;
constexpr int kLatSmallStages = 12;
constexpr int kLatSmallMMaxTokens = 384;  // 6 row tiles x 23 column tiles = 138 CTAs: the most one wave holds
// Calls of at most this many tokens run their kernel chain under programmatic dependent launch: at 4 k tokens
// the re-indexing tiles gain 7 % (2.03 -> 1.89 ms), at 16 k 3-8 %, from 32 k on it is neutral to -1 % (A/B,
// BASELINE config-5 rows, two runs each).
constexpr int kPdlMaxTokens = 16384;

int forward_latency_layer(rpx_encoder* e, const Workspace& ws, const LayerW& w, const void* next_weights,
                          size_t next_bytes, int T, int S, int max_len, cudaStream_t st) {
  const rpx_t5_config& c = e->cfg;
  const int D = c.d_model, inner = e->inner, F = c.d_ff, P = e->n_parts_lat;
  const float inv_d = 1.0f / (float)D;
  {
    Prof p(e, st, 1);
    EpiStoreBF16::Params ep{ws.qkv, 3 * inner, RowScale{ws.ssA, P, T, inv_d, c.ln_eps}};
    // the QKV projection occupies 18 x ceil(T/64) (or 18 x ceil(T/128)) SMs: the rest of the GPU fetches the
    // next layer's weights into L2
    if (T <= kLatSmallMMaxTokens) {
      RPX_TRY((launch_gemm<kLatBlockN, EpiStoreBF16, false, kLatSmallStages, false, kLatSmallM>(ws.h16, D, w.qkv, D, T, 3 * inner,
                                                                                                 D, ep, st, 0, next_weights,
                                                                                                 next_bytes)));
    } else {
      RPX_TRY((launch_gemm<kLatBlockN, EpiStoreBF16, false, kLatStages>(ws.h16, D, w.qkv, D, T, 3 * inner, D, ep, st, 0,
                                                                         next_weights, next_bytes)));
    }
  }
  {
    Prof p(e, st, 2);
    RPX_TRY(launch_t5_attention(ws.qkv, ws.attn, ws.cu_tokens, e->bias_lut, T, S, max_len, c.num_heads, c.d_kv,
                                c.rel_max_distance, st, AttnKernel::Auto));
  }
  {
    Prof p(e, st, 3);
    EpiResidual::Params ep{ws.h32, ws.h16, D, ws.ssB, T};
    if (T <= kLatSmallMMaxTokens) {
      RPX_TRY((launch_gemm<kLatBlockN, EpiResidualT<true>, false, kLatSmallStages, false, kLatSmallM>(ws.attn, inner, w.o, inner, T,
                                                                                                       D, inner, ep, st)));
    } else {
      RPX_TRY((launch_gemm<kLatBlockN, EpiResidualT<true>, false, kLatStages>(ws.attn, inner, w.o, inner, T, D, inner, ep, st)));
    }
  }
  {
    Prof p(e, st, 4);
    // hidden units per tile: 32 (64-column tiles, T <= 128: 112 CTAs) or 64 (128-column tiles: 56 x ceil(T/128))
    if (T <= kBlockM) {
      EpiGeGLUT<32>::Params ep{ws.ffn, F, RowScale{ws.ssB, P, T, inv_d, c.ln_eps}};
      RPX_TRY((launch_gemm<64, EpiGeGLUT<32>, false, kLatStages, true>(ws.h16, D, w.wi, D, T, 2 * F, D, ep, st)));
    } else {
      EpiGeGLUT<64>::Params ep{ws.ffn, F, RowScale{ws.ssB, P, T, inv_d, c.ln_eps}};
      RPX_TRY((launch_gemm<128, EpiGeGLUT<64>, false, 6, true>(ws.h16, D, w.wi, D, T, 2 * F, D, ep, st)));
    }
  }
  {
    Prof p(e, st, 5);
    EpiResidual::Params ep{ws.h32, ws.h16, D, ws.ssA, T};
    if (T <= kLatSmallMMaxTokens) {
      RPX_TRY((launch_gemm<kLatBlockN, EpiResidualT<true>, false, kLatSmallStages, false, kLatSmallM>(ws.ffn, F, w.wo, F, T, D, F,
                                                                                                       ep, st)));
    } else {
      RPX_TRY((launch_gemm<kLatBlockN, EpiResidualT<true>, false, kLatStages>(ws.ffn, F, w.wo, F, T, D, F, ep, st)));
    }
  }
  return RPX_OK;
}

// The forward pass proper.  ws.ids / ws.cu_tokens are already populated on `st`.
int forward(rpx_encoder* e, const Workspace& ws, int T, int S, int max_len, void* d_out, int out_dtype,
            cudaStream_t st) {
  const rpx_t5_config& c = e->cfg;
  const int D = c.d_model, inner = e->inner, F = c.d_ff;
  // the latency path needs d_ff in 128-unit blocks for its split-B tiles (validate_cfg) and narrow-tile n
  const bool latency = T <= e->latency_tokens && D % 32 == 0 && (3 * inner) % 32 == 0;
  const int P = latency ? e->n_parts_lat : e->n_parts;
  const float inv_d = 1.0f / (float)D;
  RPX_REQUIRE(!e->debug_hidden || T <= e->debug_tokens, RPX_ERR_WORKSPACE,
              "debug hidden-state buffer holds %lld tokens, the call has %d", (long long)e->debug_tokens, T);
  struct PdlScope {
    explicit PdlScope(bool on) { set_pdl_scope(on); }
    ~PdlScope() { set_pdl_scope(false); }
  } pdl_scope(latency || T <= kPdlMaxTokens);
  {
    Prof p(e, st, 0);
    RPX_TRY(launch_embed(ws.ids, e->emb, ws.h32, ws.h16, ws.ssA, T, P, T, D, st));
  }
  auto dump = [&](int slab) -> int {
    if (e->debug_hidden)
      RPX_CUDA_OK(cudaMemcpyAsync(e->debug_hidden + (size_t)slab * e->debug_tokens * D, ws.h32, (size_t)T * D * 4,
                                  cudaMemcpyDeviceToDevice, st));
    return RPX_OK;
  };
  RPX_TRY(dump(0));
  ResidualMaps maps;
  if (!latency) RPX_TRY(make_residual_maps(&maps, ws.h32, ws.h16, T, D));
  for (int l = 0; l < c.num_layers; ++l) {
    const LayerW& w = e->layers[l];
    if (latency) {
      const bool has_next = l + 1 < c.num_layers;
      RPX_TRY(forward_latency_layer(e, ws, w, has_next ? e->layers[l + 1].qkv : nullptr, has_next ? e->layer_bytes : 0, T, S,
                                    max_len, st));
      RPX_TRY(dump(l + 1));
      continue;
    }
    {
      Prof p(e, st, 1);
      EpiStoreBF16::Params ep{ws.qkv, 3 * inner, RowScale{ws.ssA, P, T, inv_d, c.ln_eps}};
      RPX_TRY((encoder_gemm<EpiStoreBF16>(ws.h16, D, w.qkv, D, T, 3 * inner, D, ep, st)));
    }
    {
      Prof p(e, st, 2);
      RPX_TRY(launch_t5_attention(ws.qkv, ws.attn, ws.cu_tokens, e->bias_lut, T, S, max_len, c.num_heads, c.d_kv,
                                  c.rel_max_distance, st, AttnKernel::Throughput));
    }
    {
      Prof p(e, st, 3);
      RPX_TRY(residual_gemm(maps, ws.attn, inner, w.o, inner, T, D, inner, ws.h32, ws.h16, ws.ssB, st));
    }
    {
      Prof p(e, st, 4);
      EpiGeGLU::Params ep{ws.ffn, F, RowScale{ws.ssB, P, T, inv_d, c.ln_eps}};
      RPX_TRY((encoder_gemm<EpiGeGLU>(ws.h16, D, w.wi, D, T, 2 * F, D, ep, st)));
    }
    {
      Prof p(e, st, 5);
      RPX_TRY(residual_gemm(maps, ws.ffn, F, w.wo, F, T, D, F, ws.h32, ws.h16, ws.ssA, st));
    }
    RPX_TRY(dump(l + 1));
  }
  {
    Prof p(e, st, 6);
    // latency path: per-group partial rows go where the (now dead) FFN activations were — T rows of d_ff
    // bf16 hold T rows of d_model fp32 when d_ff >= 2 d_model (else the single-kernel pool runs)
    float* scratch = latency && (size_t)F * 2 >= (size_t)D * 4 ? reinterpret_cast<float*>(ws.ffn) : nullptr;
    RPX_TRY(launch_pool_normalize(ws.h32, ws.ssA, T, P, e->final_ln, ws.cu_tokens, d_out, out_dtype, S, D,
                                  c.ln_eps, st, scratch, max_len));
  }
  return RPX_OK;
}

}  // namespace
}  // namespace rpx

using namespace rpx;

extern "C" {

size_t rpx_encoder_packed_bytes(const rpx_t5_config* cfg) {
  if (validate_cfg(cfg) != RPX_OK) return 0;
  return packed_layout(*cfg).total;
}

int rpx_encoder_create(const rpx_t5_config* cfg, const rpx_t5_weights* w, void* d_packed, size_t packed_bytes,
                       void* stream, rpx_encoder** out) {
  RPX_TRY(validate_cfg(cfg));
  RPX_REQUIRE(w && d_packed && out, RPX_ERR_INVALID, "rpx_encoder_create: null argument");
  DeviceInfo dev;
  RPX_TRY(get_device_info(&dev));
  const PackedLayout L = packed_layout(*cfg);
  RPX_REQUIRE(packed_bytes >= L.total, RPX_ERR_WORKSPACE, "packed buffer too small: %zu < %zu", packed_bytes, L.total);
  RPX_REQUIRE((reinterpret_cast<uintptr_t>(d_packed) & 255) == 0, RPX_ERR_INVALID, "packed buffer must be 256-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* base = static_cast<uint8_t*>(d_packed);
  const int D = cfg->d_model, inner = cfg->num_heads * cfg->d_kv, F = cfg->d_ff;

  rpx_encoder* e = new (std::nothrow) rpx_encoder();
  RPX_REQUIRE(e != nullptr, RPX_ERR_INVALID, "out of host memory");
  e->cfg = *cfg;
  e->inner = inner;
  e->n_parts = ceil_div(D, kBlockN) * (EpiResidual::kWarps / 4);
  e->n_parts_lat = ceil_div(D, 32) * (EpiResidual::kWarps / 4);  // one per 32-column chunk
  auto fail = [&](int code) {
    delete e;
    return code;
  };
#define TRY_E(expr)                        \
  do {                                     \
    int _s = (expr);                       \
    if (_s != RPX_OK) return fail(_s);     \
  } while (0)
#define CUDA_E(expr)                                                                                   \
  do {                                                                                                 \
    cudaError_t _c = (expr);                                                                           \
    if (_c != cudaSuccess) {                                                                           \
      set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_c));           \
      return fail(RPX_ERR_CUDA);                                                                       \
    }                                                                                                  \
  } while (0)

  CUDA_E(cudaMemcpyAsync(base + L.emb, w->d_shared, (size_t)cfg->vocab_size * D * 4, cudaMemcpyDeviceToDevice, st));
  CUDA_E(cudaMemcpyAsync(base + L.final_ln, w->d_final_ln, (size_t)D * 4, cudaMemcpyDeviceToDevice, st));
  e->emb = reinterpret_cast<const float*>(base + L.emb);
  e->final_ln = reinterpret_cast<const float*>(base + L.final_ln);

  // relative-position bias LUT: lut[h][delta + R] = rel_bias[bucket(delta)][h]
  const int R = cfg->rel_max_distance, width = 2 * R + 1;
  std::vector<int32_t> buckets(width);
  for (int j = 0; j < width; ++j) buckets[j] = rpx_t5_relative_bucket(j - R, cfg->rel_buckets, R);
  CUDA_E(cudaMemcpyAsync(base + L.bucket_tmp, buckets.data(), (size_t)width * 4, cudaMemcpyHostToDevice, st));
  bias_lut_kernel<<<ceil_div(cfg->num_heads * width, 256), 256, 0, st>>>(
      w->d_rel_bias, reinterpret_cast<const int32_t*>(base + L.bucket_tmp), reinterpret_cast<float*>(base + L.bias_lut),
      cfg->num_heads, width);
  CUDA_E(cudaGetLastError());
  e->bias_lut = reinterpret_cast<const float*>(base + L.bias_lut);

  e->layers.resize(cfg->num_layers);
  for (int l = 0; l < cfg->num_layers; ++l) {
    uint8_t* lb = base + L.layer0 + L.layer_stride * l;
    __nv_bfloat16* qkv = reinterpret_cast<__nv_bfloat16*>(lb + L.qkv);
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(lb + L.o);
    __nv_bfloat16* wi = reinterpret_cast<__nv_bfloat16*>(lb + L.wi);
    __nv_bfloat16* wo = reinterpret_cast<__nv_bfloat16*>(lb + L.wo);
    // q | k | v stacked, RMSNorm(ln0) weight folded along K
    TRY_E(launch_pack_weight(w->h_q[l], w->h_ln0[l], qkv, inner, D, 0, inner, inner, st));
    TRY_E(launch_pack_weight(w->h_k[l], w->h_ln0[l], qkv, inner, D, inner, inner, inner, st));
    TRY_E(launch_pack_weight(w->h_v[l], w->h_ln0[l], qkv, inner, D, 2 * inner, inner, inner, st));
    TRY_E(launch_pack_weight(w->h_o[l], nullptr, o, D, inner, 0, D, D, st));
    // wi_0 rows -> [j*256, j*256+128), wi_1 rows -> [j*256+128, j*256+256); ln1 folded
    TRY_E(launch_pack_weight(w->h_wi0[l], w->h_ln1[l], wi, F, D, 0, 128, 256, st));
    TRY_E(launch_pack_weight(w->h_wi1[l], w->h_ln1[l], wi, F, D, 128, 128, 256, st));
    TRY_E(launch_pack_weight(w->h_wo[l], nullptr, wo, D, F, 0, D, D, st));
    e->layers[l] = LayerW{qkv, o, wi, wo};
    e->layer_bytes = L.layer_stride;
  }
  // `buckets` is pageable host memory: make sure the H2D staging has finished before it dies.
  CUDA_E(cudaStreamSynchronize(st));
#undef TRY_E
#undef CUDA_E
  *out = e;
  return RPX_OK;
}

int rpx_encoder_destroy(rpx_encoder* enc) {
  if (!enc) return RPX_OK;
  for (auto& r : enc->prof_pending) {
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  for (auto ev : enc->event_pool) cudaEventDestroy(ev);
  delete enc;
  return RPX_OK;
}

size_t rpx_encoder_workspace_bytes(const rpx_encoder* enc, int64_t max_tokens, int64_t max_seqs) {
  if (!enc || max_tokens <= 0 || max_seqs <= 0) return 0;
  return carve(enc, nullptr, max_tokens, max_seqs).total;
}

int rpx_encode_bytes(rpx_encoder* enc, const uint8_t* d_bytes, const int64_t* h_offsets, int32_t n_seqs,
                     int32_t max_seq_len, void* d_out, int32_t out_dtype, void* d_workspace,
                     size_t workspace_bytes, void* stream) {
  RPX_REQUIRE(enc && h_offsets && d_out && d_workspace, RPX_ERR_INVALID, "rpx_encode_bytes: null argument");
  RPX_REQUIRE(n_seqs > 0, RPX_ERR_INVALID, "rpx_encode_bytes: n_seqs=%d", n_seqs);
  RPX_REQUIRE(max_seq_len >= 1, RPX_ERR_INVALID, "rpx_encode_bytes: max_seq_len=%d", max_seq_len);
  RPX_REQUIRE(h_offsets[0] >= 0, RPX_ERR_INVALID, "rpx_encode_bytes: negative offset");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto& cu = enc->h_cu_tokens;
  cu.resize((size_t)n_seqs + 1);
  cu[0] = 0;
  int max_len = 0;
  int64_t total = 0;
  for (int s = 0; s < n_seqs; ++s) {
    const int64_t nb = h_offsets[s + 1] - h_offsets[s];
    RPX_REQUIRE(nb >= 0, RPX_ERR_INVALID, "rpx_encode_bytes: offsets not monotone at %d", s);
    const int64_t nt = nb + 1 < (int64_t)max_seq_len ? nb + 1 : (int64_t)max_seq_len;
    total += nt;
    RPX_REQUIRE(total < (int64_t)INT32_MAX, RPX_ERR_UNSUPPORTED, "rpx_encode_bytes: more than 2^31 tokens in one call");
    cu[s + 1] = (int32_t)total;
    if ((int)nt > max_len) max_len = (int)nt;
  }
  RPX_REQUIRE(d_bytes != nullptr || h_offsets[n_seqs] == h_offsets[0], RPX_ERR_INVALID, "rpx_encode_bytes: d_bytes is null");
  const int T = (int)total;
  const Workspace ws = carve(enc, static_cast<uint8_t*>(d_workspace), T, n_seqs);
  RPX_REQUIRE(ws.total <= workspace_bytes, RPX_ERR_WORKSPACE, "workspace too small: need %zu, have %zu (tokens=%d seqs=%d)",
              ws.total, workspace_bytes, T, n_seqs);
  RPX_REQUIRE((reinterpret_cast<uintptr_t>(d_workspace) & 255) == 0, RPX_ERR_INVALID, "workspace must be 256-byte aligned");
  RPX_CUDA_OK(cudaMemcpyAsync(ws.cu_tokens, cu.data(), ((size_t)n_seqs + 1) * 4, cudaMemcpyHostToDevice, st));
  RPX_CUDA_OK(cudaMemcpyAsync(ws.cu_bytes, h_offsets, ((size_t)n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
  RPX_TRY(launch_tokenize_bytes(d_bytes, ws.cu_bytes, ws.cu_tokens, ws.ids, n_seqs, T, st));
  return forward(enc, ws, T, n_seqs, max_len, d_out, out_dtype, st);
}

int rpx_encode_ids(rpx_encoder* enc, const int64_t* d_input_ids, const int64_t* d_attention_mask, int32_t batch,
                   int32_t seq_len, void* d_out, int32_t out_dtype, void* d_workspace, size_t workspace_bytes,
                   void* stream) {
  RPX_REQUIRE(enc && d_input_ids && d_attention_mask && d_out && d_workspace, RPX_ERR_INVALID,
              "rpx_encode_ids: null argument");
  RPX_REQUIRE(batch > 0 && seq_len > 0, RPX_ERR_INVALID, "rpx_encode_ids: batch=%d seq_len=%d", batch, seq_len);
  RPX_REQUIRE((int64_t)batch * seq_len < (int64_t)INT32_MAX, RPX_ERR_UNSUPPORTED, "rpx_encode_ids: batch too large");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Worst case all tokens valid: the workspace must fit that (callers size it with batch*seq_len).
  const Workspace ws_max = carve(enc, static_cast<uint8_t*>(d_workspace), (int64_t)batch * seq_len, batch);
  RPX_REQUIRE(ws_max.total <= workspace_bytes, RPX_ERR_WORKSPACE, "workspace too small: need %zu, have %zu", ws_max.total,
              workspace_bytes);
  RPX_REQUIRE((reinterpret_cast<uintptr_t>(d_workspace) & 255) == 0, RPX_ERR_INVALID, "workspace must be 256-byte aligned");
  RPX_CUDA_OK(cudaMemsetAsync(ws_max.flag, 0, 4, st));
  RPX_TRY(launch_mask_lengths(d_attention_mask, ws_max.lens, ws_max.flag, batch, seq_len, st));
  auto& lens = enc->h_lens;
  lens.resize((size_t)batch + 1);
  RPX_CUDA_OK(cudaMemcpyAsync(lens.data(), ws_max.lens, (size_t)batch * 4, cudaMemcpyDeviceToHost, st));
  RPX_CUDA_OK(cudaMemcpyAsync(&lens[batch], ws_max.flag, 4, cudaMemcpyDeviceToHost, st));
  RPX_CUDA_OK(cudaStreamSynchronize(st));
  RPX_REQUIRE(lens[batch] == 0, RPX_ERR_MASK,
              "attention_mask must be a right-padded prefix of ones with at least one token per row");
  auto& cu = enc->h_cu_tokens;
  cu.resize((size_t)batch + 1);
  cu[0] = 0;
  int max_len = 0;
  for (int b = 0; b < batch; ++b) {
    cu[b + 1] = cu[b] + lens[b];
    if (lens[b] > max_len) max_len = lens[b];
  }
  const int T = cu[batch];
  // Same carve order/sizes as ws_max for the leading (S-sized) members, so cu_tokens/flag do not move;
  // the T-sized members are re-carved for the actual token count.
  const Workspace ws = carve(enc, static_cast<uint8_t*>(d_workspace), T, batch);
  RPX_CUDA_OK(cudaMemcpyAsync(ws.cu_tokens, cu.data(), ((size_t)batch + 1) * 4, cudaMemcpyHostToDevice, st));
  RPX_TRY(launch_pack_ids(d_input_ids, ws.cu_tokens, ws.ids, batch, seq_len, T, enc->cfg.vocab_size, ws.flag, st));
  RPX_TRY(forward(enc, ws, T, batch, max_len, d_out, out_dtype, st));
  // ids outside [0, vocab) are reported after the fact (the forward ran with id 0 in their place).
  int32_t flag = 0;
  RPX_CUDA_OK(cudaMemcpyAsync(&flag, ws.flag, 4, cudaMemcpyDeviceToHost, st));
  RPX_CUDA_OK(cudaStreamSynchronize(st));
  RPX_REQUIRE((flag & 2) == 0, RPX_ERR_INVALID, "input_ids contains ids outside [0, %d)", enc->cfg.vocab_size);
  return RPX_OK;
}

int rpx_encoder_set_latency_tokens(rpx_encoder* enc, int32_t max_tokens) {
  RPX_REQUIRE(enc, RPX_ERR_INVALID, "null encoder");
  RPX_REQUIRE(max_tokens >= 0, RPX_ERR_INVALID, "rpx_encoder_set_latency_tokens: %d", max_tokens);
  enc->latency_tokens = max_tokens;
  return RPX_OK;
}

int rpx_encoder_set_debug_hidden(rpx_encoder* enc, float* d_hidden, int64_t max_tokens) {
  RPX_REQUIRE(enc, RPX_ERR_INVALID, "null encoder");
  RPX_REQUIRE(!d_hidden || max_tokens > 0, RPX_ERR_INVALID, "rpx_encoder_set_debug_hidden: max_tokens=%lld",
              (long long)max_tokens);
  enc->debug_hidden = d_hidden;
  enc->debug_tokens = d_hidden ? max_tokens : 0;
  return RPX_OK;
}

int rpx_encoder_set_profiling(rpx_encoder* enc, int32_t enable) {
  RPX_REQUIRE(enc, RPX_ERR_INVALID, "null encoder");
  enc->profiling = enable != 0;
  return RPX_OK;
}

int rpx_encoder_read_profile(rpx_encoder* enc, float* h_ms, int64_t* h_launches) {
  RPX_REQUIRE(enc && h_ms && h_launches, RPX_ERR_INVALID, "null argument");
  for (auto& r : enc->prof_pending) {
    RPX_CUDA_OK(cudaEventSynchronize(r.b));
    float ms = 0.f;
    RPX_CUDA_OK(cudaEventElapsedTime(&ms, r.a, r.b));
    enc->prof_ms[r.cls] += ms;
    enc->prof_launches[r.cls] += 1;
    enc->event_pool.push_back(r.a);
    enc->event_pool.push_back(r.b);
  }
  enc->prof_pending.clear();
  for (int i = 0; i < RPX_N_KERNEL_CLASSES; ++i) {
    h_ms[i] = enc->prof_ms[i];
    h_launches[i] = enc->prof_launches[i];
    enc->prof_ms[i] = 0.f;
    enc->prof_launches[i] = 0;
  }
  return RPX_OK;
}

}  // extern "C"
