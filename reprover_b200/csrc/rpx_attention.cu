// rpx_attention.cu — T5 self-attention over packed variable-length sequences on tcgen05.
//
// Replaces HF T5Attention.forward (modeling_t5.py:253-344; SURVEY.md §2.1 K4-K7):
//   scores = q k^T            (NO 1/sqrt(d) scaling in T5)
//          + position_bias    (bucketed relative bias, shared by all layers; K5)
//          + padding mask     (packed layout: keys simply stop at the sequence end)
//   out    = softmax_fp32(scores) v, heads merged to [T, heads*64]
// without ever materialising the [B, heads, L, L] score tensor.
//
// One CTA per (128-query tile, head, sequence), 160 threads, four CTAs per SM:
//   warps 0-3  softmax: thread r owns query row r == TMEM lane r.  Per 64-key step: read the 64
//              scores from TMEM, add the bias, online softmax in fp32 (single pass), write P as bf16
//              into a 128B-swizzled K-major shared-memory tile, and rescale the output accumulator,
//              which lives in TMEM, by exp(m_old - m_new) (tcgen05.ld / st) when the row max moved.
//   warp 4     one elected thread drives both TMA and MMA: loads Q once and K / V tile by tile
//              (tensor maps over the packed qkv activation matrix, box 64 columns x 128 / 64 rows),
//              issues S = Q K^T (tcgen05.mma M128 N64 K16 x4) and O += P V (x4; V is the MN-major
//              B operand straight from the [keys, 64] tile TMA delivered), tcgen05.commit signals.
// S(j+1) is issued right behind PV(j), so the next scores are ready when the softmax warps return.
#include "rpx_common.cuh"
#include "rpx_kernels.cuh"
#include "rpx_ptx.cuh"

namespace rpx {

namespace {

constexpr int kHD = 64;    // head dim (d_kv)
// All waits of this kernel are pure spins: a try_wait suspend hint on the driver thread's long waits
// (first Q/K tiles, a whole softmax step) was measured at 300 and 1000 ns: no difference.
constexpr uint32_t kDriverHintNs = 0;
constexpr int kQT = 128;   // query rows per CTA (UMMA M)
constexpr int kKT = 64;    // keys per step (UMMA N for S, K extent for PV)
constexpr int kAttnThreads = 160;  // 4 softmax warps + 1 warp whose elected thread drives TMA and MMA
constexpr int kQBytes = 128 * 128;  // [128 rows][64 bf16], 128B-swizzled
constexpr int kKVBytes = 64 * 128;  // [64 keys][64 bf16]
constexpr int kCtasPerSm = 4;

// smem map (bytes, 1024-aligned base): Q | K | V | P | bias | barriers  (~50 KB: 4 CTAs / SM).
// K and V are single-buffered: K(j+1) is fetched as soon as S(j) has retired, V(j+1) as soon as PV(j)
// has, both well before they are needed; the other three CTAs of the SM cover what latency remains.
constexpr int kOffQ = 0;
constexpr int kOffK = kQBytes;
constexpr int kOffV = kQBytes + kKVBytes;
constexpr int kOffP = kQBytes + 2 * kKVBytes;
constexpr int kOffBias = 2 * kQBytes + 2 * kKVBytes;
constexpr int kAttnSmemFixed = kOffBias;

// MN-major (N contiguous) bf16 operand stored as rows of 128 B with the 128-byte swizzle:
// canonical layout ((8,8,m),(8,k)) : ((1,8,LBO),(64,SBO)) in elements — one 64-element atom along N
// (m = 1, LBO unused), groups of 8 K-rows 1024 B apart (SBO).  Same bit layout as the K-major
// descriptor; the "major" lives in the instruction descriptor.
RPX_DEVICE uint64_t make_smem_desc_mnmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// 2^x on the SFU (one MUFU.EX2; -inf -> 0, denormal results flushed).
RPX_DEVICE float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// idesc with B operand MN-major (bit 16)
__host__ __device__ constexpr uint32_t make_idesc_bf16_bmn(uint32_t m, uint32_t n) {
  return make_idesc_bf16(m, n) | (1u << 16);
}

// Relative-position bias in shared memory.  The table bias[clamp(key - query + R, 0, 2R)] is stored
// padded with 31 copies of its edge values on either side, so the 32 consecutive keys of a chunk
// read 32 consecutive entries starting at clamp(d0, -31, 2R) + 31 whatever the row — no per-element
// clamp and no per-lane regime (lanes of a warp sit at consecutive d0, so any branch on it diverges).
// Four copies, copy c shifted left by c entries, make that run 16-byte aligned for every start
// (8 LDS.128 per chunk instead of 32 LDS.32); the copy stride is 8 mod 32 words, which spreads the
// quarter-warp's eight loads over all 32 banks.
__host__ __device__ constexpr int bias_padded_len(int R) { return 2 * R + 63; }
__host__ __device__ constexpr int bias_copy_stride(int R) { return ((bias_padded_len(R) + 31) / 32) * 32 + 8; }

RPX_DEVICE void add_bias32(float (&s)[32], const float* __restrict__ sBias, int d0, int R, int stride) {
  const int a = min(max(d0, -31), 2 * R) + 31;
  const int c = a & 3;
  const float4* bp = reinterpret_cast<const float4*>(sBias + c * stride + (a - c));
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 b = bp[j];
    s[4 * j] += b.x;
    s[4 * j + 1] += b.y;
    s[4 * j + 2] += b.z;
    s[4 * j + 3] += b.w;
  }
}

__global__ void __launch_bounds__(kAttnThreads, kCtasPerSm)
t5_attention_tc_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_kv,
                       __nv_bfloat16* __restrict__ out, const int32_t* __restrict__ cu_seqlens,
                       const float* __restrict__ bias_lut, int n_heads, int R, int ld_out) {
  const int seq = blockIdx.z, head = blockIdx.y, qt = blockIdx.x;
  // Under programmatic dependent launch this CTA may start while the QKV projection is still running.
  // cu_seqlens and bias_lut were complete before the first kernel of the chain started, so the whole
  // prologue (bias table, barriers, TMEM) runs ahead; only the driver thread's TMA loads of q / k / v wait
  // for the predecessor (pdl_wait below).  The softmax warps touch global memory only to store `out`, after
  // MMAs that consumed those loads.
  pdl_launch_dependents();
  const int t0 = cu_seqlens[seq];
  const int len = cu_seqlens[seq + 1] - t0;
  const int q0 = qt * kQT;
  if (q0 >= len) return;  // whole CTA

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024 - (raw & 1023)) & 1023);
  float* sBias = reinterpret_cast<float*>(smem + kOffBias);
  const int lut_w = 2 * R + 1;
  const int bstride = bias_copy_stride(R);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBias + 4 * bstride * 4);
  uint64_t* bar_q = bars + 0;
  uint64_t* bar_k_full = bars + 1;
  uint64_t* bar_k_free = bars + 2;
  uint64_t* bar_v_full = bars + 3;
  uint64_t* bar_v_free = bars + 4;
  uint64_t* bar_s_full = bars + 5;
  uint64_t* bar_p_ready = bars + 6;
  uint64_t* bar_o_full = bars + 7;
  uint64_t* bar_s_free = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = n_heads * kHD;
  const int n_kt = (len + kKT - 1) / kKT;

  if (threadIdx.x < 128)
    for (int i = threadIdx.x; i < 4 * bstride; i += 128) {
      const int c = i / bstride, k = i - c * bstride;  // copy c, entry k = padded[k + c]
      sBias[i] = bias_lut[head * lut_w + min(max(k + c - 31, 0), 2 * R)];
    }
  if (warp == 4) {
    if (elect_one()) {
      mbar_init(bar_q, 1);
      mbar_init(bar_k_full, 1);
      mbar_init(bar_k_free, 1);
      mbar_init(bar_v_full, 1);
      mbar_init(bar_v_free, 1);
      mbar_init(bar_s_full, 1);
      mbar_init(bar_p_ready, 128);
      mbar_init(bar_o_full, 1);
      mbar_init(bar_s_free, 128);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, 128);  // S: columns [0,64), O: [64,128)
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + 64;

  if (warp == 4) {
    // ------------------------------------------------------------------ TMA + MMA driver (one thread)
    if (elect_one()) {
      const int kcol = inner + head * kHD, vcol = 2 * inner + head * kHD;
      pdl_wait();
      mbar_arrive_expect_tx(bar_q, kQBytes);
      tma_load_2d(smem + kOffQ, &tm_q, bar_q, head * kHD, t0 + q0);
      mbar_arrive_expect_tx(bar_k_full, kKVBytes);
      tma_load_2d(smem + kOffK, &tm_kv, bar_k_full, kcol, t0);
      mbar_arrive_expect_tx(bar_v_full, kKVBytes);
      tma_load_2d(smem + kOffV, &tm_kv, bar_v_full, vcol, t0);

      const uint32_t idesc_s = make_idesc_bf16(kQT, kKT);      // S[128 x 64]  = Q[128 x 64] K[64 x 64]^T
      const uint32_t idesc_o = make_idesc_bf16_bmn(kQT, kHD);  // O[128 x 64] += P[128 x 64] V[64 x 64]
      const uint64_t q_desc = make_smem_desc_kmajor_sw128(smem_u32(smem + kOffQ));
      const uint64_t k_desc = make_smem_desc_kmajor_sw128(smem_u32(smem + kOffK));
      const uint64_t p_desc = make_smem_desc_kmajor_sw128(smem_u32(smem + kOffP));
      const uint32_t v_base = smem_u32(smem + kOffV);
      mbar_wait<kDriverHintNs>(bar_q, 0, 12);
      mbar_wait<kDriverHintNs>(bar_k_full, 0, 13);
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < kHD / 16; ++k) umma_bf16_ss(tmem_S, q_desc + 2 * k, k_desc + 2 * k, idesc_s, k != 0);
      umma_commit(bar_s_full);
      umma_commit(bar_k_free);
      for (int kt = 0; kt < n_kt; ++kt) {
        const bool more = kt + 1 < n_kt;
        if (more) {
          // K(kt+1) as soon as S(kt) has read K(kt)
          mbar_wait<0>(bar_k_free, kt & 1, 11);
          mbar_arrive_expect_tx(bar_k_full, kKVBytes);
          tma_load_2d(smem + kOffK, &tm_kv, bar_k_full, kcol, t0 + (kt + 1) * kKT);
          // S(kt+1) as soon as every softmax warp holds S(kt) in registers: it is computed while they
          // work on step kt, so the only tensor-core round trip left between two softmax steps is
          // PV(kt), which step kt+1 needs only at its very end (P buffer, O rescale)
          mbar_wait<kDriverHintNs>(bar_s_free, kt & 1, 21);
          mbar_wait<0>(bar_k_full, (kt + 1) & 1, 15);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < kHD / 16; ++k) umma_bf16_ss(tmem_S, q_desc + 2 * k, k_desc + 2 * k, idesc_s, k != 0);
          umma_commit(bar_s_full);
          umma_commit(bar_k_free);
        }
        // O += P(kt) V(kt): needs P(kt) written (and O rescaled) and V(kt) landed
        mbar_wait<kDriverHintNs>(bar_p_ready, kt & 1, 14);
        mbar_wait<0>(bar_v_full, kt & 1, 19);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < kKT / 16; ++k) {
          // B = V (MN-major): 16 keys = two 8-row groups = 2048 B per step; A = P: 32 B per step
          const uint64_t v_desc = make_smem_desc_mnmajor_sw128(v_base + k * 2048);
          umma_bf16_ss(tmem_O, p_desc + 2 * k, v_desc, idesc_o, (kt | k) != 0);
        }
        umma_commit(bar_o_full);
        umma_commit(bar_v_free);
        if (more) {
          // V(kt+1) once PV(kt) has read V(kt)
          mbar_wait<0>(bar_v_free, kt & 1, 18);
          mbar_arrive_expect_tx(bar_v_full, kKVBytes);
          tma_load_2d(smem + kOffV, &tm_kv, bar_v_full, vcol, t0 + (kt + 1) * kKT);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax / output warps
    const int row = warp * 32 + lane;        // TMEM lane == query row inside the tile
    const int qpos = q0 + row;               // position inside the sequence
    const uint32_t lane_addr = (uint32_t)(warp * 32) << 16;
    const bool warp_live = q0 + warp * 32 < len;  // warp-uniform: some row of this warp is inside the sequence
    const float kLog2e = 1.4426950408889634f;
    const float kLazyTau = 5.545177444f;  // 8 ln 2
    float m_run = -INFINITY, l_run = 0.f;
    uint8_t* prow = smem + kOffP + row * 128;

    for (int kt = 0; kt < n_kt; ++kt) {
      const int kb = kt * kKT;
      mbar_wait<0>(bar_s_full, kt & 1, 16);
      tc_fence_after();
      if (warp_live) {  // warp-uniform
        float s0[32], s1[32];
        const bool second = kb + 32 < len;  // CTA-uniform
        {
          uint32_t v[32];
          tmem_ld_32x32(tmem_S + lane_addr, v);
          tmem_ld_wait();
          if (kb + 32 <= len) {  // CTA-uniform: only a partial chunk needs the key mask
#pragma unroll
            for (int j = 0; j < 32; ++j) s0[j] = __uint_as_float(v[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) s0[j] = (kb + j < len) ? __uint_as_float(v[j]) : -INFINITY;
          }
        }
        if (second) {
          uint32_t v[32];
          tmem_ld_32x32(tmem_S + lane_addr + 32, v);
          tmem_ld_wait();
          if (kb + 64 <= len) {
#pragma unroll
            for (int j = 0; j < 32; ++j) s1[j] = __uint_as_float(v[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) s1[j] = (kb + 32 + j < len) ? __uint_as_float(v[j]) : -INFINITY;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) s1[j] = -INFINITY;
        }
        // S(kt) now lives in registers: the driver may overwrite the TMEM tile with S(kt+1), which is
        // then computed while this step's softmax runs
        tc_fence_before();
        mbar_arrive(bar_s_free);

        // ---- single pass over the 64 scores of this row
        add_bias32(s0, sBias, kb - qpos + R, R, bstride);
        if (second) add_bias32(s1, sBias, kb + 32 - qpos + R, R, bstride);
        // row max with four independent chains (a single 64-long FMNMX chain is pure latency)
        float mx0 = fmaxf(s0[0], s1[0]), mx1 = fmaxf(s0[1], s1[1]), mx2 = fmaxf(s0[2], s1[2]),
              mx3 = fmaxf(s0[3], s1[3]);
#pragma unroll
        for (int j = 4; j < 32; j += 4) {
          mx0 = fmaxf(mx0, fmaxf(s0[j], s1[j]));
          mx1 = fmaxf(mx1, fmaxf(s0[j + 1], s1[j + 1]));
          mx2 = fmaxf(mx2, fmaxf(s0[j + 2], s1[j + 2]));
          mx3 = fmaxf(mx3, fmaxf(s0[j + 3], s1[j + 3]));
        }
        // Lazy reference maximum: the running reference only moves when the row maximum has grown by
        // more than kLazyTau (P <= 2^8 otherwise, harmless in bf16 / fp32), so most steps leave
        // scale == 1 exactly and skip the O rescale below.  exp(s - m) / sum exp(s - m) does not
        // depend on which m is used.
        const float m_cand = fmaxf(m_run, fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)));
        const float m_new = (m_cand - m_run <= kLazyTau) ? m_run : m_cand;  // first step: inf > tau
        const float mb = m_new * kLog2e;
        const float scale = fast_exp2((m_run - m_new) * kLog2e);  // 0 on the first step (m_run = -inf)
        m_run = m_new;
        // ---- PV(kt-1) has retired (it was issued a whole bias + max pass ago): the P buffer is free
        // and O may be touched
        if (kt > 0) {
          mbar_wait<0>(bar_o_full, (kt - 1) & 1, 17);
          tc_fence_after();
        }
        float la0 = 0.f, la1 = 0.f;  // two independent sum chains
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float p0 = fast_exp2(fmaf(h ? s1[j] : s0[j], kLog2e, -mb));
            const float p1 = fast_exp2(fmaf(h ? s1[j + 1] : s0[j + 1], kLog2e, -mb));
            la0 += p0;
            la1 += p1;
            pk[j >> 1] = pack_bf16x2(p0, p1);
          }
          // keys [32h, 32h+32) = 16-byte slots 4h..4h+3 of this row's 128-byte line
#pragma unroll
          for (int s4 = 0; s4 < 4; ++s4) {
            const int slot = (h * 4 + s4) ^ (row & 7);
            *reinterpret_cast<uint4*>(prow + slot * 16) =
                make_uint4(pk[4 * s4], pk[4 * s4 + 1], pk[4 * s4 + 2], pk[4 * s4 + 3]);
          }
        }
        l_run = l_run * scale + (la0 + la1);
        // O (in TMEM) *= exp(m_old - m_new) before PV(kt) accumulates onto it
        if (kt > 0 && !__all_sync(0xffffffffu, scale == 1.f)) {
#pragma unroll
          for (int c = 0; c < kHD / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(tmem_O + lane_addr + c * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * scale);
            tmem_st_32x32(tmem_O + lane_addr + c * 32, v);
          }
          tmem_st_wait();
        }
      } else {
        // rows past the sequence: P stays zero for every step.  The o_full wait keeps this warp from
        // running a step ahead of the others (its p_ready arrival must land in the right phase).
        mbar_arrive(bar_s_free);
        if (kt == 0) {
#pragma unroll
          for (int s4 = 0; s4 < 8; ++s4) *reinterpret_cast<uint4*>(prow + s4 * 16) = make_uint4(0u, 0u, 0u, 0u);
        } else {
          mbar_wait<0>(bar_o_full, (kt - 1) & 1, 22);
        }
      }
      // make the generic-proxy smem writes visible to the tensor core (async proxy), then signal
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bar_p_ready);
    }

    mbar_wait<0>(bar_o_full, (n_kt - 1) & 1, 20);
    tc_fence_after();
    if (warp_live) {
      const float inv = 1.f / l_run;
      __nv_bfloat16* dst = out + (int64_t)(t0 + qpos) * ld_out + head * kHD;
#pragma unroll
      for (int c = 0; c < kHD / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_O + lane_addr + c * 32, v);
        tmem_ld_wait();
        if (qpos < len) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint4 w;
            w.x = pack_bf16x2(__uint_as_float(v[8 * i + 0]) * inv, __uint_as_float(v[8 * i + 1]) * inv);
            w.y = pack_bf16x2(__uint_as_float(v[8 * i + 2]) * inv, __uint_as_float(v[8 * i + 3]) * inv);
            w.z = pack_bf16x2(__uint_as_float(v[8 * i + 4]) * inv, __uint_as_float(v[8 * i + 5]) * inv);
            w.w = pack_bf16x2(__uint_as_float(v[8 * i + 6]) * inv, __uint_as_float(v[8 * i + 7]) * inv);
            reinterpret_cast<uint4*>(dst + c * 32)[i] = w;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    __syncwarp();
    tmem_dealloc(tmem_base, 128);
  }
}

// ---------------------------------------------------------------------------------------------
// Latency-path variant (one or a few proof states per call, <= 1024 keys).  One proof state is a handful of
// (128-query tile, head) pairs — 12 CTAs on a 148-SM machine for 225 tokens — and in each of them one warp
// walks the whole key range of its 32 rows in 64-key steps: that walk, not the tensor core, is the critical
// path.  Here a CTA takes 32 QUERIES and all four softmax warps work on them, 256 keys at a time:
//   * the 32 query rows are loaded FOUR times, into row groups 0-31 / 32-63 / 64-95 / 96-127 of the Q tile,
//     so S[128 x 256] = Q K^T (one group of N <= 256 MMAs per key block) holds the same 32 score rows in all
//     four TMEM lane groups — a warp can only read its own lane group;
//   * warp w handles the 32-key chunks w and w + 4 of a block: block maximum and row sums are combined
//     across the warps through shared memory, each warp writes its chunks of P;
//   * O += P V from one run of MMAs per block; only rows 0-31 of P / O mean anything, warp 0 rescales them
//     between blocks (exact running maximum, at most three rescales) and stores them.
// A state of <= 256 tokens is ONE block: no running maximum, no rescale.  Four times the CTAs of the streaming
// kernel (48 for a 225-token state), a quarter of the serial softmax work in each, a quarter of the steps.
constexpr int kShortKeys = 256;                                      // keys per block
constexpr int kShortMaxKeys = 1024;                                  // longest sequence this kernel takes
constexpr int kShortQ = 32;                                          // queries per CTA
constexpr int kShortKVBytes = kShortKeys * 128;                      // one K or V block [256 keys][64 bf16]
constexpr int kShortOffQ = 0;
constexpr int kShortOffK = kQBytes;                                  // two K blocks
constexpr int kShortOffV = kShortOffK + 2 * kShortKVBytes;           // two V blocks
constexpr int kShortOffP = kShortOffV + 2 * kShortKVBytes;           // 4 tiles of [128 rows][64 keys]
constexpr int kShortOffRed = kShortOffP + 4 * kQBytes;               // max[2][4][32], sum[4][32] floats
constexpr int kShortOffBias = kShortOffRed + 3 * 4 * 32 * 4;

RPX_DEVICE void softmax_warps_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

__global__ void __launch_bounds__(kAttnThreads, 1)
t5_attention_short_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_kv,
                          __nv_bfloat16* __restrict__ out, const int32_t* __restrict__ cu_seqlens,
                          const float* __restrict__ bias_lut, int n_heads, int R, int ld_out) {
  const int seq = blockIdx.z, head = blockIdx.y, qt = blockIdx.x;
  pdl_launch_dependents();   // (prologue ahead of the predecessor's end: see t5_attention_tc_kernel)
  const int t0 = cu_seqlens[seq];
  const int len = cu_seqlens[seq + 1] - t0;   // <= kShortMaxKeys (checked by the launcher through max_len)
  const int q0 = qt * kShortQ;
  if (q0 >= len) return;  // whole CTA

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024 - (raw & 1023)) & 1023);
  float* sMax = reinterpret_cast<float*>(smem + kShortOffRed);   // [2][4][32] (alternating by block)
  float* sSum = sMax + 2 * 4 * 32;                               // [4][32]
  float* sBias = reinterpret_cast<float*>(smem + kShortOffBias);
  const int lut_w = 2 * R + 1;
  const int bstride = bias_copy_stride(R);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kShortOffBias + 4 * bstride * 4);
  uint64_t* bar_q = bars + 0;
  uint64_t* bar_k = bars + 1;   // [2]
  uint64_t* bar_v = bars + 3;   // [2]
  uint64_t* bar_s = bars + 5;
  uint64_t* bar_p = bars + 6;
  uint64_t* bar_o = bars + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = n_heads * kHD;
  const int n_blocks = (len + kShortKeys - 1) / kShortKeys;

  if (threadIdx.x < 128)
    for (int i = threadIdx.x; i < 4 * bstride; i += 128) {
      const int c = i / bstride, k = i - c * bstride;
      sBias[i] = bias_lut[head * lut_w + min(max(k + c - 31, 0), 2 * R)];
    }
  if (warp == 4) {
    if (elect_one()) {
      mbar_init(bar_q, 1);
      mbar_init(&bar_k[0], 1);
      mbar_init(&bar_k[1], 1);
      mbar_init(&bar_v[0], 1);
      mbar_init(&bar_v[1], 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, 128);
      mbar_init(bar_o, 1);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);  // S: columns [0, 256), O: [256, 320)
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + kShortKeys;

  if (warp == 4) {
    if (elect_one()) {
      const int kcol = inner + head * kHD, vcol = 2 * inner + head * kHD;
      auto load_kv = [&](int b) {   // key block b into buffer b & 1
        const int keys = min(kShortKeys, len - b * kShortKeys);
        const int n_box = (keys + kKT - 1) / kKT;   // 64-key TMA boxes
        uint8_t* kdst = smem + kShortOffK + (b & 1) * kShortKVBytes;
        uint8_t* vdst = smem + kShortOffV + (b & 1) * kShortKVBytes;
        mbar_arrive_expect_tx(&bar_k[b & 1], (uint32_t)(n_box * kKVBytes));
        for (int i = 0; i < n_box; ++i) tma_load_2d(kdst + i * kKVBytes, &tm_kv, &bar_k[b & 1], kcol, t0 + b * kShortKeys + i * kKT);
        mbar_arrive_expect_tx(&bar_v[b & 1], (uint32_t)(n_box * kKVBytes));
        for (int i = 0; i < n_box; ++i) tma_load_2d(vdst + i * kKVBytes, &tm_kv, &bar_v[b & 1], vcol, t0 + b * kShortKeys + i * kKT);
      };
      const uint32_t idesc_o = make_idesc_bf16_bmn(kQT, kHD);            // O[128 x 64] += P[128 x 16] V[16 x 64]
      const uint64_t q_desc = make_smem_desc_kmajor_sw128(smem_u32(smem + kShortOffQ));
      auto issue_s = [&](int b) {   // S[128 x n] = Q[128 x 64] K_b[n x 64]^T
        const int keys = min(kShortKeys, len - b * kShortKeys);
        const uint32_t idesc_s = make_idesc_bf16(kQT, (uint32_t)((keys + 15) & ~15));
        const uint64_t k_desc = make_smem_desc_kmajor_sw128(smem_u32(smem + kShortOffK + (b & 1) * kShortKVBytes));
        mbar_wait<0>(&bar_k[b & 1], (b >> 1) & 1, 32);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < kHD / 16; ++k) umma_bf16_ss(tmem_S, q_desc + 2 * k, k_desc + 2 * k, idesc_s, k != 0);
        umma_commit(bar_s);
      };
      pdl_wait();
      mbar_arrive_expect_tx(bar_q, kQBytes);
      for (int g = 0; g < 4; ++g)   // the same 32 query rows into every row group of the tile
        tma_load_2d(smem + kShortOffQ + g * kShortQ * 128, &tm_q, bar_q, head * kHD, t0 + q0);
      load_kv(0);
      if (n_blocks > 1) load_kv(1);
      mbar_wait<0>(bar_q, 0, 31);
      issue_s(0);
      for (int b = 0; b < n_blocks; ++b) {
        const int keys = min(kShortKeys, len - b * kShortKeys);
        const int n_mma = (keys + 15) & ~15;
        const uint32_t v_base = smem_u32(smem + kShortOffV + (b & 1) * kShortKVBytes);
        mbar_wait<0>(bar_p, b & 1, 33);
        mbar_wait<0>(&bar_v[b & 1], (b >> 1) & 1, 34);
        tc_fence_after();
        for (int j = 0; j < n_mma / 16; ++j) {
          // A = P tile j/4 (K-major, 32 B per 16 keys); B = V (MN-major): 16 keys = two 8-row groups = 2048 B
          const uint64_t p_desc = make_smem_desc_kmajor_sw128(smem_u32(smem + kShortOffP + (j >> 2) * kQBytes)) + 2 * (j & 3);
          const uint64_t v_desc = make_smem_desc_mnmajor_sw128(v_base + j * 2048);
          umma_bf16_ss(tmem_O, p_desc, v_desc, idesc_o, (b | j) != 0);
        }
        umma_commit(bar_o);
        // the next block's scores right behind this block's P V (the softmax warps are done with S: they have
        // arrived on bar_p); MMAs retire in order, so `bar_s` of block b + 1 also says P V of block b is done
        if (b + 1 < n_blocks) issue_s(b + 1);
        if (b + 2 < n_blocks) {   // K / V buffer b & 1 is free once P V of block b has read it
          mbar_wait<0>(bar_o, b & 1, 37);
          load_kv(b + 2);
        }
      }
    }
  } else {
    // query row `lane` of the CTA; this warp's copy of its scores sits in TMEM lanes [32 warp, 32 warp + 32)
    const int qpos = q0 + lane;
    const uint32_t lane_addr = (uint32_t)(warp * 32) << 16;
    const float kLog2e = 1.4426950408889634f;
    float m_run = -INFINITY, l_run = 0.f;   // l_run: this warp's share of the row sum, relative to m_run
    for (int b = 0; b < n_blocks; ++b) {
      const int kb = b * kShortKeys;                               // first key of the block
      const int keys = min(kShortKeys, len - kb);
      const int n_chunks = (((keys + 15) & ~15) + 31) >> 5;        // 32-key chunks that hold keys the MMAs read
      mbar_wait<0>(bar_s, b & 1, 35);   // (also: P V of block b - 1 has retired — P and O may be touched)
      tc_fence_after();
      // pass 1: block maximum over this warp's chunks, then over the warps
      float mx = -INFINITY;
      for (int c = warp; c < n_chunks; c += 4) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_S + lane_addr + 32 * c, v);
        tmem_ld_wait();
        float sc[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) sc[j] = __uint_as_float(v[j]);
        add_bias32(sc, sBias, kb + 32 * c - qpos + R, R, bstride);
        const int lim = keys - 32 * c;   // keys of this chunk inside the sequence
#pragma unroll
        for (int j = 0; j < 32; ++j) mx = fmaxf(mx, j < lim ? sc[j] : -INFINITY);
      }
      float* smx = sMax + (b & 1) * 128;
      smx[warp * 32 + lane] = mx;
      softmax_warps_sync();
      mx = fmaxf(fmaxf(smx[lane], smx[32 + lane]), fmaxf(smx[64 + lane], smx[96 + lane]));  // (chunk 0 is never empty)
      const float m_new = fmaxf(m_run, mx);
      const float scale = fast_exp2((m_run - m_new) * kLog2e);   // 0 for the first block (m_run = -inf)
      m_run = m_new;
      // pass 2: exponentials, row sum, P
      const float mb = m_new * kLog2e;
      float l0 = 0.f, l1 = 0.f;
      for (int c = warp; c < n_chunks; c += 4) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_S + lane_addr + 32 * c, v);
        tmem_ld_wait();
        float sc[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) sc[j] = __uint_as_float(v[j]);
        add_bias32(sc, sBias, kb + 32 * c - qpos + R, R, bstride);
        const int lim = (qpos < len) ? keys - 32 * c : 0;   // rows past the sequence contribute nothing
        uint32_t pk[16];
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float p0 = j < lim ? fast_exp2(fmaf(sc[j], kLog2e, -mb)) : 0.f;
          const float p1 = j + 1 < lim ? fast_exp2(fmaf(sc[j + 1], kLog2e, -mb)) : 0.f;
          l0 += p0;
          l1 += p1;
          pk[j >> 1] = pack_bf16x2(p0, p1);
        }
        // P row `lane` (rows 32-127 of the tiles are never written: their O rows are never read)
        uint8_t* prow = smem + kShortOffP + (c >> 1) * kQBytes + lane * 128;
        const int h = c & 1;
#pragma unroll
        for (int s4 = 0; s4 < 4; ++s4) {
          const int slot = (h * 4 + s4) ^ (lane & 7);
          *reinterpret_cast<uint4*>(prow + slot * 16) = make_uint4(pk[4 * s4], pk[4 * s4 + 1], pk[4 * s4 + 2], pk[4 * s4 + 3]);
        }
      }
      l_run = l_run * scale + (l0 + l1);
      // O rows 0-31 (warp 0's lanes) *= exp(m_old - m_new) before P V of this block accumulates onto them
      if (warp == 0 && b > 0 && !__all_sync(0xffffffffu, scale == 1.f)) {
#pragma unroll
        for (int c = 0; c < kHD / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(tmem_O + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * scale);
          tmem_st_32x32(tmem_O + c * 32, v);
        }
        tmem_st_wait();
      }
      if (b + 1 == n_blocks) sSum[warp * 32 + lane] = l_run;
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(bar_p);
    }

    if (warp == 0) {
      mbar_wait<0>(bar_o, (n_blocks - 1) & 1, 36);   // (P V needed every warp's P, so every warp's sum is in sSum)
      tc_fence_after();
      const float inv = 1.f / ((sSum[lane] + sSum[32 + lane]) + (sSum[64 + lane] + sSum[96 + lane]));
      __nv_bfloat16* dst = out + (int64_t)(t0 + qpos) * ld_out + head * kHD;
#pragma unroll
      for (int c = 0; c < kHD / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_O + c * 32, v);
        tmem_ld_wait();
        if (qpos < len) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint4 w;
            w.x = pack_bf16x2(__uint_as_float(v[8 * i + 0]) * inv, __uint_as_float(v[8 * i + 1]) * inv);
            w.y = pack_bf16x2(__uint_as_float(v[8 * i + 2]) * inv, __uint_as_float(v[8 * i + 3]) * inv);
            w.z = pack_bf16x2(__uint_as_float(v[8 * i + 4]) * inv, __uint_as_float(v[8 * i + 5]) * inv);
            w.w = pack_bf16x2(__uint_as_float(v[8 * i + 6]) * inv, __uint_as_float(v[8 * i + 7]) * inv);
            reinterpret_cast<uint4*>(dst + c * 32)[i] = w;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

bool t5_attention_bias_fits(int max_distance) {
  return 1024 + kAttnSmemFixed + (size_t)4 * bias_copy_stride(max_distance) * 4 + 128 <= 100 * 1024;
}

int launch_t5_attention(const __nv_bfloat16* qkv, __nv_bfloat16* out, const int32_t* cu_seqlens,
                        const float* bias_lut, int n_tokens, int n_seqs, int max_len, int n_heads, int d_kv,
                        int max_distance, cudaStream_t stream, AttnKernel kernel) {
  RPX_REQUIRE(d_kv == kHD, RPX_ERR_UNSUPPORTED, "attention: d_kv=%d (only 64 is implemented)", d_kv);
  RPX_REQUIRE(n_seqs > 0 && max_len > 0 && n_tokens > 0, RPX_ERR_INVALID, "attention: empty batch");
  RPX_REQUIRE(n_seqs <= 65535 && n_heads <= 65535, RPX_ERR_UNSUPPORTED, "attention: grid limits exceeded");
  const int inner = n_heads * d_kv;
  DeviceInfo dev;
  RPX_TRY(get_device_info(&dev));
  CUtensorMap tm_q, tm_kv;
  RPX_TRY(make_tmap_bf16_2d(&tm_kv, qkv, (uint64_t)n_tokens, (uint64_t)3 * inner, (uint64_t)3 * inner, kKT));
  if (kernel != AttnKernel::Throughput) {
    const size_t smem_short = 1024 + kShortOffBias + (size_t)4 * bias_copy_stride(max_distance) * 4 + 128;
    const bool short_ok = max_len <= kShortMaxKeys && smem_short <= dev.smem_optin;
    RPX_REQUIRE(short_ok || kernel == AttnKernel::Auto, RPX_ERR_UNSUPPORTED,
                "attention: the latency kernel takes at most %d keys and a bias table within %zu B of shared memory "
                "(max_len=%d, %zu B)", kShortMaxKeys, dev.smem_optin, max_len, smem_short);
    if (short_ok) {
      RPX_TRY(make_tmap_bf16_2d(&tm_q, qkv, (uint64_t)n_tokens, (uint64_t)3 * inner, (uint64_t)3 * inner, kShortQ));
      static thread_local int configured_short = -1;
      if (configured_short != dev.device) {
        RPX_CUDA_OK(cudaFuncSetAttribute(t5_attention_short_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)dev.smem_optin));
        configured_short = dev.device;
      }
      const dim3 grid32((max_len + kShortQ - 1) / kShortQ, n_heads, n_seqs);
      RPX_CUDA_OK(launch_pdl(t5_attention_short_kernel, grid32, dim3(kAttnThreads), smem_short, stream, pdl_enabled(), tm_q,
                             tm_kv, out, cu_seqlens, bias_lut, n_heads, max_distance, inner));
      return RPX_OK;
    }
  }
  RPX_TRY(make_tmap_bf16_2d(&tm_q, qkv, (uint64_t)n_tokens, (uint64_t)3 * inner, (uint64_t)3 * inner, kQT));
  const size_t smem = 1024 + kAttnSmemFixed + (size_t)4 * bias_copy_stride(max_distance) * 4 + 128;
  RPX_REQUIRE(t5_attention_bias_fits(max_distance), RPX_ERR_UNSUPPORTED,
              "attention: bias table too large (%zu B of shared memory)", smem);
  static thread_local int configured = -1;
  if (configured != dev.device) {
    RPX_CUDA_OK(cudaFuncSetAttribute(t5_attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    configured = dev.device;
  }
  const dim3 grid((max_len + kQT - 1) / kQT, n_heads, n_seqs);
  RPX_CUDA_OK(launch_pdl(t5_attention_tc_kernel, grid, dim3(kAttnThreads), smem, stream, pdl_enabled(), tm_q, tm_kv, out,
                         cu_seqlens, bias_lut, n_heads, max_distance, inner));
  return RPX_OK;
}

}  // namespace rpx

extern "C" int rpx_t5_attention_bf16(const void* d_qkv, void* d_out, const int32_t* d_cu_seqlens,
                                     const int32_t* h_cu_seqlens, int32_t n_seqs, int32_t n_heads,
                                     const float* d_bias_lut, int32_t rel_max_distance, int32_t kernel, void* stream) {
  using namespace rpx;
  RPX_REQUIRE(d_qkv && d_out && d_cu_seqlens && h_cu_seqlens && d_bias_lut, RPX_ERR_INVALID,
              "rpx_t5_attention_bf16: null pointer");
  RPX_REQUIRE(n_seqs > 0 && n_heads > 0 && rel_max_distance > 0, RPX_ERR_INVALID,
              "rpx_t5_attention_bf16: n_seqs=%d n_heads=%d rel_max_distance=%d", n_seqs, n_heads, rel_max_distance);
  RPX_REQUIRE(kernel == 0 || kernel == 1, RPX_ERR_INVALID, "rpx_t5_attention_bf16: kernel=%d (0 or 1)", kernel);
  // the grid and the tensor maps are sized from the host copy: every sequence must lie inside [0, T)
  RPX_REQUIRE(h_cu_seqlens[0] == 0, RPX_ERR_INVALID, "rpx_t5_attention_bf16: cu_seqlens[0]=%d", h_cu_seqlens[0]);
  int max_len = 0;
  for (int s = 0; s < n_seqs; ++s) {
    const int len = h_cu_seqlens[s + 1] - h_cu_seqlens[s];
    RPX_REQUIRE(len > 0, RPX_ERR_INVALID, "rpx_t5_attention_bf16: sequence %d has length %d", s, len);
    if (len > max_len) max_len = len;
  }
  return launch_t5_attention(static_cast<const __nv_bfloat16*>(d_qkv), static_cast<__nv_bfloat16*>(d_out), d_cu_seqlens,
                             d_bias_lut, h_cu_seqlens[n_seqs], n_seqs, max_len, n_heads, 64, rel_max_distance,
                             static_cast<cudaStream_t>(stream), kernel == 0 ? AttnKernel::Throughput : AttnKernel::Latency);
}
