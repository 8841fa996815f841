"""Shared test helpers (oracle access lives here: tests may import `oracle/`)."""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import reference_path as ref  # noqa: E402
from reprover_b200 import synth  # noqa: E402

# Acceptance for engine embeddings vs the fp32-"highest" HF oracle (SURVEY.md §8c):
# no worse than the reference's own GPU dtype (HF bf16 vs fp32: 1.3e-3 / 0.99992).
EMB_MAX_ABS = 2e-3
EMB_MIN_COS = 0.9999


def oracle_embeddings(cfg, sd, data: np.ndarray, offsets: np.ndarray, max_seq_len: int, batch_size: int = 8):
    """fp32 embeddings of the byte strings from the HF-based oracle (CPU)."""
    torch.set_float32_matmul_precision("highest")
    enc = ref.build_hf_encoder(cfg, sd)
    tok = ref.build_hf_tokenizer()
    texts = [s.decode("utf-8") for s in synth.split_strings(data, offsets)]
    return ref.reindex_corpus(enc, tok, texts, batch_size, max_seq_len)


def compare_embeddings(got: torch.Tensor, want: torch.Tensor):
    got = got.float().cpu()
    want = want.float().cpu()
    max_abs = float((got - want).abs().max())
    cos = torch.nn.functional.cosine_similarity(got, want, dim=1)
    return max_abs, float(cos.min())


def hf_bias_table(rel_bias: torch.Tensor, max_distance: int) -> torch.Tensor:
    """[heads][2R+1] fp32 relative-bias table built with HF's own bucket function: entry d + R is
    rel_bias[bucket(d)] for d = key - query (the layout the attention kernels consume)."""
    from transformers.models.t5.modeling_t5 import T5Attention

    d = torch.arange(-max_distance, max_distance + 1)
    buckets = T5Attention._relative_position_bucket(d, bidirectional=True, num_buckets=rel_bias.shape[0],
                                                    max_distance=max_distance)
    return rel_bias.float()[buckets].t().contiguous()


def attention_fp64(qkv: torch.Tensor, lens, n_heads: int, lut: torch.Tensor, max_distance: int, d_kv: int = 64):
    """Plain T5 self-attention in float64, per packed sequence and head: softmax(q k^T + lut[clamp(key - query)]) v
    (no 1/sqrt(d) scaling).  qkv [T, 3 * heads * d_kv] (q | k | v).  Returns (out, W |V|), both [T, heads * d_kv]."""
    x = qkv.double()
    lut = lut.to(device=qkv.device, dtype=torch.float64)
    inner = n_heads * d_kv
    o = torch.empty(x.shape[0], inner, dtype=torch.float64, device=x.device)
    wv = torch.empty_like(o)
    t0 = 0
    for L in lens:
        L = int(L)
        seq = x[t0:t0 + L]
        q, k, v = (seq[:, i * inner:(i + 1) * inner].reshape(L, n_heads, d_kv).transpose(0, 1) for i in range(3))
        pos = torch.arange(L, device=x.device)
        idx = (pos[None, :] - pos[:, None]).clamp(-max_distance, max_distance) + max_distance
        w = torch.softmax(q @ k.transpose(1, 2) + lut[:, idx], dim=-1)
        o[t0:t0 + L] = (w @ v).transpose(0, 1).reshape(L, inner)
        wv[t0:t0 + L] = (w @ v.abs()).transpose(0, 1).reshape(L, inner)
        t0 += L
    return o, wv
