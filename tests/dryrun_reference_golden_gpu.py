"""Dry run of tests/test_zz_reference_golden_gpu.py on the CPU: the CUDA engine is replaced by the HF oracle
(bf16-rounded outputs, CPU tensors), the device top-k by the C oracle.  Validates the test logic only."""
import json, sys, types
from pathlib import Path
import numpy as np, torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import reference_path as ref, c_oracle
from reprover_b200 import synth, dist as rdist, retrieval_ops
from reprover_b200.retriever import B200PremiseRetriever
import reprover_b200.corpus as corpus_mod
import tests.test_zz_reference_golden_gpu as T

class OracleEngine:
    hidden_size = 1472
    max_tokens_per_call = 1 << 18
    def __init__(self, cfg, sd):
        torch.set_float32_matmul_precision("highest")
        self.enc, self.tok = ref.build_hf_encoder(cfg, sd), ref.build_hf_tokenizer()
    def encode_strings(self, blobs, max_seq_len, out_dtype=torch.bfloat16, out=None):
        emb = ref.reindex_corpus(self.enc, self.tok, [b.decode() for b in blobs], 8, max_seq_len).to(out_dtype)
        if out is None: return emb
        out.copy_(emb); return out
    def encode_ids(self, ids, mask, out_dtype=torch.bfloat16):
        return ref.encode(self.enc, ids, mask).to(out_dtype)

def fake_load_hf(ckpt, max_seq_len, device, dtype=None):
    from reprover_b200.engine import load_hf_checkpoint
    cfg, sd = load_hf_checkpoint(ckpt)
    r = object.__new__(B200PremiseRetriever)
    r.encoder = OracleEngine(cfg, sd); r.device = torch.device("cpu"); r.dtype = torch.bfloat16
    r.max_seq_len = max_seq_len; r.num_retrieved = 100; r.corpus = None; r.corpus_embeddings = None; r.embeddings_staled = True
    return r
B200PremiseRetriever.load_hf = staticmethod(fake_load_hf)

def oracle_nearest(corpus, E, ctxs, Q, k):
    words = np.stack([corpus.accessible_mask_words(c.path, c.theorem_pos) for c in ctxs])
    s, i, cnt = c_oracle.sim_topk(c_oracle.bf16_bits(Q.bfloat16()), c_oracle.bf16_bits(E.bfloat16()), k, words)
    if (cnt < k).any(): raise ValueError
    return [[corpus.all_premises[j] for j in row] for row in i.tolist()], s.astype(np.float32).tolist()
retrieval_ops.nearest_premises_device = oracle_nearest
def loc(queries, shard, k, off, mask):
    words = None if mask is None else mask.numpy().view(np.uint32)
    s, i, _ = c_oracle.sim_topk(c_oracle.bf16_bits(queries), c_oracle.bf16_bits(shard), k, words, off)
    return torch.stack([torch.from_numpy(s).view(torch.int64), torch.from_numpy(i)], dim=-1).contiguous()
def mer(gathered):
    s64, idx = gathered[..., 0].contiguous().view(torch.float64), gathered[..., 1].contiguous()
    s, i, c = c_oracle.topk_merge(s64.numpy(), idx.numpy())
    return torch.from_numpy(s.astype(np.float32)), torch.from_numpy(i), torch.from_numpy(c), torch.from_numpy(s)
rdist.sharded_topk.__defaults__ = (None, None, loc, mer)

class TP:  # tmp_path_factory stand-in
    def mktemp(self, n):
        import tempfile, pathlib
        return pathlib.Path(tempfile.mkdtemp())
gs = T.gold_setup.__wrapped__(TP(), torch.device("cpu")) if hasattr(T.gold_setup, "__wrapped__") else None
print("fixture ok")
for name in ["test_reindex_matches_the_reference_retriever", "test_encode_matches_the_reference_retriever",
             "test_retrieve_matches_the_reference_retriever", "test_batched_predictions_match_the_reference_retriever",
             "test_sharded_mode_on_one_rank_equals_the_unsharded_retriever"]:
    getattr(T, name)(gs); print(name, "ok")
