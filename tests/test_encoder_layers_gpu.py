"""Layer-by-layer, per-token parity of the encoder on both paths, through the fp32 residual dump
(`set_debug_hidden`): each layer is recomputed in float64 from the engine's own input to that layer, so an error
in one token's row (an attention row, an RMSNorm statistic, an epilogue column) is seen where it happens instead
of after a mean over the sequence.

The reference mirrors the engine's bf16 rounding points (everything between them is float64):
    W'   = bf16(W * ln)                      weights as the packing kernel folds them (fp32 product)
    A    = bf16(h),  rs = rsqrt(mean(h^2) + eps)
    qkv  = bf16(rs * A W'_qkv^T);  attn = bf16(softmax(q k^T + bias) v)
    h   += attn O^T
    ffn  = bf16(gelu_new(rs' * A' W'_0^T) * (rs' * A' W'_1^T)),  A' = bf16(h), rs' from the updated h
    h   += ffn wo^T
Tolerance.  A layer's input slab is the engine's, so the first GEMM sees identical operands; the engine differs
from the reference by fp32 accumulation (relative ~2^-24 sqrt(K), negligible), by the odd element that lands on
the other side of a bf16 rounding point (one bf16 unit: at most 2^-7 of its value), and by the attention
kernel's own rounding (at most 2^-8 (W|V| + |o|) per element, see test_attention_gpu).  So each element x_k of
attn / ffn differs by at most about 2^-7 |x_k|, with independent signs, and an output of the residual GEMMs
moves by about 2^-7 sqrt(sum_k x_k^2 W_nk^2): 2^-7 times the size of a typical element of that token's update,
which is at most ||dh_ref||_inf.  The assertion allows twice that, 2^-6 ||dh_ref||_inf per token.
"""
import json

import numpy as np
import pytest
import torch

from reprover_b200 import _native, synth
from reprover_b200.engine import T5EncoderEngine
from tests.helpers import attention_fp64, hf_bias_table

pytestmark = pytest.mark.gpu

LAYER_TOL = 2.0 ** -6
U32 = 2.0 ** -24
_RATIOS = {}


@pytest.fixture(scope="module", autouse=True)
def _record_ratios(out_dir):
    yield
    (out_dir / "encoder_layers_err_ratio.json").write_text(json.dumps(
        {"max_ratio": max(_RATIOS.values(), default=0.0), "per_case": _RATIOS}, indent=1))


def _checkpoint(sharp):
    """ByT5-small geometry, 2 layers.  `sharp`: q weights x6 and relative bias std 3, so attention is peaked
    (scores of std ~6) instead of nearly uniform."""
    cfg = synth.tiny_config(num_layers=2)
    sd = synth.random_t5_state_dict(cfg, seed=17)
    if sharp:
        for i in range(cfg["num_layers"]):
            sd[f"encoder.block.{i}.layer.0.SelfAttention.q.weight"] = sd[f"encoder.block.{i}.layer.0.SelfAttention.q.weight"] * 6
        key = "encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"
        sd[key] = sd[key] * 6
    return cfg, sd


@pytest.fixture(scope="module", params=[False, True], ids=["standard", "sharp"])
def model(request, rpx_lib, cuda_device):
    cfg, sd = _checkpoint(request.param)
    eng = T5EncoderEngine(cfg, sd, cuda_device)
    dev = cuda_device
    bf = lambda t: t.to(dev, torch.float32).to(torch.bfloat16).double()  # noqa: E731
    layers = []
    for i in range(cfg["num_layers"]):
        a, f = f"encoder.block.{i}.layer.0.", f"encoder.block.{i}.layer.1."
        ln0 = sd[a + "layer_norm.weight"].to(dev)
        ln1 = sd[f + "layer_norm.weight"].to(dev)
        qkv_w = torch.cat([sd[a + f"SelfAttention.{n}.weight"] for n in "qkv"], 0).to(dev)
        layers.append(dict(
            qkv=bf(qkv_w * ln0[None, :]), o=bf(sd[a + "SelfAttention.o.weight"]),
            wi0=bf(sd[f + "DenseReluDense.wi_0.weight"].to(dev) * ln1[None, :]),
            wi1=bf(sd[f + "DenseReluDense.wi_1.weight"].to(dev) * ln1[None, :]),
            wo=bf(sd[f + "DenseReluDense.wo.weight"])))
    R = cfg["relative_attention_max_distance"]
    lut = hf_bias_table(sd["encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"], R).to(dev)
    m = dict(cfg=cfg, sd=sd, eng=eng, layers=layers, lut=lut, tag="sharp" if request.param else "standard")
    yield m
    eng.close()


def _gelu_new(x):
    return 0.5 * x * (1.0 + torch.tanh((2.0 / torch.pi) ** 0.5 * (x + 0.044715 * x ** 3)))


def _bf16(x):
    return x.to(torch.bfloat16).double()


def _layer_fp64(m, l, h, lens):
    """Layer l in float64 from the fp32 residual h [T, D] entering it; returns the residual leaving it."""
    cfg, w = m["cfg"], m["layers"][l]
    eps, H = cfg["layer_norm_epsilon"], cfg["num_heads"]
    h = h.double()
    rs = torch.rsqrt(h.square().mean(1, keepdim=True) + eps)
    qkv = _bf16(rs * (_bf16(h) @ w["qkv"].t()))
    attn, _ = attention_fp64(qkv, lens, H, m["lut"], cfg["relative_attention_max_distance"])
    h = h + _bf16(attn) @ w["o"].t()
    rs = torch.rsqrt(h.square().mean(1, keepdim=True) + eps)
    a = _bf16(h)
    ffn = _bf16(_gelu_new(rs * (a @ w["wi0"].t())) * (rs * (a @ w["wi1"].t())))
    return h + ffn @ w["wo"].t()


def _strings(token_lens, seed):
    """Byte strings that tokenise to exactly `token_lens` tokens (bytes + EOS); a 1-token string is empty."""
    rng = np.random.default_rng(seed)
    return [bytes(rng.choice(synth._ALPHABET, size=n - 1).tolist()) for n in token_lens]


def check_call(m, token_lens, seed, case):
    """One engine call over strings of `token_lens` tokens, checked slab by slab and at the pool."""
    cfg, eng = m["cfg"], m["eng"]
    strs = _strings(token_lens, seed)
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in strs])]).astype(np.int64)
    data = np.frombuffer(b"".join(strs), dtype=np.uint8) if offsets[-1] else np.zeros(0, dtype=np.uint8)
    T = int(sum(token_lens))
    dump = eng.set_debug_hidden(T)
    try:
        emb = eng.encode_bytes(data, offsets, 4096, out_dtype=torch.float32)
        torch.cuda.synchronize()
        slabs = dump.clone()
    finally:
        eng.set_debug_hidden(None)
    tag = f"{m['tag']}_{case}"

    # slab 0: the embedding rows of ids = byte + 3, EOS = 1, bit for bit
    ids = np.concatenate([np.append(np.frombuffer(s, dtype=np.uint8).astype(np.int64) + 3, 1) for s in strs])
    shared = m["sd"]["shared.weight"].to(slabs.device)
    assert torch.equal(slabs[0], shared[torch.from_numpy(ids).to(slabs.device)]), f"{tag}: embedding slab"

    worst = 0.0
    for l in range(cfg["num_layers"]):
        want = _layer_fp64(m, l, slabs[l], token_lens) - slabs[l].double()
        got = slabs[l + 1].double() - slabs[l].double()
        scale = want.abs().amax(1, keepdim=True)
        ratio = ((got - want).abs() / (LAYER_TOL * scale)).amax(1)
        r = int(ratio.argmax())
        worst = max(worst, float(ratio[r]))
        assert float(ratio[r]) <= 1.0, (f"{tag}: layer {l}, token {r} (sequence {int(np.searchsorted(np.cumsum(token_lens), r, 'right'))}): "
                                        f"err / tol {float(ratio[r]):.3g}; {int((ratio > 1).sum())} tokens over")
    _RATIOS[f"{tag}_layers"] = worst

    # pool: final RMSNorm + mean + L2 of the last slab in float64.  The engine sums rows of h * rs in fp32 (its
    # rs from fp32 partial sums of squares), so the bound is u (len + 2 D) sum_t |w h rs| / len / ||mean||
    # for the sums, plus u D |e| for the normalisation
    h = slabs[-1].double()
    rs = torch.rsqrt(h.square().mean(1, keepdim=True) + cfg["layer_norm_epsilon"])
    lnw = m["sd"]["encoder.final_layer_norm.weight"].to(h.device).double()
    y = h * rs * lnw
    t0, pool_worst = 0, 0.0
    for s, L in enumerate(token_lens):
        mean = y[t0:t0 + L].mean(0)
        absmean = y[t0:t0 + L].abs().mean(0)
        norm = mean.norm().clamp_min(1e-12)
        e_ref = mean / norm
        bound = U32 * ((L + 2 * cfg["d_model"]) * absmean / norm + cfg["d_model"] * e_ref.abs())
        ratio = float(((emb[s].double() - e_ref).abs() / bound).max())
        pool_worst = max(pool_worst, ratio)
        assert ratio <= 1.0, f"{tag}: pooled embedding of sequence {s} (length {L}): err / bound {ratio:.3g}"
        t0 += L
    _RATIOS[f"{tag}_pool"] = pool_worst


# 1 (empty string), 63/64/65 around the 64-row tiles, the 256-key steps, 1024 and 2048 tokens: the TMA residual
# ring (O projection) and the register epilogue (FFN down); pool tails of every length mod 4
THROUGHPUT_LENS = [1, 63, 64, 65, 255, 256, 257, 258, 511, 1024, 2048]


def test_throughput_path_per_layer(model):
    check_call(model, THROUGHPUT_LENS, seed=1, case="throughput")


# 1; 100 (FFN-up 32-unit tiles); 129, 300 (64-row tiles); 384 / 385 (64- / 128-row tiles); 700, 1024; 1535 (the
# latency GEMMs with the throughput attention kernel).  Pool groups of 16: lengths = 0, 1, 15 mod 16, > 8 groups.
@pytest.mark.parametrize("n_tok", [1, 100, 129, 300, 384, 385, 700, 1024, 1535])
def test_latency_path_single_state_per_layer(model, n_tok):
    model["eng"].set_latency_tokens(4096)
    try:
        check_call(model, [n_tok], seed=n_tok, case=f"latency_{n_tok}")
    finally:
        model["eng"].set_latency_tokens(0)


def test_latency_path_mixed_call_per_layer(model):
    model["eng"].set_latency_tokens(4096)
    try:
        check_call(model, [143, 17, 400, 1, 256, 31], seed=3, case="latency_mixed")
    finally:
        model["eng"].set_latency_tokens(0)


def test_debug_dump_capacity(rpx_lib, cuda_device):
    """The dump holds `n_tokens` rows per slab: a shorter call fills the first T rows of every slab, a longer
    one is refused instead of writing past the buffer."""
    cfg = synth.tiny_config(num_layers=1)
    sd = synth.random_t5_state_dict(cfg, seed=2)
    eng = T5EncoderEngine(cfg, sd, cuda_device)
    dump = eng.set_debug_hidden(64)
    eng.encode_strings([b"x" * 19], 512, out_dtype=torch.float32)
    torch.cuda.synchronize()
    ids = torch.tensor([ord("x") + 3] * 19 + [1], device=cuda_device)
    assert torch.equal(dump[0, :20], sd["shared.weight"].to(cuda_device)[ids])
    assert dump[1, :20].abs().sum() > 0 and not dump[:, 20:].any()
    with pytest.raises(_native.RpxError) as ei:
        eng.encode_strings([b"y" * 64], 512)
    assert ei.value.code == _native.RPX_ERR_WORKSPACE
    eng.set_debug_hidden(None)
    eng.encode_strings([b"y" * 64], 512)
    eng.close()
