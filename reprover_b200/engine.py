"""Thin Python owner of the native handles: device buffers live in torch tensors
(plumbing), every computation is a call through the C ABI (`_native`).

`T5EncoderEngine` stands where the reference holds `self.encoder =
AutoModelForTextEncoding.from_pretrained(...)` (retrieval/model.py:45): it is built
from the same HF checkpoint contents (config dict + fp32 state dict).
"""
from __future__ import annotations

import ctypes as C
import json
import os
from typing import Dict, Iterable, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _native

_LAYER_KEYS = {
    "h_q": "encoder.block.{i}.layer.0.SelfAttention.q.weight",
    "h_k": "encoder.block.{i}.layer.0.SelfAttention.k.weight",
    "h_v": "encoder.block.{i}.layer.0.SelfAttention.v.weight",
    "h_o": "encoder.block.{i}.layer.0.SelfAttention.o.weight",
    "h_ln0": "encoder.block.{i}.layer.0.layer_norm.weight",
    "h_wi0": "encoder.block.{i}.layer.1.DenseReluDense.wi_0.weight",
    "h_wi1": "encoder.block.{i}.layer.1.DenseReluDense.wi_1.weight",
    "h_wo": "encoder.block.{i}.layer.1.DenseReluDense.wo.weight",
    "h_ln1": "encoder.block.{i}.layer.1.layer_norm.weight",
}
_REL_BIAS_KEY = "encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight"


def resolve_checkpoint_dir(name_or_path: str) -> str:
    """A local HF checkpoint directory for `name_or_path`.

    The reference hands the string to `AutoModelForTextEncoding.from_pretrained` (retrieval/model.py:45),
    which also accepts hub ids such as `kaiyuy/leandojo-lean4-retriever-byt5-small`.  A directory is used
    as it is; a hub id is resolved through the local HF cache (`huggingface_hub.snapshot_download`, which
    only touches the network when the snapshot is not cached).  Anything else fails here, with the reason,
    instead of deep inside the loader."""
    if os.path.isdir(name_or_path):
        return name_or_path
    if os.path.exists(name_or_path):
        raise FileNotFoundError(f"{name_or_path!r} is a file; an HF checkpoint DIRECTORY (config.json + "
                                f"model.safetensors / pytorch_model.bin) or a hub id is expected")
    try:
        from huggingface_hub import snapshot_download

        return snapshot_download(name_or_path, allow_patterns=["config.json", "*.safetensors", "pytorch_model.bin",
                                                               "*.json", "*.txt", "*.model"])
    except Exception as exc:  # no network / not cached / not a repo id
        raise FileNotFoundError(
            f"{name_or_path!r} is neither a local checkpoint directory nor a hub snapshot available to this "
            f"machine ({type(exc).__name__}: {exc}). Download the checkpoint and pass its directory.") from exc


def load_hf_checkpoint(path: str) -> Tuple[Dict, Dict[str, torch.Tensor]]:
    """(config dict, fp32 CPU state dict) from an HF checkpoint directory or hub id
    (`config.json` + `model.safetensors` or `pytorch_model.bin`)."""
    path = resolve_checkpoint_dir(path)
    cfg_path = os.path.join(path, "config.json")
    if not os.path.exists(cfg_path):
        raise FileNotFoundError(f"{path}: no config.json — not an HF checkpoint directory")
    with open(cfg_path) as fh:
        cfg = json.load(fh)
    st_path = os.path.join(path, "model.safetensors")
    bin_path = os.path.join(path, "pytorch_model.bin")
    if os.path.exists(st_path):
        from safetensors.torch import load_file

        sd = load_file(st_path)
    elif os.path.exists(bin_path):
        sd = torch.load(bin_path, map_location="cpu", weights_only=True)
    else:
        raise FileNotFoundError(f"{path}: neither model.safetensors nor pytorch_model.bin")
    return cfg, {k: v.float() for k, v in sd.items()}


def required_weight_keys(config: Dict) -> List[str]:
    """Every state-dict key the encoder engine reads (HF T5EncoderModel names)."""
    keys = [_REL_BIAS_KEY, "encoder.final_layer_norm.weight"]
    for i in range(int(config["num_layers"])):
        keys += [pattern.format(i=i) for pattern in _LAYER_KEYS.values()]
    return keys


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class T5EncoderEngine:
    """ByT5/T5 encoder + mean-pool + L2-normalise on one GPU (`rpx_encode_*`)."""

    def __init__(self, config: Dict, state_dict: Dict[str, torch.Tensor], device: Union[int, str, torch.device],
                 max_tokens_per_call: int = 1 << 18) -> None:
        self.lib = _native.load()
        self.device = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        if self.device.type != "cuda":
            raise RuntimeError(
                f"T5EncoderEngine needs a CUDA device (got {self.device}); this engine has no CPU path")
        self.config = dict(config)
        missing = [k for k in required_weight_keys(config) if k not in state_dict]
        if "shared.weight" not in state_dict and "encoder.embed_tokens.weight" not in state_dict:
            missing.insert(0, "shared.weight (or encoder.embed_tokens.weight)")
        if missing:
            raise KeyError(f"checkpoint is not a T5/ByT5 encoder state dict: {len(missing)} weights missing, "
                           f"first: {missing[:3]}")
        # kept (by reference, no copy) so that save_pretrained can write the checkpoint back out
        self._state_dict = state_dict
        if config.get("feed_forward_proj", "gated-gelu") != "gated-gelu":
            raise NotImplementedError("only the gated-gelu T5 v1.1 / ByT5 feed-forward is implemented")
        self.hidden_size = int(config["d_model"])
        self.max_tokens_per_call = int(max_tokens_per_call)
        self.latency_tokens = 0
        self._handle = C.c_void_p()
        self._ws: Optional[torch.Tensor] = None
        self._ws_shape = (0, 0)
        self._debug_buf: Optional[torch.Tensor] = None
        self._pin_bufs: List[Optional[torch.Tensor]] = [None, None]
        self._pin_events: List[Optional[torch.cuda.Event]] = [None, None]
        self._pin_slot = 0
        with torch.cuda.device(self.device):
            _native.check(self.lib.rpx_device_check())
            cfg = _native.T5Config(
                vocab_size=config["vocab_size"], d_model=config["d_model"], d_kv=config["d_kv"], d_ff=config["d_ff"],
                num_layers=config["num_layers"], num_heads=config["num_heads"],
                rel_buckets=config.get("relative_attention_num_buckets", 32),
                rel_max_distance=config.get("relative_attention_max_distance", 128),
                ln_eps=config.get("layer_norm_epsilon", 1e-6))
            self._cfg = cfg
            nbytes = self.lib.rpx_encoder_packed_bytes(C.byref(cfg))
            if nbytes == 0:
                raise _native.RpxError(_native.RPX_ERR_UNSUPPORTED, _native.last_error())
            self._packed = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            L = cfg.num_layers
            shared = state_dict.get("shared.weight", state_dict.get("encoder.embed_tokens.weight"))
            keep = []  # device copies of the raw fp32 weights, alive until packing has run

            def dev(t: torch.Tensor) -> int:
                d = t.to(device=self.device, dtype=torch.float32).contiguous()
                keep.append(d)
                return d.data_ptr()

            w = _native.T5Weights()
            w.d_shared = dev(shared)
            w.d_rel_bias = dev(state_dict[_REL_BIAS_KEY])
            w.d_final_ln = dev(state_dict["encoder.final_layer_norm.weight"])
            arrays = []
            for field, pattern in _LAYER_KEYS.items():
                arr = (C.c_void_p * L)(*[dev(state_dict[pattern.format(i=i)]) for i in range(L)])
                arrays.append(arr)
                setattr(w, field, C.cast(arr, _native._PP))
            _native.check(self.lib.rpx_encoder_create(C.byref(cfg), C.byref(w), self._packed.data_ptr(), nbytes,
                                                      _stream_ptr(self.device), C.byref(self._handle)))
            torch.cuda.current_stream(self.device).synchronize()
            del keep

    # ------------------------------------------------------------------ lifecycle
    def close(self) -> None:
        if getattr(self, "_handle", None) and self._handle.value:
            self.lib.rpx_encoder_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def save_pretrained(self, save_directory: str) -> None:
        """`encoder.save_pretrained(dir)` as the reference's callers use it (generation/model.py:224-226
        saves the retriever's encoder next to the generator): writes `config.json` and
        `model.safetensors` with the fp32 weights this engine was built from, loadable by
        `AutoModelForTextEncoding.from_pretrained(dir)` and by `load_hf`."""
        from safetensors.torch import save_file

        os.makedirs(save_directory, exist_ok=True)
        cfg = dict(self.config)
        cfg.setdefault("architectures", ["T5EncoderModel"])
        cfg.setdefault("model_type", "t5")
        with open(os.path.join(save_directory, "config.json"), "w") as fh:
            json.dump(cfg, fh, indent=1)
        sd = self._state_dict
        tensors = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in sd.items()
                   if k != "encoder.embed_tokens.weight" or "shared.weight" not in sd}
        save_file(tensors, os.path.join(save_directory, "model.safetensors"), metadata={"format": "pt"})

    @classmethod
    def from_hf_dir(cls, path: str, device, **kw) -> "T5EncoderEngine":
        cfg, sd = load_hf_checkpoint(path)
        return cls(cfg, sd, device, **kw)

    # ------------------------------------------------------------------ helpers
    def _workspace(self, n_tokens: int, n_seqs: int) -> torch.Tensor:
        need = self.lib.rpx_encoder_workspace_bytes(self._handle, n_tokens, n_seqs)
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(int(need * 1.1) + 4096, dtype=torch.uint8, device=self.device)
        return self._ws

    @staticmethod
    def _out_dtype(dtype: torch.dtype) -> int:
        if dtype == torch.bfloat16:
            return _native.RPX_DTYPE_BF16
        if dtype == torch.float32:
            return _native.RPX_DTYPE_F32
        raise ValueError(f"unsupported output dtype {dtype}")

    MAX_SEQS_PER_CALL = 65535

    def token_counts(self, offsets: np.ndarray, max_seq_len: int) -> np.ndarray:
        """ByT5 token count of each string: bytes + EOS, truncated to max_seq_len."""
        return np.minimum(np.diff(offsets) + 1, max_seq_len)

    # ------------------------------------------------------------------ encode
    def encode_packed_bytes(self, d_bytes: torch.Tensor, offsets: np.ndarray, max_seq_len: int,
                            out: torch.Tensor) -> None:
        """One `rpx_encode_bytes` call: `d_bytes` uint8 on the device, `offsets` host int64 [n+1]
        (relative to d_bytes), `out` [n, d_model] on the device (bf16 or fp32)."""
        n = len(offsets) - 1
        assert out.shape == (n, self.hidden_size) and out.is_contiguous() and out.device == self.device
        offs = np.ascontiguousarray(offsets, dtype=np.int64)
        n_tok = int(self.token_counts(offs, max_seq_len).sum())
        with torch.cuda.device(self.device):
            ws = self._workspace(n_tok, n)
            _native.check(self.lib.rpx_encode_bytes(
                self._handle, d_bytes.data_ptr(), offs.ctypes.data_as(C.POINTER(C.c_int64)), n, max_seq_len,
                out.data_ptr(), self._out_dtype(out.dtype), ws.data_ptr(), ws.numel(), _stream_ptr(self.device)))

    def encode_bytes(self, data: np.ndarray, offsets: np.ndarray, max_seq_len: int,
                     out_dtype: torch.dtype = torch.bfloat16, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Encode n byte strings given as (concatenated uint8 bytes, int64 offsets [n+1]) on the HOST.

        The strings are cut into chunks of at most `max_tokens_per_call` packed tokens; each chunk
        is one H2D copy (from pinned memory) plus one engine call.  Row order = input order.
        """
        n = len(offsets) - 1
        if out is None:
            out = torch.empty(n, self.hidden_size, dtype=out_dtype, device=self.device)
        counts = self.token_counts(offsets, max_seq_len)
        cum = np.concatenate([[0], np.cumsum(counts)])
        lo = 0
        data_t = self._pinned_copy(data)
        while lo < n:
            hi = int(np.searchsorted(cum, cum[lo] + self.max_tokens_per_call, side="right")) - 1
            hi = max(hi, lo + 1)
            hi = min(hi, n, lo + self.MAX_SEQS_PER_CALL)   # (the attention grid takes at most 65535 sequences)
            b0, b1 = int(offsets[lo]), int(offsets[hi])
            d_bytes = data_t[b0:b1].to(self.device, non_blocking=True) if b1 > b0 else torch.empty(
                1, dtype=torch.uint8, device=self.device)
            self.encode_packed_bytes(d_bytes, offsets[lo:hi + 1] - b0, max_seq_len, out[lo:hi])
            lo = hi
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._pin_events[self._pin_slot] = ev
        return out

    def _pinned_copy(self, data: np.ndarray) -> torch.Tensor:
        """Copy host bytes into a reusable page-locked staging buffer (H2D from it is asynchronous).
        Two buffers alternate; a buffer is refilled only after the copies that read it have finished."""
        n = int(data.size)
        self._pin_slot ^= 1
        slot = self._pin_slot
        if self._pin_bufs[slot] is None or self._pin_bufs[slot].numel() < n:
            self._pin_bufs[slot] = torch.empty(max(n, 1 << 20), dtype=torch.uint8).pin_memory()
        elif self._pin_events[slot] is not None:
            self._pin_events[slot].synchronize()
        self._pin_bufs[slot][:n].numpy()[...] = np.asarray(data, dtype=np.uint8).reshape(-1)
        return self._pin_bufs[slot][:n]

    def encode_strings(self, texts: Sequence[bytes], max_seq_len: int, **kw) -> torch.Tensor:
        lens = np.fromiter((len(t) for t in texts), dtype=np.int64, count=len(texts))
        offsets = np.zeros(len(texts) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        data = np.frombuffer(b"".join(texts), dtype=np.uint8) if offsets[-1] else np.zeros(0, dtype=np.uint8)
        return self.encode_bytes(data, offsets, max_seq_len, **kw)

    def encode_ids(self, input_ids: torch.Tensor, attention_mask: torch.Tensor,
                   out_dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
        """`_encode(input_ids, attention_mask)` (reference retrieval/model.py:92-114)."""
        assert input_ids.shape == attention_mask.shape and input_ids.dim() == 2
        ids = input_ids.to(device=self.device, dtype=torch.int64).contiguous()
        mask = attention_mask.to(device=self.device, dtype=torch.int64).contiguous()
        B, L = ids.shape
        out = torch.empty(B, self.hidden_size, dtype=out_dtype, device=self.device)
        with torch.cuda.device(self.device):
            ws = self._workspace(B * L, B)
            _native.check(self.lib.rpx_encode_ids(self._handle, ids.data_ptr(), mask.data_ptr(), B, L, out.data_ptr(),
                                                  self._out_dtype(out_dtype), ws.data_ptr(), ws.numel(),
                                                  _stream_ptr(self.device)))
        return out

    def set_latency_tokens(self, max_tokens: int) -> None:
        """Engine calls with at most `max_tokens` packed tokens take the latency path (narrow tiles: one
        proof state spread over many SMs); 0 switches it off.  See `rpx_encoder_set_latency_tokens`."""
        _native.check(self.lib.rpx_encoder_set_latency_tokens(self._handle, int(max_tokens)))
        self.latency_tokens = int(max_tokens)

    # ------------------------------------------------------------------ debug / profiling
    def set_debug_hidden(self, n_tokens: Optional[int]) -> Optional[torch.Tensor]:
        """Allocate (or drop, with None) the [layers+1, n_tokens, d_model] fp32 hidden-state dump.  Each
        engine call then writes its T packed tokens to rows [0, T) of every slab; a call with more than
        `n_tokens` tokens fails with RPX_ERR_WORKSPACE."""
        if n_tokens is None:
            _native.check(self.lib.rpx_encoder_set_debug_hidden(self._handle, None, 0))
            self._debug_buf = None
            return None
        self._debug_buf = torch.zeros(self._cfg.num_layers + 1, n_tokens, self.hidden_size, dtype=torch.float32,
                                      device=self.device)
        _native.check(self.lib.rpx_encoder_set_debug_hidden(self._handle, self._debug_buf.data_ptr(), int(n_tokens)))
        return self._debug_buf

    def set_profiling(self, enable: bool) -> None:
        _native.check(self.lib.rpx_encoder_set_profiling(self._handle, int(enable)))

    def read_profile(self) -> Dict[str, Dict[str, float]]:
        ms = (C.c_float * _native.RPX_N_KERNEL_CLASSES)()
        cnt = (C.c_int64 * _native.RPX_N_KERNEL_CLASSES)()
        _native.check(self.lib.rpx_encoder_read_profile(self._handle, ms, cnt))
        return {name: {"ms": float(ms[i]), "launches": int(cnt[i])} for i, name in enumerate(_native.KERNEL_CLASS_NAMES)}
