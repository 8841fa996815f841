"""CPU-side checks of the C ABI: the library loads, exports everything include/rpx.h declares,
host-only entry points work, compute entry points fail LOUDLY without a GPU (no fallback)."""
import ctypes as C
import json
import re
from pathlib import Path

import pytest
import torch

from reprover_b200 import _native, synth

ROOT = Path(__file__).resolve().parent.parent
needs_no_gpu = pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")


def _declared_functions():
    text = (ROOT / "include" / "rpx.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rpx_[a-z0-9_]+)\s*\(", text)))


def test_header_and_library_agree(rpx_lib):
    declared = _declared_functions()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(rpx_lib, name), f"{name} declared in include/rpx.h but not exported by librpx.so"
    assert sorted(_native.EXPORTED_SYMBOLS) == declared, "ctypes signature table out of sync with the header"
    assert rpx_lib.rpx_version() == 200


def test_library_has_no_libcuda_dependency():
    """Loads on a box without libcuda.so.1 (the driver entry points are resolved at run time)."""
    import subprocess

    out = subprocess.run(["readelf", "-d", str(_native.library_path())], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out


def test_sass_is_blackwell_native():
    """The cubin carries tcgen05 MMA / TMEM / TMA instructions (UTC*MMA, LDTM, UTMALDG), sm_100a only."""
    import subprocess

    sass = subprocess.run(["cuobjdump", "-sass", str(_native.library_path())], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in sass, mnemonic


def test_host_only_entry_points(rpx_lib):
    cfg = _native.T5Config(vocab_size=384, d_model=1472, d_kv=64, d_ff=3584, num_layers=12, num_heads=6,
                           rel_buckets=32, rel_max_distance=128, ln_eps=1e-6)
    nbytes = rpx_lib.rpx_encoder_packed_bytes(C.byref(cfg))
    # bf16 copy of the 12 blocks (12 * 18,087,936 matrix params) + fp32 embedding/norm/bias tables
    assert 12 * 18_087_936 * 2 <= nbytes <= 12 * 18_087_936 * 2 + 4_000_000
    bad = _native.T5Config(vocab_size=384, d_model=1472, d_kv=32, d_ff=3584, num_layers=12, num_heads=6,
                           rel_buckets=32, rel_max_distance=128, ln_eps=1e-6)
    assert rpx_lib.rpx_encoder_packed_bytes(C.byref(bad)) == 0
    assert "d_kv" in _native.last_error()
    assert rpx_lib.rpx_sim_topk_workspace_bytes(200_000, 1472, 1024, 100) > 0
    assert rpx_lib.rpx_index_topk_workspace_bytes(200_000, 1472, 1, 100) > 200_000 * 16   # room for the exact pass
    assert rpx_lib.rpx_index_topk_workspace_bytes(200_000, 1472, 8, 1000) > 0              # k > 200: exact pass only
    assert rpx_lib.rpx_index_topk_workspace_bytes(200_000, 1472, 8, 5000) == 0             # out of range -> loud, not clamped
    assert rpx_lib.rpx_index_state_bytes() >= 64
    assert rpx_lib.rpx_encoder_workspace_bytes(None, 1000, 10) == 0


def test_packed_bytes_rejects_a_bias_table_attention_cannot_hold(rpx_lib):
    """A relative-position range whose bias table does not fit the attention kernel's shared memory is refused
    when the encoder is sized, not on its first encode call: 1584 is the largest range that fits."""
    def cfg(R):
        return _native.T5Config(vocab_size=384, d_model=1472, d_kv=64, d_ff=3584, num_layers=2, num_heads=6,
                                rel_buckets=32, rel_max_distance=R, ln_eps=1e-6)

    assert rpx_lib.rpx_encoder_packed_bytes(C.byref(cfg(1584))) > 0
    for R in (1585, 2048):
        assert rpx_lib.rpx_encoder_packed_bytes(C.byref(cfg(R))) == 0
        assert "rel_max_distance" in _native.last_error()


def test_relative_bucket_matches_hf_golden(rpx_lib):
    g = json.loads((ROOT / "tests" / "golden" / "bucket_table.json").read_text())
    got = [rpx_lib.rpx_t5_relative_bucket(r, g["num_buckets"], g["max_distance"]) for r in g["relative_position"]]
    assert got == g["bucket"]
    assert 16 not in got  # SURVEY §8 a3: bucket 16 is never produced


@needs_no_gpu
def test_compute_fails_loudly_without_gpu(rpx_lib):
    assert rpx_lib.rpx_device_check() == _native.RPX_ERR_CUDA
    buf = (C.c_uint8 * 1024)()
    rc = rpx_lib.rpx_gemm_bf16_f32(buf, buf, buf, 128, 256, 64, None)
    assert rc == _native.RPX_ERR_CUDA and _native.last_error()
    rc = rpx_lib.rpx_sim_topk(buf, 1, buf, 10, 64, 5, None, 0, buf, None, buf, None, 0, buf, 1024, None)
    assert rc != _native.RPX_OK
    rc = rpx_lib.rpx_topk_merge(buf, buf, 2, 1, 5, buf, None, buf, None, None)
    assert rc != _native.RPX_OK
    rc = rpx_lib.rpx_topk_merge_packed(buf, 2, 1, 5, buf, None, buf, None, None)
    assert rc != _native.RPX_OK
    h = C.c_void_p()
    rc = rpx_lib.rpx_index_create(buf, 4, 64, buf, None, C.byref(h))
    assert rc != _native.RPX_OK and not h.value


@needs_no_gpu
def test_python_product_path_refuses_cpu():
    from reprover_b200.engine import T5EncoderEngine
    from reprover_b200.retrieval_ops import sim_topk

    cfg = synth.tiny_config(1)
    with pytest.raises(RuntimeError, match="CUDA"):
        T5EncoderEngine(cfg, synth.random_t5_state_dict(cfg, 1), "cpu")
    q = torch.zeros(2, 64, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="CUDA"):
        sim_topk(q, q, 1)


def test_product_path_never_imports_oracle():
    """No module under reprover_b200/ may import, link or shell out to anything under oracle/
    (_build.py only *compiles* the checker)."""
    for path in list((ROOT / "reprover_b200").rglob("*.py")) + list((ROOT / "tools").rglob("*.py")):
        text = path.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), path
    # outside tests/, only the two sanctioned call sites touch it: smoke() and bench.py's CPU legs
    for name in ("bench.py", "__graft_entry__.py"):
        text = (ROOT / name).read_text()
        for m in re.finditer(r"^(\s*)(from|import)\s+oracle\b", text, flags=re.M):
            assert len(m.group(1)) >= 4, f"{name}: oracle must only be imported inside the functions that use it as checker / stopwatch"
    for path in (ROOT / "reprover_b200" / "csrc").iterdir():
        assert not re.search(r'#include\s+[<"][^>"]*oracle', path.read_text()), path
