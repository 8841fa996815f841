"""Both T5 attention kernels (`rpx_t5_attention_bf16`: 0 = throughput, 1 = latency) against a plain fp64
softmax attention of the same bf16 q / k / v and the same fp32 relative-bias table.

Error bound, per output element.  The kernels compute the scores in fp32, round P to bf16 for the P V product
but add the unrounded P into the row sum, and round the output to bf16.  bf16 carries 8 significant bits, so
rounding to nearest moves a value by at most 2^-8 of itself.  With W the fp64 softmax weights:
    |o - o_ref| <= 2^-8 (W |V|)   (P rounding)   +   2^-8 |o_ref|   (output rounding)
and both terms come close to their worst case somewhere in a few million elements.  The assertion allows twice
that (2^-7), which also covers ex2.approx, the fp32 scores and the fp32 sums (all relative 2^-20 or less).
The largest err / bound each test sees goes to attention_err_ratio.json in the suite's `out_dir`.
"""
import ctypes as C
import json

import numpy as np
import pytest
import torch

from reprover_b200 import _native
from tests.helpers import attention_fp64, hf_bias_table

pytestmark = pytest.mark.gpu

KERNELS = {"throughput": 0, "latency": 1}
HD = 64
LAT_MAX = 1024
# every tile / chunk / block edge of either kernel: 16-key MMA groups, 32-key chunks, 32- and 128-query CTAs,
# 64-key steps, 256-key blocks
LENS = [1, 2, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 383, 384, 385, 511, 512, 513,
        767, 768, 769, 1023, 1024]
LONG_LENS = [1025, 2047, 2048, 3001]   # throughput kernel only

_RATIOS = {}


@pytest.fixture(scope="module", autouse=True)
def _record_ratios(out_dir):
    yield
    (out_dir / "attention_err_ratio.json").write_text(json.dumps(
        {"max_ratio": max(_RATIOS.values(), default=0.0), "per_case": _RATIOS}, indent=1))


def _lens_for(kernel):
    return LENS + (LONG_LENS if kernel == "throughput" else [])


def run_attention(lib, qkv, lens, H, lut, R, kernel, expect=_native.RPX_OK):
    """One call over the packed sequences; `out` starts as NaN, with 64 rows past the last token."""
    cu = [0, *np.cumsum(lens).tolist()]
    T = cu[-1]
    dev = qkv.device
    out = torch.full((T + 64, H * HD), float("nan"), dtype=torch.bfloat16, device=dev)
    h_cu = (C.c_int32 * len(cu))(*cu)
    d_cu = torch.tensor(cu, dtype=torch.int32, device=dev)
    lut = lut.to(device=dev, dtype=torch.float32).contiguous()
    rc = lib.rpx_t5_attention_bf16(qkv.data_ptr(), out.data_ptr(), d_cu.data_ptr(), h_cu, len(lens), H, lut.data_ptr(), R,
                                   KERNELS[kernel], torch.cuda.current_stream().cuda_stream)
    if expect != _native.RPX_OK:
        assert rc == expect, (rc, _native.last_error())
        return None
    _native.check(rc)
    torch.cuda.synchronize()
    # every row of the call is written, nothing past it
    assert not torch.isnan(out[:T].float()).any(), "rows left unwritten"
    assert torch.isnan(out[T:].float()).all(), "write past the last sequence"
    return out[:T]


def check_against_reference(tag, got, qkv, lens, H, lut, R):
    want, wv = attention_fp64(qkv, lens, H, lut, R)
    err = (got.double() - want).abs()
    bound = 2.0 ** -7 * (wv + want.abs())
    ratio = err / bound.clamp_min(1e-300)
    worst = float(ratio.max())
    _RATIOS[tag] = max(worst, _RATIOS.get(tag, 0.0))
    if worst > 1.0:
        r = int(ratio.amax(1).argmax())
        seq = int(np.searchsorted(np.cumsum(lens), r, side="right"))
        pytest.fail(f"{tag}: err/bound {worst:.3g} at token {r} (sequence {seq}, length {lens[seq]}, row "
                    f"{r - int(np.sum(lens[:seq]))}): got {got[r, :4].tolist()} want {want[r, :4].tolist()}")
    # a sequence of one token attends to itself only: its own V row, bit for bit
    t0 = 0
    for L in lens:
        if L == 1:
            assert torch.equal(got[t0], qkv[t0, 2 * H * HD:]), f"{tag}: length-1 sequence at {t0}"
        t0 += L
    return worst


def make_qkv(lens, H, score_std, seed, dev):
    """Random q / k / v rows; q.k has standard deviation `score_std` (q, k ~ N(0, score_std / 8))."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    T = int(sum(lens))
    s = (score_std / HD ** 0.5) ** 0.5
    q = torch.randn(T, H * HD, generator=g) * s
    k = torch.randn(T, H * HD, generator=g) * s
    v = torch.randn(T, H * HD, generator=g)
    return torch.cat([q, k, v], 1).to(torch.bfloat16).to(dev)


@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("score_std", [1.0, 8.0], ids=["flat", "sharp"])
def test_random_packed(rpx_lib, cuda_device, kernel, score_std):
    """Random operands at every edge length, packed into one call (shuffled, so sequences start at every
    alignment), with the HF-bucketed table of a random 32 x 6 relative bias."""
    H, R = 6, 128
    lens = list(np.random.default_rng(1).permutation(_lens_for(kernel)))
    qkv = make_qkv(lens, H, score_std, seed=int(score_std), dev=cuda_device)
    lut = hf_bias_table(torch.randn(32, H, generator=torch.Generator().manual_seed(2)) * 0.5, R)
    got = run_attention(rpx_lib, qkv, lens, H, lut, R, kernel)
    check_against_reference(f"random_{kernel}_std{score_std:g}", got, qkv, lens, H, lut, R)


@pytest.mark.parametrize("kernel,R", [(k, r) for k in KERNELS for r in (8, 128, 480)] + [("throughput", 1584)])
@pytest.mark.parametrize("H", [1, 6, 12])
def test_bias_indexing(rpx_lib, cuda_device, kernel, R, H):
    """q = 0: the weights come from the bias table alone.  The table is random (std 3) and different for every
    delta and head, so a shifted, mis-clamped or other-head entry at any tile / block offset changes the output.
    R = 480 is the largest table the latency kernel holds, 1584 the largest the throughput kernel holds."""
    lens = _lens_for(kernel)
    qkv = make_qkv(lens, H, 1.0, seed=R + H, dev=cuda_device)
    qkv[:, :H * HD] = 0
    lut = torch.randn(H, 2 * R + 1, generator=torch.Generator().manual_seed(R * 31 + H)) * 3.0
    got = run_attention(rpx_lib, qkv, lens, H, lut, R, kernel)
    check_against_reference(f"bias_{kernel}_R{R}_H{H}", got, qkv, lens, H, lut, R)


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_uniform_weights_give_the_exact_mean(rpx_lib, cuda_device, kernel):
    """q = 0 and a zero table make every weight exactly 1, so each output is the mean of V over exactly the
    sequence's keys: bf16(mean) to within one bf16 ulp (the fp32 sum of grid values is exact, 1 / len is rounded).
    Neighbouring sequences alternate between V of order 1 and of order 2^12, so one key read across a boundary,
    or one key missed, shows at once."""
    H = 6
    lens = _lens_for(kernel)
    T = sum(lens)
    g = torch.Generator().manual_seed(7)
    v = torch.randint(-64, 65, (T, H * HD), generator=g).float() / 16
    t0 = 0
    for i, L in enumerate(lens):
        if i % 2:
            v[t0:t0 + L] *= 2 ** 12
        t0 += L
    qkv = torch.cat([torch.zeros(T, 2 * H * HD), v], 1).to(torch.bfloat16).to(cuda_device)
    lut = torch.zeros(H, 2 * 128 + 1)
    got = run_attention(rpx_lib, qkv, lens, H, lut, 128, kernel).float().cpu()
    t0 = 0
    for L in lens:
        mean = (v[t0:t0 + L].double().sum(0) / L)
        want = mean.float().to(torch.bfloat16).float()
        ulp = torch.where(want == 0, torch.zeros_like(want), 2.0 ** (torch.floor(torch.log2(want.abs())) - 7))
        bad = (got[t0:t0 + L] - want[None]).abs() > ulp[None]
        assert not bad.any(), (L, int(bad.sum()), got[t0, :4].tolist(), want[:4].tolist())
        t0 += L


def _structured_qkv(k0, q0, H, dev, seed):
    """q = q0 e_0 and k_j = k0_j e_0 in every head: the scores q0_i k0_j are exact in fp32, so the test controls
    each row's running maximum exactly.  V is random."""
    T = k0.shape[0]
    qkv = torch.zeros(T, 3 * H * HD)
    for h in range(H):
        qkv[:, h * HD] = q0
        qkv[:, H * HD + h * HD] = k0
    qkv[:, 2 * H * HD:] = torch.randn(T, H * HD, generator=torch.Generator().manual_seed(seed))
    return qkv.to(torch.bfloat16).to(dev)


def _run_structured(lib, dev, kernel, tag, k0_per_seq, q0_per_seq, lut_std=0.0, R=128):
    H = 2
    lens = [len(k) for k in k0_per_seq]
    qkv = _structured_qkv(torch.cat(k0_per_seq), torch.cat(q0_per_seq), H, dev, seed=len(tag))
    lut = torch.randn(H, 2 * R + 1, generator=torch.Generator().manual_seed(3)) * lut_std
    got = run_attention(lib, qkv, lens, H, lut, R, kernel)
    return check_against_reference(tag, got, qkv, lens, H, lut, R)


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_spike_key(rpx_lib, cuda_device, kernel):
    """One key scores far above the rest (20-40 against N(0, 1)): the first key, the last key, a key inside the
    partial 16-key MMA group at the end, and keys in the second, third and fourth key blocks."""
    g = torch.Generator().manual_seed(11)
    ks, qs = [], []
    for L, spike in [(1000, 0), (1000, 999), (1000, 995), (777, 770), (1024, 300), (1024, 600), (1024, 900),
                     (700, 64), (129, 128), (17, 16)]:
        k0 = torch.randn(L, generator=g)
        k0[spike] = 40.0
        ks.append(k0)
        qs.append(0.5 + 0.5 * torch.rand(L, generator=g))
    _run_structured(rpx_lib, cuda_device, kernel, f"spike_{kernel}", ks, qs, lut_std=0.5)


@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("step", [5.0, 6.0], ids=["under_tau", "over_tau"])
def test_rising_and_falling_maxima(rpx_lib, cuda_device, kernel, step):
    """Each 64-key step (and so each 256-key block) holds a larger maximum than the last, by just under or just
    over 8 ln 2 = 5.55, the throughput kernel's lazy-rescale threshold: its lazy path and its O / row-sum rescale
    both run, and the latency kernel rescales at every block.  Rows with q = 2 see twice the growth.  Falling
    maxima (no rescale due) run in the same call."""
    g = torch.Generator().manual_seed(int(step))
    L = 1024 if kernel == "latency" else 2048
    kstep = torch.arange(L) // 64
    top = kstep.float() * step
    rising = top - torch.randint(0, 12, (L,), generator=g).float()
    rising[torch.arange(0, L, 64) + torch.randint(0, 64, (L // 64,), generator=g)] = top[::64]
    falling = rising.flip(0)
    q = torch.tensor([1.0, 2.0, 0.5, 1.0]).repeat(L // 4)
    _run_structured(rpx_lib, cuda_device, kernel, f"maxima_{kernel}_step{step:g}",
                    [rising, falling, rising[:777]], [q, q, q[:777]])


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_large_magnitude_scores(rpx_lib, cuda_device, kernel):
    """Scores around +-500 (q = +-1, k around 500) must neither overflow nor lose the softmax."""
    g = torch.Generator().manual_seed(5)
    ks, qs = [], []
    for L in (1, 33, 300, 1024):
        ks.append(500.0 + 4.0 * torch.randn(L, generator=g))
        qs.append(torch.where(torch.rand(L, generator=g) < 0.5, -1.0, 1.0))
    mixed = torch.where(torch.rand(700, generator=g) < 0.5, -500.0, 500.0) + torch.randn(700, generator=g)
    ks.append(mixed)
    qs.append(torch.ones(700))
    _run_structured(rpx_lib, cuda_device, kernel, f"large_{kernel}", ks, qs, lut_std=0.5)


def test_refusals(rpx_lib, cuda_device):
    """The latency kernel refuses what it cannot run rather than falling back; bad offsets are refused."""
    H = 1
    qkv = make_qkv([1025], H, 1.0, seed=0, dev=cuda_device)
    lut = torch.zeros(H, 2 * 128 + 1)
    run_attention(rpx_lib, qkv, [1025], H, lut, 128, "latency", expect=_native.RPX_ERR_UNSUPPORTED)
    assert "1024" in _native.last_error()
    run_attention(rpx_lib, qkv[:1024], [1024], H, torch.zeros(H, 2 * 481 + 1), 481, "latency",
                  expect=_native.RPX_ERR_UNSUPPORTED)
    run_attention(rpx_lib, qkv, [1025], H, torch.zeros(H, 2 * 1585 + 1), 1585, "throughput",
                  expect=_native.RPX_ERR_UNSUPPORTED)
    for lens in ([5, 0, 3], [5, -2]):
        run_attention(rpx_lib, qkv, lens, H, lut, 128, "throughput", expect=_native.RPX_ERR_INVALID)
