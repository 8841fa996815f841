#!/usr/bin/env python
"""bench.py — premises encoded/s (reindex) and retrieve() queries/s on B200s, next to the
reference's own CPU path.

    python bench.py --gpus 1 --steps K --warmup W            # engine arm
    python bench.py --impl reference --steps K --warmup W    # reference arm (HF CPU path)
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU

Workload (BASELINE.json configs[1], "reindex 200k synthetic premises, seq_len <= 512, ByT5-small"):
a *step* is one re-index pass over one batch of `--premises-per-step` synthetic premises drawn from
the cfg2 distribution (byte length ~ U[16, 511] + EOS, SURVEY.md §8d), random-init ByT5-small
weights (seed 3407).  Every step uses a fresh slice of the corpus; the per-step working set
(~19 KB of activations per token, > 10 GB) is far larger than L2, so no flush is needed.
`--full` makes one step the whole 200k corpus.

  value  whole-job premises/s with the premise bytes already resident in HBM, CUDA-event timed,
         max over ranks.
  e2e    the same pass through the public API (`B200PremiseRetriever.reindex_corpus` on a `Corpus`
         of Premise objects, then `.cpu()` of the index as retrieval/index.py:37 does): host
         strings -> pinned bytes -> H2D -> engine -> D2H inside the timed region.
  retrieve   extra leg, BASELINE configs[2]/[3]: 1024 states x 200k-premise (per GPU) bf16 index,
         k = 100, fused sim+top-k (+ all-gather + merge when N > 1): queries/s and roofline, plus a
         `parity` object: 64 sampled queries re-ranked by brute force (fp64 Q.E^T of every rank's shard,
         all-gathered, exact top-k) against the engine's merged result on EVERY rank — a mismatch makes
         the run exit non-zero.
  retrieve_q1 / retrieve_q64   the same index with 1 and 64 states (the reference's production call is one
         state per retrieve(), retrieval/model.py:338-375): device time, host-to-host time, HBM roofline.
  retrieve_single (N = 1)  `B200PremiseRetriever.retrieve(state, file, theorem, pos, 100)` host to host on a
         200k-premise corpus: encode of one state + access bitmask + top-k + Premise objects.
  sweep (N = 1)  BASELINE configs[4]: encoder throughput at seq_len {128,512,1024,2048} x batch {32,128,512}.
  reindex_2048 (N = 1)  the shape retrieval/index.py:33 indexes at: max_seq_len 2048, token length ~ U[17, 2048].

`--dump-outputs DIR` writes what rank 0's timed calls returned in their last repetition, so that two builds
run with the same arguments (hence the same seeded inputs) can be compared output for output:
  reindex_embeddings.npy   float32 [rows, 1472], the last timed step's premise embeddings (bf16 widened); when a
                           step holds more than 8192 premises, 8192 of them, the same seeded sample every run,
                           and reindex_rows.npy (float64) says which
  retrieve_q{1024,64,1}_indices.npy / _scores.npy   float64 [Q, 100], the global top-k rows and their fp64 scores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from reprover_b200 import synth  # noqa: E402

D_MODEL = 1472
N_CORPUS = 200_000
MAX_SEQ_LEN = 512
# 8192 x 1472 fp32 = 48 MB: with the retrieve results a dump stays under 64 MB
DUMP_MAX_ROWS = 8192


def cpu_threads() -> int:
    """Host threads of every CPU leg: half the logical CPUs (= the physical cores on these hosts),
    set explicitly so that a torchrun launch (which exports OMP_NUM_THREADS=1) times the same thing as a
    plain one."""
    n = int(os.environ.get("RPX_CPU_THREADS", "0")) or max(1, (os.cpu_count() or 2) // 2)
    torch.set_num_threads(n)
    return n


def encoder_flops(token_lens: np.ndarray) -> float:
    """Algorithmic FLOPs of the encoder for sequences of the given token lengths (SURVEY.md §8d)."""
    l = token_lens.astype(np.float64)
    return float((l * (434_110_464.0 + 18_432.0 * l)).sum())


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # samples taken while the GPU was busy are the upper half of the clock distribution
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    # stdout carries exactly one JSON line: NCCL's own banner / debug lines (NCCL_DEBUG=VERSION|INFO) go to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def max_over_ranks(ms: float, world: int, dev) -> float:
    if world == 1:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def barrier(world: int):
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ engine arm
def run_engine(args) -> dict:
    from reprover_b200 import _native
    from reprover_b200.corpus import Corpus, File, Pos, Premise
    from reprover_b200.engine import T5EncoderEngine
    from reprover_b200.retrieval_ops import IndexHandle
    from reprover_b200.retriever import B200PremiseRetriever

    rank, world, local = dist_env()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N > 1)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    K, W = args.steps, args.warmup
    P = N_CORPUS if args.full else args.premises_per_step

    cfg = dict(synth.BYT5_SMALL)
    sd = synth.random_t5_state_dict(cfg, seed=synth.SEED)
    eng = T5EncoderEngine(cfg, sd, dev, max_tokens_per_call=args.max_tokens_per_call)

    # this rank's premises for all steps (rank r draws from seed 3407 + r: SURVEY §8d cfg4)
    n_steps = K + W
    data, offsets = synth.synth_premises(P * n_steps if not args.full else P, seed=synth.SEED + rank)
    if args.full:
        step_slices = [(0, P)] * n_steps
    else:
        step_slices = [(i * P, (i + 1) * P) for i in range(n_steps)]
    tok_lens = np.minimum(np.diff(offsets) + 1, MAX_SEQ_LEN)

    d_data = torch.from_numpy(data.copy()).to(dev)
    out = torch.empty(P, D_MODEL, dtype=torch.bfloat16, device=dev)

    def device_step(i):
        lo, hi = step_slices[i]
        cum = np.concatenate([[0], np.cumsum(tok_lens[lo:hi])])
        a = 0
        n = hi - lo
        while a < n:
            b = int(np.searchsorted(cum, cum[a] + eng.max_tokens_per_call, side="right")) - 1
            b = min(max(b, a + 1), n)
            b0, b1 = int(offsets[lo + a]), int(offsets[lo + b])
            eng.encode_packed_bytes(d_data[b0:b1], offsets[lo + a:lo + b + 1] - b0, MAX_SEQ_LEN, out[a:b])
            a = b

    # ---- device-resident throughput
    for i in range(W):
        device_step(i)
    eng.set_profiling(True)
    eng.read_profile()
    sampler = ClockSampler(local)
    barrier(world)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(W, W + K):
        device_step(i)
    e1.record()
    barrier(world)
    clocks = sampler.stop()
    ms_dev = max_over_ranks(e0.elapsed_time(e1), world, dev)
    prof = eng.read_profile()
    eng.set_profiling(False)
    dump = {} if args.dump_outputs and rank == 0 else None
    if dump is not None:
        rows = np.arange(P)
        if P > DUMP_MAX_ROWS:
            rows = np.sort(np.random.default_rng(synth.SEED).choice(P, DUMP_MAX_ROWS, replace=False))
            dump["reindex_rows"] = rows.astype(np.float64)
        dump["reindex_embeddings"] = out[torch.from_numpy(rows).to(dev)].float().cpu().numpy()
    timed_tokens = sum(int(tok_lens[lo:hi].sum()) for lo, hi in step_slices[W:W + K])
    timed_flops = sum(encoder_flops(tok_lens[lo:hi]) for lo, hi in step_slices[W:W + K])
    value = world * P * K / (ms_dev / 1e3)

    # dominant kernel: the FFN up-projection GEMM (58 % of the FLOPs)
    ffn = prof["ffn_up_gemm"]
    ffn_flops = 2.0 * timed_tokens * 7168 * 1472 * cfg["num_layers"]
    ffn_tf = ffn_flops / (ffn["ms"] / 1e3) / 1e12 if ffn["ms"] > 0 else 0.0
    traffic = None
    tpath = ROOT / "profiles" / "roofline_traffic.json"
    if tpath.exists():
        traffic = json.loads(tpath.read_text()).get("ffn_up_gemm_dram_bytes_per_launch")
    launches = sum(v["launches"] for v in prof.values())

    # ---- end to end through the public API (host strings in, host index out)
    e2e = None
    if not args.skip_e2e:
        ckpt = Path(args.tmp) / f"byt5_small_synth_rank{rank}"
        synth.save_hf_checkpoint(str(ckpt), cfg, sd)
        del eng
        torch.cuda.empty_cache()
        retr = B200PremiseRetriever.load_hf(str(ckpt), MAX_SEQ_LEN, dev)
        retr.encoder.max_tokens_per_call = args.max_tokens_per_call

        def make_corpus(i):
            lo, hi = step_slices[i]
            prem = []
            for j in range(lo, hi):
                code = data[offsets[j]:offsets[j + 1]].tobytes().decode()
                prem.append(Premise("Synth.lean", f"Synth.p{j}", Pos(j + 1, 0), Pos(j + 1, 1), code))
            return Corpus.from_files([(File("Synth.lean", prem), [])])

        corpora = [make_corpus(0)] * n_steps if args.full else [make_corpus(i) for i in range(n_steps)]
        h2d = d2h = 0
        host_index = None
        for i in range(W):
            retr.load_corpus(corpora[i])
            retr.reindex_corpus(batch_size=64)
            host_index = retr.corpus_embeddings.to(torch.float32).cpu()
        barrier(world)
        t0 = time.perf_counter()
        e0.record()
        for i in range(W, W + K):
            retr.load_corpus(corpora[i])
            retr.reindex_corpus(batch_size=64)
            host_index = retr.corpus_embeddings.to(torch.float32).cpu()   # retrieval/index.py:37: fp32 host copy
            lo, hi = step_slices[i]
            h2d += int(offsets[hi] - offsets[lo])
            d2h += host_index.numel() * host_index.element_size()
        e1.record()
        barrier(world)
        ms_e2e = max_over_ranks(e0.elapsed_time(e1), world, dev)
        wall_e2e = time.perf_counter() - t0
        e2e = {"value": world * P * K / (ms_e2e / 1e3), "unit": "premises/s", "h2d_bytes_per_step": h2d // K,
               "d2h_bytes_per_step": d2h // K, "ms_per_step": ms_e2e / K, "host_wall_s": wall_e2e}
        eng_for_retrieve = retr.encoder
    else:
        eng_for_retrieve = eng

    # ---- retrieve legs (cfg3 per GPU; cfg4 when world == 8; plus the 1- and 64-state shapes)
    retrieve = retrieve_q1 = retrieve_q64 = None
    if not args.skip_retrieve:
        n_idx, k = N_CORPUS, 100
        E = synth.random_unit_rows(n_idx, D_MODEL, 1000 + rank, dev)
        handle = IndexHandle(E)
        Q_all = synth.random_unit_rows(1024, D_MODEL, 999, dev)   # same queries on every rank
        retrieve = retrieve_leg(Q_all, E, handle, k, rank, world, dev, peaks, e0, e1, K, W, check_parity=True, dump=dump)
        retrieve_q64 = retrieve_leg(Q_all[:64].contiguous(), E, handle, k, rank, world, dev, peaks, e0, e1, K, W, dump=dump)
        retrieve_q1 = retrieve_leg(Q_all[:1].contiguous(), E, handle, k, rank, world, dev, peaks, e0, e1, K, W, dump=dump)
        retrieve["guard"] = handle.stats()
        if rank == 0 and world == 1 and not args.skip_cpu_baseline:
            retrieve["cpu_baseline"] = cpu_baseline_retrieve(E, Q_all, k)
        del handle, E

    # ---- single-GPU extras: retrieve() as the prover calls it, the config-5 sweep, max_seq_len 2048
    retrieve_single = sweep = reindex_2048 = None
    if world == 1 and not args.skip_extras:
        if e2e is not None:
            retrieve_single = retrieve_single_leg(retr, dev)
        sweep = sweep_leg(eng_for_retrieve, dev, peaks)
        reindex_2048 = reindex_2048_leg(eng_for_retrieve, dev, peaks)

    result = {
        "metric": "premises encoded/sec (reindex_corpus, ByT5-small, seq_len<=512)",
        "value": value, "unit": "premises/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: reindex synthetic premises, byte len~U[16,511]+EOS, ByT5-small random-init seed 3407",
                   "premises_per_step_per_gpu": P, "tokens_per_step_per_gpu": timed_tokens // K, "max_seq_len": MAX_SEQ_LEN,
                   "parallelism": f"row-sharded corpus x{world}, no data-path collective in reindex",
                   "l2": "inputs larger than L2 (fresh premises every step; ~19 KB activations/token)",
                   "max_tokens_per_call": args.max_tokens_per_call},
        "encoder_roofline": {"achieved_tflops": timed_flops / (ms_dev / 1e3) / 1e12, "peak": peaks["tf_sustained"],
                             "frac": timed_flops / (ms_dev / 1e3) / 1e12 / peaks["tf_sustained"],
                             "note": "WHOLE PATH: algorithmic FLOPs sum F(l_i) of SURVEY 8d over the whole step (per GPU) / step time; "
                                     "`roofline` below is the dominant kernel alone"},
        "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel<6,EpiGeGLU> (FFN up-projection, 2-CTA tcgen05, 58% of FLOPs)",
                     "achieved": ffn_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                     "frac": ffn_tf / peaks["tf_sustained"], "peak_source": peaks["source"] + " (sustained bf16)",
                     "traffic": traffic, "launches": ffn["launches"], "avg_launch_ms": ffn["ms"] / max(ffn["launches"], 1)},
        "kernel_ms": {k2: v["ms"] for k2, v in prof.items()},
        "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "retrieve": retrieve,
        "retrieve_q1": retrieve_q1, "retrieve_q64": retrieve_q64, "retrieve_single": retrieve_single,
        "sweep": sweep, "reindex_2048": reindex_2048,
    }
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    parity = (retrieve or {}).get("parity")
    if parity is not None and parity["mismatches"] != 0:
        exc = SystemExit(f"[bench] retrieve parity FAILED: {parity}")
        exc.bench_result = result if rank == 0 else None
        raise exc
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        result["cpu_baseline"] = cpu_baseline_encode(cfg, sd, data, offsets, n_premises=args.cpu_sample)
    if world > 1:
        torch.distributed.destroy_process_group()
    return result if rank == 0 else None


# ------------------------------------------------------------------------------------------ retrieve legs
def brute_force_parity(Q, E, k, rank, world, dev, got_idx, got_s64, n_sample=64):
    """Checker (not the product): fp64 Q.E^T of this rank's shard for `n_sample` queries, exact local
    top-(k+8), all-gather, global exact top-k under (score desc, index asc); compared on EVERY rank with
    the engine's merged result.  fp64 torch sums in another order than the engine's canonical one, so a
    position only counts as a mismatch when the scores around it differ by more than 1e-12."""
    nq = Q.shape[0]
    sel = torch.linspace(0, nq - 1, steps=min(n_sample, nq), device=dev).round().long().unique()
    S = Q[sel].double() @ E.double().t()                                   # [s, n_idx] fp64
    top = torch.topk(S, k + 8, dim=1)
    loc_s, loc_i = top.values, top.indices + rank * E.shape[0]
    if world > 1:
        gs = [torch.empty_like(loc_s) for _ in range(world)]
        gi = [torch.empty_like(loc_i) for _ in range(world)]
        torch.distributed.all_gather(gs, loc_s)
        torch.distributed.all_gather(gi, loc_i)
        loc_s, loc_i = torch.cat(gs, dim=1), torch.cat(gi, dim=1)
    # order: score desc, index asc (stable sort on index first, then on score)
    o = torch.argsort(loc_i, dim=1, stable=True)
    loc_s, loc_i = torch.gather(loc_s, 1, o), torch.gather(loc_i, 1, o)
    o = torch.argsort(loc_s, dim=1, descending=True, stable=True)
    want_s, want_i = torch.gather(loc_s, 1, o)[:, :k + 1], torch.gather(loc_i, 1, o)[:, :k + 1]
    g_i, g_s = got_idx[sel], got_s64[sel]
    differs = g_i != want_i[:, :k]
    # a differing position is tolerated only inside a run of (numerically) tied scores
    gap_ok = (g_s - want_s[:, :k]).abs() < 1e-12
    mism = int((differs & ~gap_ok).sum())
    score_err = float((g_s - want_s[:, :k]).abs().max())
    bad_scores = int(((g_s - want_s[:, :k]).abs() >= 1e-12).sum())
    out = {"checked_queries": int(sel.numel()), "k": k, "mismatches": mism + bad_scores, "index_positions_differing_within_ties": int((differs & gap_ok).sum()),
           "max_abs_score_diff": score_err, "checker": "torch fp64 matmul + exact top-k per shard, all-gathered, on every rank"}
    if world > 1:
        t = torch.tensor([out["mismatches"]], device=dev)
        torch.distributed.all_reduce(t)                                   # any rank's mismatch fails the run
        out["mismatches"] = int(t.item())
        out["ranks_checked"] = world
    return out


def retrieve_leg(Q, E, handle, k, rank, world, dev, peaks, e0, e1, K, W, check_parity=False, dump=None):
    from reprover_b200.dist import sharded_topk
    from reprover_b200.retrieval_ops import sim_topk

    nq, n_idx = Q.shape[0], E.shape[0]
    Q_host = Q.cpu().pin_memory()
    # one retrieve is 0.1-0.6 ms: a handful of repetitions would be timed while the SM clock is still
    # ramping after the host-side legs; 50 repetitions after 10 warm-ups are past that
    reps, warm_r = max(50, K), max(10, W)

    def retrieve_dev(q=Q):
        if world == 1:
            return sim_topk(q, handle, k, want_scores64=True)
        s32, idx, cnt, s64 = sharded_topk(q, handle, k, row_offset=rank * n_idx)
        return s32, idx, cnt, s64

    for _ in range(warm_r):
        retrieve_dev()
    barrier(world)
    e0.record()
    for _ in range(reps):
        last = retrieve_dev()
    e1.record()
    barrier(world)
    ms_r = max_over_ranks(e0.elapsed_time(e1), world, dev) / reps
    if dump is not None:
        dump[f"retrieve_q{nq}_indices"] = last[1].double().cpu().numpy()
        dump[f"retrieve_q{nq}_scores"] = last[3].cpu().numpy()
    # e2e: queries from pinned host memory, results back to the host
    res_scores = torch.empty(nq, k, dtype=torch.float32).pin_memory()
    res_idx = torch.empty(nq, k, dtype=torch.int64).pin_memory()

    def retrieve_host():
        r = retrieve_dev(Q_host.to(dev, non_blocking=True))
        res_scores.copy_(r[0], non_blocking=True)
        res_idx.copy_(r[1], non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the caller reads the host result here

    for _ in range(3):
        retrieve_host()   # warm-up (allocator, pinned staging)
    barrier(world)
    e0.record()
    for _ in range(reps):
        retrieve_host()
    e1.record()
    barrier(world)
    ms_re = max_over_ranks(e0.elapsed_time(e1), world, dev) / reps
    flops = 2.0 * nq * n_idx * D_MODEL
    bytes_alg = n_idx * D_MODEL * 2 + nq * D_MODEL * 2 + nq * k * 12
    t_mma = flops / (peaks["tf_burst"] * 1e12)
    t_hbm = bytes_alg / (peaks["hbm_gbs"] * 1e9)
    bound = "tensor" if t_mma > t_hbm else "hbm"
    leg = {
        "metric": "retrieve queries/s", "config": {"queries": nq, "index_rows_per_gpu": n_idx, "index_rows_total": n_idx * world,
                                                  "k": k, "dtype": "bf16", "merge": "nccl all_gather + device merge" if world > 1 else "none",
                                                  "path": "streaming kernel (HBM-bound)" if nq <= 2 else "tcgen05 MMA + fused top-k",
                                                  "warmup": warm_r, "repetitions": reps, "l2": "index (589 MB) larger than L2"},
        "value": nq / (ms_r / 1e3), "ms": ms_r,
        "e2e": {"value": nq / (ms_re / 1e3), "ms": ms_re, "h2d_bytes": nq * D_MODEL * 2, "d2h_bytes": nq * k * 12},
        "roofline": {"bound": bound,
                     "achieved": (flops / (ms_r / 1e3) / 1e12) if bound == "tensor" else (bytes_alg / (ms_r / 1e3) / 1e9),
                     "peak": peaks["tf_burst"] if bound == "tensor" else peaks["hbm_gbs"],
                     "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                     "frac": max(t_mma, t_hbm) / (ms_r / 1e3), "hbm_frac": t_hbm / (ms_r / 1e3),
                     # the same against the sustained tensor rate (what a power-capped B200 holds over a step)
                     "frac_of_sustained": (max(flops / (peaks["tf_sustained"] * 1e12), t_hbm) / (ms_r / 1e3)) if bound == "tensor" else None,
                     "algorithmic_bytes": bytes_alg, "peak_source": peaks["source"] + (" (burst bf16)" if bound == "tensor" else ""),
                     "note": "whole retrieve (every launch of the call [+ all-gather + merge]) vs max(t_MMA, t_HBM) of one pass over the index"},
    }
    if bound == "hbm" and nq <= 2:
        tpath = ROOT / "profiles" / "roofline_traffic.json"
        if tpath.exists():
            leg["roofline"]["traffic"] = json.loads(tpath.read_text()).get("smallq_topk_dram_bytes_per_launch")
            leg["roofline"]["kernel"] = "smallq_topk_kernel<1,6> (one streaming pass over the bf16 index, fused per-warp heaps + fp64 re-score + rank)"
    if check_parity:
        r = retrieve_dev()
        torch.cuda.synchronize()
        leg["parity"] = brute_force_parity(Q, E, k, rank, world, dev, r[1], r[3])
    return leg


def retrieve_single_leg(retr, dev):
    """`retrieve()` host to host, one state per call, on a 200k-premise corpus split into 2000 files
    (a chain of imports, so the access bitmask is a real one)."""
    from reprover_b200.corpus import Corpus, File, Pos, Premise

    N, n_files = N_CORPUS, 2000
    files = []
    for f in range(n_files):
        prem = [Premise(f"F{f}.lean", f"F{f}.p{j}", Pos(j + 1, 0), Pos(j + 1, 5), f"theorem p{j} : True := trivial")
                for j in range(N // n_files)]
        files.append((File(f"F{f}.lean", prem), [f"F{f - 1}.lean"] if f else []))
    retr.load_corpus(Corpus.from_files(files))
    retr.corpus_embeddings = synth.random_unit_rows(N, D_MODEL, 7, dev)   # latency does not depend on the values
    retr.embeddings_staled = False
    sdat, soff = synth.synth_states(80, seed=5, min_len=50, max_len=400)
    states = [s.decode() for s in synth.split_strings(sdat, soff)]
    where = (f"F{n_files - 1}.lean", "t", Pos(50, 0))
    for st in states[:16]:
        retr.retrieve(st, *where, 100)
    torch.cuda.synchronize()
    lat = []
    for st in states[16:]:
        t0 = time.perf_counter()
        prem, sc = retr.retrieve(st, *where, 100)
        lat.append((time.perf_counter() - t0) * 1e3)
    assert len(prem) == 100
    # where the time goes: the encode of the one state (latency path) alone, CUDA events around the call
    # (tokenisation, the copy of its bytes and the ~65 launches included)
    enc_ms = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for st in states[16:48]:
        torch.cuda.synchronize()
        e0.record()
        retr._encode_states([st])
        e1.record()
        torch.cuda.synchronize()
        enc_ms.append(e0.elapsed_time(e1))
    return {"metric": "retrieve() latency, one state per call, host to host", "unit": "ms",
            "median": float(np.median(lat)), "p90": float(np.percentile(lat, 90)), "min": float(min(lat)), "calls": len(lat),
            "encode_state_ms_median": float(np.median(enc_ms)),
            "config": {"index_rows": N, "files": n_files, "k": 100, "state_bytes": "U[50,400]", "max_seq_len": retr.max_seq_len,
                       "accessible_rows": int(N - N // n_files + 49)}}


def sweep_leg(eng, dev, peaks):
    """BASELINE configs[4]: seq_len {128,512,1024,2048} x batch {32,128,512}, ids ~ U[3,258], full-length
    rows (SURVEY 8d), device-timed with CUDA events, 3 warm-ups per point."""
    rng = np.random.default_rng(synth.SEED)
    rows = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for L in (128, 512, 1024, 2048):
        for B in (32, 128, 512):
            data = rng.integers(0, 256, size=B * (L - 1), dtype=np.uint8)   # ids 3..258 = bytes 0..255, + EOS
            offsets = np.arange(B + 1, dtype=np.int64) * (L - 1)
            d = torch.from_numpy(data).to(dev)
            out = torch.empty(B, D_MODEL, dtype=torch.bfloat16, device=dev)
            per_call = max(1, eng.max_tokens_per_call // L)

            def step():
                for a in range(0, B, per_call):
                    b = min(B, a + per_call)
                    eng.encode_packed_bytes(d[offsets[a]:offsets[b]], offsets[a:b + 1] - offsets[a], L, out[a:b])

            for _ in range(3):
                step()
            reps = max(2, min(20, int(4e5 // (B * L))))
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            tf = B * L * (434_110_464.0 + 18_432.0 * L) / ms / 1e9
            rows.append({"seq_len": L, "batch": B, "ms": ms, "seq_per_s": B / ms * 1e3, "tflops": tf,
                         "frac_of_sustained_peak": tf / peaks["tf_sustained"], "reps": reps})
    return {"metric": "encoder sequences/s and roofline fraction, BASELINE configs[4]", "peak": peaks["tf_sustained"],
            "peak_source": peaks["source"] + " (sustained bf16)", "rows": rows,
            "frac_min": min(r["frac_of_sustained_peak"] for r in rows), "frac_max": max(r["frac_of_sustained_peak"] for r in rows)}


def reindex_2048_leg(eng, dev, peaks, P=2048):
    """The shape the reference indexes at (retrieval/index.py:33: max_seq_len 2048): byte length ~ U[16, 2047]."""
    data, offsets = synth.synth_premises(P * 3, seed=synth.SEED + 7, min_len=16, max_len=2047)
    tok = np.minimum(np.diff(offsets) + 1, 2048)
    d_data = torch.from_numpy(data.copy()).to(dev)
    out = torch.empty(P, D_MODEL, dtype=torch.bfloat16, device=dev)

    def step(i):
        lo, hi = i * P, (i + 1) * P
        cum = np.concatenate([[0], np.cumsum(tok[lo:hi])])
        a = 0
        while a < P:
            b = int(np.searchsorted(cum, cum[a] + eng.max_tokens_per_call, side="right")) - 1
            b = min(max(b, a + 1), P)
            b0, b1 = int(offsets[lo + a]), int(offsets[lo + b])
            eng.encode_packed_bytes(d_data[b0:b1], offsets[lo + a:lo + b + 1] - b0, 2048, out[a:b])
            a = b

    step(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    step(1)
    step(2)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 2
    fl = encoder_flops(tok[P:3 * P]) / 2
    tf = fl / ms / 1e9
    return {"metric": "premises encoded/sec at max_seq_len 2048", "value": P / ms * 1e3, "unit": "premises/s", "ms_per_step": ms,
            "config": {"premises_per_step": P, "token_len": "U[17,2048]", "tokens_per_step": int(tok[P:3 * P].sum() // 2), "warmup_steps": 1, "steps": 2},
            "encoder_roofline": {"achieved_tflops": tf, "peak": peaks["tf_sustained"], "frac": tf / peaks["tf_sustained"]}}


# ------------------------------------------------------------------------------------------ CPU reference
def cpu_baseline_encode(cfg, sd, data, offsets, n_premises: int, precision: str = "medium") -> dict:
    """The reference's own path on the host cores: HF T5EncoderModel fp32, reference batching
    (batch 64, pad to longest, corpus order), `torch.set_float32_matmul_precision("medium")` as
    retrieval/model.py:26 sets it.  Bounded sample; this is the oracle used as a stopwatch."""
    from oracle import reference_path as ref

    cpu_threads()
    torch.set_float32_matmul_precision(precision)
    enc = ref.build_hf_encoder(cfg, sd)
    tok = ref.build_hf_tokenizer()
    texts = [s.decode() for s in synth.split_strings(data, offsets[: n_premises + 1])]
    ref.reindex_corpus(enc, tok, texts[:2], 64, MAX_SEQ_LEN)  # warm-up
    t0 = time.perf_counter()
    ref.reindex_corpus(enc, tok, texts, 64, MAX_SEQ_LEN)
    dt = time.perf_counter() - t0
    torch.set_float32_matmul_precision("highest")
    return {"value": n_premises / dt, "unit": "premises/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(),
            "kind": "port", "sample": f"first {n_premises} premises of the cfg2 corpus, batch 64 pad-to-longest, fp32 matmul precision '{precision}', {dt:.1f} s",
            "note": "oracle/reference_path.py = reference algorithm on HF T5EncoderModel (the reference modules need lean_dojo/lightning/deepspeed, absent here)"}


def cpu_baseline_retrieve(E_dev: torch.Tensor, Q_dev: torch.Tensor, k: int, n_queries: int = 64) -> dict:
    """Reference retrieve arithmetic on the host cores (common.py:307-324: fp32 matmul, full argsort,
    .tolist(), Python walk) for a bounded sample of the same queries against the same index."""
    from oracle import reference_path as ref

    cpu_threads()
    torch.set_float32_matmul_precision("medium")
    E = E_dev.float().cpu()
    Q = Q_dev[:n_queries].float().cpu()
    ref.nearest_unfiltered_verbatim(E, Q[:1], k)  # warm-up
    t0 = time.perf_counter()
    ref.nearest_unfiltered_verbatim(E, Q, k)
    dt = time.perf_counter() - t0
    torch.set_float32_matmul_precision("highest")
    return {"value": n_queries / dt, "unit": "queries/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "sample": f"{n_queries} of the 1024 states against the full {E.shape[0]}-row fp32 index, k={k}, {dt:.1f} s"}


def run_reference(args) -> dict:
    """--impl reference: the reference's CPU implementation of the path, all host threads,
    each step a bounded sample of the same workload."""
    rank, world, _ = dist_env()
    if rank != 0:
        return None
    from oracle import reference_path as ref

    K, W = args.steps, args.warmup
    S = args.reference_premises_per_step
    cfg = dict(synth.BYT5_SMALL)
    sd = synth.random_t5_state_dict(cfg, seed=synth.SEED)
    cpu_threads()
    torch.set_float32_matmul_precision("medium")  # retrieval/model.py:26
    enc = ref.build_hf_encoder(cfg, sd)
    tok = ref.build_hf_tokenizer()
    data, offsets = synth.synth_premises(S * (K + W), seed=synth.SEED)
    texts = [s.decode() for s in synth.split_strings(data, offsets)]
    for i in range(W):
        ref.reindex_corpus(enc, tok, texts[i * S:(i + 1) * S], 64, MAX_SEQ_LEN)
    t0 = time.perf_counter()
    for i in range(W, W + K):
        ref.reindex_corpus(enc, tok, texts[i * S:(i + 1) * S], 64, MAX_SEQ_LEN)
    dt = time.perf_counter() - t0
    v = S * K / dt
    return {
        "impl": "reference",
        "metric": "premises encoded/sec (reindex_corpus, ByT5-small, seq_len<=512)",
        "value": v, "unit": "premises/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": dt / K * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (matmul precision 'medium')", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: reindex synthetic premises, byte len~U[16,511]+EOS, ByT5-small random-init seed 3407",
                   "premises_per_step": S, "max_seq_len": MAX_SEQ_LEN, "batching": "reference: batch 64, pad to longest, corpus order"},
        "cpu_baseline": {"value": v, "unit": "premises/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
                         "sample": f"{S} premises per step x {K} steps of the cfg2 corpus ({dt:.1f} s)"},
        "e2e": {"value": v, "unit": "premises/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--premises-per-step", type=int, default=8192)
    ap.add_argument("--full", action="store_true", help="one step = the whole 200k-premise corpus")
    ap.add_argument("--max-tokens-per-call", type=int, default=1 << 18)
    ap.add_argument("--cpu-sample", type=int, default=64, help="premises timed on the CPU baseline")
    ap.add_argument("--reference-premises-per-step", type=int, default=8)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-retrieve", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="skip retrieve_single / sweep / reindex_2048 (N = 1 legs)")
    ap.add_argument("--tmp", default=None,
                    help="where the e2e leg's checkpoint goes, in a fresh directory removed at exit (default: the system's temp dir)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed calls' last outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs applies to the engine arm")
    if args.impl == "engine" and args.warmup < 3:
        print(f"[bench] --warmup {args.warmup} raised to 3 (timing rules: at least 3 warm-up steps)", file=sys.stderr)
        args.warmup = 3
    # stdout carries exactly ONE JSON line: anything a library prints to file descriptor 1 meanwhile
    # (NCCL's version banner with NCCL_DEBUG=VERSION, for one) is sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        with tempfile.TemporaryDirectory(prefix="rpx_bench_", dir=args.tmp) as tmp:
            args.tmp = tmp
            res = run_reference(args) if args.impl == "reference" else run_engine(args)
    except SystemExit as exc:
        res = getattr(exc, "bench_result", None)
        if res is not None:
            os.write(real_stdout, (json.dumps(res) + "\n").encode())
        raise
    if res is not None:
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(res) + "\n").encode())


if __name__ == "__main__":
    main()
