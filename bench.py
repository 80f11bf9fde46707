#!/usr/bin/env python
"""bench.py -- headline metric of BASELINE.json: basecalled samples/s on B200.

One "step" = one pass of the hot path (network forward + CRF decode) over one batch of synthetic chunks.
Workload at N=1: BASELINE.json configs[1] -- dna_r10.4.1 fast@v5 topology, batch 512, chunksize 10000
(normalised to 9996 = 1666 blocks of stride 6), synthetic N(0,1) signal, seeded synthetic weights.
Multi-GPU: one process per GPU (torchrun), each with its own engine replica and its own batch (reads shard
embarrassingly; no collective on the data path) -> weak scaling; time = max over ranks of the device time.

  value  whole-job samples/s with the batches already resident in HBM (CUDA events bracketing the runners' streams);
         `--runners` batches are in flight per GPU (dorado's --num-runners; default here 4 for fast / hac, 2 for sup): the
         recurrences and the beam search are latency chains, so each runner's kernels are sized for a share of the SMs and
         several batches run side by side -- every step is still a full forward + decode of one batch
  e2e    same metric through the C ABI call the adapter makes (b200_runner_call_chunks via
         B200ModelRunner.call_chunks_raw) from pinned host buffers, one host thread per runner:
         H2D of the fp16 batch and D2H of moves/sequence/qstring inside the timed region
  roofline      dominant kernel of the step, timed live per launch with CUDA events (one runner alone, its launch plan
                unchanged); per-kernel table beside it.  A kernel sized for a share of the SMs reports `frac` against the
                whole-GPU peak as the contract defines it, and `frac_of_sms_used` against the peak of the SMs it occupies
                (each decode kernel is charged the bytes of its own interface; `decode` is the three together against the
                algorithmic 2C+3 bytes per chunk-block of SURVEY.md 8d)
  cpu_baseline  the reference's own CPU runner (dorado::basecall::ModelRunner::call_chunks, compiled from the reference
                sources into oracle/_ref) on all host cores -- one runner per core, torch intra-op threads = 1 as dorado
                configures it -- 4 chunks per runner per pass, median of 5 passes after a warm-up; plus the
                single-runner N=1 / N=8 figures with ModelRunner's own model_ms / decode_ms split (SURVEY.md 8d)
  configs       (default run only) the same measurement for hac@512 and sup@128: value / e2e / roofline per model

`--impl reference` times only the CPU runner: a step is one pass of every runner over its 4 chunks; W warm-up passes,
then exactly K timed passes, value = samples of the K passes / their wall time.

`--steps K` / `--warmup W` apply to every timed run: the flagship and, in the default run, the hac / sup sub-results
and their auto-batch runs (device-resident and e2e loops alike).

`--dump-outputs DIR` writes, after the timed steps, what the last timed e2e step returned to its caller for each model
timed (the flagship, plus hac and sup in the default run): DIR/<model>_{moves,sequence,qstring,n_bases,chunk_index}.npy
in float32.  DIR must be new or empty.  Inputs and weights are seeded, so two builds run with the same arguments can be
compared output for output.  Not available with `--impl reference`, whose timed passes discard their outputs.
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

MODELS = {
    "fast": "dna_r10.4.1_e8.2_400bps_fast@v5.0.0",
    "hac": "dna_r10.4.1_e8.2_400bps_hac@v5.0.0",
    "sup": "dna_r10.4.1_e8.2_400bps_sup@v5.0.0",
}
# SURVEY.md section 8(d): algorithmic FLOP per input sample
FLOP_PER_SAMPLE = {"fast": 0.1435e6, "hac": 2.139e6, "sup": 14.35e6}
SUB_MODELS = {"hac": dict(batch=512), "sup": dict(batch=128)}
NUM_SMS = 148
DEFAULT_RUNNERS = {"fast": 4, "hac": 4, "sup": 2}   # batches in flight per GPU (dorado's --num-runners; see --runners)
METRIC = "basecalled samples/s"
DUMP_LIMIT = 64 << 20   # bytes of .npy data one --dump-outputs directory may receive


def model_dir(kind):
    return ROOT / "tests" / "data" / "model_configs" / MODELS[kind]


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, t_begin=None, t_end=None):
        """Summarise the samples whose nvidia-smi timestamp falls inside [t_begin, t_end] (time.time() values)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        out = self._summarise(t_begin, t_end, 0.02)
        if t_begin is not None and out["samples"] < 2:
            # timed region shorter than nvidia-smi's real sampling period: also take the samples of the warm-up
            # (the same kernels, run back to back just before the timed region)
            out = self._summarise(t_begin, t_end, 0.4)
            out["window_widened_s"] = 0.4
        return out

    def _summarise(self, t_begin, t_end, slack):
        import datetime
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                if t_begin is not None:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    if ts < t_begin - slack or ts > t_end + slack:
                        continue
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU reference arm: dorado::basecall::ModelRunner (oracle/_ref), the only place bench.py executes oracle/
# ---------------------------------------------------------------------------------------------------------------------
class CpuReference:
    """`runners` ModelRunners of batch `chunks_per_runner`, each driven by its own host thread (BasecallerNode drives every
    runner from its own worker thread); torch intra-op threads = 1 (dorado/torch_utils/torch_utils.cpp:20)."""

    def __init__(self, kind, chunk_size, runners, chunks_per_runner):
        from dorado_b200.config import load_model_config
        from dorado_b200.weights import synthetic_weights
        from oracle.oracle import Reference, ReferenceRunner
        self.kind = kind
        self.cfg = load_model_config(model_dir(kind))
        self.T = self.cfg.normalise_chunk_size(chunk_size)
        self.ref = Reference()
        self.ref.set_num_threads(1)
        w = synthetic_weights(self.cfg, 42)
        first = ReferenceRunner(self.ref, model_dir(kind), w, chunks_per_runner, chunk_size)
        self.runners = [first] + [ReferenceRunner(self.ref, model_dir(kind), None, chunks_per_runner, chunk_size, share_with=first)
                                  for _ in range(runners - 1)]
        self.B = chunks_per_runner
        rng = np.random.default_rng(1234)
        for r in self.runners:
            sig = rng.standard_normal((self.B, self.T)).astype(np.float32)
            for i in range(self.B):
                r.accept_chunk(i, sig[i])

    def passes(self, n):
        """n passes; every runner calls call_chunks(B) once per pass, all runners start a pass together.  Returns the wall
        time of each pass."""
        R = len(self.runners)
        bar = threading.Barrier(R + 1)
        times = []

        def drive(r):
            for _ in range(n):
                bar.wait()
                r.call_chunks(self.B, want_output=False)
                bar.wait()

        ths = [threading.Thread(target=drive, args=(r,)) for r in self.runners]
        for th in ths:
            th.start()
        for _ in range(n):
            bar.wait()
            t0 = time.perf_counter()
            bar.wait()
            times.append(time.perf_counter() - t0)
        for th in ths:
            th.join()
        return times

    def samples_per_pass(self):
        return len(self.runners) * self.B * self.T

    def close(self):
        for r in self.runners[1:]:
            r.close()
        self.runners[0].close()


def cpu_single_runner(kind, chunk_size, batch, iters=5):
    """One ModelRunner, batch N: wall ms per call_chunks and ModelRunner's own model_ms / decode_ms (ModelRunner.cpp:32-57)."""
    c = CpuReference(kind, chunk_size, 1, batch)
    c.passes(1)
    s0 = c.runners[0].sample_stats()
    times = c.passes(iters)
    s1 = c.runners[0].sample_stats()
    c.close()
    return {"batch": batch, "iters": iters, "ms_per_call": 1e3 * float(np.mean(times)),
            "model_ms": (s1["model_ms"] - s0["model_ms"]) / iters, "decode_ms": (s1["decode_ms"] - s0["decode_ms"]) / iters,
            "samples_per_s": batch * c.T / float(np.mean(times))}


def cpu_reference_budget(kind):
    """runners x chunks per runner for the all-cores figure, bounded so that six passes stay within ~30 s of wall time
    and the replicas fit host memory (sup holds 315 MB of fp32 weights per runner)."""
    cores = os.cpu_count() or 1
    if kind == "fast":
        return cores, 4
    if kind == "hac":
        return cores, 2
    return min(cores, 32), 1


def run_reference_arm(args, config):
    kind = args.model
    runners, per = cpu_reference_budget(kind)
    c = CpuReference(kind, args.chunksize, runners, per)
    W, K = max(0, args.warmup), max(1, args.steps)
    c.passes(max(1, W))
    t0 = time.perf_counter()
    times = c.passes(K)
    total = time.perf_counter() - t0
    value = K * c.samples_per_pass() / total
    sample = (f"{runners} ModelRunners (one per core, torch threads = 1) x {per} chunks of {c.T} samples per pass, {kind} topology, "
              f"ModelRunner::call_chunks (forward + CPUDecoder); {K} passes after {max(1, W)} warm-up")
    c.close()
    config = dict(config, parallelism="host cores only", runners_per_gpu=0, batch_per_gpu=runners * per)
    return {"impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus, "steps": K,
            "warmup": max(1, W), "ms_per_step": 1e3 * total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": runners, "kind": "reference", "sample": sample,
                             "median_pass_ms": 1e3 * float(np.median(times))},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def cpu_baseline_leg(kind, chunksize):
    """The bounded CPU sample reported next to the GPU line (rank 0, N=1 only)."""
    runners, per = cpu_reference_budget(kind)
    c = CpuReference(kind, chunksize, runners, per)
    c.passes(1)
    times = c.passes(5)
    med = float(np.median(times))
    out = {"value": c.samples_per_pass() / med, "unit": "samples/s", "cores": runners, "kind": "reference",
           "sample": f"{runners} ModelRunners (one per core, torch threads = 1) x {per} chunks of {c.T} samples per pass, {kind} "
                     f"topology, ModelRunner::call_chunks; median of 5 passes after 1 warm-up",
           "pass_ms": [round(1e3 * t, 1) for t in times]}
    c.close()
    out["single_runner"] = {"n1": cpu_single_runner(kind, chunksize, 1), "n8": cpu_single_runner(kind, chunksize, 8, iters=3)}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------------------
def kernel_work(cfg, kind, N, T, T_out):
    """Algorithmic work of ONE launch of each kernel (SURVEY.md 8d; DESIGN.md section 4): name -> (bound, amount)."""
    C = cfg.outsize
    S = C // 4
    if cfg.is_tx_model:
        M = N * (T // cfg.stride_inner())          # transformer tokens in the batch
        d, ff = cfg.tx.d_model, cfg.tx.dim_feedforward
        work = {"qkv_gemm": ("tensor", 2.0 * M * d * 3 * d), "out_proj_gemm": ("tensor", 2.0 * M * d * d),
                "fc1_swiglu_gemm": ("tensor", 2.0 * M * d * 2 * ff), "fc2_gemm": ("tensor", 2.0 * M * ff * d),
                "tx_attention": ("tensor", 4.0 * M * cfg.tx.nhead * 64 * (sum(cfg.tx.attn_window) + 1)),
                "upsample_gemm": ("tensor", 2.0 * M * d * cfg.tx.upsample_scale * d),
                "crf_gemm": ("tensor", 2.0 * M * cfg.tx.upsample_scale * d * C),
                "rmsnorm": ("hbm", 2.0 * M * d * 2),
                "tx_conv1": ("hbm", (2.0 + 2.0 * cfg.convs[0].size) * T * N)}
    else:
        Cl = cfg.lstm_size
        work = {"lstm_layer": ("tensor", 16.0 * Cl * Cl * T_out * N),   # 2*(2C)*(4C) per chunk-step
                "lstm_rec": ("tensor", 8.0 * Cl * Cl * T_out * N),      # W_hh half; the W_ih half is lstm_gx_gemm
                "lstm_gx_gemm": ("tensor", 8.0 * Cl * Cl * T_out * N),
                "conv3_gemm": ("tensor", 2.0 * cfg.convs[2].winlen * 16 * Cl * T_out * N),
                "linear_gemm": ("tensor", 2.0 * Cl * C * T_out * N),
                "conv12": ("hbm", (2.0 + 32.0) * T * N)}
    # decode: every kernel is charged the bytes of its own interface (what it must read and write once)
    work["crf_bwd_scan"] = ("hbm", (2.0 * C + 4.0 * S) * T_out * N)               # scores in, fp32 guides out
    work["crf_fwd_beam"] = ("hbm", (2.0 * C + 4.0 * S + 8.0 * 32) * T_out * N)    # scores + guides in, beam records out
    work["crf_traceback"] = ("hbm", (4.0 * 32 + 32.0 + 3.0) * T_out * N)          # meta plane + one 32 B sector of the prob plane per block in, moves/seq/qstring out
    return work


def dump_outputs(out_dir, kind, result, budget):
    """One step's call_chunks_raw result (moves, sequence, qstring [N, T_out] uint8; n_bases [N]) as float32 .npy files.
    Sequence and qstring are zeroed past each chunk's n_bases: a caller's DecodedChunk ends there and the rest of the
    buffer is not part of the result.  Above `budget` bytes, a fixed seeded sample of chunks is written; chunk_index
    lists the chunks kept."""
    moves, seq, qs, nb = (np.array(a) for a in result)
    N, T = moves.shape
    valid = np.arange(T)[None, :] < nb[:, None]
    seq, qs = np.where(valid, seq, 0), np.where(valid, qs, 0)
    keep = min(N, max(1, budget // (3 * T * 4 + 8)))
    rows = np.arange(N) if keep == N else np.sort(np.random.default_rng(0).choice(N, keep, replace=False))
    out_dir = pathlib.Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in (("moves", moves), ("sequence", seq), ("qstring", qs), ("n_bases", nb), ("chunk_index", np.arange(N))):
        np.save(out_dir / f"{kind}_{name}.npy", a[rows].astype(np.float32))


def bench_b200(kind, batch, chunksize, steps, warmup, R, rank, local_rank, world, sampler=None, want_cpu=False,
               dump=None, dump_budget=DUMP_LIMIT):
    import torch
    import torch.distributed as dist
    from dorado_b200.config import load_model_config
    from dorado_b200.runner import B200Caller, B200ModelRunner
    from dorado_b200.weights import synthetic_weights
    cfg = load_model_config(model_dir(kind))
    T = cfg.normalise_chunk_size(chunksize)
    caller = B200Caller(cfg, synthetic_weights(cfg, 42), device=local_rank, num_runners=R)
    runners = [B200ModelRunner(caller, batch, chunksize) for _ in range(R)]
    runner = runners[0]
    rng = np.random.default_rng(1234 + rank)
    for r in runners:
        r.input_view()[:] = rng.standard_normal((batch, T)).astype(np.float16)
    N = batch
    samples_per_step = N * T

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput: step i runs on runner i % R (own stream, own buffers) ----
    for r in runners:
        r.upload()
    W = max(3, warmup)
    B200ModelRunner.step_device_runners(runners, N, W * R)
    launches0 = caller.stats()["gpu_launches"]
    barrier()
    t_begin = time.time()
    tot_ms = B200ModelRunner.step_device_runners(runners, N, steps)
    barrier()
    t_end = time.time()
    launches = caller.stats()["gpu_launches"] - launches0
    clocks = None
    if sampler is not None:
        time.sleep(0.05)
        clocks = sampler.stop(t_begin, t_end)
    _, fwd_ms, dec_ms = runner.step_device(N, steps)  # un-overlapped stage split, outside the timed region
    tot_ms = max_over_ranks(tot_ms)
    value = world * samples_per_step * steps / (tot_ms * 1e-3)

    # ---- end to end through the public API (host buffers), one host thread per runner ----
    last = [None] * R

    def drive(i, n_calls):
        for _ in range(n_calls):
            last[i] = runners[i].call_chunks_raw(N)  # the C-ABI call the C++ adapter makes; results land in pinned host memory

    def run_calls(total):
        ths = [threading.Thread(target=drive, args=(i, total // R + (1 if i < total % R else 0))) for i in range(R)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()

    run_calls(W * R)
    barrier()
    t0 = time.perf_counter()
    run_calls(steps)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    if dump is not None and rank == 0:
        dump_outputs(dump, kind, last[(steps - 1) % R], dump_budget)   # step i ran on runner i % R
    bases_last = int(next(c for c in last if c is not None)[3][:N].sum())
    e2e_value = world * samples_per_step * steps / e2e_s
    h2d = N * T * 2
    d2h = N * runner.out_len() * 3 + 4 * N
    out = {"value": value, "ms_per_step": tot_ms / steps, "steps": steps, "warmup": W,
           "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "ms_per_step": e2e_s / steps * 1e3},
           "gpu_launches": int(launches), "forward_ms_per_step": fwd_ms / steps, "decode_ms_per_step": dec_ms / steps,
           "bases_called_last_step": bases_last, "batch_per_gpu": N, "chunk_samples": T, "runners_per_gpu": R}
    if clocks is not None:
        out["clocks"] = clocks
    if rank != 0:
        for r in runners:
            r.close()
        caller.close()
        return out

    # ---- roofline of the dominant kernel (rank 0, live CUDA events per launch) ----
    pk = peaks()
    prof = {}
    for _ in range(3):
        for name, ms in runner.profile(N):
            prof.setdefault(name, []).append(ms)
    agg = {k: (float(np.mean(v)), len(v) // 3) for k, v in prof.items()}  # mean ms per launch, launches per step
    step_ms = sum(m * c for m, c in agg.values())
    dom = max(agg, key=lambda k: agg[k][0] * agg[k][1])
    dom_ms, dom_cnt = agg[dom]
    C, T_out = cfg.outsize, runner.out_len()
    work = kernel_work(cfg, kind, N, T, T_out)
    bound, amount = work.get(dom, ("tensor", FLOP_PER_SAMPLE[kind] * samples_per_step))
    unit_div, peak, unit = (1e12, pk["tflops"], "TFLOP/s") if bound == "tensor" else (1e9, pk["hbm_gbs"], "GB/s")
    roof = {"kernel": dom, "bound": bound, "achieved": amount / (dom_ms * 1e-3) / unit_div, "peak": peak, "unit": unit,
            "traffic": None}
    roof["frac"] = roof["achieved"] / roof["peak"]

    def entry(k):
        b, amt = work[k]
        div, pkv = (1e12, pk["tflops"]) if b == "tensor" else (1e9, pk["hbm_gbs"])
        ach = amt / (agg[k][0] * 1e-3) / div
        return {"bound": b, "ms_per_launch": round(agg[k][0], 4), "launches": agg[k][1], "achieved": round(ach, 2),
                "frac": round(ach / pkv, 4)}

    roof["per_kernel"] = {k: entry(k) for k in agg if k in work}
    # Kernels that are deliberately launched on a share of the SMs (several runners' latency-bound kernels side by side,
    # b200_engine_set_num_runners): `frac` above stays launch work / launch time / whole-GPU peak; `frac_of_sms_used` scales
    # the peak to the SMs the launch occupies (one CTA per SM), which is the efficiency of the SM-time it consumes.
    plan = runner.plan_info()
    for k, e in roof["per_kernel"].items():
        ctas = plan.get(k + ".ctas")
        if ctas and ctas < NUM_SMS:
            e["ctas"] = ctas
            e["frac_of_sms_used"] = round(e["frac"] * NUM_SMS / ctas, 4)
    if dom in roof["per_kernel"] and "ctas" in roof["per_kernel"][dom]:
        roof["ctas"] = roof["per_kernel"][dom]["ctas"]
        roof["frac_of_sms_used"] = roof["frac"] * NUM_SMS / roof["ctas"]
        roof["note"] = (f"{dom} runs on {roof['ctas']} of {NUM_SMS} SMs by design ({R} batches in flight share the GPU); frac = "
                        f"launch work / launch time / whole-GPU peak, frac_of_sms_used = the same against the peak of the SMs used")
    if plan:
        roof["plan"] = plan
    dec_kernels = [k for k in ("crf_bwd_scan", "crf_fwd_beam", "crf_traceback") if k in agg]
    dec_total_ms = sum(agg[k][0] * agg[k][1] for k in dec_kernels)
    dec_alg = (2.0 * C + 3.0) * T_out * N
    roof["decode"] = {"bound": "hbm", "algorithmic_bytes": dec_alg, "ms": round(dec_total_ms, 4),
                      "achieved": round(dec_alg / (dec_total_ms * 1e-3) / 1e9, 2),
                      "frac": round(dec_alg / (dec_total_ms * 1e-3) / 1e9 / pk["hbm_gbs"], 4)}
    # DRAM bytes per launch from this round's `ncu --set full` captures of the same workload (profiles/r02_traffic.json,
    # written by tools/ncu_summary.py): for the dominant kernel as roofline.traffic, and per kernel; null when not captured
    try:
        tr_all = json.loads((ROOT / "profiles" / "r02_traffic.json").read_text())
    except (OSError, ValueError):
        tr_all = {}
    for k, e in roof["per_kernel"].items():
        tr = tr_all.get(f"{kind}_n{N}_{k}")
        if tr:
            e["traffic"] = tr["dram_bytes"]
    tr = tr_all.get(f"{kind}_n{N}_{dom}")
    if tr:
        roof["traffic"] = tr["dram_bytes"]
        roof["traffic_source"] = f"profiles/{tr['file']} launch {tr['launch']} ({tr['kernel']})"
    roof["peak_source"] = pk["source"]
    roof["ms_per_launch"] = dom_ms
    roof["launches_per_step"] = dom_cnt
    roof["share_of_step"] = dom_ms * dom_cnt / step_ms
    roof["kernels_ms"] = {k: round(m * c, 4) for k, (m, c) in agg.items()}
    roof["forward_tflops"] = FLOP_PER_SAMPLE[kind] * samples_per_step / (fwd_ms / steps * 1e-3) / 1e12
    out["roofline"] = roof

    if want_cpu:
        try:
            out["cpu_baseline"] = cpu_baseline_leg(kind, chunksize)
        except Exception as e:  # the checker is optional for the headline number
            out["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": os.cpu_count(), "kind": "reference",
                                   "sample": f"unavailable: {e}"}
    for r in runners:
        r.close()
    caller.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="fast", choices=list(MODELS))
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--chunksize", type=int, default=10000)
    ap.add_argument("--runners", type=int, default=None,
                    help="runners (batches in flight) per GPU = dorado's --num-runners (default there 2 per device, "
                         "api/runner_creation.cpp:91-123).  Default here: 4 for fast (its recurrence and beam search are latency "
                         "chains; four batches side by side fill the SMs, profiles/r02_b11_*), 2 for hac and sup")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU reference leg (batch sweeps)")
    ap.add_argument("--no-sub-models", action="store_true", help="skip the hac@512 / sup@128 sub-results of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned (moves, sequence, qstring, n_bases) "
                         "as DIR/<model>_<name>.npy, float32, at most 64 MB in all; DIR must be new or empty")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None:
        if args.impl == "reference":
            ap.error("--dump-outputs records the B200 path; the reference arm's timed passes return no outputs")
        d = pathlib.Path(args.dump_outputs)
        if d.exists() and (not d.is_dir() or any(d.iterdir())):
            ap.error(f"--dump-outputs {d}: must be a new or empty directory, so that no earlier run's files mix in")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    kind = args.model

    from dorado_b200.config import load_model_config
    cfg = load_model_config(model_dir(kind))
    T = cfg.normalise_chunk_size(args.chunksize)
    config = {"workload": f"{MODELS[kind]} topology (synthetic weights), batch {args.batch} per GPU, chunksize "
                          f"{args.chunksize} -> {T} samples/chunk, synthetic N(0,1) fp16 signal",
              "model": kind, "batch_per_gpu": args.batch, "chunk_samples": T, "parallelism": f"replica x{args.gpus}",
              "runners_per_gpu": args.runners if args.runners is not None else DEFAULT_RUNNERS[kind],
              "l2": "per-step working set (conv activations + scores > 400 MB) exceeds the 126 MB L2; no explicit flush"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        print(json.dumps(run_reference_arm(args, config)))
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)  # let nvidia-smi reach its sampling loop
    R = max(1, args.runners if args.runners is not None else DEFAULT_RUNNERS[kind])
    config["runners_per_gpu"] = R
    default_run = kind == "fast" and args.batch == 512 and not args.no_sub_models
    dump_budget = DUMP_LIMIT // (1 + len(SUB_MODELS) if default_run else 1)
    main_res = bench_b200(kind, args.batch, args.chunksize, args.steps, args.warmup, R, rank, local_rank, world, sampler=sampler,
                          want_cpu=(world == 1 and not args.no_cpu_baseline), dump=args.dump_outputs, dump_budget=dump_budget)
    subs = {}
    if default_run:
        for sk, sc in SUB_MODELS.items():
            res = bench_b200(sk, sc["batch"], args.chunksize, args.steps, args.warmup, DEFAULT_RUNNERS[sk], rank, local_rank, world,
                             dump=args.dump_outputs, dump_budget=dump_budget)
            if rank == 0:
                keep = ("value", "ms_per_step", "steps", "e2e", "forward_ms_per_step", "decode_ms_per_step", "batch_per_gpu",
                        "chunk_samples", "runners_per_gpu", "gpu_launches", "bases_called_last_step")
                subs[sk] = {k: res[k] for k in keep}
                r = res["roofline"]
                subs[sk]["roofline"] = {k: r[k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "share_of_step",
                                                          "per_kernel", "decode", "forward_tflops", "traffic")}
        # BASELINE.json configs[2], [3]: the same models at the batch size the engine picks itself -- the counterpart of
        # CudaCaller::determine_batch_dims (pre-computed "NVIDIA B200" table + exact memory cap at 80 % of the free HBM)
        from dorado_b200 import batching
        from dorado_b200.config import load_model_config as _lc
        from dorado_b200.runner import B200Caller
        from dorado_b200.weights import synthetic_weights
        for sk, sc in SUB_MODELS.items():
            cfg_s = _lc(model_dir(sk))
            probe = B200Caller(cfg_s, synthetic_weights(cfg_s, 42), device=local_rank, num_runners=DEFAULT_RUNNERS[sk])
            free_b, _tot = torch.cuda.mem_get_info(local_rank)
            dims, source = batching.determine_batch_dims(probe, MODELS[sk], args.chunksize, int(0.8 * free_b),
                                                         num_runners=DEFAULT_RUNNERS[sk])
            probe.close()
            auto_batch = int(dims[0][0])
            res = bench_b200(sk, auto_batch, args.chunksize, args.steps, args.warmup, DEFAULT_RUNNERS[sk], rank, local_rank,
                             world)
            if rank == 0:
                subs[sk + "_auto_batch"] = {k: res[k] for k in ("value", "ms_per_step", "steps", "e2e", "batch_per_gpu",
                                                               "chunk_samples", "runners_per_gpu", "gpu_launches")}
                subs[sk + "_auto_batch"]["batch_source"] = f"determine_batch_dims: {source}, chunk-size buckets {dims}"
    if rank != 0:
        return 0
    line = {"metric": METRIC, "value": main_res["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": main_res["warmup"], "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 (fp32 accumulate; fp32 decode)", "data": "synthetic",
            "config": config, "clocks": main_res.get("clocks"), "e2e": main_res["e2e"],
            "gpu_launches": main_res["gpu_launches"], "forward_ms_per_step": main_res["forward_ms_per_step"],
            "decode_ms_per_step": main_res["decode_ms_per_step"], "roofline": main_res["roofline"],
            "cpu_baseline": main_res.get("cpu_baseline", {"value": None, "unit": "samples/s", "cores": os.cpu_count(),
                                                            "kind": "reference", "sample": "reported at N=1 only"}),
            "bases_called_last_step": main_res["bases_called_last_step"]}
    if subs:
        line["configs"] = subs
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
