#!/usr/bin/env python
"""bench.py -- decode tokens/s at batch 1 on B200 (BASELINE.json metric), plus roofline, parity and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload nano-168m-q80|qwen3-0.6b-q80|qwen3-0.6b-q4k|...]
    python bench.py --impl reference ...        # the reference's own OpenMP CPU engine on the host cores

A *step* is one pass of the hot path over one batch of synthetic input: a 16-token prompt is pushed through the
token-at-a-time path (infer.c:1258-1260), then greedy decode (temperature 0, repetition penalty 1.0) runs to `seq`
(SURVEY 8(d)).  tokens/s is counted over the decode segment only, like the reference's own TPS.

  value    : device-resident loop (nb200_decode_greedy: the token is fed back on the GPU, inputs already in HBM), decode
             segments timed with CUDA events on the launching stream, max over ranks.  No host can reach this loop through
             the reference API: it is the kernel-side number; the drop-in number is `e2e`.
  e2e      : the same metric through the per-token C-ABI call a reference host makes (nb200_next_greedy ==
             generate_next_token): every token does a pinned H2D of the step descriptor + token id and a D2H of the
             resulting id; wall-clock over the decode segment.
  roofline : dominant kernel.  Streaming path: the one persistent kernel (algorithmic bytes of the launch / launch duration).
             Multi-kernel path: the W1|W3 + SwiGLU matvec, from a live CUDA-event pass over every launch (graph/PDL off).
  parity   : the ids of a timed run, checked position by position against the oracle fed with the same ids (first divergence
             and the oracle's top-1/top-2 margin there); `exact_mode` = tok/s of the bit-exact mode on the same workload.
  configs  : the other single-GPU BASELINE configs (Qwen3-0.6B Q80 / Q4K at 2048) measured in the same run (N = 1 only).
  tp       : N > 1: BASELINE config 5 -- ONE Qwen3-4B Q80 session at seq 4096 row-sharded over the N GPUs (activations through
             NVLink peer memory), beside the same path on one GPU measured in the same job.
  cpu_baseline : the unmodified reference (oracle/_ref, Makefile flags) on the host cores over a bounded sample.

N > 1 (torchrun): `value` = N independent batch-1 sessions (the path shards by session: no data-path collective => "weak").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from nano_b200 import modelfile as mf  # noqa: E402

WORKLOADS = {
    # name: (preset, quant, gs, seq)   -- BASELINE.json configs[1..4]
    "nano-168m-q80": ("nano-168m", mf.QUANT_Q80, 128, 512),
    "qwen3-0.6b-q80": ("qwen3-0.6b", mf.QUANT_Q80, 128, 2048),
    "qwen3-0.6b-q4k": ("qwen3-0.6b", mf.QUANT_Q4K, 0, 2048),
    "nano-168m-f32": ("nano-168m", mf.QUANT_F32, 0, 128),
    "nano-168m-q4k": ("nano-168m", mf.QUANT_Q4K, 0, 512),
    "qwen3-1.7b-q80": ("qwen3-1.7b", mf.QUANT_Q80, 128, 2048),
    "qwen3-4b-q80": ("qwen3-4b", mf.QUANT_Q80, 128, 4096),
    "toy-qwen3-q80": ("toy-qwen3", mf.QUANT_Q80, 64, 128),
}
FAST_FILE = {"qwen3-1.7b-q80": True, "qwen3-4b-q80": True}      # multi-GB files: synthesise codes/scales directly (seconds, not minutes)
EXTRA_CONFIGS = ["qwen3-0.6b-q80", "qwen3-0.6b-q4k"]            # measured beside the headline config at N = 1
TP_WORKLOAD = "qwen3-4b-q80"                                     # BASELINE config 5
PROMPT = 16
DTYPE = {mf.QUANT_Q80: "int8xint8->int32 + f32", mf.QUANT_Q4K: "u4xu4->int32 + f32", mf.QUANT_F32: "f32"}


def _metric_name():
    """The headline metric exactly as BASELINE.json names it (tokens/s is `value`; the GB/s-vs-roofline half is `roofline`)."""
    try:
        return json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    except Exception:
        return "decode tokens/sec at batch=1; achieved HBM GB/s vs roofline"


METRIC = _metric_name()
CLASS_NAMES = ["embed", "qkv", "attention", "o_proj", "w13_swiglu", "w2", "classifier"]
BPW = {mf.QUANT_F32: lambda gs: 4.0, mf.QUANT_Q80: lambda gs: 1.0 + 4.0 / max(gs, 1), mf.QUANT_Q4K: lambda gs: 148.0 / 256.0}


def workload_config(name):
    """The `config` object: identical in the B200 arm and in the reference arm."""
    preset, quant, gs, seq = WORKLOADS[name]
    spec = mf.PRESETS[preset]
    wbytes = spec.n_weights() * BPW[quant](gs)
    return {"workload": f"{name} greedy decode, seq={seq}, prompt={PROMPT}, max_seq_len={seq}",
            "l2": "inputs larger than L2: %.0f MB of weights (+ the KV cache) are streamed per token vs 126 MB of L2" % (wbytes / 1e6),
            "timing": "decode segment of each step (tokens %d..%d); GPU: CUDA events on the launching stream, max over ranks; CPU: wall clock" % (PROMPT, seq - 1)}


def prompt_ids(spec, seq):
    ids = np.zeros(seq + 1, np.uint32)
    ids[:PROMPT] = [(17 + i % 10) if spec.arch == mf.ARCH_NANO else 1000 + i for i in range(PROMPT)]
    return ids


def model_path(name):
    preset, quant, gs, _seq = WORKLOADS[name]
    return mf.cached_model(mf.PRESETS[preset], quant, gs or 128, fast=FAST_FILE.get(name, False))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# CPU reference (runs in a subprocess so OMP_* take effect before libgomp loads)
# --------------------------------------------------------------------------------------------------
CPU_CHILD = r"""
import json, os, sys, time
import numpy as np
sys.path.insert(0, {root!r})
from oracle import bindings as ob
path, seq, sample_end, P, kind, flavour, arch, runs = {path!r}, {seq}, {sample_end}, {P}, {kind!r}, {flavour!r}, {arch}, {runs}
if kind == "reference":
    eng = ob.RefEngine(path, seq, flavour, penalty=1.0, temperature=0.0)
else:
    eng = ob.NanoOracle(path, seq)
    ob.NanoOracle.lib().nor_set_threads(int(os.environ.get("OMP_NUM_THREADS", "1")))
out = []
for _ in range(runs):
    ids = np.zeros(seq + 1, np.uint32)
    ids[:P] = [(17 + i % 10) if arch == 0 else 1000 + i for i in range(P)]
    step = (lambda pos, pre: eng.next(ids, pos, pre)) if kind == "reference" else (lambda pos, pre: eng.next_greedy(ids, pos, pre, 1.0))
    for pos in range(P - 1):
        ids[pos + 1] = step(pos, 1)
    t0 = time.perf_counter()
    n = 0
    for pos in range(P - 1, sample_end - 1):
        ids[pos + 1] = step(pos, 0); n += 1
    out.append({{"tokens": n, "seconds": time.perf_counter() - t0}})
print(json.dumps(out))
"""


def _cpu_run(path, spec, seq, sample_end, kind, flavour, threads, bind, runs, timeout=600):
    env = dict(os.environ, OMP_NUM_THREADS=str(threads))
    if bind:
        env.update(OMP_PROC_BIND="true", OMP_WAIT_POLICY="active")
    else:
        env.pop("OMP_PROC_BIND", None); env.pop("OMP_WAIT_POLICY", None)
    code = CPU_CHILD.format(root=ROOT, path=path, seq=seq, sample_end=sample_end, P=PROMPT, kind=kind, flavour=flavour or "",
                            arch=spec.arch, runs=runs)
    try:
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=timeout)
        return [r["tokens"] / r["seconds"] for r in json.loads(out.stdout.strip().splitlines()[-1])]
    except Exception:
        return []


def cpu_sweep(path, spec, seq, budget_s=30.0):
    """BASELINE.md section 3: OMP_NUM_THREADS x {default, OMP_PROC_BIND=true OMP_WAIT_POLICY=active} on a short probe
    (README.md:73: N 'must be found by experiment'); returns the best (threads, bind) and the probe table."""
    from oracle import bindings as ob
    flavour = ob.best_fast_flavour()
    kind = "reference" if flavour else "port"
    ncpu = os.cpu_count() or 1
    probe_end = min(seq, PROMPT + (16 if spec.n_embd >= 1024 else 48))
    # most promising counts first (a matvec of these sizes stops scaling around 16-32 threads); the budget cuts the tail
    order = [t for t in (16, 32, 8, 64, 4, ncpu // 2, ncpu, 2, 1) if 1 <= t <= ncpu]
    cands = [t for i, t in enumerate(order) if t not in order[:i]]
    table, best, t0 = [], None, time.time()
    for th in cands:
        for bind in (True, False):
            if time.time() - t0 > budget_s and best is not None:
                break
            r = _cpu_run(path, spec, seq, probe_end, kind, flavour, th, bind, 1, timeout=45)
            if not r:
                continue
            table.append({"threads": th, "bind": bind, "tok_s": round(r[0], 1)})
            if best is None or r[0] > best[0]:
                best = (r[0], th, bind)
    return kind, flavour, best, table, ncpu, probe_end


def cpu_baseline(workload, path, spec, seq, runs=1):
    """`cpu_baseline` of the B200 arm: thread sweep on a probe, then the bounded sample (prompt + 64 decode positions) at the best setting."""
    kind, flavour, best, table, ncpu, _ = cpu_sweep(path, spec, seq, budget_s=20.0)
    if best is None:
        return {"value": None, "unit": "tokens/s", "cores": 0, "kind": kind, "sample": "failed"}
    sample_end = min(seq, PROMPT + (32 if spec.n_embd >= 1024 else 64))
    r = _cpu_run(path, spec, seq, sample_end, kind, flavour, best[1], best[2], runs)
    v = float(np.median(r)) if r else best[0]
    return {"value": v, "unit": "tokens/s", "cores": best[1], "kind": kind,
            "sample": f"{workload}: prompt {PROMPT} + decode positions {PROMPT - 1}..{sample_end - 2} ({sample_end - PROMPT} tokens) of the seq-{seq} run; "
                      f"OMP_NUM_THREADS={best[1]}{' OMP_PROC_BIND=true OMP_WAIT_POLICY=active' if best[2] else ''} = best of the sweep {table}; "
                      f"host has {ncpu} logical cores; build {flavour or 'oracle port -O2 strict'}"}


def run_reference_arm(args, workload):
    """--impl reference: the unmodified reference CPU engine on the SAME workload: every step is one full prompt + decode run
    (tokens PROMPT..seq-1 timed), at the best thread setting of the BASELINE.md section-3 sweep; value = median over the K steps."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    preset, quant, gs, seq = WORKLOADS[workload]
    spec = mf.PRESETS[preset]
    path = model_path(workload)
    t_all = time.time()
    kind, flavour, best, table, ncpu, _ = cpu_sweep(path, spec, seq, budget_s=40.0)
    vals, sample_end = [], seq
    if best is not None:
        # bounded: if a full run would take more than ~12 s, time the first 128 decode positions of the same run instead
        full_s = (seq - PROMPT) / best[0]
        sample_end = seq if full_s <= 12.0 else min(seq, PROMPT + 128)
        r = _cpu_run(path, spec, seq, sample_end, kind, flavour, best[1], best[2], args.warmup + args.steps, timeout=1500)
        vals = r[args.warmup:]
    v = float(np.median(vals)) if vals else None
    cb = {"value": v, "unit": "tokens/s", "cores": best[1] if best else 0, "kind": kind,
          "sample": (f"{workload}: {args.steps} timed runs (after {args.warmup} warm-up runs) of prompt {PROMPT} + decode positions {PROMPT - 1}..{sample_end - 2}; median; "
                     f"OMP_NUM_THREADS={best[1]}{' OMP_PROC_BIND=true OMP_WAIT_POLICY=active' if best[2] else ''} = best of the sweep {table}; "
                     f"host has {ncpu} logical cores; build {flavour or 'oracle port -O2 strict'}") if best else "failed"}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": (time.time() - t_all) * 1e3 / max(1, args.steps + args.warmup),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[quant], "data": "synthetic",
            "config": workload_config(workload),
            "run": {"mode": "reference CPU engine (oracle/_ref: the unmodified infer/*.c at the Makefile's flags; the oracle port if absent)", "all_runs_tok_s": [round(x, 1) for x in vals]},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
def dist_setup(n, backend=None):
    """One process per GPU (torchrun); NCCL when CUDA is present, gloo otherwise (CPU tests of the host logic)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch
        import torch.distributed as dist
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
        return rank, world, local, dist
    return rank, world, local, None


def barrier_max(dist, local, value):
    """barrier + max over ranks of a float (the timing rule: a multi-GPU time is the max over ranks)."""
    if dist is None:
        return value
    import torch
    dev = f"cuda:{local}" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def aggregate_tokens_per_s(world, steps, tokens_per_step, ms_per_rank_max):
    """Whole-job throughput of `world` independent batch-1 replicas: all ranks' tokens over the slowest rank's time."""
    return world * steps * tokens_per_step / (ms_per_rank_max * 1e-3)


def parity_check(eng_ids, path, spec, seq, n_check=64):
    """Feed the oracle the ids of the timed run; at each of the first `n_check` decode positions compare its greedy choice
    with the id the GPU run produced.  Fast mode may legitimately differ where the oracle's own top-1/top-2 margin is inside
    fast-mode noise, so the margin at the first divergence is reported."""
    from oracle import bindings as ob
    o = ob.NanoOracle(path, seq)
    ob.NanoOracle.lib().nor_set_threads(min(32, os.cpu_count() or 1))
    first, margin_at, agree, min_margin = None, None, 0, None
    end = min(seq - 1, PROMPT - 1 + n_check)
    for pos in range(end):
        lg = o.forward(int(eng_ids[pos]), pos)
        if pos < PROMPT - 1:
            continue
        top2 = np.partition(lg, -2)[-2:]
        m = float(top2[1] - top2[0])
        min_margin = m if min_margin is None else min(min_margin, m)
        if int(np.argmax(lg)) == int(eng_ids[pos + 1]):
            agree += 1
        elif first is None:
            first, margin_at = pos + 1, m
    o.close()
    return {"checked_decode_positions": end - (PROMPT - 1), "agree": agree, "first_divergence": first, "oracle_margin_at_divergence": margin_at,
            "min_oracle_margin": min_margin, "oracle": "oracle/nano_oracle.c (bit-identical to the strict reference), teacher-forced with the timed run's ids"}


def measure(E, workload, steps, warmup, local, dist=None, world=1, flags=0, e2e=True, parity=True, per_kernel=True):
    """One workload on this rank's GPU: device-loop tok/s, e2e tok/s, roofline, parity."""
    preset, quant, gs, seq = WORKLOADS[workload]
    spec = mf.PRESETS[preset]
    path = model_path(workload)
    eng = E.Engine(path, seq, device=local, flags=flags)
    n_dec = seq - PROMPT
    for _ in range(warmup):
        ids = prompt_ids(spec, seq)
        eng.decode_greedy(ids, PROMPT, seq)
    barrier_max(dist, local, 0.0)
    launches0 = eng.launches
    t0 = time.perf_counter()
    dec_ms = 0.0
    for _ in range(steps):
        ids = prompt_ids(spec, seq)
        _pre, dec = eng.decode_greedy(ids, PROMPT, seq)
        dec_ms += dec
    wall = time.perf_counter() - t0
    launches = eng.launches - launches0
    dec_ms = barrier_max(dist, local, dec_ms)
    wall = barrier_max(dist, local, wall)
    value = aggregate_tokens_per_s(world, steps, n_dec, dec_ms)
    timed_ids = ids.copy()
    res = {"value": value, "ms_per_step": wall * 1e3 / steps, "gpu_launches": int(launches), "launches_per_token": eng.launches_per_token,
           "engine": eng.path, "path_calibration": eng.calibration, "dec_ms": dec_ms, "ids": timed_ids[:seq]}

    if e2e:
        e2e_steps = max(1, min(steps, 2))
        t_e2e = 0.0
        for _ in range(e2e_steps):
            ids2 = prompt_ids(spec, seq)
            for pos in range(PROMPT - 1):
                ids2[pos + 1] = eng.next_greedy(ids2, pos, 1)
            t1 = time.perf_counter()
            for pos in range(PROMPT - 1, seq - 1):
                ids2[pos + 1] = eng.next_greedy(ids2, pos, 0)
            t_e2e += time.perf_counter() - t1
        t_e2e = barrier_max(dist, local, t_e2e)
        res["e2e"] = {"value": world * e2e_steps * n_dec / t_e2e, "unit": "tokens/s", "h2d_bytes_per_step": 48 * n_dec, "d2h_bytes_per_step": 4 * n_dec,
                      "api": "nb200_next_greedy per token (pinned H2D of the 48 B step descriptor incl. token id, D2H of the next id)",
                      "same_ids_as_device_loop": bool(np.array_equal(ids2[:seq], timed_ids[:seq]))}

    # ---- roofline ----
    peak, peak_src = peaks()
    E_, F_, Q_, K_ = spec.n_embd, spec.n_hidden, spec.q_dim, spec.kv_dim
    bpw = BPW[quant](gs)
    avg_pos = (PROMPT + seq - 1) / 2.0
    bytes_tok = spec.bytes_per_token(quant, gs, avg_pos)
    per_gpu_gbs = bytes_tok * (value / world) / 1e9
    res["token_roofline"] = {"alg_bytes_per_token": bytes_tok, "achieved_gbs_per_gpu": per_gpu_gbs, "frac_of_peak": per_gpu_gbs / peak,
                             "roofline_tok_s_per_session": peak * 1e9 / bytes_tok}
    per_class = {}
    if per_kernel:
        nprof = min(64, seq - 1 - PROMPT)
        start = max(PROMPT, (seq // 2) - nprof // 2)
        eng.profile_tokens(timed_ids, start, 4)                        # warm
        ms, cnt = eng.profile_tokens(timed_ids, start, nprof)
        mid = start + nprof / 2.0
        alg = {"qkv": (Q_ + 2 * K_) * E_ * bpw + 4 * E_ + 4 * K_,
               "attention": 8 * K_ * (mid + 1) + 4 * K_ + (8 * spec.hd if spec.arch == mf.ARCH_QWEN3 else 0),
               "o_proj": E_ * Q_ * bpw, "w13_swiglu": 2 * F_ * E_ * bpw + 4 * E_, "w2": E_ * F_ * bpw,
               "classifier": spec.vocab * E_ * bpw + 4 * E_, "embed": 4 * E_}
        tot_ms = float(ms.sum())
        for i, name in enumerate(CLASS_NAMES):
            if cnt[i]:
                dur = float(ms[i]) / int(cnt[i]) * 1e-3
                per_class[name] = {"launches": int(cnt[i]), "mean_us": dur * 1e6, "share": float(ms[i]) / tot_ms, "alg_bytes": alg[name], "gbs": alg[name] / dur / 1e9}
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json"))).get(workload + (":stream" if eng.path.startswith("streaming") else ":multikernel"))
    except Exception:
        pass
    if eng.path.startswith("streaming"):
        # the step IS one kernel: a launch decodes n_dec tokens, so the dominant kernel's roofline is the token roofline
        res["roofline"] = {"bound": "hbm", "kernel": f"k_decode_stream (one launch decodes {n_dec} tokens: all layers + classifier + argmax)",
                           "achieved": per_gpu_gbs, "peak": peak, "unit": "GB/s", "frac": per_gpu_gbs / peak,
                           "traffic": traffic * n_dec if traffic else None,
                           "traffic_source": f"ncu --set full capture of one k_decode_stream launch: DRAM bytes per token x {n_dec} tokens (profiles/r2_ncu_stream.md)" if traffic else None,
                           "peak_source": peak_src, "alg_bytes_per_launch": bytes_tok * n_dec, "mean_launch_us": dec_ms / steps * 1e3, "share_of_step": 1.0,
                           "phase_profile_note": "per_kernel = the multi-kernel path's kernels for the same phases (graph/PDL off, CUDA events per launch), for orientation only",
                           "per_kernel": per_class}
    elif per_class:
        dom = "w13_swiglu"
        res["roofline"] = {"bound": "hbm", "kernel": f"k_matvec<{'Q80' if quant == mf.QUANT_Q80 else 'Q4K' if quant == mf.QUANT_Q4K else 'F32'},SWIGLU> (W1|W3 + SwiGLU)",
                           "achieved": per_class[dom]["gbs"], "peak": peak, "unit": "GB/s", "frac": per_class[dom]["gbs"] / peak,
                           "traffic": traffic, "traffic_source": "ncu --set full capture (profiles/r2_ncu_multikernel.md)" if traffic else None,
                           "peak_source": peak_src, "alg_bytes_per_launch": per_class[dom]["alg_bytes"], "mean_launch_us": per_class[dom]["mean_us"],
                           "share_of_step": per_class[dom]["share"], "per_kernel": per_class}
    if parity:
        try:
            res["parity"] = parity_check(timed_ids, path, spec, seq)
        except Exception as ex:        # the oracle is test infrastructure: its absence must not break the measurement
            res["parity"] = {"error": str(ex)}
    eng.close()
    return res


def tp_block(E, rank, world, local, dist):
    """BASELINE config 5: one Qwen3-4B Q80 session at seq 4096, row-sharded over the `world` GPUs, and the same (multi-kernel)
    path on one GPU in the same job.  Every rank takes part in the sharded run; rank 0 alone runs the one-GPU point."""
    preset, quant, gs, seq = WORKLOADS[TP_WORKLOAD]
    spec = mf.PRESETS[preset]
    if rank == 0:
        model_path(TP_WORKLOAD)
    dist.barrier()
    path = model_path(TP_WORKLOAD)
    n_dec = seq - PROMPT
    eng = E.Engine(path, seq, device=local, tp=(rank, world))
    handles = [None] * world
    dist.all_gather_object(handles, eng.tp_export())
    eng.tp_attach_ipc(handles)
    dist.barrier()
    ids = prompt_ids(spec, seq)
    eng.decode_greedy(ids, PROMPT, seq)                     # warm-up
    barrier_max(dist, local, 0.0)
    ids = prompt_ids(spec, seq)
    _pre, dec = eng.decode_greedy(ids, PROMPT, seq)
    dec = barrier_max(dist, local, dec)
    tp_ids = ids.copy()
    eng.close()
    dist.barrier()
    out = None
    if rank == 0:
        one = E.Engine(path, seq, device=local, flags=E.FLAG_NO_STREAM)
        ids1 = prompt_ids(spec, seq)
        one.decode_greedy(ids1, PROMPT, seq)
        ids1 = prompt_ids(spec, seq)
        _p1, dec1 = one.decode_greedy(ids1, PROMPT, seq)
        path1 = one.path
        one.close()
        dflt = E.Engine(path, seq, device=local)               # the one-GPU engine a user gets by default (path chosen by calibration)
        ids2 = prompt_ids(spec, seq)
        dflt.decode_greedy(ids2, PROMPT, seq)
        ids2 = prompt_ids(spec, seq)
        _p2, dec2 = dflt.decode_greedy(ids2, PROMPT, seq)
        path2, calib2 = dflt.path, dflt.calibration
        dflt.close()
        tp_tok, one_tok = n_dec / (dec * 1e-3), n_dec / (dec1 * 1e-3)
        nx = 4 * spec.n_layer + 1
        out = {"workload": workload_config(TP_WORKLOAD)["workload"], "n_gpus": world, "scaling": "strong",
               "parallelism": f"tp{world}: one batch-1 session; every weight matrix row-sharded over {world} GPUs (QKV and the KV cache by kv head); "
                              f"{nx} activation exchanges per token pushed into every rank's copy through NVLink peer memory from inside the kernels (no NCCL on the data path)",
               "value": tp_tok, "unit": "tokens/s", "one_gpu_same_path": one_tok, "one_gpu_engine": path1, "speedup_vs_one_gpu": tp_tok / one_tok,
               "one_gpu_default": {"value": n_dec / (dec2 * 1e-3), "engine": path2, "path_calibration": calib2},
               "exchanges_per_token": nx,
               "per_exchange_us_model": ((dec / n_dec) - (dec1 / n_dec) / world) * 1e3 / nx,
               "per_exchange_note": "(ms/token at tp - ms/token on one GPU / N) / exchanges: what an exchange costs beyond perfectly divided streaming time",
               "ids_identical_to_one_gpu": bool(np.array_equal(tp_ids[:seq], ids1[:seq]))}
    dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (each one full prompt + greedy decode run)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="nano-168m-q80", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="replicas", choices=["replicas", "tp"],
                    help="replicas: one independent batch-1 session per GPU (weak scaling, the default the driver runs; a `tp` block is added for N > 1); "
                         "tp: only the tensor-parallel block (ONE session sharded over the GPUs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra configs / exact-mode / tp blocks (quick runs)")
    ap.add_argument("--exact", action="store_true", help="run the engine in exact (reference-order) mode")
    ap.add_argument("--no-pdl", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-stream", action="store_true", help="forbid the streaming kernel")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last step (the token ids of the greedy decode) as DIR/ids.npy, "
                         "float64; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "replicas"):
        ap.error("--dump-outputs writes the outputs of the default path (--impl b200 --mode replicas) only")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    preset, quant, gs, seq = WORKLOADS[args.workload]
    spec = mf.PRESETS[preset]
    if args.impl == "reference":
        run_reference_arm(args, args.workload)
        return

    from nano_b200 import engine as E
    rank, world, local, dist = dist_setup(args.gpus)
    if rank == 0 or int(os.environ.get("LOCAL_WORLD_SIZE", "1")) == 1:
        model_path(args.workload)
    if dist is not None:
        dist.barrier()
    flags = (E.FLAG_EXACT if args.exact else 0) | (E.FLAG_NO_PDL if args.no_pdl else 0) | (E.FLAG_NO_GRAPH if args.no_graph else 0) | (E.FLAG_NO_STREAM if args.no_stream else 0)

    if args.mode == "tp" and world > 1:
        tp = tp_block(E, rank, world, local, dist)
        if rank == 0:
            line = {"metric": METRIC, "value": tp["value"], "unit": "tokens/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": None,
                    "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE[mf.QUANT_Q80], "data": "synthetic",
                    "config": workload_config(TP_WORKLOAD), "tp": tp}
            print(json.dumps(line))
        dist.destroy_process_group()
        return

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    res = measure(E, args.workload, args.steps, args.warmup, local, dist, world, flags, parity=(rank == 0))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "ids.npy"), res["ids"].astype(np.float64))

    tp = None
    if world > 1 and not args.no_extra:
        try:
            tp = tp_block(E, rank, world, local, dist)
        except Exception as ex:
            tp = {"error": str(ex)}
    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return

    extra, exact = None, None
    if world == 1 and not args.no_extra and not args.exact:
        try:
            r = measure(E, args.workload, 1, 1, local, flags=flags | E.FLAG_EXACT, e2e=False, parity=False, per_kernel=False)
            exact = {"value": r["value"], "unit": "tokens/s", "engine": r["engine"],
                     "note": "NB200_FLAG_EXACT: reference-order fp32 reductions + glibc-equivalent expf; logits, KV rows and greedy ids bit-identical to the strict reference (tests)"}
        except Exception as ex:
            exact = {"error": str(ex)}
        extra = {}
        for w in EXTRA_CONFIGS:
            if w == args.workload:
                continue
            try:
                r = measure(E, w, 2, 1, local, flags=flags)
                extra[w] = {"config": workload_config(w), "value": r["value"], "unit": "tokens/s", "e2e": r.get("e2e"), "engine": r["engine"], "path_calibration": r.get("path_calibration"),
                            "gpu_launches": r["gpu_launches"], "roofline": {k: v for k, v in (r.get("roofline") or {}).items() if k != "per_kernel"},
                            "token_roofline": r["token_roofline"], "parity": r.get("parity"), "dtype": DTYPE[WORKLOADS[w][1]]}
            except Exception as ex:
                extra[w] = {"error": str(ex)}

    cb = None
    if not args.no_cpu_baseline and world == 1:
        cb = cpu_baseline(args.workload, model_path(args.workload), spec, seq)

    line = {
        "metric": METRIC, "value": res["value"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE[quant], "data": "synthetic",
        "config": workload_config(args.workload),
        "run": {"parallelism": f"{world} independent batch-1 session(s), one per GPU, no data-path collective", "mode": "exact" if args.exact else "fast",
                "engine": res["engine"], "path_calibration": res.get("path_calibration"),
                "value_path": "device-resident greedy loop (nb200_decode_greedy); the drop-in per-token number is e2e"},
        "clocks": clocks, "e2e": res.get("e2e"), "gpu_launches": res["gpu_launches"], "launches_per_token": res["launches_per_token"],
        "roofline": res.get("roofline"), "token_roofline": res["token_roofline"], "parity": res.get("parity"),
        "exact_mode": exact, "configs": extra, "tp": tp, "cpu_baseline": cb,
    }
    print(json.dumps(line))
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
