#!/usr/bin/env python
"""bench.py -- streaming Whisper on B200 behind WhisperLiveKit's AlignAtt seam.

Headline config (`--config alignatt-large-v3`, the default; BASELINE.json's metric): Whisper large-v3, 0.5 s
chunks, 30 s rolling window fully re-encoded per chunk (the reference's parity mode), B concurrent streams per GPU.

One "step" = one 0.5 s tick of the hot path for every stream of the job, AlignAtt-style:
    append 0.5 s of PCM (host -> device) and drop the oldest 0.5 s of the full 30 s window,
    log-mel -> 32-layer encoder over all 1500 positions -> cross-K/V for 32 decoder layers,
    decoder prefill of a PREFIX-token prompt, then STEPS_PER_CHUNK greedy iterations of
    (suppress -> argmax/logprob -> alignment-head reduction -> most attended frame -> 1-token decode).

Numbers in the one JSON line:
  value       audio seconds processed per wall second with the windows resident in HBM (scripted tick above,
              CUDA events on the engine stream) = concurrent real-time streams the GPU sustains.
  e2e         THROUGH THE SEAM, REAL-TIME PACED: B `StreamingAlignAtt` policies (the token-id mirror of
              AlignAttBase.infer, whisperlivekit_b200/alignatt.py) on B caller threads over `BatchingEngine`, each
              fed one 0.5 s host chunk every 0.5 s of wall clock at its own phase; the policy decides prefix and step
              count; value = the largest probed B for which p95 latency (chunk arrival -> infer() returns) < 0.5 s
              and the backlog does not grow.  Host->device chunk copies and device->host results are inside.
  roofline    encoder GEMM class: algorithmic FLOPs / CUDA-event time inside the timed run vs the measured peak.
  exact_mode  the same scripted tick in WLK_PREC_BF16X3 (1e-3-on-logits mode): the price of exactness.
  other_configs  BASELINE configs 2, 3, 4 (per-GPU share: 64 streams + Sortformer), 5 in brief (each also the main line with --config).
  incremental_mode  the LABELLED APPROXIMATE incremental encoder: streams per GPU and agreement with the parity mode (also --config
              alignatt-large-v3-incremental as the main line).
  cpu_baseline / --impl reference: the STAGED UNMODIFIED reference (oracle/_ref: vendored torch Whisper behind its own
              AlignAtt hooks) on the host cores, same per-chunk workload (oracle/ref_driver.py).

--dump-outputs DIR (headline config, rank 0): what the last timed tick returned to its caller, as float32 / float64 .npy
files -- content frames per stream, no-speech probability, token / logprob / attended frame of every decode iteration --
and the logits its last decode left for the next one (the first streams' rows, up to 32 MB).  Weights, audio and prompts
are seeded, so two builds run with the same arguments can be compared output for output, with a tolerance: the bf16
path is not bit-reproducible (two runs of one build on a B200 at 1000 W: tokens identical, logits within 0.04).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--config C] [--streams B] [--no-extras]
                    [--dump-outputs DIR]
Multi-GPU: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...  (one rank per GPU; sessions are
sharded, NCCL is used once to broadcast the packed weights; weak scaling, no data-path collective).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

CHUNK_S = 0.5
CHUNK = 8000
WINDOW = 480000
PREFIX = int(os.environ.get("WLK_BENCH_PREFIX", "48"))            # the headline workload: 48 + 8 (overrides are for experiments)
STEPS_PER_CHUNK = int(os.environ.get("WLK_BENCH_STEPS", "8"))
UNIT = "concurrent real-time streams (audio-s per wall-s)"
CONFIGS = ["alignatt-large-v3", "alignatt-base-en-1stream", "localagreement-large-v3-64", "alignatt-large-v3-sortformer-64",
           "qwen-tower-128", "alignatt-large-v3-incremental"]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_tflops=d.get("bf16_tflops_sustained") or d.get("bf16_tflops"), hbm_gbs=d.get("hbm_gbs"),
                    source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(bf16_tflops=1400.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(self.rows))


# ------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the staged, unmodified reference on the host cores (oracle/ref_driver.py)
# ------------------------------------------------------------------------------------------
def reference_available() -> bool:
    from oracle import stage_reference
    return stage_reference.staged()


def cpu_baseline_leg(dims, sd, heads, n_chunks=2):
    """One stream, all host threads, `n_chunks` stream-chunks of the headline workload.  -> dict"""
    from oracle import ref_driver as rd
    cores = rd.default_threads()
    if reference_available():
        model = rd.build_model(dims, sd, heads)
        per, threads = rd.time_single_stream(model, dims, PREFIX, STEPS_PER_CHUNK, n_chunks, cores, warmup=0)
        kind, what = "reference", "staged unmodified reference (oracle/_ref): its AlignAtt hooks over its vendored torch Whisper, fp32"
    else:                                                     # the recipe could not run (no /root/reference at build time)
        import torch
        torch.set_num_threads(cores)
        per, threads = oracle_port_chunks(dims, sd, heads, n_chunks), torch.get_num_threads()
        kind, what = "port", "oracle port of the reference CPU path (oracle/_ref not staged)"
    sec = float(np.mean(per))
    return dict(value=CHUNK_S / sec, unit=UNIT, cores=threads, kind=kind, cpu_model=rd.cpu_model(), nproc=os.cpu_count(),
                cpu_quota=rd.cpu_quota(), sample=f"{n_chunks} stream-chunks of the same workload, 1 stream, {threads} threads; {what}",
                seconds_per_stream_chunk=sec)


def oracle_port_chunks(dims, sd, heads, n_chunks):
    from oracle import whisper_oracle as wo
    from whisperlivekit_b200.weights import synthetic_audio
    eng = wo.OracleEngine(dims, sd, heads)
    sid = eng.open_session()
    eng.append_audio(sid, synthetic_audio(30.0, seed=1))
    prefix = list(eng.specials.sot_sequence_including_notimestamps()) + list(range(1000, 1000 + PREFIX - 4))
    sup = eng.specials.alignatt_suppress_tokens()
    per = []
    for c in range(n_chunks):
        t0 = time.perf_counter()
        eng.drop_audio(sid, CHUNK)
        eng.append_audio(sid, synthetic_audio(CHUNK_S, seed=100 + c))
        eng.encode([sid])
        eng.decode([sid], [prefix])
        for _ in range(STEPS_PER_CHUNK):
            eng.suppress([sid], sup)
            tok, _, _ = eng.greedy_and_align([sid])[0]
            eng.decode([sid], [[tok]])
        per.append(time.perf_counter() - t0)
    return per


def reference_arm(args, dims, heads, metric, workload):
    """bench.py --impl reference: rank 0 only.  Two figures (BASELINE.md section 4): (ii) `cores` single-thread
    streams in parallel, then (i) one stream on all cores; `value` is the better of the two (CPU throughput)."""
    from oracle import ref_driver as rd
    from whisperlivekit_b200.weights import synthetic_state_dict
    import torch
    torch.set_num_threads(1)                                  # nothing multi-threaded before the fork of figure (ii)
    cores = rd.default_threads()                              # torch's own default here, torchrun's OMP_NUM_THREADS=1 ignored
    sd = synthetic_state_dict(dims, seed=0)
    if not reference_available():
        per = oracle_port_chunks(dims, sd, heads, 1)
        torch.set_num_threads(cores)
        per = oracle_port_chunks(dims, sd, heads, max(1, min(args.steps, 3)))
        sec = float(np.mean(per))
        base = dict(value=CHUNK_S / sec, unit=UNIT, cores=torch.get_num_threads(), kind="port",
                    sample="oracle port (oracle/_ref not staged)")
        fig_i, fig_ii = base, None
    else:
        model = rd.build_model(dims, sd, heads)
        del sd
        procs = cores
        budget = float(os.environ.get("WLK_REF_PARALLEL_TIMEOUT", "240"))
        wall, done = rd.time_parallel_single_thread(model, dims, PREFIX, STEPS_PER_CHUNK, procs, timeout_s=budget)
        fig_ii = dict(procs=procs, finished=done, wall_s=wall,
                      value=(done * CHUNK_S / wall) if done == procs else 0.0,
                      note=("every process ran one stream-chunk at 1 thread" if done == procs else
                            f"only {done}/{procs} single-thread stream-chunks finished within {budget:.0f} s: below "
                            f"{procs * CHUNK_S / budget:.3f} streams"))
        n = max(1, min(args.steps, 3))
        per, threads = rd.time_single_stream(model, dims, PREFIX, STEPS_PER_CHUNK, n, cores, warmup=1)
        sec = float(np.mean(per))
        fig_i = dict(value=CHUNK_S / sec, unit=UNIT, cores=threads, kind="reference", seconds_per_stream_chunk=sec,
                     sample=f"{n} stream-chunks, 1 stream on {threads} threads")
    value = max(fig_i["value"], fig_ii["value"] if fig_ii else 0.0)
    best = "one stream on all cores" if value == fig_i["value"] else f"{fig_ii['procs']} single-thread streams in parallel"
    line = dict(metric=metric, value=value, unit=UNIT, n_gpus=args.gpus, steps=max(1, min(args.steps, 3)), warmup=1,
                ms_per_step=CHUNK_S / value * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=workload.replace(f"{args.streams} streams/GPU", "host CPU"), model=args.model,
                            note="staged unmodified reference (oracle/_ref), `--backend whisper` path: its own AlignAtt hooks over "
                                 "its vendored torch Whisper, fp32, scripted to the same per-chunk work as the B200 arm"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind=fig_i.get("kind", "reference"),
                                  cpu_model=rd.cpu_model(), nproc=os.cpu_count(), cpu_quota=rd.cpu_quota(),
                                  omp_env=os.environ.get("OMP_NUM_THREADS"),
                                  sample=f"better of two figures ({best}); each step is one stream-chunk of the workload",
                                  one_stream_all_cores=fig_i, parallel_single_thread=fig_ii),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# through-the-seam, real-time paced load (e2e)
# ------------------------------------------------------------------------------------------
def _seam_policies(eng_like, eng, B, rng, context_tokens):
    """B policies mid-conversation: a full 30 s window, ~4 hypothesis tokens per second of window and `context_tokens` of
    left context (a long stream saturates the reference's context at n_text_ctx - 20 tokens, align_att_base.py:100-113)."""
    from whisperlivekit_b200.alignatt import AlignAttConfig, StreamingAlignAtt
    from whisperlivekit_b200.weights import synthetic_audio
    base = synthetic_audio(36.0, seed=7)
    pols = []
    for _ in range(B):
        p = StreamingAlignAtt(eng_like, AlignAttConfig(nonspeech_prob=1.01))     # the no-speech exit would hide the decode loop on random weights
        off = int(rng.integers(0, 16000 * 5))
        p.segments = [CHUNK] * (WINDOW // CHUNK)
        eng.append_audio(p.sid, base[off: off + WINDOW])
        p.tokens = [list(p.initial_tokens)] + [[int(t) for t in rng.integers(1000, 40000, 2)] for _ in range(WINDOW // CHUNK - 1)]
        p.context = [int(t) for t in rng.integers(1000, 40000, context_tokens)]
        pols.append(p)
    return pols


def _seam_summary(B, mode, n_ticks, warm_ticks, lat, lag, aborted, errors, stats, wall, extra):
    L = lat[:, warm_ticks:].reshape(-1)
    G = lag[:, warm_ticks:]
    third = max(1, n_ticks // 3)
    lag_first, lag_last = float(G[:, :third].mean()), float(G[:, -third:].mean())
    p95 = float(np.percentile(L, 95))
    ok = (not errors) and (not aborted) and p95 < CHUNK_S and lag_last < 0.1 + lag_first and float(G[:, -1].max()) < CHUNK_S
    out = dict(streams=B, ok=bool(ok), aborted=bool(aborted), mode=mode, ticks=n_ticks, p50_latency_s=float(np.percentile(L, 50)),
               p95_latency_s=p95, max_latency_s=float(L.max()), start_lag_first_third_s=lag_first,
               start_lag_last_third_s=lag_last, wall_s=wall, errors=errors[:3],
               mean_prefix_tokens=float(np.mean(stats["prefix"])) if stats["prefix"] else 0.0,
               mean_decode_iterations=float(np.mean(stats["iters"])) if stats["iters"] else 0.0, stops=stats["stops"])
    out.update(extra)
    return out


def seam_probe(eng, B, n_ticks, warm_ticks, rng, mode="cohort", context_tokens=300):
    """Real-time paced load through the policy seam: stream i's chunk k ARRIVES (host buffer) at t0 + phase_i + k * 0.5 s,
    phases spread uniformly over the chunk period; latency = arrival -> infer() returned.
    mode "cohort":  one scheduler thread; the streams whose chunk has arrived form a cohort, `cohort.CohortRunner` advances
                    their policies in lockstep, every round one batched engine call (no thread per stream).
    mode "threads": one OS thread per stream calling the blocking per-session API through `batching.BatchingEngine`
                    (WhisperLiveKit's own calling convention, audio_processor.py:543-551).
    -> dict(ok, p50/p95/max latency, start lag, policy statistics)"""
    if mode == "threads":
        return seam_probe_threads(eng, B, n_ticks, warm_ticks, rng, context_tokens)
    if mode == "continuous":
        return seam_probe_continuous(eng, B, n_ticks, warm_ticks, rng, context_tokens)
    from whisperlivekit_b200.cohort import CohortRunner
    pols = _seam_policies(eng, eng, B, rng, context_tokens)
    runner = CohortRunner(eng, max_batch=eng.max_batch)
    chunks = (0.05 * rng.standard_normal((8, CHUNK))).astype(np.float32)
    phases = np.arange(B) / B * CHUNK_S
    total = warm_ticks + n_ticks
    lat = np.full((B, total), 10.0); lag = np.full((B, total), 10.0)
    nxt = np.zeros(B, np.int64)                                              # next chunk index of every stream
    stats = dict(prefix=[], iters=[], stops={})
    errors, aborted = [], False
    t_start = time.perf_counter() + 0.2
    try:
        while (nxt < total).any():
            now = time.perf_counter()
            arrival = t_start + phases + nxt * CHUNK_S
            due = np.nonzero((nxt < total) & (arrival <= now))[0]
            if len(due) == 0:
                time.sleep(max(0.0, float(arrival[nxt < total].min() - now)))
                continue
            t0 = time.perf_counter()
            if (nxt[due] >= warm_ticks).any() and float((t0 - arrival[due]).max()) > 2.0:
                aborted = True                                               # the backlog ran away: this B has failed
                break
            for i in due:
                pols[i].insert_audio(chunks[(i + nxt[i]) % 8])               # H2D of the chunk + window slide
            traces = runner.run([pols[i] for i in due])
            t1 = time.perf_counter()
            for i, tr in zip(due, traces):
                k = nxt[i]
                lat[i, k] = t1 - arrival[i]; lag[i, k] = t0 - arrival[i]
                if k >= warm_ticks:
                    stats["prefix"].append(tr.prefix_len); stats["iters"].append(len(tr.step_tokens))
                    stats["stops"][tr.stop] = stats["stops"].get(tr.stop, 0) + 1
                nxt[i] += 1
    except Exception as e:                                                   # noqa: BLE001
        errors.append(repr(e))
    wall = time.perf_counter() - t_start
    rs = runner.stats
    for p in pols:
        p.close()
    return _seam_summary(B, "cohort", n_ticks, warm_ticks, lat, lag, aborted, errors, stats, wall,
                         dict(engine_calls=rs["calls"], mean_sessions_per_call=rs["sessions"] / max(1, rs["calls"]),
                              cohorts=rs["cohorts"], mean_cohort=rs["cohort_sessions"] / max(1, rs["cohorts"])))


ADMIT_WAIT_S = float(os.environ.get("WLK_ADMIT_WAIT_S", "0.06"))


def seam_probe_continuous(eng, B, n_ticks, warm_ticks, rng, context_tokens=300):
    """Same load as the cohort mode, scheduled with continuous batching (cohort.CohortRunner.admit / round): streams whose
    chunk has arrived are admitted BETWEEN rounds, their encode / prefill is served next, and they then share the token-step
    rounds of the streams already running, instead of waiting for the running cohort to finish all of its rounds."""
    from whisperlivekit_b200.cohort import CohortRunner
    pols = _seam_policies(eng, eng, B, rng, context_tokens)
    runner = CohortRunner(eng, max_batch=eng.max_batch)
    chunks = (0.05 * rng.standard_normal((8, CHUNK))).astype(np.float32)
    phases = np.arange(B) / B * CHUNK_S
    total = warm_ticks + n_ticks
    lat = np.full((B, total), 10.0); lag = np.full((B, total), 10.0)
    nxt = np.zeros(B, np.int64)
    flying = np.zeros(B, bool)
    started = np.zeros(B)
    stats = dict(prefix=[], iters=[], stops={})
    errors, aborted = [], False
    t_start = time.perf_counter() + 0.2

    def finish(i, tr, t1):
        k = nxt[i]
        arrival = t_start + phases[i] + k * CHUNK_S
        lat[i, k] = t1 - arrival; lag[i, k] = started[i] - arrival
        if k >= warm_ticks:
            stats["prefix"].append(tr.prefix_len); stats["iters"].append(len(tr.step_tokens))
            stats["stops"][tr.stop] = stats["stops"].get(tr.stop, 0) + 1
        nxt[i] += 1; flying[i] = False

    try:
        while (nxt < total).any():
            now = time.perf_counter()
            arrival = t_start + phases + nxt * CHUNK_S
            idle = (~flying) & (nxt < total)
            due = np.nonzero(idle & (arrival <= now))[0]
            # admission: an encoder batch of one or two streams wastes the tensor cores, so arrivals wait until the engine is
            # idle, or enough of them have gathered, or the oldest has waited ADMIT_WAIT_S
            if len(due) and runner.busy() and len(due) < max(4, B // 8) and float((now - arrival[due]).max()) < ADMIT_WAIT_S:
                due = due[:0]
            if len(due):
                if (nxt[due] >= warm_ticks).any() and float((now - arrival[due]).max()) > 2.0:
                    aborted = True
                    break
                for i in due:
                    pols[i].insert_audio(chunks[(i + nxt[i]) % 8])
                    started[i] = now; flying[i] = True
                for i, tr in runner.admit_many([(int(i), pols[i]) for i in due]):
                    finish(i, tr, time.perf_counter())
            if runner.busy():
                done = runner.round()
                t1 = time.perf_counter()
                for i, tr in done:
                    finish(i, tr, t1)
            elif not len(due):
                time.sleep(max(0.0, float(arrival[idle].min() - now)))
    except Exception as e:                                                   # noqa: BLE001
        errors.append(repr(e))
    wall = time.perf_counter() - t_start
    rs = runner.stats
    for p in pols:
        p.close()
    return _seam_summary(B, "continuous", n_ticks, warm_ticks, lat, lag, aborted, errors, stats, wall,
                         dict(engine_calls=rs["calls"], mean_sessions_per_call=rs["sessions"] / max(1, rs["calls"]),
                              cohorts=rs["cohorts"], mean_cohort=rs["cohort_sessions"] / max(1, rs["cohorts"])))


def seam_probe_threads(eng, B, n_ticks, warm_ticks, rng, context_tokens=300):
    from whisperlivekit_b200.batching import BatchingEngine
    beng = BatchingEngine(eng, max_batch=eng.max_batch, max_wait_s=0.004)
    pols = _seam_policies(beng, eng, B, rng, context_tokens)
    chunks = (0.05 * rng.standard_normal((8, CHUNK))).astype(np.float32)
    phases = np.arange(B) / B * CHUNK_S
    total = warm_ticks + n_ticks
    lat = np.full((B, total), 10.0); lag = np.full((B, total), 10.0)
    stats = dict(prefix=[], iters=[], stops={})
    slock = threading.Lock()
    errors = []
    abort = threading.Event()                                                # the backlog ran away: the probe has failed
    t_start = time.perf_counter() + 0.3

    def worker(i):
        p, ph = pols[i], phases[i]
        try:
            for k in range(total):
                if abort.is_set():
                    return
                due = t_start + ph + k * CHUNK_S
                now = time.perf_counter()
                if now < due:
                    time.sleep(due - now)
                t0 = time.perf_counter()
                if k >= warm_ticks and t0 - due > 2.0:
                    abort.set()
                    return
                p.insert_audio(chunks[(i + k) % 8])                      # H2D of the chunk + window slide
                tr = p.infer()
                t1 = time.perf_counter()
                lat[i, k] = t1 - due
                lag[i, k] = t0 - due
                if k >= warm_ticks:
                    with slock:
                        stats["prefix"].append(tr.prefix_len); stats["iters"].append(len(tr.step_tokens))
                        stats["stops"][tr.stop] = stats["stops"].get(tr.stop, 0) + 1
        except Exception as e:                                           # noqa: BLE001
            errors.append(repr(e))

    th = [threading.Thread(target=worker, args=(i,), daemon=True) for i in range(B)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    wall = time.perf_counter() - t_start
    bst = beng.stats
    for p in pols:
        p.close()
    beng.close()
    return _seam_summary(B, "threads", n_ticks, warm_ticks, lat, lag, abort.is_set(), errors, stats, wall,
                         dict(engine_calls=bst["calls"], mean_sessions_per_call=bst["sessions"] / max(1, bst["calls"]),
                              cohorts=bst["cohorts"], mean_cohort=bst["cohort_sessions"] / max(1, bst["cohorts"]),
                              max_cohort=bst["max_cohort"]))


def seam_search(eng, B0, Bmax, world, rng, n_ticks, warm_ticks, mode="cohort"):
    """Probe B0, then walk up (pass) or down (fail) in steps of 8: at most four probes.  All ranks probe the same B
    at the same time and a probe passes only if it passes on every rank."""
    import torch
    import torch.distributed as dist

    def probe(B):
        if world > 1:
            dist.barrier()
        r = seam_probe(eng, B, n_ticks, warm_ticks, rng, mode=mode)
        ok = r["ok"]
        if world > 1:
            t = torch.tensor([1 if ok else 0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = bool(t.item())
        r["ok_all_ranks"] = ok
        return r

    probes = [probe(B0)]
    step = 8
    if probes[0]["ok_all_ranks"]:
        B = B0
        while len(probes) < 4 and B + step <= Bmax:
            r = probe(B + step)
            probes.append(r)
            if not r["ok_all_ranks"]:
                break
            B += step
    else:
        B = B0
        while len(probes) < 4 and B - step >= step:
            B -= step
            r = probe(B)
            probes.append(r)
            if r["ok_all_ranks"]:
                break
    passed = [p for p in probes if p["ok_all_ranks"]]
    best = max(passed, key=lambda p: p["streams"]) if passed else None
    return best, probes


# ------------------------------------------------------------------------------------------
# the other BASELINE configs, in brief (each is also a main line with --config)
# ------------------------------------------------------------------------------------------
def config_base_en_single_stream(device=0, chunks=24):
    """Config 2: whisper base.en, AlignAtt, 0.5 s chunks, ONE stream: per-chunk latency through StreamingAlignAtt
    (host chunk in, tokens out), 10 s of audio growing to 22 s."""
    from whisperlivekit_b200.alignatt import AlignAttConfig, StreamingAlignAtt
    from whisperlivekit_b200.dims import ALIGNMENT_HEADS, DIMS
    from whisperlivekit_b200.engine import WhisperEngine
    from whisperlivekit_b200.weights import synthetic_audio, synthetic_state_dict
    dims = DIMS["base.en"]
    eng = WhisperEngine(dims, synthetic_state_dict(dims, seed=0), ALIGNMENT_HEADS["base.en"], precision="bf16", device=device,
                        max_sessions=1, max_batch=1)
    pol = StreamingAlignAtt(eng, AlignAttConfig(nonspeech_prob=1.01))
    audio = synthetic_audio(10.0 + chunks * CHUNK_S, seed=5)
    pol.segments = [CHUNK] * 20
    eng.append_audio(pol.sid, audio[: 20 * CHUNK])
    lat, iters = [], []
    for k in range(chunks + 4):
        seg = audio[(20 + k) * CHUNK: (21 + k) * CHUNK]
        t0 = time.perf_counter()
        pol.insert_audio(seg)
        tr = pol.infer()
        if k >= 4:
            lat.append(time.perf_counter() - t0); iters.append(len(tr.step_tokens))
    pol.close(); eng.close()
    lat = np.asarray(lat) * 1e3
    return dict(workload="whisper base.en AlignAtt greedy, 0.5 s chunks, 1 stream, host chunk in / tokens out per call",
                metric="ms per 0.5 s chunk (process_iter latency)", ms_p50=float(np.percentile(lat, 50)),
                ms_p95=float(np.percentile(lat, 95)), rtf=float(lat.mean() / 1e3 / CHUNK_S),
                mean_decode_iterations=float(np.mean(iters)), chunks=chunks, timed_steps=chunks, warmup_steps=4)


def config_localagreement_64(device=0, streams=64, ticks=3, eng=None):
    """Config 3: large-v3, LocalAgreement shape of work, 1.0 s chunks, 64 ragged streams (5-15 s buffers): per tick and
    stream the audio buffer is encoded (device log-mel + encoder + cross-K/V), a 32-token hypothesis is decoded greedily
    (batched over the streams), then the word-timestamp pass runs (all-position logits + alignment rows, no second
    encode: SURVEY.md 8f-2).  Scripted over the engine entry points the LocalAgreement shim uses."""
    from whisperlivekit_b200.dims import ALIGNMENT_HEADS, DIMS
    from whisperlivekit_b200.engine import WhisperEngine
    from whisperlivekit_b200.weights import synthetic_audio, synthetic_state_dict
    dims = DIMS["large-v3"]
    own = eng is None
    if own:
        eng = WhisperEngine(dims, synthetic_state_dict(dims, seed=0), ALIGNMENT_HEADS["large-v3"], precision="bf16", device=device,
                            max_sessions=streams, max_batch=streams)
    sp = eng.specials
    rng = np.random.default_rng(3)
    base = synthetic_audio(20.0, seed=11)
    sids = [eng.open_session() for _ in range(streams)]
    for s in sids:
        eng.append_audio(s, base[: int(rng.integers(5, 15)) * 16000])
    prompt = list(sp.sot_sequence_including_notimestamps())
    sup = sp.alignatt_suppress_tokens()
    per = []
    for k in range(ticks + 1):
        t0 = time.perf_counter()
        for s in sids:
            eng.drop_audio(s, 16000); eng.append_audio(s, base[:16000])          # 1.0 s chunk in, buffer trimmed by 1.0 s
        eng.encode(sids)
        eng.decode(sids, [prompt] * streams)
        toks = [list(prompt) for _ in sids]
        for _ in range(32):
            r = eng.select(sids, sup)
            for i, t in enumerate(r):
                toks[i].append(t[0])
            eng.decode(sids, [[t[0]] for t in r])
        for i, s in enumerate(sids):                                              # word-timestamp pass per stream
            eng.reset_decoder(s)
            eng.decode_all_logits(s, toks[i], sot_index=0)
        eng.sync()
        if k >= 1:
            per.append(time.perf_counter() - t0)
    for s in sids:
        eng.close_session(s)
    if own:
        eng.close()
    sec = float(np.mean(per))
    return dict(workload=f"whisper large-v3, LocalAgreement-shaped tick, 1.0 s chunks, {streams} ragged streams (5-15 s buffers), "
                         "32-token greedy hypothesis + word-timestamp pass per stream-tick",
                metric=UNIT, value=streams * 1.0 / sec, ms_per_tick=sec * 1e3, rtf_per_stream=sec / 1.0, streams=streams,
                timed_steps=ticks, warmup_steps=1)


def config_alignatt_sortformer(device=0, streams=64, seconds=4, eng=None):
    """Config 4 per GPU: whisper large-v3 AlignAtt ticks at 0.5 s chunks PLUS the streaming Sortformer at its native 1.0 s
    step (two Whisper ticks per diarization step, SURVEY.md 8d), `streams` streams on one GPU (512 streams = 64 per GPU x 8).
    Host chunks in for both engines, tokens / speaker segments out.  Weights: seeded, true geometries (no checkpoint in
    either container; the Sortformer oracle is parity-unpinned, see oracle/sortformer_oracle.py)."""
    import torch
    from whisperlivekit_b200.dims import ALIGNMENT_HEADS, DIMS
    from whisperlivekit_b200.engine import WhisperEngine
    from whisperlivekit_b200.sortformer_dims import SORTFORMER_DIMS, synthetic_sortformer_state_dict, synthetic_two_speaker_audio
    from whisperlivekit_b200.sortformer_engine import B200SortformerDiarization, B200SortformerDiarizationOnline, diarize_batch
    from whisperlivekit_b200.weights import synthetic_audio, synthetic_state_dict
    dims = DIMS["large-v3"]
    own = eng is None
    if own:
        eng = WhisperEngine(dims, synthetic_state_dict(dims, seed=0), ALIGNMENT_HEADS["large-v3"], precision="bf16", device=device,
                            max_sessions=streams, max_batch=streams)
    sd = SORTFORMER_DIMS["diar_streaming_sortformer_4spk-v2"]
    shared = B200SortformerDiarization(sd, synthetic_sortformer_state_dict(sd, 0), precision="bf16", device=device,
                                       max_sessions=streams, max_batch=streams)
    ons = [B200SortformerDiarizationOnline(shared) for _ in range(streams)]
    rng = np.random.default_rng(5)
    base = synthetic_audio(36.0, seed=7)
    two = synthetic_two_speaker_audio(seconds + 14.0, seed=3)
    sids = [eng.open_session() for _ in range(streams)]
    for s in sids:
        off = int(rng.integers(0, 16000 * 5))
        eng.append_audio(s, base[off: off + WINDOW])
    sp = eng.specials
    prefix = list(sp.sot_sequence_including_notimestamps()) + list(range(1000, 1000 + PREFIX - 4))
    sup = sp.alignatt_suppress_tokens()

    def whisper_tick(k):
        for i, s in enumerate(sids):
            eng.drop_audio(s, CHUNK)
            eng.append_audio(s, two[(k * CHUNK + 131 * i) % 100000: (k * CHUNK + 131 * i) % 100000 + CHUNK])
        eng.encode(sids)
        eng.decode(sids, [prefix] * streams)
        eng.no_speech_prob(sids)
        for _ in range(STEPS_PER_CHUNK):
            r = eng.select(sids, sup)
            eng.decode(sids, [[t[0]] for t in r])

    def second(k):
        whisper_tick(2 * k)
        segs = diarize_batch(ons, [np.roll(two[k * 16000:(k + 1) * 16000], 37 * i) for i in range(streams)])
        whisper_tick(2 * k + 1)
        eng.sync()
        return segs

    for k in range(10):                                   # fill the speaker caches (188 + 188 rows) before timing
        diarize_batch(ons, [np.roll(two[k * 16000:(k + 1) * 16000], 37 * i) for i in range(streams)])
    second(10)
    per, diar = [], []
    for k in range(seconds):
        t0 = time.perf_counter()
        second(11 + k)
        per.append(time.perf_counter() - t0)
    for k in range(3):                                    # the diarization leg alone, same state
        t0 = time.perf_counter()
        diarize_batch(ons, [np.roll(two[k * 16000:(k + 1) * 16000], 37 * i) for i in range(streams)])
        diar.append(time.perf_counter() - t0)
    for o in ons:
        o.close()
    shared.close()
    for s in sids:
        eng.close_session(s)
    if own:
        eng.close()
    sec = float(np.mean(per))
    return dict(workload=f"whisper large-v3 AlignAtt (0.5 s chunks, {PREFIX}+{STEPS_PER_CHUNK} tokens per chunk, full 30 s re-encode) + streaming "
                         f"Sortformer 4spk-v2 geometry (1.0 s steps, caches full: 401 rows per stream), {streams} streams per GPU, host chunks in",
                metric=UNIT, value=streams * 1.0 / sec, ms_per_audio_second=sec * 1e3, rtf_per_stream=sec,
                sortformer_ms_per_step=float(np.mean(diar) * 1e3), streams=streams, timed_steps=seconds, warmup_steps=1)


def incremental_leg(eng, scripted, B, world, rng, base, pairs=8, ticks=10, seam_bmax=0):
    """The LABELLED APPROXIMATE incremental encoder (wlk_encode_incremental: encoder K/V retained, ~27 positions per chunk
    run through the encoder instead of 1500) next to the parity mode: (1) agreement -- `pairs` streams are held twice on the
    same engine, one session encoded in parity mode, one incrementally, same audio, same forced prefix, greedy steps
    compared token by token and frame by frame over `ticks` slides of the full 30 s window; (2) throughput -- the scripted
    tick with the window sliding by one host chunk per tick (the device-resident variant would leave the encoder nothing
    to do)."""
    sp = eng.specials
    prefix = list(sp.sot_sequence_including_notimestamps()) + list(range(1000, 1000 + PREFIX - 4))
    sup = sp.alignatt_suppress_tokens()
    par = [eng.open_session() for _ in range(pairs)]
    inc = [eng.open_session() for _ in range(pairs)]
    offs = [int(rng.integers(0, 16000 * 5)) for _ in range(pairs)]
    for i in range(pairs):
        for s in (par[i], inc[i]):
            eng.append_audio(s, base[offs[i]: offs[i] + WINDOW])
    eng.encode(par, incremental=False); eng.encode(inc, incremental=True)          # first blocks: the whole window
    tok_same = frm_same = frm_close = total = 0
    dlog, cos = [], []
    chunk_src = (0.05 * rng.standard_normal((ticks, pairs, CHUNK))).astype(np.float32)
    rows = []
    for k in range(ticks):
        for i in range(pairs):
            for s in (par[i], inc[i]):
                eng.drop_audio(s, CHUNK); eng.append_audio(s, chunk_src[k, i])
        eng.encode(par, incremental=False)
        eng.encode(inc, incremental=True)
        rows.append(int(np.mean(eng.last_block_rows)))
        out = {}
        for name, sids in (("par", par), ("inc", inc)):
            eng.decode(sids, [prefix] * pairs)
            seq = []
            for _ in range(STEPS_PER_CHUNK):
                r = eng.select(sids, sup)
                seq.append(r)
                eng.decode(sids, [[t[0]] for t in (out["par"][len(seq) - 1] if name == "inc" else r)])   # teacher-forced on the parity tokens
            out[name] = seq
        for i in range(0, pairs, 4):                                   # logits after the last forced step, encoder rows
            lp_, li_ = eng.read_logits(par[i]), eng.read_logits(inc[i])
            fin = np.isfinite(lp_) & np.isfinite(li_)
            dlog.append(float(np.abs(lp_[fin] - li_[fin]).max()))
            xp_, xi_ = eng.read_encoder(par[i]), eng.read_encoder(inc[i])
            cos.append(float(np.mean(np.sum(xp_ * xi_, 1) / (np.linalg.norm(xp_, axis=1) * np.linalg.norm(xi_, axis=1) + 1e-9))))
        for a, b in zip(out["par"], out["inc"]):
            for (ta, _, fa), (tb, _, fb) in zip(a, b):
                tok_same += ta == tb; frm_same += fa == fb; frm_close += abs(fa - fb) <= 2; total += 1
    for s in par + inc:
        eng.close_session(s)
    was = eng.incremental_encoder
    eng.incremental_encoder = True
    seam = None
    try:
        r = scripted(eng, B, 6, 3, profile_pass=False, io_only=True)
        if seam_bmax and world == 1:
            # the same real-time paced run through the policy seam as the headline's e2e, in this mode: two probes
            p1 = seam_probe(eng, min(96, seam_bmax), 12, 6, rng, mode="cohort")
            nxt = min(seam_bmax, 128) if p1["ok"] else 64
            p2 = seam_probe(eng, nxt, 12, 6, rng, mode="cohort") if nxt != p1["streams"] else p1
            ok = [p for p in (p1, p2) if p["ok"]]
            seam = dict(value=max((p["streams"] for p in ok), default=0),
                        probes=[dict(streams=p["streams"], ok=p["ok"], p50_latency_s=p["p50_latency_s"], p95_latency_s=p["p95_latency_s"],
                                     mean_prefix_tokens=p["mean_prefix_tokens"]) for p in (p1, p2)],
                        how="largest of two probed stream counts with p95(chunk arrival -> infer() returned) < 0.5 s, same policies, "
                            "pacing and context-saturated prefixes as the headline's e2e")
    finally:
        eng.incremental_encoder = was
    ms = r["ms_io"] / 6
    return dict(mode="incremental encoder, LABELLED APPROXIMATE (north_star item 2; not 1e-3-comparable by construction, SURVEY 7-H1): "
                     "per chunk ~27 of 1500 positions run through the conv stem and the 32 layers against the retained K/V of the rest; "
                     "ring-addressed buffers, nothing moves when the 30 s window slides",
                value=B * world * CHUNK_S / (ms / 1e3), unit=UNIT, streams_per_gpu=B, ms_per_step=ms,
                note="sliding full 30 s window, one host chunk in per stream and tick (H2D inside), same decoder work as the headline tick",
                encoder_rows_per_chunk=float(np.mean(rows)), e2e_through_seam=seam,
                agreement=dict(streams=pairs, ticks=ticks, compared=total, tokens_identical_pct=100.0 * tok_same / total,
                               frames_identical_pct=100.0 * frm_same / total, frames_within_2_pct=100.0 * frm_close / total,
                               max_abs_dlogits=float(np.max(dlog)), encoder_row_cosine_mean=float(np.mean(cos)),
                               how="teacher-forced on the parity mode's greedy tokens; seeded random weights at large-v3 dims (no "
                                   "checkpoint in either container), synthetic speech-like audio: token agreement measures the "
                                   "logit perturbation, frame agreement is pessimistic (random alignment heads have flat rows)"))


def config_qwen_tower(device=0, streams=128, ticks=24):
    """Config 5: Qwen3-ASR-0.6B causal audio tower, 0.25 s chunks (raw audio in, device log-mel), encoder fires per
    192-frame block, `streams` streams with staggered block phases."""
    from whisperlivekit_b200.qwen_dims import QWEN_DIMS, synthetic_tower_state_dict
    from whisperlivekit_b200.qwen_engine import QwenTowerEngine
    from whisperlivekit_b200.weights import synthetic_audio
    dims = QWEN_DIMS["qwen3-asr-0.6b"]
    eng = QwenTowerEngine(dims, synthetic_tower_state_dict(dims, seed=0), precision="bf16", device=device,
                          max_sessions=streams, max_batch=streams)
    eng.load_mel_filters()
    sids = [eng.open_session() for _ in range(streams)]
    rng = np.random.default_rng(0)
    pcm = synthetic_audio(40.0, seed=3)
    mel = np.clip(0.3 + rng.standard_normal((256, dims.n_mels)).astype(np.float32), -1, 1.5)
    eng.forward_chunk(sids, [mel[: int(p)] for p in rng.integers(0, 192, streams)])

    def tick(k):
        chunks = [pcm[(4000 * k + 997 * i) % 500000: (4000 * k + 997 * i) % 500000 + 4000] for i in range(streams)]
        return eng.forward_chunk(sids, eng.mel_append(sids, chunks))

    for k in range(8):
        tick(k)
    per, rows = [], 0
    for k in range(ticks):
        t0 = time.perf_counter()
        out = tick(8 + k)
        per.append(time.perf_counter() - t0)
        rows += sum(o.shape[0] for o in out)
    eng.close()
    per = np.asarray(per)
    return dict(workload=f"qwen3-asr-0.6b causal audio tower, 0.25 s chunks, raw audio in (device log-mel), {streams} streams, "
                         "host audio in / encoder rows out per call (e2e by construction)",
                metric=UNIT, value=float(streams * 0.25 / per.mean()), ms_per_tick_mean=float(per.mean() * 1e3),
                ms_per_tick_p95=float(np.percentile(per, 95) * 1e3), encoder_steps=int(rows), streams=streams,
                timed_steps=ticks, warmup_steps=8)


def run_side_config(name, device):
    fn = {"alignatt-base-en-1stream": config_base_en_single_stream, "localagreement-large-v3-64": config_localagreement_64,
          "alignatt-large-v3-sortformer-64": config_alignatt_sortformer, "qwen-tower-128": config_qwen_tower}[name]
    try:
        return fn(device)
    except Exception as e:                                                # noqa: BLE001
        return dict(error=repr(e))


def scripted_tick(eng, sids, prefix, sup, host, last, sync_before_prefill=False):
    """The device part of one scripted tick (module docstring) for the sessions `sids`: encode, prefill of `prefix`,
    STEPS_PER_CHUNK greedy iterations suppressing `sup`.  Host time inside the engine calls accumulates in `host`; what
    the tick returns to its caller goes to `last`: content frames, no-speech probabilities, and per iteration the
    (token, logprob, attended frame) of every session."""
    B = len(sids)
    t0 = time.perf_counter()
    last["content"] = eng.encode(sids)
    t1 = time.perf_counter()
    if sync_before_prefill:
        eng.sync()
        t1 = time.perf_counter()
    eng.decode(sids, [prefix] * B)
    t2 = time.perf_counter()
    if sync_before_prefill:
        host["prefill_synced"] += t2 - t1; host["ns"] += 1
    else:
        host["encode"] += t1 - t0; host["prefill"] += t2 - t1; host["n"] += 1
    last["no_speech_prob"] = eng.no_speech_prob(sids)
    last["select"] = []
    for _ in range(STEPS_PER_CHUNK):
        r = eng.select(sids, sup)                            # suppress -> greedy token/logprob -> alignment reduce -> frame
        last["select"].append(r)
        t3 = time.perf_counter()
        eng.decode(sids, [[t[0]] for t in r])
        if not sync_before_prefill:
            host["step"] += time.perf_counter() - t3


def scripted_tick_outputs(eng, sids, last, logits_bytes=32 << 20):
    """--dump-outputs: the `last` of a tick as float arrays, and the logits its last decode left for the next iteration
    (the first sessions' rows, up to `logits_bytes`)."""
    sel = np.asarray(last["select"], np.float64)                           # [iteration, session, (token, logprob, frame)]
    return dict(content_frames=np.asarray(last["content"], np.float64),
                no_speech_prob=np.asarray(last["no_speech_prob"], np.float32),
                tokens=sel[..., 0], logprobs=sel[..., 1].astype(np.float32), frames=sel[..., 2],
                logits=np.stack([eng.read_logits(s) for s in sids[:max(1, logits_bytes // (4 * eng.dims.n_vocab))]]).astype(np.float32))


def dump_outputs(out_dir, outputs, limit=64 << 20):
    """outputs: name -> float32 / float64 array.  -> DIR/<name>.npy, at most `limit` bytes in all."""
    total = sum(a.nbytes for a in outputs.values())
    if total > limit:
        raise ValueError(f"outputs of {total} bytes exceed the {limit}-byte dump limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="alignatt-large-v3", choices=CONFIGS)
    ap.add_argument("--streams", type=int, default=int(os.environ.get("WLK_BENCH_STREAMS", "96")), help="streams per GPU")
    ap.add_argument("--model", default="large-v3")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip exact_mode and other_configs")
    ap.add_argument("--no-seam", action="store_true", help="skip the real-time paced run through the seam")
    ap.add_argument("--seam-ticks", type=int, default=16)
    ap.add_argument("--seam-mode", default="cohort", choices=["cohort", "continuous", "threads"],
                    help="cohort: closed cohorts (best p95 capacity); continuous: arrivals join between rounds (measured: p50 0.20 s "
                         "instead of 0.34 s at 64 streams, same p95, but the small encoder batches cost capacity: 80 streams run away)")
    ap.add_argument("--seam-streams", type=int, default=0, help="first stream count probed through the seam (default: 2/3 of --streams)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed tick returned as DIR/<name>.npy (headline config; module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != "alignatt-large-v3" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the headline config (alignatt-large-v3) of --impl b200")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from whisperlivekit_b200.dims import ALIGNMENT_HEADS, DIMS, default_alignment_heads
    from whisperlivekit_b200.weights import synthetic_audio, synthetic_state_dict
    dims = DIMS[args.model]
    heads = ALIGNMENT_HEADS.get(args.model) or default_alignment_heads(dims)
    workload = (f"whisper {args.model} AlignAtt greedy, {CHUNK_S}s chunks, 30 s rolling window fully re-encoded per chunk, "
                f"{PREFIX}-token prefill + {STEPS_PER_CHUNK} decode steps per chunk, {args.streams} streams/GPU")
    metric = "realtime_streams_large_v3_0.5s_chunks"

    # ---------------------------------------------------------------- reference arm (CPU), rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        reference_arm(args, dims, heads, metric, workload)
        return

    # ---------------------------------------------------------------- side configs as the main line
    if args.config not in ("alignatt-large-v3", "alignatt-large-v3-incremental"):
        import torch
        torch.cuda.set_device(local_rank)
        sharded = args.config == "alignatt-large-v3-sortformer-64" and world > 1      # config 4: every rank carries 64 streams
        if rank != 0 and not sharded:
            return
        if sharded:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        sampler = ClockSampler(local_rank); sampler.start()
        r = run_side_config(args.config, local_rank)
        clocks = sampler.summary()
        if sharded:
            t = torch.tensor([r.get("rtf_per_stream", 1e9)], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                                 # the slowest rank sets the rate
            r["rtf_per_stream"] = float(t.item())
            r["value"] = r["streams"] * world / r["rtf_per_stream"]
            dist.barrier(); dist.destroy_process_group()
            if rank != 0:
                return
        hib = args.config != "alignatt-base-en-1stream"
        print(json.dumps(dict(metric=r.get("metric"), value=r.get("value", r.get("ms_p50")), unit=r.get("metric"), n_gpus=world if sharded else 1,
                              steps=r.get("timed_steps"), warmup=r.get("warmup_steps"), higher_is_better=hib, scaling="weak", vs_baseline=None,
                              dtype="bf16", data="synthetic", config=dict(workload=r.get("workload"), name=args.config),
                              e2e=dict(value=r.get("value", r.get("ms_p50")), unit=r.get("metric"),
                                       note="these configs are timed through the host-buffer API: chunk H2D and result D2H are inside"),
                              clocks=clocks, detail=r)))
        return

    # ---------------------------------------------------------------- B200 arm, headline config
    import torch
    import torch.distributed as dist
    from whisperlivekit_b200.engine import WhisperEngine
    from whisperlivekit_b200.sharding import broadcast_blob
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    B = args.streams
    seam_bmax = 0 if args.no_seam else B + 32
    sd = synthetic_state_dict(dims, seed=0) if rank == 0 else None

    def make_engine(precision, max_sessions, max_batch):
        eng = WhisperEngine(dims, None, heads, precision=precision, device=local_rank, max_sessions=max_sessions,
                            max_batch=max_batch, attn_backend=os.environ.get("WLK_ATTN", "auto"))
        if rank == 0:
            eng.load_state_dict(sd)
        if world > 1:                                        # NCCL: weight broadcast at init, nothing else
            ptr, nbytes = eng.weight_blob()

            class _Blob:
                __cuda_array_interface__ = dict(shape=(nbytes,), typestr="|u1", data=(ptr, False), version=2)
            blob = torch.as_tensor(_Blob(), device=f"cuda:{local_rank}")
            broadcast_blob(blob, src=0)
            torch.cuda.synchronize()
            if rank != 0:
                eng.adopt_weights()
        return eng

    rng = np.random.default_rng(1000 + rank)
    base = synthetic_audio(36.0, seed=7)

    def scripted(eng, B, steps, warmup, profile_pass=True, io_only=False, dump=False):
        """The scripted tick (module docstring).  -> (ms device-resident, ms with per-chunk IO, profile, host enqueue);
        dump: also what the last device-resident timed tick returned (module docstring, --dump-outputs)."""
        sp = eng.specials
        sids = [eng.open_session() for _ in range(B)]
        for s in sids:
            off = int(rng.integers(0, 16000 * 5))
            eng.append_audio(s, base[off: off + WINDOW] + 0.001 * rng.standard_normal(WINDOW).astype(np.float32))
        prefix = list(sp.sot_sequence_including_notimestamps()) + list(range(1000, 1000 + PREFIX - 4))
        sup = sp.alignatt_suppress_tokens()
        chunk_host = torch.empty(B, CHUNK, dtype=torch.float32).pin_memory()
        host = dict(encode=0.0, prefill=0.0, prefill_synced=0.0, step=0.0, n=0, ns=0)
        last = {}                                            # the caller-visible results of the latest tick

        def step(with_io, sync_before_prefill=False):
            if with_io:
                chunk_host.copy_(torch.from_numpy(0.05 * rng.standard_normal((B, CHUNK)).astype(np.float32)))
                cn = chunk_host.numpy()
                for i, s in enumerate(sids):
                    eng.drop_audio(s, CHUNK)
                    eng.append_audio(s, cn[i])
            scripted_tick(eng, sids, prefix, sup, host, last, sync_before_prefill)

        def timed(with_io, steps, warmup, profile):
            for _ in range(warmup):
                step(with_io)
            eng.sync()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            if profile:
                eng.profile_reset(); eng.profile_enable(True)
            eng.timer_record(0)
            for _ in range(steps):
                step(with_io)
            eng.timer_record(1)
            eng.sync()
            ms = eng.timer_elapsed_ms(0, 1)
            prof = eng.profile_read() if profile else None
            eng.profile_enable(False)
            if world > 1:
                t = torch.tensor([ms], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
                dist.barrier()
            return ms, prof

        if os.environ.get("WLK_NCU"):
            # profiler capture mode: warm up, then exactly one step between cudaProfilerStart/Stop
            # (ncu --profile-from-start off ...).  Numbers printed under a profiler are never bench values.
            for _ in range(warmup):
                step(False)
            eng.sync()
            torch.cuda.profiler.start()
            step(False)
            eng.sync()
            torch.cuda.profiler.stop()
            print(json.dumps(dict(ncu_capture=True, streams=B)))
            sys.exit(0)

        if io_only:                                          # the sliding-window tick only (host chunk in every tick)
            ms_io, _ = timed(True, steps, warmup, False)
            for s in sids:
                eng.close_session(s)
            return dict(ms_io=ms_io)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        if sampler:
            sampler.start()
        ms_dev, _ = timed(False, steps, warmup, False)
        clocks = sampler.summary() if sampler else None
        outputs = None
        if dump:
            outputs = scripted_tick_outputs(eng, sids, last)
        ms_io, prof, ms_prof = None, None, None
        if profile_pass:
            ms_io, _ = timed(True, steps, max(1, warmup // 3), False)
            # same steps once more with a CUDA-event pair around every kernel class launch (engine stream): per-class
            # device time for the roofline; kept out of `value`: ~10^4 event records per step cost host launch throughput
            ms_prof, prof = timed(False, steps, 0, True)
            step(False, sync_before_prefill=True)            # what the prefill call costs the host when the queue is empty
            eng.sync()
        for s in sids:
            eng.close_session(s)
        return dict(ms_dev=ms_dev, ms_io=ms_io, ms_prof=ms_prof, prof=prof, host=host, clocks=clocks, outputs=outputs)

    def note(msg):
        if rank == 0:
            print(f"[bench] {msg}", file=sys.stderr, flush=True)

    if args.config == "alignatt-large-v3-incremental":
        # the LABELLED APPROXIMATE mode as the main line (every rank carries B streams; max over ranks)
        eng = make_engine("bf16", B + 16, B + 16)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        if sampler:
            sampler.start()
        inc = incremental_leg(eng, scripted, B, world, rng, base)
        clocks = sampler.summary() if sampler else None
        eng.close()
        if rank == 0:
            print(json.dumps(dict(metric=metric + "_incremental_encoder_approximate", value=inc["value"], unit=UNIT, n_gpus=world, steps=6,
                                  warmup=3, ms_per_step=inc["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None,
                                  dtype="bf16", data="synthetic (seeded random weights at true large-v3 dims, synthetic speech-like audio)",
                                  config=dict(workload=workload.replace("fully re-encoded per chunk", "incremental encoder (approximate): "
                                              "~27 of 1500 positions encoded per chunk"), model=args.model, streams_per_gpu=B,
                                              parallelism=f"sessions sharded x{world}", approximate=True),
                                  e2e=dict(value=inc["value"], unit=UNIT, h2d_bytes_per_step=B * world * CHUNK * 4,
                                           d2h_bytes_per_step=B * world * 16 * (STEPS_PER_CHUNK + 1),
                                           note="the timed tick takes one host chunk per stream (H2D) and returns per-token results (D2H)"),
                                  clocks=clocks, detail=inc)))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    eng = make_engine(args.precision, max(B, seam_bmax), max(B, seam_bmax))
    r = scripted(eng, B, args.steps, args.warmup, dump=bool(args.dump_outputs) and rank == 0)
    if r["outputs"] is not None:
        dump_outputs(args.dump_outputs, r["outputs"])
    note(f"scripted tick: {r['ms_dev'] / args.steps:.1f} ms device-resident, {r['ms_io'] / args.steps:.1f} ms with host chunks")
    seam_best, seam_probes = None, []
    if not args.no_seam:
        b0 = args.seam_streams or max(16, (2 * B // 3) // 16 * 16)
        seam_best, seam_probes = seam_search(eng, b0, seam_bmax, world, rng, args.seam_ticks, 6, mode=args.seam_mode)
        note("seam probes: " + json.dumps(seam_probes))
    inc_mode = None
    if not args.no_extras and args.precision == "bf16":
        try:
            inc_mode = incremental_leg(eng, scripted, B, world, rng, base, seam_bmax=seam_bmax)
            note(f"incremental encoder (approximate): {inc_mode['ms_per_step']:.1f} ms per tick at {B} streams/GPU, "
                 f"token agreement {inc_mode['agreement']['tokens_identical_pct']:.1f} %")
        except Exception as e:                                            # noqa: BLE001
            inc_mode = dict(error=repr(e))
    la64, diar64 = None, None
    if not args.no_extras and args.precision == "bf16" and rank == 0 and world == 1 and max(B, seam_bmax) >= 64:
        try:
            la64 = config_localagreement_64(local_rank, eng=eng)
        except Exception as e:                                            # noqa: BLE001
            la64 = dict(error=repr(e))
        try:
            diar64 = config_alignatt_sortformer(local_rank, eng=eng)
        except Exception as e:                                            # noqa: BLE001
            diar64 = dict(error=repr(e))
    eng.close()

    exact, others = None, None
    if not args.no_extras and args.precision == "bf16":
        Bx = min(B, 32)
        engx = make_engine("bf16x3", Bx, Bx)
        rx = scripted(engx, Bx, 2, 3, profile_pass=False)
        engx.close()
        msx = rx["ms_dev"] / 2
        note(f"bf16x3 tick at {Bx} streams: {msx:.1f} ms")
        exact = dict(mode="bf16x3 (WLK_PREC_BF16X3: split operands, 3 tcgen05 MMAs per product; fp32 activations, softmax, K/V)",
                     parity="|dlogits| 2.4e-4 vs the reference at large-v3, tokens and frames identical (tests/test_gpu_large_v3.py)",
                     value=Bx * world * CHUNK_S / (msx / 1e3), unit=UNIT, streams_per_gpu=Bx, ms_per_step=msx)
        if rank == 0 and world == 1:
            reuse = {"localagreement-large-v3-64": la64, "alignatt-large-v3-sortformer-64": diar64}
            others = {c: (reuse[c] if reuse.get(c) is not None else run_side_config(c, local_rank))
                      for c in CONFIGS[1:] if c != "alignatt-large-v3-incremental"}      # that one is `incremental_mode` above

    if rank == 0:
        peaks = load_peaks()
        total_streams = B * world
        ms_dev, ms_io, prof, host = r["ms_dev"], r["ms_io"], r["prof"], r["host"]
        value = total_streams * CHUNK_S * args.steps / (ms_dev / 1e3)
        g = prof["gemm_enc"]
        traffic, tnote = None, "no ncu capture for this configuration"
        for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath) and B == 96 and args.model == "large-v3":
                tj = json.load(open(tpath))
                traffic = tj["mean_dram_bytes_per_launch"]
                tnote = (f"dram__bytes_read+write per launch, mean of one encoder layer's GEMMs, ncu --set full at 96 streams "
                         f"(profiles/{name}); algorithmic {tj.get('algorithmic_bytes_per_launch', 2.04e9) / 1e9:.2f} GB")
                break
        ach = g["flops"] / (g["ms"] / 1e3) / 1e12 if g["ms"] else 0.0
        mult = dict(mel=2, align=3)
        launches = int(sum(v["launches"] * mult.get(k, 1) for k, v in prof.items()))
        classes = {k: dict(ms_per_step=v["ms"] / args.steps, launches_per_step=v["launches"] / args.steps,
                           tflops=(v["flops"] / (v["ms"] / 1e3) / 1e12) if v["ms"] and v["flops"] else None)
                   for k, v in prof.items() if v["launches"]}
        scripted_io = dict(value=total_streams * CHUNK_S * args.steps / (ms_io / 1e3), ms_per_step=ms_io / args.steps,
                           note="the scripted tick with per-chunk H2D append + window shift and per-token D2H, engine driven directly")
        if seam_best is not None:
            e2e = dict(value=float(seam_best["streams"] * world), unit=UNIT,
                       h2d_bytes_per_step=seam_best["streams"] * world * CHUNK * 4,
                       d2h_bytes_per_step=int(seam_best["streams"] * world * 16 * (seam_best["mean_decode_iterations"] + 1)),
                       how="largest probed B per GPU with p95(chunk arrival -> infer() returned) < 0.5 s and no backlog growth; B "
                           "StreamingAlignAtt policies fed host chunks at real time with staggered phases, " +
                           {"continuous": "one scheduler thread, continuous batching over policy requests (cohort.CohortRunner.admit / round): "
                                          "arrivals are admitted between rounds and share the running streams' token-step rounds",
                            "cohort": "advanced in closed cohorts by one scheduler thread (cohort.CohortRunner.run), one batched engine call per round",
                            "threads": "one OS thread per stream over batching.BatchingEngine"}[args.seam_mode],
                       best=seam_best, probes=[dict(streams=p["streams"], ok=p["ok_all_ranks"], p95_latency_s=p["p95_latency_s"],
                                                    start_lag_last_third_s=p["start_lag_last_third_s"]) for p in seam_probes],
                       scripted_with_io=scripted_io)
        else:
            e2e = dict(value=scripted_io["value"] if not seam_probes else 0.0, unit=UNIT, h2d_bytes_per_step=B * world * CHUNK * 4,
                       d2h_bytes_per_step=B * world * 16 * (STEPS_PER_CHUNK + 1),
                       how=("scripted tick with host chunks (seam run skipped)" if not seam_probes else
                            "no probed stream count met p95 < 0.5 s through the seam"),
                       probes=[dict(streams=p["streams"], ok=p["ok_all_ranks"], p95_latency_s=p["p95_latency_s"],
                                    start_lag_last_third_s=p["start_lag_last_third_s"], errors=p["errors"]) for p in seam_probes],
                       scripted_with_io=scripted_io)
        line = dict(
            metric=metric, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
            ms_per_step=ms_dev / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="bf16" if args.precision == "bf16" else "bf16x3",
            data="synthetic (seeded random weights at true large-v3 dims, synthetic speech-like audio)",
            config=dict(workload=workload, model=args.model, streams_per_gpu=B, parallelism=f"sessions sharded x{world}",
                        chunk_s=CHUNK_S, l2="working set (3.4 GB weights + per-stream KV) exceeds the 126 MB L2",
                        rtf_per_stream=(ms_dev / args.steps / 1e3) / CHUNK_S,
                        frac_of_encoder_gemm_stream_ceiling=value / world / (peaks["bf16_tflops"] / 5.18),
                        parity="bf16 mode: tokens identical to the reference wherever its top-2 logit gap exceeds the test's epsilon (63-64 of 64 "
                               "teacher-forced steps on two large-v3 streams; the one flip seen has a reference gap of 0.006), max |dlogits| 0.05-0.075 "
                               "(tests/test_gpu_large_v3.py, profiles/r02_parity_large_v3_bf16.json); fp32 and bf16x3 modes: 1e-3 on logits, identical"),
            e2e=e2e,
            gpu_launches=launches,
            clocks=r["clocks"],
            roofline=dict(bound="tensor", kernel="gemm_tc2_kernel (cta_group::2 pair GEMM; encoder GEMMs, class gemm_enc)", achieved=ach,
                          peak=peaks["bf16_tflops"], unit="TFLOP/s", frac=ach / peaks["bf16_tflops"], traffic=traffic,
                          traffic_note=tnote, peak_source=peaks["source"],
                          flops_per_launch=g["flops"] / max(1, g["launches"]), ms_per_launch=g["ms"] / max(1, g["launches"])),
            kernel_classes=classes,
            profiled_ms_per_step=r["ms_prof"] / args.steps,
            host_enqueue_ms=dict(encode_call=1e3 * host["encode"] / max(1, host["n"]), prefill_call=1e3 * host["prefill"] / max(1, host["n"]),
                                 prefill_call_queue_empty=1e3 * host["prefill_synced"] / max(1, host["ns"]),
                                 decode_step_call=1e3 * host["step"] / max(1, host["n"]) / STEPS_PER_CHUNK,
                                 note="host time inside the asynchronous engine calls; prefill_call is back-pressure of the ~1000-deep "
                                      "launch queue behind the encoder's launches -- with the queue drained first it is prefill_call_queue_empty"),
        )
        if exact is not None:
            line["exact_mode"] = exact
        if inc_mode is not None:
            line["incremental_mode"] = inc_mode
        if others is not None:
            line["other_configs"] = others
        if not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline_leg(dims, sd, heads, 2)
            except Exception as e:                                            # noqa: BLE001  (the line must still print)
                line["cpu_baseline"] = dict(value=None, error=repr(e))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
