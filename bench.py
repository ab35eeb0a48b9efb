#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on B200: decode tokens/s + RTF, Voxtral-Mini-4B Q4_0, 16 s audio.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--streams B] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[4] -- concurrent 16 s streams, B=8 per GPU
(64 at 8 GPUs), weights replicated, no steady-state collective -- with the single-stream
configs[3] numbers measured in the same run and reported under "single_stream".
A *step* = one full transcribe of the GPU's B streams: (peak-normalise + pad + mel) -> encoder ->
adapter -> 38-token prefill -> 107 greedy decode steps -> 108 token ids per stream.
`value` = aggregate decode tokens/s with the reference's definition (tokens / decode seconds,
prefill included; src/bin/e2e_bench.rs:231-240), PCM already resident in HBM, device-timed (CUDA
events on the session stream), max over ranks.  `e2e` = the same through the host-buffer C-ABI
call (pinned host PCM in, token ids out, copies inside the timed region).
Weights are synthetic (random Q4_0 blocks with the real tensor names/shapes: no checkpoint exists
offline) and the audio is a synthetic speech-like signal; token-count, shapes and bytes moved are
identical to the real model's (the decode loop never stops at EOS).

`--impl reference`: the reference has no CPU backend and cannot be built here (Rust, SURVEY F1-F2),
so the reference arm times the oracle port (oracle/: C q4 matvec with OpenMP on all host cores +
torch CPU f32 ops) on a bounded sample of the same workload (single-token decode steps).
"""
from __future__ import annotations

import argparse
import json
import os

# the CPU legs interleave torch-CPU ops with an OpenMP C kernel: spinning worker pools of two
# runtimes would fight over the cores, so make idle OpenMP threads sleep (must be set before import)
os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
os.environ.setdefault("GOMP_SPINCOUNT", "0")
os.environ.setdefault("KMP_BLOCKTIME", "0")
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AUDIO_SECONDS = 16.0
SAMPLE_RATE = 16000
SEED_WEIGHTS = 42
GGUF_PATH = os.environ.get("VOX_BENCH_GGUF", "/dev/shm/voxtral_synth_s42.gguf")
METRIC = "decode_tokens_per_sec"
UNIT = "tokens/s"


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class RankReducer:
    """max / sum of a scalar over the ranks of the (already initialised) process group; identity
    at world size 1.  Device 'cpu' works with gloo (tests), 'cuda:<i>' with nccl (bench)."""

    def __init__(self, dist_mod=None, device="cpu"):
        self.dist, self.device = dist_mod, device

    def _reduce(self, x: float, op_name: str) -> float:
        if self.dist is None:
            return float(x)
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=self.device)
        self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op_name))
        return float(t.item())

    def max(self, x: float) -> float:
        return self._reduce(x, "MAX")

    def sum(self, x: float) -> float:
        return self._reduce(x, "SUM")

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()


def aggregate_throughput(red: RankReducer, local_tokens: int, local_seconds: float):
    """Whole-job throughput: all ranks' tokens / the slowest rank's time (max over ranks)."""
    total = red.sum(float(local_tokens))
    t = red.max(float(local_seconds))
    return total / t, total, t


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def ensure_gguf(rank: int, barrier):
    """Rank 0 writes the deterministic full-size synthetic GGUF (2.5 GB) once per box."""
    from voxtral_mini_realtime_rs_b200 import synth
    if rank == 0 and not os.path.exists(GGUF_PATH):
        t0 = time.time()
        synth.write_synthetic_gguf(GGUF_PATH, synth.VoxtralConfig(), seed=SEED_WEIGHTS)
        sys.stderr.write(f"[bench] wrote {GGUF_PATH} in {time.time() - t0:.1f}s\n")
    barrier()


def dump_outputs(out_dir: str, **arrays):
    """Writes each array as out_dir/<name>.npy in float64 (token ids are exact in it), so that the outputs of two
    builds on the same seeded inputs can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, np.float64))


def make_audio(n_streams: int, rank: int) -> np.ndarray:
    from voxtral_mini_realtime_rs_b200 import synth
    return np.stack([synth.speechlike(AUDIO_SECONDS, seed=1234 + rank * 1000 + i) for i in range(n_streams)])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc, self.th = gpu_index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
def cpu_port_decode_sample(n_steps: int, threads: int, streams: int = 1, with_prefill: bool = False):
    """Oracle port, bounded sample of the GPU arm's decode workload: `streams` concurrent streams batched exactly as the
    GPU batches them (every weight matrix swept ONCE per step for all streams; attention per stream), optionally the
    38-token prefill of all streams, then `n_steps` single-token steps (26 layers + tied lm_head + argmax) with the
    full-size weights on all host threads.  Returns dict(prefill_s, step_s, steps, streams).
    Timed with the vectorised (AVX2 + FMA) re-association of the port (oracle/q4_fast.c), not the strict shader-order
    loop the parity tests use: the baseline should be what these cores can do."""
    import torch
    from oracle import mel as omel, q4 as oq4
    from oracle.model import OracleModel, PREFIX_LEN
    torch.set_num_threads(threads if with_prefill else 1)   # M=1..8 torch ops are tiny; the prefill GEMMs want the cores
    oq4.FAST = True
    om = OracleModel(GGUF_PATH, threads=threads)
    cfg = om.cfg
    ada = om.ada_scales(omel.time_embedding(6.0, cfg.dec_dim))
    caches = [om.new_cache() for _ in range(streams)]
    prefill_s = 0.0
    if with_prefill:
        prefix = [1] + [32] * (PREFIX_LEN - 1)
        x = torch.cat([om.embed_tokens(prefix) for _ in range(streams)])
        t0 = time.perf_counter()
        h = om.decoder_forward_batched(x, ada, caches, PREFIX_LEN)
        last = h.reshape(streams, PREFIX_LEN, -1)[:, -1]
        toks = [int(t) for t in torch.argmax(om.lm_head(last), dim=1)]
        prefill_s = time.perf_counter() - t0
        torch.set_num_threads(1)
    else:
        toks = [1] * streams
        h = om.decoder_forward_batched(torch.cat([om.embed_tokens([t]) for t in toks]), ada, caches, 1)   # untimed: faults the weights in
        toks = [int(t) for t in torch.argmax(om.lm_head(h), dim=1)]
    t0 = time.perf_counter()
    for _ in range(n_steps):
        h = om.decoder_forward_batched(torch.cat([om.embed_tokens([t]) for t in toks]), ada, caches, 1)
        toks = [int(t) for t in torch.argmax(om.lm_head(h), dim=1)]
    dt = time.perf_counter() - t0
    return {"prefill_s": prefill_s, "step_s": dt / max(n_steps, 1), "steps": n_steps, "streams": streams, "seconds": dt + prefill_s}


def cpu_decode_tokens_per_sec(sample: dict, tokens_per_stream: int = 108) -> float:
    """The metric's definition (e2e_bench.rs:231-240: tokens / decode seconds, prefill included) evaluated on the
    sampled prefill time + per-step time: tokens_per_stream * streams / (prefill + (tokens_per_stream - 1) * step)."""
    return tokens_per_stream * sample["streams"] / (sample["prefill_s"] + (tokens_per_stream - 1) * sample["step_s"])


def cpu_threads() -> int:
    """Threads for the CPU port: all cores up to 64 (the matvec is memory-bound beyond that)."""
    return max(1, min(os.cpu_count() or 1, 64))


def run_reference(args, rank, world):
    """The reference's own CPU implementation does not exist (Rust + wgpu only, SURVEY F1-F2): the oracle port is timed,
    on the SAME workload as our arm -- `--streams` (8) concurrent 16 s streams batched per weight sweep, 38-token
    prefill + single-token steps -- each step a bounded sample (one prefill + 3 decode steps) evaluated with the
    metric's own definition.  Rank 0 only."""
    if rank != 0:
        return
    ensure_gguf(0, lambda: None)
    threads = cpu_threads()
    B = args.streams
    cpu_port_decode_sample(1, threads, streams=B)      # warm-up: faults the 2.5 GB of weights in (W honoured as >= 1)
    vals, t_all, pf, st = [], 0.0, 0.0, 0.0
    for _ in range(args.steps):
        smp = cpu_port_decode_sample(3, threads, streams=B, with_prefill=True)
        vals.append(cpu_decode_tokens_per_sec(smp))
        t_all += smp["seconds"]
        pf += smp["prefill_s"]
        st += smp["step_s"]
    K = args.steps
    value = 108 * B / (pf / K + 107 * st / K)
    sample = (f"per step: 38-token prefill of {B} streams + 3 batched single-token decode steps ({B} streams per weight sweep), "
              f"full-size synthetic weights, f32, AVX2 port; tokens/s = 108*{B} / (prefill {pf / K:.2f} s + 107 x step {st / K * 1e3:.0f} ms)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * t_all / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[4]: {B} concurrent 16 s streams per GPU, decode (38-token prefill + 107 steps -> 108 tokens/stream); "
                               "bounded CPU sample of the same batched workload",
                   "model": "Voxtral-Mini-4B-Realtime Q4_0 GGUF layout, synthetic weights (seed 42)",
                   "audio_seconds": AUDIO_SECONDS, "streams_per_gpu": B, "tokens_per_stream": 108,
                   "note": "reference cannot be built here (Rust; no CPU backend at this commit): oracle port timed"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def streaming_leg(vx, model, audio, B, max_ticks=260):
    """B live sessions, each fed 1280 samples (80 ms) per tick, all opened together (worst case: every session steps in
    every second tick).  Returns per-tick device latency statistics and the real-time headroom."""
    pool = vx.StreamingPool(model, max_sessions=B, max_seconds=20.0)
    try:
        peak = np.abs(audio).max(axis=1, keepdims=True)
        sig = (audio * (0.95 / np.maximum(peak, 1e-10))).astype(np.float32)
        sids = [pool.open() for _ in range(B)]
        n = sig.shape[1]
        ticks_ms, steps, out = [], 0, [[] for _ in range(B)]
        first = pool.tick()                      # the left padding (6.08 s of silence): encoder backlog + prefill
        fed = 0
        while fed < n and len(ticks_ms) < max_ticks:
            for i, sid in enumerate(sids):
                pool.push(sid, sig[i, fed:fed + 1280])
            st = pool.tick()
            ticks_ms.append(st["gpu_ms"])
            steps += st["decode_steps"]
            fed += 1280
        for sid in sids:
            pool.finish(sid)
        last = pool.tick()
        for i, sid in enumerate(sids):
            out[i] = pool.poll(sid)[0]
        t = np.array(ticks_ms)
        return {"sessions": B, "tick_audio_ms": 80.0, "ticks": int(t.size), "tick_gpu_ms_mean": float(t.mean()),
                "tick_gpu_ms_p50": float(np.percentile(t, 50)), "tick_gpu_ms_p95": float(np.percentile(t, 95)),
                "tick_gpu_ms_max": float(t.max()), "open_tick_gpu_ms": first["gpu_ms"], "finish_tick_gpu_ms": last["gpu_ms"],
                "decode_steps": int(steps), "tokens_per_session": len(out[0]),
                "realtime_factor": float(t.mean() / 80.0),
                "sessions_at_realtime_estimate": int(B * 80.0 / max(float(np.percentile(t, 95)), 1e-6)),
                "note": "device time per 80 ms tick for all sessions (incremental mel+conv, 32 encoder layers over K/V rings, adapter, "
                        "one shared paged-KV decoder step every 2nd tick); estimate = sessions x 80 ms / p95 tick"}
    finally:
        pool.close()


# --------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import voxtral_mini_realtime_rs_b200 as vx

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod

    red = RankReducer(dist, f"cuda:{local_rank}")
    barrier = red.barrier
    max_over_ranks = red.max

    assert vx.device_count() > local_rank, "bench needs one CUDA device per rank (no CPU fallback)"
    ensure_gguf(rank, barrier)
    B = args.streams
    n = int(AUDIO_SECONDS * SAMPLE_RATE)
    audio = make_audio(B, rank)
    t0 = time.time()
    model = vx.Q4ModelLoader.from_file(GGUF_PATH).load(local_rank, max_batch=B, max_mel_frames=2400)
    load_s = time.time() - t0
    info = model.info
    dev_audio = vx.DeviceBuffer.from_numpy(audio, local_rank)
    pinned = vx.PinnedArray((B, n), np.float32)
    pinned.array[...] = audio

    # ---- warm-up (also captures the decode CUDA graph)
    tm = vx.Timings()
    for _ in range(max(args.warmup, 1)):
        ids = model.transcribe_pcm_dev(dev_audio, B, n, timings=tm)
    n_tok = ids.shape[1]
    launches0 = model.launch_count()

    # ---- timed: device-resident input
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    vx.lib().vox_dev_sync(local_rank)
    wall0 = time.perf_counter()
    dec_ms = pre_ms = enc_ms = tot_ms = pf_ms = 0.0
    for _ in range(args.steps):
        ids = model.transcribe_pcm_dev(dev_audio, B, n, timings=tm)
        dec_ms += tm.decode_ms; pre_ms += tm.preprocess_ms; enc_ms += tm.encode_ms; tot_ms += tm.total_ms
        pf_ms += tm.prefill_ms
    vx.lib().vox_dev_sync(local_rank)
    wall = time.perf_counter() - wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, token_ids=ids)
    barrier()
    launches = model.launch_count() - launches0
    K = args.steps
    value, total_tokens, dec_s = aggregate_throughput(red, B * n_tok * K, dec_ms / 1e3)
    tot_s = max_over_ranks(tot_ms / 1e3)
    wall_s = max_over_ranks(wall)
    step_ms_loop = (dec_ms - pf_ms) / K / max(n_tok - 1, 1)   # one decode-step graph replay, this rank

    # ---- timed: end-to-end through the host-buffer C ABI (pinned PCM in, ids out)
    model.transcribe_pcm(pinned.array, timings=tm)
    barrier()
    vx.lib().vox_dev_sync(local_rank)
    e0 = time.perf_counter()
    for _ in range(K):
        ids_e2e = model.transcribe_pcm(pinned.array, timings=tm)
    e2e_wall = max_over_ranks(time.perf_counter() - e0)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = total_tokens / e2e_wall
    same = bool(np.array_equal(ids_e2e, ids))

    # ---- single stream (configs[3]) in the same run, rank 0's GPU only contributes the number
    tm1 = vx.Timings()
    for _ in range(2):
        model.transcribe_pcm_dev(dev_audio, 1, n, timings=tm1)
    s_dec = s_tot = s_pf = 0.0
    for _ in range(K):
        model.transcribe_pcm_dev(dev_audio, 1, n, timings=tm1)
        s_dec += tm1.decode_ms; s_tot += tm1.total_ms; s_pf += tm1.prefill_ms
    s_step_ms = (s_dec - s_pf) / K / max(n_tok - 1, 1)
    # single-stream end to end through the host-buffer C ABI (pinned PCM in, ids out)
    model.transcribe_pcm(pinned.array[0], timings=tm1)
    vx.lib().vox_dev_sync(local_rank)
    e1 = time.perf_counter()
    for _ in range(K):
        model.transcribe_pcm(pinned.array[0], timings=tm1)
    s_e2e_wall = time.perf_counter() - e1
    single = {"decode_tokens_per_sec": n_tok * K / (s_dec / 1e3), "rtf": (s_tot / K / 1e3) / AUDIO_SECONDS,
              "e2e": {"tokens_per_sec": n_tok * K / s_e2e_wall, "rtf": (s_e2e_wall / K) / AUDIO_SECONDS,
                      "h2d_bytes_per_step": int(n * 4), "d2h_bytes_per_step": int(n_tok * 4),
                      "definition": "108 tokens / wall time of vox_transcribe_pcm for one stream (whole pipeline)"},
              "decode_ms": s_dec / K, "total_ms": s_tot / K, "prefill_ms": s_pf / K, "ms_per_decode_step": s_step_ms,
              "published_gb10_tokens_per_sec": 19.4, "published_gb10_rtf": 0.416}

    # ---- isolated Q4 matvec (configs[1]): [1,3072] x [N,3072]^T for N = 9216 (the reference's bench shape,
    # benches/q4_ops.rs:57-65) and N = 8192 (BASELINE.json's stated shape), 24 rotating weight copies each
    mv = None
    try:
        from voxtral_mini_realtime_rs_b200 import synth
        mv = {}
        for nn in (9216, 8192):
            kk = 3072
            raw = synth.random_q4_blocks(np.random.Generator(np.random.PCG64(7)), nn * kk, 0.02)
            ws = [vx.Q4Tensor.from_q4_bytes(raw, (nn, kk), local_rank) for _ in range(24)]
            ms = vx.q4_matmul_bench(ws, 1, iters=480, warmup=48)
            mv_bytes = nn * kk * 18 // 32 + 4 * kk + 4 * nn
            mv[f"n{nn}"] = {"shape": f"[1,3072]x[{nn},3072]^T", "ms": ms, "bytes": mv_bytes, "gbs": mv_bytes / ms / 1e6,
                            "l2": f"24 rotating weight copies ({24 * mv_bytes / 1e6:.0f} MB) > 126 MB L2"}
            del ws
        mv.update(mv["n9216"])      # top-level keys = the reference's shape (as in round 1)
    except Exception as e:  # pragma: no cover
        mv = {"error": str(e)}

    # ---- streaming sessions (SURVEY 8(f)-1): `B` live sessions fed 80 ms per tick through vox_stream_*; per-tick
    # device latency and how many such sessions one GPU sustains at real time (tick budget = 80 ms of audio)
    streaming = None
    if not args.no_streaming:
        try:
            streaming = streaming_leg(vx, model, audio, B)
        except Exception as e:  # pragma: no cover
            streaming = {"error": str(e)}

    if rank != 0:
        return
    peaks, peak_src = measured_peaks()
    step_bytes = int(info["decode_step_bytes"])
    achieved = step_bytes / (step_ms_loop / 1e3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("decode_step_dram_bytes")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                "traffic_source": "static: profiles/traffic.json (ncu --set full capture of this kernel; not re-measured in this run)",
                "peak_source": peak_src,
                "launch": f"one decode step for B={B} streams = one launch of the persistent decode kernel (CUDA-graph replay)",
                "algorithmic_bytes_per_launch": step_bytes, "ms_per_launch": step_ms_loop,
                "single_stream": {"achieved": step_bytes / (s_step_ms / 1e3) / 1e9,
                                  "frac": step_bytes / (s_step_ms / 1e3) / 1e9 / peaks["hbm_gbs"],
                                  "ms_per_launch": s_step_ms},
                "isolated_matvec": mv}
    # CPU baseline (oracle port) on a bounded sample, N=1 only
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        smp = cpu_port_decode_sample(args.cpu_tokens, threads, streams=B, with_prefill=True)
        cpu = {"value": cpu_decode_tokens_per_sec(smp, int(n_tok)), "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"38-token prefill of {B} streams ({smp['prefill_s']:.1f} s) + {args.cpu_tokens} batched single-token decode steps "
                         f"({smp['step_s'] * 1e3:.0f} ms/step, {B} streams per weight sweep), full-size weights, AVX2 port; "
                         f"tokens/s by the metric's definition: {int(n_tok)}*{B} / (prefill + {int(n_tok) - 1} steps)"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_s / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[4]: {B} concurrent 16 s streams per GPU ({B * world} total), full Q4 transcribe "
                               "(mel+encode+adapter+38-token prefill+107 decode steps -> 108 tokens/stream); "
                               "configs[3] single stream reported under single_stream",
                   "model": "Voxtral-Mini-4B-Realtime Q4_0 GGUF layout, synthetic weights (seed 42)",
                   "audio_seconds": AUDIO_SECONDS, "streams_per_gpu": B, "tokens_per_stream": int(n_tok),
                   "parallelism": f"replicas x{world}, no data-path collective",
                   "l2": "decode reads 1.93 GB of weights per step >> 126 MB L2 (no flush needed)"},
        "rtf": (tot_s / K) / AUDIO_SECONDS, "rtf_per_stream_amortised": (tot_s / K) / (AUDIO_SECONDS * B),
        "stage_ms": {"preprocess": pre_ms / K, "encode": enc_ms / K, "decode": dec_ms / K, "prefill": pf_ms / K},
        "wall_s_timed_region": wall_s, "model_load_s": load_s,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(B * n * 4), "d2h_bytes_per_step": int(B * n_tok * 4),
                "definition": "tokens / wall time of vox_transcribe_pcm (pinned host PCM in, ids out)",
                "ids_match_device_path": same},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "single_stream": single, "streaming": streaming,
        # SURVEY 8(d) config 3: encoder + adapter of the same streams, algorithmic 1.235 TFLOP per 16 s stream
        # (f32-equivalent; the tcgen05 GEMM spends 5 bf16 MMAs per product for f32-grade accuracy)
        "encoder": {"ms": enc_ms / K, "algorithmic_tflop": 1.235 * B,
                    "tflops": 1.235 * B / (enc_ms / K / 1e3) if enc_ms > 0 else None,
                    "frac_of_bf16_dense_peak": (1.235 * B / (enc_ms / K / 1e3)) / peaks.get("bf16_tflops", 1700.9) if enc_ms > 0 else None},
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--streams", type=int, default=8, help="concurrent 16 s streams per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-tokens", type=int, default=6)
    ap.add_argument("--no-streaming", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the token ids of the last timed step (rank 0's streams) to DIR/token_ids.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    rank, local_rank, world = dist_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
