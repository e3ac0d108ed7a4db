#!/usr/bin/env python3
"""bench.py -- headline benchmark of the streaming hot path (BASELINE.json metric: RTFx = audio seconds
processed per wall second, summed over streams; per-chunk latency alongside).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C] [--only-headline] [--dump-outputs DIR]

Headline (top-level keys of the JSON line) = BASELINE.json configs[1] ("config 2"): nemotron-speech-streaming-en-0.6b
(24 layers, random-init synthetic weights of that architecture), bf16 compute, 64 concurrent streams per GPU, 160 ms chunks
(att_right_context = 1). A "step" = one batched engine step = one chunk for every stream.
The same line carries a `configs` record with the other BASELINE.json configs measured the same way in the same run:
  3: Q8_0 weights (dequantisation fused into the GEMM operand path), 256 streams x 560 ms -- STRONG scaling under --gpus N
     (256 streams in total, 256 / N per GPU, sharded by nemotron-speech.cpp_b200/sharding.py)
  4: 80 ms chunks, 128 streams per GPU (1024 over 8 GPUs), host-to-host p50 / p99 chunk latency
  5: 1.12 s chunks (full lookahead), 64 long-form streams per GPU
N > 1 (torchrun, one rank per GPU): streams are independent, every rank runs its own engine, no data-path collective;
torch.distributed is used only for the barrier, the max-over-ranks of the timed regions and the gather of token checksums.

Per config:
  value   : device-resident throughput -- PCM of the step already in HBM, K steps enqueued back to back on the engine's stream,
            CUDA events around them
  e2e     : the same K steps through the public C ABI with HOST buffers, up to three steps in flight: nsb_push_pcm_batch,
            nsb_engine_step_begin (pinned staging + H2D + step + D2H of the token ids enqueued), the next chunk pushed meanwhile,
            nsb_engine_step_end, nsb_pop_tokens_batch; wall clock. The tokens of this leg are check-summed and compared with a
            re-run of the same audio WITHOUT the CUDA graph, one step at a time (`token_check`)
  latency : host-to-host, one chunk at a time as a real-time feed sees it: clock starts when the chunk's last sample is handed to
            nsb_push_pcm_batch and stops when its token ids are back on the host (graph-capture step excluded)
  roofline: the dominant kernel class (tcgen05 layer GEMMs) timed alone, live, against MEASURED_PEAKS.json

--dump-outputs DIR writes, for the headline config, what its last timed step computed: encoder_out.npy = the encoder output of the
last device-resident step [streams x (1 + R), 1024], tokens.npy = the token ids the last e2e step handed back [streams, 12 (1 + R)],
-1 past each stream's count. The inputs are seeded, so two builds run with the same arguments can be compared array for array.

--impl reference times the CPU oracle port of the reference path (oracle/liboracle.so, all host threads): every step = one chunk
of a bounded number of streams, `ms_per_step` is its measured wall time. The reference's own ggml build cannot be produced
offline (DESIGN.md section 2).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

N_LAYERS = int(os.environ.get("NSB_BENCH_LAYERS", 24))
PROFILE = os.environ.get("NSB_BENCH_PROFILE", "speech")   # synthetic-model calibration: "speech" = ~4.5 tokens per audio second, "parity" = the tests' dense emission
IN_FLIGHT = max(1, min(3, int(os.environ.get("NSB_BENCH_IN_FLIGHT", 3))))   # steps between step_begin and step_end in the e2e leg
BENCH_CHUNKS = 8                                          # distinct chunks staged in HBM for the device-resident leg, cycled

# BASELINE.json configs by number (configs[0] is the CPU case = --impl reference).
#   streams per GPU at N = 1, att_right_context, GGUF type, compute, K/V ring, scaling under --gpus N
CONFIGS = {2: dict(streams=64, R=1, weights="f16", compute="bf16", kv="bf16", scaling="weak"),
           3: dict(streams=256, R=6, weights="q8_0", compute="q8_0", kv="f16", scaling="strong"),
           4: dict(streams=128, R=0, weights="f16", compute="bf16", kv="bf16", scaling="weak"),
           5: dict(streams=64, R=13, weights="f16", compute="bf16", kv="bf16", scaling="weak")}
if "NSB_BENCH_STREAMS" in os.environ:
    CONFIGS[2]["streams"] = int(os.environ["NSB_BENCH_STREAMS"])
if "NSB_BENCH_R" in os.environ:
    CONFIGS[2]["R"] = int(os.environ["NSB_BENCH_R"])


def stream_recording(g: int) -> int:
    """Which of the 8 synthetic recordings global stream g carries (shifted by 977 (g // 8) samples). Must not be a function of g mod G
    alone for any G the streams are sharded over (sharding.py: stream -> rank g mod G), or a rank's whole batch is one recording."""
    return (g + g // 8) % 8


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        # the GEMM roofline times the kernel ALONE (back-to-back launches): the burst bf16 figure is its denominator, not the sustained one
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", d.get("bf16_tflops_sustained", 1400.0))), "measured"
    return 6650.0, 1400.0, "fallback"


def measured_traffic(rows: int):
    """DRAM bytes per launch of the layer GEMM class from this round's `ncu --set full` capture (tools/ncu_summary.py writes the file)."""
    p = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    e = d.get(str(rows))
    return (e["dram_bytes_per_launch"], f"profiles/r02_gemm_traffic.json ({e['source']})") if e else (None, None)


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe). NVML polled every 5 ms from a thread
    (the timed region is ~0.1 s: `nvidia-smi -lms 100` would give one sample); nvidia-smi is the fallback."""

    def __init__(self, device: int):
        self.rows, self.proc, self.device = [], None, device
        self.sm, self.mx, self.reason_bits, self.stop_flag, self.thread, self.nvml = [], None, 0, False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.device)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml = (pynvml, h)

            def poll():
                while not self.stop_flag:
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.reason_bits |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.thread = threading.Thread(target=poll, daemon=True); self.thread.start()
            return
        except Exception:
            self.nvml = None
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            pynvml = self.nvml[0]
            bits = {"hw_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            reasons = sorted(k for k, b in bits.items() if self.reason_bits & b)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.sm), "source": "nvml"}
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi"}


def gemm_roofline(eng, rows: int, elem: int = 2, iters: int = 10, w_elem: float | None = None):
    """Dominant kernel = the tcgen05 layer GEMM (8 launches per conformer layer). Timed live, alone: for each of the six
    distinct shapes, 24 layers x `iters` launches back to back on the engine's stream (every launch on a different layer's
    weights: 24 x 2-8 MB > L2, so weights stream from HBM), CUDA events around the loop; same tile / split-K choice as the
    step. achieved = algorithmic bytes (weights + A operand + C result, once each) / mean launch duration, weighted by how
    often each shape occurs in a layer."""
    # kind: (N, K, bytes per C element incl. read-modify-write, occurrences per layer)
    kinds = {0: (4096, 1024, elem, 2), 1: (1024, 4096, 8, 2), 2: (3072, 1024, 4, 1), 3: (1024, 1024, 8, 1), 4: (2048, 1024, 4, 1), 5: (1024, 1024, 8, 1)}
    w_elem = elem if w_elem is None else w_elem       # HBM bytes per weight (Q8_0 blocks: 34 / 32)
    tot_us = tot_bytes = tot_flops = 0.0; n = 0; per = {}
    for kind, (N, K, cb, occ) in kinds.items():
        us = eng.bench_gemm(kind, rows, 0, 0, -1, 0, iters)    # splits = -1: the engine's own split-K choice for this shape
        b = N * K * w_elem + rows * K * elem + rows * N * cb
        per[("ff_up", "ff_down", "qkv", "attn_out", "pw1", "pw2")[kind]] = {"us": round(us, 2), "GBps": round(b / us / 1e3, 1),
                                                                           "TFLOPs": round(2.0 * rows * N * K / us / 1e6, 1)}
        tot_us += us * occ; tot_bytes += b * occ; tot_flops += 2.0 * rows * N * K * occ; n += occ
    return tot_bytes / n, tot_us / n, per, tot_flops / n


def host_threads():
    try:
        return len(os.sched_getaffinity(0))         # torchrun exports OMP_NUM_THREADS=1: ignored, all cores this process may use
    except AttributeError:
        return os.cpu_count() or 1


def oracle_chunk_loop(R: int, streams: int, steps: int, warmup: int, threads: int):
    """Oracle port (reference arithmetic restated, OpenMP over output rows): `steps` timed steps, each = one chunk of every one of
    `streams` streams pushed through the reference's per-chunk driver. Returns (seconds per timed step list, chunks per step)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    import synth
    T = 1 + R
    O.lib().orc_set_threads(threads)
    path = synth.cached_model("f32", N_LAYERS, R=R, profile=PROFILE)
    m = O.Model(path, O.MM_REF)
    first, shift = 160 * (8 * T - 1) + 256, 1280 * T
    need = first + shift * (steps + warmup)
    pcm = [synth.synth_pcm(s, need / 16000.0 + 0.01) for s in range(streams)]
    st = [O.Stream(m, R) for _ in range(streams)]
    pos = first
    for s in range(streams):
        st[s].push(pcm[s][:first])                      # chunk 0 (its graph-build analogue is excluded like the GPU arm's capture step)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        for s in range(streams):
            st[s].push(pcm[s][pos:pos + shift])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
        pos += shift
    assert all(x.chunks == 1 + warmup + steps for x in st)
    return times, streams


def cpu_baseline(R: int, threads: int | None = None, steps: int | None = None, streams: int = 2):
    threads = threads or host_threads()
    T = 1 + R
    steps = steps or max(4, int(12.8 / (0.08 * T * streams)))      # ~13 s of audio: 5-10 s of CPU work on a 16-core host
    times, n = oracle_chunk_loop(R, streams, steps, 1, threads)
    dt = float(np.sum(times))
    audio = n * steps * 0.08 * T
    return {"value": audio / dt, "unit": "audio_s/s", "cores": threads, "kind": "port",
            "sample": f"{streams} streams x {steps} chunks of {int(80 * T)} ms (after 2 untimed chunks per stream), f32 weights, {N_LAYERS} layers, R={R} "
                      f"({dt:.1f} s wall); oracle/liboracle.so = CPU restatement of the reference streaming path "
                      f"(ggml build not reproducible offline)"}


def run_reference(args, rank: int):
    if rank != 0:
        return
    c = CONFIGS[args.config]
    R, T, threads = c["R"], 1 + c["R"], host_threads()
    ref_streams = 2
    steps = max(1, min(args.steps, int(120.0 / (0.14 * T * ref_streams)) or 1))      # bounded: ~0.07 s of CPU per stream-frame
    warm = max(1, min(args.warmup, 3))
    times, n = oracle_chunk_loop(R, ref_streams, steps, warm, threads)
    dt = float(np.sum(times))
    value = n * steps * 0.08 * T / dt
    base = {"value": value, "unit": "audio_s/s", "cores": threads, "kind": "port",
            "sample": f"each step = one {int(80 * T)} ms chunk of {ref_streams} streams through the oracle port (f32 weights, {N_LAYERS} layers, R={R}); "
                      f"{steps} timed steps ({dt:.1f} s wall) after {warm} warm-up steps -- a bounded sample of the {c['streams']}-stream workload"}
    line = {"impl": "reference", "metric": "rtfx", "value": value, "unit": "audio_s/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": f"0.6B streaming FastConformer RNN-T, {N_LAYERS} layers, {int(80 * T)} ms chunks (R={R}), "
                                                        f"bounded CPU sample ({ref_streams} streams per step) of the {c['streams']}-stream workload",
                                            "baseline_config": args.config, "steps_requested": args.steps},
            "cpu_baseline": base, "e2e": {"value": value, "unit": "audio_s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_LIMIT = 64 << 20


def write_dump(d: str, arrays: dict) -> None:
    """--dump-outputs: each array as DIR/<name>.npy in float32. An array whose share of the 64 MB limit is too small keeps a fixed,
    seeded sample of its rows, and DIR/<name>_rows.npy (float64) says which."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_LIMIT // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        if a.nbytes > share:
            keep = share // (a[0].nbytes + 8)                # + its float64 row index
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            np.save(os.path.join(d, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(d, f"{name}.npy"), a)


def token_checksum(per_stream):
    """Order-sensitive checksum of {global stream id: token list}."""
    c = 0
    for sid in sorted(per_stream):
        c = zlib.crc32(np.asarray([sid, len(per_stream[sid])] + list(per_stream[sid]), dtype=np.int64).tobytes(), c)
    return c


def run_config(no: int, args, ctx, headline: bool):
    """All legs of one BASELINE.json config on this rank's GPU; returns the record (rank 0 fills the aggregate fields)."""
    import torch
    import torch.distributed as dist
    import nsb200
    import synth
    from nemotron_speech_cpp_b200 import sharding
    rank, world, local = ctx["rank"], ctx["world"], ctx["local"]
    c = CONFIGS[no]
    R, T = c["R"], 1 + c["R"]
    chunk_s = 0.08 * T
    # which global streams this rank owns: weak = its own `streams`; strong = its share of a fixed total (sharding.py: stream s -> rank s mod G)
    total = c["streams"] * (world if c["scaling"] == "weak" else 1)
    if c["scaling"] == "strong" and os.environ.get("NSB_BENCH_EMULATE_WORLD"):
        # one GPU plays ONE rank of a k-GPU strong-scaling run (its 1 / k share of the fixed stream population): per-rank timing of the
        # 4- and 8-GPU cases on a box with fewer GPUs; the ranks share nothing, so the k-GPU aggregate is k times this rank's value
        total = max(1, total // int(os.environ["NSB_BENCH_EMULATE_WORLD"]))
    mine = sharding.local_streams(range(total), rank, world)
    S = len(mine)
    steps = args.steps
    warm_chunks = 40 if no == 2 else max(8, 70 // T + 3)          # > 70 / T: the attention cache is full (steady state) before timing
    hbm_peak, tf_peak, peak_kind = peaks()

    path = synth.cached_model(c["weights"], N_LAYERS, R=R, profile=PROFILE)
    compute = {"f16": nsb200.COMPUTE_F16, "bf16": nsb200.COMPUTE_BF16, "q8_0": nsb200.COMPUTE_Q8_0}[c["compute"]]
    kv = {"f16": nsb200.KV_F16, "bf16": nsb200.KV_BF16}[c["kv"]]
    t_load = time.perf_counter()
    eng = nsb200.Engine(path, right_context=R, max_streams=S, compute=compute, kv_dtype=kv, device=local,
                        cuda_graph=os.environ.get("NSB_BENCH_GRAPH", "1") != "0")
    t_load = time.perf_counter() - t_load
    shift = eng.shift_samples
    need = 160 * (8 * T * (warm_chunks + BENCH_CHUNKS) - 1) + 256
    base = [synth.synth_pcm(1000 * no + s, need / 16000.0 + 0.01)[:need] for s in range(8)]
    # distinct streams from 8 seeds, keyed by GLOBAL stream id g: recording (g + g // 8) % 8 rolled by 977 (g // 8) samples. (g % 8 alone
    # would hand every stream of a rank the SAME recording under s mod G sharding with G = 8: the whole batch then bursts together and
    # the max over ranks reports the burstiest recording instead of the workload -- seen as 2.07 vs 1.77 ms per step at 8 vs 1 GPU.)
    pcm = np.stack([np.roll(base[stream_recording(g)], 977 * (g // 8)) for g in mine])
    eng.bench_prepare(pcm, warm_chunks)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    # ---- device-resident timing: K steps, CUDA events inside the engine per step (engine stream) ----
    for _ in range(max(args.warmup, BENCH_CHUNKS)):       # >= W untimed steps; at least one pass over every staged chunk (one CUDA graph each)
        eng.bench_step()
    eng.bench_steps(2 * BENCH_CHUNKS)                     # ... and over the graphs of the pipelined form (decode overlap: other decode graphs, both sides)
    st0 = eng.stats()
    sampler = ClockSampler(local); sampler.start()
    sync_all()
    t0 = time.perf_counter()
    dev_ms, _ = eng.bench_steps(steps)                    # K steps enqueued back to back, CUDA events on the engine stream
    sync_all()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    dump = {}
    if headline and args.dump_outputs and rank == 0:
        dump["encoder_out"] = eng.debug_get("x", S)       # the last timed step's encoder output, before anything else runs
    launches = int(eng.stats().kernel_launches - st0.kernel_launches)
    dev_lat = sorted(eng.bench_step() for _ in range(min(steps, 30)))     # device time of single host-synchronised steps
    t_dev_s, wall_s = max_over_ranks(dev_ms / 1e3, wall)
    audio_s = total * chunk_s * steps
    value = audio_s / t_dev_s

    # ---- per-kernel-class breakdown + roofline of the dominant kernel class (layer GEMMs) ----
    prof, prof_total = eng.bench_profile()
    g_ms, _ = prof["layer_gemm"]
    rows = S * T
    q8 = c["compute"] == "q8_0"
    b_launch, us_launch, per_shape, f_launch = gemm_roofline(eng, rows, w_elem=34.0 / 32.0 if q8 else None, iters=10 if headline else 4)
    achieved = b_launch / us_launch / 1e3
    traffic, traffic_src = measured_traffic(rows)
    roofline = {"bound": "hbm", "kernel": f"tcgen05 layer GEMMs (8 launches per conformer layer, M = {rows} token rows)",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_kind": peak_kind, "share_of_step": g_ms / prof_total if prof_total else None,
                "algorithmic_bytes_per_launch": b_launch, "avg_launch_us": us_launch, "per_shape": per_shape,
                "how": "CUDA events on the engine stream around 24 layers x back-to-back launches per shape (kernel timed alone, weights from HBM)"}
    if rows >= 512:
        # configs 3 and 5: past the ridge (~208 rows at 2-byte weights) the layer GEMMs are bound by the tensor pipe, not by HBM
        tf = f_launch / us_launch / 1e6
        roofline.update({"bound": "tensor", "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": tf / tf_peak,
                         "algorithmic_flops_per_launch": f_launch, "peak_kind": peak_kind + " (burst bf16: kernel timed alone)"})
    # whole step against its HBM bound (SURVEY 8d: weights once + K/V ring + activations)
    w_bytes = 578.8e6 * (34.0 / 32.0 if q8 else 2.0) + 27e6
    step_bytes = w_bytes + S * (24 * 2 * (70 + T) * 1024 * 2 + 2 * 24 * 8 * 1024 * 4 + 10 * 24 * T * 1024 * 4)
    step_flops = S * T * 1.1576e9 + S * 24 * 6 * T * (70 + T) * 1024
    t_bound = max(step_bytes / (hbm_peak * 1e9), step_flops / (tf_peak * 1e12))
    step_roof = {"bytes": step_bytes, "flops": step_flops, "bound_ms": 1e3 * t_bound, "bound": "hbm" if step_bytes / (hbm_peak * 1e9) >= step_flops / (tf_peak * 1e12) else "tensor",
                 "frac": t_bound / (t_dev_s / steps)}
    breakdown = {k: {"ms": round(v[0], 4), "launches": v[1]} for k, v in prof.items()}

    # ---- end to end through the public C ABI with host buffers ----
    for s in range(S):
        eng.reset_stream(s)
    e2e_warm = max(args.warmup, 70 // T + 2)              # the 70-frame cache is full before the timed region here too
    n_lat = min(steps, 30)
    e2e_chunks = steps + e2e_warm + n_lat + 1
    need2 = 160 * (8 * T * e2e_chunks - 1) + 256
    reps = -(-need2 // pcm.shape[1])
    pcm2 = np.ascontiguousarray(np.tile(pcm, (1, reps))[:, :need2])
    first = 160 * (8 * T - 1) + 256
    ids = np.arange(S, dtype=np.int32)
    pos = 0
    toks = {g: [] for g in mine}
    popped = None

    def feed(n):
        nonlocal pos
        eng.push_batch(ids, pcm2[:, pos:pos + n]); pos += n

    def pop():
        nonlocal popped
        out, cnt = eng.pop_tokens_batch(ids, 12 * T)
        for i, g in enumerate(mine):
            toks[g] += out[i, :cnt[i]].tolist()
        popped = (out, cnt)
        return int(cnt.sum())

    feed(first)
    for _ in range(e2e_warm):
        assert eng.step() == S
        feed(shift)
    pop()
    sync_all()
    t0 = time.perf_counter()
    ntok = 0
    # steps in flight (IN_FLIGHT, default 3 = the C ABI's limit): while the device runs step i the host hands over the next chunks of
    # every stream and stages + enqueues steps i+1 (and i+2) (pinned staging, H2D, all kernels, D2H of the token ids), then waits for
    # step i and pops its tokens. The third slot keeps the engine stream busy while a long greedy decode is still running on its own.
    begun = 0
    for i in range(steps):
        while begun < steps and begun - i < IN_FLIGHT:
            if begun:
                feed(shift)
            assert eng.step_begin() == S
            begun += 1
        assert eng.step_end() == S                        # wait for the OLDEST step in flight, queue its tokens
        ntok += pop()
    sync_all()
    e2e_wall = time.perf_counter() - t0
    (t_e2e,) = max_over_ranks(e2e_wall)
    if dump:
        out, cnt = popped                                  # token ids of the last timed step, per stream, -1 past each count
        dump["tokens"] = np.where(np.arange(out.shape[1]) < cnt[:, None], out, -1)
        write_dump(args.dump_outputs, dump)
    # ---- host-to-host chunk latency: one chunk at a time, as a real-time feed sees it ----
    lat = []
    for _ in range(n_lat):
        t0 = time.perf_counter()
        feed(shift)                                       # the chunk's last sample is handed over here
        assert eng.step_begin() == S
        assert eng.step_end() == S
        pop()                                             # ... and its token ids are on the host here
        lat.append(1e3 * (time.perf_counter() - t0))
    lat.sort()
    (p50, p99) = max_over_ranks(lat[len(lat) // 2], lat[min(len(lat) - 1, int(0.99 * len(lat)))])
    # ---- token check: the same audio again, no CUDA graph, one plain step at a time ----
    n_done = e2e_warm + steps + n_lat
    eng.set_cuda_graph(False)
    for s in range(S):
        eng.reset_stream(s)
    toks_ng = {g: [] for g in mine}
    eng.push_batch(ids, pcm2[:, :first + shift * (n_done - 1)])
    while eng.step() == S:
        pass
    out, cnt = eng.pop_tokens_batch(ids, 12 * T * (n_done + 1))
    for i, g in enumerate(mine):
        toks_ng[g] = out[i, :cnt[i]].tolist()
    eng.set_cuda_graph(True)
    all_g = sharding.gather_results({g: toks[g] for g in mine}, rank, world) if world > 1 else toks
    all_ng = sharding.gather_results({g: toks_ng[g] for g in mine}, rank, world) if world > 1 else toks_ng
    rec = None
    if rank == 0:
        ck, ck_ng = token_checksum(all_g), token_checksum(all_ng)
        rl = 1280 * T + 353
        e2e = {"value": audio_s / t_e2e, "unit": "audio_s/s", "h2d_bytes_per_step": S * rl * 2 + S * 4,
               "d2h_bytes_per_step": S * (10 * T + 1) * 4, "ms_per_step": 1e3 * t_e2e / steps, "tokens": ntok,
               "tokens_per_audio_s": ntok / (S * chunk_s * steps)}
        rec = {"baseline_config": no, "metric": "rtfx", "value": value, "unit": "audio_s/s", "ms_per_step": 1e3 * t_dev_s / steps, "steps": steps,
               "scaling": c["scaling"], "streams_total": total, "streams_per_gpu": S, "chunk_ms": int(chunk_s * 1000), "token_rows_per_step": rows,
               "dtype": c["compute"], "kv_ring": c["kv"], "weights_file": c["weights"],
               "e2e": e2e,
               "latency_ms": {"p50": p50, "p99": p99, "n": n_lat, "definition": "host to host: chunk handed to nsb_push_pcm_batch -> its token ids popped "
                              "(one chunk at a time, graph-capture step excluded); max over ranks",
                              "device_p50": dev_lat[len(dev_lat) // 2], "device_p99": dev_lat[min(len(dev_lat) - 1, int(0.99 * len(dev_lat)))]},
               "token_check": {"crc32_graph_steps_in_flight": ck, "crc32_no_graph_single_steps": ck_ng, "identical": ck == ck_ng,
                               "tokens": sum(len(v) for v in all_g.values()), "chunks_per_stream": n_done},
               "roofline": roofline, "step_roofline": step_roof, "breakdown": breakdown, "gpu_launches": launches, "clocks": clocks,
               "wall_ms_per_step": 1e3 * wall_s / steps, "engine_load_s": round(t_load, 2)}
        if not rec["token_check"]["identical"]:
            raise SystemExit(f"bench: config {no}: tokens of the CUDA-graph / two-in-flight leg differ from the un-graphed re-run "
                             f"({ck:#x} vs {ck_ng:#x})")
    eng.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json config in the headline keys (default 2)")
    ap.add_argument("--only-headline", action="store_true", help="skip the `configs` record (the other BASELINE.json configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the headline config's last timed step computed to DIR/*.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    import nsb200  # noqa: F401
    import synth
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    ctx = {"rank": rank, "world": world, "local": local}
    side = [] if args.only_headline else [n for n in sorted(CONFIGS) if n != args.config]
    # synthetic models (one GGUF per weight type, variants per latency mode derived by patching two small tensors): rank 0 writes
    if rank == 0:
        for n in [args.config] + side:
            synth.cached_model(CONFIGS[n]["weights"], N_LAYERS, R=CONFIGS[n]["R"], profile=PROFILE)
    if world > 1:
        dist.barrier()

    head = run_config(args.config, args, ctx, headline=True)
    others = {}
    for n in side:
        try:
            r = run_config(n, args, ctx, headline=False)
            if rank == 0:
                others[str(n)] = r
        except SystemExit:
            raise
        except Exception as e:                              # a side config must not take the headline down with it
            if world > 1:
                raise
            others[str(n)] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        c = CONFIGS[args.config]
        T = 1 + c["R"]
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(c["R"])
        q8 = c["compute"] == "q8_0"
        line = {"metric": "rtfx", "value": head["value"], "unit": "audio_s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": c["scaling"], "vs_baseline": None,
                "dtype": c["compute"], "data": "synthetic",
                "config": {"workload": f"nemotron-speech-streaming-en-0.6b architecture ({N_LAYERS} conformer layers, random-init synthetic weights), "
                                       f"{c['compute']} tcgen05 GEMMs" + (" (Q8_0 weights resident in HBM as int8 + block scales; dequantised to fp16 inside every step, one layer ahead on a side "
                                       "stream into two L2-sized fp16 shadows)" if q8 else "")
                                       + f", {c['kv']} K/V ring, {head['streams_per_gpu']} concurrent streams per GPU, {head['chunk_ms']} ms chunks "
                                       f"(att_right_context={c['R']}), steady state (70-frame attention cache full); joint blank bias calibrated to a "
                                       f"{'speech-like' if PROFILE == 'speech' else 'dense (parity-test)'} token rate ({head['e2e']['tokens_per_audio_s']:.1f} tokens per audio second measured in the e2e leg)",
                           "baseline_config": args.config, "streams_per_gpu": head["streams_per_gpu"], "chunk_ms": head["chunk_ms"],
                           "l2_policy": f"per-step working set (weights {0.62 if q8 else 1.16} GB + K/V ring {head['streams_per_gpu'] * 6.88e-3:.2f} GB) > 126 MB L2",
                           "token_profile": PROFILE, "device_resident_input": f"{BENCH_CHUNKS} consecutive chunks per stream staged in HBM, cycled"},
                "p50_chunk_latency_ms": head["latency_ms"]["p50"], "p99_chunk_latency_ms": head["latency_ms"]["p99"], "latency": head["latency_ms"],
                "wall_ms_per_step": head["wall_ms_per_step"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
                "roofline": head["roofline"], "step_roofline": head["step_roofline"], "breakdown": head["breakdown"], "token_check": head["token_check"],
                "engine_load_s": head["engine_load_s"], "configs": others}
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
