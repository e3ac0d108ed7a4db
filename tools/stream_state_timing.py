#!/usr/bin/env python3
"""Cost of stream snapshots (nsb_stream_export / nsb_stream_import) at 24 layers, in the two BASELINE.json setups they matter most for:
config 2 (R = 1, bf16 GEMMs and K/V, 64 streams) and config 3 (R = 6, Q8_0 weights, fp16 K/V, 256 streams).

For each: the streams are warmed with a few chunks of audio (so every snapshot carries a token queue and buffered PCM), then
  * per stream: export, and import into a second engine of the same config, each timed on its own (host clock; both calls return
    after the engine stream is synchronised);
  * whole engine: every stream exported, then imported into a fresh engine on the same GPU.
Snapshot bytes and effective GB/s (snapshot bytes / wall time) are printed with the card name and power limit, read in the same run.
Usage: python tools/stream_state_timing.py [--reps N]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)
import nsb200  # noqa: E402
import synth  # noqa: E402

SETUPS = [  # name, GGUF, compute, K/V, R, streams
    ("config2_bf16_R1_64", "f16", nsb200.COMPUTE_BF16, nsb200.KV_BF16, 1, 64),
    ("config3_q8_0_R6_256", "q8_0", nsb200.COMPUTE_AUTO, nsb200.KV_F16, 6, 256),
]


def gpu_info() -> str:
    return subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3, help="whole-engine moves per setup")
    a = ap.parse_args()
    print(f"# GPU: {gpu_info()}")
    for name, wtype, compute, kv, R, n in SETUPS:
        T = 1 + R
        path = synth.cached_model(wtype, 24, R=R, profile="speech")
        mk = lambda: nsb200.Engine(path, right_context=R, max_streams=n, compute=compute, kv_dtype=kv, cuda_graph=True)
        A = mk()
        ids = np.array([A.open_stream() for _ in range(n)], np.int32)
        warm = 160 * (8 * T * 4 - 1) + 256 + 1000                   # 4 chunks and a partial one
        A.push_batch(ids, np.stack([synth.synth_pcm(s, warm / 16000.0 + 0.01)[:warm] for s in range(n)]))
        A.drain()
        B = mk()
        blob = A.export_stream(int(ids[0]))
        s = B.import_stream(blob); B.close_stream(s)                # first calls: allocation of the checksum word, page faults
        size = len(blob)
        t_exp, t_imp = [], []
        for i in ids:
            t0 = time.perf_counter(); blob = A.export_stream(int(i)); t_exp.append(time.perf_counter() - t0)
            t0 = time.perf_counter(); s = B.import_stream(blob); t_imp.append(time.perf_counter() - t0)
            B.close_stream(s)
        B.close()
        me, mi = float(np.median(t_exp)), float(np.median(t_imp))
        print(f"{name}: snapshot {size} bytes ({size / 1e6:.2f} MB) per stream; export median {me * 1e3:.3f} ms ({size / me / 1e9:.1f} GB/s), "
              f"import median {mi * 1e3:.3f} ms ({size / mi / 1e9:.1f} GB/s)", flush=True)
        for r in range(a.reps):
            B = mk()
            t0 = time.perf_counter()
            blobs = [A.export_stream(int(i)) for i in ids]
            t1 = time.perf_counter()
            for b in blobs:
                B.import_stream(b)
            t2 = time.perf_counter()
            total = sum(len(b) for b in blobs)
            print(f"{name}: whole engine ({n} streams, {total / 1e9:.3f} GB) rep {r}: export {(t1 - t0) * 1e3:.1f} ms "
                  f"({total / (t1 - t0) / 1e9:.1f} GB/s), import into a new engine {(t2 - t1) * 1e3:.1f} ms ({total / (t2 - t1) / 1e9:.1f} GB/s)",
                  flush=True)
            B.close()
        A.close()


if __name__ == "__main__":
    main()
