"""Pooled live-stream ticks for clients that send int16 PCM at 48 kHz or 44.1 kHz (default spec, random-init weights seed 0,
2.0 s contexts, every session in steady state).

Three batchers serve n sessions each on one engine, one tokenize_audio call per tick:

    host    each chunk prepared on the host as AudioTokenizer does (int16 / 32768, audio_io.resample: scipy polyphase in
            float64), then SessionBatcher.tokenize_audio on the float32 arrays (mc_pool_push_audio); the tick time includes
            the preparation, which is also reported alone (host_prep)
    device  SessionBatcher.tokenize_audio on (sr, int16 array) tuples: conversion and resampling inside the push
            (mc_pool_push_pcm, pool_ingest_kernel)
    floor   SessionBatcher.tokenize_audio on 16 kHz float32 chunks of the same resampled length (mc_pool_push_audio)

The three alternate tick by tick.  Every graph key is warmed up first (the contexts fill, then each key is captured on its
second use), then --ticks ticks are timed: host wall clock around one call, which ends in a device synchronise.  The
card's name, power limit and maximum SM clock are read in the same run.

    python tools/bench_pool_ingest.py [--out profiles/r05_pool_ingest.json] [--ticks 100] [--sessions 1,4,16]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rca_b200_loader  # noqa: E402,F401
import realtime_codec_agent_b200 as pkg  # noqa: E402
from realtime_codec_agent_b200 import audio_io as aio  # noqa: E402
from realtime_codec_agent_b200.audio_tokenizer import prep_audio_for_tokenization  # noqa: E402
from realtime_codec_agent_b200.session_batcher import SessionBatcher  # noqa: E402

SR, CONTEXT_SECS = 16000, 2.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:                                                       # noqa: BLE001
        q = f"unavailable ({ex!r})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def stats(ms):
    a = np.asarray(ms)
    return {"p50_ms": float(np.percentile(a, 50)), "p90_ms": float(np.percentile(a, 90)), "mean_ms": float(a.mean())}


def run(gen, n, sr, n_out, ticks):
    n_in = -(-n_out * sr // SR)
    assert aio.resample_plan(sr, SR).n_out(n_in) == n_out
    warm = int(CONTEXT_SECS * SR) // n_out + 3
    total = warm + ticks
    rng = np.random.default_rng(sr + n_out + n)
    src = pkg.synth_audio(total * n_in + n * 997, file_id=7).numpy()
    pcm = [(0.8 * src[s * 997:s * 997 + total * n_in] * 32767).astype(np.int16) for s in range(n)]
    floor_audio = [rng.standard_normal(total * n_out).astype(np.float32) * 0.1 for _ in range(n)]
    bats = {k: SessionBatcher(gen, context_secs=CONTEXT_SECS, max_sessions=n) for k in ("host", "device", "floor")}
    sids = {k: [b.open_session() for _ in range(n)] for k, b in bats.items()}
    times = {k: [] for k in ("host", "device", "floor", "host_prep")}
    for t in range(total):
        chunks = [(sr, x[t * n_in:(t + 1) * n_in]) for x in pcm]
        for k in np.roll(np.array(["host", "device", "floor"]), t % 3):
            bat, ss = bats[k], sids[k]
            a = time.perf_counter()
            if k == "host":
                prepped = [prep_audio_for_tokenization(c, SR, 1) for c in chunks]
                b = time.perf_counter()
                bat.tokenize_audio(dict(zip(ss, prepped)))
            elif k == "device":
                bat.tokenize_audio(dict(zip(ss, chunks)))
            else:
                bat.tokenize_audio({s: x[t * n_out:(t + 1) * n_out] for s, x in zip(ss, floor_audio)})
            e = time.perf_counter()
            if t >= warm:
                times[k].append((e - a) * 1e3)
                if k == "host":
                    times["host_prep"].append((b - a) * 1e3)
    graphs = {k: list(b.pool.graph_count()) for k, b in bats.items()}
    return {"sessions": n, "rate": sr, "chunk_ms": n_out * 1000 // SR, "n_in": n_in, "n_out": n_out,
            **{k: stats(v) for k, v in times.items()}, "graphs_keys_captured": graphs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r05_pool_ingest.json"))
    ap.add_argument("--ticks", type=int, default=100)
    ap.add_argument("--sessions", default="1,4,16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (B200)")
    spec = pkg.DEFAULT_SPEC
    gen = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda")
    rows = []
    for n in [int(v) for v in args.sessions.split(",")]:
        for n_out in (1600, 320):
            for sr in (48000, 44100):
                r = run(gen, n, sr, n_out, args.ticks)
                rows.append(r)
                print(f"n={n:2d} {r['chunk_ms']:3d} ms int16 @ {sr}: host {r['host']['p50_ms']:.3f}/{r['host']['p90_ms']:.3f} "
                      f"(prep {r['host_prep']['p50_ms']:.3f}) device {r['device']['p50_ms']:.3f}/{r['device']['p90_ms']:.3f} "
                      f"floor {r['floor']['p50_ms']:.3f}/{r['floor']['p90_ms']:.3f} ms p50/p90", flush=True)
    res = {"card": card(), "spec": "DEFAULT_SPEC, random init seed 0", "context_secs": CONTEXT_SECS, "timed_ticks": args.ticks,
           "results": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
