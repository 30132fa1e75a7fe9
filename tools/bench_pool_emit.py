"""The agent output chain for n live sessions on one GPU, per 0.1 s tick (default spec, random-init weights seed 0,
5 codes per chunk, 20 ms crossfade, target_volume_rms 0, 2.0 s code contexts).  Three ways to serve n agents:

    pool_emit         SessionBatcher.emit_output_chunks: decoder + pad_or_trim + RMS + crossfade of all n sessions in
                      one engine call (mc_pool_push_codes_emit, one CUDA graph replay in the steady state)
    sequential        n private AudioTokenizer + OutputChunkEmitter pairs called one after another (n single-session
                      mc_stream_push_codes_emit calls)
    pool_decode_host  SessionBatcher.detokenize_audio(preroll = L) of all n sessions in one call, then the chain in host
                      numpy per session (OutputChunkEmitter over the decoded window)

The three run side by side on their own sessions, one after another within every tick, so they share the machine's
state.  Every shape is warmed up first (contexts filled, graphs captured), then --ticks steady ticks are timed.  Each
time is host wall clock around one tick's calls, which end in a device synchronise.  The card's name, power limit and
maximum SM clock are read in the same run.

    python tools/bench_pool_emit.py --out DIR [--ticks 2000] [--sessions 1,2,4,8,16]
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
from realtime_codec_agent_b200.codec_chars import UNICODE_OFFSET_LARGE, codes_to_chars  # noqa: E402
from realtime_codec_agent_b200.session_batcher import SessionBatcher  # noqa: E402

CHUNK_SECS, FADE_SECS, CODES_PER_CHUNK = 0.1, 0.02, 5


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:                                                       # noqa: BLE001
        q = f"unavailable ({ex!r})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


class _Window:
    """detokenize_audio handing back a window decoded elsewhere, so OutputChunkEmitter runs its numpy chain on it."""
    num_channels, _native = 1, False

    def __init__(self, sr):
        self.sampling_rate, self.result = sr, None

    def detokenize_audio(self, s, preroll_samples=0):
        return self.result


def stats(ms):
    a = np.asarray(ms)
    return {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "mean_ms": float(a.mean())}


def run_n(gen, n, ticks, warmup, rng):
    K = gen.codebook_size
    pool = SessionBatcher(gen, max_sessions=n)
    pool.arm_emit(CHUNK_SECS, FADE_SECS)
    psid = [pool.open_session() for _ in range(n)]
    seq = [pkg.OutputChunkEmitter(pkg.AudioTokenizer(codec_model=gen, device="cuda"), CHUNK_SECS, FADE_SECS) for _ in range(n)]
    dec = SessionBatcher(gen, max_sessions=n)
    dsid = [dec.open_session() for _ in range(n)]
    shims = [_Window(gen.sample_rate) for _ in range(n)]
    host = [pkg.OutputChunkEmitter(w, CHUNK_SECS, FADE_SECS) for w in shims]
    L = host[0].crossfade_ramps[0]
    times = {"pool_emit": [], "sequential": [], "pool_decode_host": []}
    for t in range(warmup + ticks):
        strs = [codes_to_chars(rng.integers(0, K, size=(1, CODES_PER_CHUNK)), K, unicode_offset=UNICODE_OFFSET_LARGE)
                for _ in range(n)]
        a = time.perf_counter()
        pool.emit_output_chunks({psid[i]: strs[i] for i in range(n)})
        b = time.perf_counter()
        for i in range(n):
            seq[i].emit(strs[i])
        c = time.perf_counter()
        wins = dec.detokenize_audio({dsid[i]: strs[i] for i in range(n)}, preroll_samples=L)
        for i in range(n):
            shims[i].result = wins[dsid[i]]
            host[i].emit(strs[i])
        d = time.perf_counter()
        if t >= warmup:
            times["pool_emit"].append((b - a) * 1e3)
            times["sequential"].append((c - b) * 1e3)
            times["pool_decode_host"].append((d - c) * 1e3)
    return {k: stats(v) for k, v in times.items()}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for pool_emit.json")
    ap.add_argument("--ticks", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=60, help="ticks before timing (contexts fill after 20)")
    ap.add_argument("--sessions", default="1,2,4,8,16")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_pool_emit needs the B200")
    os.makedirs(args.out, exist_ok=True)
    spec = pkg.DEFAULT_SPEC
    gen = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda")
    rng = np.random.default_rng(0)
    res = {"card": card(), "spec": "DEFAULT_SPEC", "chunk_secs": CHUNK_SECS, "fade_secs": FADE_SECS, "target_volume_rms": 0.0,
           "context_secs": 2.0, "ticks": args.ticks, "warmup_ticks": args.warmup, "results": []}
    for n in [int(x) for x in args.sessions.split(",")]:
        r = run_n(gen, n, args.ticks, args.warmup, rng)
        r["n"] = n
        res["results"].append(r)
        print(f"n={n:2d}  pool_emit p50 {r['pool_emit']['p50_ms']:.3f} / p99 {r['pool_emit']['p99_ms']:.3f} ms   "
              f"sequential p50 {r['sequential']['p50_ms']:.3f} / p99 {r['sequential']['p99_ms']:.3f} ms   "
              f"pool_decode_host p50 {r['pool_decode_host']['p50_ms']:.3f} / p99 {r['pool_decode_host']['p99_ms']:.3f} ms",
              flush=True)
    with open(os.path.join(args.out, "pool_emit.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
