"""Grouped vs ragged session-pool batches per tick (default spec, random-init weights seed 0, 0.1 s chunks, 2.0 s contexts,
5 codes per emitted chunk, 20 ms crossfade, target_volume_rms 0).

n sessions are served per tick; m of them are in their warm-up at distinct context lengths (each restarts every 20 ticks,
the m phases spread over those 20), the other n - m are in steady state.  Two batchers serve identical inputs on their
own sessions of one engine:

    grouped  SessionBatcher(ragged=False): one engine call per context length (1 + m calls per kind and tick)
    ragged   SessionBatcher(ragged=True):  one engine call per kind and tick (mc_pool_push_*_ragged)

Per tick each batcher runs tokenize_audio (encode) and emit_output_chunks (decode + the agent's output chain); the two
batchers alternate which goes first.  Every graph key is warmed up first (the warm-up pattern repeats every 20 ticks and
a key is captured on its second use), then --ticks ticks are timed.  Each time is host wall clock around one call, which
ends in a device synchronise.  The output also gives the engine calls per tick, the graphs each pool captured, and the
share of encode characters on which the two batchers agree (the default split-K kernels differ in summation order
between batch sizes, so near-tie codes may differ).  The card's name, power limit and maximum SM clock are read in the
same run.

    python tools/bench_pool_ragged.py --out DIR [--ticks 200] [--sessions 4,8,16]
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

CHUNK, CODES_PER_CHUNK, WARMUP_TICKS_PER_SESSION = 1600, 5, 20
CALLS = ("push_audio", "push_codes_emit", "push_audio_ragged", "push_codes_emit_ragged")


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


def _count_calls(pool):
    calls = []
    for name in CALLS:
        f = getattr(pool, name)
        setattr(pool, name, lambda *a, _f=f, _n=name, **k: (calls.append(_n), _f(*a, **k))[1])
    return calls


def run_mix(gen, n, m, ticks, warmup, audio, rng):
    K = gen.codebook_size
    bats = {"grouped": SessionBatcher(gen, max_sessions=n), "ragged": SessionBatcher(gen, max_sessions=n, ragged=True)}
    sids, calls = {}, {}
    for name, bat in bats.items():
        bat.arm_emit(0.1, 0.02)
        sids[name] = [bat.open_session() for _ in range(n)]
        calls[name] = _count_calls(bat.pool)
    phase = [round(i * WARMUP_TICKS_PER_SESSION / m) for i in range(m)]       # warming sessions: distinct lengths every tick
    pos = [0] * n
    times = {f"{b}_{k}": [] for b in bats for k in ("encode", "emit")}
    per_tick = {f"{b}_{k}": [] for b in bats for k in ("encode", "emit")}
    agree = []
    for t in range(warmup + ticks):
        for i in range(m):
            if t >= WARMUP_TICKS_PER_SESSION and (t - phase[i]) % WARMUP_TICKS_PER_SESSION == 0:
                for name, bat in bats.items():
                    bat.reset_context(sids[name][i])
        chunks = []
        for i in range(n):
            if pos[i] + CHUNK > audio[i].shape[0]:
                pos[i] = 0
            chunks.append(audio[i][pos[i]:pos[i] + CHUNK])
            pos[i] += CHUNK
        strs = [codes_to_chars(rng.integers(0, K, size=(1, CODES_PER_CHUNK)), K, unicode_offset=UNICODE_OFFSET_LARGE) for _ in range(n)]
        order = list(bats) if t % 2 == 0 else list(reversed(bats))
        enc = {}
        for name in order:
            bat, sd = bats[name], sids[name]
            for kind, call in (("encode", lambda: bat.tokenize_audio({sd[i]: chunks[i] for i in range(n)})),
                               ("emit", lambda: bat.emit_output_chunks({sd[i]: strs[i] for i in range(n)}))):
                del calls[name][:]
                a = time.perf_counter()
                out = call()
                b = time.perf_counter()
                if kind == "encode":
                    enc[name] = out
                if t >= warmup:
                    times[f"{name}_{kind}"].append((b - a) * 1e3)
                    per_tick[f"{name}_{kind}"].append(len(calls[name]))
        if t >= warmup:
            for i in range(n):
                x, y = enc["grouped"][sids["grouped"][i]], enc["ragged"][sids["ragged"][i]]
                agree += [p == q for p, q in zip(x, y)]
    res = {"n": n, "m_warming": m}
    for k, v in times.items():
        res[k] = stats(v)
        res[k]["calls_per_tick"] = float(np.mean(per_tick[k]))
    res["graphs_captured"] = {name: bat.pool.graph_count()[1] for name, bat in bats.items()}
    res["graph_keys"] = {name: bat.pool.graph_count()[0] for name, bat in bats.items()}
    res["encode_chars_equal"] = float(np.mean(agree)) if agree else None
    return res


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for pool_ragged.json")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=60, help="ticks before timing (every key is seen twice by tick 40)")
    ap.add_argument("--sessions", default="4,8,16")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_pool_ragged needs the B200")
    os.makedirs(args.out, exist_ok=True)
    spec = pkg.DEFAULT_SPEC
    gen = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda")
    ns = [int(x) for x in args.sessions.split(",")]
    audio = [pkg.synth_audio(16000 * 20, file_id=200 + i).numpy() for i in range(max(ns))]
    rng = np.random.default_rng(0)
    res = {"card": card(), "spec": "DEFAULT_SPEC", "chunk_samples": CHUNK, "context_secs": 2.0, "fade_secs": 0.02,
           "target_volume_rms": 0.0, "ticks": args.ticks, "warmup_ticks": args.warmup, "results": []}
    for n in ns:
        for m in sorted({1, n // 4, n // 2} - {0}):
            r = run_mix(gen, n, m, args.ticks, args.warmup, audio, rng)
            res["results"].append(r)
            print(f"n={n:2d} m={m:2d}  encode p50 grouped {r['grouped_encode']['p50_ms']:.3f} / ragged {r['ragged_encode']['p50_ms']:.3f} ms"
                  f"  (p90 {r['grouped_encode']['p90_ms']:.3f} / {r['ragged_encode']['p90_ms']:.3f}; calls "
                  f"{r['grouped_encode']['calls_per_tick']:.1f} / {r['ragged_encode']['calls_per_tick']:.1f})"
                  f"   emit p50 grouped {r['grouped_emit']['p50_ms']:.3f} / ragged {r['ragged_emit']['p50_ms']:.3f} ms"
                  f"  (p90 {r['grouped_emit']['p90_ms']:.3f} / {r['ragged_emit']['p90_ms']:.3f}; calls "
                  f"{r['grouped_emit']['calls_per_tick']:.1f} / {r['ragged_emit']['calls_per_tick']:.1f})"
                  f"   graphs {r['graphs_captured']}  chars equal {r['encode_chars_equal']:.4f}", flush=True)
    with open(os.path.join(args.out, "pool_ragged.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
