"""Offline corpus decode throughput on one GPU: 1 h of codes (6 x 10 min, corpus.encode_streams of synth_audio with
bench.py's seeds, default spec, random-init weights seed 0), resident in HBM.  Modes, alternated round by round in one
process after a warm-up round:

    chunked    corpus.decode_streams (0.1 s chunks, 2.0 s context)
    render     corpus.render_streams (the same windows with 20 ms preroll + the crossfade chain)
    one_shot   gen.decode of each whole file
    cli        codes_to_audio.decode_corpus end to end: .npy files on tmpfs -> 16-bit .wav files on tmpfs

Audio seconds are NEW audio (what the files hold), as in bench.py.  Device time by CUDA events around each mode (the cli
mode: wall clock, it ends in a synchronise).  GEMM rate = GEMM FLOPs of the planned windows (MagiCodecSpec.decode_flops per
window; decode_impl skips rows no kept sample depends on, so this counts a little more than is executed) over the GEMM
class time of mc_profile_*, from a separate profiled pass.  The card's name and power limit are read in the same process.

    python tools/bench_decode_corpus.py [--rounds 3] [--out profiles/r03_bench_decode_corpus.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rca_b200_loader  # noqa: E402,F401
import realtime_codec_agent_b200 as pkg  # noqa: E402
from realtime_codec_agent_b200 import codes_to_audio, corpus  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:                                                       # noqa: BLE001
        q = f"unavailable ({ex!r})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def planned_gemm_flops(spec, n_frames, cf=5, ctx=100):
    irr, steady = corpus.plan_decode_stream(n_frames, cf, ctx, 0, spec.hop)
    warm = [w for w in irr if w.start_frame == 0]
    flops = spec.decode_flops(max(w.frames for w in warm)) if len(warm) >= 2 else 0
    flops += sum(spec.decode_flops(w.frames) for w in irr if not (len(warm) >= 2 and w.start_frame == 0))
    if steady is not None:
        flops += steady[1] * spec.decode_flops(steady[0].frames)
    return flops


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--files", type=int, default=6)
    ap.add_argument("--file_secs", type=float, default=600.0)
    ap.add_argument("--batch_size", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_decode_corpus needs a CUDA device (sm_100)")
    spec = pkg.DEFAULT_SPEC
    dev = torch.device("cuda", 0)
    gen = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device=dev)
    sr, hop = gen.sample_rate, gen.hop
    wavs = [pkg.synth_audio(int(args.file_secs * sr), seed=1234, file_id=f).to(dev) for f in range(args.files)]
    codes = corpus.encode_streams(gen, wavs, 0.1, 2.0, 256, 4)
    del wavs
    audio_secs = sum(int(c.numel()) * hop for c in codes) / sr
    tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    src = os.path.join(tmp, "codes")
    os.makedirs(src)
    with open(os.path.join(src, "codec_info.json"), "w") as f:
        json.dump({"framerate": sr / hop, "num_codebooks": 1, "codebook_size": gen.codebook_size, "sampling_rate": sr,
                   "chunk_size_secs": 0.1, "context_secs": 2.0, "stereo": False}, f)
    for i, c in enumerate(codes):
        np.save(os.path.join(src, f"f{i}_c0.npy"), c.cpu().numpy().astype(np.int32)[None])

    def chunked():
        return corpus.decode_streams(gen, codes, 0.1, 2.0, args.batch_size)

    def render():
        return corpus.render_streams(gen, codes, 0.1, 2.0, 0.02, 0.0, 0.003, args.batch_size)

    def one_shot():
        return [gen.decode(c[None]) for c in codes]

    def cli():
        return codes_to_audio.decode_corpus(gen, src, os.path.join(tmp, "audio"), "chunked", batch_size=args.batch_size,
                                            overwrite=True)

    modes = {"chunked": chunked, "render": render, "one_shot": one_shot, "cli": cli}
    errors = {}
    times = {k: [] for k in modes}
    for rnd in range(args.rounds + 1):                                              # round 0 warms every shape up
        for name, fn in modes.items():
            if name in errors:
                continue
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            try:
                out = fn()
            except Exception as ex:                                                 # noqa: BLE001  (reported, e.g. a size limit)
                errors[name] = repr(ex)
                continue
            e1.record()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            if name == "cli":
                assert not out[1], out[1]
            if rnd > 0:
                times[name].append(wall if name == "cli" else e0.elapsed_time(e1) / 1e3)
            del out
    prof = {}
    for name in ("chunked", "render", "one_shot"):
        if name in errors:
            continue
        torch.cuda.synchronize()
        gen.profile_begin()
        modes[name]()
        p = gen.profile_end()
        flops = (sum(spec.decode_flops(int(c.numel())) for c in codes) if name == "one_shot"
                 else sum(planned_gemm_flops(spec, int(c.numel())) for c in codes))
        prof[name] = {"gemm_ms": p["gemm"]["ms"], "gemm_planned_tflop": flops / 1e12,
                      "gemm_tflops_per_s": flops / (p["gemm"]["ms"] / 1e3) / 1e12 if p["gemm"]["ms"] > 0 else None,
                      "classes_ms": {k: v["ms"] for k, v in p.items()}}
    res = {"metric": "offline corpus decode, audio-s per s (new audio)", "audio_secs": audio_secs, "files": args.files,
           "batch_size": args.batch_size, "rounds": args.rounds, "card": card(), "errors": errors,
           "modes": {k: {"secs": v, "audio_s_per_s": [audio_secs / t for t in v],
                         "median_audio_s_per_s": float(np.median([audio_secs / t for t in v])) if v else None}
                     for k, v in times.items()},
           "profile": prof,
           "timing": "CUDA events around each call with codes resident in HBM (cli: wall clock, .npy -> .wav on tmpfs); "
                     "modes alternated per round after one warm-up round"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
