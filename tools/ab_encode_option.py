"""A/B of one engine option on the offline chunked encode, in one process on one GPU.

Every launch is the benchmark's shape: 1024 overlapping windows of 2.0 s (100 frames) read from one flat buffer with a
0.1 s stride, the last 5 frames of each kept (corpus.encode_streams with batch 256 x 4 fused).  Launches cycle through
eight different stretches of a 2 min signal, and the option value alternates between blocks so that clock and power
drift hit every arm alike.  Per arm: median and spread of the per-launch device time (CUDA events), the per-class
device time of mc_profile (in a separate pass: its event pairs add overhead), the kernel launches per call, and a
check that every arm returns the same codes and margins bit for bit.

    python tools/ab_encode_option.py exact_cut 0 1 [--blocks 8 --per-block 10 --out result.json]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rca_b200_loader  # noqa: E402,F401
import realtime_codec_agent_b200 as pkg  # noqa: E402

WINDOWS, LD, T, KEEP = 1024, 1600, 32000, 5


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("option")
    ap.add_argument("values", type=int, nargs="+")
    ap.add_argument("--blocks", type=int, default=8)
    ap.add_argument("--per-block", type=int, default=10)
    ap.add_argument("--out", help="also write the result as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ab_encode_option: needs a CUDA device")

    spec = pkg.DEFAULT_SPEC
    gen = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda")
    span = (WINDOWS - 1) * LD + T
    n_seg = 8
    audio = pkg.synth_audio(n_seg * span, seed=1234, file_id=0).cuda()
    segs = [audio[i * span:(i + 1) * span] for i in range(n_seg)]

    def launch(i, margin=False):
        return gen.encode(segs[i % n_seg], keep_last_frames=KEEP, return_margin=margin, row_stride=LD,
                          num_windows=WINDOWS, window_samples=T)

    ref = {}
    for v in args.values:                                     # warm-up and output check per arm
        gen.set_option(args.option, v)
        for i in range(3):
            launch(i)
        ref[v] = [launch(i, margin=True) for i in range(2)]
    v0 = args.values[0]
    identical = all(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
                    for v in args.values for a, b in zip(ref[v], ref[v0]))

    times = {v: [] for v in args.values}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.per_block)]
    k = 0
    for _ in range(args.blocks):
        for v in args.values:
            gen.set_option(args.option, v)
            launch(k)                                         # one untimed launch after the switch
            torch.cuda.synchronize()
            for e0, e1 in ev:
                e0.record()
                launch(k)
                e1.record()
                k += 1
            torch.cuda.synchronize()
            times[v] += [e0.elapsed_time(e1) for e0, e1 in ev]

    prof, launches = {}, {}
    for v in args.values:
        gen.set_option(args.option, v)
        torch.cuda.synchronize()
        l0 = gen.launch_count
        gen.profile_begin()
        for i in range(args.per_block):
            launch(i)
        p = gen.profile_end()
        launches[v] = (gen.launch_count - l0) / args.per_block
        prof[v] = {c: {"ms": r["ms"] / args.per_block, "launches": r["launches"] / args.per_block,
                       "TFLOPs": r["flops"] / r["ms"] / 1e9 if r["ms"] > 0 else 0.0} for c, r in p.items()}

    props = torch.cuda.get_device_properties(0)
    res = {"option": args.option, "gpu": props.name, "shape": f"{WINDOWS} windows x {T} samples, stride {LD}, keep {KEEP}",
           "outputs_identical": identical, "arms": {}}
    med0 = float(np.median(times[v0]))
    for v in args.values:
        t = np.array(times[v])
        res["arms"][str(v)] = {"median_ms": float(np.median(t)), "p10_ms": float(np.percentile(t, 10)),
                               "p90_ms": float(np.percentile(t, 90)), "min_ms": float(t.min()), "max_ms": float(t.max()),
                               "n": int(t.size), "vs_first_arm": float(np.median(t)) / med0 - 1.0,
                               "gpu_launches_per_call": launches[v], "profile_ms_per_call": prof[v]}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not identical:
        sys.exit("ab_encode_option: the arms returned different codes or margins")


if __name__ == "__main__":
    main()
