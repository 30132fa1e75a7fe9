#!/usr/bin/env python
"""bench.py — encode throughput of the MagiCodec tokenization path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference ...                      (the reference's CPU path, oracle port)
    python bench.py ... --dump-outputs DIR                    (also write the codes of the last timed step as .npy)

Workload (BASELINE.json configs[1], the prep_lm_dataset_magicodec shape): per rank, 1 h of synthetic
16 kHz mono audio as 6 x 10 min files, encoded the way encode_audio_gpu_N.sh does it — 0.1 s chunks,
2.0 s context, 256 windows per batch, random-init default-spec weights.  One "step" = one pass over
that hour.  `value` = audio-seconds per second over all ranks with the audio resident in HBM;
`e2e` = the same through the host-facing call with pinned HOST buffers (H2D of the audio and D2H of
the codes inside the timed region).  Weak scaling: every rank encodes its own hour (file-sharded, no
data-path collective); at N>1 the timed region ends with ONE NCCL all-gather of the per-rank manifests (once per
run, as the corpus CLI does).  Extra keys on the line: `e2e_cli` (the same hour through audio_to_codes.encode_corpus
from .wav files on tmpfs: loader threads, pinned staging, device ingest, writer thread), `stereo` (configs[2]),
`one_shot_10s` (configs[0] on the GPU, and on the CPU in `cpu_baseline`), `streaming` (configs[3], >= 5 000 steady
steps), and with `--scaling strong` a load-imbalance figure for ONE uneven file list sharded by duration.
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
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np
import torch

import rca_b200_loader  # noqa: F401
import realtime_codec_agent_b200 as pkg
from realtime_codec_agent_b200 import corpus

METRIC = "encode audio-sec/sec"
UNIT = "audio-s/s"
FILES_PER_RANK = 6
FILE_SECS = 600.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch-size", type=int, default=256, help="windows per batch (the reference CLI's --batch_size)")
    ap.add_argument("--fuse-batches", type=int, default=4, help="consecutive batches issued as one engine launch "
                    "(results are independent of launch grouping; tests/test_gpu_parity.py checks this bit-exactly)")
    ap.add_argument("--file-secs", type=float, default=FILE_SECS)
    ap.add_argument("--files", type=int, default=FILES_PER_RANK)
    ap.add_argument("--cpu-sample-secs", type=float, default=0.0, help="0 = pick ~15 s of CPU work")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: ONE list of uneven files (the N=1 hour) sharded over the ranks with corpus.shard_by_duration")
    ap.add_argument("--stream-steps", type=int, default=5000, help="steady 20 ms steps of the streaming measurement (configs[3])")
    ap.add_argument("--no-extras", action="store_true", help="skip the auxiliary keys (e2e_cli, stereo, one-shot, decode, streaming)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the codes of the last timed step to DIR/codes_fileNNNNN.npy "
                    "(float32; the same arguments give the same inputs, so two builds can be compared file by file)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path only")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, file_ids, codes, n_files_total: int) -> None:
    """One .npy per file of what corpus.encode_streams returned: the int64 codes as float32 (exact below 2**24).  Past
    DUMP_BYTES over all files, each file keeps a seeded sample of its codes and their positions (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // n_files_total - 256                     # bytes per file; 256 covers two .npy headers
    for f, c in zip(file_ids, codes):
        a = c.cpu().numpy()
        name = os.path.join(out_dir, f"codes_file{f:05d}")
        if a.size * 4 > budget:
            pos = np.sort(np.random.default_rng(f).choice(a.size, budget // 12, replace=False))
            np.save(name + "_positions.npy", pos.astype(np.float64))
            a = a[pos]
        np.save(name + ".npy", a.astype(np.float32))


# ------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------- CPU reference arm
def cpu_reference_run(sample_secs: float, steps: int, warmup: int, cores: int, one_shot: bool = False):
    """The reference's CPU path: AudioTokenizer.chunked_tokenize_audio semantics (0.1 s chunks, 2.0 s
    context) around the fp32 oracle port of the network, all host threads.  The unmodified reference
    wrapper cannot travel to the GPU box (/root/reference is absent there), so the host side is this
    repo's AudioTokenizer, which the CPU tests prove string-identical to it."""
    from oracle.magicodec_oracle import OracleGenerator

    torch.set_num_threads(cores)
    spec = pkg.DEFAULT_SPEC
    model = OracleGenerator(spec, pkg.init_random_weights(spec, seed=0))
    tok = pkg.AudioTokenizer(codec_model=model, device="cpu")
    wav = pkg.synth_audio(int((2.0 + 60.0) * 16000), seed=1234, file_id=0).numpy()
    tok.tokenize_audio(wav[:32000])                          # fill the 2.0 s context
    pos = 32000
    t0 = time.perf_counter()
    tok.tokenize_audio(wav[pos:pos + 1600]); pos += 1600
    per_chunk = time.perf_counter() - t0
    if sample_secs <= 0:
        sample_secs = max(0.2, min(6.0, round(15.0 / max(per_chunk, 1e-3)) * 0.1 / max(1, steps + warmup)))
    n_chunks = max(1, int(round(sample_secs / 0.1)))
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for _ in range(n_chunks):
            if pos + 1600 > wav.shape[0]:
                pos = 32000
            tok.tokenize_audio(wav[pos:pos + 1600]); pos += 1600
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    out = {"value": n_chunks * 0.1 * len(times) / total, "ms_per_step": 1e3 * total / len(times),
           "sample": f"{n_chunks} chunks of 0.1 s with a full 2.0 s context per step ({n_chunks * 0.1:.1f} s of audio), "
                     f"fp32 oracle port, default spec", "cores": cores}
    if one_shot:                                   # configs[0] as the reference runs it: one 10 s waveform, CPU, fp32
        wav10 = pkg.synth_audio(160000, seed=1234, file_id=77).numpy()
        tok.reset_context()
        t0 = time.perf_counter(); s = tok.tokenize_audio(wav10); t1 = time.perf_counter()
        tok.detokenize_audio(s); t2 = time.perf_counter()
        out["one_shot_10s"] = {"encode_ms": (t1 - t0) * 1e3, "decode_ms": (t2 - t1) * 1e3, "cores": cores, "kind": "port",
                               "sample": "one 10 s waveform, tokenize_audio + detokenize_audio, one run"}
    return out


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the block GEMMs AT THE BENCH SHAPE (1 024 windows,
    8 layers; profiles/ncu_traffic.json, written by tools/ncu_gemm_traffic.py from an `ncu --set full` capture of
    tools/profile_step.py 1024).  `traffic` on the line is the launch-weighted mean over QKV / Wo / W1 / W2 (one of
    each per layer); the per-GEMM figures sit beside it.  None if the capture is absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        per = t["per_gemm"]
        mean = sum(v["dram_bytes_per_launch"] for v in per.values()) / len(per)
        return mean, {"per_gemm": per, "source": t["source"]}
    except Exception:
        return None, None


# --------------------------------------------------------------------------------- GPU arm
def _write_wav16(path: str, wav: torch.Tensor, sr: int) -> None:
    import struct
    pcm = (wav.clamp(-1, 1) * 32767.0).round().to(torch.int16).cpu().numpy()
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 36 + pcm.nbytes) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, sr, sr * 2, 2, 16) +
                b"data" + struct.pack("<I", pcm.nbytes))
        pcm.tofile(f)


def uneven_durations(total_secs: float, n_files: int):
    """ONE corpus of uneven files (strong scaling): deterministic lengths between 0.25x and 2.5x the mean, whole chunks."""
    rng = np.random.default_rng(7)
    w = rng.uniform(0.25, 2.5, size=n_files)
    secs = np.maximum(1.0, np.round(w / w.sum() * total_secs, 1))
    return [float(x) for x in secs]


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1
    strong = args.scaling == "strong"
    config = {"workload": f"1 h synthetic 16 kHz mono per GPU ({args.files} x {args.file_secs:.0f} s files), chunk 0.1 s, "
                          f"context 2.0 s, batch {args.batch_size} windows ({args.fuse_batches} batches fused per engine "
                          f"launch), MagiCodec default spec (8+8 layers, d=1024), random-init weights seed 0",
              "windows_per_step_per_gpu": int(args.files * args.file_secs * 10), "l2": "inputs_exceed_l2",
              "sharding": "files across ranks, no data-path collective; ONE manifest all_gather at the end of the timed region at N>1"}
    if strong:
        config["workload"] = (f"strong scaling: ONE corpus of {4 * args.files} uneven files ({args.files * args.file_secs:.0f} s in total) "
                              "sharded over the ranks with corpus.shard_by_duration; " + config["workload"].split(", chunk", 1)[1])

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(args.cpu_sample_secs, args.steps, max(args.warmup, 1), cores)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    import torch.distributed as dist
    # Anything a library prints while the job runs (NCCL's version banner goes to stdout) must not land in front of
    # the ONE JSON line: fd 1 points at stderr until the line is printed.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spec = pkg.DEFAULT_SPEC
    gen = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device=dev)
    sr = spec.sample_rate

    if strong:
        durations = uneven_durations(args.files * args.file_secs, 4 * args.files)
        shards = corpus.shard_by_duration(durations, world)
        file_ids = shards[rank]
        file_secs = [durations[f] for f in file_ids]
        rank_secs = [sum(durations[f] for f in sh) for sh in shards]
        total_audio_secs = float(sum(durations))
        imbalance = max(rank_secs) / (sum(rank_secs) / world)
    else:
        file_ids = [rank * args.files + i for i in range(args.files)]
        file_secs = [args.file_secs] * args.files
        total_audio_secs = world * args.files * args.file_secs
        imbalance = 1.0
    # synthesised on the host: the phase is a cumsum over the whole file, and a CUDA cumsum's summation order (so its
    # rounding) changes from run to run, which would change the audio and the codes of every run
    dev_files = [pkg.synth_audio(int(secs * sr), seed=1234, file_id=f).to(dev) for f, secs in zip(file_ids, file_secs)]
    host_files = [torch.empty(d.numel(), dtype=torch.float32).pin_memory() for d in dev_files]
    for h, d in zip(host_files, dev_files):
        h.copy_(d)
    staging = [torch.empty_like(d) for d in dev_files]

    def manifests(codes_list):
        local = [corpus.manifest_entry(f, 0, c, int(c.numel() // 5), rank) for f, c in zip(file_ids, codes_list)]
        return corpus.gather_manifests(local, dev)

    last = {}

    def step_device():
        last["codes"] = corpus.encode_streams(gen, dev_files, 0.1, 2.0, args.batch_size, args.fuse_batches)
        return last["codes"]

    host_codes = [torch.empty(int(d.numel() // 320), dtype=torch.int64).pin_memory() for d in dev_files]
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [torch.cuda.Event() for _ in file_ids]

    def step_e2e():
        # what a corpus job does: the upload of file i+1 (pinned host -> HBM, side stream) runs under the encode of file i
        main_s = torch.cuda.current_stream()
        copy_stream.wait_stream(main_s)                   # staging buffers are free again
        with torch.cuda.stream(copy_stream):
            for s_, h, ev in zip(staging, host_files, copied):
                s_.copy_(h, non_blocking=True)
                ev.record(copy_stream)
        codes = []
        for s_, hc, ev in zip(staging, host_codes, copied):
            main_s.wait_event(ev)
            c = corpus.encode_streams(gen, [s_], 0.1, 2.0, args.batch_size, args.fuse_batches)[0]
            hc[: c.numel()].copy_(c, non_blocking=True)
            codes.append(c)
        main_s.synchronize()
        last["codes"] = codes
        return codes

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile=False):
        """K steps, then (N>1) the one manifest all-gather of the run, between barriers; device time = max over ranks."""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = gen.launch_count
        if profile:
            gen.profile_begin()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        if world > 1:
            manifests(last["codes"])
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        prof = gen.profile_end() if profile else None
        ms = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), gen.launch_count - l0, prof

    for _ in range(max(args.warmup, 3)):
        codes = step_device()
    if world > 1:
        manifests(codes)                                   # NCCL communicator warm-up, outside the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dev_ms, _, launches, _ = timed(step_device, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, file_ids, last["codes"], len(durations) if strong else world * args.files)
    # the same K steps once more with an event pair around every kernel launch: per-class device time for the
    # roofline object.  Kept out of the pass above so that `value` carries no instrumentation overhead.
    prof_ms, _, _, prof = timed(step_device, args.steps, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    step_e2e()
    _, e2e_wall_ms, _, _ = timed(step_e2e, args.steps)
    sync_all()

    value = total_audio_secs * args.steps / (dev_ms / 1e3)
    e2e_value = total_audio_secs * args.steps / (e2e_wall_ms / 1e3)

    # ---- e2e_cli: the same audio through the real consumer path, audio_to_codes.encode_corpus over .wav files on tmpfs
    cli = None
    if not args.no_extras:
        try:
            cli = bench_cli(args, gen, dev, rank, world, dev_files, file_ids, total_audio_secs, sync_all)
        except Exception as ex:                             # never lose the main line to an auxiliary metric
            cli = {"error": repr(ex)}

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else \
            "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
        g = prof["gemm"]
        achieved = g["flops"] / (g["ms"] / 1e3) / 1e12 if g["ms"] > 0 else 0.0
        traffic, traffic_detail = ncu_traffic()
        roofline = {"bound": "tensor", "kernel": "gemm_bf16_sm100_kernel (linears + implicit-GEMM convs)",
                    "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                    "peak_source": peak_src, "traffic": traffic, "traffic_detail": traffic_detail,
                    "launches": g["launches"], "avg_launch_ms": g["ms"] / max(1, g["launches"]),
                    "share_of_step": g["ms"] / prof_ms, "instrumented_ms_per_step": prof_ms / args.steps,
                    "other_classes_ms_per_step": {k: v["ms"] / args.steps for k, v in prof.items()},
                    "hbm_kernels_achieved_GBps": (prof["elementwise"]["bytes"] / (prof["elementwise"]["ms"] / 1e3) / 1e9)
                    if prof["elementwise"]["ms"] > 0 else None,
                    "hbm_peak_GBps": peaks.get("hbm_gbs")}
        exec_flops = sum(v["flops"] for v in prof.values()) / args.steps
        roofline["whole_step_TFLOPs"] = exec_flops / (dev_ms / args.steps / 1e3) / 1e12
        roofline["whole_step_frac"] = roofline["whole_step_TFLOPs"] / peak_tf
        windows = config["windows_per_step_per_gpu"]
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_wall_ms / args.steps,
                        "h2d_bytes_per_step": int(sum(d.numel() for d in dev_files) * 4), "d2h_bytes_per_step": int(sum(h.numel() for h in host_codes) * 8),
                        "api": "corpus.encode_streams per file -> B200Generator.encode -> mc_encode (pinned host audio in on a side stream, "
                               "pinned host codes out)"},
                "e2e_cli": cli,
                "gpu_launches": int(launches),
                "roofline": roofline,
                "executed_tflop_per_step_per_gpu": exec_flops / 1e12,
                "reference_equivalent_tflop_per_step_per_gpu": windows * spec.encode_flops(100) / 1e12,
                "codes_checksum": int(sum(int(c.sum().item()) for c in codes) % (1 << 31))}
        if strong:
            line["load_imbalance"] = {"max_over_mean_rank_audio_secs": imbalance, "rank_audio_secs": rank_secs,
                                      "partition": "corpus.shard_by_duration (longest-processing-time first)"}
        if world == 1 and not args.no_extras:
            extras_single_gpu(args, gen, dev, spec, codes, dev_files, line)
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(args.cpu_sample_secs, 1, 1, cores, one_shot=not args.no_extras)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]}
            if "one_shot_10s" in r and isinstance(line.get("one_shot_10s"), dict):
                line["one_shot_10s"]["cpu_reference"] = r["one_shot_10s"]
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def bench_cli(args, gen, dev, rank, world, dev_files, file_ids, total_audio_secs, sync_all):
    """`e2e_cli`: audio_to_codes.encode_corpus (the body of `python -m rca_b200_loader audio_to_codes`) over this
    run's audio as 16-bit .wav files on tmpfs: header probe + duration-balanced sharding, loader threads reading into
    pinned buffers, H2D of the int16 payload on a copy stream, device ingest kernels, corpus encode, writer thread with
    atomic .npy writes, and the manifest all-gather — wall clock between barriers, max over ranks."""
    import shutil
    import torch.distributed as dist
    from realtime_codec_agent_b200 import audio_to_codes

    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    tag = os.environ.get("MASTER_PORT", "0") + "_" + str(os.environ.get("TORCHELASTIC_RUN_ID", os.getppid()))
    root = os.path.join(base, f"rca_b200_bench_{tag}")
    raw, out = os.path.join(root, "raw"), os.path.join(root, "codes")
    os.makedirs(os.path.join(raw, f"rank{rank:02d}"), exist_ok=True)
    for f, d in zip(file_ids, dev_files):
        _write_wav16(os.path.join(raw, f"rank{rank:02d}", f"file{f:05d}.wav"), d, gen.sample_rate)
    sync_all()
    try:
        walls = []
        nfiles = 0
        for it in range(1 + args.steps):                                   # one untimed pass, then K timed ones
            sync_all()
            t0 = time.perf_counter()
            man, errs = audio_to_codes.encode_corpus(gen, raw, out, batch_size=args.batch_size, fuse_batches=args.fuse_batches,
                                                     rank=rank, world_size=world, overwrite=True, loader_threads=6, prefetch_files=5)
            merged = corpus.gather_manifests(man, dev)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            t = torch.tensor([wall], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if it > 0:
                walls.append(float(t[0]))
            nfiles = len(merged)
            if errs:
                raise RuntimeError(f"e2e_cli: {errs[:2]}")
        total = sum(walls)
        return {"value": total_audio_secs * len(walls) / total, "unit": UNIT, "ms_per_step": 1e3 * total / len(walls),
                "files": nfiles, "input": "16-bit PCM .wav on tmpfs", "h2d_bytes_per_step": int(sum(d.numel() for d in dev_files) * 2),
                "api": "audio_to_codes.encode_corpus (what `python -m rca_b200_loader audio_to_codes` runs after loading the model)"}
    finally:
        sync_all()
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)


def extras_single_gpu(args, gen, dev, spec, codes, dev_files, line):
    """The other BASELINE configs as keys on the line (N = 1 only): configs[2] stereo hour, configs[0] 10 s one-shot
    encode + decode, the decode half at the offline batch shape, configs[3] streaming."""
    def cuda_time(fn, iters):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters, out

    try:                                              # configs[2]: 1 h of two-channel dialogue -> _c0 / _c1
        ch1 = [pkg.synth_audio(int(d.numel()), seed=1234, file_id=1000 + i, channel=1, device=dev) for i, d in enumerate(dev_files)]
        streams = [s for pair in zip(dev_files, ch1) for s in pair]
        ms, st_codes = cuda_time(lambda: corpus.encode_streams(gen, streams, 0.1, 2.0, args.batch_size, args.fuse_batches), 2)
        secs = sum(d.numel() for d in dev_files) / spec.sample_rate
        tok2 = pkg.AudioTokenizer(codec_model=gen, num_channels=2, device=dev)
        n = 16000 * 3
        s2 = tok2.chunked_tokenize_audio(torch.stack([dev_files[0][:n], ch1[0][:n]]).cpu().numpy(), 0.1)
        inter = torch.stack([st_codes[0][:150], st_codes[1][:150]], dim=1).reshape(-1).cpu().tolist()
        line["stereo"] = {"value": secs / (ms / 1e3), "unit": "dialogue audio-s/s (two channels each)", "channel_audio_s_per_s": 2 * secs / (ms / 1e3),
                          "ms_per_step": ms, "config": "configs[2]: 1 h synthetic two-channel dialogue (encode_audio_stereo.sh shape), "
                          "channels encoded as independent streams -> _c0 / _c1",
                          "interleave_matches_tokenizer": [ord(c) - tok2.unicode_offset for c in s2] == inter}
        del ch1, streams, st_codes
    except Exception as ex:
        line["stereo"] = {"error": repr(ex)}
    try:                                              # configs[0]: one 10 s waveform, one-shot encode + decode
        tok = pkg.AudioTokenizer(codec_model=gen, device=dev)
        wav10 = pkg.synth_audio(160000, seed=1234, file_id=77).numpy()
        enc, dec = [], []
        for it in range(23):
            tok.reset_context()
            t0 = time.perf_counter(); s = tok.tokenize_audio(wav10); t1 = time.perf_counter()
            (_, rec), _, _ = tok.detokenize_audio(s); t2 = time.perf_counter()
            if it >= 3:
                enc.append((t1 - t0) * 1e3); dec.append((t2 - t1) * 1e3)
        line["one_shot_10s"] = {"config": "configs[0] on the GPU: AudioTokenizer.tokenize_audio(10 s) -> 500 chars, detokenize_audio -> 160 000 samples; "
                                "wall clock around the Python calls (host numpy in, host numpy out)",
                                "encode_ms_p50": float(np.percentile(enc, 50)), "decode_ms_p50": float(np.percentile(dec, 50)),
                                "chars": len(s), "samples": int(rec.shape[-1])}
    except Exception as ex:
        line["one_shot_10s"] = {"error": repr(ex)}
    try:                                      # the decode half of the path at the offline batch shape
        ctx = torch.stack([c[:25600] for c in codes]).reshape(-1, 100)[:1024].contiguous()    # 1024 windows x 100 codes
        gen.decode(ctx)
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gen.profile_begin()
        d0.record()
        for _ in range(5):
            gen.decode(ctx)
        d1.record()
        torch.cuda.synchronize()
        dprof = gen.profile_end()
        dms = d0.elapsed_time(d1) / 5
        line["decode"] = {"value": ctx.shape[0] * 2.0 / (dms / 1e3), "unit": "audio-s/s", "ms_per_launch": dms,
                          "config": "mc_decode of 1024 windows x 100 codes -> 1024 x 2.0 s of waveform (every sample kept), "
                                    "codes resident in HBM",
                          "gemm_TFLOPs": dprof["gemm"]["flops"] / (dprof["gemm"]["ms"] / 1e3) / 1e12 if dprof["gemm"]["ms"] else None,
                          "class_ms_per_launch": {k: v["ms"] / 5 for k, v in dprof.items()}}
    except Exception as ex:
        line["decode"] = {"error": repr(ex)}
    try:                                      # BASELINE metric, second half: p50 streaming decode ms/frame
        from tools.bench_stream import run as stream_run, run_emit
        tok = pkg.AudioTokenizer(codec_model=gen, device=dev)
        st = stream_run(tok, 0.02, args.stream_steps, 120)
        st100 = stream_run(tok, 0.1, 300, 30)
        emit = run_emit(tok, 300, 30)
        line["streaming"] = {"config": f"configs[3]: batch-1, 20 ms frames, 2.0 s context, tokenize_audio + detokenize_audio per frame, "
                                       f"{args.stream_steps} steady steps after 120 warm-up steps (device-resident context, CUDA-graph replay), "
                                       "wall clock around the Python call",
                             "p50_decode_ms_per_frame": st["decode_wall_ms"]["p50"], "decode_wall_ms": st["decode_wall_ms"],
                             "encode_wall_ms": st["encode_wall_ms"], "decode_cuda_ms": st["decode_cuda_ms"],
                             "encode_cuda_ms": st["encode_cuda_ms"],
                             "chunk_100ms": {"decode_wall_ms": st100["decode_wall_ms"], "encode_wall_ms": st100["encode_wall_ms"],
                                             "note": "the agent's default chunk (realtime_agent_config.py): 5 frames per call"},
                             "emit_chain_100ms": {"emit_wall_ms": emit["emit_wall_ms"],
                                                  "note": "OutputChunkEmitter.emit = decoder + pad_or_trim + normalize_audio_rms + "
                                                          "smooth_join in one engine call (realtime_agent_v2.py:556-579)"}}
    except Exception as ex:                   # never lose the main line to the auxiliary metric
        line["streaming"] = {"error": repr(ex)}


if __name__ == "__main__":
    main()
