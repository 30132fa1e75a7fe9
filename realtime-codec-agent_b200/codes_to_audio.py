"""Offline corpus decode CLI — the way back from what ``audio_to_codes`` wrote to audio files:

    python -m rca_b200_loader codes_to_audio --codes_path data/audio/codes/MagiCodec-50Hz-Base/0.1s_2.0s/mono \
        --audio_path data/audio/decoded [--mode chunked|render|one_shot] [--format pcm16|float]

Modes:
    chunked    every chunk decoded from the trailing context of codes, its own samples kept (corpus.decode_streams):
               what a loop of AudioTokenizer.detokenize_audio over the chunks returns — how the agent decodes
    render     the agent's recording: chunked decode with preroll + RMS normalisation + crossfade
               (corpus.render_streams, one emit_chunks_kernel launch per channel) — what OutputChunkEmitter plays
    one_shot   the whole file as one window (one gen.decode per file), like detokenize_audio(whole_string)

Inputs: ``<rel>_c<channel>.npy`` (int16 / int32 / int64, shape (1, T) or (T,)), grouped by <rel> into one file of C
channels (the name regex of lm_dataset_builder.py:79), next to ``codec_info.json``.  Outputs:
    <audio_path>/<rel>.wav                 16-bit PCM or 32-bit float, channels interleaved
    <audio_path>/manifest.json             file, channels, samples, crc32 of the data chunk, rank
    <audio_path>/errors.json               files that could not be decoded (the run goes on without them)

The job is a pipeline: loader threads read and range-check the .npy files into pinned host buffers, the copy stream
uploads file i+1 under the decode of file i, mc_op_f32_to_pcm stores the samples straight into pinned memory, and a
writer thread waits for them and writes tmp + rename.  Existing complete .wav files of the right length are skipped
(resume).  Under torchrun every rank decodes its duration-balanced share of the files and rank 0 writes the merged
manifest.
"""
from __future__ import annotations

import argparse
import json
import os
import queue
import re
import threading
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import audio_io, corpus
from .audio_to_codes import _PinnedPool, _atomic_write

NAME_RE = re.compile(r"(.+)_c(\d+)[_.]")                  # lm_dataset_builder.py:79
MODES = ("chunked", "render", "one_shot")
FORMATS = {"pcm16": audio_io.PCM_S16, "float": audio_io.PCM_F32}


class RefusedToStart(RuntimeError):
    """The codes directory does not belong to the loaded model; nothing was written."""


def read_codec_info(codes_path: str, gen) -> dict:
    path = os.path.join(codes_path, "codec_info.json")
    if not os.path.isfile(path):
        raise RefusedToStart(f"{path} is missing: --codes_path must be a directory written by audio_to_codes")
    with open(path) as f:
        info = json.load(f)
    want = {"codebook_size": gen.codebook_size, "sampling_rate": gen.sample_rate, "framerate": gen.sample_rate / gen.hop}
    for key, value in want.items():
        if key not in info or abs(float(info[key]) - float(value)) > 1e-9:
            raise RefusedToStart(f"codec_info.json has {key}={info.get(key)!r}, the loaded model has {value!r}")
    return info


def find_code_files(codes_path: str, filters: Optional[Sequence[str]] = None) -> Dict[str, Dict[int, str]]:
    """<rel> -> {channel: path} for every <rel>_c<channel>.npy under codes_path."""
    groups: Dict[str, Dict[int, str]] = {}
    for d, _, files in os.walk(codes_path):
        for f in files:
            if not f.endswith(".npy"):
                continue
            p = os.path.join(d, f)
            m = NAME_RE.match(os.path.relpath(p, codes_path))
            if m is None or (filters and not any(s in p for s in filters)):
                continue
            groups.setdefault(m.group(1), {})[int(m.group(2))] = p
    return dict(sorted(groups.items()))


def _frames_of(path: str) -> int:
    try:
        return int(np.load(path, mmap_mode="r").shape[-1])
    except Exception:                                               # noqa: BLE001  (reported when the file is loaded)
        return 0


def load_codes(paths: Dict[int, str], channels: int, codebook_size: int, alloc) -> Tuple[int, np.ndarray]:
    """Channel files -> (frames, int64 [channels, frames] in the buffer `alloc(nbytes)` returns).  Raises ValueError with
    the reason for a file the run has to skip."""
    if sorted(paths) != list(range(channels)):
        raise ValueError(f"channels {sorted(paths)} are not 0..{channels - 1}")
    arrays = []
    for c in range(channels):
        try:
            a = np.load(paths[c], allow_pickle=False)
        except Exception as ex:                                     # noqa: BLE001
            raise ValueError(f"{paths[c]}: unreadable ({ex!r})") from None
        if a.dtype not in (np.int16, np.int32, np.int64) or not (a.ndim == 1 or (a.ndim == 2 and a.shape[0] == 1)):
            raise ValueError(f"{paths[c]}: {a.dtype} array of shape {a.shape}; expected int16/32/64 of shape (1, T) or (T,)")
        arrays.append(a.reshape(-1))
    frames = arrays[0].shape[0]
    if any(a.shape[0] != frames for a in arrays):
        raise ValueError(f"channels of unequal length {[a.shape[0] for a in arrays]}")
    if frames == 0:
        raise ValueError("no codes")
    for c, a in enumerate(arrays):                                  # the engine clamps silently, F.embedding would raise
        lo, hi = int(a.min()), int(a.max())
        if lo < 0 or hi >= codebook_size:
            raise ValueError(f"{paths[c]}: codes in [{lo}, {hi}] outside [0, {codebook_size})")
    out = alloc(8 * channels * frames)[: 8 * channels * frames].view(np.int64).reshape(channels, frames)
    for c, a in enumerate(arrays):
        out[c] = a
    return frames, out


def decode_corpus(gen, codes_path: str, audio_path: str, mode: str = "chunked", chunk_size_secs: Optional[float] = None,
                  context_secs: Optional[float] = None, fade_secs: float = 0.02, target_rms: float = 0.0,
                  silence_rms_threshold: float = 0.003, fmt: str = "pcm16", batch_size: int = 256,
                  codes_filter: Optional[Sequence[str]] = None, rank: int = 0, world_size: int = 1, overwrite: bool = False,
                  loader_threads: int = 4, prefetch_files: int = 3, fuse_batches: int = 1, ingest=None,
                  stats: Optional[Dict[str, float]] = None) -> Tuple[List[dict], List[Dict[str, str]]]:
    """Decodes this rank's share of the code files.  Returns (manifest entries incl. resumed files, per-file errors).
    Raises RefusedToStart (before writing anything) when codec_info.json is missing or does not match `gen`.
    `ingest`: the staging interface (default audio_io.DeviceIngest(gen); the CPU tests pass a host stand-in)."""
    if mode not in MODES:
        raise ValueError(f"mode must be one of {MODES}")
    info = read_codec_info(codes_path, gen)
    chunk_size_secs = float(info.get("chunk_size_secs", 0.1) if chunk_size_secs is None else chunk_size_secs)
    context_secs = float(info.get("context_secs", 2.0) if context_secs is None else context_secs)
    if mode != "one_shot":
        corpus._chunk_frames(gen, chunk_size_secs)                 # reject a chunk that is not whole frames up front
    pcm_fmt = FORMATS[fmt]
    width = audio_io.BYTES_PER_SAMPLE[pcm_fmt]
    sr, hop = gen.sample_rate, gen.hop
    groups = find_code_files(codes_path, codes_filter)
    rels = list(groups)
    default_c = (2 if info["stereo"] else 1) if "stereo" in info else None

    cost = [len(groups[r]) * _frames_of(next(iter(groups[r].values()))) for r in rels]
    mine = corpus.shard_by_duration(cost, world_size)[rank]
    os.makedirs(audio_path, exist_ok=True)

    manifest: List[dict] = []
    errors: List[Dict[str, str]] = []
    todo = []
    for fid in mine:
        rel = rels[fid]
        dst = os.path.join(audio_path, rel + ".wav")
        channels = default_c or len(groups[rel])
        if not overwrite:
            frames = _frames_of(groups[rel].get(0, next(iter(groups[rel].values()))))
            have = audio_io.wav_info(dst)
            if frames > 0 and have == (sr, channels, pcm_fmt, frames * hop):   # resume: the entry comes back from disk
                with open(dst, "rb") as f:
                    f.seek(44)
                    crc = zlib.crc32(f.read()) & 0xFFFFFFFF
                manifest.append({"file": rel + ".wav", "channels": channels, "samples": frames * hop, "crc32": crc, "rank": rank})
                continue
        todo.append((fid, rel, dst, channels))

    if ingest is None:                                              # one per engine, reused by later runs in the process
        ingest = getattr(gen, "_corpus_ingest", None)
        if ingest is None:
            ingest = audio_io.DeviceIngest(gen)
            try:
                gen._corpus_ingest = ingest
            except AttributeError:
                pass
    pool = _PinnedPool(prefetch_files + 1, ingest.host_buffer)
    write_q: "queue.Queue" = queue.Queue(maxsize=4 * (prefetch_files + 1))
    lock = threading.Lock()

    def load(item):
        fid, rel, dst, channels = item
        holder = {"buf": None}

        def alloc(nbytes: int) -> np.ndarray:
            holder["buf"] = pool.acquire(nbytes, holder["buf"])
            return holder["buf"].numpy()

        try:
            frames, _ = load_codes(groups[rel], channels, gen.codebook_size, alloc)
            if frames * hop * channels * width > audio_io.WAV_MAX_DATA_BYTES:
                raise ValueError(f"{frames * hop * channels * width} bytes of audio exceed the 4 GiB RIFF limit")
            return item, frames, holder["buf"], None
        except Exception as ex_:                                    # noqa: BLE001  (the file goes to errors.json)
            if holder["buf"] is None:
                holder["buf"] = pool.acquire(1)
            return item, 0, holder["buf"], f"{rel}: {ex_}"

    def writer():
        while True:
            job = write_q.get()
            if job is None:
                return
            rel, dst, channels, pcm, wait = job
            try:
                wait()
                os.makedirs(os.path.dirname(dst) or ".", exist_ok=True)
                crc = {}
                _atomic_write(dst, lambda f: crc.setdefault("v", audio_io.write_wav(f, pcm, sr)))
                with lock:
                    manifest.append({"file": rel + ".wav", "channels": channels, "samples": int(pcm.shape[0]),
                                     "crc32": crc["v"], "rank": rank})
            except Exception as ex_:                                # noqa: BLE001
                with lock:
                    errors.append({"file": rel, "error": f"write failed: {ex_!r}"})
            finally:
                pcm = None
                release = getattr(wait, "release", None)
                if release is not None:
                    release()

    def decode(codes: torch.Tensor, channels: int) -> torch.Tensor:
        streams = [codes[c] for c in range(channels)]
        if mode == "chunked":
            return torch.stack(corpus.decode_streams(gen, streams, chunk_size_secs, context_secs, batch_size, fuse_batches))
        if mode == "render":
            return torch.stack(corpus.render_streams(gen, streams, chunk_size_secs, context_secs, fade_secs, target_rms,
                                                     silence_rms_threshold, batch_size, fuse_batches))
        return gen.decode(codes)

    wt = threading.Thread(target=writer, daemon=True)
    wt.start()
    decoded_secs = 0.0
    ex = ThreadPoolExecutor(max(1, loader_threads))
    try:
        inflight = []
        it = iter(todo)
        for _ in range(prefetch_files + 1):
            nxt = next(it, None)
            if nxt is not None:
                inflight.append(ex.submit(load, nxt))
        while inflight:
            item, frames, buf, err = inflight.pop(0).result()
            fid, rel, dst, channels = item
            if err is None:
                staged = ingest.upload_codes(buf, 8 * channels * frames)   # copy stream: under the previous file's decode
                try:
                    wav = decode(ingest.codes_on_device(staged, channels, frames), channels)
                except Exception as ex_:                            # noqa: BLE001  (e.g. one_shot beyond the single-call limit)
                    err = f"{rel}: decode failed: {ex_}"
                else:
                    pcm, wait = ingest.pcm_to_host(wav, pcm_fmt)
                    decoded_secs += channels * frames * hop / float(sr)
                    write_q.put((rel, dst, channels, pcm, wait))
                ingest.wait_uploaded(staged)
            if err is not None:
                with lock:
                    errors.append({"file": rel, "error": err})
            pool.release(buf)
            nxt = next(it, None)
            if nxt is not None:
                inflight.append(ex.submit(load, nxt))
    finally:
        ex.shutdown(wait=True, cancel_futures=True)
        write_q.put(None)
        wt.join()
        if hasattr(ingest, "recycle"):
            for b in pool.drain():
                ingest.recycle(b)
    if stats is not None:
        stats["decoded_audio_secs"] = stats.get("decoded_audio_secs", 0.0) + decoded_secs
    manifest.sort(key=lambda e: e["file"])
    return manifest, errors


def main(argv: Optional[Sequence[str]] = None) -> None:
    ap = argparse.ArgumentParser(prog="python -m rca_b200_loader codes_to_audio", description=__doc__.split("\n\n")[0])
    ap.add_argument("--codes_path", required=True, help="directory holding codec_info.json (audio_to_codes output)")
    ap.add_argument("--audio_path", required=True, help="output root for the .wav files")
    ap.add_argument("--mode", choices=MODES, default="chunked")
    ap.add_argument("--chunk_size_secs", type=float, default=None, help="default: codec_info.json")
    ap.add_argument("--context_secs", type=float, default=None, help="default: codec_info.json")
    ap.add_argument("--fade_secs", type=float, default=0.02, help="render only")
    ap.add_argument("--target_rms", type=float, default=0.0, help="render only; 0 = no normalisation")
    ap.add_argument("--silence_rms_threshold", type=float, default=0.003, help="render only")
    ap.add_argument("--format", choices=tuple(FORMATS), default="pcm16")
    ap.add_argument("--batch_size", type=int, default=256)
    ap.add_argument("--codec_model", default="MagiCodec-50Hz-Base")
    ap.add_argument("--codes_filter", nargs="+")
    ap.add_argument("--overwrite", action="store_true")
    ap.add_argument("--loader_threads", type=int, default=4)
    ap.add_argument("--prefetch_files", type=int, default=3)
    args = ap.parse_args(argv)

    import torch.distributed as dist
    from .audio_tokenizer import load_magicodec_model

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gen = load_magicodec_model(args.codec_model, dev)[0]
    try:
        local_manifest, local_errors = decode_corpus(
            gen, args.codes_path, args.audio_path, args.mode, args.chunk_size_secs, args.context_secs, args.fade_secs,
            args.target_rms, args.silence_rms_threshold, args.format, args.batch_size, args.codes_filter, rank, world,
            overwrite=args.overwrite, loader_threads=args.loader_threads, prefetch_files=args.prefetch_files)
    except RefusedToStart as ex:
        raise SystemExit(f"codes_to_audio: {ex}") from None
    merged = sorted(corpus.gather_objects(local_manifest, dev), key=lambda e: e["file"])
    all_errors = corpus.gather_objects(local_errors, dev)
    if rank == 0:
        _atomic_write(os.path.join(args.audio_path, "manifest.json"), lambda f: f.write(json.dumps(merged, indent=1).encode()))
        _atomic_write(os.path.join(args.audio_path, "errors.json"), lambda f: f.write(json.dumps(all_errors, indent=1).encode()))
        print(f"decoded {len(merged)} files -> {args.audio_path}" + (f"; {len(all_errors)} file(s) skipped, see errors.json" if all_errors else ""))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
