"""Offline corpus encode: the ``python -m codec_bpe.audio_to_codes --chunk_size_secs 0.1
--context_secs 2.0 --batch_size 256`` path of /root/reference/encode_audio_gpu_1.sh:1-8 (and
encode_audio_stereo.sh), whose per-file semantics are pinned in-tree by
``AudioTokenizer.chunked_tokenize_audio`` (audio_tokenizer.py:52-65, used for exactly this purpose at
realtime_agent_v2.py:77).

Every 0.1 s chunk is encoded from the trailing 2.0 s of context ending at that chunk, and only the
chunk's own frames are kept.  Here all steady-state windows of a stream are read through ONE
overlapping strided view of the audio already in HBM (row stride = chunk samples), so the 20x
window amplification never exists in memory; warm-up windows (shorter context at the start of a
file) and a ragged last chunk are batched across streams by shape.

Multi-GPU: files are partitioned by duration (longest-processing-time first) across ranks, each
rank encodes its shard with no communication, then per-rank manifests are all-gathered (NCCL on
GPUs, gloo in the CPU tests) — SURVEY.md §8(e).
"""
from __future__ import annotations

import json
import zlib
from dataclasses import asdict, dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch


@dataclass(frozen=True)
class Window:
    start: int      # first sample of the context window
    length: int     # samples in the window
    keep: int       # frames kept (0 never occurs here: the [-0:] quirk is resolved to "all frames")
    chunk: int      # chunk index inside the stream


def plan_stream(n_samples: int, chunk_samples: int, context_samples: int, sample_rate: int, framerate: float,
                hop: int) -> Tuple[List[Window], Optional[Tuple[int, int, int]]]:
    """Windows of one mono stream under chunked_tokenize_audio semantics.

    Returns (irregular windows, steady) where steady = (first_chunk, count, keep) describes the run of
    full-context, full-chunk windows  start = (first_chunk + j + 1) * chunk - context, j < count.
    """
    irregular: List[Window] = []
    n_chunks = -(-n_samples // chunk_samples) if n_samples > 0 else 0
    steady_first, steady_count, steady_keep = None, 0, 0
    for i in range(n_chunks):
        end = min((i + 1) * chunk_samples, n_samples)
        n_new = end - i * chunk_samples
        ctx = max(n_new, context_samples)                      # audio_tokenizer.py:74
        start = max(0, end - ctx)
        length = end - start
        frames = -(-length // hop)
        keep = int(n_new / sample_rate * framerate)            # :99-100 (mono: num_channels == 1 per stream)
        if keep <= 0 or keep > frames:
            keep = frames                                      # :101 — s[-0:] is the whole string
        if n_new == chunk_samples and length == context_samples and start == end - context_samples:
            if steady_first is None:
                steady_first, steady_keep = i, keep
            steady_count += 1
        else:
            irregular.append(Window(start, length, keep, i))
    steady = (steady_first, steady_count, steady_keep) if steady_first is not None else None
    return irregular, steady


def encode_streams(gen, streams: Sequence[torch.Tensor], chunk_secs: float = 0.1, context_secs: float = 2.0,
                   batch_size: int = 256, fuse_batches: int = 1, causal_warmup: bool = True) -> List[torch.Tensor]:
    """Encode mono streams (1-D fp32 device tensors) -> one int64 code tensor per stream.

    ``batch_size`` is the reference CLI's windows-per-forward flag.  Per-window results do not depend on
    how windows are grouped into launches (tested bit-exact), so ``fuse_batches`` consecutive batches may
    be issued as ONE engine call: fewer, larger launches quantise better onto 74 CTA pairs.

    ``causal_warmup``: the warm-up windows of a stream (chunks 0..18 at the default sizes: context shorter than
    2.0 s) all start at sample 0, so each is a PREFIX of the longest one.  The network is causal end to end
    (causal convs, causal windowed attention, window-relative RoPE), so frame t of a prefix equals frame t of the
    longer window: ONE full-frame encode of the longest warm-up window yields every warm-up chunk's codes instead
    of 19 launches of growing length per stream.  On the engine this is bit-identical (masked keys add exact
    zeros; tested on the GPU against ``causal_warmup=False``).  The shortcut is only taken when the spec really is
    causal (``window_right == 0``): with any look-ahead a prefix frame would attend to audio beyond its own window,
    so such specs go through the per-window path."""
    batch_size = batch_size * max(1, int(fuse_batches))
    causal_warmup = causal_warmup and int(getattr(getattr(gen, "spec", None), "window_right", 0)) == 0
    sr, hop = gen.sample_rate, gen.hop
    framerate = sr / hop
    chunk = int(chunk_secs * sr)
    context = int(context_secs * sr)
    plans = [plan_stream(int(s.numel()), chunk, context, sr, framerate, hop) for s in streams]
    # chunk -> (codes tensor) per stream, assembled at the end in chunk order
    pieces: List[Dict[int, torch.Tensor]] = [dict() for _ in streams]

    # steady state: one overlapping strided view per stream, `batch_size` windows per launch
    for si, (s, (_, steady)) in enumerate(zip(streams, plans)):
        if steady is None:
            continue
        first, count, keep = steady
        base = (first + 1) * chunk - context
        flat = s if s.is_contiguous() else s.contiguous()
        for b0 in range(0, count, batch_size):
            nb = min(batch_size, count - b0)
            view = flat[base + b0 * chunk:]
            codes = gen.encode(view, keep_last_frames=keep, row_stride=chunk, num_windows=nb, window_samples=context)
            pieces[si][first + b0] = codes.reshape(-1)          # consecutive chunks, already in order

    # warm-up windows as prefixes of the longest one (see docstring)
    done: List[set] = [set() for _ in streams]
    if causal_warmup and chunk % hop == 0:
        cf = chunk // hop
        prefix_groups: Dict[int, List[Tuple[int, List[Window]]]] = {}
        for si, (irr, _) in enumerate(plans):
            warm = [w for w in irr if w.start == 0 and w.length == (w.chunk + 1) * chunk and w.keep == cf]
            if len(warm) >= 2:
                prefix_groups.setdefault(max(w.length for w in warm), []).append((si, warm))
        for length, items in prefix_groups.items():
            for b0 in range(0, len(items), batch_size):
                part = items[b0:b0 + batch_size]
                batch = torch.stack([streams[si][:length] for si, _ in part])
                codes = gen.encode(batch, keep_last_frames=0)                      # every frame of the longest prefix
                for row, (si, warm) in enumerate(part):
                    for w in warm:
                        pieces[si][w.chunk] = codes[row, (w.chunk + 1) * cf - w.keep:(w.chunk + 1) * cf]
                        done[si].add(w.chunk)

    # remaining warm-up / ragged windows: group across streams by (length, keep)
    groups: Dict[Tuple[int, int], List[Tuple[int, Window]]] = {}
    for si, (irr, _) in enumerate(plans):
        for w in irr:
            if w.chunk not in done[si]:
                groups.setdefault((w.length, w.keep), []).append((si, w))
    for (length, keep), items in groups.items():
        for b0 in range(0, len(items), batch_size):
            part = items[b0:b0 + batch_size]
            batch = torch.stack([streams[si][w.start:w.start + length] for si, w in part])
            codes = gen.encode(batch, keep_last_frames=keep)
            for row, (si, w) in enumerate(part):
                pieces[si][w.chunk] = codes[row]

    out = []
    for si in range(len(streams)):
        if not pieces[si]:
            out.append(torch.empty(0, dtype=torch.int64, device=gen.device))
            continue
        out.append(torch.cat([pieces[si][k] for k in sorted(pieces[si])]))
    return out


# --------------------------------------------------------------------------------- decode
@dataclass(frozen=True)
class DecodeWindow:
    start_frame: int    # first frame of the code context window
    frames: int         # frames in the window
    keep_samples: int   # decoded samples kept: the last min(new * hop + preroll, frames * hop)
    chunk: int          # chunk index inside the stream


def plan_decode_stream(n_frames: int, chunk_frames: int, context_frames: int, preroll_samples: int,
                       hop: int) -> Tuple[List[DecodeWindow], Optional[Tuple[DecodeWindow, int]]]:
    """Windows of one code stream under the bookkeeping of a detokenize_audio loop that starts from an empty context
    (audio_tokenizer.py:105-113): chunk i is decoded from the last max(n_new, context_frames) frames ending at it, and
    the last n_new * hop + preroll samples (at most the whole window) are kept.

    Returns (irregular windows, steady) where steady = (first window, count) describes the run of full-context,
    full-chunk windows  start_frame = (first.chunk + j + 1) * chunk_frames - first.frames, j < count."""
    irregular: List[DecodeWindow] = []
    n_chunks = -(-n_frames // chunk_frames) if n_frames > 0 else 0
    full = max(chunk_frames, context_frames)
    steady_first, steady_count = None, 0
    for i in range(n_chunks):
        end = min((i + 1) * chunk_frames, n_frames)
        n_new = end - i * chunk_frames
        start = max(0, end - max(n_new, context_frames))
        w = DecodeWindow(start, end - start, min(n_new * hop + preroll_samples, (end - start) * hop), i)
        if n_new == chunk_frames and w.frames == full:
            if steady_first is None:
                steady_first = w
            steady_count += 1
        else:
            irregular.append(w)
    return irregular, ((steady_first, steady_count) if steady_first is not None else None)


def _chunk_frames(gen, chunk_secs: float) -> int:
    exact = chunk_secs * gen.sample_rate / gen.hop
    cf = int(round(exact))
    if cf < 1 or abs(exact - cf) > 1e-6:
        raise ValueError(f"chunk_secs={chunk_secs} is {exact} frames; the chunked decode needs a whole number >= 1")
    return cf


def _decode_windows(gen, code_streams: Sequence[torch.Tensor], cf: int, context_frames: int, preroll: int,
                    batch_size: int, causal_warmup: bool, sink) -> None:
    """Decodes every planned window of every stream; sink(stream, first_chunk, wav [n, keep]) receives the kept samples
    of n consecutive chunks."""
    hop = gen.hop
    causal_warmup = causal_warmup and int(getattr(getattr(gen, "spec", None), "window_right", 0)) == 0
    plans = [plan_decode_stream(int(s.numel()), cf, context_frames, preroll, hop) for s in code_streams]

    # steady state: the overlapping windows of a stream as an unfolded view, materialised per launch by gen.decode
    for si, (s, (_, steady)) in enumerate(zip(code_streams, plans)):
        if steady is None:
            continue
        first, count = steady
        base = first.start_frame
        view = s[base: base + (count - 1) * cf + first.frames].unfold(0, first.frames, cf)        # [count, frames]
        for b0 in range(0, count, batch_size):
            nb = min(batch_size, count - b0)
            sink(si, first.chunk + b0, gen.decode(view[b0:b0 + nb], keep_last_samples=first.keep_samples))

    # warm-up windows (start_frame 0) as prefixes of the longest one: the decoder is causal end to end (causal windowed
    # attention, causal transposed convolutions, window-relative RoPE), so sample t of a prefix's output equals sample t
    # of the longer window's; one full decode per stream replaces up to context/chunk launches of growing length
    done: List[set] = [set() for _ in code_streams]
    if causal_warmup:
        prefix_groups: Dict[int, List[Tuple[int, List[DecodeWindow]]]] = {}
        for si, (irr, _) in enumerate(plans):
            warm = [w for w in irr if w.start_frame == 0]
            if len(warm) >= 2:
                prefix_groups.setdefault(max(w.frames for w in warm), []).append((si, warm))
        for frames, items in prefix_groups.items():
            for b0 in range(0, len(items), batch_size):
                part = items[b0:b0 + batch_size]
                wav = gen.decode(torch.stack([code_streams[si][:frames] for si, _ in part]), keep_last_samples=0)
                for row, (si, warm) in enumerate(part):
                    for w in warm:
                        end = w.frames * hop
                        sink(si, w.chunk, wav[row:row + 1, end - w.keep_samples:end])
                        done[si].add(w.chunk)

    # remaining warm-up / ragged windows: grouped across streams by (frames, keep)
    groups: Dict[Tuple[int, int], List[Tuple[int, DecodeWindow]]] = {}
    for si, (irr, _) in enumerate(plans):
        for w in irr:
            if w.chunk not in done[si]:
                groups.setdefault((w.frames, w.keep_samples), []).append((si, w))
    for (frames, keep), items in groups.items():
        for b0 in range(0, len(items), batch_size):
            part = items[b0:b0 + batch_size]
            wav = gen.decode(torch.stack([code_streams[si][w.start_frame:w.start_frame + frames] for si, w in part]),
                             keep_last_samples=keep)
            for row, (si, w) in enumerate(part):
                sink(si, w.chunk, wav[row:row + 1])


def decode_streams(gen, code_streams: Sequence[torch.Tensor], chunk_secs: float = 0.1, context_secs: float = 2.0,
                   batch_size: int = 256, fuse_batches: int = 1, causal_warmup: bool = True) -> List[torch.Tensor]:
    """Chunked decode of code streams (1-D int64 device tensors) -> one fp32 waveform per stream: exactly what a loop
    of AudioTokenizer.detokenize_audio over chunk_secs pieces returns when it starts from an empty context.  The twin
    of encode_streams: steady windows `batch_size * fuse_batches` per engine call, warm-up chunks from ONE decode of
    the longest warm-up prefix (causal specs only, ``window_right == 0``; any look-ahead takes the per-window path),
    the rest grouped across streams by shape."""
    cf = _chunk_frames(gen, chunk_secs)
    context_frames = int(context_secs * gen.sample_rate / gen.hop)
    pieces: List[Dict[int, torch.Tensor]] = [dict() for _ in code_streams]

    def sink(si, first, wav):
        pieces[si][first] = wav.reshape(-1)

    _decode_windows(gen, code_streams, cf, context_frames, 0, batch_size * max(1, int(fuse_batches)), causal_warmup, sink)
    return [torch.cat([p[k] for k in sorted(p)]) if p else torch.empty(0, dtype=torch.float32, device=gen.device)
            for p in pieces]


def render_streams(gen, code_streams: Sequence[torch.Tensor], chunk_secs: float = 0.1, context_secs: float = 2.0,
                   fade_secs: float = 0.02, target_rms: float = 0.0, silence_rms_threshold: float = 0.003,
                   batch_size: int = 256, fuse_batches: int = 1, causal_warmup: bool = True) -> List[torch.Tensor]:
    """The agent's recording of each code stream: every chunk after the first decoded with preroll_samples = L, then
    pad_or_trim -> normalize_audio_rms (target_rms > 0) -> smooth_join, i.e. np.concatenate(audio_history_ch1) of an
    OutputChunkEmitter fed the chunk strings in order (the emitted stream shifted left by L), frames * hop samples long.
    Windows are decoded as in decode_streams, gathered into one [n_chunks, chunk + L] matrix per stream, and the whole
    crossfade chain is one render_chunks launch per stream."""
    from .audio_utils import create_crossfade_ramps
    cf = _chunk_frames(gen, chunk_secs)
    chunk = cf * gen.hop
    context_frames = int(context_secs * gen.sample_rate / gen.hop)
    L, fade_in, _ = create_crossfade_ramps(gen.sample_rate, fade_secs)
    if not 0 < L <= chunk:
        raise ValueError(f"fade_secs={fade_secs} gives {L} fade samples; the render needs 0 < fade <= chunk ({chunk})")
    mats = [torch.zeros((-(-int(s.numel()) // cf), chunk + L), dtype=torch.float32, device=gen.device) for s in code_streams]

    def sink(si, first, wav):
        mats[si][first:first + wav.shape[0], :wav.shape[1]] = wav

    _decode_windows(gen, code_streams, cf, context_frames, L, batch_size * max(1, int(fuse_batches)), causal_warmup, sink)
    ramp = torch.from_numpy(fade_in).to(gen.device)
    out = []
    for s, m in zip(code_streams, mats):
        n = int(s.numel())
        if n == 0:
            out.append(torch.empty(0, dtype=torch.float32, device=gen.device))
            continue
        last_len = (n - (m.shape[0] - 1) * cf) * gen.hop
        out.append(gen.render_chunks(m, chunk, ramp, last_len=last_len, target_rms=target_rms,
                                     silence_rms_threshold=silence_rms_threshold))
    return out


# ------------------------------------------------------------------------------- sharding
def shard_by_duration(durations: Sequence[float], world_size: int) -> List[List[int]]:
    """Longest-processing-time-first partition; deterministic (ties by index)."""
    order = sorted(range(len(durations)), key=lambda i: (-durations[i], i))
    loads = [0.0] * world_size
    shards: List[List[int]] = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: (loads[k], k))
        shards[r].append(i)
        loads[r] += durations[i]
    return [sorted(s) for s in shards]


@dataclass
class ManifestEntry:
    file_id: int
    channel: int
    n_frames: int
    n_windows: int
    crc32: int
    rank: int
    path: str = ""          # file path relative to --audio_path, without extension (the CLI fills it in)


def manifest_entry(file_id: int, channel: int, codes: torch.Tensor, n_windows: int, rank: int) -> ManifestEntry:
    raw = codes.detach().cpu().numpy().astype("<i4").tobytes()
    return ManifestEntry(file_id, channel, int(codes.numel()), n_windows, zlib.crc32(raw) & 0xFFFFFFFF, rank)


def gather_objects(local: list, device: Optional[torch.device] = None) -> list:
    """all_gather of one JSON-serialisable list per rank, concatenated in rank order: lengths first, then zero-padded
    byte buffers (two small collectives; NCCL over NVLink on GPUs, gloo in the CPU tests)."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return list(local)
    world = dist.get_world_size()
    backend = dist.get_backend()
    dev = device if (device is not None and backend == "nccl") else torch.device("cpu")
    payload = json.dumps(local).encode()
    n = torch.tensor([len(payload)], dtype=torch.int64, device=dev)
    sizes = torch.zeros(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(sizes, n)
    sizes = sizes.cpu().tolist()                                   # one D2H for all ranks' lengths
    cap = max(1, int(max(sizes)))
    buf = torch.zeros(cap, dtype=torch.uint8, device=dev)
    if payload:
        buf[: len(payload)] = torch.frombuffer(bytearray(payload), dtype=torch.uint8).to(dev)
    bufs = torch.zeros(world * cap, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(bufs, buf)
    host = bufs.cpu().numpy().reshape(world, cap)
    merged = []
    for r in range(world):
        merged.extend(json.loads(host[r, : int(sizes[r])].tobytes().decode()))
    return merged


def gather_manifests(local: List[ManifestEntry], device: Optional[torch.device] = None) -> List[ManifestEntry]:
    """all_gather of per-rank manifests (two small collectives per corpus run; no collective touches the data path)."""
    merged = [ManifestEntry(**d) for d in gather_objects([asdict(e) for e in local], device)]
    merged.sort(key=lambda e: (e.file_id, e.channel))
    return merged


def codes_to_array(codes: torch.Tensor) -> np.ndarray:
    """On-disk shape of one stream: (num_codebooks=1, T) — lm_dataset_builder.py:404-408 accepts rank
    2-4 with trailing (num_codebooks, T); tools/total_duration_codes.py:8 reads shape[-1] as frames."""
    return codes.detach().cpu().numpy().astype(np.int32)[None, :]
