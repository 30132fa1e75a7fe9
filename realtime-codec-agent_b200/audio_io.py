"""Audio ingest for the offline corpus encode (SURVEY.md §8 f1) and for
``AudioTokenizer._prep_audio_for_tokenization`` (audio_tokenizer.py:203-215).

The reference's loader is librosa (soundfile / audioread underneath) and its corpora are wav, flac (libri-light) and
sph -> mp3 telephone speech (tools/sph_to_mp3.py, prep_channel_map.py:7-8 ``SUPPORTED_EXTENSIONS``).  None of those
libraries exists in the offline image, so containers are parsed here:

    .wav / .wave   RIFF / RIFX / RF64: PCM 8/16/24/32, IEEE float 32/64, G.711 mu-law / A-law, WAVE_FORMAT_EXTENSIBLE
    .sph           NIST SPHERE: pcm (either byte order), ulaw, alaw (shorten-compressed files need sph2pipe, as upstream)
    .flac          native decoder in libmagicodec_b200.so (csrc/audio_decode.cpp), CRC-checked
    .npy           raw arrays [T] or [C,T]
    .mp3 .ogg .opus .m4a   torchaudio(+torchcodec), soundfile or an ffmpeg binary when one is present; otherwise a
                   per-file ``UnsupportedAudio`` that the CLI records and skips (never a run-level failure)

``read_audio`` stops at the container's PCM payload (1-2 bytes per sample for the telephone corpora): sample
conversion, mono mix and resampling to 16 kHz run ON THE DEVICE in the corpus path (``DeviceIngest``; kernels
``pcm_to_f32_kernel`` / ``resample_poly_kernel``).  ``load_audio`` is the host-side equivalent (numpy + scipy polyphase
with the same filter taps) for callers that want an array, like ``librosa.load``.
"""
from __future__ import annotations

import functools
import math
import os
import shutil
import struct
import subprocess
import zlib
from dataclasses import dataclass
from typing import Callable, Optional, Tuple

import numpy as np

PCM_U8, PCM_S16, PCM_S24, PCM_S32, PCM_F32, PCM_F64, PCM_ULAW, PCM_ALAW = range(8)
BYTES_PER_SAMPLE = {PCM_U8: 1, PCM_S16: 2, PCM_S24: 3, PCM_S32: 4, PCM_F32: 4, PCM_F64: 8, PCM_ULAW: 1, PCM_ALAW: 1}

SUPPORTED_EXTENSIONS = (".wav", ".wave", ".npy", ".flac", ".mp3", ".ogg", ".opus", ".m4a", ".sph")


class UnsupportedAudio(RuntimeError):
    """This file cannot be decoded in this environment (the run continues without it)."""


@dataclass
class PcmAudio:
    sample_rate: int
    channels: int
    frames: int
    fmt: int                 # PCM_* (== MC_PCM_* of the C ABI)
    big_endian: bool
    payload: np.ndarray      # uint8, interleaved frames [frames][channels] in `fmt`

    @property
    def duration(self) -> float:
        return self.frames / float(self.sample_rate)


Alloc = Callable[[int], np.ndarray]       # nbytes -> writable uint8 array (e.g. a view of pinned host memory)


def _default_alloc(nbytes: int) -> np.ndarray:
    return np.empty(nbytes, dtype=np.uint8)


# ------------------------------------------------------------------------------------- WAV
_WAVE_TAGS = {1: "pcm", 3: "float", 6: "alaw", 7: "ulaw"}


def _wav_header(f) -> Tuple[int, int, int, int, bool, int, int]:
    """-> (sample_rate, channels, fmt, frames, big_endian, data_offset, data_bytes)"""
    head = f.read(12)
    if len(head) < 12 or head[:4] not in (b"RIFF", b"RIFX", b"RF64") or head[8:12] != b"WAVE":
        raise UnsupportedAudio("not a RIFF/WAVE file")
    big = head[:4] == b"RIFX"
    en = ">" if big else "<"
    rf64 = head[:4] == b"RF64"
    fmt_info, data64 = None, None
    file_size = os.fstat(f.fileno()).st_size
    while True:
        ck = f.read(8)
        if len(ck) < 8:
            raise UnsupportedAudio("no data chunk")
        cid, size = ck[:4], struct.unpack(en + "I", ck[4:])[0]
        if cid == b"ds64":
            body = f.read(size)
            data64 = struct.unpack("<Q", body[8:16])[0]
        elif cid == b"fmt ":
            body = f.read(size)
            tag, ch, sr, _, align, bits = struct.unpack(en + "HHIIHH", body[:16])
            if tag == 0xFFFE and size >= 26:
                tag = struct.unpack(en + "H", body[24:26])[0]
            fmt_info = (tag, ch, sr, align, bits)
        elif cid == b"data":
            if fmt_info is None:
                raise UnsupportedAudio("data chunk before fmt chunk")
            off = f.tell()
            if rf64 and size == 0xFFFFFFFF and data64 is not None:
                size = data64
            if size == 0 or size == 0xFFFFFFFF or off + size > file_size:
                size = file_size - off                      # streamed / truncated header: take what is there
            tag, ch, sr, align, bits = fmt_info
            kind = _WAVE_TAGS.get(tag)
            if kind == "pcm" and bits in (8, 16, 24, 32):
                fmt = {8: PCM_U8, 16: PCM_S16, 24: PCM_S24, 32: PCM_S32}[bits]
            elif kind == "float" and bits in (32, 64):
                fmt = PCM_F32 if bits == 32 else PCM_F64
            elif kind == "alaw" and bits == 8:
                fmt = PCM_ALAW
            elif kind == "ulaw" and bits == 8:
                fmt = PCM_ULAW
            else:
                raise UnsupportedAudio(f"WAVE format tag {tag:#x} with {bits} bits per sample")
            if ch < 1 or sr < 1:
                raise UnsupportedAudio("bad fmt chunk")
            frame_bytes = BYTES_PER_SAMPLE[fmt] * ch
            return sr, ch, fmt, size // frame_bytes, big, off, (size // frame_bytes) * frame_bytes
        else:
            f.seek(size, os.SEEK_CUR)
        if size & 1:
            f.seek(1, os.SEEK_CUR)


def _read_wav(path: str, alloc: Alloc) -> PcmAudio:
    with open(path, "rb") as f:
        sr, ch, fmt, frames, big, off, nbytes = _wav_header(f)
        buf = alloc(nbytes)
        f.seek(off)
        got = f.readinto(memoryview(buf)[:nbytes])
        if got != nbytes:
            raise UnsupportedAudio("short read")
    return PcmAudio(sr, ch, frames, fmt, big, buf[:nbytes])


WAV_MAX_DATA_BYTES = 0xFFFFFFFF - 36          # RIFF sizes are 32-bit; RF64 is not written


def wav_header(sample_rate: int, channels: int, fmt: int, frames: int) -> bytes:
    """44-byte canonical RIFF/WAVE header for interleaved PCM_S16 (format tag 1) or PCM_F32 (format tag 3) data."""
    if fmt not in (PCM_S16, PCM_F32):
        raise ValueError("write_wav writes 16-bit PCM or 32-bit float only")
    width = BYTES_PER_SAMPLE[fmt]
    data = frames * channels * width
    if data > WAV_MAX_DATA_BYTES:
        raise ValueError(f"{data} bytes of audio exceed the 4 GiB RIFF limit")
    return (b"RIFF" + struct.pack("<I", 36 + data) + b"WAVE"
            + b"fmt " + struct.pack("<IHHIIHH", 16, 1 if fmt == PCM_S16 else 3, channels, sample_rate,
                                    sample_rate * channels * width, channels * width, 8 * width)
            + b"data" + struct.pack("<I", data))


def write_wav(f, pcm: np.ndarray, sample_rate: int) -> int:
    """Write interleaved audio [frames, channels] (or [frames]) of dtype int16 or float32 as a .wav file to the binary
    file object `f`.  Returns the crc32 of the data chunk."""
    pcm = np.ascontiguousarray(pcm)
    if pcm.dtype not in (np.int16, np.float32):
        raise ValueError("write_wav writes int16 or float32 samples")
    frames, channels = (pcm.shape[0], 1) if pcm.ndim == 1 else pcm.shape
    body = pcm.astype(pcm.dtype.newbyteorder("<"), copy=False).reshape(-1).view(np.uint8)
    f.write(wav_header(sample_rate, channels, PCM_S16 if pcm.dtype == np.int16 else PCM_F32, frames))
    f.write(body)
    return zlib.crc32(body) & 0xFFFFFFFF


def wav_info(path: str) -> Optional[Tuple[int, int, int, int]]:
    """(sample_rate, channels, fmt, frames) of a complete .wav file, or None when it is missing, unreadable or shorter
    than its header says."""
    try:
        with open(path, "rb") as f:
            head = f.read(44)
            f.seek(0)
            sr, ch, fmt, frames, _, off, nbytes = _wav_header(f)
        declared = struct.unpack("<I", head[40:44])[0] if head[36:40] == b"data" else nbytes
        if declared != nbytes or off + nbytes > os.path.getsize(path):
            return None
        return sr, ch, fmt, frames
    except (OSError, UnsupportedAudio, struct.error):
        return None


# ------------------------------------------------------------------------------ NIST SPHERE
def _sph_header(f):
    first = f.read(16)
    if not first.startswith(b"NIST_1A"):
        raise UnsupportedAudio("not a NIST SPHERE file")
    hsize = int(first[8:16].split()[0])
    f.seek(0)
    text = f.read(hsize).decode("latin-1")
    fields = {}
    for line in text.split("\n")[2:]:
        if line.startswith("end_head"):
            break
        parts = line.split(None, 2)
        if len(parts) == 3:
            fields[parts[0]] = parts[2].strip() if parts[1].startswith("-s") else parts[2].split()[0]
    coding = fields.get("sample_coding", "pcm").lower()
    if "shorten" in coding or "wavpack" in coding:
        raise UnsupportedAudio(f"SPHERE sample_coding '{coding}' is compressed: run sph2pipe first (tools/sph_to_mp3.py does the same upstream)")
    nbytes = int(fields.get("sample_n_bytes", 2))
    ch = int(fields.get("channel_count", 1))
    sr = int(fields["sample_rate"])
    big = fields.get("sample_byte_format", "01") == "10"
    if coding.startswith("ulaw") or coding.startswith("mu-law"):
        fmt = PCM_ULAW
    elif coding.startswith("alaw"):
        fmt = PCM_ALAW
    elif coding.startswith("pcm") and nbytes in (1, 2, 3, 4):
        fmt = {1: PCM_U8, 2: PCM_S16, 3: PCM_S24, 4: PCM_S32}[nbytes]
    else:
        raise UnsupportedAudio(f"SPHERE sample_coding '{coding}' / {nbytes} bytes per sample")
    size = os.fstat(f.fileno()).st_size - hsize
    frame_bytes = BYTES_PER_SAMPLE[fmt] * ch
    frames = size // frame_bytes
    if "sample_count" in fields:
        frames = min(frames, int(fields["sample_count"]))
    return sr, ch, fmt, frames, big, hsize


def _read_sph(path: str, alloc: Alloc) -> PcmAudio:
    with open(path, "rb") as f:
        sr, ch, fmt, frames, big, off = _sph_header(f)
        nbytes = frames * ch * BYTES_PER_SAMPLE[fmt]
        buf = alloc(nbytes)
        f.seek(off)
        if f.readinto(memoryview(buf)[:nbytes]) != nbytes:
            raise UnsupportedAudio("short read")
    return PcmAudio(sr, ch, frames, fmt, big, buf[:nbytes])


# -------------------------------------------------------------------------------------- FLAC
def _flac_lib():
    from . import _native
    return _native.load_library()


def _flac_info(data: np.ndarray):
    import ctypes as C
    sr, ch, bits, total = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    rc = _flac_lib().mc_flac_info(data.ctypes.data, data.size, C.byref(sr), C.byref(ch), C.byref(bits), C.byref(total))
    if rc != 0:
        raise UnsupportedAudio("not a FLAC stream (no fLaC marker / STREAMINFO)")
    return sr.value, ch.value, bits.value, total.value


def _read_flac(path: str, alloc: Alloc) -> PcmAudio:
    import ctypes as C
    data = np.fromfile(path, dtype=np.uint8)
    sr, ch, bits, total = _flac_info(data)
    if total <= 0:
        raise UnsupportedAudio("FLAC stream without a sample count in STREAMINFO")
    width = 2 if bits <= 16 else 4
    buf = alloc(total * ch * width)
    got = C.c_int64()
    rc = _flac_lib().mc_flac_decode(data.ctypes.data, data.size, buf.ctypes.data, total, C.byref(got))
    if rc != 0:
        raise UnsupportedAudio(f"FLAC decode failed after {got.value} of {total} frames (corrupt or truncated file)")
    return PcmAudio(sr, ch, total, PCM_S16 if width == 2 else PCM_S32, False, buf[: total * ch * width])


# ------------------------------------------------------------------------------ other formats
def _from_planar_float(arr: np.ndarray, sr: int, alloc: Alloc) -> PcmAudio:
    arr = np.asarray(arr)
    if arr.ndim == 1:
        arr = arr[None]
    ch, frames = arr.shape
    inter = np.ascontiguousarray(arr.T, dtype=np.float32)               # [frames][channels]
    buf = alloc(inter.nbytes)
    buf[: inter.nbytes] = inter.view(np.uint8).reshape(-1)
    return PcmAudio(int(sr), ch, frames, PCM_F32, False, buf[: inter.nbytes])


def _read_npy(path: str, alloc: Alloc, default_sr: int) -> PcmAudio:
    arr = np.load(path)
    if np.issubdtype(arr.dtype, np.integer):
        arr = arr.astype(np.float32) / float(np.iinfo(arr.dtype).max + 1)
    return _from_planar_float(arr, default_sr, alloc)


def _read_external(path: str, alloc: Alloc) -> PcmAudio:
    """Compressed lossy containers: whatever decoder the deployment has."""
    errors = []
    try:
        import torchaudio
        wav, sr = torchaudio.load(path)
        return _from_planar_float(wav.numpy(), sr, alloc)
    except Exception as ex:                                          # noqa: BLE001 (ImportError: torchcodec absent)
        errors.append(f"torchaudio: {type(ex).__name__}")
    try:
        import soundfile as sf
        arr, sr = sf.read(path, dtype="float32", always_2d=True)
        return _from_planar_float(arr.T, sr, alloc)
    except Exception as ex:                                          # noqa: BLE001
        errors.append(f"soundfile: {type(ex).__name__}")
    ff = shutil.which("ffmpeg")
    if ff:
        try:
            probe = subprocess.run([ff, "-v", "error", "-i", path, "-f", "f32le", "-acodec", "pcm_f32le", "-ar", "16000", "-"],
                                   capture_output=True, check=True)
            ch = 1
            info = subprocess.run([shutil.which("ffprobe") or "ffprobe", "-v", "error", "-select_streams", "a:0", "-show_entries",
                                   "stream=channels", "-of", "csv=p=0", path], capture_output=True, text=True)
            if info.returncode == 0 and info.stdout.strip().isdigit():
                ch = int(info.stdout.strip())
            arr = np.frombuffer(probe.stdout, dtype=np.float32).reshape(-1, ch).T
            return _from_planar_float(arr, 16000, alloc)
        except Exception as ex:                                      # noqa: BLE001
            errors.append(f"ffmpeg: {type(ex).__name__}")
    else:
        errors.append("ffmpeg: not on PATH")
    raise UnsupportedAudio(f"no decoder for {os.path.splitext(path)[1]} in this environment ({'; '.join(errors)})")


def read_audio(path: str, alloc: Optional[Alloc] = None, default_sr: int = 16000) -> PcmAudio:
    """Container -> interleaved PCM payload (no sample conversion).  Raises UnsupportedAudio per file."""
    alloc = alloc or _default_alloc
    ext = os.path.splitext(path)[1].lower()
    try:
        if ext in (".wav", ".wave"):
            return _read_wav(path, alloc)
        if ext == ".sph":
            return _read_sph(path, alloc)
        if ext == ".flac":
            return _read_flac(path, alloc)
        if ext == ".npy":
            return _read_npy(path, alloc, default_sr)
        return _read_external(path, alloc)
    except UnsupportedAudio as ex:
        raise UnsupportedAudio(f"{path}: {ex}") from None
    except (OSError, ValueError, struct.error, KeyError) as ex:
        raise UnsupportedAudio(f"{path}: {type(ex).__name__}: {ex}") from None


def probe_audio(path: str, default_sr: int = 16000) -> Tuple[int, int, int]:
    """(sample_rate, channels, frames) from the header only — the corpus CLI balances ranks on DECODED duration,
    not file size (an mp3 and a wav of equal size differ 10x in audio)."""
    ext = os.path.splitext(path)[1].lower()
    try:
        if ext in (".wav", ".wave"):
            with open(path, "rb") as f:
                sr, ch, _, frames, _, _, _ = _wav_header(f)
            return sr, ch, frames
        if ext == ".sph":
            with open(path, "rb") as f:
                sr, ch, _, frames, _, _ = _sph_header(f)
            return sr, ch, frames
        if ext == ".flac":
            with open(path, "rb") as f:
                head = np.frombuffer(f.read(1 << 16), dtype=np.uint8)
            sr, ch, _, total = _flac_info(head)
            return sr, ch, total
        if ext == ".npy":
            arr = np.load(path, mmap_mode="r")
            return default_sr, (1 if arr.ndim == 1 else arr.shape[0]), arr.shape[-1]
    except Exception:                                                # noqa: BLE001 — fall through to the size estimate
        pass
    # compressed containers: ~64 kbit/s is what tools/sph_to_mp3.py-style corpora use; only the relative order matters
    return default_sr, 1, int(os.path.getsize(path) * 8 / 64000.0 * default_sr)


# ------------------------------------------------------------------- host-side sample conversion
_ULAW = None
_ALAW = None


def _g711_tables():
    global _ULAW, _ALAW
    if _ULAW is None:
        u = (~np.arange(256, dtype=np.uint8)).astype(np.int32)
        t = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4)
        _ULAW = np.where(u & 0x80, 0x84 - t, t - 0x84).astype(np.int16)
        a = (np.arange(256, dtype=np.uint8) ^ 0x55).astype(np.int32)
        t = (a & 0x0F) << 4
        seg = (a & 0x70) >> 4
        t = np.where(seg == 0, t + 8, np.where(seg == 1, t + 0x108, (t + 0x108) << np.maximum(seg - 1, 0)))
        _ALAW = np.where(a & 0x80, t, -t).astype(np.int16)
    return _ULAW, _ALAW


def pcm_to_float(pcm: PcmAudio, mono: bool = False) -> np.ndarray:
    """Host mirror of mc_op_pcm_to_f32: -> float32 [C, frames] ([1, frames] with mono=True: mean over channels)."""
    raw, ch, n = pcm.payload, pcm.channels, pcm.frames
    en = ">" if pcm.big_endian else "<"
    if pcm.fmt == PCM_U8:
        x = (raw.astype(np.float32) - 128.0) / 128.0
    elif pcm.fmt == PCM_S16:
        x = raw.view(en + "i2").astype(np.float32) / 32768.0
    elif pcm.fmt == PCM_S24:
        b = raw.reshape(-1, 3).astype(np.int32)
        v = (b[:, 0] << 16 | b[:, 1] << 8 | b[:, 2]) if pcm.big_endian else (b[:, 2] << 16 | b[:, 1] << 8 | b[:, 0])
        x = ((v << 8) >> 8).astype(np.float32) / 8388608.0
    elif pcm.fmt == PCM_S32:
        x = raw.view(en + "i4").astype(np.float32) / 2147483648.0
    elif pcm.fmt == PCM_F32:
        x = raw.view(en + "f4").astype(np.float32)
    elif pcm.fmt == PCM_F64:
        x = raw.view(en + "f8").astype(np.float32)
    else:
        table = _g711_tables()[0 if pcm.fmt == PCM_ULAW else 1]
        x = table[raw].astype(np.float32) / 32768.0
    x = np.ascontiguousarray(x.reshape(n, ch).T)
    if mono and ch > 1:
        acc = np.zeros(n, dtype=np.float32)
        for c in range(ch):                                           # same left-to-right fp32 sum as the kernel
            acc += x[c]
        x = (acc / np.float32(ch))[None]
    return x


# ------------------------------------------------------------------------------- resampling
@dataclass(frozen=True)
class ResamplePlan:
    up: int
    down: int
    taps: np.ndarray          # float32, scaled by `up`, left-padded for alignment (what the kernel consumes)
    fir: np.ndarray           # float64 unscaled linear-phase prototype (scipy.signal.resample_poly(window=fir))
    pre_remove: int

    def n_out(self, n_in: int) -> int:
        return -(-n_in * self.up // self.down)


@functools.lru_cache(maxsize=64)
def resample_plan(sr_in: int, sr_out: int) -> Optional[ResamplePlan]:
    """Linear-phase Kaiser FIR to the specification of librosa.resample's default kernel (res_type 'soxr_hq',
    audio_tokenizer.py:213-214): pass band up to 0.913 of the lower Nyquist, stop band from the Nyquist, ~125 dB
    (20-bit) rejection.  soxr itself is not available offline; this is a filter of the same class, not its taps."""
    from scipy.signal import firwin, kaiserord

    g = math.gcd(int(sr_in), int(sr_out))
    up, down = int(sr_out) // g, int(sr_in) // g
    if up == down:
        return None
    max_rate = max(up, down)
    numtaps, beta = kaiserord(125.0, (1.0 - 0.913) / max_rate)
    numtaps |= 1
    fir = firwin(numtaps, (1.0 + 0.913) / 2.0 / max_rate, window=("kaiser", beta))
    half_len = (numtaps - 1) // 2
    n_pre_pad = down - half_len % down                               # scipy.signal.resample_poly's alignment
    pre_remove = (half_len + n_pre_pad) // down
    taps = np.concatenate([np.zeros(n_pre_pad), fir * up]).astype(np.float32)
    return ResamplePlan(up, down, taps, fir, pre_remove)


def resample(wav: np.ndarray, sr_in: int, sr_out: int) -> np.ndarray:
    """Host polyphase resampler (float32 in/out, last axis); length ceil(n * sr_out / sr_in) like librosa.resample."""
    plan = resample_plan(int(sr_in), int(sr_out))
    if plan is None:
        return np.asarray(wav, dtype=np.float32)
    from scipy.signal import resample_poly
    return resample_poly(np.asarray(wav, dtype=np.float64), plan.up, plan.down, axis=-1, window=plan.fir).astype(np.float32)


def load_audio(path: str, target_sr: int, mono: bool) -> np.ndarray:
    """-> float32 [C, T] at target_sr on the host (librosa.load(sr=target_sr, mono=mono) stand-in)."""
    pcm = read_audio(path, default_sr=target_sr)
    x = pcm_to_float(pcm, mono=mono)
    if pcm.sample_rate != target_sr:
        x = resample(x, pcm.sample_rate, target_sr)
    return np.ascontiguousarray(x)


# ------------------------------------------------------------------------------ device ingest
class DeviceIngest:
    """PCM payload (pinned host) -> fp32 planar audio at the codec's rate in HBM:
    H2D of the raw payload on a copy stream (file i+1 uploads under the encode of file i), then on the main stream
    mc_op_pcm_to_f32 (convert / de-interleave / mono mix) and mc_op_resample; codes return through pinned memory.
    The corpus pipeline (audio_to_codes.encode_corpus) only talks to this interface."""

    def __init__(self, gen):
        import torch
        if not getattr(gen, "is_b200_native", False) or gen.device.type != "cuda":
            raise RuntimeError("DeviceIngest needs a B200Generator on its CUDA device; there is no host fallback")
        self.gen, self.torch = gen, torch
        self._taps = {}
        self._host_free = []                 # pinned staging buffers handed back by finished runs (cudaHostAlloc is ~ms per call)
        self._host_lock = __import__("threading").Lock()
        self.copy_stream = torch.cuda.Stream(device=gen.device)

    # ---- buffers
    def host_buffer(self, nbytes: int):
        """A pinned uint8 tensor of at least nbytes: the smallest recycled one that fits, else a new allocation."""
        with self._host_lock:
            fits = [b for b in self._host_free if nbytes <= b.numel() <= max(4 * nbytes, 1 << 20)]
            if fits:
                buf = min(fits, key=lambda b: b.numel())
                self._host_free = [b for b in self._host_free if b is not buf]
                return buf
        return self.torch.empty(nbytes, dtype=self.torch.uint8).pin_memory()

    def recycle(self, buf) -> None:
        """Hand a pinned buffer back (staging buffers at the end of a run, code buffers after the write); at most 64 are kept."""
        with self._host_lock:
            if buf is not None and len(self._host_free) < 64:
                self._host_free.append(buf)

    def _taps_on_device(self, plan: ResamplePlan):
        key = (plan.up, plan.down)
        if key not in self._taps:
            self._taps[key] = self.torch.from_numpy(plan.taps).to(self.gen.device)
        return self._taps[key]

    # ---- stages
    def upload(self, pcm: PcmAudio, host_tensor=None):
        """H2D of the raw payload on the copy stream -> (device bytes, event).  `host_tensor`: the pinned uint8 tensor
        that backs pcm.payload (else the payload goes through pageable memory)."""
        torch = self.torch
        nbytes = pcm.payload.nbytes
        src = host_tensor[:nbytes] if host_tensor is not None else torch.from_numpy(np.ascontiguousarray(pcm.payload))
        with torch.cuda.stream(self.copy_stream):
            raw = torch.empty(nbytes + 8, dtype=torch.uint8, device=self.gen.device)[:nbytes]
            raw.copy_(src, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self.copy_stream)
        return raw, done

    def convert(self, pcm: PcmAudio, staged, mono: bool):
        """Device payload -> fp32 [C_out, T] at gen.sample_rate on the CURRENT stream (mc_op_pcm_to_f32, mc_op_resample)."""
        torch, gen = self.torch, self.gen
        from . import _native as nat
        raw, done = staged
        main = torch.cuda.current_stream(gen.device)
        main.wait_event(done)
        raw.record_stream(main)
        mix = bool(mono and pcm.channels > 1)
        c_out = 1 if mix else pcm.channels
        if pcm.frames == 0:
            return torch.zeros((c_out, 0), dtype=torch.float32, device=gen.device)
        x = torch.empty((c_out, pcm.frames), dtype=torch.float32, device=gen.device)
        with gen._serial():
            rc = gen._lib.mc_op_pcm_to_f32(gen._handle, raw.data_ptr(), pcm.fmt, int(pcm.big_endian), pcm.channels, pcm.frames,
                                           int(mix), x.data_ptr(), pcm.frames, gen._stream())
            nat.check(gen._lib, gen._handle, rc, "mc_op_pcm_to_f32")
        plan = resample_plan(int(pcm.sample_rate), int(gen.sample_rate))
        if plan is None:
            return x
        n_out = plan.n_out(pcm.frames)
        y = torch.empty((c_out, n_out), dtype=torch.float32, device=gen.device)
        taps = self._taps_on_device(plan)
        with gen._serial():
            rc = gen._lib.mc_op_resample(gen._handle, x.data_ptr(), pcm.frames, c_out, pcm.frames, plan.up, plan.down, taps.data_ptr(),
                                         taps.numel(), plan.pre_remove, y.data_ptr(), n_out, n_out, gen._stream())
            nat.check(gen._lib, gen._handle, rc, "mc_op_resample")
        return y

    def wait_uploaded(self, staged) -> None:
        staged[1].synchronize()

    def to_device(self, pcm: PcmAudio, mono: bool, host_tensor=None):
        """upload + convert."""
        return self.convert(pcm, self.upload(pcm, host_tensor), mono)

    def upload_codes(self, host_tensor, nbytes: int):
        """H2D of `nbytes` of a pinned uint8 tensor (int64 codes, the offline decode) on the copy stream -> (device bytes,
        event); codes_on_device() hands them to the current stream."""
        torch = self.torch
        with torch.cuda.stream(self.copy_stream):
            raw = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=self.gen.device)[:nbytes]
            raw.copy_(host_tensor[:nbytes], non_blocking=True)
            done = torch.cuda.Event()
            done.record(self.copy_stream)
        return raw, done

    def codes_on_device(self, staged, channels: int, frames: int):
        """The uploaded codes as int64 [channels, frames], ordered after the upload on the current stream."""
        raw, done = staged
        main = self.torch.cuda.current_stream(self.gen.device)
        main.wait_event(done)
        raw.record_stream(main)
        return raw.view(self.torch.int64).view(channels, frames)

    def pcm_to_host(self, wav, fmt: int):
        """Planar fp32 [C, T] on the device -> (interleaved [T, C] int16 / float32 numpy view of pinned memory, wait):
        mc_op_f32_to_pcm stores straight into the pinned buffer on the current stream; wait() blocks until it has, and
        wait.release() hands the buffer back."""
        torch = self.torch
        C, T = wav.shape
        width = BYTES_PER_SAMPLE[fmt]
        raw = self.host_buffer(max(C * T * width, 8))
        out = raw[: C * T * width].view(torch.int16 if fmt == PCM_S16 else torch.float32)
        if T > 0:
            self.gen.f32_to_pcm(wav, fmt, out=out)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.gen.device))

        def wait():
            ev.synchronize()

        def release():
            self.recycle(raw)

        wait.release = release
        return out.numpy().reshape(T, C), wait

    def codes_to_host(self, codes):
        """Device int64 code tensors -> (pinned host tensors, wait) — async D2H on the current stream.  wait() blocks until
        the copies have landed; wait.release() (optional, once the caller is done with the host tensors) hands the
        pinned memory back for the next file."""
        torch = self.torch
        host, bufs = [], []
        for c in codes:
            raw = self.host_buffer(max(8 * c.numel(), 8))
            hc = raw[: 8 * c.numel()].view(torch.int64)
            hc.copy_(c, non_blocking=True)
            host.append(hc)
            bufs.append(raw)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.gen.device))

        def wait():
            ev.synchronize()

        def release():
            for b in bufs:
                self.recycle(b)

        wait.release = release
        return host, wait
