"""Multi-session batching for the streaming path (SURVEY.md §8 f2).

The reference serves several live streams through one codec: ``tts_server.py:59,158`` tokenizes every 0.1 s chunk
of every active TTS request on ONE ``AudioTokenizer`` shared by Flask threads, ``realtime_agent_resources.py:41-49``
hands one model to two agents, ``inference_client_self_play.py:148-159`` runs two agents side by side.  Alone, each
session is a batch-1 pass that streams every weight of the network for 100 rows; here the rolling contexts of up to
``max_sessions`` sessions live in one device pool (``mc_pool_*`` in the C ABI) and the sessions that are due at the
same time go through the engine as ONE ``B = n * channels`` launch.

``SessionBatcher`` keeps, per session, exactly the host-side state of ``AudioTokenizer`` (context length, code
string context, the ``[-0:]`` / hanging-code quirks of audio_tokenizer.py:99-101,144,161-168), so every session's
outputs are what its own ``AudioTokenizer`` would have returned.  Sessions whose contexts differ in length (a stream
that has just started next to one in steady state) are grouped by length: one launch per group.  With
``ragged=True`` they share one launch (``mc_pool_push_*_ragged``): each window starts at row 0 of the batch and reads
zeros past its own end, which the causal codec never looks at.

``SessionBatcher.emit_output_chunks`` is ``OutputChunkEmitter.emit`` for many agents at once: decoder, ``pad_or_trim``,
``normalize_audio_rms`` and ``smooth_join`` of every session of a group run as ONE engine call (``mc_pool_push_codes_emit``,
one CUDA graph), and each session keeps the agent's ``audio_history_ch1``.

``ThreadedSessionBatcher`` adds the tts_server.py calling pattern: request threads call ``tokenize_audio_one``,
``detokenize_audio_one`` or ``emit_output_chunk_one`` and block; a dispatcher thread collects whatever arrived within
``max_wait_ms`` and runs it as one batch per kind.
"""
from __future__ import annotations

import ctypes as C
import threading
from concurrent.futures import Future
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _native as nat
from . import audio_io as aio
from .audio_tokenizer import prep_audio_for_tokenization
from .audio_utils import create_crossfade_ramps
from .codec_chars import UNICODE_OFFSET_LARGE, chars_to_codes, codes_to_chars


class SessionPool:
    """Thin binding of mc_pool_*: slots with device-resident audio / code contexts, pushed in batches."""

    def __init__(self, gen, channels: int, context_samples: int, max_sessions: int, max_chunk_samples: int = 0):
        self.gen, self.channels, self.max_sessions = gen, channels, max_sessions
        self.cap_samples = max(context_samples, max_chunk_samples)
        self.cap_frames = -(-self.cap_samples // gen.hop)
        gen.ensure_positions(self.cap_frames)
        self._p = C.c_void_p()
        rc = gen._lib.mc_pool_create(gen._handle, channels, context_samples, self.cap_samples, max_sessions, C.byref(self._p))
        nat.check(gen._lib, gen._handle, rc, "mc_pool_create")

    def reset(self, slot: int, audio: bool = True, codes: bool = True) -> None:
        self.gen._lib.mc_pool_reset(self._p, slot, int(audio), int(codes))

    def context_len(self, slot: int) -> Tuple[int, int]:
        a, c = C.c_int32(), C.c_int32()
        self.gen._lib.mc_pool_context_len(self._p, slot, C.byref(a), C.byref(c))
        return a.value, c.value

    def set_graphs(self, enabled: bool) -> None:
        self.gen._lib.mc_pool_set_graphs(self._p, int(enabled))

    def push_audio(self, slots, chunks: np.ndarray, keep_frames: int) -> np.ndarray:
        """chunks float32 [n, C, len] -> int64 codes [n, C, keep]."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        chunks = np.ascontiguousarray(chunks, dtype=np.float32).reshape(len(slots), self.channels, -1)
        out = np.empty((len(slots) * self.channels * self.cap_frames,), dtype=np.int64)
        got = C.c_int32(0)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_audio(self._p, slots.ctypes.data, len(slots), chunks.ctypes.data, chunks.shape[2],
                                                  keep_frames, out.ctypes.data, C.byref(got), self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_audio")
        return out[: len(slots) * self.channels * got.value].reshape(len(slots), self.channels, got.value)

    def push_codes(self, slots, codes: np.ndarray, keep_samples: int) -> np.ndarray:
        """codes int64 [n, C, len] -> float32 wav [n, C, keep]."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(len(slots), self.channels, -1)
        out = np.empty((len(slots) * self.channels * self.cap_samples,), dtype=np.float32)
        got = C.c_int32(0)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_codes(self._p, slots.ctypes.data, len(slots), codes.ctypes.data, codes.shape[2],
                                                  keep_samples, out.ctypes.data, C.byref(got), self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_codes")
        return out[: len(slots) * self.channels * got.value].reshape(len(slots), self.channels, got.value)

    def set_emit(self, chunk_samples: int, fade_samples: int, target_rms: float, silence_rms_threshold: float, fade_in) -> None:
        """Arm the post-decode chain for every slot (mc_pool_set_emit); every slot forgets its previous chunk."""
        ramp = np.ascontiguousarray(fade_in, dtype=np.float32)
        if ramp.shape != (fade_samples,):
            raise ValueError("fade_in must hold fade_samples values")
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_set_emit(self._p, chunk_samples, fade_samples, float(target_rms),
                                                float(silence_rms_threshold), ramp.ctypes.data)
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_set_emit")
        self._emit_floats = 2 * chunk_samples + fade_samples

    def push_codes_emit(self, slots, codes: np.ndarray) -> Tuple[np.ndarray, bool]:
        """codes int64 [n, len] -> (float32 [n, 2*chunk + fade]: per session emitted ++ cross-faded tail ++ new history
        chunk, had_prev shared by the batch)."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(len(slots), -1)
        out = np.empty((len(slots), getattr(self, "_emit_floats", 0)), dtype=np.float32)
        had = C.c_int32(0)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_codes_emit(self._p, slots.ctypes.data, len(slots), codes.ctypes.data, codes.shape[1],
                                                       out.ctypes.data, C.byref(had), self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_codes_emit")
        return out, bool(had.value)

    def push_audio_ragged(self, slots, chunks: np.ndarray, keep_frames: int) -> np.ndarray:
        """push_audio for sessions whose contexts may differ in length: chunks float32 [n, C, len] -> int64 codes
        [n, C, keep_frames], each session's own last keep_frames frames (1 <= keep_frames <= ceil(len / hop))."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        chunks = np.ascontiguousarray(chunks, dtype=np.float32).reshape(len(slots), self.channels, -1)
        out = np.empty((len(slots), self.channels, keep_frames), dtype=np.int64)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_audio_ragged(self._p, slots.ctypes.data, len(slots), chunks.ctypes.data, chunks.shape[2],
                                                         keep_frames, out.ctypes.data, self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_audio_ragged")
        return out

    def push_codes_ragged(self, slots, codes: np.ndarray, keep_samples: int) -> Tuple[np.ndarray, np.ndarray]:
        """push_codes for sessions whose contexts may differ in length: codes int64 [n, C, len] -> (float32 wav
        [n, C, keep_samples], int32 samples [n]); session j's samples fill the first samples[j] of its row."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(len(slots), self.channels, -1)
        out = np.empty((len(slots), self.channels, keep_samples), dtype=np.float32)
        got = np.zeros(len(slots), dtype=np.int32)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_codes_ragged(self._p, slots.ctypes.data, len(slots), codes.ctypes.data, codes.shape[2],
                                                         keep_samples, out.ctypes.data, got.ctypes.data, self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_codes_ragged")
        return out, got

    def push_codes_emit_ragged(self, slots, codes: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """push_codes_emit for sessions whose contexts may differ in length, first chunks mixed with continuing ones:
        codes int64 [n, len] -> (float32 [n, 2*chunk + fade], bool had_prev [n])."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(len(slots), -1)
        out = np.empty((len(slots), getattr(self, "_emit_floats", 0)), dtype=np.float32)
        had = np.zeros(len(slots), dtype=np.int32)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_codes_emit_ragged(self._p, slots.ctypes.data, len(slots), codes.ctypes.data,
                                                              codes.shape[1], out.ctypes.data, had.ctypes.data, self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_codes_emit_ragged")
        return out, had.astype(bool)

    def set_resampler(self, sr_in: int, plan) -> None:
        """Register the polyphase plan of one client rate for push_pcm (mc_pool_set_resampler): the ResamplePlan of
        audio_io.resample_plan(sr_in, codec rate)."""
        taps = np.ascontiguousarray(plan.taps, dtype=np.float32)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_set_resampler(self._p, int(sr_in), plan.up, plan.down, taps.ctypes.data, taps.size,
                                                     plan.pre_remove)
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_set_resampler")

    def reserve_pcm(self, max_in_samples: int, max_in_channels: int) -> None:
        """Fix push_pcm's pinned staging at max_in_channels x max_in_samples per session (mc_pool_reserve_pcm)."""
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_reserve_pcm(self._p, int(max_in_samples), int(max_in_channels))
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_reserve_pcm")

    @staticmethod
    def _pcm_items(pcm) -> Tuple[np.ndarray, np.ndarray]:
        """[(sr, int16 / float32 [T] or [C_in, T])] -> (mc_pcm_chunk table, payload bytes)."""
        items = np.zeros(len(pcm), dtype=nat.PCM_CHUNK_DTYPE)
        parts, off = [], 0
        for j, (sr, x) in enumerate(pcm):
            x = np.ascontiguousarray(x)
            if x.dtype not in (np.int16, np.float32) or x.ndim not in (1, 2):
                raise ValueError(f"item {j}: push_pcm takes int16 / float32 [T] or [C_in, T], got {x.dtype} {x.shape}")
            rows = x.reshape(-1, x.shape[-1])
            items[j] = (aio.PCM_S16 if x.dtype == np.int16 else aio.PCM_F32, rows.shape[0], rows.shape[1], int(sr), off, rows.shape[1])
            parts.append(rows.reshape(-1).view(np.uint8))
            off += rows.nbytes
        return items, np.concatenate(parts) if parts else np.zeros(1, np.uint8)

    def push_pcm(self, slots, pcm, length: int, keep_frames: int) -> np.ndarray:
        """push_audio on raw client chunks: pcm = [(sr, int16 / float32 [T] or [C_in, T])], each at the codec's rate or a
        registered one and resampling to `length` samples; converted, mixed and resampled on the device -> int64 codes
        [n, C, keep]."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        items, payload = self._pcm_items(pcm)
        out = np.empty((len(slots) * self.channels * self.cap_frames,), dtype=np.int64)
        got = C.c_int32(0)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_pcm(self._p, slots.ctypes.data, len(slots), items.ctypes.data, payload.ctypes.data, int(length),
                                                keep_frames, out.ctypes.data, C.byref(got), self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_pcm")
        return out[: len(slots) * self.channels * got.value].reshape(len(slots), self.channels, got.value)

    def push_pcm_ragged(self, slots, pcm, length: int, keep_frames: int) -> np.ndarray:
        """push_audio_ragged on raw client chunks (see push_pcm) -> int64 codes [n, C, keep_frames]."""
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        items, payload = self._pcm_items(pcm)
        out = np.empty((len(slots), self.channels, keep_frames), dtype=np.int64)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_push_pcm_ragged(self._p, slots.ctypes.data, len(slots), items.ctypes.data, payload.ctypes.data,
                                                       int(length), keep_frames, out.ctypes.data, self.gen._stream())
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_push_pcm_ragged")
        return out

    def read_audio(self, slot: int, n: int) -> np.ndarray:
        """The last n samples of a slot's audio context, float32 [C, n] (mc_pool_read_audio)."""
        out = np.empty((self.channels, n), dtype=np.float32)
        with self.gen._serial():
            rc = self.gen._lib.mc_pool_read_audio(self._p, int(slot), out.ctypes.data, int(n))
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_pool_read_audio")
        return out

    def graph_count(self) -> Tuple[int, int]:
        """(distinct graph keys seen, graphs captured) over every push of this pool."""
        k, c = C.c_int32(), C.c_int32()
        with self.gen._serial():
            self.gen._lib.mc_pool_graph_count(self._p, C.byref(k), C.byref(c))
        return k.value, c.value

    def __del__(self):
        try:
            if getattr(self, "_p", None) and self.gen._handle:
                self.gen._lib.mc_pool_destroy(self._p)
                self._p = None
        except Exception:
            pass


class _SessionState:
    def __init__(self, slot: int):
        self.slot = slot
        self.audio_len = 0            # samples in the rolling audio context (len(tokenize_context[-1]))
        self.detok_context = ""       # the code-string context (detokenize_context)
        self.history: List[np.ndarray] = []   # the agent's audio_history_ch1 (emit_output_chunks)


class SessionBatcher:
    """Batched ``tokenize_audio`` / ``detokenize_audio`` over many independent sessions of one engine."""

    def __init__(self, codec_model, num_channels: int = 1, context_secs: float = 2.0, max_sessions: int = 8,
                 unicode_offset: int = UNICODE_OFFSET_LARGE, ragged: bool = False):
        """ragged=True: sessions whose contexts differ in length go through one engine call per kind and tick (split only by
        chunk length, and by decode length and preroll) instead of one call per context length.  Off by default: with the
        default split-K kernels a mixed batch has another row count than today's groups, so near-tie codes may change."""
        if not getattr(codec_model, "is_b200_native", False):
            raise RuntimeError("SessionBatcher needs the B200 engine (B200Generator); there is no fallback")
        self.gen = codec_model
        self.ragged = ragged
        self.num_channels, self.context_secs, self.unicode_offset = num_channels, context_secs, unicode_offset
        self.sampling_rate = codec_model.sample_rate
        self.framerate = self.sampling_rate / codec_model.hop
        self.codebook_size = codec_model.codebook_size
        self.context_samples = int(context_secs * self.sampling_rate)
        self.context_frames = int(context_secs * self.framerate * num_channels)
        self.pool = SessionPool(codec_model, num_channels, self.context_samples, max_sessions)
        self._free = list(range(max_sessions - 1, -1, -1))
        self._sessions: Dict[int, _SessionState] = {}
        self._next_id = 0
        self._lock = threading.RLock()
        self._emit: Optional[Tuple[int, int]] = None   # (chunk samples, fade samples) once arm_emit ran
        self._rates: set = set()                       # client rates whose resampler the pool holds

    # ---- session lifetime
    def open_session(self) -> int:
        with self._lock:
            if not self._free:
                raise RuntimeError(f"all {self.pool.max_sessions} session slots are in use")
            slot = self._free.pop()
            self.pool.reset(slot)
            sid = self._next_id
            self._next_id += 1
            self._sessions[sid] = _SessionState(slot)
            return sid

    def close_session(self, sid: int) -> None:
        with self._lock:
            self._free.append(self._sessions.pop(sid).slot)

    def reset_context(self, sid: int) -> None:
        with self._lock:
            st = self._sessions[sid]
            self.pool.reset(st.slot)
            st.audio_len, st.detok_context, st.history = 0, "", []

    # ---- encode
    def tokenize_audio(self, chunks: Dict[int, object]) -> Dict[int, str]:
        """{session: chunk} -> {session: code string}, each exactly what that session's AudioTokenizer.tokenize_audio
        (audio_tokenizer.py:67-103) would return for the same chunk.  A chunk is what AudioTokenizer takes: a float32/int16
        array [T] or [C,T] at the codec's rate, or an (sr, array) tuple.  Tuples of int16 data, or of float32 data at another
        rate, are converted, mixed and resampled on the device inside the push (SessionPool.push_pcm; the first chunk at a
        new rate registers its resampler); every other chunk is prepared on the host as AudioTokenizer does.  When a group
        holds such a tuple, all its chunks go through push_pcm, so a tick stays one engine call per group."""
        C_ = self.num_channels
        with self._lock:
            groups: Dict[Tuple[int, int], List[int]] = {}
            prepped, raw, rates = {}, {}, set()
            for sid, chunk in chunks.items():                    # validate everything before any state changes
                if sid not in self._sessions:
                    raise KeyError(f"unknown session {sid}")
                ingest = self._device_ingest(chunk)
                if ingest is not None:
                    sr, x = raw[sid] = ingest
                    if sr == self.sampling_rate:
                        n_new = x.shape[-1]
                    else:
                        n_new = aio.resample_plan(sr, self.sampling_rate).n_out(x.shape[-1])
                        rates.add(sr)
                else:
                    if isinstance(chunk, tuple):
                        x = prep_audio_for_tokenization((int(chunk[0]), np.asarray(chunk[1])), self.sampling_rate, C_)
                    else:
                        x = np.asarray(chunk)
                        if x.dtype == np.int16:
                            x = x.astype("float32") / 32768.0
                        if C_ == 1 and x.ndim > 1:
                            x = np.mean(x, axis=0)
                    x = np.ascontiguousarray(x, dtype=np.float32).reshape(C_, -1)
                    n_new = x.shape[1]
                    prepped[sid] = x
                if not 0 < n_new <= self.pool.cap_samples:
                    raise ValueError(f"session {sid}: chunks must hold 1..{self.pool.cap_samples} samples at {self.sampling_rate} Hz")
                # ragged: one call per chunk length; the [-0:] case keeps every frame of each window, so it stays grouped
                ragged = self.ragged and self._n_chars(n_new) > 0
                groups.setdefault((-1 if ragged else self._sessions[sid].audio_len, n_new), []).append(sid)
            if len(self._rates | rates) > nat.MC_POOL_MAX_RESAMPLERS:
                raise ValueError(f"a session pool converts at most {nat.MC_POOL_MAX_RESAMPLERS} client rates on the device, "
                                 f"this tick would need {sorted(self._rates | rates)}")
            for sr in sorted(rates - self._rates):
                self.pool.set_resampler(sr, aio.resample_plan(sr, self.sampling_rate))
                self._rates.add(sr)
            out: Dict[int, str] = {}
            for (ctx_len, n_new), sids in groups.items():
                n_chars = self._n_chars(n_new)
                frames_needed = -(-n_chars // C_) if n_chars > 0 else 0                  # 0 -> all frames ([-0:])
                slots = [self._sessions[s].slot for s in sids]
                if any(s in raw for s in sids):
                    push = self.pool.push_pcm_ragged if ctx_len < 0 else self.pool.push_pcm
                    pcm = [raw[s] if s in raw else (self.sampling_rate, prepped[s]) for s in sids]
                    codes = push(slots, pcm, n_new, frames_needed)                       # [n,C,k]
                else:
                    push = self.pool.push_audio_ragged if ctx_len < 0 else self.pool.push_audio
                    codes = push(slots, np.stack([prepped[s] for s in sids]), frames_needed)   # [n,C,k]
                for j, sid in enumerate(sids):
                    st = self._sessions[sid]
                    st.audio_len = min(st.audio_len + n_new, max(n_new, self.context_samples))
                    frame_major = np.ascontiguousarray(codes[j].T).reshape(1, -1)
                    text = codes_to_chars(frame_major, self.codebook_size, unicode_offset=self.unicode_offset)
                    out[sid] = text[-n_chars:]
            return out

    def _device_ingest(self, chunk) -> Optional[Tuple[int, np.ndarray]]:
        """(sr, array) when the chunk is converted on the device: an (sr, int16 / float32 array) tuple that needs more than a
        cast (int16 data, or another rate) and has a shape the pool takes ([T] or [1..8, T] on a mono pool, [C, T] else);
        None for everything the host prepares."""
        if not isinstance(chunk, tuple) or len(chunk) != 2:
            return None
        sr, x = int(chunk[0]), np.asarray(chunk[1])
        if x.dtype not in (np.int16, np.float32) or sr <= 0 or (x.dtype == np.float32 and sr == self.sampling_rate):
            return None
        if self.num_channels == 1:
            fits = x.ndim == 1 or (x.ndim == 2 and 1 <= x.shape[0] <= nat.MC_POOL_MAX_MIX_CHANNELS)
        else:
            fits = x.ndim == 2 and x.shape[0] == self.num_channels
        return (sr, x) if fits else None

    def _n_chars(self, n_new: int) -> int:
        return int(n_new / self.sampling_rate * self.framerate * self.num_channels)

    # ---- decode
    def detokenize_audio(self, strings: Dict[int, str], preroll_samples: int = 0):
        """{session: code string} -> {session: ((sr, wav), end_hanging, preroll_left)} like
        AudioTokenizer.detokenize_audio (audio_tokenizer.py:105-149)."""
        C_ = self.num_channels
        with self._lock:
            groups: Dict[Tuple[int, int], List[int]] = {}
            new_codes, hanging, wants, trimmed = {}, {}, {}, {}
            for sid, s in strings.items():                       # validate everything before any state changes
                if sid not in self._sessions:
                    raise KeyError(f"unknown session {sid}")
                extra = len(s) % C_
                if extra:
                    s = s[:-extra]
                    hanging[sid] = s[-extra:]
                else:
                    hanging[sid] = ""
                if not 0 < len(s) // C_ <= self.pool.cap_frames:
                    raise ValueError(f"session {sid}: strings must hold 1..{self.pool.cap_frames} frames")
                flat = chars_to_codes(s, 1, self.codebook_size, unicode_offset=self.unicode_offset)[0]
                new_codes[sid] = np.ascontiguousarray(np.asarray(flat).reshape(-1, C_).T)
                trimmed[sid] = s
            for sid, s in trimmed.items():
                st = self._sessions[sid]
                st.detok_context = (st.detok_context + s)[-max(len(s), self.context_frames):]
                wants[sid] = int(len(s) / (self.framerate * C_) * self.sampling_rate) + preroll_samples
                ctx_frames_before = -1 if self.ragged else self.pool.context_len(st.slot)[1]
                groups.setdefault((ctx_frames_before, len(s) // C_, wants[sid]), []).append(sid)
            out = {}
            for (ctx_len, _, want), sids in groups.items():
                slots = [self._sessions[s].slot for s in sids]
                codes = np.stack([new_codes[s] for s in sids])
                if ctx_len < 0:       # no window holds more than cap_frames * hop samples: the clamp changes no session's samples
                    wav, got = self.pool.push_codes_ragged(slots, codes, min(want, self.pool.cap_frames * self.gen.hop))
                    wav = [wav[j][..., :got[j]] for j in range(len(sids))]
                else:
                    wav = self.pool.push_codes(slots, codes, want)   # [n,C,k]
                for j, sid in enumerate(sids):
                    w = wav[j]
                    preroll_left = max(0, preroll_samples - want + w.shape[-1])
                    out[sid] = ((self.sampling_rate, (w[0] if C_ == 1 else w).copy()), hanging[sid], preroll_left)
            return out

    # ---- decode + the agent's output chain
    def arm_emit(self, chunk_size_secs: float = 0.1, chunk_fade_secs: float = 0.02, target_volume_rms: float = 0.0,
                 silence_rms_threshold: float = 0.003) -> None:
        """OutputChunkEmitter's parameters, shared by every session (agents cloned from one RealtimeAgentConfig).
        Every session forgets its previous chunk and its recording."""
        if self.num_channels != 1:
            raise ValueError("the agent's output chain is mono (pad_or_trim rejects [C,T] arrays)")
        chunk = int(chunk_size_secs * self.sampling_rate)                                   # realtime_agent_v2.py:129
        L, fade_in, _ = create_crossfade_ramps(self.sampling_rate, fade_secs=chunk_fade_secs)   # :131
        if not 0 < L <= chunk:
            raise ValueError("chunk_fade_secs must give 0 < fade samples <= chunk samples")
        with self._lock:
            self.pool.set_emit(chunk, L, target_volume_rms, silence_rms_threshold, fade_in)
            self._emit = (chunk, L)
            for st in self._sessions.values():
                st.history = []

    def audio_history_ch1(self, sid: int) -> List[np.ndarray]:
        """The session's audio_history_ch1: ``np.concatenate`` of it is the agent's recording (realtime_agent_v2.py:744)."""
        with self._lock:
            return self._sessions[sid].history

    def emit_output_chunks(self, strings: Dict[int, str]) -> Dict[int, np.ndarray]:
        """{session: output code string of one chunk} -> {session: float32 [chunk]}, each exactly what that session's own
        ``OutputChunkEmitter.emit`` returns; the code contexts advance as in ``detokenize_audio``.  Sessions are grouped by
        code-context length, one engine call per group (ragged: one call for all of them)."""
        with self._lock:
            if self._emit is None:
                raise ValueError("call arm_emit first")
            chunk, L = self._emit
            hop = self.gen.hop
            new_codes, groups = {}, {}
            for sid, s in strings.items():                       # validate everything before any state changes
                if sid not in self._sessions:
                    raise KeyError(f"unknown session {sid}")
                st = self._sessions[sid]
                if len(s) * hop != chunk:
                    raise ValueError(f"session {sid}: {len(s)} codes decode to {len(s) * hop} samples, the chunk is {chunk}")
                if not st.history and st.detok_context:
                    raise ValueError(f"session {sid}: the first emitted chunk needs an empty code context (reset_context first)")
                new_codes[sid] = chars_to_codes(s, 1, self.codebook_size, unicode_offset=self.unicode_offset)[0]
                key = (-1, None) if self.ragged else (self.pool.context_len(st.slot)[1], bool(st.history))
                groups.setdefault(key, []).append(sid)
            for sid, s in strings.items():
                st = self._sessions[sid]
                st.detok_context = (st.detok_context + s)[-max(len(s), self.context_frames):]
            out = {}
            for (ctx_len, has_prev), sids in groups.items():
                slots, codes = [self._sessions[s].slot for s in sids], np.stack([new_codes[s] for s in sids])
                if ctx_len < 0:
                    blocks, had = self.pool.push_codes_emit_ragged(slots, codes)
                else:
                    blocks, had_prev = self.pool.push_codes_emit(slots, codes)
                    had = [had_prev] * len(sids)
                for j, sid in enumerate(sids):                   # OutputChunkEmitter._emit_native, session by session
                    block, hist = blocks[j], self._sessions[sid].history
                    if bool(had[j]) != bool(hist):
                        raise RuntimeError("emit chain state diverged from audio_history_ch1")
                    if had[j]:
                        hist[-1] = np.concatenate((hist[-1][:chunk - L], block[chunk:chunk + L]))
                    hist.append(block[chunk + L:].copy())
                    out[sid] = block[:chunk].copy()
            return out


class ThreadedSessionBatcher(SessionBatcher):
    """tts_server.py's calling pattern: every request thread calls ``tokenize_audio_one(session, chunk)``,
    ``detokenize_audio_one(session, codes)`` or ``emit_output_chunk_one(session, codes)`` and blocks; each tick the
    dispatcher thread runs everything that arrived within ``max_wait_ms``: the encode batch, then one decode batch per
    ``preroll_samples`` value, then the emit batch.  A session has at most one request of each kind in a tick; later
    ones wait for the next tick.  Encode and decode contexts are independent, so the order of the kinds changes no
    result."""

    def __init__(self, *args, max_wait_ms: float = 2.0, **kw):
        super().__init__(*args, **kw)
        self.max_wait = max_wait_ms / 1e3
        self._cv = threading.Condition()
        self._pending: List[Tuple[tuple, int, object, Future]] = []   # (kind, session, payload, future)
        self._stop = False
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _submit(self, kind: tuple, sid: int, payload, timeout: Optional[float]):
        fut: Future = Future()
        with self._cv:
            self._pending.append((kind, sid, payload, fut))
            self._cv.notify()
        return fut.result(timeout=timeout)

    def tokenize_audio_one(self, sid: int, chunk, timeout: Optional[float] = 30.0) -> str:
        """chunk: an array at the codec's rate or an (sr, array) tuple, as SessionBatcher.tokenize_audio takes it."""
        return self._submit(("encode",), sid, chunk, timeout)

    def detokenize_audio_one(self, sid: int, code_str: str, preroll_samples: int = 0, timeout: Optional[float] = 30.0):
        """-> ((sr, wav), end_hanging, preroll_left), as SessionBatcher.detokenize_audio gives it for this session."""
        return self._submit(("decode", int(preroll_samples)), sid, code_str, timeout)

    def emit_output_chunk_one(self, sid: int, code_str: str, timeout: Optional[float] = 30.0) -> np.ndarray:
        """The session's OutputChunkEmitter.emit(code_str), batched with the other sessions' emits of the tick."""
        return self._submit(("emit",), sid, code_str, timeout)

    def shutdown(self) -> None:
        with self._cv:
            self._stop = True
            self._cv.notify()
        self._thread.join(timeout=5)

    def _run(self) -> None:
        import time
        while True:
            with self._cv:
                while not self._pending and not self._stop:
                    self._cv.wait()
                if self._stop and not self._pending:
                    return
            time.sleep(self.max_wait)                      # let the other streams' chunks of this tick arrive
            with self._cv:
                batches: Dict[tuple, List[Tuple[int, object, Future]]] = {}
                rest, seen = [], set()
                for kind, sid, payload, fut in self._pending:   # one request per (session, kind) per tick, in arrival order
                    if (sid, kind[0]) in seen:
                        rest.append((kind, sid, payload, fut))
                    else:
                        seen.add((sid, kind[0]))
                        batches.setdefault(kind, []).append((sid, payload, fut))
                self._pending = rest
            self._serve(self.tokenize_audio, batches.pop(("encode",), []))
            for kind in sorted(k for k in batches if k[0] == "decode"):
                self._serve(lambda reqs, pre=kind[1]: self.detokenize_audio(reqs, preroll_samples=pre), batches[kind])
            self._serve(self.emit_output_chunks, batches.get(("emit",), []))

    @staticmethod
    def _serve(call, batch: List[Tuple[int, object, Future]]) -> None:
        if not batch:
            return
        try:
            res = call({sid: payload for sid, payload, _ in batch})
            for sid, _, fut in batch:
                fut.set_result(res[sid])
        except (ValueError, KeyError):
            # a malformed request (bad chunk length or string, closed session, emit not armed) is rejected BEFORE anything
            # is pushed: serve the others, fail only the offender
            for sid, payload, fut in batch:
                try:
                    fut.set_result(call({sid: payload})[sid])
                except Exception as ex:                    # noqa: BLE001
                    fut.set_exception(ex)
        except Exception as ex:                            # noqa: BLE001  (engine failure: state unknown, everyone in the batch hears about it)
            for _, _, fut in batch:
                if not fut.done():
                    fut.set_exception(ex)
