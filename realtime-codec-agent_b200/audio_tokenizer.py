"""Drop-in ``AudioTokenizer`` for the B200 engine.

Public surface, argument meaning, return shapes and quirks are those of
/root/reference/realtime_codec_agent/audio_tokenizer.py (class at :10, ctor :11-42,
tokenize_audio :67-103, detokenize_audio :105-149, get_codec_embeddings :151-159,
_drop_hanging_channel_codes :161-168, _encode_silence :170-179, _compute_framerate :181-187,
_prep_audio_for_tokenization :203-215).  What differs is what runs underneath:

* ``codec_model="MagiCodec-50Hz-Base"`` (or a checkpoint path) builds a ``B200Generator``
  (hand-written sm_100a kernels behind the C-ABI in include/magicodec_b200.h); there is no
  CPU fallback — constructing it without a B200 and the built extension raises.
* with a ``B200Generator`` all channels go through ONE batched engine call per
  tokenize/detokenize (the reference loops batch-1 per channel, :83-86 and :136-139), only
  the frames/samples the caller keeps are computed past the last attention layer and copied
  back (:99-101, :141-144), and the projected codebook is cached (the reference re-projects
  131 072 rows on every decode, :198).
* any other duck-typed model object (``pad_audio/encoder/quantizer/decoder``) is driven
  through exactly the calls the reference makes, so host-side behaviour can be compared
  against the reference wrapper with the same model on either side.
"""
from __future__ import annotations

import math
import threading
from typing import Any, Optional, Tuple, Union

import numpy as np
import torch

from .codec_chars import UNICODE_OFFSET_LARGE, chars_to_codes, codes_to_chars

AudioLike = Union[Tuple[int, np.ndarray], np.ndarray]


def load_magicodec_model(name_or_path: str, device: torch.device):
    """Counterpart of codec_bpe.tools.codec_utils.load_magicodec_model (audio_tokenizer.py:8,27).

    Returns ``(model, None, None)`` like upstream's 3-tuple.  Resolution order: an existing
    checkpoint file path; ``$MAGICODEC_B200_CHECKPOINT``; else seeded random-init weights of the
    default spec (no checkpoint is reachable offline — BASELINE.json prescribes random init).
    """
    import os

    from .generator import B200Generator
    from .spec import DEFAULT_SPEC
    from .weights import init_random_weights, load_checkpoint

    path = name_or_path if os.path.isfile(name_or_path) else os.environ.get("MAGICODEC_B200_CHECKPOINT")
    if path:
        spec, weights = load_checkpoint(path)
    else:
        import warnings
        warnings.warn(f"load_magicodec_model({name_or_path!r}): no checkpoint file and $MAGICODEC_B200_CHECKPOINT is not set — "
                      "using SEEDED RANDOM weights of the default spec (benchmark / test mode; the codes carry no audio meaning). "
                      "Convert a real checkpoint with weights.save_checkpoint and point $MAGICODEC_B200_CHECKPOINT at it.",
                      RuntimeWarning, stacklevel=2)
        spec, weights = DEFAULT_SPEC, init_random_weights(DEFAULT_SPEC, seed=0)
    return B200Generator(spec, weights, device=device), None, None


class AudioTokenizer:
    def __init__(
        self,
        codec_model: Union[str, Any] = "MagiCodec-50Hz-Base",
        num_channels: int = 1,
        context_secs: float = 2.0,
        unicode_offset: int = UNICODE_OFFSET_LARGE,
        device: Optional[Union[str, torch.device]] = None,
    ):
        if device is None:
            device = "cuda" if torch.cuda.is_available() else "cpu"
        self.device = torch.device(device)
        self.autocast_bfloat16 = self.device.type == "cuda" and torch.cuda.is_bf16_supported()

        if isinstance(codec_model, str):
            codec_model = load_magicodec_model(codec_model, self.device)[0]
        self.codec_model = codec_model.eval().to(self.device)
        self._native = bool(getattr(self.codec_model, "is_b200_native", False))

        self.num_channels = num_channels
        self.num_codebooks = 1
        self.codebook_size = self.codec_model.codebook_size
        self.context_secs = context_secs
        self.unicode_offset = unicode_offset
        self.sampling_rate = self.codec_model.sample_rate
        self.framerate = self._compute_framerate()
        self.context_samples = int(self.context_secs * self.sampling_rate)
        self.context_frames = int(self.context_secs * self.framerate * self.num_channels)
        self._session = None
        # One tokenizer may be shared by threads (tts_server.py:59,158 runs Flask with threaded=True on a single
        # AudioTokenizer): the rolling contexts and the engine call that consumes them change together or not at all.
        self._lock = threading.RLock()
        self.reset_context()

    # ------------------------------------------------------------------ state
    def reset_context(self):
        with self._lock:
            self.tokenize_context = np.zeros((self.num_channels, 0), dtype=np.float32)
            self._ctx_buf = None
            self.detokenize_context = ""
            if getattr(self, "_session", None) is not None:
                self._session.reset()
            self._session_audio_ok = self._session_codes_ok = True      # device context mirrors the host context

    def _stream_session(self):
        """Device-resident twin of the two contexts (native engine only), created on first use."""
        if self._session is None:
            self._session = self.codec_model.open_stream(self.num_channels, self.context_samples)
            self._session_audio_ok = self.tokenize_context.shape[-1] == 0
            self._session_codes_ok = len(self.detokenize_context) == 0
        return self._session

    def get_audio_codes_str_secs(self, audio_codes_str: str) -> float:
        return len(audio_codes_str) / (self.framerate * self.num_channels)

    # ----------------------------------------------------------------- encode
    def chunked_tokenize_audio(self, audio: AudioLike, chunk_size_secs: float) -> str:
        sr, wav = (self.sampling_rate, audio) if isinstance(audio, np.ndarray) else audio
        step = int(chunk_size_secs * sr)
        total = wav.shape[-1]
        with self._lock:
            fast = self._chunked_tokenize_batched(sr, wav, step, chunk_size_secs) if self._native else None
            if fast is not None:
                return fast
            return "".join(self.tokenize_audio((sr, wav[..., s:s + step])) for s in range(0, total, step))

    @torch.inference_mode()
    def _chunked_tokenize_batched(self, sr: int, wav: np.ndarray, step: int, chunk_size_secs: float) -> Optional[str]:
        """The loop above as ONE batched corpus encode (corpus.encode_streams: every chunk's 2.0 s window in a few
        launches) — the same kernels, hence the same codes, as the offline training-data encode, which is what the
        agent wants for its enrolment prompt (realtime_agent_v2.py:77).  Taken only where it is provably the loop's
        result: empty context, no per-chunk resampling, and chunk sizes for which the per-chunk character count
        int(secs * framerate * C) is a whole number of frames.  Leaves the contexts as the loop would."""
        from . import corpus
        C = self.num_channels
        if self.tokenize_context.shape[-1] != 0 or sr != self.sampling_rate or step <= 0 or wav.shape[-1] == 0:
            return None
        full = self._prep_audio_for_tokenization((sr, wav)).reshape(C, -1)
        total = full.shape[-1]
        per_chunk = int(step / self.sampling_rate * self.framerate)
        if int(step / self.sampling_rate * self.framerate * C) != C * per_chunk or per_chunk <= 0:
            return None
        if C > 1 and total % step != 0:
            return None                                    # a ragged tail can cut a frame in two across channels (:99-101)
        gen = self.codec_model
        dev = torch.from_numpy(np.ascontiguousarray(full)).to(self.device)
        codes = corpus.encode_streams(gen, [dev[c] for c in range(C)], chunk_size_secs, self.context_secs)
        per_channel = torch.stack(codes).cpu().numpy()[:, None, :]             # [C,1,F]
        text = self._interleave_chars(per_channel)
        last_new = total - ((total - 1) // step) * step
        keep = max(last_new, self.context_samples)
        self.tokenize_context = full[..., -keep:].astype(np.float32, copy=True)
        self._stream_session().load_audio(self.tokenize_context[..., -self.context_samples:])
        self._session_audio_ok = True
        return text

    def tokenize_audio(self, audio: AudioLike) -> str:
        with self._lock:
            new = self._prep_audio_for_tokenization(audio)
            if self._native:
                text = self._tokenize_on_session(new)
                if text is not None:
                    return text
            return self._tokenize_audio_locked(new)

    def _tokenize_on_session(self, new: np.ndarray) -> Optional[str]:
        """The steady state of the full-duplex loop (one chunk per call, device-resident context): no torch call, no
        context manager — every microsecond here is on the per-frame latency (the engine call is ~0.35 ms).  Returns None
        WITHOUT touching any state when the call has to take the general path."""
        C = self.num_channels
        n_new = new.shape[-1]
        sess = self._stream_session()                                # before the context changes: mirrors it from the start
        if not (self._session_audio_ok and 0 < n_new <= sess.cap_samples):
            return None
        chunk = new.reshape(C, -1)
        self._append_context(chunk)
        n_chars = int(n_new / self.sampling_rate * self.framerate * C)
        frames_needed = -(-n_chars // C) if n_chars > 0 else 0       # 0 -> all frames ([-0:] keeps everything)
        codes = sess.push_audio(chunk, frames_needed)                # [C, k] int64
        pts = (codes[0] if C == 1 else np.ascontiguousarray(codes.T).reshape(-1)) + self.unicode_offset
        text = pts.astype("<u4").tobytes().decode("utf-32-le", errors="surrogatepass")
        return text[-n_chars:]

    @torch.inference_mode()
    def _tokenize_audio_locked(self, new: np.ndarray) -> str:
        n_new = new.shape[-1]
        C = self.num_channels
        sess = self._stream_session() if self._native else None      # before the context changes: mirrors it from the start
        self._append_context(new.reshape(C, -1))

        # chars the caller keeps: int(secs*framerate*C); a zero count slices [-0:] == whole string
        n_chars = int(n_new / self.sampling_rate * self.framerate * C)

        if self._native:
            frames_needed = -(-n_chars // C) if n_chars > 0 else 0          # 0 -> all frames
            if self._session_audio_ok and 0 < n_new <= sess.cap_samples:
                # steady state: only the new chunk crosses PCIe; the context lives in HBM
                per_channel = sess.push_audio(new.reshape(C, -1), frames_needed)[:, None, :]
            else:
                window = torch.from_numpy(np.ascontiguousarray(self.tokenize_context)).to(self.device, non_blocking=True)
                codes = self.codec_model.encode(window, keep_last_frames=frames_needed)  # [C,Fk] int64
                per_channel = codes.cpu().numpy()[:, None, :]                   # [C,1,Fk]
                # re-seed the device context with what the next call can still see (an upload, no compute)
                sess.load_audio(self.tokenize_context[..., -self.context_samples:])
                self._session_audio_ok = True
        else:
            window = torch.tensor(self.tokenize_context).to(self.device)
            with self._autocast():
                per_channel = torch.cat([self._magicodec_encode(ch[None]) for ch in window], dim=0)
            per_channel = per_channel.cpu().numpy()

        text = self._interleave_chars(per_channel)
        return text[-n_chars:]

    def _append_context(self, new: np.ndarray) -> None:
        """tokenize_context <- the last max(len(new), context_samples) samples of (tokenize_context ++ new)
        (audio_tokenizer.py:72-74; [-0:] keeps everything, as upstream).  The reference concatenates and slices — a
        128 KB copy per 20 ms frame; here the context is a view that slides through a buffer of a few context lengths
        and is moved back to its start only when it reaches the end."""
        C, n_new = new.shape
        old = self.tokenize_context
        keep = max(n_new, self.context_samples)
        keep_old = min(old.shape[-1], keep - n_new) if n_new < keep else 0
        buf = getattr(self, "_ctx_buf", None)
        base = old.base if old.base is not None else old
        if buf is None or base is not buf or buf.shape[0] != C or keep > buf.shape[1] // 4:
            buf = np.empty((C, 8 * max(keep, self.context_samples)), dtype=np.float32)
            buf[:, :keep_old] = old[:, old.shape[-1] - keep_old:]
            self._ctx_buf, self._ctx_end = buf, keep_old
        elif self._ctx_end + n_new > buf.shape[1]:
            buf[:, :keep_old] = old[:, old.shape[-1] - keep_old:]              # regions cannot overlap: keep_old <= size / 8
            self._ctx_end = keep_old
        end = self._ctx_end
        buf[:, end:end + n_new] = new
        self._ctx_end = end + n_new
        self.tokenize_context = buf[:, self._ctx_end - keep_old - n_new:self._ctx_end]

    def _interleave_chars(self, codes_c1f: np.ndarray) -> str:
        """[C,1,F] codes -> 'c0[0] c1[0] c0[1] c1[1] ...' (audio_tokenizer.py:89-96)."""
        C = codes_c1f.shape[0]
        if C == 1:
            return codes_to_chars(codes_c1f[0], self.codebook_size, unicode_offset=self.unicode_offset)
        # same offset on every channel: channels are not codebooks
        frame_major = np.ascontiguousarray(codes_c1f[:, 0, :].T).reshape(1, -1)
        return codes_to_chars(frame_major, self.codebook_size, unicode_offset=self.unicode_offset)

    # ----------------------------------------------------------------- decode
    def detokenize_audio(self, audio_codes_str: str, preroll_samples: int = 0):
        with self._lock:
            if self._native:
                fast = self._detokenize_on_session(audio_codes_str, preroll_samples)
                if fast is not None:
                    return fast
            return self._detokenize_audio_locked(audio_codes_str, preroll_samples)

    def chunked_detokenize_audio(self, audio_codes_str: str, chunk_size_secs: float):
        """The twin of chunked_tokenize_audio: ``detokenize_audio`` over pieces of int(chunk_size_secs * framerate * C)
        characters, outputs concatenated -> (sampling_rate, float32 [T] or [C, T]).  Each piece is decoded from the
        trailing context_secs of codes and only its own samples are kept, which is how the agent hears its codes.

        With the B200 engine, an empty ``detokenize_context``, whole frames per piece and no hanging code, the loop runs as
        ONE batched corpus decode (corpus.decode_streams); otherwise it runs as written.  Either way the contexts are left
        as the loop leaves them.  The batched path runs the stateless corpus kernels, the loop's calls run on the streaming
        session's few-rows kernels (DESIGN.md §5, "Two kernel regimes"): the two agree bit for bit with
        ``small_m_split_k = 0`` and to the decode parity bar (SNR >= 38 dB) with the default setting."""
        C = self.num_channels
        step = int(chunk_size_secs * self.framerate * C)
        if step <= 0:
            raise ValueError(f"chunk_size_secs={chunk_size_secs} is less than one code per chunk")
        with self._lock:
            fast = self._chunked_detokenize_batched(audio_codes_str, step) if self._native else None
            if fast is not None:
                return self.sampling_rate, fast
            parts = [self.detokenize_audio(audio_codes_str[s:s + step])[0][1] for s in range(0, len(audio_codes_str), step)]
            if not parts:
                return self.sampling_rate, np.zeros((0,) if C == 1 else (C, 0), dtype=np.float32)
            return self.sampling_rate, np.concatenate(parts, axis=-1)

    @torch.inference_mode()
    def _chunked_detokenize_batched(self, text: str, step: int) -> Optional[np.ndarray]:
        """The loop of chunked_detokenize_audio as corpus.decode_streams, taken only where it provably decodes the same
        windows and keeps the same samples; None (nothing touched) otherwise."""
        from . import corpus
        C, sr = self.num_channels, self.sampling_rate
        n = len(text)
        if self.detokenize_context or n == 0 or step % C or n % C or self.context_frames % C:
            return None
        cf, hop = step // C, self.codec_model.hop
        last = n - ((n - 1) // step) * step
        for piece in (step, last):                                   # samples the loop keeps per piece (:283)
            if int(piece / (self.framerate * C) * sr) != piece // C * hop:
                return None
        if int(self.context_secs * sr / hop) != self.context_frames // C:            # decode_streams' context in frames
            return None
        flat = chars_to_codes(text, 1, self.codebook_size, unicode_offset=self.unicode_offset)[0]
        codes = np.ascontiguousarray(flat.reshape(-1, C).T)                   # [C, F]
        dev = torch.from_numpy(codes).to(self.device)
        wav = corpus.decode_streams(self.codec_model, [dev[c] for c in range(C)], cf * hop / sr, self.context_secs)
        out = torch.stack(wav).cpu().numpy()
        keep = max(last, self.context_frames)
        self.detokenize_context = text[-keep:]
        ctx = np.ascontiguousarray(chars_to_codes(self.detokenize_context, 1, self.codebook_size,
                                                  unicode_offset=self.unicode_offset)[0].reshape(-1, C).T)
        self._stream_session().load_codes(ctx[:, -(self.context_frames // C):])
        self._session_codes_ok = True
        return out[0] if C == 1 else out

    def _detokenize_on_session(self, audio_codes_str: str, preroll_samples: int):
        """Steady-state twin of _detokenize_audio_locked (same bookkeeping, same results) without a torch call; returns
        None WITHOUT touching any state when the general path has to run."""
        C = self.num_channels
        audio_codes_str, end_hanging = self._drop_hanging_channel_codes(audio_codes_str)
        sess = self._stream_session()
        n_chars = len(audio_codes_str)
        if not (self._session_codes_ok and 0 < n_chars // C <= sess.cap_frames):
            return None
        self.detokenize_context = (self.detokenize_context + audio_codes_str)[-max(n_chars, self.context_frames):]
        want = int(self.get_audio_codes_str_secs(audio_codes_str) * self.sampling_rate) + preroll_samples
        pts = np.frombuffer(audio_codes_str.encode("utf-32-le", errors="surrogatepass"), dtype="<u4").astype(np.int64)
        pts -= self.unicode_offset
        codes = pts[None] if C == 1 else np.ascontiguousarray(pts.reshape(-1, C).T)      # [C, F] (:116)
        wav = sess.push_codes(codes, want)                           # [C, Tk] float32, a fresh array
        preroll_left = max(0, preroll_samples - want + wav.shape[-1])
        return (self.sampling_rate, wav[0] if C == 1 else wav), end_hanging, preroll_left

    @torch.inference_mode()
    def _detokenize_audio_locked(self, audio_codes_str: str, preroll_samples: int = 0):
        audio_codes_str, end_hanging = self._drop_hanging_channel_codes(audio_codes_str)
        C = self.num_channels
        sess = self._stream_session() if self._native else None
        self.detokenize_context += audio_codes_str
        keep = max(len(audio_codes_str), self.context_frames)
        self.detokenize_context = self.detokenize_context[-keep:]

        want = int(self.get_audio_codes_str_secs(audio_codes_str) * self.sampling_rate) + preroll_samples
        n_new_frames = len(audio_codes_str) // C
        on_session = self._native and self._session_codes_ok and 0 < n_new_frames <= sess.cap_frames
        # de-interleave (:116); on the session path only the NEW codes cross to the device, so only they are converted
        text = audio_codes_str if on_session else self.detokenize_context
        flat = chars_to_codes(text, 1, self.codebook_size, unicode_offset=self.unicode_offset)[0]
        codes = np.ascontiguousarray(flat.reshape(-1, C).T)                  # [C,F]

        if self._native:
            if on_session:
                wav = torch.from_numpy(sess.push_codes(codes, want))[None]          # [1,C,Tk]
            else:
                dev_codes = torch.from_numpy(codes).to(self.device, non_blocking=True)
                wav = self.codec_model.decode(dev_codes, keep_last_samples=want)[None].cpu()   # [1,C,Tk] fp32
                sess.load_codes(codes[:, -(self.context_frames // C):])
                self._session_codes_ok = True
        else:
            dev_codes = torch.from_numpy(codes)[:, None, :].to(self.device)  # [C,1,F]
            with self._autocast():
                wav = torch.cat([self._magicodec_decode(ch[None]) for ch in dev_codes], dim=1)
            wav = wav[..., -want:]                                            # [-0:] == everything

        preroll_left = max(0, preroll_samples - want + wav.shape[-1])
        out = wav[0, 0] if C == 1 else wav[0]
        return (self.sampling_rate, out.cpu().numpy()), end_hanging, preroll_left

    # ------------------------------------------------- decode + emit chain (native engine only)
    def arm_emit(self, chunk_samples: int, fade_samples: int, target_rms: float, silence_rms_threshold: float,
                 fade_in: np.ndarray) -> None:
        """Configure the device-side output chain (OutputChunkEmitter); forgets the previous chunk."""
        if not self._native:
            raise RuntimeError("the fused emit chain needs the B200 engine")
        self._stream_session().set_emit(chunk_samples, fade_samples, target_rms, silence_rms_threshold, fade_in)

    def detokenize_audio_emit(self, audio_codes_str: str):
        """detokenize_audio(str, preroll_samples=L) + pad_or_trim + normalize_audio_rms + smooth_join in one
        engine call.  Context bookkeeping is that of detokenize_audio (:105-113).  Returns
        (float32[2*chunk + L] = emitted ++ cross-faded tail of the previous chunk ++ new history chunk, had_prev).

        The FIRST emitted chunk of a session needs an empty code context (the engine rejects it otherwise): with
        a non-empty context the reference keeps an (n + L)-sample history chunk and its own length assert
        (realtime_agent_v2.py:566-568) fires on the next chunk, so that state is unreachable upstream as well."""
        with self._lock, torch.inference_mode():
            audio_codes_str, _ = self._drop_hanging_channel_codes(audio_codes_str)
            sess = self._stream_session()
            before = self.detokenize_context
            self.detokenize_context += audio_codes_str
            keep = max(len(audio_codes_str), self.context_frames)
            self.detokenize_context = self.detokenize_context[-keep:]
            if not self._session_codes_ok:
                # device context out of step with the string (a one-shot decode ran in between): re-seed it
                tail = before[-self.context_frames:]
                sess.load_codes(chars_to_codes(tail, 1, self.codebook_size, unicode_offset=self.unicode_offset))
                self._session_codes_ok = True
            new_codes = chars_to_codes(audio_codes_str, 1, self.codebook_size, unicode_offset=self.unicode_offset)
            return sess.push_codes_emit(new_codes)

    # ---------------------------------------------------------- codec details
    @torch.inference_mode()
    def get_codec_embeddings(self) -> torch.Tensor:
        q = self.codec_model.quantizer
        with self._autocast():
            return q.codebook_proj(q.codebook.weight)

    def _drop_hanging_channel_codes(self, audio_str: str) -> Tuple[str, str]:
        extra = len(audio_str) % self.num_channels
        if extra == 0:
            return audio_str, ""
        trimmed = audio_str[:-extra]
        # upstream returns the tail of the ALREADY trimmed string (:164-165); kept bug-compatible
        return trimmed, trimmed[-extra:]

    @torch.inference_mode()
    def _encode_silence(self, secs: float) -> torch.Tensor:
        silence = torch.zeros(int(secs * self.sampling_rate), device=self.device)
        with self._autocast():
            return self._magicodec_encode(silence[None])

    def _compute_framerate(self) -> float:
        probe_secs = 10.0
        frames = self._encode_silence(probe_secs).shape[-1]
        samples_per_frame = math.ceil(int(probe_secs * self.sampling_rate) / frames)
        return self.sampling_rate / samples_per_frame

    def _magicodec_encode(self, x: torch.Tensor) -> torch.Tensor:
        m = self.codec_model
        if self._native:
            return m.encode(x)[:, None, :]
        z_e = m.encoder(m.pad_audio(x))
        return m.quantizer.inference(z_e)[1].unsqueeze(1)

    def _magicodec_decode(self, codes: torch.Tensor) -> torch.Tensor:
        m = self.codec_model
        codes = codes.squeeze(1)
        if self._native:
            return m.decode(codes)[:, None, :]
        table = m.quantizer.codebook_proj(m.quantizer.codebook.weight)
        return m.decoder(torch.nn.functional.embedding(codes, table)).float()

    def _prep_audio_for_tokenization(self, audio: AudioLike) -> np.ndarray:
        sr, wav = (self.sampling_rate, audio) if isinstance(audio, np.ndarray) else audio
        if wav.dtype == np.int16:
            wav = wav.astype("float32") / 32768.0
        if self.num_channels == 1 and wav.ndim > 1:
            wav = np.mean(wav, axis=0)                       # librosa.to_mono
        if sr != self.sampling_rate:
            wav = _resample(wav, sr, self.sampling_rate)
        return wav

    def _autocast(self):
        return torch.autocast(device_type="cuda", dtype=torch.bfloat16, enabled=self.autocast_bfloat16)


def _resample(wav: np.ndarray, orig_sr: int, target_sr: int) -> np.ndarray:
    """Stand-in for ``librosa.resample`` (audio_tokenizer.py:214; default res_type 'soxr_hq'): a linear-phase
    polyphase FIR designed to soxr-HQ's specification (audio_io.resample_plan).  soxr itself is not available
    offline, so sample values differ from the reference's in the transition band; INTEGRATION.md states by how much."""
    from .audio_io import resample

    return resample(wav, int(orig_sr), int(target_sr))
