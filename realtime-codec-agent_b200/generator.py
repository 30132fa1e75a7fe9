"""B200Generator — the MagiCodec model object of the B200 engine.

Implements the duck type the reference wrapper drives
(/root/reference/realtime_codec_agent/audio_tokenizer.py:28,32,36,158,190-200):
``eval() to() sample_rate codebook_size pad_audio encoder quantizer.{inference,codebook,
codebook_proj} decoder`` — so the UNMODIFIED reference ``AudioTokenizer`` runs on these kernels —
plus the batched fast entry points ``encode`` / ``decode`` our own ``AudioTokenizer`` uses.

Everything that computes is a kernel of libmagicodec_b200.so reached through the C ABI; torch only
owns the device buffers and the stream.  Nothing here falls back to PyTorch ops or to the CPU.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import Dict, Optional

import torch

from . import _native as nat
from .spec import MagiCodecSpec

BF16, F32 = torch.bfloat16, torch.float32


# ------------------------------------------------------------------------------------ packing
def rope_tables(max_positions: int, head_dim: int, base: float):
    """cos/sin [max_positions, head_dim/2] fp32 — flash-attn rotary convention (non-interleaved)."""
    half = head_dim // 2
    inv_freq = 1.0 / (base ** (torch.arange(0, half, dtype=torch.float32) * 2.0 / head_dim))
    freqs = torch.outer(torch.arange(max_positions, dtype=torch.float32), inv_freq)
    return torch.cos(freqs).contiguous(), torch.sin(freqs).contiguous()


def split_bf16(x: torch.Tensor, parts: int):
    """x (fp32) = sum of `parts` bf16 tensors, each the rounding of the running remainder."""
    out, rem = [], x.to(F32).clone()
    for _ in range(parts):
        p = rem.to(BF16)
        out.append(p)
        rem = rem - p.to(F32)
    return out


def pack_weights(spec: MagiCodecSpec, w: Dict[str, torch.Tensor], max_positions: int,
                 gemm_dtype: torch.dtype = torch.bfloat16) -> Dict[str, torch.Tensor]:
    """fp32 master weights (weights.param_shapes layout) -> the engine's packed CPU tensors.

    Layouts (also DESIGN.md §"Packed weights"):
      enc.conv0.w      fp32 [2*s0, C0]            (tap-major)            enc.conv0.b fp32 [C0]
      enc.conv{i}.w    bf16 [Cout, 2*s*Cin]       K index = tap*Cin + c  (i >= 1)
      dec.up{i}.w      bf16 [s*Cout, 2*Cin]       row = j*Cout + co; K = [x[t-1] | x[t]]   (i < n-1)
      dec.up{i}.b      fp32 [s*Cout]              bias repeated per tap
      dec.up{n-1}.w    fp32 [Cin, 2*s]            (Cout = 1)             dec.up{n-1}.b fp32 [1]
      *.wqkv/.wo/.w1/.w2, enc.proj.w  bf16 [N,K] as torch Linear stores them; biases / norms fp32
      dec.in_proj.w    bf16 [d, 64]               K zero-padded 16 -> 64
      vq.codebook      fp32 [K,16]  = codebook_proj(codebook.weight), computed in fp32 on the CPU
      vq.c2            fp32 [K]     = |row|^2
      vq.packed        bf16 [K,64]  = [c_hi | c_lo | c_hi | n1 n2 n3 0...]  (vq_sm100.cuh)
      rope.cos/.sin    fp32 [32, max_positions]   (transposed: coalesced per-row lookups in the QKV epilogue)
    """
    n = len(spec.conv_strides)
    BF16 = gemm_dtype          # tests pack in fp32 to check layouts exactly (tests/packed_emulator.py)
    p: Dict[str, torch.Tensor] = {}
    p["enc.conv0.w"] = w["enc.conv0.weight"][:, 0, :].t().contiguous().to(F32)
    p["enc.conv0.b"] = w["enc.conv0.bias"].to(F32)
    for i in range(1, n):
        cw = w[f"enc.conv{i}.weight"]                                  # [Cout, Cin, k]
        p[f"enc.conv{i}.w"] = cw.permute(0, 2, 1).reshape(cw.shape[0], -1).to(BF16).contiguous()
        p[f"enc.conv{i}.b"] = w[f"enc.conv{i}.bias"].to(F32)
    for i, s in enumerate(spec.dec_strides):
        tw = w[f"dec.up{i}.weight"]                                    # [Cin, Cout, 2s]
        if i < n - 1:
            both = torch.cat([tw[:, :, s:], tw[:, :, :s]], dim=0)       # [2Cin, Cout, s]: prev-frame taps first
            p[f"dec.up{i}.w"] = both.permute(2, 1, 0).reshape(s * tw.shape[1], -1).to(BF16).contiguous()
            p[f"dec.up{i}.b"] = w[f"dec.up{i}.bias"].to(F32).repeat(s).contiguous()
        else:
            p[f"dec.up{i}.w"] = tw[:, 0, :].to(F32).contiguous()        # [Cin, 2s]
            p[f"dec.up{i}.b"] = w[f"dec.up{i}.bias"].to(F32).contiguous()
    for stack, layers in (("enc", spec.enc_layers), ("dec", spec.dec_layers)):
        for l in range(layers):
            s_, d_ = f"{stack}.layers.{l}", f"{stack}.layers.{l}"
            p[f"{d_}.norm1"] = w[f"{s_}.norm1.weight"].to(F32)
            p[f"{d_}.wqkv"] = w[f"{s_}.attn.wqkv.weight"].to(BF16).contiguous()
            p[f"{d_}.bqkv"] = w[f"{s_}.attn.wqkv.bias"].to(F32)
            p[f"{d_}.wo"] = w[f"{s_}.attn.wo.weight"].to(BF16).contiguous()
            p[f"{d_}.bo"] = w[f"{s_}.attn.wo.bias"].to(F32)
            p[f"{d_}.norm2"] = w[f"{s_}.norm2.weight"].to(F32)
            p[f"{d_}.w1"] = w[f"{s_}.mlp.w1.weight"].to(BF16).contiguous()
            p[f"{d_}.b1"] = w[f"{s_}.mlp.w1.bias"].to(F32)
            p[f"{d_}.w2"] = w[f"{s_}.mlp.w2.weight"].to(BF16).contiguous()
            p[f"{d_}.b2"] = w[f"{s_}.mlp.w2.bias"].to(F32)
    p["enc.norm_f"] = w["enc.norm_f.weight"].to(F32)
    p["enc.proj.w"] = w["enc.proj.weight"].to(BF16).contiguous()
    p["enc.proj.b"] = w["enc.proj.bias"].to(F32)
    p["dec.norm_f"] = w["dec.norm_f.weight"].to(F32)
    ip = torch.zeros(spec.d_model, 64, dtype=F32)                    # K padded to one 64-wide block
    ip[:, : spec.codebook_dim] = w["dec.in_proj.weight"]
    p["dec.in_proj.w"] = ip.to(BF16).contiguous()
    p["dec.in_proj.b"] = w["dec.in_proj.bias"].to(F32)

    # projected codebook, once, in fp32 on the CPU (same arithmetic the fp32 oracle performs)
    cb = torch.nn.functional.linear(w["quantizer.codebook.weight"].to(F32),
                                    w["quantizer.codebook_proj.weight"].to(F32),
                                    w["quantizer.codebook_proj.bias"].to(F32)).contiguous()
    c2 = cb.pow(2).sum(-1).contiguous()
    p["vq.codebook_raw"] = w["quantizer.codebook.weight"].to(F32).contiguous()
    p["vq.codebook"] = cb
    p["vq.c2"] = c2
    c_hi, c_lo = split_bf16(cb, 2)
    n1, n2, n3 = split_bf16(-0.5 * c2, 3)
    packed = torch.zeros(cb.shape[0], 64, dtype=torch.bfloat16)
    packed[:, 0:16], packed[:, 16:32], packed[:, 32:48] = c_hi, c_lo, c_hi
    packed[:, 48], packed[:, 49], packed[:, 50] = n1, n2, n3
    p["vq.packed"] = packed.contiguous()
    cos, sin = rope_tables(max_positions, spec.head_dim, spec.rope_base)
    p["rope.cos"], p["rope.sin"] = cos.t().contiguous(), sin.t().contiguous()   # [32, max_positions]: position contiguous
    return {k: v.contiguous() for k, v in p.items()}


def mc_spec_struct(spec: MagiCodecSpec, max_positions: int) -> nat.McSpec:
    """The C ABI's mc_spec for `spec` (not validated: mc_create applies the same rules as spec.validate())."""
    cs = nat.McSpec()
    cs.sample_rate, cs.n_convs = spec.sample_rate, len(spec.conv_strides)
    for i, c in enumerate(tuple(spec.conv_channels) + (spec.d_model,)):
        cs.conv_channels[i] = c
    for i, s in enumerate(spec.conv_strides):
        cs.conv_strides[i] = s
    cs.d_model, cs.n_heads, cs.ffn_dim = spec.d_model, spec.n_heads, spec.ffn_dim
    cs.enc_layers, cs.dec_layers = spec.enc_layers, spec.dec_layers
    cs.window_left, cs.window_right = spec.window_left, spec.window_right
    cs.norm_eps = spec.norm_eps
    cs.codebook_size, cs.codebook_dim = spec.codebook_size, spec.codebook_dim
    cs.max_positions = max_positions
    return cs


# ------------------------------------------------------------------------------- streaming
class StreamSession:
    """Device-resident rolling context of one AudioTokenizer (mc_stream_* in the C ABI): each push
    uploads only the new chunk / codes; the steady state replays one captured CUDA graph per call."""

    def __init__(self, gen: "B200Generator", channels: int, context_samples: int, max_chunk_samples: int):
        import numpy as np
        self._np = np
        self.gen, self.channels = gen, channels
        self.cap_samples = max(context_samples, max_chunk_samples)
        self.cap_frames = -(-self.cap_samples // gen.hop)
        self._h = C.c_void_p()
        rc = gen._lib.mc_stream_create(gen._handle, channels, context_samples, max_chunk_samples, C.byref(self._h))
        nat.check(gen._lib, gen._handle, rc, "mc_stream_create")

    def reset(self) -> None:
        self.gen._lib.mc_stream_reset(self._h)

    def reset_audio(self) -> None:
        self.gen._lib.mc_stream_reset_part(self._h, 1, 0)

    def reset_codes(self) -> None:
        self.gen._lib.mc_stream_reset_part(self._h, 0, 1)

    def load_audio(self, audio) -> None:
        """float32 [C,n] -> the session's audio context (its last `context` samples); no compute."""
        np = self._np
        audio = np.ascontiguousarray(audio, dtype=np.float32).reshape(self.channels, -1)
        rc = self.gen._lib.mc_stream_load_audio(self._h, audio.ctypes.data, audio.shape[1])
        nat.check(self.gen._lib, self.gen._handle, rc, "mc_stream_load_audio")

    def load_codes(self, codes) -> None:
        """int64 [C,n] -> the session's code context (its last `context` frames); no compute."""
        np = self._np
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(self.channels, -1)
        rc = self.gen._lib.mc_stream_load_codes(self._h, codes.ctypes.data, codes.shape[1])
        nat.check(self.gen._lib, self.gen._handle, rc, "mc_stream_load_codes")

    def set_graphs(self, enabled: bool) -> None:
        self.gen._lib.mc_stream_set_graphs(self._h, 1 if enabled else 0)

    def push_audio(self, chunk, keep_frames: int):
        """chunk float32 [C,n] (numpy) -> int64 codes [C,keep] (numpy)."""
        np = self._np
        chunk = np.ascontiguousarray(chunk, dtype=np.float32).reshape(self.channels, -1)
        n = chunk.shape[1]
        out = np.empty((self.channels, self.cap_frames), dtype=np.int64)
        got = C.c_int32(0)
        with self.gen._serial() as st:
            rc = self.gen._lib.mc_stream_push_audio(self._h, chunk.ctypes.data, n, keep_frames, out.ctypes.data, C.byref(got),
                                                    st.cuda_stream)
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_stream_push_audio")
        return out.reshape(-1)[: self.channels * got.value].reshape(self.channels, got.value)

    def push_codes(self, codes, keep_samples: int):
        """codes int64 [C,n] (numpy) -> float32 wav [C,keep] (numpy)."""
        np = self._np
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(self.channels, -1)
        n = codes.shape[1]
        out = np.empty((self.channels * self.cap_samples,), dtype=np.float32)
        got = C.c_int32(0)
        with self.gen._serial() as st:
            rc = self.gen._lib.mc_stream_push_codes(self._h, codes.ctypes.data, n, keep_samples, out.ctypes.data, C.byref(got),
                                                    st.cuda_stream)
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_stream_push_codes")
        return out[: self.channels * got.value].reshape(self.channels, got.value)

    def set_emit(self, chunk_samples: int, fade_samples: int, target_rms: float, silence_rms_threshold: float, fade_in) -> None:
        """Arm the post-decode chain (mc_stream_set_emit); forgets the previous chunk."""
        np = self._np
        ramp = np.ascontiguousarray(fade_in, dtype=np.float32)
        if ramp.shape != (fade_samples,):
            raise ValueError("fade_in must hold fade_samples values")
        rc = self.gen._lib.mc_stream_set_emit(self._h, chunk_samples, fade_samples, float(target_rms),
                                              float(silence_rms_threshold), ramp.ctypes.data)
        nat.check(self.gen._lib, self.gen._handle, rc, "mc_stream_set_emit")
        self._emit_floats = 2 * chunk_samples + fade_samples

    def push_codes_emit(self, codes):
        """codes int64 [n] -> (float32 [2*chunk + fade] = emitted ++ cross-faded tail ++ new history chunk, had_prev)."""
        np = self._np
        codes = np.ascontiguousarray(codes, dtype=np.int64).reshape(-1)
        out = np.empty((self._emit_floats,), dtype=np.float32)
        had = C.c_int32(0)
        with self.gen._serial() as st:
            rc = self.gen._lib.mc_stream_push_codes_emit(self._h, codes.ctypes.data, codes.shape[0], out.ctypes.data, C.byref(had),
                                                         st.cuda_stream)
            nat.check(self.gen._lib, self.gen._handle, rc, "mc_stream_push_codes_emit")
        return out, bool(had.value)

    def __del__(self):
        try:
            if getattr(self, "_h", None) and self.gen._handle:
                self.gen._lib.mc_stream_destroy(self._h)
                self._h = None
        except Exception:
            pass


# --------------------------------------------------------------------------------- duck type
class _Codebook:
    def __init__(self, raw: torch.Tensor):
        self.weight = raw


class _Quantizer:
    def __init__(self, gen: "B200Generator"):
        self._gen = gen
        self.codebook = _Codebook(gen._dev["vq.codebook_raw"])
        self._table_bf16 = None

    def codebook_proj(self, weight: torch.Tensor) -> torch.Tensor:
        """codebook_proj(codebook.weight) -> the cached projected table (audio_tokenizer.py:158,198).
        Under CUDA autocast the reference's Linear returns bf16; the dtype is mirrored."""
        if weight is not self.codebook.weight and not torch.equal(weight, self.codebook.weight):
            raise NotImplementedError("B200Generator projects its own (frozen) codebook only")
        table = self._gen._dev["vq.codebook"]
        if torch.is_autocast_enabled("cuda"):
            if self._table_bf16 is None:                       # cast once: the reference re-projects 131 072 rows per decode
                self._table_bf16 = table.to(BF16)
            return self._table_bf16
        return table

    def inference(self, z_e: torch.Tensor):
        """(z_q, indices[B,F]) like quantizer.inference (audio_tokenizer.py:192)."""
        gen = self._gen
        cached = gen._last_encoded
        if cached is not None and cached[0] is z_e:
            idx = cached[1]
        else:
            idx = gen.vq_search(z_e.reshape(-1, z_e.shape[-1])).view(z_e.shape[:-1])
        z_q = torch.nn.functional.embedding(idx, gen._dev["vq.codebook"])
        return z_q, idx


class _Serial:
    """Context manager behind B200Generator._serial (a plain class: this sits on the per-frame latency path, and a
    generator-based context manager plus an event record per call cost more than the bookkeeping they do).  The device
    ordering is established only when the stream CHANGES: the new stream then waits for everything queued on the old one
    (Stream.wait_stream records the event at that moment, i.e. after the earlier call's kernels)."""
    __slots__ = ("gen",)

    def __init__(self, gen: "B200Generator"):
        self.gen = gen

    def __enter__(self):
        gen = self.gen
        gen._lock.acquire()
        try:
            st = torch.cuda.current_stream(gen.device)
            last = gen._last_stream
            if last is not None and last.cuda_stream != st.cuda_stream:
                st.wait_stream(last)
            gen._last_stream = st
            return st
        except BaseException:
            gen._lock.release()
            raise

    def __exit__(self, *exc):
        self.gen._lock.release()
        return False


class B200Generator:
    is_b200_native = True

    def __init__(self, spec: MagiCodecSpec, weights: Dict[str, torch.Tensor],
                 device: Optional[torch.device | str] = None, max_positions: int = 2048):
        spec.validate()
        if not torch.cuda.is_available():
            raise RuntimeError("B200Generator needs a CUDA device (sm_100); there is no CPU fallback")
        self.spec = spec
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError(f"B200Generator cannot run on {self.device}; there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.sample_rate = spec.sample_rate
        self.codebook_size = spec.codebook_size
        self.hop = spec.hop
        self.max_positions = max_positions
        self._lib = nat.load_library()
        self._handle = C.c_void_p()
        cs = mc_spec_struct(spec, max_positions)
        rc = self._lib.mc_create(C.byref(cs), self.device.index, C.byref(self._handle))
        nat.check(self._lib, None, rc, "mc_create")
        packed = pack_weights(spec, weights, max_positions)
        self._dev = {k: v.to(self.device) for k, v in packed.items()}
        for name, t in self._dev.items():
            rc = self._lib.mc_set_tensor(self._handle, name.encode(), t.data_ptr(), t.numel())
            nat.check(self._lib, self._handle, rc, f"mc_set_tensor({name})")
        nat.check(self._lib, self._handle, self._lib.mc_finalize(self._handle), "mc_finalize")
        self.quantizer = _Quantizer(self)
        self._last_encoded = None
        # The handle owns ONE workspace arena and its sessions own captured graphs over it: calls on one handle are
        # serialised on the host (threads: tts_server.py:158 runs Flask threaded on one tokenizer; two tokenizers on
        # one model: realtime_agent_resources.py:41-49) and ordered on the device across streams.
        self._lock = threading.RLock()
        self._last_stream = None          # torch stream of the previous engine call (ordering across streams: _Serial)

    # ---- nn.Module-ish surface used by AudioTokenizer.__init__ (:28)
    def eval(self):
        return self

    def to(self, device):
        if torch.device(device).type != "cuda":
            raise RuntimeError("B200Generator lives on its CUDA device; there is no CPU fallback")
        return self

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                self._lib.mc_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    # ---- helpers
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _serial(self) -> "_Serial":
        """Host lock + device ordering for one engine call: work queued on ANOTHER stream by an earlier call must be
        finished with the shared workspace before this call's kernels touch it.  `with gen._serial() as st:` yields the
        calling thread's current torch stream (st.cuda_stream is what the C ABI takes)."""
        return _Serial(self)

    def frames_for(self, samples: int) -> int:
        return -(-samples // self.hop)

    @property
    def launch_count(self) -> int:
        return int(self._lib.mc_launch_count(self._handle))

    def open_stream(self, channels: int, context_samples: int, max_chunk_samples: int = 0) -> StreamSession:
        cap = max(max_chunk_samples, context_samples)
        self.ensure_positions(self.frames_for(cap))
        return StreamSession(self, channels, context_samples, cap)

    def ensure_positions(self, frames: int) -> None:
        """Grow the RoPE tables so that inputs of `frames` frames are accepted (the reference's AudioTokenizer takes
        any length: run_demo.py:55,109 encode / decode whole files in one call).  The new tables are registered under
        the same names; captured stream graphs notice the changed tensor generation and re-capture."""
        if frames <= self.max_positions:
            return
        new_max = 1 << (int(frames) - 1).bit_length()
        cos, sin = rope_tables(new_max, self.spec.head_dim, self.spec.rope_base)
        torch.cuda.synchronize(self.device)                       # nothing in flight reads the old tables
        for name, t in (("rope.cos", cos), ("rope.sin", sin)):
            dev = t.t().contiguous().to(self.device)
            self._dev[name] = dev
            rc = self._lib.mc_set_tensor(self._handle, name.encode(), dev.data_ptr(), dev.numel())
            nat.check(self._lib, self._handle, rc, f"mc_set_tensor({name})")
        self.set_option("max_positions", new_max)
        nat.check(self._lib, self._handle, self._lib.mc_finalize(self._handle), "mc_finalize")
        self.max_positions = new_max

    def set_debug_impl(self, attention: int = 0, vq: int = 0) -> None:
        nat.check(self._lib, self._handle, self._lib.mc_set_debug_impl(self._handle, attention, vq), "mc_set_debug_impl")

    def set_option(self, key: str, value: int) -> None:
        nat.check(self._lib, self._handle, self._lib.mc_set_option(self._handle, key.encode(), int(value)), "mc_set_option")

    PROFILE_CLASSES = ("gemm", "attention", "vq", "elementwise")

    def profile_begin(self) -> None:
        nat.check(self._lib, self._handle, self._lib.mc_profile_begin(self._handle), "mc_profile_begin")

    def profile_end(self) -> Dict[str, Dict[str, float]]:
        n = len(self.PROFILE_CLASSES)
        ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        rc = self._lib.mc_profile_end(self._handle, ms, fl, by, cnt, n)
        nat.check(self._lib, self._handle, rc, "mc_profile_end")
        return {name: {"ms": ms[i], "flops": fl[i], "bytes": by[i], "launches": int(cnt[i])}
                for i, name in enumerate(self.PROFILE_CLASSES)}

    # ---- fast batched entry points
    def encode(self, wav: torch.Tensor, keep_last_frames: int = 0, return_margin: bool = False,
               return_latents: bool = False, row_stride: Optional[int] = None, num_windows: Optional[int] = None,
               window_samples: Optional[int] = None):
        """wav fp32 [B,T] on the engine's device -> int64 codes [B,Fk].

        ``row_stride/num_windows/window_samples`` describe overlapping windows over a flat buffer
        (window b = wav.view(-1)[b*row_stride : b*row_stride + window_samples]) — the chunked
        encode with context never materialises its 20x amplified input."""
        if wav.device != self.device:
            wav = wav.to(self.device)
        wav = wav.to(F32)
        if row_stride is None:
            if wav.dim() == 1:
                wav = wav[None]
            wav = wav.contiguous()
            B, T, ld = wav.shape[0], wav.shape[1], wav.shape[1]
        else:
            wav = wav.contiguous().view(-1)
            B, T, ld = int(num_windows), int(window_samples), int(row_stride)
            if (B - 1) * ld + T > wav.numel():
                raise ValueError("windows exceed the audio buffer")
        F = self.frames_for(T)
        self.ensure_positions(F)
        keep = F if keep_last_frames <= 0 or keep_last_frames > F else keep_last_frames
        codes = torch.empty((B, keep), dtype=torch.int64, device=self.device)
        margin = torch.empty((B, keep), dtype=F32, device=self.device) if return_margin else None
        z_e = torch.empty((B, F, self.spec.codebook_dim), dtype=F32, device=self.device) if return_latents else None
        with self._serial():
            rc = self._lib.mc_encode(self._handle, wav.data_ptr(), ld, B, T, keep, codes.data_ptr(), nat.ptr(margin),
                                     nat.ptr(z_e), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_encode")
        if return_margin or return_latents:
            return codes, margin, z_e
        return codes

    def decode(self, codes: torch.Tensor, keep_last_samples: int = 0) -> torch.Tensor:
        """int64 codes [B,F] -> fp32 wav [B,Tk]."""
        codes = codes.to(self.device, torch.int64).contiguous()
        if codes.dim() == 1:
            codes = codes[None]
        B, F = codes.shape
        self.ensure_positions(F)
        total = F * self.hop
        keep = total if keep_last_samples <= 0 or keep_last_samples > total else keep_last_samples
        wav = torch.empty((B, keep), dtype=F32, device=self.device)
        with self._serial():
            rc = self._lib.mc_decode(self._handle, codes.data_ptr(), B, F, keep, wav.data_ptr(), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_decode")
        return wav

    def render_chunks(self, windows: torch.Tensor, chunk: int, fade_in: torch.Tensor, last_len: Optional[int] = None,
                      target_rms: float = 0.0, silence_rms_threshold: float = 0.003) -> torch.Tensor:
        """The agent's output chain over every chunk of one mono stream in ONE launch (mc_render_chunks).
        windows fp32 [n_chunks, ld >= chunk + L] on the device: row 0 = the first chunk, rows i >= 1 = L preroll ++ chunk;
        fade_in fp32 [L] (create_crossfade_ramps).  Returns fp32 [(n_chunks-1)*chunk + last_len] =
        np.concatenate(OutputChunkEmitter.audio_history_ch1) cut to the real samples of the last chunk."""
        windows = windows.to(self.device, F32).contiguous()
        n_chunks, ld = windows.shape
        last_len = chunk if last_len is None else int(last_len)
        fade_in = fade_in.to(self.device, F32).contiguous()
        out = torch.empty(((n_chunks - 1) * chunk + last_len,), dtype=F32, device=self.device)
        with self._serial():
            rc = self._lib.mc_render_chunks(self._handle, windows.data_ptr(), ld, n_chunks, chunk, fade_in.numel(),
                                            last_len, float(target_rms), float(silence_rms_threshold), fade_in.data_ptr(),
                                            out.data_ptr(), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_render_chunks")
        return out

    PCM_S16, PCM_F32 = 1, 4                     # MC_PCM_* of include/magicodec_b200.h

    def f32_to_pcm(self, wav: torch.Tensor, fmt: int = 1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Planar fp32 [C, T] (or [T]) on the device -> interleaved PCM [T, C] (mc_op_f32_to_pcm): int16 for
        fmt = PCM_S16 (clamp(rint(x * 32768)), NaN -> 0), float32 for PCM_F32.  `out` may be a pinned host tensor of
        that dtype with at least T*C elements; the kernel writes into it directly (wait on the stream before reading)."""
        if wav.dim() == 1:
            wav = wav[None]
        if wav.stride(-1) != 1:
            wav = wav.contiguous()
        C, T = wav.shape
        dtype = torch.int16 if fmt == self.PCM_S16 else F32
        if out is None:
            out = torch.empty((T, C), dtype=dtype, device=self.device)
        if out.dtype != dtype or out.numel() < T * C or not out.is_contiguous():
            raise ValueError(f"f32_to_pcm: out must be a contiguous {dtype} buffer of at least {T * C} elements")
        with self._serial():
            rc = self._lib.mc_op_f32_to_pcm(self._handle, wav.data_ptr(), wav.stride(0) if C > 1 else T, C, T, int(fmt),
                                            out.data_ptr(), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_op_f32_to_pcm")
        return out.view(-1)[: T * C].view(T, C)

    def vq_search(self, z: torch.Tensor, return_margin: bool = False):
        z = z.to(self.device, F32).contiguous()
        M = z.shape[0]
        codes = torch.empty((M,), dtype=torch.int64, device=self.device)
        margin = torch.empty((M,), dtype=F32, device=self.device) if return_margin else None
        with self._serial():
            rc = self._lib.mc_vq_search(self._handle, z.data_ptr(), M, codes.data_ptr(), nat.ptr(margin), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_vq_search")
        return (codes, margin) if return_margin else codes

    def embed_distance(self, ids: torch.Tensor, vocab_start: int = 0, ref: Optional[torch.Tensor] = None,
                       want_mean: bool = False):
        """ids int64 [rows,n] -> mean_j ||E[ids - vocab_start] - ref|| per row (fp32 [rows]) and, optionally,
        the mean embedding per row (fp32 [rows,dq]) — external_tts_duplex_aligner.py:14-24 on the cached codebook."""
        ids = ids.to(self.device, torch.int64).contiguous()
        if ids.dim() == 1:
            ids = ids[None]
        rows, n = ids.shape
        ref = None if ref is None else ref.to(self.device, F32).contiguous()
        dist = torch.empty((rows,), dtype=F32, device=self.device)
        mean = torch.empty((rows, self.spec.codebook_dim), dtype=F32, device=self.device) if want_mean else None
        with self._serial():
            rc = self._lib.mc_embed_distance(self._handle, ids.data_ptr(), rows, n, int(vocab_start), nat.ptr(ref),
                                             dist.data_ptr(), nat.ptr(mean), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_embed_distance")
        return (dist, mean) if want_mean else dist

    # ---- the reference wrapper's call sequence (audio_tokenizer.py:190-192, 198-200)
    def pad_audio(self, x: torch.Tensor) -> torch.Tensor:
        return x                     # right padding to the hop multiple happens inside the first conv kernel

    def encoder(self, x: torch.Tensor) -> torch.Tensor:
        codes, _, z_e = self.encode(x, return_latents=True)
        self._last_encoded = (z_e, codes)
        return z_e

    def decoder(self, z_q: torch.Tensor) -> torch.Tensor:
        z = z_q.to(self.device, F32).contiguous()
        B, F = z.shape[0], z.shape[1]
        self.ensure_positions(F)
        wav = torch.empty((B, F * self.hop), dtype=F32, device=self.device)
        with self._serial():
            rc = self._lib.mc_decode_latents(self._handle, z.data_ptr(), B, F, 0, wav.data_ptr(), self._stream())
            nat.check(self._lib, self._handle, rc, "mc_decode_latents")
        return wav[:, None, :]

    # ---- operator-level hooks (parity tests / profiling)
    def op_gemm(self, A, W, bias=None, act=0, out_mode=0, out=None, a_k_wrap=None, M=None, K=None,
                grp_in=0, grp_valid=0, grp_stride=0, grp_off=0, ldo=None, rope_cols=0, rope_period=0, block_n=0):
        N = W.shape[0]
        K = W.shape[1] if K is None else K
        a_k_wrap = A.shape[-1] if a_k_wrap is None else a_k_wrap
        a_rows = A.numel() // a_k_wrap
        M = a_rows if M is None else M
        ldo = N if ldo is None else ldo
        if out is None:
            out = torch.zeros((M, N), dtype=BF16 if out_mode == 0 else F32, device=self.device)
        rc = self._lib.mc_op_gemm(self._handle, A.data_ptr(), a_rows, a_k_wrap, W.data_ptr(), nat.ptr(bias), M, N, K,
                                  act, out_mode, out.data_ptr(), ldo, grp_in, grp_valid, grp_stride, grp_off,
                                  rope_cols, rope_period, block_n, self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_gemm")
        return out

    def op_gemm_fused(self, A, W, bias=None, act=0, out_mode=1, out=None, row_stats=None, xb_gamma=None, rope_cols=0,
                      rope_period=0, block_n=0):
        """GEMM with the fused-RMSNorm roles: row_stats [M, n] -> consumer; xb_gamma [N] -> producer (returns out, xb, stats)."""
        M, K = A.shape
        N = W.shape[0]
        if out is None:
            out = torch.zeros((M, N), dtype=BF16 if out_mode == 0 else F32, device=self.device)
        xb = torch.zeros((M, N), dtype=BF16, device=self.device) if xb_gamma is not None else None
        st = torch.zeros((M, N // 64), dtype=F32, device=self.device) if xb_gamma is not None else None
        rc = self._lib.mc_op_gemm_fused(self._handle, A.data_ptr(), W.data_ptr(), nat.ptr(bias), M, N, K, act, out_mode, out.data_ptr(),
                                        nat.ptr(row_stats), 0 if row_stats is None else row_stats.shape[1], nat.ptr(xb), nat.ptr(xb_gamma),
                                        nat.ptr(st), rope_cols, rope_period, block_n, self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_gemm_fused")
        return (out, xb, st) if xb_gamma is not None else out

    def op_rowstats(self, x, gamma):
        M, d = x.shape
        xb = torch.empty((M, d), dtype=BF16, device=self.device)
        st = torch.empty((M, d // 64), dtype=F32, device=self.device)
        rc = self._lib.mc_op_rowstats(self._handle, x.data_ptr(), gamma.data_ptr(), xb.data_ptr(), st.data_ptr(), M, d, self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_rowstats")
        return xb, st

    def op_emit_chunk(self, wav, chunk, fade, has_prev, target_rms, silence_thr, fade_in, prev_tail):
        out = torch.empty((2 * chunk + fade,), dtype=F32, device=self.device)
        rc = self._lib.mc_op_emit_chunk(self._handle, wav.data_ptr(), wav.numel(), chunk, fade, int(has_prev), float(target_rms),
                                        float(silence_thr), fade_in.data_ptr(), prev_tail.data_ptr(), out.data_ptr(), self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_emit_chunk")
        return out

    def op_embed_distance(self, table, ids, vocab_start=0, ref=None, want_mean=False):
        rows, n = ids.shape
        dist = torch.empty((rows,), dtype=F32, device=self.device)
        mean = torch.empty((rows, 16), dtype=F32, device=self.device) if want_mean else None
        rc = self._lib.mc_op_embed_distance(self._handle, table.data_ptr(), table.shape[0], ids.data_ptr(), rows, n,
                                            int(vocab_start), nat.ptr(ref), dist.data_ptr(), nat.ptr(mean), self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_embed_distance")
        return (dist, mean) if want_mean else dist

    def op_rmsnorm(self, x, gamma):
        out = torch.empty(x.shape, dtype=BF16, device=self.device)
        rc = self._lib.mc_op_rmsnorm(self._handle, x.data_ptr(), gamma.data_ptr(), out.data_ptr(), x.shape[0],
                                     x.shape[1], self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_rmsnorm")
        return out

    def op_attention(self, qkv, B, F, impl=0, out_rows=None, phase=0):
        out_rows = F if out_rows is None else out_rows
        out = torch.empty((B * out_rows, self.spec.d_model), dtype=BF16, device=self.device)
        rc = self._lib.mc_op_attention(self._handle, qkv.data_ptr(), out.data_ptr(), B, F, out_rows, phase, impl,
                                       self._stream())
        nat.check(self._lib, self._handle, rc, "mc_op_attention")
        return out
