"""MagiCodecSpec — the single source of truth for the codec architecture.

The reference never shows the network: ``AudioTokenizer`` only touches
``model.sample_rate``, ``.codebook_size``, ``.pad_audio``, ``.encoder``,
``.quantizer.{inference,codebook,codebook_proj}`` and ``.decoder``
(/root/reference/realtime_codec_agent/audio_tokenizer.py:28,32,36,158,190-200).
What the reference pins is: 16 kHz, 50 Hz frames (hop 320), one codebook of
131 072 entries, projected codebook dim 16
(/root/reference/realtime_codec_agent/codec_llama.py:17-19).  Everything else
(depth, width, window, conv stack) is a field here, shared by the oracle, the
weight packer and the CUDA engine; the defaults are the SURVEY.md §7.0
"unverified default".

Layout of the network this spec describes
-----------------------------------------
encode:  wav[B,T] --pad to hop multiple--> causal strided conv stack
         (kernel = 2*stride each, tanh-GELU between layers) --> [B,F,d]
         --> enc_layers x pre-RMSNorm transformer block (RoPE, sliding-window
         attention keys j in [i-wl, i+wr], tanh-GELU MLP) --> RMSNorm -->
         Linear d->dq --> nearest neighbour over codebook_proj(codebook)
decode:  codes --> rows of codebook_proj(codebook) --> Linear dq->d -->
         dec_layers x block --> RMSNorm --> causal transposed-conv stack
         (mirror of the encoder stack) --> wav[B,1,F*hop]
"""
from __future__ import annotations

import dataclasses
import math
from dataclasses import dataclass
from typing import Tuple


@dataclass(frozen=True)
class MagiCodecSpec:
    sample_rate: int = 16000
    # encoder conv stack: channels after each layer (last one is d_model) and strides
    conv_channels: Tuple[int, ...] = (32, 128, 512)
    conv_strides: Tuple[int, ...] = (4, 4, 4, 5)
    d_model: int = 1024
    n_heads: int = 16
    ffn_dim: int = 4096
    enc_layers: int = 8
    dec_layers: int = 8
    window_left: int = 32
    window_right: int = 0
    rope_base: float = 10000.0
    norm_eps: float = 1e-5
    codebook_size: int = 131072
    codebook_dim: int = 16

    # ---- derived -----------------------------------------------------
    @property
    def hop(self) -> int:
        return math.prod(self.conv_strides)

    @property
    def head_dim(self) -> int:
        return self.d_model // self.n_heads

    @property
    def enc_channels(self) -> Tuple[int, ...]:
        """Channel count entering/leaving each encoder conv: (1, c0, c1, ..., d)."""
        return (1,) + tuple(self.conv_channels) + (self.d_model,)

    @property
    def dec_channels(self) -> Tuple[int, ...]:
        """Channel count entering/leaving each decoder transposed conv: (d, ..., c0, 1)."""
        return tuple(reversed(self.enc_channels))

    @property
    def dec_strides(self) -> Tuple[int, ...]:
        return tuple(reversed(self.conv_strides))

    def validate(self) -> None:
        assert len(self.conv_strides) == len(self.conv_channels) + 1
        assert len(self.conv_strides) >= 2, "need a first (CUDA-core) conv and at least one GEMM conv"
        assert self.d_model % self.n_heads == 0
        assert self.head_dim == 64, "attention kernels are instantiated for head_dim 64"
        assert self.d_model % 64 == 0 and self.ffn_dim % 64 == 0
        assert self.codebook_dim == 16, "VQ kernel packs split-bf16 16-d rows into one 128-byte line"
        assert self.codebook_size % 256 == 0
        assert 0 <= self.window_left <= 96 and 0 <= self.window_right <= 32
        ch = self.enc_channels
        s0, c0 = self.conv_strides[0], ch[1]
        # conv_first_kernel is instantiated for 8 and 16 taps and gives each thread 8 channels of a 256-thread block;
        # the last transposed conv (Cout = 1) mirrors it and reads 16-byte groups of 8 channels
        assert s0 in (4, 8), f"conv 0: stride {s0} unsupported (the first conv runs strides 4 and 8)"
        assert c0 % 8 == 0 and 256 % (c0 // 8) == 0, \
            f"conv 0: {c0} channels unsupported (need 8 * 2^k channels, at most 2048)"
        for i, s in enumerate(self.conv_strides):
            if i >= 1:
                # GEMM convs: the K loop walks stride*Cin-wide row blocks in 64-element steps
                assert (s * ch[i]) % 64 == 0, f"conv {i}: stride*Cin must be a multiple of 64"
        dch = self.dec_channels
        for i, s in enumerate(self.dec_strides[:-1]):
            assert dch[i] % 64 == 0, f"tconv {i}: Cin must be a multiple of 64"
        assert dch[-2] % 8 == 0

    # ---- algorithmic work (shared by bench.py's roofline and DESIGN.md) -------
    def conv_flops(self, frames: int) -> int:
        """FLOPs of the encoder conv stack for `frames` output frames of one window."""
        total, t = 0, frames * self.hop
        ch = self.enc_channels
        for i, s in enumerate(self.conv_strides):
            t //= s
            total += 2 * t * (2 * s * ch[i]) * ch[i + 1]
        return total

    def tconv_flops(self, frames: int) -> int:
        total, t = 0, frames
        ch = self.dec_channels
        for i, s in enumerate(self.dec_strides):
            total += 2 * t * (2 * ch[i]) * (s * ch[i + 1])
            t *= s
        return total

    def block_flops(self, frames: int) -> int:
        """One transformer block over a window of `frames` frames (full window computed)."""
        d, f = self.d_model, self.ffn_dim
        span = min(frames, self.window_left + self.window_right + 1)
        return (2 * frames * d * 3 * d + 2 * frames * d * d + 2 * 2 * frames * d * f
                + 4 * frames * span * d)

    def vq_flops(self, frames: int) -> int:
        return 2 * frames * self.codebook_size * self.codebook_dim

    def encode_flops(self, frames: int, vq_frames: int | None = None) -> int:
        vq_frames = frames if vq_frames is None else vq_frames
        return (self.conv_flops(frames) + self.enc_layers * self.block_flops(frames)
                + 2 * frames * self.d_model * self.codebook_dim + self.vq_flops(vq_frames))

    def decode_flops(self, frames: int) -> int:
        return (2 * frames * self.codebook_dim * self.d_model
                + self.dec_layers * self.block_flops(frames) + self.tconv_flops(frames))

    def weight_bytes_bf16(self, stack: str = "enc") -> int:
        d, f = self.d_model, self.ffn_dim
        n_layers = self.enc_layers if stack == "enc" else self.dec_layers
        per_layer = 2 * (3 * d * d + d * d + 2 * d * f)
        ch = self.enc_channels
        conv = sum(2 * (2 * s * ch[i]) * ch[i + 1] for i, s in enumerate(self.conv_strides))
        return n_layers * per_layer + conv + 2 * d * self.codebook_dim

    def replace(self, **kw) -> "MagiCodecSpec":
        return dataclasses.replace(self, **kw)


#: the configuration every BASELINE.json workload is quoted on ("MagiCodec-50Hz-Base")
DEFAULT_SPEC = MagiCodecSpec()

#: a small spec the fp32 CPU oracle finishes in seconds; exercised by the parity tests
TINY_SPEC = MagiCodecSpec(
    conv_channels=(32, 64, 64), d_model=128, n_heads=2, ffn_dim=256,
    enc_layers=2, dec_layers=2, codebook_size=4096,
)

#: mid-size spec: full-width kernels' tile shapes, shallow enough for the CPU oracle
MID_SPEC = MagiCodecSpec(
    conv_channels=(32, 128, 256), d_model=512, n_heads=8, ffn_dim=1024,
    enc_layers=3, dec_layers=3, codebook_size=16384,
)
