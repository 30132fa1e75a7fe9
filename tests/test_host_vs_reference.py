"""CPU: the product AudioTokenizer and the UNMODIFIED reference wrapper, each driving the same oracle model object, must agree
call by call (strings equal, waveforms equal, bookkeeping equal) across the call patterns the reference's callers use
(realtime_agent_v2.py:504-579, run_stream_codes.py:14-68, tts_server.py:59).

The reference wrapper is not part of this repository, so every call pattern below is also pinned by
tests/golden/golden_host_calls.npz (tests/golden/make_golden_host_calls.py): strings and bookkeeping exactly, waveforms and
embeddings by shape and a fixed sample of values.  The product is checked against those vectors everywhere, and against the
reference itself, bit for bit, wherever the reference is installed."""
import os

import numpy as np
import pytest

import realtime_codec_agent_b200 as pkg
from oracle.magicodec_oracle import OracleGenerator
from oracle.reference_wrapper import load_reference_audio_tokenizer, reference_available
from tests.golden_calls import assert_identical, assert_matches_golden, ords

CHANNELS = [1, 2]
CHUNK_MS = [20, 100, 580, 1000]


def streaming_calls(Tok, model, channels, chunk_ms):
    """Streaming tokenize_audio / detokenize_audio in chunk_ms pieces with a 320-sample preroll -> {name: array}."""
    tok = Tok(codec_model=model, num_channels=channels, device="cpu")
    out = {"framerate": np.float64(tok.framerate), "context_frames": np.int64(tok.context_frames)}
    n = chunk_ms * 16
    total = min(3.0, 12 * chunk_ms / 1000.0)
    wav = np.stack([pkg.synth_audio(int(total * 16000), file_id=3, channel=c).numpy() for c in range(channels)])
    wav = wav[0] if channels == 1 else wav
    for i, s0 in enumerate(range(0, wav.shape[-1], n)):
        s = tok.tokenize_audio(wav[..., s0:s0 + n])
        (sr, w), h, pre = tok.detokenize_audio(s, preroll_samples=320)
        out.update({f"{i}_codes": ords(s), f"{i}_sr": np.int64(sr), f"{i}_hanging": ords(h), f"{i}_preroll": np.int64(pre),
                    f"{i}_wav": np.asarray(w)})
    out["tokenize_context"] = np.asarray(tok.tokenize_context)
    out["detokenize_context"] = ords(tok.detokenize_context)
    return out


def int16_calls(Tok, model):
    """int16 (sr, pcm) tuples with a stereo->mono downmix, stereo strings cut mid-frame, and the small helpers."""
    out = {}
    tok = Tok(codec_model=model, device="cpu")
    st = np.stack([pkg.synth_audio(8000, channel=c).numpy() for c in range(2)])
    out["int16_mono_codes"] = ords(tok.tokenize_audio((16000, (st * 32767).astype(np.int16))))
    tok2 = Tok(codec_model=model, num_channels=2, device="cpu")
    s = tok2.tokenize_audio(st)
    out["stereo_codes"] = ords(s)
    for cut in (len(s) - 1, len(s) - 3, 7):
        tok2.reset_context()
        (_, w), h, p = tok2.detokenize_audio(s[:cut], preroll_samples=100)
        out.update({f"cut{cut}_wav": np.asarray(w), f"cut{cut}_hanging": ords(h), f"cut{cut}_preroll": np.int64(p)})
    out["codes_str_secs"] = np.float64(tok.get_audio_codes_str_secs(s))
    out["codec_embeddings"] = tok.get_codec_embeddings().detach().cpu().numpy()
    out["silence_codes"] = tok._encode_silence(1.0).cpu().numpy()
    kept, hanging = tok._drop_hanging_channel_codes("abc")
    out["drop_hanging_kept"], out["drop_hanging_hanging"] = ords(kept), ords(hanging)
    return out


@pytest.fixture(scope="module")
def model():
    return OracleGenerator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0))


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "golden_host_calls.npz"))


@pytest.mark.parametrize("channels", CHANNELS)
@pytest.mark.parametrize("chunk_ms", CHUNK_MS)
def test_streaming_encode_decode_agree(model, golden, channels, chunk_ms):
    ours = streaming_calls(pkg.AudioTokenizer, model, channels, chunk_ms)
    assert_matches_golden(ours, golden, f"stream_c{channels}_{chunk_ms}ms")
    if reference_available():
        assert_identical(ours, streaming_calls(load_reference_audio_tokenizer(), model, channels, chunk_ms))


def test_int16_tuple_mono_downmix_and_hanging(model, golden):
    ours = int16_calls(pkg.AudioTokenizer, model)
    assert_matches_golden(ours, golden, "int16")
    if reference_available():
        assert_identical(ours, int16_calls(load_reference_audio_tokenizer(), model))


def test_codec_chars_match_shim():
    from oracle.shims.codec_bpe.core import converter as shim
    rng = np.random.default_rng(0)
    for nb, K in ((1, 131072), (2, 1024), (4, 2048)):
        codes = rng.integers(0, K, size=(nb, 37))
        for off in (pkg.UNICODE_OFFSET, pkg.UNICODE_OFFSET_LARGE):
            if off + nb * K > 0x110000:
                continue
            a = shim.codes_to_chars(codes, K, unicode_offset=off)
            assert a == pkg.codes_to_chars(codes, K, unicode_offset=off)
            assert np.array_equal(shim.chars_to_codes(a, nb, K, unicode_offset=off),
                                  pkg.chars_to_codes(a, nb, K, unicode_offset=off))
            assert np.array_equal(pkg.chars_to_codes(a, nb, K, unicode_offset=off), codes)
