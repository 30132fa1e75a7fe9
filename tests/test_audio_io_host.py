"""CPU: container parsing, the native FLAC decoder, G.711 tables, host sample conversion and the polyphase
resampler of audio_io.py (the host half of the corpus ingest path, SURVEY §8 f1 / a13)."""
import glob
import hashlib
import os
import struct

import numpy as np
import pytest

from realtime_codec_agent_b200 import audio_io as aio
from tests import flac_writer as fw

SCIPY_WAVS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wav")    # SciPy's WAV test vectors


def _write_wav(path, sr, data, tag=1, bits=16, extensible=False):
    """data: interleaved raw bytes."""
    ch = data[1]
    raw = data[0]
    align = ch * bits // 8
    if extensible:
        fmt = struct.pack("<HHIIHHHHIH14s", 0xFFFE, ch, sr, sr * align, align, bits, 22, bits, 0, tag, b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71")
    else:
        fmt = struct.pack("<HHIIHH", tag, ch, sr, sr * align, align, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"LIST" + struct.pack("<I", 3) + b"abc\x00" + \
        b"data" + struct.pack("<I", len(raw)) + raw
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_wav_variants_match_scipy(tmp_path):
    from scipy.io import wavfile
    checked = 0
    for p in sorted(glob.glob(os.path.join(SCIPY_WAVS, "test-*.wav"))):
        try:
            pcm = aio.read_audio(p)
        except aio.UnsupportedAudio:
            continue                                     # odd container bit depths (20/36/53-bit) are not corpus formats
        try:
            sr, ref = wavfile.read(p)
        except Exception:                                # scipy has no G.711 decoder; those files are checked below
            continue
        ref = ref[:, None] if ref.ndim == 1 else ref
        if ref.dtype == np.uint8:
            want = (ref.astype(np.float32) - 128.0) / 128.0
        elif np.issubdtype(ref.dtype, np.integer):
            want = ref.astype(np.float32) / float(np.iinfo(ref.dtype).max + 1)
        else:
            want = ref.astype(np.float32)
        got = aio.pcm_to_float(pcm)
        assert pcm.sample_rate == sr and got.shape == want.T.shape, p
        assert np.array_equal(got, want.T), p
        checked += 1
    assert checked >= 8
    # our own writer: extensible header, a LIST chunk with odd size before the data, 24-bit, 8-bit unsigned, stereo
    rng = np.random.default_rng(0)
    s16 = rng.integers(-32768, 32767, size=(1000, 2), dtype=np.int16)
    _write_wav(tmp_path / "a.wav", 8000, (s16.tobytes(), 2), extensible=True)
    pcm = aio.read_audio(str(tmp_path / "a.wav"))
    assert (pcm.sample_rate, pcm.channels, pcm.frames, pcm.fmt) == (8000, 2, 1000, aio.PCM_S16)
    assert np.array_equal(aio.pcm_to_float(pcm), s16.T.astype(np.float32) / 32768.0)
    assert np.array_equal(aio.pcm_to_float(pcm, mono=True)[0], (s16[:, 0].astype(np.float32) / 32768 + s16[:, 1].astype(np.float32) / 32768) / 2)
    u8 = rng.integers(0, 255, size=500, dtype=np.uint8)
    _write_wav(tmp_path / "b.wav", 16000, (u8.tobytes(), 1), bits=8)
    assert np.array_equal(aio.pcm_to_float(aio.read_audio(str(tmp_path / "b.wav")))[0], (u8.astype(np.float32) - 128) / 128)
    v24 = rng.integers(-(1 << 23), (1 << 23) - 1, size=300)
    raw = b"".join(int(v).to_bytes(3, "little", signed=True) for v in v24)
    _write_wav(tmp_path / "c.wav", 44100, (raw, 1), bits=24)
    assert np.array_equal(aio.pcm_to_float(aio.read_audio(str(tmp_path / "c.wav")))[0], v24.astype(np.float32) / 8388608.0)
    assert aio.probe_audio(str(tmp_path / "c.wav")) == (44100, 1, 300)


def test_g711_known_answers_and_ulaw_wav(tmp_path):
    ulaw, alaw = aio._g711_tables()
    # ITU-T G.711 corner values
    assert ulaw[0xFF] == 0 and ulaw[0x7F] == 0 and ulaw[0x80] == 32124 and ulaw[0x00] == -32124 and ulaw[0xFE] == 8 and ulaw[0x7E] == -8
    assert alaw[0xD5] == 8 and alaw[0x55] == -8 and alaw[0xAA] == 32256 and alaw[0x2A] == -32256
    assert np.array_equal(ulaw[128:], -ulaw[:128]) and np.array_equal(alaw[128:], -alaw[:128])
    p = os.path.join(SCIPY_WAVS, "test-8000Hz-le-1ch-1byte-ulaw.wav")
    pcm = aio.read_audio(p)
    assert pcm.fmt == aio.PCM_ULAW and pcm.sample_rate == 8000 and pcm.channels == 1
    x = aio.pcm_to_float(pcm)
    assert x.shape == (1, pcm.frames) and np.abs(x).max() <= 1.0
    raw = bytes(range(256))
    _write_wav(tmp_path / "a.wav", 8000, (raw, 1), tag=6, bits=8)
    assert np.array_equal(aio.pcm_to_float(aio.read_audio(str(tmp_path / "a.wav")))[0], alaw.astype(np.float32) / 32768)


def test_sphere_files(tmp_path):
    rng = np.random.default_rng(1)

    def sph(path, fields, payload):
        body = "NIST_1A\n   1024\n" + "".join(f"{k} {t} {v}\n" for k, t, v in fields) + "end_head\n"
        with open(path, "wb") as f:
            f.write(body.encode().ljust(1024, b" ") + payload)

    s = rng.integers(-32768, 32767, size=(700, 2), dtype=np.int16)
    sph(tmp_path / "be.sph", [("sample_count", "-i", 700), ("sample_n_bytes", "-i", 2), ("channel_count", "-i", 2),
                              ("sample_byte_format", "-s2", "10"), ("sample_rate", "-i", 8000), ("sample_coding", "-s3", "pcm")],
        s.astype(">i2").tobytes())
    pcm = aio.read_audio(str(tmp_path / "be.sph"))
    assert (pcm.sample_rate, pcm.channels, pcm.frames, pcm.big_endian) == (8000, 2, 700, True)
    assert np.array_equal(aio.pcm_to_float(pcm), s.T.astype(np.float32) / 32768)
    u = rng.integers(0, 255, size=(900, 2), dtype=np.uint8)
    sph(tmp_path / "ul.sph", [("sample_count", "-i", 900), ("sample_n_bytes", "-i", 1), ("channel_count", "-i", 2),
                              ("sample_byte_format", "-s1", "1"), ("sample_rate", "-i", 8000), ("sample_coding", "-s4", "ulaw")], u.tobytes())
    pcm = aio.read_audio(str(tmp_path / "ul.sph"))
    assert pcm.fmt == aio.PCM_ULAW and aio.probe_audio(str(tmp_path / "ul.sph")) == (8000, 2, 900)
    assert np.array_equal(aio.pcm_to_float(pcm), (aio._g711_tables()[0][u].T.astype(np.float32)) / 32768)
    sph(tmp_path / "sh.sph", [("sample_count", "-i", 10), ("sample_n_bytes", "-i", 2), ("channel_count", "-i", 1),
                              ("sample_rate", "-i", 8000), ("sample_coding", "-s26", "pcm,embedded-shorten-v2.00")], b"\x00" * 20)
    with pytest.raises(aio.UnsupportedAudio, match="sph2pipe"):
        aio.read_audio(str(tmp_path / "sh.sph"))


def _speechlike(n, bits, seed, channels=1):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    amp = (1 << (bits - 1)) * 0.4
    out = []
    for c in range(channels):
        x = amp * np.sin(2 * np.pi * (0.011 + 0.003 * c) * t) * (0.5 + 0.5 * np.sin(2 * np.pi * 0.0007 * t + c)) + rng.normal(0, amp * 0.01, n)
        out.append(np.round(x).astype(np.int64))
    if channels == 2:
        out[1] = (0.8 * out[0] + 0.2 * out[1]).astype(np.int64)            # correlated channels: side coding is meaningful
    return np.stack(out)


def _decode_to_int(path_or_bytes, tmp_path, name="x.flac"):
    p = tmp_path / name
    p.write_bytes(path_or_bytes)
    pcm = aio.read_audio(str(p))
    raw = pcm.payload
    if pcm.fmt == aio.PCM_S16:
        v = raw.view("<i2").astype(np.int64)
    else:
        v = raw.view("<i4").astype(np.int64)
    return pcm, v.reshape(pcm.frames, pcm.channels).T


@pytest.mark.parametrize("case", ["fixed_mono16", "lpc_stereo16_modes", "verbatim_constant", "escape_rice2", "wasted_24bit", "odd_blocks_8bit"])
def test_flac_decoder_against_the_test_encoder(tmp_path, case):
    if case == "fixed_mono16":
        pcm = _speechlike(9000, 16, 1)
        plan = lambda b, c: ("fixed", {"order": b % 5, "porder": b % 4})
        data, bps, sr, bs = fw.encode_flac(pcm, 16000, 16, 4096, plan), 16, 16000, 4096
    elif case == "lpc_stereo16_modes":
        pcm = _speechlike(5000, 16, 2, channels=2)
        plan = lambda b, c: ("lpc", {"order": 1 + (3 * b + 5 * c) % 12, "porder": 3, "precision": 12 + b % 3})
        plan.stereo = lambda b: [0, 8, 9, 10][b % 4]
        data, bps, sr, bs = fw.encode_flac(pcm, 8000, 16, 1024, plan), 16, 8000, 1024
    elif case == "verbatim_constant":
        pcm = _speechlike(2048, 16, 3, channels=2)
        pcm[1, :] = -1234
        plan = lambda b, c: ("constant", {}) if c == 1 else ("verbatim", {})
        data, bps, sr, bs = fw.encode_flac(pcm, 44100, 16, 512, plan, id3=True), 16, 44100, 512
    elif case == "escape_rice2":
        pcm = _speechlike(4096, 16, 4)
        pcm[0, 1000:1010] = 32767                                            # outliers: large residuals
        plan = lambda b, c: ("fixed", {"order": 3, "porder": 2, "method": 1, "escape": True})
        data, bps, sr, bs = fw.encode_flac(pcm, 22050, 16, 2048, plan), 16, 22050, 2048
    elif case == "wasted_24bit":
        pcm = _speechlike(3000, 20, 5, channels=2) << 4                      # 24-bit container, 4 wasted bits
        plan = lambda b, c: ("lpc" if c else "fixed", {"order": 4, "porder": 1, "wasted": 4})
        plan.stereo = lambda b: 0
        data, bps, sr, bs = fw.encode_flac(pcm, 48000, 24, 1152, plan), 24, 48000, 1152
    else:
        pcm = _speechlike(1000, 8, 6)
        plan = lambda b, c: ("fixed", {"order": 1, "porder": 0})
        data, bps, sr, bs = fw.encode_flac(pcm, 12345, 8, 300, plan), 8, 12345, 300
    info, got = _decode_to_int(data, tmp_path)
    assert (info.sample_rate, info.channels, info.frames) == (sr, pcm.shape[0], pcm.shape[1])
    shift = (16 - bps) if bps <= 16 else (32 - bps)                          # left-justified output
    assert np.array_equal(got, pcm << shift)
    # the MD5 the ENCODER stored over the original PCM equals the MD5 of what the DECODER produced
    stored = data[data.index(b"fLaC") + 8 + 18: data.index(b"fLaC") + 8 + 34]
    nbytes = (bps + 7) // 8
    md5 = hashlib.md5(b"".join(int(v).to_bytes(nbytes, "little", signed=True) for v in (got >> shift).T.reshape(-1))).digest()
    assert md5 == stored
    assert aio.probe_audio(str(tmp_path / "x.flac")) == (sr, pcm.shape[0], pcm.shape[1])
    # float conversion: left-justified ints scale to [-1, 1)
    x = aio.pcm_to_float(info)
    assert np.allclose(x, pcm / float(1 << (bps - 1)), atol=1e-7)


def test_flac_corruption_is_detected(tmp_path):
    pcm = _speechlike(6000, 16, 9)
    data = bytearray(fw.encode_flac(pcm, 16000, 16, 1024))
    good = bytes(data)
    _decode_to_int(good, tmp_path)
    bad = bytearray(good); bad[len(bad) // 2] ^= 0x10                        # a flipped bit inside a frame: CRC-16 (or the header CRC-8)
    (tmp_path / "bad.flac").write_bytes(bytes(bad))
    with pytest.raises(aio.UnsupportedAudio, match="decode failed"):
        aio.read_audio(str(tmp_path / "bad.flac"))
    (tmp_path / "cut.flac").write_bytes(good[: len(good) * 2 // 3])         # truncated download
    with pytest.raises(aio.UnsupportedAudio):
        aio.read_audio(str(tmp_path / "cut.flac"))
    (tmp_path / "not.flac").write_bytes(b"RIFF" + b"\x00" * 100)
    with pytest.raises(aio.UnsupportedAudio):
        aio.read_audio(str(tmp_path / "not.flac"))
    (tmp_path / "x.mp3").write_bytes(b"\xff\xfb" + b"\x00" * 400)
    with pytest.raises(aio.UnsupportedAudio, match="no decoder"):
        aio.read_audio(str(tmp_path / "x.mp3"))


@pytest.mark.parametrize("sr_in", [8000, 48000, 44100, 24000, 11025])
def test_resampler_specification(sr_in):
    """soxr_hq-class behaviour: unity gain and linear phase up to 0.9 of the lower Nyquist, > 100 dB rejection of
    what would alias, output length ceil(n * ratio) (librosa.resample's length rule)."""
    sr_out = 16000
    n = sr_in // 2 + 37
    t = np.arange(n) / sr_in
    nyq = min(sr_in, sr_out) / 2
    f_pass = 0.9 * nyq
    x = np.sin(2 * np.pi * f_pass * t).astype(np.float32)
    y = aio.resample(x, sr_in, sr_out)
    assert y.dtype == np.float32 and y.shape[0] == -(-n * sr_out // sr_in)
    to = np.arange(y.shape[0]) / sr_out
    mid = slice(y.shape[0] // 4, 3 * y.shape[0] // 4)
    assert np.abs(y[mid] - np.sin(2 * np.pi * f_pass * to)[mid]).max() < 2e-4
    if sr_in > sr_out:                                                        # a tone above the new Nyquist must vanish
        x2 = np.sin(2 * np.pi * (nyq * 1.09) * t).astype(np.float32)
        assert np.abs(aio.resample(x2, sr_in, sr_out)[mid]).max() < 1e-5
    plan = aio.resample_plan(sr_in, sr_out)
    assert plan.taps.dtype == np.float32 and plan.n_out(n) == y.shape[0]
    # the kernel's formula, evaluated in numpy on a short signal, equals scipy's upfirdn-based result
    xs = np.random.default_rng(0).standard_normal(400).astype(np.float32)
    ref = aio.resample(xs, sr_in, sr_out)
    i = np.arange(ref.shape[0])
    tt = (i + plan.pre_remove) * plan.down
    got = np.zeros(ref.shape[0])
    for k_out in range(ref.shape[0]):
        phase, base = tt[k_out] % plan.up, tt[k_out] // plan.up
        j = np.arange(0, (plan.taps.shape[0] - 1 - phase) // plan.up + 1)
        ok = (base - j >= 0) & (base - j < xs.shape[0])
        got[k_out] = np.dot(plan.taps[phase + j[ok] * plan.up].astype(np.float64), xs[base - j[ok]].astype(np.float64))
    assert np.abs(got - ref).max() < 2e-6
    assert aio.resample_plan(16000, 16000) is None
