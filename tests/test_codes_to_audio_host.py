"""CPU: the offline corpus decode's host logic — window planning against a replay of the detokenize_audio bookkeeping,
the render chain against OutputChunkEmitter, write_wav, and the codes_to_audio CLI (layout, channel grouping,
codec_info checks, per-file errors, resume, rank partition) around the fp32 oracle."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch
from scipy.io import wavfile

import realtime_codec_agent_b200 as pkg
from oracle.magicodec_oracle import OracleGenerator
from realtime_codec_agent_b200 import audio_io, codes_to_audio, corpus
from realtime_codec_agent_b200.audio_utils import create_crossfade_ramps, normalize_audio_rms, pad_or_trim, smooth_join
from realtime_codec_agent_b200.codec_chars import codes_to_chars
from realtime_codec_agent_b200.output_chunks import OutputChunkEmitter
from tests.fake_gen import HostIngest, OracleBackedGen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def host_render(windows, chunk, fade_in, last_len, target_rms, silence_thr):
    """numpy mirror of emit_chunks_kernel: the OutputChunkEmitter chain replayed on the decoded window rows."""
    L = fade_in.shape[0]
    hist = []
    n = windows.shape[0]
    for i in range(n):
        valid = (L if i else 0) + (last_len if i == n - 1 else chunk)
        x = pad_or_trim(windows[i, :valid], chunk + (L if i else 0))
        if target_rms > 0:
            x = normalize_audio_rms(x, target_rms=target_rms, silence_rms_threshold=silence_thr)
        if hist:
            joined = smooth_join(hist[-1], x, L, fade_in, fade_in[::-1])
            hist[-1] = joined[:chunk]
            hist.append(joined[chunk:])
        else:
            hist.append(x)
    return np.concatenate(hist)[: (n - 1) * chunk + last_len]


def host_f32_to_pcm(x, fmt):
    x = np.asarray(x, dtype=np.float32)
    if fmt == audio_io.PCM_F32:
        return x.copy()
    with np.errstate(invalid="ignore", over="ignore"):
        v = np.clip(np.rint(x * np.float32(32768)), -32768, 32767)
    return np.where(np.isnan(v), 0, v).astype(np.int16)


class DecodeGen(OracleBackedGen):
    """OracleBackedGen plus the decode-side entry points: decode (one oracle call per window, exactly as the host
    AudioTokenizer decodes) and host mirrors of mc_render_chunks / mc_op_f32_to_pcm."""

    def __init__(self, oracle):
        super().__init__(oracle)
        self.decode_calls = []

    def decode(self, codes, keep_last_samples=0):
        codes = codes.reshape(1, -1) if codes.dim() == 1 else codes
        self.decode_calls.append(tuple(codes.shape))
        q = self.oracle.quantizer
        with torch.no_grad():
            table = q.codebook_proj(q.codebook.weight)
            rows = [self.oracle.decoder(torch.nn.functional.embedding(r[None].long(), table)).float()[0, 0] for r in codes]
        wav = torch.stack(rows)
        total = wav.shape[-1]
        keep = total if keep_last_samples <= 0 or keep_last_samples > total else keep_last_samples
        return wav[:, total - keep:]

    def render_chunks(self, windows, chunk, fade_in, last_len=None, target_rms=0.0, silence_rms_threshold=0.003):
        last_len = chunk if last_len is None else last_len
        return torch.from_numpy(host_render(windows.numpy(), chunk, fade_in.numpy(), last_len, target_rms, silence_rms_threshold))

    def f32_to_pcm(self, wav, fmt=1, out=None):
        wav = wav.reshape(1, -1) if wav.dim() == 1 else wav
        pcm = torch.from_numpy(np.ascontiguousarray(host_f32_to_pcm(wav.numpy(), fmt).T))
        if out is not None:
            out.view(-1)[: pcm.numel()] = pcm.reshape(-1)
        return pcm


class DecodeIngest(HostIngest):
    def upload_codes(self, host_tensor, nbytes):
        return host_tensor[:nbytes].clone()

    def codes_on_device(self, staged, channels, frames):
        return staged.view(torch.int64).view(channels, frames)

    def pcm_to_host(self, wav, fmt):
        return self.gen.f32_to_pcm(wav, fmt).numpy(), (lambda: None)


@pytest.fixture(scope="module")
def oracle():
    return OracleGenerator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0))


def _codes(n, seed, k):
    return torch.from_numpy(np.random.default_rng(seed).integers(0, k, n)).long()


def replay_detokenize_windows(n_frames, cf, context_frames, preroll, hop):
    """The context bookkeeping of a detokenize_audio loop from an empty context (audio_tokenizer.py:105-113), on strings."""
    text = "".join(chr(0x100 + i) for i in range(n_frames))
    ctx, out = "", []
    for i, s in enumerate(range(0, n_frames, cf)):
        piece = text[s:s + cf]
        ctx = (ctx + piece)[-max(len(piece), context_frames):]
        start = ord(ctx[0]) - 0x100
        keep = min(len(piece) * hop + preroll, len(ctx) * hop)
        out.append((start, len(ctx), keep, i))
    return out


@pytest.mark.parametrize("n_frames,cf,ctx,pre", [(3000, 5, 100, 0), (117, 5, 100, 320), (3, 5, 100, 0), (250, 7, 20, 64),
                                                  (40, 10, 4, 0)])
def test_plan_decode_stream_matches_the_detokenize_bookkeeping(n_frames, cf, ctx, pre):
    irr, steady = corpus.plan_decode_stream(n_frames, cf, ctx, pre, 320)
    got = [(w.start_frame, w.frames, w.keep_samples, w.chunk) for w in irr]
    if steady is not None:
        first, count = steady
        got += [(first.start_frame + j * cf, first.frames, first.keep_samples, first.chunk + j) for j in range(count)]
    assert sorted(got, key=lambda t: t[3]) == replay_detokenize_windows(n_frames, cf, ctx, pre, 320)
    if (n_frames, cf, ctx) == (3000, 5, 100):
        assert len(irr) == 19 and steady[1] == 581 and steady[0].frames == 100


@pytest.mark.parametrize("n_frames", [5 * 23 + 3, 5 * 4, 2])
def test_decode_streams_equals_the_detokenize_loop(oracle, n_frames):
    gen = DecodeGen(oracle)
    codes = _codes(n_frames, n_frames, oracle.codebook_size)
    got = corpus.decode_streams(gen, [codes], 0.1, 0.4, batch_size=4, causal_warmup=False)[0].numpy()
    tok = pkg.AudioTokenizer(codec_model=oracle, context_secs=0.4, device="cpu")
    text = codes_to_chars(codes.numpy()[None], oracle.codebook_size, unicode_offset=tok.unicode_offset)
    sr, ref = tok.chunked_detokenize_audio(text, 0.1)                        # host model: the loop itself
    assert sr == 16000 and got.shape == (n_frames * 320,) and np.array_equal(got, ref)
    with pytest.raises(ValueError):
        corpus.decode_streams(gen, [codes], 0.07)                            # 3.5 frames per chunk


@pytest.mark.parametrize("target_rms,n_frames", [(0.0, 5 * 12), (0.05, 5 * 12 + 2), (0.05, 3)])
def test_render_streams_equals_output_chunk_emitter(oracle, target_rms, n_frames):
    gen = DecodeGen(oracle)
    codes = _codes(n_frames, 7 + n_frames, oracle.codebook_size)
    got = corpus.render_streams(gen, [codes], 0.1, 0.4, 0.02, target_rms, 0.003, batch_size=3, causal_warmup=False)[0].numpy()
    tok = pkg.AudioTokenizer(codec_model=oracle, context_secs=0.4, device="cpu")
    em = OutputChunkEmitter(tok, 0.1, 0.02, target_rms, 0.003)
    text = codes_to_chars(codes.numpy()[None], oracle.codebook_size, unicode_offset=tok.unicode_offset)
    for s in range(0, len(text), 5):
        em.emit(text[s:s + 5])
    ref = np.concatenate(em.audio_history_ch1)[: n_frames * 320]
    assert got.shape == (n_frames * 320,) and np.array_equal(got, ref)


def test_write_wav_round_trips(tmp_path):
    rng = np.random.default_rng(0)
    for dtype, fmt in ((np.int16, audio_io.PCM_S16), (np.float32, audio_io.PCM_F32)):
        for C in (1, 2):
            x = (rng.standard_normal((1001, C)) * (3000 if dtype == np.int16 else 0.3)).astype(dtype)
            p = tmp_path / f"x_{C}_{fmt}.wav"
            with open(p, "wb") as f:
                crc = audio_io.write_wav(f, x, 16000)
            sr, back = wavfile.read(p)
            assert sr == 16000 and np.array_equal(back.reshape(1001, C), x)
            pcm = audio_io.read_audio(str(p))
            assert (pcm.sample_rate, pcm.channels, pcm.frames, pcm.fmt) == (16000, C, 1001, fmt)
            assert np.array_equal(pcm.payload.view(dtype).reshape(1001, C), x)
            assert crc == zlib.crc32(x.tobytes()) & 0xFFFFFFFF
            assert audio_io.wav_info(str(p)) == (16000, C, fmt, 1001)
            p.write_bytes(p.read_bytes()[:-10])
            assert audio_io.wav_info(str(p)) is None                         # truncated: not complete


def test_pcm16_formula_inverts_the_int16_input_scaling():
    grid = np.arange(-32768, 32768, dtype=np.int16)
    assert np.array_equal(host_f32_to_pcm(grid.astype(np.float32) / 32768.0, audio_io.PCM_S16), grid)
    assert host_f32_to_pcm(np.array([1.0, -1.0, 2.0, -3.0, np.nan], np.float32), audio_io.PCM_S16).tolist() == \
        [32767, -32768, 32767, -32768, 0]


def _make_corpus(root, oracle, stereo, files):
    sub = "stereo" if stereo else "mono"
    out = root / "codes" / sub
    out.mkdir(parents=True)
    info = {"codec_model": "x", "framerate": 50.0, "num_codebooks": 1, "codebook_size": oracle.codebook_size,
            "sampling_rate": 16000, "chunk_size_secs": 0.1, "context_secs": 0.4, "stereo": stereo}
    (out / "codec_info.json").write_text(json.dumps(info))
    for rel, arrs in files.items():
        (out / rel).parent.mkdir(parents=True, exist_ok=True)
        for c, a in enumerate(arrs):
            np.save(out / f"{rel}_c{c}.npy", a)
    return out


@pytest.mark.parametrize("mode", ["chunked", "render", "one_shot"])
def test_cli_layout_grouping_errors_and_resume(tmp_path, oracle, mode):
    K = oracle.codebook_size
    a, b = _codes(33, 1, K).numpy(), _codes(33, 2, K).numpy()
    files = {"A/one": [a[None].astype(np.int32), b.astype(np.int64)], "two": [b[None, :20].astype(np.int32)] * 2,
             "bad_range": [a[None], np.full((1, 33), K, np.int32)], "unequal": [a[None], b[None, :30]],
             "missing": [a[None]]}
    src = _make_corpus(tmp_path, oracle, True, files)
    np.save(src / "missing_c2.npy", a[None])                              # channels 0 and 2: not 0..1
    (src / "corrupt_c0.npy").write_bytes(b"\x93NUMPY garbage")
    np.save(src / "corrupt_c1.npy", a[None])
    gen = DecodeGen(oracle)
    dst = tmp_path / "audio"
    man, errs = codes_to_audio.decode_corpus(gen, str(src), str(dst), mode, batch_size=4, ingest=DecodeIngest(gen))
    assert sorted(e["file"].split(":")[0] for e in errs) == ["bad_range", "corrupt", "missing", "unequal"]
    assert [e["file"] for e in man] == ["A/one.wav", "two.wav"]
    assert sorted(os.path.relpath(os.path.join(d, f), dst) for d, _, fs in os.walk(dst) for f in fs) == ["A/one.wav", "two.wav"]
    sr, got = wavfile.read(dst / "A/one.wav")
    assert sr == 16000 and got.dtype == np.int16 and got.shape == (33 * 320, 2)
    streams = [torch.from_numpy(a), torch.from_numpy(b)]
    if mode == "chunked":
        want = torch.stack(corpus.decode_streams(gen, streams, 0.1, 0.4, batch_size=4))
    elif mode == "render":
        want = torch.stack(corpus.render_streams(gen, streams, 0.1, 0.4, batch_size=4))
    else:
        want = gen.decode(torch.stack(streams))
    assert np.array_equal(got, host_f32_to_pcm(want.numpy(), audio_io.PCM_S16).T)
    assert man[0]["crc32"] == zlib.crc32(got.tobytes()) & 0xFFFFFFFF and man[0]["samples"] == 33 * 320
    # resume: no decode, same manifest; a truncated file is decoded again
    calls = len(gen.decode_calls)
    man2, _ = codes_to_audio.decode_corpus(gen, str(src), str(dst), mode, ingest=DecodeIngest(gen))
    assert len(gen.decode_calls) == calls and man2 == man
    victim = dst / "two.wav"
    victim.write_bytes(victim.read_bytes()[:100])
    man3, _ = codes_to_audio.decode_corpus(gen, str(src), str(dst), mode, ingest=DecodeIngest(gen))
    assert len(gen.decode_calls) > calls and man3 == man


def test_cli_mono_float_output(tmp_path, oracle):
    a = _codes(12, 3, oracle.codebook_size).numpy()
    src = _make_corpus(tmp_path, oracle, False, {"m": [a.astype(np.int16)]})
    gen = DecodeGen(oracle)
    man, errs = codes_to_audio.decode_corpus(gen, str(src), str(tmp_path / "o"), fmt="float", ingest=DecodeIngest(gen))
    assert errs == [] and man[0]["channels"] == 1
    sr, got = wavfile.read(tmp_path / "o" / "m.wav")
    want = corpus.decode_streams(gen, [torch.from_numpy(a.astype(np.int64))], 0.1, 0.4)[0].numpy()
    assert got.dtype == np.float32 and np.array_equal(got, want)


@pytest.mark.parametrize("key,value", [(None, None), ("codebook_size", 17), ("sampling_rate", 24000), ("framerate", 75.0)])
def test_codec_info_mismatch_refuses_to_start(tmp_path, oracle, key, value):
    src = _make_corpus(tmp_path, oracle, False, {"m": [_codes(12, 3, oracle.codebook_size).numpy()]})
    if key is None:
        os.remove(src / "codec_info.json")
    else:
        info = json.loads((src / "codec_info.json").read_text())
        info[key] = value
        (src / "codec_info.json").write_text(json.dumps(info))
    gen = DecodeGen(oracle)
    with pytest.raises(codes_to_audio.RefusedToStart):
        codes_to_audio.decode_corpus(gen, str(src), str(tmp_path / "o"), ingest=DecodeIngest(gen))
    assert not (tmp_path / "o").exists() and gen.decode_calls == []


def test_two_ranks_partition_the_files(tmp_path, oracle):
    K = oracle.codebook_size
    files = {f"f{i}": [_codes(10 + 7 * i, i, K).numpy()] for i in range(5)}
    src = _make_corpus(tmp_path, oracle, False, files)
    seen = []
    for rank in range(2):
        gen = DecodeGen(oracle)
        man, errs = codes_to_audio.decode_corpus(gen, str(src), str(tmp_path / "o"), rank=rank, world_size=2,
                                                 ingest=DecodeIngest(gen))
        assert errs == [] and all(e["rank"] == rank for e in man) and man
        seen += [e["file"] for e in man]
    assert sorted(seen) == [f"f{i}.wav" for i in range(5)]


def test_cli_help_resolves():
    p = subprocess.run([sys.executable, "-m", "rca_b200_loader", "codes_to_audio", "--help"], cwd=ROOT, capture_output=True,
                       text=True, timeout=120)
    assert p.returncode == 0 and "--mode" in p.stdout and "one_shot" in p.stdout
