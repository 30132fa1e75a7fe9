"""GPU (B200): the offline corpus decode — emit_chunks_kernel against emit_chunk_kernel run chunk by chunk, f32_to_pcm_kernel
against the numpy formula, corpus.decode_streams / render_streams against hand-built windows, the detokenize_audio loop,
OutputChunkEmitter and the fp32 oracle, and the codes_to_audio CLI end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.io import wavfile

import realtime_codec_agent_b200 as pkg
from oracle.magicodec_oracle import OracleGenerator
from realtime_codec_agent_b200 import audio_io, audio_to_codes, codes_to_audio, corpus
from realtime_codec_agent_b200._native import McError
from realtime_codec_agent_b200.audio_utils import create_crossfade_ramps
from realtime_codec_agent_b200.codec_chars import codes_to_chars
from realtime_codec_agent_b200.output_chunks import OutputChunkEmitter
from tests.test_codes_to_audio_host import host_f32_to_pcm

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SNR_MIN_DB, WAV_TOL = 38.0, 0.02                # the decode bar of tests/test_gpu_parity.py


@pytest.fixture(scope="module")
def gen():
    return pkg.B200Generator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0), device="cuda", max_positions=1024)


def _snr_db(ref, got):
    ref, got = np.asarray(ref, np.float64), np.asarray(got, np.float64)
    return 10.0 * np.log10((ref ** 2).sum() / max(((ref - got) ** 2).sum(), 1e-30))


def _codes(n, seed, k, device="cuda"):
    return torch.from_numpy(np.random.default_rng(seed).integers(0, k, n)).long().to(device)


class split_k_off:
    def __init__(self, gen):
        self.gen = gen

    def __enter__(self):
        self.gen.set_option("small_m_split_k", 0)

    def __exit__(self, *exc):
        self.gen.set_option("small_m_split_k", 1)


# ----------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("chunk,L,last_len,target", [(1600, 320, 1600, 0.0), (1600, 320, 1600, 0.05), (1600, 1600, 1600, 0.05),
                                                      (1600, 320, 640, 0.05), (1600, 320, 960, 0.0), (640, 64, 320, 0.1)])
def test_emit_chunks_kernel_equals_the_sequential_kernel(gen, chunk, L, last_len, target):
    n = 9
    rng = np.random.default_rng(chunk + L + last_len)
    win = (rng.standard_normal((n, chunk + L)) * 0.2).astype(np.float32)
    win[3] *= 1e-3                                                          # a chunk below the silence threshold
    _, fade_np, _ = create_crossfade_ramps(16000, L / 16000)
    fade_in = torch.from_numpy(fade_np).cuda()
    dev = torch.from_numpy(win).cuda()
    got = gen.render_chunks(dev, chunk, fade_in, last_len=last_len, target_rms=target, silence_rms_threshold=0.003).cpu().numpy()
    prev_tail = torch.zeros(L, device="cuda")
    hist = []
    for i in range(n):
        have = (L if i else 0) + (last_len if i == n - 1 else chunk)
        out = gen.op_emit_chunk(dev[i, :have].contiguous(), chunk, L, i > 0, target, 0.003, fade_in, prev_tail).cpu().numpy()
        if i:
            hist[-1] = np.concatenate((hist[-1][:chunk - L], out[chunk:chunk + L]))
        hist.append(out[chunk + L:])
    want = np.concatenate(hist)[: (n - 1) * chunk + last_len]
    assert got.shape == want.shape and np.array_equal(got, want)
    one = gen.render_chunks(dev[:1], chunk, fade_in, last_len=last_len, target_rms=target).cpu().numpy()
    assert one.shape == (last_len,)
    with pytest.raises(McError):
        gen.render_chunks(dev, chunk, fade_in, last_len=chunk + 1)


def test_f32_to_pcm_into_pinned_memory_equals_the_formula(gen):
    vals = np.array([1.0, -1.0, 0.5 / 32768, 1.5 / 32768, -2.5 / 32768, 1.0001, -1.2, 3e38, -np.inf, np.nan, 0.0, -0.0],
                     dtype=np.float32)
    x = np.concatenate([vals, np.random.default_rng(0).standard_normal(4001).astype(np.float32)])
    stereo = np.stack([x, -x[::-1]])
    for wav in (x[None], stereo):
        dev = torch.from_numpy(np.ascontiguousarray(wav)).cuda()
        for fmt, dtype in ((audio_io.PCM_S16, torch.int16), (audio_io.PCM_F32, torch.float32)):
            pinned = torch.empty(wav.size, dtype=dtype).pin_memory()
            got = gen.f32_to_pcm(dev, fmt, out=pinned)
            torch.cuda.current_stream().synchronize()
            want = host_f32_to_pcm(wav, fmt).T
            assert np.array_equal(got.numpy(), want, equal_nan=fmt == audio_io.PCM_F32)
    planar_view = torch.from_numpy(stereo).cuda()[:, 10:]                   # row stride > frames
    assert np.array_equal(gen.f32_to_pcm(planar_view, audio_io.PCM_S16).cpu().numpy(), host_f32_to_pcm(stereo[:, 10:], 1).T)


# ------------------------------------------------------------------------------------- chunked decode
def _hand_built(gen, s, cf, ctx, preroll=0):
    out, hop, n = [], gen.hop, int(s.numel())
    for i in range(0, n, cf):
        end = min(i + cf, n)
        lo = max(0, end - max(end - i, ctx))
        out.append(gen.decode(s[None, lo:end], keep_last_samples=(end - i) * hop + preroll)[0])
    return out


@pytest.mark.parametrize("bs,fuse", [(16, 1), (7, 3), (256, 1)])
def test_decode_streams_equals_hand_built_windows(gen, bs, fuse):
    K = gen.codebook_size
    streams = [_codes(3000 + 3, 1, K), _codes(250, 2, K), _codes(42, 3, K), _codes(5 * 19, 4, K), _codes(2, 5, K)]
    fast = corpus.decode_streams(gen, streams, 0.1, 2.0, batch_size=bs, fuse_batches=fuse)
    slow = corpus.decode_streams(gen, streams, 0.1, 2.0, batch_size=bs, causal_warmup=False)
    for s, a, b in zip(streams, fast, slow):
        assert torch.equal(a, b)
        assert torch.equal(a, torch.cat(_hand_built(gen, s, 5, 100)))
        assert a.numel() == s.numel() * gen.hop


def test_look_ahead_spec_skips_the_causal_warmup_shortcut_in_decode():
    spec = pkg.TINY_SPEC.replace(window_left=24, window_right=8)
    g = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda", max_positions=256)
    streams = [_codes(150, 10 + i, g.codebook_size) for i in range(2)]
    fast = corpus.decode_streams(g, streams, 0.1, 2.0, batch_size=16)
    slow = corpus.decode_streams(g, streams, 0.1, 2.0, batch_size=16, causal_warmup=False)
    assert all(torch.equal(a, b) for a, b in zip(fast, slow))
    assert torch.equal(fast[0], torch.cat(_hand_built(g, streams[0], 5, 100)))
    whole = g.decode(streams[0][None, :100])[0]                             # the prefix trick WOULD have been wrong here
    assert not torch.equal(whole[:95 * 320], fast[0][:95 * 320])


@pytest.mark.parametrize("C", [1, 2])
def test_chunked_detokenize_equals_the_loop(gen, C):
    tok = pkg.AudioTokenizer(codec_model=gen, num_channels=C, device="cuda")
    codes = np.stack([_codes(5 * 31 + 3, 20 + c, gen.codebook_size, "cpu").numpy() for c in range(C)])
    text = codes_to_chars(np.ascontiguousarray(codes.T).reshape(1, -1), gen.codebook_size, unicode_offset=tok.unicode_offset)
    sr, fast = tok.chunked_detokenize_audio(text, 0.1)
    assert sr == 16000 and fast.shape == ((codes.shape[1] * 320,) if C == 1 else (C, codes.shape[1] * 320))
    ctx_fast = tok.detokenize_context
    step = 5 * C

    def loop():
        tok.reset_context()
        return np.concatenate([tok.detokenize_audio(text[s:s + step])[0][1] for s in range(0, len(text), step)], axis=-1)

    with split_k_off(gen):
        assert np.array_equal(loop(), fast) and tok.detokenize_context == ctx_fast
        (_, a), _, _ = tok.detokenize_audio(text[:step])                     # the session context is the loop's, too
        tok.reset_context()
        tok.chunked_detokenize_audio(text, 0.1)
        (_, b), _, _ = tok.detokenize_audio(text[:step])
        assert np.array_equal(a, b)
    snr = _snr_db(loop(), fast)
    print(f"[decode corpus] C={C} chunked_detokenize batched vs session loop (split-K few-rows kernels): {snr:.1f} dB")
    assert snr >= SNR_MIN_DB


def test_render_streams_equals_the_native_emitter(gen):
    codes = _codes(5 * 40, 30, gen.codebook_size)
    tok = pkg.AudioTokenizer(codec_model=gen, device="cuda")
    text = codes_to_chars(codes.cpu().numpy()[None], gen.codebook_size, unicode_offset=tok.unicode_offset)
    for target in (0.0, 0.05):
        with split_k_off(gen):
            got = corpus.render_streams(gen, [codes], 0.1, 2.0, 0.02, target, 0.003, batch_size=16)[0].cpu().numpy()
            tok.reset_context()
            em = OutputChunkEmitter(tok, 0.1, 0.02, target, 0.003)
            for s in range(0, len(text), 5):
                em.emit(text[s:s + 5])
        assert np.array_equal(got, np.concatenate(em.audio_history_ch1))


@pytest.mark.parametrize("name", ["tiny", "mid"])
def test_chunked_decode_and_render_meet_the_oracle_bar(name):
    spec = {"tiny": pkg.TINY_SPEC, "mid": pkg.MID_SPEC}[name]
    w = pkg.init_random_weights(spec, seed=0)
    g = pkg.B200Generator(spec, w, device="cuda", max_positions=1024)
    oracle = OracleGenerator(spec, w)
    codes = _codes(5 * 26 + 2, 40, spec.codebook_size)
    host = pkg.AudioTokenizer(codec_model=oracle, device="cpu")
    text = codes_to_chars(codes.cpu().numpy()[None], spec.codebook_size, unicode_offset=host.unicode_offset)
    _, ref = host.chunked_detokenize_audio(text, 0.1)
    got = corpus.decode_streams(g, [codes], 0.1, 2.0)[0].cpu().numpy()
    host.reset_context()
    em = OutputChunkEmitter(host, 0.1, 0.02, 0.05, 0.003)
    for s in range(0, len(text), 5):
        em.emit(text[s:s + 5])
    ref_r = np.concatenate(em.audio_history_ch1)[: codes.numel() * 320]
    got_r = corpus.render_streams(g, [codes], 0.1, 2.0, 0.02, 0.05, 0.003)[0].cpu().numpy()
    for what, r, x in (("chunked", ref, got), ("render", ref_r, got_r)):
        snr, rel = _snr_db(r, x), np.abs(r - x).max() / np.abs(r).max()
        print(f"[decode corpus {name}] {what} vs fp32 oracle: snr={snr:.1f} dB max_rel={rel:.4f}")
        assert snr >= SNR_MIN_DB and rel <= WAV_TOL


# ------------------------------------------------------------------------------------------------ CLI
def _encode_corpus(tmp_path, stereo):
    raw = tmp_path / "raw"
    raw.mkdir(exist_ok=True)
    a = pkg.synth_audio(16000 * 3 + 800, file_id=51).numpy()
    b = pkg.synth_audio(16000 * 2, file_id=52, channel=1).numpy()
    wavfile.write(raw / "x.wav", 16000, (np.stack([a[:len(b)], b], axis=1) * 32767).astype(np.int16))
    wavfile.write(raw / "y.wav", 16000, (a * 32767).astype(np.int16))
    spec = pkg.TINY_SPEC
    ckpt = tmp_path / "tiny.pt"
    pkg.save_checkpoint(str(ckpt), spec, pkg.init_random_weights(spec, seed=0))
    audio_to_codes.main(["--audio_path", str(raw), "--codes_path", str(tmp_path / "codes"), "--batch_size", "16"]
                        + (["--stereo"] if stereo else []))
    return tmp_path / "codes" / "MagiCodec-50Hz-Base" / "0.1s_2.0s" / ("stereo" if stereo else "mono"), ckpt


@pytest.mark.parametrize("stereo", [False, True])
def test_cli_on_the_engine(tmp_path, monkeypatch, gen, stereo):
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("MAGICODEC_B200_CHECKPOINT", str(tmp_path / "tiny.pt"))
    src, _ = _encode_corpus(tmp_path, stereo)
    C = 2 if stereo else 1
    for mode in codes_to_audio.MODES:
        dst = tmp_path / f"audio_{mode}"
        codes_to_audio.main(["--codes_path", str(src), "--audio_path", str(dst), "--mode", mode])
        man = json.load(open(dst / "manifest.json"))
        assert json.load(open(dst / "errors.json")) == [] and [e["file"] for e in man] == ["x.wav", "y.wav"]
        for e in man:
            rel = e["file"][:-4]
            streams = [torch.from_numpy(np.load(src / f"{rel}_c{c}.npy")[0].astype(np.int64)).cuda() for c in range(C)]
            if mode == "chunked":
                want = torch.stack(corpus.decode_streams(gen, streams, 0.1, 2.0))
            elif mode == "render":
                want = torch.stack(corpus.render_streams(gen, streams, 0.1, 2.0))
            else:
                want = gen.decode(torch.stack(streams))
            sr, got = wavfile.read(dst / e["file"])
            assert sr == 16000 and np.array_equal(got.reshape(-1, C), host_f32_to_pcm(want.cpu().numpy(), 1).T)
    # resume: every output is complete, so the engine launches nothing
    g2 = pkg.B200Generator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0), device="cuda")
    man1, _ = codes_to_audio.decode_corpus(g2, str(src), str(tmp_path / "audio_render"), "render")
    assert g2.launch_count == 0 and len(man1) == 2


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (one process per GPU)")
def test_cli_under_torchrun_on_two_gpus(tmp_path, monkeypatch):
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("MAGICODEC_B200_CHECKPOINT", str(tmp_path / "tiny.pt"))
    src, ckpt = _encode_corpus(tmp_path, False)
    env = dict(os.environ, MAGICODEC_B200_CHECKPOINT=str(ckpt), PYTHONPATH=ROOT)

    def run(nproc, dst):
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
               "--master-port", "29613", "-m", "rca_b200_loader", "codes_to_audio", "--codes_path", str(src), "--audio_path", str(dst)]
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
        return json.load(open(dst / "manifest.json"))

    man2, man1 = run(2, tmp_path / "a2"), run(1, tmp_path / "a1")
    assert {e["rank"] for e in man2} == {0, 1}
    assert [(e["file"], e["samples"], e["crc32"]) for e in man1] == [(e["file"], e["samples"], e["crc32"]) for e in man2]
