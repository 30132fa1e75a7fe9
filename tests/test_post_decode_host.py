"""CPU: rows f3 / f4 (SURVEY §8) — the post-decode output chain and the duplex aligner.

* the oracle restatement (oracle/post_decode_oracle.py) reproduces the golden vectors the reference's OWN
  utils/audio_utils.py and ExternalTTSDuplexAligner produced (tests/golden/make_golden_post.py);
* the product's host utilities and OutputChunkEmitter / ExternalTTSDuplexAligner (non-native branch)
  reproduce them too, and agree with the stored outputs of the reference modules (tests/golden/golden_host_calls.npz)
  and, wherever the reference is installed, with those modules imported unmodified.
"""
import os

import numpy as np
import pytest
import torch

import realtime_codec_agent_b200 as pkg
from oracle import post_decode_oracle as po
from tests.golden_calls import assert_identical, assert_matches_golden

SR, CHUNK, L = 16000, 1600, 320


@pytest.fixture(scope="module")
def g(golden_dir):
    return np.load(os.path.join(golden_dir, "golden_post.npz"))


class ReplayTokenizer:
    sampling_rate, num_channels = SR, 1

    def __init__(self, flat, lengths):
        ends = np.cumsum(lengths)
        self.decoded = [flat[e - n:e] for e, n in zip(ends, lengths)]
        self.i = 0

    def detokenize_audio(self, s, preroll_samples=0):
        wav = self.decoded[self.i]
        self.i += 1
        return (SR, wav), "", wav.shape[-1] - CHUNK


UTIL_SETS = {"oracle": po.RESTATED_UTILS,
             "product": {"create_crossfade_ramps": pkg.create_crossfade_ramps, "smooth_join": pkg.smooth_join,
                         "pad_or_trim": pkg.pad_or_trim, "normalize_audio_rms": pkg.normalize_audio_rms}}


@pytest.mark.parametrize("which", ["oracle", "product"])
def test_audio_utils_match_reference_golden(g, which):
    u = UTIL_SETS[which]
    n, fi, fo = u["create_crossfade_ramps"](SR, 0.02)
    assert n == int(g["ramp_L"]) == L
    assert np.array_equal(fi, g["fade_in"]) and np.array_equal(fo, g["fade_out"])
    a, b = g["join_a"], g["join_b"]
    assert np.array_equal(u["smooth_join"](a, b, n, fi, fo), g["join_out"])
    assert np.array_equal(u["smooth_join"](a[:0], b, n, fi, fo), b)
    assert np.array_equal(u["smooth_join"](a, b, 0, fi[:0], fo[:0]), np.concatenate((a, b)))
    assert np.array_equal(u["pad_or_trim"](a[:1000], 1600), g["pad_right"])
    assert np.array_equal(u["pad_or_trim"](a[:1000], 1600, pad_side="left"), g["pad_left"])
    assert np.array_equal(u["pad_or_trim"](b, 1600), g["trim"])
    assert u["pad_or_trim"](a, 1600) is a
    with pytest.raises(ValueError):
        u["pad_or_trim"](np.zeros((2, 10), np.float32), 5)
    assert np.array_equal(u["normalize_audio_rms"](b, target_rms=0.05), g["norm_loud"])
    assert np.array_equal(u["normalize_audio_rms"](b * 1e-3, target_rms=0.05), g["norm_silent"])


@pytest.mark.parametrize("tag,target", [("plain", 0.0), ("rms", 0.05)])
def test_output_chain_matches_reference_golden(g, tag, target):
    chain = po.OracleOutputChain(ReplayTokenizer(g["chain_decoded"], g["chain_lengths"]), 0.1, 0.02, target)
    emitter = pkg.OutputChunkEmitter(ReplayTokenizer(g["chain_decoded"], g["chain_lengths"]), 0.1, 0.02, target)
    for want in g[f"chain_emitted_{tag}"]:
        assert np.array_equal(chain.step(""), want)
        assert np.array_equal(emitter.emit(""), want)
    assert np.array_equal(np.concatenate(chain.history), g[f"chain_history_{tag}"])
    assert np.array_equal(np.concatenate(emitter.audio_history_ch1), g[f"chain_history_{tag}"])
    emitter.reset()
    assert emitter.audio_history_ch1 == []


def test_emitter_rejects_what_the_reference_cannot_do():
    tok = ReplayTokenizer(np.zeros(10, np.float32), [10])
    with pytest.raises(ValueError):
        pkg.OutputChunkEmitter(tok, 0.1, 0.0)           # L = 0: the reference's [:-L] slices are empty
    with pytest.raises(ValueError):
        pkg.OutputChunkEmitter(tok, 0.01, 0.02)         # fade > chunk (realtime_agent_config.py:58)
    tok.num_channels = 2
    with pytest.raises(ValueError):
        pkg.OutputChunkEmitter(tok, 0.1, 0.02)


class AlignerStubTokenizer:
    _native = False

    def __init__(self, table, silence_codes):
        self.table, self.silence = table, silence_codes

    def get_codec_embeddings(self):
        return self.table

    def _encode_silence(self, secs):
        assert secs == 10.0
        return self.silence[None, None]


def test_interrupt_score_matches_reference_golden(g):
    table, sil = torch.from_numpy(g["ali_table"]), torch.from_numpy(g["ali_silence_codes"])
    emb = po.oracle_silence_embedding(table, sil)
    assert np.array_equal(emb.numpy(), g["ali_silence_embedding"])
    ours = pkg.ExternalTTSDuplexAligner(AlignerStubTokenizer(table, sil), codec_vocab_start=128256)
    assert np.array_equal(ours.silence_embedding.numpy(), g["ali_silence_embedding"])
    for t, d, want in zip(g["ali_tts"], g["ali_duplex"], g["ali_scores"]):
        assert po.oracle_interrupt_score(table, emb, 128256, t.tolist(), d.tolist()) == want
        assert ours.interrupt_score(t.tolist(), d.tolist()) == want


def test_aligner_reads_vocab_start_from_a_config_dir(g, tmp_path):
    import json
    (tmp_path / "config.json").write_text(json.dumps({"model_type": "llama", "codec_vocab_start": 777}))
    table, sil = torch.from_numpy(g["ali_table"]), torch.from_numpy(g["ali_silence_codes"])
    al = pkg.ExternalTTSDuplexAligner(AlignerStubTokenizer(table, sil), str(tmp_path))
    assert al.codec_vocab_start == 777


def util_calls(u):
    """Ramps, joins and RMS normalisation over seeded inputs for three fade lengths -> {name: array}."""
    rng = np.random.default_rng(5)
    out = {}
    for L_secs in (0.02, 0.005, 0.1):
        n, fi, fo = u["create_crossfade_ramps"](SR, L_secs)
        a = rng.standard_normal(CHUNK).astype(np.float32)
        b = rng.standard_normal(CHUNK + n).astype(np.float32)
        out.update({f"{L_secs}_n": np.int64(n), f"{L_secs}_fade_in": fi, f"{L_secs}_fade_out": np.ascontiguousarray(fo),
                    f"{L_secs}_join": u["smooth_join"](a, b, n, fi, fo)})
        for tr in (0.05, 0.2):
            out[f"{L_secs}_norm_{tr}"] = u["normalize_audio_rms"](b, target_rms=tr)
    return out


def chain_calls(step, history, s):
    """The output chain fed 0.1 s (5-char) pieces of ``s`` -> {name: array}."""
    out = {f"{i}_emitted": np.array(step(s[i:i + 5])) for i in range(0, len(s), 5)}      # a copy: buffers may be reused
    out["history"] = np.concatenate(history())
    return out


def oracle_model_tokenizer_and_codes():
    from oracle.magicodec_oracle import OracleGenerator
    model = OracleGenerator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0))
    our_tok = pkg.AudioTokenizer(codec_model=model, device="cpu")
    s = our_tok.tokenize_audio(pkg.synth_audio(16000, file_id=2).numpy())
    our_tok.reset_context()
    return model, our_tok, s


def test_live_against_the_unmodified_reference_modules(golden_dir):
    """The utilities and the chain over a real (oracle-model) tokenizer, against tests/golden/golden_host_calls.npz and,
    wherever the reference is installed, against the reference's own modules bit for bit."""
    golden = np.load(os.path.join(golden_dir, "golden_host_calls.npz"))
    utils = {which: util_calls(u) for which, u in UTIL_SETS.items()}
    for got in utils.values():
        assert_matches_golden(got, golden, "post_utils", sample=False)
    model, our_tok, s = oracle_model_tokenizer_and_codes()
    emitter = pkg.OutputChunkEmitter(our_tok, 0.1, 0.02, 0.05)
    ours = chain_calls(emitter.emit, lambda: emitter.audio_history_ch1, s)
    assert_matches_golden(ours, golden, "post_chain")
    if po.reference_available():
        from oracle.reference_wrapper import load_reference_audio_tokenizer
        au = po.load_reference_module("utils.audio_utils")
        ref_utils = {k: getattr(au, k) for k in UTIL_SETS["oracle"]}
        for got in utils.values():
            assert_identical(got, util_calls(ref_utils))
        chain = po.OracleOutputChain(load_reference_audio_tokenizer()(codec_model=model, device="cpu"), 0.1, 0.02, 0.05,
                                     utils=ref_utils)
        assert_identical(ours, chain_calls(chain.step, lambda: chain.history, s))
