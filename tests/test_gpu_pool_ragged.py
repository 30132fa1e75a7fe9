"""GPU (B200): ragged session-pool batches (mc_pool_push_*_ragged, SessionBatcher(ragged=True)).

Sessions in their warm-up share one launch with sessions in steady state: every window starts at row 0 of the batch and
reads zeros past its own end.  With the batch-invariant kernels (small_m_split_k = 0) every session must get exactly
what its own AudioTokenizer + OutputChunkEmitter gives, with one engine call per kind and tick."""
import numpy as np
import pytest

import realtime_codec_agent_b200 as pkg
from realtime_codec_agent_b200._native import McError
from realtime_codec_agent_b200.audio_utils import create_crossfade_ramps
from realtime_codec_agent_b200.codec_chars import UNICODE_OFFSET_LARGE, codes_to_chars
from realtime_codec_agent_b200.session_batcher import SessionBatcher, SessionPool, ThreadedSessionBatcher

pytestmark = pytest.mark.gpu
SR, CHUNK = 16000, 1600
KINDS = ("push_audio", "push_codes", "push_codes_emit", "push_audio_ragged", "push_codes_ragged", "push_codes_emit_ragged")


@pytest.fixture(scope="module")
def gen():
    return pkg.B200Generator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0), device="cuda", max_positions=256)


class batch_invariant:
    def __init__(self, gen):
        self.gen = gen

    def __enter__(self):
        self.gen.set_option("small_m_split_k", 0)

    def __exit__(self, *exc):
        self.gen.set_option("small_m_split_k", 1)


def _audio(i, secs=8.0):
    return pkg.synth_audio(int(SR * secs), file_id=90 + i).numpy()


def _count_calls(pool):
    """Record the name of every engine call the batcher makes on `pool`."""
    calls = []
    for name in KINDS:
        f = getattr(pool, name)
        setattr(pool, name, lambda *a, _f=f, _n=name, **k: (calls.append(_n), _f(*a, **k))[1])
    return calls


def _chunk_len(tick):
    return {4: 320, 9: 1000, 13: 320}.get(tick, CHUNK)       # 20 ms ticks and one non-hop-multiple chunk among 0.1 s ones


def _run_equality(gen, joins, ticks, context_secs, target):
    bat = SessionBatcher(gen, context_secs=context_secs, max_sessions=8, ragged=True)
    emb = SessionBatcher(gen, context_secs=context_secs, max_sessions=8, ragged=True)
    emb.arm_emit(0.1, 0.02, target)
    calls, ecalls = _count_calls(bat.pool), _count_calls(emb.pool)
    wav = [_audio(i) for i in range(len(joins))]
    sids, esids, toks, ems, pos = {}, {}, {}, {}, [0] * len(joins)
    for t in range(ticks):
        for i, j in enumerate(joins):
            if t == j:
                sids[i], esids[i] = bat.open_session(), emb.open_session()
                toks[i] = pkg.AudioTokenizer(codec_model=gen, context_secs=context_secs, device="cuda")
                ems[i] = pkg.OutputChunkEmitter(pkg.AudioTokenizer(codec_model=gen, context_secs=context_secs, device="cuda"),
                                                0.1, 0.02, target)
        n = _chunk_len(t)
        del calls[:]
        got = bat.tokenize_audio({sids[i]: wav[i][pos[i]:pos[i] + n] for i in sids})
        assert calls == ["push_audio_ragged"], (t, calls)
        strings = {}
        for i in sids:
            strings[i] = toks[i].tokenize_audio(wav[i][pos[i]:pos[i] + n])
            assert got[sids[i]] == strings[i], f"encode tick {t} session {i}"
            pos[i] += n
        for pre in (0, 320):
            del calls[:]
            out = bat.detokenize_audio({sids[i]: strings[i] for i in sids}, preroll_samples=pre)
            assert calls == ["push_codes_ragged"], (t, calls)
            for i in sids:
                (sr, w), hang, left = out[sids[i]]
                (sr2, w2), hang2, left2 = toks[i].detokenize_audio(strings[i], preroll_samples=pre)
                assert (sr, hang, left) == (sr2, hang2, left2) and w.shape == w2.shape and np.array_equal(w, w2), \
                    f"decode tick {t} session {i} preroll {pre}"
        if n == CHUNK:
            pieces = {i: strings[i] for i in sids}
            del ecalls[:]
            eout = emb.emit_output_chunks({esids[i]: pieces[i] for i in sids})
            assert ecalls == ["push_codes_emit_ragged"], (t, ecalls)
            for i in sids:
                assert np.array_equal(eout[esids[i]], ems[i].emit(pieces[i])), f"emit tick {t} session {i}"
    for i in sids:
        assert np.array_equal(np.concatenate(emb.audio_history_ch1(esids[i])), np.concatenate(ems[i].audio_history_ch1))


@pytest.mark.parametrize("context_secs,target", [(2.0, 0.0), (2.0, 0.05), (3.0, 0.05)])
def test_ragged_sessions_equal_lone_sessions(gen, context_secs, target):
    """Sessions join at different ticks; a 3.0 s context (150 frames) takes the attention halo kernel."""
    with batch_invariant(gen):
        _run_equality(gen, [0, 0, 2, 5, 11], 36 if context_secs > 2 else 26, context_secs, target)


def test_ragged_sessions_equal_lone_sessions_default_spec():
    spec = pkg.DEFAULT_SPEC
    g = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda")
    with batch_invariant(g):
        _run_equality(g, [0, 1, 3, 8], 24, 2.0, 0.05)


def test_equal_lengths_match_the_uniform_call(gen):
    """Default kernels: with equal lengths a ragged call is the uniform call (same graph, same bits)."""
    a, b = SessionPool(gen, 1, 32000, 6), SessionPool(gen, 1, 32000, 6)
    fade = create_crossfade_ramps(SR, fade_secs=0.02)[1]
    for p in (a, b):
        p.set_emit(CHUNK, 320, 0.05, 0.003, fade)
    wav = np.stack([_audio(i) for i in range(3)])[:, None]
    rng = np.random.default_rng(5)
    for t in range(24):
        x = wav[..., t * CHUNK:(t + 1) * CHUNK]
        assert np.array_equal(a.push_audio([0, 1, 2], x, 5), b.push_audio_ragged([0, 1, 2], x, 5))
        c = rng.integers(0, gen.codebook_size, size=(3, 1, 5))
        w1 = a.push_codes([0, 1, 2], c, 1920)
        w2, got = b.push_codes_ragged([0, 1, 2], c, 1920)
        assert np.array_equal(got, [w1.shape[-1]] * 3) and np.array_equal(w1, w2[..., :w1.shape[-1]])
        assert not w2[..., w1.shape[-1]:].any()
        e = rng.integers(0, gen.codebook_size, size=(3, 5))
        (o1, h1), (o2, h2) = a.push_codes_emit([3, 4, 5], e), b.push_codes_emit_ragged([3, 4, 5], e)
        assert np.array_equal(o1, o2) and list(h2) == [h1] * 3


def test_default_kernels_agree_with_lone_sessions(gen):
    """Default kernels: the mixed batch and the lone session take different GEMM kernels (different fp32 summation
    order), so near-tie codes may differ, as in test_gpu_pool.py."""
    joins = [0, 0, 1, 3, 3, 6, 9, 12]
    bat = SessionBatcher(gen, max_sessions=8, ragged=True)
    sids, toks, agree = {}, {}, []
    for t in range(30):
        for i, j in enumerate(joins):
            if t == j:
                sids[i], toks[i] = bat.open_session(), pkg.AudioTokenizer(codec_model=gen, device="cuda")
        got = bat.tokenize_audio({sids[i]: _audio(i)[(t - joins[i]) * CHUNK:(t - joins[i] + 1) * CHUNK] for i in sids})
        for i in sids:
            ref = toks[i].tokenize_audio(_audio(i)[(t - joins[i]) * CHUNK:(t - joins[i] + 1) * CHUNK])
            agree += [x == y for x, y in zip(got[sids[i]], ref)]
    print(f"[pool ragged] mixed batches (default kernels) vs lone sessions: {np.mean(agree):.4f} of {len(agree)} codes equal")
    assert np.mean(agree) > 0.9


def test_ragged_errors_change_nothing(gen):
    wav = np.stack([_audio(i) for i in range(3)])[:, None]
    fade = create_crossfade_ramps(SR, fade_secs=0.02)[1]
    codes = np.random.default_rng(3).integers(0, gen.codebook_size, size=(3, 1, 5))

    def prime(p):
        p.push_audio_ragged([0], wav[:1, :, :CHUNK], 5)                  # slot 0: 1600 samples, slots 1, 2: none
        p.push_codes_ragged([1], codes[:1], 320)                          # slot 1: 5 frames of code context

    a, ref = SessionPool(gen, 1, 32000, 3), SessionPool(gen, 1, 32000, 3)
    prime(a); prime(ref)
    lens = [a.context_len(s) for s in range(3)]
    x = wav[:, :, CHUNK:2 * CHUNK]
    bad = [(lambda: a.push_audio_ragged([0, 0], x[:2], 5), "listed twice"),
           (lambda: a.push_audio_ragged([0, 3], x[:2], 5), "out of range"),
           (lambda: a.push_audio_ragged([0, 1], np.zeros((2, 1, 32001), np.float32), 5), "exceeds"),
           (lambda: a.push_audio_ragged([0, 1], x[:2], 0), "keep_frames"),
           (lambda: a.push_audio_ragged([0, 1], x[:2], 6), "keep_frames"),
           (lambda: a.push_codes_ragged([0, 1], np.zeros((2, 1, 101), np.int64), 320), "exceed"),
           (lambda: a.push_codes_emit_ragged([0, 1], codes[:2, 0]), "set_emit")]
    for call, msg in bad:
        with pytest.raises(McError, match=msg):
            call()
        assert [a.context_len(s) for s in range(3)] == lens
    a.set_emit(CHUNK, 320, 0.0, 0.003, fade); ref.set_emit(CHUNK, 320, 0.0, 0.003, fade)
    with pytest.raises(McError, match="empty code context"):
        a.push_codes_emit_ragged([0, 1], codes[:2, 0])                    # slot 1 holds codes but emitted no chunk
    assert [a.context_len(s) for s in range(3)] == lens
    # later results are those of a pool that never saw the errors
    assert np.array_equal(a.push_audio_ragged([0, 1, 2], x, 5), ref.push_audio_ragged([0, 1, 2], x, 5))
    wa, ga = a.push_codes_ragged([0, 1, 2], codes, 1920)
    wr, gr = ref.push_codes_ragged([0, 1, 2], codes, 1920)
    assert np.array_equal(wa, wr) and np.array_equal(ga, gr) and list(ga) == [1600, 1920, 1600]
    # mixed lengths need causal attention
    spec = pkg.TINY_SPEC.replace(window_left=24, window_right=8)
    g2 = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda", max_positions=256)
    p = SessionPool(g2, 1, 32000, 2)
    p.push_audio_ragged([0], wav[:1, :, :CHUNK], 5)
    p.push_codes_ragged([0], codes[:1], 320)
    with pytest.raises(McError, match="causal"):
        p.push_audio_ragged([0, 1], x[:2], 5)
    with pytest.raises(McError, match="causal"):
        p.push_codes_ragged([0, 1], codes[:2], 320)
    assert p.context_len(0) == (CHUNK, 5) and p.context_len(1) == (0, 0)
    assert p.push_audio_ragged([0], x[:1], 5).shape == (1, 1, 5)          # equal lengths still work there


def test_a_second_warm_up_cohort_captures_no_new_graphs(gen):
    """One steady session; three sessions warm up next to it (joining 2 ticks apart), leave, and a second and a third
    cohort do the same: the per-item lengths live in the uploaded table, so the graph keys repeat exactly."""
    bat = ThreadedSessionBatcher(gen, max_sessions=4, ragged=True)
    try:
        bat.arm_emit()
        steady = bat.open_session()
        for t in range(22):
            bat.tokenize_audio({steady: _audio(0)[t * CHUNK:(t + 1) * CHUNK]})
        rng = np.random.default_rng(9)

        def cohort():
            sids = {}
            for t in range(10):
                if t in (0, 2, 4):
                    sids[t] = bat.open_session()
                bat.tokenize_audio({s: _audio(1)[t * CHUNK:(t + 1) * CHUNK] for s in [steady, *sids.values()]})
                bat.emit_output_chunks({s: codes_to_chars(rng.integers(0, gen.codebook_size, size=(1, 5)), gen.codebook_size,
                                                          unicode_offset=UNICODE_OFFSET_LARGE) for s in sids.values()})
            for s in sids.values():
                bat.close_session(s)
            return bat.pool.graph_count()

        keys_a, _ = cohort()
        keys_b, captured_b = cohort()
        keys_c, captured_c = cohort()
        assert keys_a == keys_b == keys_c and captured_c == captured_b, (keys_a, keys_b, keys_c, captured_b, captured_c)
    finally:
        bat.shutdown()
