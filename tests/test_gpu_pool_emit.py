"""GPU (B200): the agent's output chain for many pooled sessions in one launch (mc_pool_set_emit /
mc_pool_push_codes_emit, SessionBatcher.emit_output_chunks, ThreadedSessionBatcher.emit_output_chunk_one).

Every session must get what its own AudioTokenizer + OutputChunkEmitter gives: bit for bit with the batch-invariant
kernels (small_m_split_k = 0, as in test_gpu_pool.py); with the default kernels, the chain is held to the oracle chain
fed with a decode of the same batch (bit for bit at target_rms = 0, test_gpu_post.py's tolerances with RMS on)."""
import threading

import numpy as np
import pytest

import realtime_codec_agent_b200 as pkg
from oracle import post_decode_oracle as po
from realtime_codec_agent_b200._native import McError
from realtime_codec_agent_b200.audio_utils import create_crossfade_ramps
from realtime_codec_agent_b200.codec_chars import UNICODE_OFFSET_LARGE, chars_to_codes
from realtime_codec_agent_b200.session_batcher import SessionBatcher, SessionPool, ThreadedSessionBatcher

pytestmark = pytest.mark.gpu
SR, CHUNK, L, CODES = 16000, 1600, 320, 5
RMS_RTOL, RMS_ATOL = 2e-6, 1e-7                 # test_gpu_post.py


@pytest.fixture(scope="module")
def gen():
    return pkg.B200Generator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0), device="cuda", max_positions=256)


@pytest.fixture(scope="module")
def strings(gen):
    """An output code string of 4 s per agent (the codes of synthetic speech-like audio)."""
    out = []
    for i in range(8):
        tok = pkg.AudioTokenizer(codec_model=gen, device="cuda")
        out.append(tok.tokenize_audio(pkg.synth_audio(4 * SR, file_id=70 + i).numpy()))
    return out


class batch_invariant:
    def __init__(self, gen):
        self.gen = gen

    def __enter__(self):
        self.gen.set_option("small_m_split_k", 0)

    def __exit__(self, *exc):
        self.gen.set_option("small_m_split_k", 1)


def _piece(s, k):
    return s[k * CODES:(k + 1) * CODES]


def _codes(gen, s):
    return chars_to_codes(s, 1, gen.codebook_size, unicode_offset=UNICODE_OFFSET_LARGE)        # [1, len]


@pytest.mark.parametrize("target", [0.0, 0.05])
def test_pool_emit_equals_lone_agents(gen, strings, target):
    """6 sessions join at different ticks (first-chunk groups next to steady ones) for 40 ticks."""
    joins = [0, 0, 2, 5, 5, 9]
    with batch_invariant(gen):
        bat = SessionBatcher(gen, max_sessions=8)
        bat.arm_emit(0.1, 0.02, target)
        sids, ems = {}, {}
        for tick in range(40):
            for i, j in enumerate(joins):
                if tick == j:
                    sids[i] = bat.open_session()
                    ems[i] = pkg.OutputChunkEmitter(pkg.AudioTokenizer(codec_model=gen, device="cuda"), 0.1, 0.02, target)
            out = bat.emit_output_chunks({sids[i]: _piece(strings[i], tick - joins[i]) for i in sids})
            for i in sids:
                want = ems[i].emit(_piece(strings[i], tick - joins[i]))
                assert out[sids[i]].shape == (CHUNK,) and np.array_equal(out[sids[i]], want), f"tick {tick} session {i}"
        for i in sids:
            assert np.array_equal(np.concatenate(bat.audio_history_ch1(sids[i])), np.concatenate(ems[i].audio_history_ch1))
            assert bat._sessions[sids[i]].detok_context == ems[i].audio_tokenizer.detokenize_context


class _Decoded:
    """detokenize_audio returning a result computed elsewhere (the oracle chain's decoder input)."""
    sampling_rate = SR

    def __init__(self):
        self.result = None

    def detokenize_audio(self, s, preroll_samples=0):
        assert preroll_samples == L
        return self.result


@pytest.mark.parametrize("target", [0.0, 0.05])
def test_pool_emit_equals_oracle_chain_with_default_kernels(gen, strings, target):
    """A second batcher decodes the same batches (same B, same rows -> the same bits) with preroll L; the oracle chain
    turns each session's window into the agent's chunk."""
    joins = [0, 0, 3, 3, 6]
    bat, dec = SessionBatcher(gen, max_sessions=8), SessionBatcher(gen, max_sessions=8)
    bat.arm_emit(0.1, 0.02, target)
    sids, dsids, shims, chains = {}, {}, {}, {}
    tol = dict(rtol=RMS_RTOL, atol=RMS_ATOL) if target else dict(rtol=0.0, atol=0.0)
    for tick in range(30):
        for i, j in enumerate(joins):
            if tick == j:
                sids[i], dsids[i], shims[i] = bat.open_session(), dec.open_session(), _Decoded()
                chains[i] = po.OracleOutputChain(shims[i], 0.1, 0.02, target)
        out = bat.emit_output_chunks({sids[i]: _piece(strings[i], tick - joins[i]) for i in sids})
        wins = dec.detokenize_audio({dsids[i]: _piece(strings[i], tick - joins[i]) for i in sids}, preroll_samples=L)
        for i in sids:
            shims[i].result = wins[dsids[i]]
            want = chains[i].step(_piece(strings[i], tick - joins[i]))
            assert np.allclose(out[sids[i]], want, **tol), f"tick {tick} session {i}"
    for i in sids:
        a, b = np.concatenate(bat.audio_history_ch1(sids[i])), np.concatenate(chains[i].history)
        assert a.shape == b.shape and np.allclose(a, b, **tol)


def test_a_steady_tick_is_one_graph_replay(gen, strings):
    bat = SessionBatcher(gen, max_sessions=8)
    bat.arm_emit()
    sids = [bat.open_session() for _ in range(5)]
    for tick in range(25):                                               # fill the 2 s contexts, capture the graph
        bat.emit_output_chunks({s: _piece(strings[i], tick) for i, s in enumerate(sids)})
    l0 = gen.launch_count
    bat.emit_output_chunks({s: _piece(strings[i], 25) for i, s in enumerate(sids)})
    assert gen.launch_count - l0 == 1


def test_reset_recycle_and_rearm_start_fresh(gen, strings):
    with batch_invariant(gen):
        bat = SessionBatcher(gen, max_sessions=2)
        bat.arm_emit()
        a, b = bat.open_session(), bat.open_session()
        tok = pkg.AudioTokenizer(codec_model=gen, device="cuda")
        em = pkg.OutputChunkEmitter(tok, 0.1, 0.02)
        for k in range(4):
            bat.emit_output_chunks({a: _piece(strings[0], k), b: _piece(strings[1], k)})
            em.emit(_piece(strings[0], k))
        bat.reset_context(a)                                             # mid-stream: the next chunk is a first chunk
        em.reset(); tok.reset_context()
        slot = bat._sessions[a].slot
        blocks, had_prev = bat.pool.push_codes_emit([slot], _codes(gen, _piece(strings[0], 4)))
        assert had_prev is False
        want = em.emit(_piece(strings[0], 4))
        assert np.array_equal(blocks[0, :CHUNK], want) and np.all(blocks[0, :L] == 0)
        bat.close_session(b)                                             # a recycled slot starts from nothing
        b2 = bat.open_session()
        fresh = pkg.OutputChunkEmitter(pkg.AudioTokenizer(codec_model=gen, device="cuda"), 0.1, 0.02)
        assert np.array_equal(bat.emit_output_chunks({b2: _piece(strings[2], 0)})[b2], fresh.emit(_piece(strings[2], 0)))
        bat.arm_emit()                                                   # forgets every previous chunk
        assert bat.audio_history_ch1(b2) == []
        with pytest.raises(McError, match="empty code context"):
            bat.pool.push_codes_emit([bat._sessions[b2].slot], _codes(gen, _piece(strings[2], 1)))
        bat.reset_context(b2)
        assert bat.pool.push_codes_emit([bat._sessions[b2].slot], _codes(gen, _piece(strings[2], 0)))[1] is False


def test_pool_emit_errors_leave_contexts_unchanged(gen, strings):
    codes = _codes(gen, _piece(strings[0], 0))
    ramp = create_crossfade_ramps(SR, 0.02)[1]
    pool = SessionPool(gen, 1, 2 * SR, 4)
    with pytest.raises(McError, match="set_emit"):
        pool.push_codes_emit([0], codes)
    pool.set_emit(CHUNK, L, 0.0, 0.003, ramp)
    with pytest.raises(McError):
        pool.set_emit(CHUNK, CHUNK + 1, 0.0, 0.003, np.zeros(CHUNK + 1, np.float32))     # fade > chunk
    pool.set_emit(CHUNK, L, 0.0, 0.003, ramp)
    pool.push_codes_emit([0], codes)                                     # slot 0: one chunk emitted
    pool.push_codes([1], codes[:, None], 0)                              # slot 1: a plain decode, no previous chunk
    lens = [pool.context_len(s) for s in range(4)]
    with pytest.raises(McError, match="decode to"):
        pool.push_codes_emit([2], codes[:, :4])                          # len * hop != chunk
    with pytest.raises(McError, match="empty code context"):
        pool.push_codes_emit([1], codes)                                 # first emit after a plain push_codes
    with pytest.raises(McError, match="different length"):
        pool.push_codes_emit([0, 2], np.concatenate([codes, codes]))
    with pytest.raises(McError):
        pool.push_codes_emit([0, 0], np.concatenate([codes, codes]))     # a slot twice
    assert [pool.context_len(s) for s in range(4)] == lens
    stereo = SessionPool(gen, 2, 2 * SR, 2)
    stereo.set_emit(CHUNK, L, 0.0, 0.003, ramp)
    with pytest.raises(McError, match="mono"):
        stereo.push_codes_emit([0], codes)
    assert stereo.context_len(0) == (0, 0)
    with pytest.raises(ValueError, match="mono"):
        SessionBatcher(gen, num_channels=2, max_sessions=2).arm_emit()
    bat = SessionBatcher(gen, max_sessions=2)
    s = bat.open_session()
    with pytest.raises(ValueError, match="arm_emit"):
        bat.emit_output_chunks({s: _piece(strings[0], 0)})
    assert bat.pool.context_len(bat._sessions[s].slot) == (0, 0) and bat._sessions[s].detok_context == ""


def test_threaded_agents_emit_like_private_agents(gen, strings):
    """S request threads each run an agent loop: tokenize their input chunk, emit their output chunk, every tick.  One
    more thread sends a malformed emit request, which fails alone."""
    S, ticks = 4, 16
    with batch_invariant(gen):
        bat = ThreadedSessionBatcher(gen, max_sessions=8, max_wait_ms=1.0)
        try:
            bat.arm_emit()
            inputs = [pkg.synth_audio(ticks * CHUNK, file_id=90 + i).numpy() for i in range(S)]
            refs = []
            for i in range(S):                                           # the private agent: one tokenizer, one emitter
                tok = pkg.AudioTokenizer(codec_model=gen, device="cuda")
                em = pkg.OutputChunkEmitter(tok, 0.1, 0.02)
                refs.append([(tok.tokenize_audio(inputs[i][t * CHUNK:(t + 1) * CHUNK]), em.emit(_piece(strings[i], t)))
                             for t in range(ticks)])
            got, errs, bad = {}, [], {}

            def agent(i):
                try:
                    sid = bat.open_session()
                    got[i] = [(bat.tokenize_audio_one(sid, inputs[i][t * CHUNK:(t + 1) * CHUNK]),
                               bat.emit_output_chunk_one(sid, _piece(strings[i], t))) for t in range(ticks)]
                except Exception as ex:                                  # noqa: BLE001
                    errs.append(ex)

            def malformed():
                sid = bat.open_session()
                for t in range(3):
                    try:
                        bat.emit_output_chunk_one(sid, _piece(strings[7], t)[:3])
                    except Exception as ex:                              # noqa: BLE001
                        bad[t] = ex

            ts = [threading.Thread(target=agent, args=(i,)) for i in range(S)] + [threading.Thread(target=malformed)]
            [t.start() for t in ts]; [t.join(timeout=120) for t in ts]
            assert not errs, errs
            assert len(bad) == 3 and all(isinstance(e, ValueError) for e in bad.values())
            for i in range(S):
                for t in range(ticks):
                    assert got[i][t][0] == refs[i][t][0], f"agent {i} tick {t} (encode)"
                    assert np.array_equal(got[i][t][1], refs[i][t][1]), f"agent {i} tick {t} (emit)"
        finally:
            bat.shutdown()
