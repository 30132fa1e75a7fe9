"""CPU: the host logic of SessionBatcher.emit_output_chunks and the ThreadedSessionBatcher dispatcher, with a numpy
stand-in for the engine's session pool (``session_batcher.SessionPool`` is swapped for ``FakePool`` in this file only).

FakePool keeps each slot's code context like mc_pool_* does, "decodes" a context with a deterministic function of its
codes, and runs the agent's output chain with the numpy utilities, so a session driven through the batcher can be held
to an OutputChunkEmitter over a tokenizer that decodes the same way."""
import threading
from concurrent.futures import Future

import numpy as np
import pytest

import realtime_codec_agent_b200 as pkg
from realtime_codec_agent_b200 import audio_utils, session_batcher
from realtime_codec_agent_b200.codec_chars import UNICODE_OFFSET_LARGE, codes_to_chars

SR, HOP, K = 16000, 320, 4096
CHUNK, L = 1600, 320                     # 0.1 s chunks (5 codes), 0.02 s fade


def fake_decode(codes: np.ndarray) -> np.ndarray:
    """[F] codes -> [F*HOP] samples; every sample depends on the whole window, so a wrong context shows."""
    codes = np.asarray(codes, dtype=np.float64)
    phase = np.cumsum(codes)[:, None] * 1e-3 + codes[:, None] * 0.37 + np.arange(HOP)[None] * 0.05
    return (0.2 * np.sin(phase)).reshape(-1).astype(np.float32)


class FakeGen:
    is_b200_native = True
    sample_rate, hop, codebook_size = SR, HOP, K


class FakePool:
    """mc_pool_* bookkeeping and the emit chain of mc_pool_push_codes_emit, in numpy."""

    def __init__(self, gen, channels, context_samples, max_sessions, max_chunk_samples=0):
        self.gen, self.channels, self.max_sessions = gen, channels, max_sessions
        self.cap_samples = max(context_samples, max_chunk_samples)
        self.cap_frames = -(-self.cap_samples // HOP)
        self.ctx_frames = context_samples // HOP
        self.ctx = [np.zeros(0, np.int64) for _ in range(max_sessions)]
        self.audio_len = [0] * max_sessions
        self.has_prev = [False] * max_sessions
        self.tails = [None] * max_sessions
        self.emit = None
        self.calls = []

    def reset(self, slot, audio=True, codes=True):
        if audio:
            self.audio_len[slot] = 0
        if codes:
            self.ctx[slot] = np.zeros(0, np.int64)
            self.has_prev[slot] = False

    def context_len(self, slot):
        return self.audio_len[slot], len(self.ctx[slot])

    def _check(self, slots):
        assert len(set(slots)) == len(slots), "slot listed twice"
        if len({len(self.ctx[s]) for s in slots}) != 1:
            raise AssertionError("contexts of different length in one launch")

    def _roll(self, slot, new):
        self.ctx[slot] = np.concatenate((self.ctx[slot], new))[-max(len(new), self.ctx_frames):]
        return fake_decode(self.ctx[slot])

    def push_audio(self, slots, chunks, keep_frames):
        self.calls.append(("encode", list(slots)))
        out = []
        for s, x in zip(slots, chunks):
            self.audio_len[s] = min(self.audio_len[s] + x.shape[-1], max(x.shape[-1], self.cap_samples))
            frames = -(-x.shape[-1] // HOP) if keep_frames <= 0 else keep_frames
            out.append((np.abs(x[:, :frames * HOP:HOP]) * 1000).astype(np.int64) % K)
        return np.stack(out)

    def push_codes(self, slots, codes, keep_samples):
        self.calls.append(("decode", list(slots)))
        self._check(slots)
        return np.stack([self._roll(s, c.reshape(-1))[-keep_samples:][None] for s, c in zip(slots, codes)])

    def set_emit(self, chunk, fade, target_rms, silence_thr, fade_in):
        self.emit = (chunk, fade, target_rms, silence_thr, np.asarray(fade_in, np.float32))
        self.has_prev = [False] * self.max_sessions

    def push_codes_emit(self, slots, codes):
        self.calls.append(("emit", list(slots)))
        self._check(slots)
        chunk, fade, target, thr, fade_in = self.emit
        had = self.has_prev[slots[0]]
        assert all(self.has_prev[s] == had for s in slots)
        blocks = []
        for s, c in zip(slots, codes):
            w = self._roll(s, c)[-(chunk + fade):]
            assert len(w) == (chunk + fade if had else chunk)
            x = audio_utils.pad_or_trim(w, chunk + fade if had else chunk)
            if target > 0:
                x = audio_utils.normalize_audio_rms(x, target_rms=target, silence_rms_threshold=thr)
            if had:
                cross = self.tails[s] * fade_in[::-1] + x[:fade] * fade_in
                block = np.concatenate((cross, x[fade:chunk], cross, x[fade:fade + chunk]))
                self.tails[s] = x[chunk:chunk + fade].copy()
            else:
                block = np.concatenate((np.zeros(fade, np.float32), x[:chunk - fade], np.zeros(fade, np.float32), x))
                self.tails[s] = x[chunk - fade:].copy()
            self.has_prev[s] = True
            blocks.append(block.astype(np.float32))
        return np.stack(blocks), had


class FakeTokenizer:
    """AudioTokenizer.detokenize_audio over the fake decoder (string context of max(len, context) chars)."""
    num_channels, sampling_rate, _native = 1, SR, False

    def __init__(self, context_frames=100):
        self.context_frames, self.detokenize_context = context_frames, ""

    def detokenize_audio(self, s, preroll_samples=0):
        self.detokenize_context = (self.detokenize_context + s)[-max(len(s), self.context_frames):]
        codes = np.array([ord(ch) - UNICODE_OFFSET_LARGE for ch in self.detokenize_context], np.int64)
        want = len(s) * HOP + preroll_samples
        wav = fake_decode(codes)[-want:]
        return (SR, wav), "", max(0, preroll_samples - want + wav.shape[-1])


class NativeFakeTokenizer:
    """The native tokenizer's emit surface (arm_emit / detokenize_audio_emit) on a one-slot FakePool."""
    num_channels, sampling_rate, _native = 1, SR, True

    def __init__(self):
        self.pool = FakePool(FakeGen(), 1, 2 * SR, 1)

    def arm_emit(self, chunk, fade, target, thr, fade_in):
        self.pool.set_emit(chunk, fade, target, thr, fade_in)

    def detokenize_audio_emit(self, s):
        blocks, had = self.pool.push_codes_emit([0], np.array([[ord(ch) - UNICODE_OFFSET_LARGE for ch in s]], np.int64))
        return blocks[0], had


@pytest.fixture(autouse=True)
def fake_pool(monkeypatch):
    monkeypatch.setattr(session_batcher, "SessionPool", FakePool)


def _codes(i, tick):
    rng = np.random.default_rng(1000 * i + tick)
    return codes_to_chars(rng.integers(0, K, size=(1, 5)), K, unicode_offset=UNICODE_OFFSET_LARGE)


def _run_agents(bat, joins, ticks):
    """Sessions i joins at tick joins[i]; -> (sids, per-session emitted chunks, launches per tick)."""
    sids, got, launches = {}, {i: [] for i in range(len(joins))}, []
    for t in range(ticks):
        for i, j in enumerate(joins):
            if t == j:
                sids[i] = bat.open_session()
        n0 = len(bat.pool.calls)
        out = bat.emit_output_chunks({sids[i]: _codes(i, t) for i in sids})
        launches.append(bat.pool.calls[n0:])
        for i in sids:
            got[i].append(out[sids[i]])
    return sids, got, launches


@pytest.mark.parametrize("target", [0.0, 0.05])
def test_emit_equals_private_emitters_and_groups_by_context_length(target):
    joins = [0, 0, 3, 7, 7, 12]
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=8)
    bat.arm_emit(0.1, 0.02, target)
    ticks = 40                                                                # every context full by the end
    sids, got, launches = _run_agents(bat, joins, ticks)
    for i, j in enumerate(joins):
        ref = pkg.OutputChunkEmitter(FakeTokenizer(), 0.1, 0.02, target)          # numpy chain, call for call the reference
        nat = pkg.OutputChunkEmitter(NativeFakeTokenizer(), 0.1, 0.02, target)    # _emit_native's history assembly
        for t in range(j, ticks):
            want = ref.emit(_codes(i, t))
            assert np.array_equal(got[i][t - j], want), (i, t)
            assert np.array_equal(nat.emit(_codes(i, t)), want)
        hist = np.concatenate(bat.audio_history_ch1(sids[i]))
        assert np.array_equal(hist, np.concatenate(ref.audio_history_ch1))
        assert np.array_equal(hist, np.concatenate(nat.audio_history_ch1))
        assert bat._sessions[sids[i]].detok_context == ref.audio_tokenizer.detokenize_context
    for t, calls in enumerate(launches):                                      # one launch per context length
        lens = {min(5 * (t - j), 100) for j in joins if j <= t}
        assert len(calls) == len(lens) and all(k == "emit" for k, _ in calls), (t, calls)
    assert len(launches[-1]) == 1 and sorted(launches[-1][0][1]) == sorted(bat._sessions[s].slot for s in sids.values())


def test_a_rejected_batch_changes_nothing():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=4)
    with pytest.raises(ValueError, match="arm_emit"):
        bat.emit_output_chunks({})
    bat.arm_emit()
    a, b, c = bat.open_session(), bat.open_session(), bat.open_session()
    bat.emit_output_chunks({a: _codes(0, 0), b: _codes(1, 0)})
    bat.detokenize_audio({c: _codes(2, 0)})                                    # c: a code context but no previous chunk

    def snapshot():
        return ({s: bat._sessions[s].detok_context for s in (a, b, c)},
                {s: [h.copy() for h in bat.audio_history_ch1(s)] for s in (a, b, c)}, len(bat.pool.calls))

    before = snapshot()
    for bad in ({a: _codes(0, 1), b: _codes(1, 1)[:4]},                          # 4 codes are not one chunk
                {a: _codes(0, 1), 999: _codes(1, 1)},                            # unknown session
                {a: _codes(0, 1), c: _codes(2, 1)}):                             # first emit after a plain decode
        with pytest.raises((ValueError, KeyError)):
            bat.emit_output_chunks(bad)
        after = snapshot()
        assert after[0] == before[0] and after[2] == before[2]
        assert all(len(after[1][s]) == len(before[1][s]) and all(np.array_equal(x, y) for x, y in zip(after[1][s], before[1][s]))
                   for s in (a, b, c))


def test_reset_close_reopen_and_rearm_clear_the_history():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=2)
    bat.arm_emit()
    a, b = bat.open_session(), bat.open_session()
    for t in range(3):
        bat.emit_output_chunks({a: _codes(0, t), b: _codes(1, t)})
    assert len(bat.audio_history_ch1(a)) == 3
    bat.reset_context(a)
    assert bat.audio_history_ch1(a) == [] and bat._sessions[a].detok_context == ""
    first = bat.emit_output_chunks({a: _codes(0, 0)})[a]                        # a first chunk again: L zeros, then audio
    assert np.array_equal(first, pkg.OutputChunkEmitter(FakeTokenizer(), 0.1, 0.02).emit(_codes(0, 0)))
    bat.close_session(b)
    b2 = bat.open_session()
    assert bat.audio_history_ch1(b2) == []
    assert np.array_equal(bat.emit_output_chunks({b2: _codes(5, 0)})[b2][:L], np.zeros(L, np.float32))
    bat.arm_emit()
    assert bat.audio_history_ch1(a) == [] and bat.audio_history_ch1(b2) == []


def test_arm_emit_checks_like_the_emitter():
    with pytest.raises(ValueError, match="mono"):
        session_batcher.SessionBatcher(FakeGen(), num_channels=2).arm_emit()
    bat = session_batcher.SessionBatcher(FakeGen())
    with pytest.raises(ValueError, match="fade"):
        bat.arm_emit(0.1, 0.0)
    with pytest.raises(ValueError, match="fade"):
        bat.arm_emit(0.1, 0.2)


def _enqueue(bat, reqs):
    """Queue requests for ONE dispatcher tick without blocking (the *_one calls block on their own request)."""
    futs = []
    with bat._cv:
        for kind, sid, payload in reqs:
            futs.append(Future())
            bat._pending.append((kind, sid, payload, futs[-1]))
        bat._cv.notify()
    return futs


def test_dispatcher_routes_kinds_defers_repeats_and_fails_bad_requests_alone():
    bat = session_batcher.ThreadedSessionBatcher(FakeGen(), max_sessions=4, max_wait_ms=1.0)
    ref = session_batcher.SessionBatcher(FakeGen(), max_sessions=4)
    try:
        bat.arm_emit(); ref.arm_emit()
        a, b, c = bat.open_session(), bat.open_session(), bat.open_session()
        rb, rc = ref.open_session(), ref.open_session()
        audio = np.linspace(-0.5, 0.5, 1600, dtype=np.float32)
        futs = _enqueue(bat, [(("emit",), a, _codes(0, 0)),
                              (("emit",), a, _codes(0, 1)),                   # same (session, kind): next tick
                              (("decode", 320), c, _codes(2, 0)),
                              (("encode",), b, audio),
                              (("emit",), b, _codes(1, 0)[:3]),                # malformed: fails alone
                              (("decode", 0), b, _codes(1, 0)),
                              (("emit",), 999, _codes(2, 0))])                 # closed session: fails alone
        res = [f.result(timeout=10) if f.exception(timeout=10) is None else f.exception() for f in futs]
        # tick 1: encode, decode (preroll 0), decode (preroll 320), the emit batch (rejected, then served one by one);
        # tick 2: a's second emit
        assert bat.pool.calls == [("encode", [bat._sessions[b].slot]), ("decode", [bat._sessions[b].slot]),
                                  ("decode", [bat._sessions[c].slot]), ("emit", [bat._sessions[a].slot]),
                                  ("emit", [bat._sessions[a].slot])]
        assert isinstance(res[4], ValueError) and isinstance(res[6], KeyError)
        em = pkg.OutputChunkEmitter(FakeTokenizer(), 0.1, 0.02)
        assert np.array_equal(res[0], em.emit(_codes(0, 0))) and np.array_equal(res[1], em.emit(_codes(0, 1)))
        assert res[3] == ref.tokenize_audio({rb: audio})[rb]
        for got, sid, pre, i in ((res[5], rb, 0, 1), (res[2], rc, 320, 2)):
            (_, w), hang, left = got
            (_, w2), hang2, left2 = ref.detokenize_audio({sid: _codes(i, 0)}, preroll_samples=pre)[sid]
            assert np.array_equal(w, w2) and (hang, left) == (hang2, left2)
        # the blocking entry points from a request thread
        c = bat.open_session()
        outs, errs = [], []

        def agent():
            try:
                for t in range(4):
                    bat.tokenize_audio_one(c, audio)
                    outs.append(bat.emit_output_chunk_one(c, _codes(3, t)))
            except Exception as ex:                                      # noqa: BLE001
                errs.append(ex)

        th = threading.Thread(target=agent)
        th.start(); th.join(timeout=30)
        assert not errs and len(outs) == 4
        em = pkg.OutputChunkEmitter(FakeTokenizer(), 0.1, 0.02)
        assert all(np.array_equal(o, em.emit(_codes(3, t))) for t, o in enumerate(outs))
        assert np.array_equal(np.concatenate(bat.audio_history_ch1(c)), np.concatenate(em.audio_history_ch1))
    finally:
        bat.shutdown()
