"""CPU: SessionBatcher(ragged=True) host logic, with a numpy stand-in for the engine's session pool
(``session_batcher.SessionPool`` is swapped for ``RaggedFakePool`` in this file only).

RaggedFakePool keeps each slot's audio and code context like mc_pool_* does and "encodes" / "decodes" a context with a
causal deterministic function of it, so a wrong context or a wrong window offset shows.  Its ragged methods run every
slot by the lone semantics of the uniform ones; its uniform methods refuse contexts of different length as the engine
does.  Each session driven through a ragged batcher is held to the same session alone on a grouped batcher
(tokenize / detokenize) and to an OutputChunkEmitter (emit)."""
import threading

import numpy as np
import pytest

import realtime_codec_agent_b200 as pkg
from realtime_codec_agent_b200 import audio_utils, session_batcher
from realtime_codec_agent_b200.codec_chars import UNICODE_OFFSET_LARGE, codes_to_chars

SR, HOP, K = 16000, 320, 4096
CHUNK, L = 1600, 320


def fake_encode(x: np.ndarray) -> np.ndarray:
    """[C, T] audio -> [C, ceil(T/HOP)] codes; frame f depends on samples < (f+1)*HOP only (causal, zero padded)."""
    F = -(-x.shape[1] // HOP)
    pad = np.zeros((x.shape[0], F * HOP), np.float64)
    pad[:, :x.shape[1]] = x
    return (np.floor(np.abs(np.cumsum(pad, axis=1)[:, HOP - 1::HOP]) * 997) % K).astype(np.int64)


def fake_decode(codes: np.ndarray) -> np.ndarray:
    """[F] codes -> [F*HOP] samples; every sample depends on the whole window prefix."""
    codes = np.asarray(codes, dtype=np.float64)
    phase = np.cumsum(codes)[:, None] * 1e-3 + codes[:, None] * 0.37 + np.arange(HOP)[None] * 0.05
    return (0.2 * np.sin(phase)).reshape(-1).astype(np.float32)


class FakeGen:
    is_b200_native = True
    sample_rate, hop, codebook_size = SR, HOP, K


class RaggedFakePool:
    def __init__(self, gen, channels, context_samples, max_sessions, max_chunk_samples=0):
        self.gen, self.channels, self.max_sessions = gen, channels, max_sessions
        self.cap_samples = max(context_samples, max_chunk_samples)
        self.cap_frames = -(-self.cap_samples // HOP)
        self.ctx_samples, self.ctx_frames = context_samples, context_samples // HOP
        self.audio = [np.zeros((channels, 0), np.float32) for _ in range(max_sessions)]
        self.codes = [np.zeros((channels, 0), np.int64) for _ in range(max_sessions)]
        self.has_prev = [False] * max_sessions
        self.tails = [None] * max_sessions
        self.emit = None
        self.calls = []

    def reset(self, slot, audio=True, codes=True):
        if audio:
            self.audio[slot] = np.zeros((self.channels, 0), np.float32)
        if codes:
            self.codes[slot] = np.zeros((self.channels, 0), np.int64)
            self.has_prev[slot] = False

    def context_len(self, slot):
        return self.audio[slot].shape[1], self.codes[slot].shape[1]

    def _check(self, slots, ctx, ragged):
        assert len(set(slots)) == len(slots), "slot listed twice"
        if not ragged and len({ctx[s].shape[1] for s in slots}) != 1:
            raise AssertionError("contexts of different length in one launch")

    def _encode(self, slot, x, keep_frames):
        self.audio[slot] = np.concatenate((self.audio[slot], x), axis=1)[:, -max(x.shape[1], self.ctx_samples):]
        codes = fake_encode(self.audio[slot])
        return codes[:, -keep_frames:] if keep_frames > 0 else codes

    def _decode(self, slot, c):
        self.codes[slot] = np.concatenate((self.codes[slot], c), axis=1)[:, -max(c.shape[1], self.ctx_frames):]
        return np.stack([fake_decode(row) for row in self.codes[slot]])

    def push_audio(self, slots, chunks, keep_frames):
        self.calls.append(("encode", list(slots)))
        self._check(slots, self.audio, False)
        return np.stack([self._encode(s, x, keep_frames) for s, x in zip(slots, chunks)])

    def push_audio_ragged(self, slots, chunks, keep_frames):
        self.calls.append(("encode_ragged", list(slots)))
        self._check(slots, self.audio, True)
        assert 1 <= keep_frames <= -(-chunks.shape[-1] // HOP)
        return np.stack([self._encode(s, x, keep_frames) for s, x in zip(slots, chunks)])

    def push_codes(self, slots, codes, keep_samples):
        self.calls.append(("decode", list(slots)))
        self._check(slots, self.codes, False)
        return np.stack([self._decode(s, c)[:, -keep_samples:] for s, c in zip(slots, codes)])

    def push_codes_ragged(self, slots, codes, keep_samples):
        self.calls.append(("decode_ragged", list(slots)))
        self._check(slots, self.codes, True)
        assert 1 <= keep_samples <= self.cap_frames * HOP
        out = np.zeros((len(slots), self.channels, keep_samples), np.float32)
        got = np.zeros(len(slots), np.int32)
        for j, (s, c) in enumerate(zip(slots, codes)):
            w = self._decode(s, c)[:, -keep_samples:]
            out[j, :, :w.shape[1]], got[j] = w, w.shape[1]
        return out, got

    def set_emit(self, chunk, fade, target_rms, silence_thr, fade_in):
        self.emit = (chunk, fade, target_rms, silence_thr, np.asarray(fade_in, np.float32))
        self.has_prev = [False] * self.max_sessions

    def _emit_one(self, s, c):
        chunk, fade, target, thr, fade_in = self.emit
        had = self.has_prev[s]
        w = self._decode(s, c[None])[0][-(chunk + fade):]
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
        return block.astype(np.float32), had

    def push_codes_emit(self, slots, codes):
        self.calls.append(("emit", list(slots)))
        self._check(slots, self.codes, False)
        assert len({self.has_prev[s] for s in slots}) == 1
        res = [self._emit_one(s, c) for s, c in zip(slots, codes)]
        return np.stack([b for b, _ in res]), res[0][1]

    def push_codes_emit_ragged(self, slots, codes):
        self.calls.append(("emit_ragged", list(slots)))
        self._check(slots, self.codes, True)
        res = [self._emit_one(s, c) for s, c in zip(slots, codes)]
        return np.stack([b for b, _ in res]), np.array([h for _, h in res])


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


@pytest.fixture(autouse=True)
def fake_pool(monkeypatch):
    monkeypatch.setattr(session_batcher, "SessionPool", RaggedFakePool)


def _audio(i, channels=1, secs=12.0):
    rng = np.random.default_rng(77 + i)
    return (0.3 * rng.standard_normal((channels, int(SR * secs)))).astype(np.float32)


def _codes(i, tick):
    rng = np.random.default_rng(1000 * i + tick)
    return codes_to_chars(rng.integers(0, K, size=(1, 5)), K, unicode_offset=UNICODE_OFFSET_LARGE)


def _chunk_len(tick):
    return {5: 320, 11: 1000, 17: 100}.get(tick, 1600)         # 20 ms, a non-hop-multiple chunk, and a [-0:] chunk


@pytest.mark.parametrize("channels", [1, 2])
def test_one_call_per_kind_and_tick_equals_lone_sessions(channels):
    joins = [0, 0, 2, 6, 9, 13]
    ticks = 30                                                            # 0.1 s ticks: the earliest sessions reach steady state
    bat = session_batcher.SessionBatcher(FakeGen(), num_channels=channels, max_sessions=8, ragged=True)
    lone = [session_batcher.SessionBatcher(FakeGen(), num_channels=channels, max_sessions=1) for _ in joins]
    lsid = [b.open_session() for b in lone]
    wav = [_audio(i, channels)[0] if channels == 1 else _audio(i, channels) for i in range(len(joins))]
    sids, pos = {}, [0] * len(joins)
    for t in range(ticks):
        for i, j in enumerate(joins):
            if t == j:
                sids[i] = bat.open_session()
        n = _chunk_len(t)
        n0 = len(bat.pool.calls)
        got = bat.tokenize_audio({sids[i]: wav[i][..., pos[i]:pos[i] + n] for i in sids})
        enc_calls = bat.pool.calls[n0:]
        strings = {}
        for i in sids:
            ref = lone[i].tokenize_audio({lsid[i]: wav[i][..., pos[i]:pos[i] + n]})[lsid[i]]
            assert got[sids[i]] == ref, (t, i)
            pos[i] += n
            strings[i] = ref
        lens = {lone[i].pool.context_len(0)[0] for i in sids}
        if n == 100:                                                      # [-0:]: every frame of each window, grouped
            assert [k for k, _ in enc_calls] == ["encode"] * len({bat.pool.context_len(bat._sessions[sids[i]].slot)[0] for i in sids})
        else:
            assert [k for k, _ in enc_calls] == ["encode_ragged"], (t, enc_calls, lens)
        for pre in (0, 320):
            dec_in = {sids[i]: strings[i] for i in sids if len(strings[i]) >= channels}
            if not dec_in:
                continue
            n0 = len(bat.pool.calls)
            out = bat.detokenize_audio(dec_in, preroll_samples=pre)
            by_len = {len(s) // channels for s in dec_in.values()}
            assert [k for k, _ in bat.pool.calls[n0:]] == ["decode_ragged"] * len(by_len), t
            for i in sids:
                if sids[i] not in dec_in:
                    continue
                (sr, w), hang, left = out[sids[i]]
                (sr2, w2), hang2, left2 = lone[i].detokenize_audio({lsid[i]: strings[i]}, preroll_samples=pre)[lsid[i]]
                assert (sr, hang, left) == (sr2, hang2, left2) and w.shape == w2.shape and np.array_equal(w, w2), (t, i, pre)


@pytest.mark.parametrize("target", [0.0, 0.05])
def test_emit_is_one_call_per_tick_and_equals_private_emitters(target):
    joins = [0, 0, 3, 7, 7, 12]
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=8, ragged=True)
    bat.arm_emit(0.1, 0.02, target)
    ticks = 30
    sids, got = {}, {i: [] for i in range(len(joins))}
    for t in range(ticks):
        for i, j in enumerate(joins):
            if t == j:
                sids[i] = bat.open_session()
        n0 = len(bat.pool.calls)
        out = bat.emit_output_chunks({sids[i]: _codes(i, t) for i in sids})
        calls = bat.pool.calls[n0:]
        assert calls == [("emit_ragged", [bat._sessions[sids[i]].slot for i in sids])], (t, calls)   # first and continuing mixed
        for i in sids:
            got[i].append(out[sids[i]])
    for i, j in enumerate(joins):
        ref = pkg.OutputChunkEmitter(FakeTokenizer(), 0.1, 0.02, target)
        for t in range(j, ticks):
            assert np.array_equal(got[i][t - j], ref.emit(_codes(i, t))), (i, t)
        assert np.array_equal(np.concatenate(bat.audio_history_ch1(sids[i])), np.concatenate(ref.audio_history_ch1))
        assert bat._sessions[sids[i]].detok_context == ref.audio_tokenizer.detokenize_context


def test_a_rejected_ragged_batch_changes_nothing():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=4, ragged=True)
    bat.arm_emit()
    a, b, c = bat.open_session(), bat.open_session(), bat.open_session()
    bat.emit_output_chunks({a: _codes(0, 0)})
    bat.emit_output_chunks({a: _codes(0, 1), b: _codes(1, 0)})                  # a: continuing, b: first chunk, one call
    bat.detokenize_audio({c: _codes(2, 0)})                                    # c: a code context but no previous chunk
    bat.tokenize_audio({a: _audio(0)[0, :1600]})

    def snapshot():
        return ({s: bat._sessions[s].detok_context for s in (a, b, c)}, {s: bat._sessions[s].audio_len for s in (a, b, c)},
                {s: [h.copy() for h in bat.audio_history_ch1(s)] for s in (a, b, c)}, len(bat.pool.calls))

    before = snapshot()
    bad_calls = [(bat.emit_output_chunks, {a: _codes(0, 2), b: _codes(1, 1)[:4]}),     # 4 codes are not one chunk
                 (bat.emit_output_chunks, {a: _codes(0, 2), 999: _codes(1, 1)}),       # unknown session
                 (bat.emit_output_chunks, {a: _codes(0, 2), c: _codes(2, 1)}),         # first emit after a plain decode
                 (bat.tokenize_audio, {a: _audio(0)[0, :1600], b: np.zeros(0, np.float32)}),   # empty chunk
                 (bat.tokenize_audio, {a: _audio(0)[0, :1600], b: np.zeros(40000, np.float32)}),  # over the capacity
                 (bat.detokenize_audio, {c: _codes(2, 1), b: ""})]                      # empty string
    for call, req in bad_calls:
        with pytest.raises((ValueError, KeyError)):
            call(req)
        after = snapshot()
        assert after[0] == before[0] and after[1] == before[1] and after[3] == before[3]
        assert all(len(after[2][s]) == len(before[2][s]) and all(np.array_equal(x, y) for x, y in zip(after[2][s], before[2][s]))
                   for s in (a, b, c))


def test_default_stays_grouped():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=4)
    assert bat.ragged is False
    a, b = bat.open_session(), bat.open_session()
    bat.tokenize_audio({a: _audio(0)[0, :1600]})
    bat.tokenize_audio({a: _audio(0)[0, 1600:3200], b: _audio(1)[0, :1600]})
    assert [k for k, _ in bat.pool.calls] == ["encode", "encode", "encode"]


def test_threaded_batcher_forwards_ragged():
    bat = session_batcher.ThreadedSessionBatcher(FakeGen(), max_sessions=4, max_wait_ms=1.0, ragged=True)
    ref = [session_batcher.SessionBatcher(FakeGen(), max_sessions=1) for _ in range(3)]
    try:
        assert bat.ragged is True
        bat.arm_emit()
        sids = [bat.open_session() for _ in range(3)]
        rsid = [r.open_session() for r in ref]
        outs, errs = {i: [] for i in range(3)}, []

        def agent(i, start):
            try:
                for t in range(start, 6):
                    chunk = _audio(i)[0, t * 1600:(t + 1) * 1600]
                    outs[i].append((bat.tokenize_audio_one(sids[i], chunk), bat.emit_output_chunk_one(sids[i], _codes(i, t))))
            except Exception as ex:                                      # noqa: BLE001
                errs.append(ex)

        ths = [threading.Thread(target=agent, args=(i, s)) for i, s in enumerate((0, 2, 4))]   # sessions at different points
        [th.start() for th in ths]; [th.join(timeout=30) for th in ths]
        assert not errs, errs
        for i, start in enumerate((0, 2, 4)):
            em = pkg.OutputChunkEmitter(FakeTokenizer(), 0.1, 0.02)
            for k, t in enumerate(range(start, 6)):
                s, w = outs[i][k]
                assert s == ref[i].tokenize_audio({rsid[i]: _audio(i)[0, t * 1600:(t + 1) * 1600]})[rsid[i]]
                assert np.array_equal(w, em.emit(_codes(i, t)))
        assert {k for k, _ in bat.pool.calls} <= {"encode_ragged", "emit_ragged"}
    finally:
        bat.shutdown()
