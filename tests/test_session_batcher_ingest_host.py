"""CPU: SessionBatcher.tokenize_audio fed (sr, array) tuples, with a numpy stand-in for the session pool whose push_pcm
converts and resamples on the host (audio_io.pcm_to_float + audio_io.resample) and then encodes as push_audio does.

Checks the routing: tuples that need conversion go to push_pcm (one call per group, mixed rates included), plain arrays
keep today's calls, n_chars follows the resampled length, bad input changes nothing, and every session's strings equal
a lone session fed what AudioTokenizer._prep_audio_for_tokenization makes of the same tuple."""
import threading

import numpy as np
import pytest

from realtime_codec_agent_b200 import audio_io as aio
from realtime_codec_agent_b200 import session_batcher
from realtime_codec_agent_b200.audio_tokenizer import prep_audio_for_tokenization
from tests.test_session_batcher_ragged_host import SR, FakeGen, RaggedFakePool


class IngestFakePool(RaggedFakePool):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.rates = {}

    def set_resampler(self, sr, plan):
        self.calls.append(("set_resampler", sr))
        self.rates[sr] = plan

    def _convert(self, pcm, length):
        out = []
        for sr, x in pcm:
            assert x.dtype in (np.int16, np.float32) and (sr == SR or sr in self.rates)
            rows = x.reshape(-1, x.shape[-1])
            fmt = aio.PCM_S16 if x.dtype == np.int16 else aio.PCM_F32
            p = aio.PcmAudio(sr, rows.shape[0], rows.shape[1], fmt, False, np.ascontiguousarray(rows.T).view(np.uint8).reshape(-1))
            y = aio.resample(aio.pcm_to_float(p, mono=self.channels == 1), sr, SR)
            assert y.shape == (self.channels, length)
            out.append(y)
        return np.stack(out)

    def push_pcm(self, slots, pcm, length, keep_frames):
        chunks = self._convert(pcm, length)
        self.calls.append(("encode_pcm", list(slots)))
        self._check(slots, self.audio, False)
        return np.stack([self._encode(s, x, keep_frames) for s, x in zip(slots, chunks)])

    def push_pcm_ragged(self, slots, pcm, length, keep_frames):
        chunks = self._convert(pcm, length)
        self.calls.append(("encode_pcm_ragged", list(slots)))
        self._check(slots, self.audio, True)
        return np.stack([self._encode(s, x, keep_frames) for s, x in zip(slots, chunks)])


@pytest.fixture(autouse=True)
def fake_pool(monkeypatch):
    monkeypatch.setattr(session_batcher, "SessionPool", IngestFakePool)


def _n_in(sr, n_out):
    if sr == SR:
        return n_out
    plan = aio.resample_plan(sr, SR)
    n = n_out * sr // SR
    while plan.n_out(n) < n_out:
        n += 1
    return n


def _client(i, sr, channels, dtype, secs=4.0):
    x = 0.3 * np.random.default_rng(500 + i).standard_normal((max(channels, 1), int(sr * secs)))
    x = (x * 32767).clip(-32768, 32767).astype(np.int16) if dtype == np.int16 else x.astype(np.float32)
    return x[0] if channels == 0 else x


MIX = [(48000, 0, np.int16), (44100, 2, np.float32), (16000, 0, np.int16), (24000, 0, np.int16), (16000, 0, "bare")]


def _tick(t):
    return {3: 320, 7: 1000}.get(t, 1600)                  # 20 ms and a non-hop-multiple chunk among 0.1 s ones


@pytest.mark.parametrize("ragged", [False, True])
def test_tuples_take_push_pcm_and_equal_lone_sessions(ragged):
    joins = [0, 0, 1, 4, 6]
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=8, ragged=ragged)
    lone = [session_batcher.SessionBatcher(FakeGen(), max_sessions=1) for _ in joins]
    lsid = [b.open_session() for b in lone]
    sig = [_client(i, sr, ch, np.float32 if d == "bare" else d) for i, (sr, ch, d) in enumerate(MIX)]
    sids, pos = {}, [0] * len(joins)
    for t in range(14):
        for i, j in enumerate(joins):
            if t == j:
                sids[i] = bat.open_session()
        req, ref_in = {}, {}
        for i in sids:
            sr, _, d = MIX[i]
            n = _n_in(sr, _tick(t))
            x = sig[i][..., pos[i]:pos[i] + n]
            pos[i] += n
            req[sids[i]] = x if d == "bare" else (sr, x)
            ref_in[i] = prep_audio_for_tokenization(req[sids[i]], SR, 1)   # AudioTokenizer's host preparation
        lens = {bat._sessions[sids[i]].audio_len for i in sids}
        n0 = len(bat.pool.calls)
        got = bat.tokenize_audio(req)
        calls = [k for k, _ in bat.pool.calls[n0:] if k != "set_resampler"]
        if ragged:
            assert calls == ["encode_pcm_ragged"], (t, calls)
        else:
            assert len(calls) == len(lens) and set(calls) <= {"encode_pcm", "encode"}, (t, calls)
        for i in sids:
            want = lone[i].tokenize_audio({lsid[i]: ref_in[i]})[lsid[i]]
            assert got[sids[i]] == want, (t, i)
            assert len(got[sids[i]]) == int(_tick(t) / SR * 50)             # n_chars of the resampled length
    assert sorted(sr for k, sr in bat.pool.calls if k == "set_resampler") == [24000, 44100, 48000]   # once per rate


def test_plain_arrays_make_todays_calls():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=4)
    a, b = bat.open_session(), bat.open_session()
    x = _client(0, SR, 0, np.float32)
    bat.tokenize_audio({a: x[:1600]})
    bat.tokenize_audio({a: x[1600:3200], b: (x[:1600] * 32767).astype(np.int16)})
    bat.tokenize_audio({a: (SR, x[3200:4800]), b: (SR, x[1600:3200])})       # float32 at the codec's rate: nothing to convert
    assert [k for k, _ in bat.pool.calls] == ["encode"] * 5                    # a and b hold contexts of different length


def test_other_dtypes_are_prepared_on_the_host():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=2)
    ref = session_batcher.SessionBatcher(FakeGen(), max_sessions=1)
    a, r = bat.open_session(), ref.open_session()
    x = _client(1, 48000, 2, np.float32).astype(np.float64)
    got = bat.tokenize_audio({a: (48000, x[:, :4800])})
    assert [k for k, _ in bat.pool.calls] == ["encode"]
    assert got[a] == ref.tokenize_audio({r: prep_audio_for_tokenization((48000, x[:, :4800]), SR, 1)})[r]


def test_invalid_input_changes_nothing():
    bat = session_batcher.SessionBatcher(FakeGen(), max_sessions=4, ragged=True)
    a, b = bat.open_session(), bat.open_session()
    x = _client(0, 48000, 0, np.int16)
    bat.tokenize_audio({a: (48000, x[:4800]), b: (48000, x[4800:9600])})

    def snapshot():
        return [bat._sessions[s].audio_len for s in (a, b)], len(bat.pool.calls), set(bat._rates)

    bad = [{a: (48000, x[:4800]), b: (48000, x[:0])},                         # empty
           {a: (48000, x[:4800]), b: (48000, np.zeros(3 * 32001, np.int16))},  # over the capacity once resampled
           {a: (48000, x[:4800]), 99: (48000, x[:4800])},                      # unknown session
           {a: (48000, x[:4800]), b: (96000, x[:9600])}]                         # a ninth client rate
    for sr in (8000, 11025, 22050, 24000, 32000, 44100, 88200):                   # fill the rate table: 48 kHz + 7 = 8
        bat.tokenize_audio({a: (sr, _client(9, sr, 0, np.int16)[:_n_in(sr, 320)])})
    before = snapshot()
    for req in bad:
        with pytest.raises((ValueError, KeyError)):
            bat.tokenize_audio(req)
        assert snapshot() == before, req


def test_threaded_batcher_forwards_tuples():
    bat = session_batcher.ThreadedSessionBatcher(FakeGen(), max_sessions=4, max_wait_ms=1.0, ragged=True)
    ref = [session_batcher.SessionBatcher(FakeGen(), max_sessions=1) for _ in range(3)]
    rates = (48000, 44100, 24000)
    sig = [_client(i, r, 0, np.int16) for i, r in enumerate(rates)]
    try:
        sids = [bat.open_session() for _ in rates]
        rsid = [r.open_session() for r in ref]
        outs, errs = {i: [] for i in range(3)}, []

        def client(i):
            try:
                n = _n_in(rates[i], 1600)
                for t in range(5):
                    outs[i].append(bat.tokenize_audio_one(sids[i], (rates[i], sig[i][t * n:(t + 1) * n])))
            except Exception as ex:                                  # noqa: BLE001
                errs.append(ex)

        ths = [threading.Thread(target=client, args=(i,)) for i in range(3)]
        [th.start() for th in ths]; [th.join(timeout=30) for th in ths]
        assert not errs, errs
        for i, r in enumerate(rates):
            n = _n_in(r, 1600)
            for t in range(5):
                x = prep_audio_for_tokenization((r, sig[i][t * n:(t + 1) * n]), SR, 1)
                assert outs[i][t] == ref[i].tokenize_audio({rsid[i]: x})[rsid[i]], (i, t)
        assert {k for k, _ in bat.pool.calls} <= {"encode_pcm_ragged", "encode_pcm", "set_resampler"}
    finally:
        bat.shutdown()
