"""GPU (B200): pooled live-stream chunks at the client's rate and sample format (mc_pool_push_pcm / _ragged,
SessionBatcher fed (sr, array) tuples).

The device route is held to the kernels that already exist: the staged samples equal DeviceIngest.to_device
(mc_op_pcm_to_f32 + mc_op_resample) on the same bytes bit for bit, and a batcher fed tuples returns exactly what a twin fed
those converted float32 chunks returns.  Against the drop-in AudioTokenizer (float64 host resampler) codes are compared
only where the frame's top-2 margin exceeds what the input difference can move it by."""
import threading

import numpy as np
import pytest
import torch

import realtime_codec_agent_b200 as pkg
from realtime_codec_agent_b200 import audio_io as aio
from realtime_codec_agent_b200._native import MC_POOL_MAX_RESAMPLERS, McError
from realtime_codec_agent_b200.codec_chars import UNICODE_OFFSET_LARGE
from realtime_codec_agent_b200.session_batcher import SessionBatcher, SessionPool, ThreadedSessionBatcher

pytestmark = pytest.mark.gpu
SR = 16000
RATES = (8000, 16000, 22050, 24000, 44100, 48000)
KINDS = ("push_audio", "push_audio_ragged", "push_pcm", "push_pcm_ragged")


@pytest.fixture(scope="module")
def gen():
    return pkg.B200Generator(pkg.TINY_SPEC, pkg.init_random_weights(pkg.TINY_SPEC, seed=0), device="cuda", max_positions=256)


@pytest.fixture(scope="module")
def ingest(gen):
    return aio.DeviceIngest(gen)


class batch_invariant:
    def __init__(self, gen):
        self.gen = gen

    def __enter__(self):
        self.gen.set_option("small_m_split_k", 0)

    def __exit__(self, *exc):
        self.gen.set_option("small_m_split_k", 1)


def _count_calls(pool):
    calls = []
    for name in KINDS:
        f = getattr(pool, name)
        setattr(pool, name, lambda *a, _f=f, _n=name, **k: (calls.append(_n), _f(*a, **k))[1])
    return calls


def _n_in(sr, n_out):
    """The smallest chunk at `sr` that resamples to n_out samples."""
    if sr == SR:
        return n_out
    plan = aio.resample_plan(sr, SR)
    n = n_out * sr // SR
    while plan.n_out(n) < n_out:
        n += 1
    assert plan.n_out(n) == n_out
    return n


def _client(i, sr, channels, secs, dtype):
    """A client's signal at its own rate: [T] (channels = 0) or [channels, T], int16 or float32."""
    n = int(sr * secs)
    x = np.stack([pkg.synth_audio(n, file_id=200 + i, channel=c).numpy() for c in range(max(channels, 1))])
    x = 0.8 * x / max(np.abs(x).max(), 1e-6)
    x = (x * 32767).astype(np.int16) if dtype == np.int16 else x.astype(np.float32)
    return x[0] if channels == 0 else x


def _device_ref(ingest, sr, x, mono):
    """DeviceIngest.to_device of the same chunk: the existing kernels on an interleaved payload."""
    rows = x.reshape(-1, x.shape[-1])
    fmt = aio.PCM_S16 if x.dtype == np.int16 else aio.PCM_F32
    pcm = aio.PcmAudio(sr, rows.shape[0], rows.shape[1], fmt, False, np.ascontiguousarray(rows.T).view(np.uint8).reshape(-1))
    return ingest.to_device(pcm, mono=mono).cpu().numpy()


@pytest.mark.parametrize("sr", RATES)
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
@pytest.mark.parametrize("layout", ["mono", "stereo_to_mono", "stereo"])
def test_staging_is_bit_exact(gen, ingest, sr, dtype, layout):
    C = 2 if layout == "stereo" else 1
    pool = SessionPool(gen, C, 32000, 2)
    if sr != SR:
        pool.set_resampler(sr, aio.resample_plan(sr, SR))
    ch = {"mono": 0, "stereo_to_mono": 2, "stereo": 2}[layout]
    sig = _client(1, sr, ch, 3.0, dtype)
    prev = (0.1 * np.random.default_rng(3).standard_normal((1, C, 1600))).astype(np.float32)
    pool.push_audio([1], prev, 0)
    ctx = prev[0]
    pos = 0
    for n_out in (1600, 320, 1000):                                # 0.1 s, 20 ms and a length that is no hop multiple
        n = _n_in(sr, n_out)
        x = sig[..., pos:pos + n]
        pos += n
        pool.push_pcm([1], [(sr, x)], n_out, 0)
        want = _device_ref(ingest, sr, x, mono=C == 1)
        ctx = np.concatenate([ctx, want], axis=1)[:, -32000:]
        got = pool.read_audio(1, ctx.shape[1])
        assert got.shape == ctx.shape and np.array_equal(got.view(np.uint32), ctx.view(np.uint32)), (sr, n_out)
        host = x.astype(np.float32) / 32768.0 if dtype == np.int16 else x
        if C == 1 and host.ndim > 1:
            host = np.mean(host, axis=0)
        host = aio.resample(host, sr, SR).reshape(C, -1)
        err = np.abs(want - host).max()
        assert err < 3e-6, (sr, n_out, err)


def _mix():
    """Session i: (rate, channels, dtype) -- 0 channels: a [T] array; bare: a float32 array at the codec's rate."""
    return [(48000, 0, np.int16), (44100, 2, np.float32), (16000, 0, np.int16), (24000, 2, np.int16), ("bare", 0, np.float32),
            (22050, 0, np.int16), (8000, 0, np.float32)]


def _tick_len(t):
    return 320 if t % 5 == 4 else 1600                              # 20 ms ticks among 0.1 s ones


def _drive(gen, ingest, ragged, joins, ticks, C=1):
    bat = SessionBatcher(gen, num_channels=C, max_sessions=8, ragged=ragged)
    twin = SessionBatcher(gen, num_channels=C, max_sessions=8, ragged=ragged)
    calls = _count_calls(bat.pool)
    mix = _mix()[:len(joins)] if C == 1 else [(48000, 2, np.int16), (44100, 2, np.float32), (16000, 2, np.int16)][:len(joins)]
    sig = [_client(i, SR if r == "bare" else r, ch, 6.0, d) for i, (r, ch, d) in enumerate(mix)]
    pos = [0] * len(joins)
    sids, tsids = {}, {}
    for t in range(ticks):
        for i, j in enumerate(joins):
            if t == j:
                sids[i], tsids[i] = bat.open_session(), twin.open_session()
        n_out = _tick_len(t)
        req, treq = {}, {}
        for i in sids:
            r, ch, d = mix[i]
            n = n_out if r == "bare" else _n_in(r, n_out)
            x = sig[i][..., pos[i]:pos[i] + n]
            pos[i] += n
            if r == "bare":
                req[sids[i]], treq[tsids[i]] = x, x
            else:
                req[sids[i]] = (r, x)
                treq[tsids[i]] = _device_ref(ingest, r, x, mono=C == 1)
        lens = {bat._sessions[sids[i]].audio_len for i in sids}
        del calls[:]
        got = bat.tokenize_audio(req)
        want = twin.tokenize_audio(treq)
        for i in sids:
            assert got[sids[i]] == want[tsids[i]], (ragged, t, i)
        if ragged:                                                  # one engine call per tick
            assert calls == ["push_pcm_ragged"], (t, calls)
        else:                                                       # one per context length; a group of bare arrays only: today's call
            assert len(calls) == len(lens) and set(calls) <= {"push_pcm", "push_audio"}, (t, calls)
    return bat


@pytest.mark.parametrize("ragged", [False, True])
def test_codes_equal_the_converted_twin(gen, ingest, ragged):
    with batch_invariant(gen):
        _drive(gen, ingest, ragged, [0, 0, 1, 3, 4, 8, 11], 26)


def test_codes_equal_the_converted_twin_stereo_pool(gen, ingest):
    with batch_invariant(gen):
        _drive(gen, ingest, True, [0, 2, 5], 18, C=2)


def test_codes_equal_the_converted_twin_default_spec(ingest):
    spec = pkg.DEFAULT_SPEC
    g = pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda")
    with batch_invariant(g):
        _drive(g, aio.DeviceIngest(g), True, [0, 1, 3, 6], 16)


def test_against_the_drop_in_tokenizer(gen):
    """Lone AudioTokenizers resample on the host in float64.  A frame's code must agree wherever the device window's top-2
    margin exceeds the bound on how far the input difference can move it: the squared distances to codewords e differ by
    ||z'||^2 - ||z||^2 - 2<z' - z, e>, so the best code cannot change while margin > 2 ||z' - z|| max_k ||e_k - e_best||."""
    cb = gen.quantizer.codebook_proj(gen.quantizer.codebook.weight).float()
    joins, ticks = [0, 0, 2, 4], 16
    mix = [(48000, 0, np.int16), (44100, 2, np.float32), (24000, 0, np.int16), (22050, 0, np.int16)]
    with batch_invariant(gen):
        bat = SessionBatcher(gen, max_sessions=8, ragged=True)
        sig = [_client(i, r, ch, 4.0, d) for i, (r, ch, d) in enumerate(mix)]
        pos, sids, toks = [0] * len(joins), {}, {}
        same = total = asserted = 0
        for t in range(ticks):
            for i, j in enumerate(joins):
                if t == j:
                    sids[i] = bat.open_session()
                    toks[i] = pkg.AudioTokenizer(codec_model=gen, device="cuda")
            n_out = _tick_len(t)
            req = {}
            for i in sids:
                r = mix[i][0]
                n = _n_in(r, n_out)
                req[sids[i]] = (r, sig[i][..., pos[i]:pos[i] + n])
                pos[i] += n
            got = bat.tokenize_audio(req)
            for i in sids:
                ref = toks[i].tokenize_audio(req[sids[i]])
                k = len(ref)
                a = np.array([ord(c) - UNICODE_OFFSET_LARGE for c in got[sids[i]]])
                b = np.array([ord(c) - UNICODE_OFFSET_LARGE for c in ref])
                slot = bat._sessions[sids[i]].slot
                dev_win = bat.pool.read_audio(slot, bat.pool.context_len(slot)[0])
                host_win = np.ascontiguousarray(toks[i].tokenize_context, dtype=np.float32)
                assert dev_win.shape == host_win.shape
                _, m, z = gen.encode(torch.from_numpy(dev_win).cuda(), keep_last_frames=k, return_margin=True, return_latents=True)
                _, _, z2 = gen.encode(torch.from_numpy(host_win).cuda(), keep_last_frames=k, return_latents=True)
                z, z2, m = z[0, -k:], z2[0, -k:], m[0]
                best = cb[torch.from_numpy(a).cuda()]
                reach = torch.stack([(cb - e).norm(dim=-1).max() for e in best])
                bound = 2 * (z2 - z).norm(dim=-1) * reach + 1e-3       # + slack for the fp32 distances themselves
                clear = (m > bound).cpu().numpy()
                same += int((a == b).sum()); total += k; asserted += int(clear.sum())
                assert np.array_equal(a[clear], b[clear]), (t, i)
        print(f"[pool ingest] device vs host-float64 resampling: {same}/{total} codes equal; "
              f"{asserted} frames above their margin bound asserted equal")


def _state(bat, sids):
    return [(bat.pool.context_len(bat._sessions[s].slot), bat._sessions[s].audio_len) for s in sids]


def _raw_push(pool, slots, pcm, length, keep, ragged=False, **override):
    """mc_pool_push_pcm(_ragged) with the item table patched after SessionPool builds it -> the C return code."""
    items, payload = SessionPool._pcm_items(pcm)
    for k, v in override.items():
        items[k] = v
    slots = np.ascontiguousarray(slots, dtype=np.int32)
    out = np.empty(len(slots) * pool.channels * pool.cap_frames, np.int64)
    lib = pool.gen._lib
    if ragged:
        return lib.mc_pool_push_pcm_ragged(pool._p, slots.ctypes.data, len(slots), items.ctypes.data, payload.ctypes.data, length,
                                           keep, out.ctypes.data, pool.gen._stream())
    return lib.mc_pool_push_pcm(pool._p, slots.ctypes.data, len(slots), items.ctypes.data, payload.ctypes.data, length, keep,
                                out.ctypes.data, None, pool.gen._stream())


def test_errors_change_nothing_and_graphs_stay(gen):
    MC_ERR_ARG = -1
    pool = SessionPool(gen, 1, 32000, 4)
    pool.set_resampler(48000, aio.resample_plan(48000, SR))
    x48 = _client(0, 48000, 0, 1.0, np.int16)
    pool.push_pcm([0, 1], [(48000, x48[:4800]), (48000, x48[4800:9600])], 1600, 0)
    pool.push_pcm([2], [(48000, x48[:960])], 320, 0)

    def snapshot():
        return [pool.context_len(s) for s in range(4)], pool.read_audio(0, 1600), pool.read_audio(2, 320)

    before = snapshot()
    one = [(48000, x48[:4800])]
    bad = [
        dict(slots=[0], pcm=[(44100, x48[:4410])], length=1600, keep=0),                             # unknown rate
        dict(slots=[0], pcm=one, length=1600, keep=0, format=aio.PCM_S32),                           # format
        dict(slots=[0], pcm=[(48000, np.zeros((9, 4800), np.int16))], length=1600, keep=0),          # 9 channels, mono pool
        dict(slots=[0], pcm=one, length=1601, keep=0),                                               # resampled length
        dict(slots=[0], pcm=[(48000, np.zeros(3 * 32001, np.int16))], length=32001, keep=0),         # over the capacity
        dict(slots=[0], pcm=one, length=1600, keep=0, n_in=0),                                       # empty chunk
        dict(slots=[0, 0], pcm=one * 2, length=1600, keep=0),                                        # slot twice
        dict(slots=[0], pcm=one, length=1600, keep=6, ragged=True),                                  # keep_frames > ceil(len/hop)
        dict(slots=[0, 2], pcm=one * 2, length=1600, keep=0, ragged=True),                           # keep_frames 0
    ]
    if gen.spec.window_right != 0:
        bad.append(dict(slots=[0, 2], pcm=one * 2, length=1600, keep=5, ragged=True))               # causal rule
    for kw in bad:
        assert _raw_push(pool, **kw) == MC_ERR_ARG, kw
        after = snapshot()
        assert after[0] == before[0] and np.array_equal(after[1], before[1]) and np.array_equal(after[2], before[2]), kw
    with pytest.raises(McError):
        pool.read_audio(3, 10)                                                                       # empty context
    pool.reserve_pcm(4800, 2)
    assert _raw_push(pool, [0], [(48000, np.zeros((3, 4800), np.int16))], 1600, 0) == MC_ERR_ARG    # over the reserved staging
    assert _raw_push(pool, [0], [(48000, np.zeros(4803, np.int16))], 1601, 0) == MC_ERR_ARG
    assert snapshot()[0] == before[0]
    stereo = SessionPool(gen, 2, 32000, 2)
    stereo.set_resampler(48000, aio.resample_plan(48000, SR))
    assert _raw_push(stereo, [0], one, 1600, 0) == MC_ERR_ARG                                       # 1 channel, C = 2 pool
    assert stereo.context_len(0) == (0, 0)
    others = (8000, 11025, 22050, 24000, 32000, 44100, 88200)
    assert len(others) + 1 == MC_POOL_MAX_RESAMPLERS
    for sr in others:
        pool.set_resampler(sr, aio.resample_plan(sr, SR))
    with pytest.raises(McError):                                                                     # a ninth rate
        pool.set_resampler(96000, aio.resample_plan(96000, SR))
    with pytest.raises(McError):                                                                     # another rate's plan
        pool.set_resampler(44100, aio.resample_plan(48000, SR))
    # steady ticks replay captured graphs: 50 of them add none
    bat = SessionBatcher(gen, max_sessions=4, ragged=True)
    rates = (48000, 44100, 16000)
    sig = [_client(i, r, 0, 8.0, np.int16) for i, r in enumerate(rates)]
    sids = [bat.open_session() for _ in rates]
    for t in range(80):
        if t == 30:
            counts = bat.pool.graph_count()
        bat.tokenize_audio({s: (r, x[t * _n_in(r, 1600):(t + 1) * _n_in(r, 1600)]) for s, r, x in zip(sids, rates, sig)})
    assert bat.pool.graph_count() == counts


def test_batcher_rejects_before_state_changes(gen):
    bat = SessionBatcher(gen, max_sessions=4, ragged=True)
    a, b = bat.open_session(), bat.open_session()
    x = _client(0, 48000, 0, 1.0, np.int16)
    bat.tokenize_audio({a: (48000, x[:4800]), b: (44100, _client(1, 44100, 0, 1.0, np.int16)[:4410])})
    before = _state(bat, (a, b))
    for req in ({a: (48000, x[:4800]), b: (48000, np.zeros(0, np.int16))},
                {a: (48000, x[:4800]), b: (48000, np.zeros(3 * 32001, np.int16))},
                {a: (48000, x[:4800]), 99: (48000, x[:4800])}):
        with pytest.raises((ValueError, KeyError)):
            bat.tokenize_audio(req)
        assert _state(bat, (a, b)) == before


def test_threaded_batcher_takes_tuples(gen, ingest):
    with batch_invariant(gen):
        bat = ThreadedSessionBatcher(gen, max_sessions=4, max_wait_ms=1.0, ragged=True)
        ref = [SessionBatcher(gen, max_sessions=1) for _ in range(3)]
        rates = (48000, 44100, 24000)
        sig = [_client(i, r, 0, 2.0, np.int16) for i, r in enumerate(rates)]
        try:
            sids = [bat.open_session() for _ in range(3)]
            rsid = [r.open_session() for r in ref]
            outs, errs = {i: [] for i in range(3)}, []

            def client(i):
                try:
                    n = _n_in(rates[i], 1600)
                    for t in range(8):
                        outs[i].append(bat.tokenize_audio_one(sids[i], (rates[i], sig[i][t * n:(t + 1) * n])))
                except Exception as ex:                                   # noqa: BLE001
                    errs.append(ex)

            ths = [threading.Thread(target=client, args=(i,)) for i in range(3)]
            [th.start() for th in ths]; [th.join(timeout=60) for th in ths]
            assert not errs, errs
            for i in range(3):
                n = _n_in(rates[i], 1600)
                for t in range(8):
                    x = _device_ref(ingest, rates[i], sig[i][t * n:(t + 1) * n], mono=True)[0]
                    assert outs[i][t] == ref[i].tokenize_audio({rsid[i]: x})[rsid[i]], (i, t)
        finally:
            bat.shutdown()
