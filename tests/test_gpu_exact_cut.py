"""GPU (B200): dead-output elimination cuts a window at the exact row its kept outputs need (engine option "exact_cut",
default 1) instead of at multiples of 16 frames (0).  The attention kernels lay a cut window out on the key groups of
the full-window pass, so codes, margins, latents and decoded samples must be bit-identical under both plans and equal
to the full pass sliced."""
import pytest
import torch

import realtime_codec_agent_b200 as pkg

pytestmark = pytest.mark.gpu

SPECS = {"tiny": pkg.TINY_SPEC, "mid": pkg.MID_SPEC, "default": pkg.DEFAULT_SPEC}


@pytest.fixture(scope="module", params=["tiny", "mid", "default"])
def gen(request):
    spec = SPECS[request.param]
    return pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda", max_positions=1024)


@pytest.fixture(scope="module")
def gen_default():
    spec = pkg.DEFAULT_SPEC
    return pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda", max_positions=1024)


def _both_plans(gen, fn):
    try:
        gen.set_option("exact_cut", 1)
        exact = fn()
        gen.set_option("exact_cut", 0)
        aligned = fn()
    finally:
        gen.set_option("exact_cut", 1)
    return exact, aligned


def _qkv(B, F, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((B * F, 3 * d), generator=g, device="cuda").to(torch.bfloat16)


@pytest.mark.parametrize("F_full", [100, 140, 300])
def test_attention_at_every_cut_phase_equals_the_full_window(gen_default, F_full):
    """A window cut to its last Ri rows, laid out with phase (F_full - Ri) mod 16, gives the full pass's kept rows bit for
    bit (v4 and v3; the SIMT kernel is cut-invariant by construction).  F_full = 140 also crosses from the halo kernel
    (full window) to the single-tile one (cut window); at 300 the phase rows push some cut windows of <= 128 rows onto
    two tiles."""
    gen = gen_default
    d, wl, B = gen.spec.d_model, gen.spec.window_left, 3
    qkv = _qkv(B, F_full, d, seed=F_full)
    full = {}
    for impl, p_tmem in ((0, 1), (0, 0), (1, 1)):
        gen.set_option("attn_p_tmem", p_tmem)
        full[impl, p_tmem] = gen.op_attention(qkv, B, F_full, impl=impl).view(B, F_full, d)
    gen.set_option("attn_p_tmem", 1)
    assert torch.equal(full[0, 1], full[0, 0])
    assert (full[0, 1].float() - full[1, 1].float()).abs().max().item() < 0.03
    base = 37 if F_full < 300 else 115   # 115 .. 130: some cut windows fit one tile, some need two once the phase is added
    phases = set()
    for Ri in range(base, base + 16):
        phase, Ro = (F_full - Ri) % 16, Ri - wl
        phases.add(phase)
        cut = qkv.view(B, F_full, 3 * d)[:, F_full - Ri:].reshape(B * Ri, 3 * d).contiguous()
        try:
            for impl, p_tmem in ((0, 1), (0, 0), (1, 1)):
                gen.set_option("attn_p_tmem", p_tmem)
                out = gen.op_attention(cut, B, Ri, impl=impl, out_rows=Ro, phase=phase).view(B, Ro, d)
                assert torch.equal(out, full[impl, p_tmem][:, -Ro:]), f"impl {impl} p_tmem {p_tmem}: Ri {Ri} phase {phase}"
        finally:
            gen.set_option("attn_p_tmem", 1)
    assert phases == set(range(16))


def test_attention_rejects_a_bad_phase(gen_default):
    qkv = _qkv(2, 50, gen_default.spec.d_model, seed=1)
    with pytest.raises(Exception):
        gen_default.op_attention(qkv, 2, 50, out_rows=10, phase=16)


@pytest.mark.parametrize("T", [32000, 27200, 16000, 4800])
def test_encode_exact_cut_matches_aligned_cut_and_full_pass(gen, T):
    """Overlapping strided windows (ld = 1600, the chunked encode); T < 32000 are the warm-up windows of a stream."""
    ld, B = 1600, 24
    wav = pkg.synth_audio((B - 1) * ld + T, seed=11).cuda()
    kw = dict(row_stride=ld, num_windows=B, window_samples=T)
    c_full, m_full, _ = gen.encode(wav, return_margin=True, **kw)
    F = c_full.shape[1]
    for keep in (1, 5, 17):
        (c1, m1, _), (c0, m0, _) = _both_plans(gen, lambda: gen.encode(wav, keep_last_frames=keep, return_margin=True, **kw))
        k = min(keep, F)
        assert torch.equal(c1, c0) and torch.equal(m1, m0), f"keep {keep}"
        assert torch.equal(c1, c_full[:, -k:]) and torch.equal(m1, m_full[:, -k:]), f"keep {keep}"


def test_encode_bench_shape(gen_default):
    """The benchmark's launch shape: 1024 windows of 100 frames over one strided buffer, 5 frames kept."""
    gen = gen_default
    ld, T, B = 1600, 32000, 1024
    wav = pkg.synth_audio((B - 1) * ld + T, seed=5).cuda()
    kw = dict(row_stride=ld, num_windows=B, window_samples=T)
    (c1, m1, _), (c0, m0, _) = _both_plans(gen, lambda: gen.encode(wav, keep_last_frames=5, return_margin=True, **kw))
    assert torch.equal(c1, c0) and torch.equal(m1, m0)
    c_full, m_full, _ = gen.encode(wav[: 127 * ld + T], return_margin=True, row_stride=ld, num_windows=128, window_samples=T)
    assert torch.equal(c1[:128], c_full[:, -5:]) and torch.equal(m1[:128], m_full[:, -5:])


@pytest.mark.parametrize("keep", [320, 1600, 4000])
def test_decode_exact_cut_matches_aligned_cut_and_full_pass(gen, keep):
    B = 6
    wav = pkg.synth_audio((B - 1) * 1600 + 32000, seed=3).cuda()
    codes = gen.encode(wav, row_stride=1600, num_windows=B, window_samples=32000)
    full = gen.decode(codes)
    s1, s0 = _both_plans(gen, lambda: gen.decode(codes, keep_last_samples=keep))
    assert torch.equal(s1, s0)
    assert torch.equal(s1, full[:, -keep:])
