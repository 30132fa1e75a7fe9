"""The kernel variants that specs other than the three shipped ones select, against float64 references.

`MagiCodecSpec` is meant to be overridden (a checkpoint carries its own spec), but the shipped specs share one shape:
window (32, 0), strides (4, 4, 4, 5), first conv width 32.  This module runs what other accepted specs select:
`conv_first_kernel<16>` (first stride 8), the last transposed conv at stride 8 and with a weight table over 48 KB,
stride-1 layers, the generic RMSNorm (d = 192, 384, 768), the SIMT attention (wide or look-ahead windows), the tcgen05
attention at window_left != 32, zero-layer stacks and a VQ over 1 or 3 codebook tiles.

  1. the attention op against a float64 masked softmax over the same bf16 inputs;
  2. each conv stack alone (zero-layer specs) against the float64 oracle;
  3. the whole network on a small spec matrix: oracle bars of tests/test_gpu_parity.py, plus the exactness properties
     the engine promises (keep_last_*, shared stem, batching, stream sessions, exact cut);
  4. every spec rule: validate() and mc_create refuse the same specs, at construction.

Widths stay small so the CPU oracle is quick; no case is dropped for time.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import realtime_codec_agent_b200 as pkg
from oracle.magicodec_oracle import OracleGenerator
from realtime_codec_agent_b200 import _native as nat
from realtime_codec_agent_b200.generator import mc_spec_struct
from tests.test_gpu_parity import EPS_MARGIN, NEAR_TIE_MAX, SNR_MIN_DB, WAV_TOL, Z_TOL

Spec = pkg.MagiCodecSpec


def _small(**kw):
    base = dict(conv_channels=(32, 64, 64), conv_strides=(4, 4, 4, 5), d_model=128, n_heads=2, ffn_dim=256,
                enc_layers=0, dec_layers=0, window_left=32, window_right=0, codebook_size=256)
    base.update(kw)
    return Spec(**base)


def tconv_margin_frames(spec):
    """Frames a decode cut from a longer window needs before its first kept sample (engine.cu, tconv_margin_frames):
    transposed conv i reads input steps t-1 and t, so the zero pad of a cut window spoils L = sum_i hop / prod_{j<i} ds[j]
    samples (ds: the decoder strides)."""
    hop, look_back, step = spec.hop, 0, spec.hop
    for s in spec.dec_strides:
        look_back += step
        step //= s
    return -(-look_back // hop)


_ENGINES = {}


def _engine(spec, seed=0):
    """One engine (and its fp32 master weights) per spec for the whole module."""
    key = (spec, seed)
    if key not in _ENGINES:
        w = pkg.init_random_weights(spec, seed=seed)
        _ENGINES[key] = (pkg.B200Generator(spec, w, device="cuda", max_positions=1024), w)
    return _ENGINES[key]


@pytest.fixture(scope="module", autouse=True)
def _release_engines():
    yield
    _ENGINES.clear()


def _oracle64(spec, w):
    return OracleGenerator(spec, w).double()


def _snr_db(ref, got):
    noise = (ref.double() - got.double()).pow(2).sum().item()
    return 10.0 * np.log10(ref.double().pow(2).sum().item() / max(noise, 1e-30))


# ============================================================================ 1. attention op
def attention_ref64(qkv, B, F, H, wl, wr, out_rows):
    """float64 softmax over keys j in [i - wl, i + wr] ∩ [0, F), scale 0.125, on the same bf16 inputs.  Returns the
    output rows [B*out_rows, H*64] and, per element, sum_j p_j |v_j| (the bound on the error of bf16 probabilities)."""
    d = H * 64
    x = qkv.double().cpu().view(B, F, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)   # [B,H,F,64]
    i = torch.arange(F)[:, None]
    j = torch.arange(F)[None, :]
    allowed = (j >= i - wl) & (j <= i + wr)
    s = (q @ k.transpose(-1, -2)) * 0.125
    s = s.masked_fill(~allowed, float("-inf"))
    p = torch.softmax(s, dim=-1)
    o = (p @ v).transpose(1, 2)[:, F - out_rows:].reshape(B * out_rows, d)
    pv_abs = (p @ v.abs()).transpose(1, 2)[:, F - out_rows:].reshape(B * out_rows, d)
    return o, pv_abs


def assert_attention_close(got, ref, pv_abs, what):
    """Tolerance: |got - ref| <= 2^-8 |ref| + 2^-8 sum_j p_j |v_j| + 2^-16.
    The first term is one bf16 ulp of the output (the store rounds to nearest: half an ulp, 2^-9 relative, plus fp32
    accumulation far below it).  The second is the tcgen05 kernels' P.V product, which consumes the probabilities in bf16
    (each p_j off by at most 2^-9 relative, so the sum moves by at most 2^-9 sum_j p_j |v_j|), doubled for the fp32 row
    sum taken from unrounded values.  The last term covers outputs that round to (near) zero.  A reference whose window is
    one key off moves outputs by about p_j |v_j - o| ~ 1/span, tens of ulps."""
    err = (got.double().cpu() - ref).abs()
    tol = ref.abs() * 2.0 ** -8 + pv_abs * 2.0 ** -8 + 2.0 ** -16
    bad = err > tol
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {err.numel()} outside the bf16 bound, "
                           f"max err {err.max().item():.3g}, max err/tol {(err / tol).max().item():.2f}")


def _qkv(B, F, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn((B * F, 3 * d), generator=g, device="cuda") * 1.5).to(torch.bfloat16)


TC_WINDOWS = [0, 1, 7, 31, 32]
TC_FRAMES = [1, 37, 100, 128, 129, 300]


@pytest.mark.gpu
@pytest.mark.parametrize("wl", TC_WINDOWS)
def test_tcgen05_attention_against_float64(wl):
    """v4 (P in tensor memory) and v3 (attn_p_tmem = 0) at window (wl, 0): one tile (F <= 128) and the halo kernel
    (F = 129, 300); full windows and cut ones (out_rows < F) at several phases.  The SIMT cross-check runs the same
    cases."""
    gen, _ = _engine(_small(window_left=wl))
    d, H, B = 128, 2, 3
    for F in TC_FRAMES:
        qkv = _qkv(B, F, d, seed=100 * wl + F)
        cuts = [(F, 0)] + [(r, ph) for r, ph in ((F - 1, 1), (F // 2, 7), (max(1, F // 3), 15), (1, 3)) if 1 <= r < F]
        for out_rows, phase in cuts:
            ref, pv_abs = attention_ref64(qkv, B, F, H, wl, 0, out_rows)
            for impl, p_tmem in ((0, 1), (0, 0), (1, 1)):
                gen.set_option("attn_p_tmem", p_tmem)
                try:
                    out = gen.op_attention(qkv, B, F, impl=impl, out_rows=out_rows, phase=phase)
                finally:
                    gen.set_option("attn_p_tmem", 1)
                assert_attention_close(out, ref, pv_abs, f"wl {wl} F {F} out_rows {out_rows} phase {phase} impl {impl}/{p_tmem}")


SIMT_WINDOWS = [(wl, wr) for wl in (33, 64, 96) for wr in (0, 1, 8, 32)] + [(0, 32)]


@pytest.mark.gpu
@pytest.mark.parametrize("wl,wr", SIMT_WINDOWS)
def test_simt_attention_against_float64(wl, wr):
    """Windows the tcgen05 kernels are not built for (window_left > 32 or window_right > 0) run the SIMT kernel in
    production (impl 0 selects it); full windows and kept tails, F from 1 to past the widest span."""
    gen, _ = _engine(_small(window_left=wl, window_right=wr))
    d, H, B = 128, 2, 2
    for F in (1, 20, 130, 200):
        qkv = _qkv(B, F, d, seed=1000 + 7 * wl + wr + F)
        for out_rows in sorted({F, max(1, F - 33), 1}):
            ref, pv_abs = attention_ref64(qkv, B, F, H, wl, wr, out_rows)
            out = gen.op_attention(qkv, B, F, out_rows=out_rows)
            assert_attention_close(out, ref, pv_abs, f"window ({wl}, {wr}) F {F} out_rows {out_rows}")


# ============================================================================ 2. conv stacks alone
CONV_STACKS = {
    "4445_control": dict(conv_strides=(4, 4, 4, 5), conv_channels=(32, 128, 256)),
    "885_c64": dict(conv_strides=(8, 8, 5), conv_channels=(64, 128)),        # conv_first<16>, last tconv at stride 8
    "885_c8": dict(conv_strides=(8, 8, 5), conv_channels=(8, 128)),          # first conv C0 = 8: one channel group
    "4451_stride1": dict(conv_strides=(4, 4, 5, 1), conv_channels=(32, 64, 64)),
    "4445_c256": dict(conv_strides=(4, 4, 4, 5), conv_channels=(256, 128, 128)),
    "845_c1024": dict(conv_strides=(8, 4, 5), conv_channels=(1024, 128)),    # last tconv: 64 KB weight table
}


def _stack_spec(name):
    return _small(**CONV_STACKS[name])


def assert_latents_close(z, z_ref, what):
    """Encoder latents: max |z - z_ref| <= Z_TOL (tests/test_gpu_parity.py: bf16 products with fp32 accumulation against
    the oracle measured 0.031 - 0.035 on the shipped specs with 2 - 8 transformer layers; the conv stack alone carries
    less of that error), and the rms error within 2 % of the latent rms (bf16 rounding of every conv output and weight,
    about 2^-9 relative each, over at most five roundings in a row)."""
    err = (z.double().cpu() - z_ref.double())
    rel_rms = err.pow(2).mean().sqrt().item() / z_ref.double().pow(2).mean().sqrt().item()
    assert err.abs().max().item() <= Z_TOL and rel_rms <= 0.02, f"{what}: max {err.abs().max().item():.4f} rel rms {rel_rms:.4f}"


def assert_audio_close(rec, ref, what):
    """Decoded audio: SNR >= SNR_MIN_DB and max |error| <= WAV_TOL x peak (tests/test_gpu_parity.py)."""
    snr = _snr_db(ref, rec.cpu())
    max_rel = (rec.double().cpu() - ref.double()).abs().max().item() / ref.double().abs().max().item()
    assert snr >= SNR_MIN_DB and max_rel <= WAV_TOL, f"{what}: snr {snr:.1f} dB, max err {max_rel:.4f} x peak"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONV_STACKS))
def test_encoder_conv_stack_against_float64(name):
    """enc_layers = 0: the latents are proj(norm_f(conv stack)).  Lengths 1 sample, hop - 1, hop + 1 and a batch of
    strided windows (the shared stem) of several frames."""
    spec = _stack_spec(name)
    gen, w = _engine(spec)
    oracle = _oracle64(spec, w)
    hop = spec.hop
    wav = pkg.synth_audio(40 * hop + 3 * hop, seed=21)
    cases = [wav[None, :1], wav[None, :hop - 1], torch.stack([wav[:hop + 1], wav[hop:2 * hop + 1]])]
    for x in cases:
        _, _, z = gen.encode(x.cuda(), return_latents=True)
        with torch.no_grad():
            z_ref = oracle.encoder(oracle.pad_audio(x.double()))
        assert z.shape == z_ref.shape
        assert_latents_close(z, z_ref, f"{name} T {x.shape[1]}")
    ld, T, B = hop, 40 * hop, 4
    _, _, z = gen.encode(wav.cuda(), row_stride=ld, num_windows=B, window_samples=T, return_latents=True)
    mat = torch.stack([wav[b * ld: b * ld + T] for b in range(B)])
    with torch.no_grad():
        z_ref = oracle.encoder(mat.double())
    assert_latents_close(z, z_ref, f"{name} strided windows")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONV_STACKS))
def test_decoder_conv_stack_against_float64(name):
    """dec_layers = 0: the waveform is embed -> in_proj -> norm_f -> the transposed-conv stack.  1, 2 and 40 frames."""
    spec = _stack_spec(name)
    gen, w = _engine(spec)
    oracle = _oracle64(spec, w)
    g = torch.Generator().manual_seed(5)
    for F in (1, 2, 40):
        codes = torch.randint(0, spec.codebook_size, (2, F), generator=g)
        rec = gen.decode(codes.cuda())
        with torch.no_grad():
            ref = oracle.decoder(torch.nn.functional.embedding(codes, oracle.quantizer.projected()))[:, 0]
        assert rec.shape == ref.shape
        assert_audio_close(rec, ref, f"{name} F {F}")


def test_tconv_margin_makes_a_cut_decode_exact_in_float64():
    """CPU, float64 oracle with a zero-layer decoder (the transformer is per row, so a cut window is exact iff the convs
    are): decoding the last ceil(keep / hop) + margin frames gives the full decode's last `keep` samples.  With the
    former fixed margin of 2 frames, specs whose late encoder strides are small come out wrong."""
    for strides, channels, margin in (((4, 4, 4, 5), (32, 128, 256), 2), ((4, 4, 5, 1), (32, 64, 64), 3),
                                      ((8, 8, 5), (64, 128), 2), ((4, 4, 1, 1), (32, 64, 64), 4)):
        spec = _small(conv_strides=strides, conv_channels=channels)
        assert tconv_margin_frames(spec) == margin
        oracle = _oracle64(spec, pkg.init_random_weights(spec, seed=0))
        hop, F = spec.hop, 12
        codes = torch.randint(0, spec.codebook_size, (1, F), generator=torch.Generator().manual_seed(2))
        emb = torch.nn.functional.embedding(codes, oracle.quantizer.projected())
        with torch.no_grad():
            full = oracle.decoder(emb)[0, 0]
            worst_fixed = 0.0
            for keep in range(1, 6 * hop + 1, max(1, hop // 16)):
                kf = -(-keep // hop)
                cut = oracle.decoder(emb[:, F - min(F, kf + margin):])[0, 0]
                assert torch.allclose(cut[-keep:], full[-keep:], rtol=0, atol=1e-12), (strides, keep)
                fixed = oracle.decoder(emb[:, F - min(F, kf + 2):])[0, 0]
                worst_fixed = max(worst_fixed, (fixed[-keep:] - full[-keep:]).abs().max().item())
        assert (worst_fixed > 1e-3) == (margin > 2), (strides, worst_fixed)


# ============================================================================ 3. whole network, spec matrix
MATRIX = {
    "d128_w00_s4451": _small(d_model=128, n_heads=2, ffn_dim=192, window_left=0, enc_layers=1, dec_layers=1,
                             conv_strides=(4, 4, 5, 1), conv_channels=(32, 64, 64), codebook_size=256),
    "d192_w80_s885": _small(d_model=192, n_heads=3, ffn_dim=320, window_left=8, enc_layers=2, dec_layers=1,
                            conv_strides=(8, 8, 5), conv_channels=(64, 128), codebook_size=768),
    "d384_w640_s4445": _small(d_model=384, n_heads=6, ffn_dim=448, window_left=64, enc_layers=1, dec_layers=2,
                              conv_strides=(4, 4, 4, 5), conv_channels=(32, 128, 256), codebook_size=4096),
    "d768_w248_s885c8": _small(d_model=768, n_heads=12, ffn_dim=1088, window_left=24, window_right=8, enc_layers=1,
                               dec_layers=1, conv_strides=(8, 8, 5), conv_channels=(8, 128), codebook_size=1024),
    "d128_w9632_c256": _small(d_model=128, n_heads=2, ffn_dim=320, window_left=96, window_right=32, enc_layers=2,
                              dec_layers=2, conv_strides=(4, 4, 4, 5), conv_channels=(256, 128, 128), codebook_size=2048),
    "d192_w320_s4451": _small(d_model=192, n_heads=3, ffn_dim=192, window_left=32, enc_layers=2, dec_layers=2,
                              conv_strides=(4, 4, 5, 1), conv_channels=(32, 64, 64), codebook_size=512),
    "d384_w032_s845c1024": _small(d_model=384, n_heads=6, ffn_dim=576, window_left=0, window_right=32, enc_layers=1,
                                  dec_layers=1, conv_strides=(8, 4, 5), conv_channels=(1024, 128), codebook_size=256),
}


@pytest.fixture(scope="module", params=list(MATRIX))
def matrix_case(request):
    spec = MATRIX[request.param]
    gen, w = _engine(spec)
    return request.param, spec, gen, w


def _audio(spec, frames, n, seed):
    return torch.stack([pkg.synth_audio(frames * spec.hop, seed=seed, file_id=i) for i in range(n)])


@pytest.mark.gpu
def test_matrix_against_the_oracle(matrix_case):
    """Encode latents and codes (margin-qualified) and decoded audio against the float64 oracle, with the bars of
    tests/test_gpu_parity.py."""
    name, spec, gen, w = matrix_case
    oracle = _oracle64(spec, w)
    wav = _audio(spec, 60, 4, seed=31)
    codes, _, z = gen.encode(wav.cuda(), return_margin=True, return_latents=True)
    with torch.no_grad():
        z_ref = oracle.encoder(oracle.pad_audio(wav.double()))
        z_q, idx_ref, margin = oracle.quantizer.inference(z_ref, return_margin=True)
        rec_ref = oracle.decoder(z_q.double())[:, 0]
    z_err = (z.double().cpu() - z_ref).abs().max().item()
    clear = margin > EPS_MARGIN
    assert z_err <= Z_TOL, f"{name}: max |dz| {z_err:.4f}"
    assert torch.equal(codes.cpu()[clear], idx_ref[clear]), name
    assert 1 - clear.float().mean().item() <= NEAR_TIE_MAX, name
    rec = gen.decode(idx_ref.cuda())
    assert_audio_close(rec, rec_ref, name)


def _each_plan(gen, key, values, fn):
    outs = []
    try:
        for v in values:
            gen.set_option(key, v)
            outs.append(fn())
    finally:
        gen.set_option(key, values[0])
    return outs


@pytest.mark.gpu
def test_matrix_keep_last_and_exact_cut(matrix_case):
    """keep_last_frames and keep_last_samples equal slicing the full result, under the exact cut (1) and the 16-frame
    plan (0).  keep_last_samples k in {1, hop - 1, hop, hop + 1, 5 hop + 17}: a margin too small for the strides spoils
    the first kept samples."""
    name, spec, gen, w = matrix_case
    hop = spec.hop
    wav = _audio(spec, 40, 3, seed=41).cuda()
    full = gen.encode(wav)
    for keep in (1, 5, 17):
        a, b = _each_plan(gen, "exact_cut", (1, 0), lambda: gen.encode(wav, keep_last_frames=keep))
        assert torch.equal(a, full[:, -keep:]) and torch.equal(b, a), f"{name} keep_last_frames {keep}"
    codes = torch.randint(0, spec.codebook_size, (2, 30), generator=torch.Generator().manual_seed(4)).cuda()
    rec = gen.decode(codes)
    for k in (1, hop - 1, hop, hop + 1, 5 * hop + 17):
        a, b = _each_plan(gen, "exact_cut", (1, 0), lambda: gen.decode(codes, keep_last_samples=k))
        assert torch.equal(a, rec[:, -k:]), f"{name} keep_last_samples {k}: max err {(a - rec[:, -k:]).abs().max().item():.3g}"
        assert torch.equal(b, a), f"{name} keep_last_samples {k}, exact_cut 0"


@pytest.mark.gpu
def test_matrix_shared_stem_and_batching(matrix_case):
    """The shared conv stem equals per-window stacks, and a batch of windows equals its windows run one at a time."""
    name, spec, gen, w = matrix_case
    hop = spec.hop
    ld, T, B = 2 * hop, 40 * hop, 10
    wav = pkg.synth_audio((B - 1) * ld + T, seed=51).cuda()
    kw = dict(row_stride=ld, num_windows=B, window_samples=T, return_margin=True, return_latents=True)
    (c1, m1, z1), (c0, m0, z0) = _each_plan(gen, "shared_stem", (1, 0), lambda: gen.encode(wav, **kw))
    assert torch.equal(z1, z0) and torch.equal(c1, c0) and torch.equal(m1, m0), name
    mat = torch.stack([wav[b * ld: b * ld + T] for b in range(B)])
    assert torch.equal(gen.encode(mat), c0), name
    single = torch.cat([gen.encode(mat[i:i + 1]) for i in range(B)])
    assert torch.equal(single, c0), name
    dec_all = gen.decode(c0[:4])
    dec_one = torch.cat([gen.decode(c0[i:i + 1]) for i in range(4)])
    assert torch.equal(dec_all, dec_one), name


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 2])
def test_matrix_stream_session_equals_stateless_calls(matrix_case, mode):
    """A stream session (device-resident context, graph replay) equals re-sending the whole window, for encode and
    decode, with the batch-invariant kernels (small_m_split_k 0) and the split-K few-rows kernels on both sides (2)."""
    name, spec, gen, w = matrix_case
    hop, ctx_frames = spec.hop, 40
    gen.set_option("small_m_split_k", mode)
    try:
        wav = _audio(spec, 120, 1, seed=61).numpy()
        sess = gen.open_stream(1, ctx_frames * hop)
        ctx = np.zeros((1, 0), dtype=np.float32)
        pos, pushed = 0, []
        for i, n in enumerate([hop] * 3 + [5 * hop] * 10 + [hop // 2, 17 * hop, hop]):
            if pos + n > wav.shape[1]:
                break
            chunk = wav[:, pos:pos + n]
            pos += n
            ctx = np.concatenate([ctx, chunk], axis=1)[:, -max(n, ctx_frames * hop):]
            keep = max(1, n // hop)
            got = sess.push_audio(chunk, keep)
            ref = gen.encode(torch.from_numpy(np.ascontiguousarray(ctx)).cuda(), keep_last_frames=keep).cpu().numpy()
            assert np.array_equal(got, ref), f"{name} push_audio {i} (n={n})"
            pushed.append(got)
        codes = np.concatenate(pushed, axis=1)
        cctx = np.zeros((1, 0), dtype=np.int64)
        for i, n in enumerate([1] * 4 + [5] * 8 + [1] * 3):
            new = codes[:, 2 * i: 2 * i + n]
            cctx = np.concatenate([cctx, new], axis=1)[:, -max(n, ctx_frames):]
            want = n * hop + hop // 2 + 1
            got = sess.push_codes(new, want)
            ref = gen.decode(torch.from_numpy(np.ascontiguousarray(cctx)).cuda(), keep_last_samples=want).cpu().numpy()
            assert got.shape == ref.shape and np.array_equal(got, ref), f"{name} push_codes {i}"
    finally:
        gen.set_option("small_m_split_k", 1)


@pytest.mark.gpu
@pytest.mark.parametrize("codebook_size", [256, 768])
def test_vq_over_few_codebook_tiles(codebook_size):
    """Codebooks of 1 and 3 tiles of 256 rows: the split count is clamped to the tiles.  Codes equal the float64 argmin
    wherever its top-2 margin exceeds 2e-3 (the split-bf16 product is fp32-accurate; tests/test_gpu_parity.py)."""
    spec = _small(codebook_size=codebook_size)
    gen, w = _engine(spec)
    table = gen._dev["vq.codebook"].double().cpu()
    g = torch.Generator().manual_seed(codebook_size)
    for M in (1, 127, 128, 129, 1000, 5000):
        z = torch.randn((M, 16), generator=g) * 1.3
        codes, margin = gen.vq_search(z.cuda(), return_margin=True)
        dist = (z.double()[:, None, :] - table[None]).pow(2).sum(-1)
        top2 = torch.topk(dist, 2, dim=-1, largest=False)
        clear = (top2.values[:, 1] - top2.values[:, 0]) > 2e-3
        assert torch.equal(codes.cpu()[clear], top2.indices[:, 0][clear]), f"K {codebook_size} M {M}"


# ============================================================================ 4. accepted means it runs
REFUSED = {
    "one_conv": dict(conv_strides=(320,), conv_channels=()),
    "heads_not_64_wide": dict(n_heads=4),
    "d_not_multiple_of_64": dict(d_model=160, n_heads=2),
    "ffn_not_multiple_of_64": dict(ffn_dim=200),
    "codebook_dim_8": dict(codebook_dim=8),
    "codebook_not_multiple_of_256": dict(codebook_size=1000),
    "window_left_97": dict(window_left=97),
    "window_right_33": dict(window_right=33),
    "conv1_stride_cin_not_64": dict(conv_strides=(4, 3, 4, 5), conv_channels=(32, 64, 64)),
    "tconv_cin_not_64": dict(conv_channels=(32, 96, 64)),
    "conv0_stride_5": dict(conv_strides=(5, 4, 4, 4)),                        # engine: conv0 stride unsupported
    "conv0_stride_16": dict(conv_strides=(16, 4, 5), conv_channels=(32, 64)),   # engine: conv0 and last tconv stride
    "conv0_channels_24": dict(conv_strides=(8, 8, 5), conv_channels=(24, 128)),  # engine: conv0 channels unsupported
    "conv0_channels_4096": dict(conv_channels=(4096, 64, 64)),                 # engine: conv0 channels unsupported
}


@pytest.mark.parametrize("name", list(REFUSED))
def test_validate_refuses(name):
    with pytest.raises(AssertionError):
        _small(**REFUSED[name]).validate()


@pytest.mark.parametrize("name", list(CONV_STACKS) + list(MATRIX))
def test_validate_accepts_the_specs_tested_here(name):
    spec = _stack_spec(name) if name in CONV_STACKS else MATRIX[name]
    spec.validate()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(REFUSED))
def test_refused_specs_fail_at_construction(name):
    """Every spec validate() refuses fails when B200Generator is built, and mc_create refuses it on its own with a
    message (the C ABI does not rely on the Python check)."""
    spec = _small(**REFUSED[name])
    with pytest.raises(AssertionError):
        pkg.B200Generator(spec, {}, device="cuda")
    lib = nat.load_library()
    cs = mc_spec_struct(spec, 1024)
    h = C.c_void_p()
    rc = lib.mc_create(C.byref(cs), torch.cuda.current_device(), C.byref(h))
    assert rc == -1 and not h.value, name                    # MC_ERR_ARG, no handle
    assert b"unsupported spec" in lib.mc_last_error(None), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONV_STACKS) + list(MATRIX))
def test_accepted_specs_run_every_entry_point(name):
    """A spec validate() accepts builds an engine whose encode, decode, keep_last cuts and stream calls all run."""
    spec = _stack_spec(name) if name in CONV_STACKS else MATRIX[name]
    gen, _ = _engine(spec)
    wav = pkg.synth_audio(7 * spec.hop + 3, seed=71).cuda()
    codes = gen.encode(wav[None])
    assert codes.shape == (1, 8) and int(codes.min()) >= 0 and int(codes.max()) < spec.codebook_size
    assert gen.encode(wav[None], keep_last_frames=3).shape == (1, 3)
    rec = gen.decode(codes)
    assert rec.shape == (1, 8 * spec.hop) and torch.isfinite(rec).all()
    assert torch.equal(gen.decode(codes, keep_last_samples=spec.hop + 1), rec[:, -(spec.hop + 1):])
    sess = gen.open_stream(1, 20 * spec.hop)
    assert sess.push_audio(wav[None, :spec.hop].cpu().numpy(), 1).shape == (1, 1)
    assert sess.push_codes(codes[:, :2].cpu().numpy(), 2 * spec.hop).shape == (1, 2 * spec.hop)
