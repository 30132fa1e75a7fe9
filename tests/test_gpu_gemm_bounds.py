"""Every GEMM kernel and epilogue against a float64 reference, element by element, within a derived error bound.

Kernels, forced through ``block_n``: the single-CTA kernel with 128 x 64 / 128 / 256 tiles (64, 128, 256), its form with
four k-blocks per pipeline stage (4064), the CTA-pair kernel (512) with the specialised and the generic epilogues
(``fast_epilogue`` 1 / 0), the split-K cluster kernel with S = 2 / 4 / 8 (1002 / 1004 / 1008), and the automatic choice
(0) under ``small_m_split_k`` 0 and 2.  The reference is computed on the device in float64 from the kernel's own bf16
operands, fp32 bias, gamma, row statistics and fp32 RoPE tables.

Error bound per output element (u = 2^-24, the fp32 unit roundoff; |.| of an intermediate means |reference| plus its
bound):

* Accumulator.  bf16 x bf16 products are exact in fp32.  tcgen05.mma kind::f16 sums 16-deep k-groups and adds the K/16
  group partials into the fp32 accumulator in tensor memory.  Granting each of those K/16 + 16 additions a relative
  error of 2^-23 (twice the round-to-nearest unit, in case the adds truncate):
      E_acc = (K/16 + 16) 2^-23 sum_k |a_k w_k|.
  The summation precision inside the tensor core is not documented, so this is a derivation, not a measurement; the
  module prints the largest err / bound it met per (kernel, mode).
* Split-K over S CTAs: the S partial tiles are added in a fixed order over DSMEM.  Every running sum is bounded by
  sum_k |a_k w_k| (not by |ref|: partials can cancel), so the S - 1 fp32 adds add at most S u sum_k |a_k w_k|.
* Bias add, residual add: one fp32 rounding each, u |result|.
* Fused-RMSNorm consumer y = fmaf(acc, rs, bias), rs = rsqrtf(fmaf(sum_c st_c, 1/K, eps)) (row_rs): the in-order sum of
  n non-negative chunk statistics is off by at most (n - 1) u relative, 1/K and the fma by u each, and rsqrtf by 2 ulp
  (CUDA C++ Programming Guide, single-precision mathematical functions), so rel(rs) = (n + 1) u / 2 + 2^-22 and
      E = rs E_acc + rs |acc| rel(rs) + u |y|.
* tanh-GELU y = x/2 + x/2 tanh(u) (gelu_tanh_f): |GELU'| <= 1.13 carries the input error.  tanh.approx.f32 is documented
  in the PTX ISA (tanh) with a maximum error of 2^-10.987 ~ 2^-11; as |tanh| <= 1 we use it as an absolute error of t.
  The three fp32 roundings that form u move t by at most 2^-22 more:
      E = 1.13 E_x + |x|/2 (2^-10.987 + 2^-22) + u |y|.
* RoPE (x1, x2) -> (x1 c - x2 s, x1 s + x2 c) on 64-wide heads below rope_cols, one product and one fma or subtraction:
      E1' = |c| E1 + |s| E2 + 2^-23 (|x1 c| + |x2 s|),   E2' = |s| E1 + |c| E2 + 2^-23 (|x1 s| + |x2 c|).
* bf16 store: round to nearest, 2^-8 |y| (half an ulp).
* Fused-RMSNorm producer: x as for the residual epilogue; xb must equal bf16(fp32(x * gamma)) of the kernel's own x bit
  for bit, and each 64-column statistic, an fma chain (or, split-K, partial chains and a butterfly) over x^2, is within
  65 u sum x^2 of the float64 sum.

A NaN or infinite output, or one outside the bound, fails the element check and is recorded as an infinite ratio.

The self-checks (no GPU) apply each bug the bound must catch to the float64 reference and assert that it is rejected.
The GPU tests also write every output into a larger buffer whose extra rows (and columns N .. ldo, more than one
64-column chunk, where the entry point takes an ldo) hold a NaN sentinel.  They check that the sentinel survives and
that every element in range was written.  They check that every single-accumulator kernel returns the same bits for
the same (mode, shape) (the batch invariance of DESIGN §5), and that the automatic choice under small_m_split_k 2
returns the bits of a kernel it may pick: bn64's above 256 rows, bn64's or a split-K kernel's below.  They check that
each split-K kernel repeats itself, and that the launcher refuses what the kernels cannot do without touching the
output.

The ``pair_fast`` column of the printed table runs a specialised epilogue only where launch_gemm_pair selects one: a
bias, N % 256 == 0 and a mode with a specialised form (bf16 RoPE, bf16 GELU, fp32 residual, the producer).  Everywhere
else, including the fp32, plain bf16 and consumer modes, it runs the generic epilogue, as ``pair_generic`` does.
"""
import contextlib
import math

import pytest
import torch

import realtime_codec_agent_b200 as pkg
from realtime_codec_agent_b200 import _native as nat

U = 2.0 ** -24
U_BF16 = 2.0 ** -8
EPS_TANH = 2.0 ** -10.987          # PTX ISA, tanh.approx.f32
GELU_SLOPE = 1.13                  # max |d/dx gelu_tanh(x)| = 1.1289...
GELU_C0, GELU_C1 = 0.7978845608028654, 0.044715

SENT_F32 = 0x7FC0DEAD              # quiet NaN with a payload no kernel produces
SENT_BF16 = 0x7FC1


# --------------------------------------------------------------------------------------------- float64 reference

def gelu64(x, tanh_scale=1.0):
    return 0.5 * x * (1.0 + torch.tanh(GELU_C0 * (x + GELU_C1 * x ** 3)) * tanh_scale)


def gemm_reference(A, W, *, bias=None, act=0, out_mode=1, x0=None, rope=None, row_stats=None, norm_eps=0.0, split=1,
                   exact_acc=False, tanh_scale=1.0):
    """float64 value and error bound (module docstring) of every element of epilogue(A @ W^T).

    rope = (rope_cols, cos, sin) with cos / sin [M, 32]: the table row of each output row.
    row_stats [M, K/64]: consumer.
    exact_acc: the accumulator is exact (identity weights), so only the epilogue is bounded.  tanh_scale exists to model
    a wrong tanh in the self-checks."""
    a, w = A.double(), W.double()
    K = a.shape[1]
    v = a @ w.t()
    s1 = a.abs() @ w.abs().t()
    E = torch.zeros_like(v) if exact_acc else (K / 16 + 16) * 2.0 ** -23 * s1
    if split > 1:
        E = E + split * U * s1
    if row_stats is not None:
        st = row_stats.double()
        rs = torch.rsqrt(st.sum(1, keepdim=True) / K + norm_eps)
        rel = (st.shape[1] + 1) * U / 2 + 2.0 ** -22
        E = rs * E + rs * v.abs() * rel
        v = v * rs
        if bias is not None:
            v = v + bias.double()
        E = E + U * (v.abs() + E)
    elif bias is not None:
        v = v + bias.double()
        E = E + U * (v.abs() + E)
    if act:
        x, ex = v, E
        v = gelu64(x, tanh_scale)
        E = GELU_SLOPE * ex + 0.5 * (x.abs() + ex) * (EPS_TANH + 2.0 ** -22)
        E = E + U * (v.abs() + E)
    if rope is not None and rope[0] > 0:
        cols, c, s = rope
        M = v.shape[0]
        c, s = c.double()[:, None, :], s.double()[:, None, :]
        h = v[:, :cols].reshape(M, cols // 64, 2, 32)
        eh = E[:, :cols].reshape(M, cols // 64, 2, 32)
        x1, x2, e1, e2 = h[:, :, 0], h[:, :, 1], eh[:, :, 0], eh[:, :, 1]
        a1, a2 = x1.abs() + e1, x2.abs() + e2
        y1, y2 = x1 * c - x2 * s, x1 * s + x2 * c
        f1 = c.abs() * e1 + s.abs() * e2 + 2.0 ** -23 * (a1 * c.abs() + a2 * s.abs())
        f2 = s.abs() * e1 + c.abs() * e2 + 2.0 ** -23 * (a1 * s.abs() + a2 * c.abs())
        v = torch.cat((torch.stack((y1, y2), 2).reshape(M, cols), v[:, cols:]), 1)
        E = torch.cat((torch.stack((f1, f2), 2).reshape(M, cols), E[:, cols:]), 1)
    if out_mode == 2:
        v = x0.double() + v
        E = E + U * (v.abs() + E)
    if out_mode == 0:
        E = E + U_BF16 * (v.abs() + E)
    return v, E


def stats_reference(x):
    """float64 sum of x^2 per 64-column chunk of the kernel's own fp32 x, and its bound (a chain of 64 fp32 fmas)."""
    sq = x.double().pow(2).reshape(x.shape[0], -1, 64).sum(-1)
    return sq, 65 * U * sq


def rope_rows(cos_t, sin_t, rows, period, shift=0):
    """cos / sin [rows, 32] of output rows 0..rows-1 (position row % period, plus a shift for the self-checks) from the
    transposed [32, max_positions] tables."""
    pos = torch.arange(rows, device=cos_t.device) % period + shift
    return cos_t[:, pos].t(), sin_t[:, pos].t()


def rope_cols_for(N):
    """q and k heads of a QKV-like output: two thirds of the 64-wide heads (at least one)."""
    return 64 * max(1, (2 * (N // 64)) // 3)


def exceed(got, ref, bound):
    """(number of elements outside the bound, largest err / bound).  A NaN output is outside, with ratio inf."""
    err = (got.double() - ref).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    ratio = torch.where(torch.isnan(err), torch.full_like(err, math.inf), ratio)
    return int((~(err <= bound)).sum()), float(ratio.max()) if ratio.numel() else 0.0


# --------------------------------------------------------------------------------------------- self-checks (CPU)

def _cpu_tables(max_pos=64):
    inv = 1.0 / (10000.0 ** (torch.arange(0, 32, dtype=torch.float32) * 2.0 / 64))
    f = torch.outer(torch.arange(max_pos, dtype=torch.float32), inv)
    return torch.cos(f).t().contiguous(), torch.sin(f).t().contiguous()


def _cpu_case(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    A = torch.randn((M, K), generator=g).to(torch.bfloat16)
    W = (torch.randn((N, K), generator=g) / math.sqrt(K)).to(torch.bfloat16)
    bias = torch.randn((N,), generator=g)
    x0 = torch.randn((M, N), generator=g)
    stats = 64.0 * (0.25 + 2.0 * torch.rand((M, K // 64), generator=g))
    return A, W, bias, x0, stats


SELF_CASES = [(37, 192, 256), (5, 320, 1024), (64, 64, 448), (3, 1152, 4096), (129, 16, 64), (2, 576, 192)]


@pytest.mark.parametrize("M,N,K", SELF_CASES)
def test_bound_rejects_each_bug(M, N, K):
    """Each mutation is a bug the bound must catch: applied to the float64 reference, at least one element of every case
    must fall outside the bound of the correct result."""
    A, W, bias, x0, stats = _cpu_case(M, N, K, seed=M * 7 + N + K)
    cos_t, sin_t = _cpu_tables()
    eps, period = 1e-5, 7

    def rejected(mut, ref_bound):
        return exceed(mut, *ref_bound)[0] > 0

    # fp32 output rounded to bf16 somewhere
    ref, bound = gemm_reference(A, W, bias=bias, out_mode=1)
    assert rejected(ref.float().to(torch.bfloat16).double(), (ref, bound)), "fp32 output rounded to bf16"
    for out_mode in (1, 0):
        # the bias dropped from the last 64-column chunk
        ok = gemm_reference(A, W, bias=bias, out_mode=out_mode)
        b = bias.clone()
        b[(N - 1) // 64 * 64:] = 0
        assert rejected(gemm_reference(A, W, bias=b, out_mode=out_mode)[0], ok), f"bias dropped, out_mode {out_mode}"
        # one 64-wide k-block dropped
        for kb in sorted({0, K // 64 - 1}):
            a = A.clone()
            a[:, kb * 64:(kb + 1) * 64] = 0
            assert rejected(gemm_reference(a, W, bias=bias, out_mode=out_mode)[0], ok), f"k-block {kb} dropped"
    # the residual read from the wrong row
    if M > 1:
        ok = gemm_reference(A, W, bias=bias, out_mode=2, x0=x0)
        assert rejected(gemm_reference(A, W, bias=bias, out_mode=2, x0=x0.roll(1, 0))[0], ok), "residual row"
    # the consumer's row scale taken from the neighbouring row
    if M > 1:
        for act in (0, 1):
            ok = gemm_reference(A, W, bias=bias, act=act, out_mode=0, row_stats=stats, norm_eps=eps)
            mut = gemm_reference(A, W, bias=bias, act=act, out_mode=0, row_stats=stats.roll(1, 0), norm_eps=eps)[0]
            assert rejected(mut, ok), f"row scale of the neighbouring row, act {act}"
    # GELU whose tanh is 2^-7 off
    ok = gemm_reference(A, W, bias=bias, act=1, out_mode=0)
    assert rejected(gemm_reference(A, W, bias=bias, act=1, out_mode=0, tanh_scale=1 + 2.0 ** -7)[0], ok), "tanh 2^-7"
    # RoPE: position off by one, rope_cols off by 64 (either way)
    if N >= 64:
        cols = rope_cols_for(N)
        for out_mode in (0, 1):
            c, s = rope_rows(cos_t, sin_t, M, period)
            ok = gemm_reference(A, W, bias=bias, out_mode=out_mode, rope=(cols, c, s))
            c1, s1 = rope_rows(cos_t, sin_t, M, period, shift=1)
            assert rejected(gemm_reference(A, W, bias=bias, out_mode=out_mode, rope=(cols, c1, s1))[0], ok), "position"
            for dc in (-64, 64):
                if 0 <= cols + dc <= N // 64 * 64:
                    mut = gemm_reference(A, W, bias=bias, out_mode=out_mode, rope=(cols + dc, c, s))[0]
                    assert rejected(mut, ok), f"rope_cols {cols + dc} instead of {cols}"


def test_bound_accepts_fp32_rounding_of_the_exact_result():
    """The bound is not vacuous in the other direction: the correctly rounded fp32 / bf16 results of every epilogue are
    inside it."""
    A, W, bias, x0, stats = _cpu_case(33, 320, 1024, seed=5)
    cos_t, sin_t = _cpu_tables()
    c, s = rope_rows(cos_t, sin_t, 33, 7)
    for kw in (dict(out_mode=1), dict(out_mode=0, act=1), dict(out_mode=2, x0=x0), dict(out_mode=0, rope=(192, c, s)),
               dict(out_mode=0, row_stats=stats, norm_eps=1e-5, act=1)):
        ref, bound = gemm_reference(A, W, bias=bias, **kw)
        got = ref.float() if kw["out_mode"] else ref.float().to(torch.bfloat16)
        assert exceed(got, ref, bound)[0] == 0, kw


@pytest.mark.parametrize("bad", [math.nan, math.inf, -math.inf])
def test_element_check_rejects_non_finite_outputs(bad):
    """A NaN or infinite output element is outside the bound and shows as an infinite ratio in the printed table."""
    A, W, bias, _, _ = _cpu_case(9, 64, 192, seed=3)
    ref, bound = gemm_reference(A, W, bias=bias, out_mode=1)
    got = ref.float()
    got[4] = bad                  # a whole row
    got[7, 5] = bad               # and one more element
    n, r = exceed(got, ref, bound)
    assert n == 65 and r == math.inf
    table = {}
    _record(table, ("k", "m"), r)
    _record(table, ("k", "m"), 0.5)
    assert table[("k", "m")] == math.inf


# --------------------------------------------------------------------------------------------- GPU: fixtures, helpers

KERNELS = [  # name, block_n, options
    ("bn64", 64, {}), ("bn128", 128, {}), ("bn256", 256, {}), ("kps4", 4064, {}),
    ("pair_fast", 512, {"fast_epilogue": 1}), ("pair_generic", 512, {"fast_epilogue": 0}),
    ("splitk2", 1002, {}), ("splitk4", 1004, {}), ("splitk8", 1008, {}),
    ("auto_sk0", 0, {"small_m_split_k": 0}), ("auto_sk2", 0, {"small_m_split_k": 2}),
]
# one fp32 accumulator per output tile: the same products in the same order, so the same bits whatever the tiling
SINGLE_ACC = ("bn64", "bn128", "bn256", "kps4", "pair_fast", "pair_generic", "auto_sk0")
OPTION_DEFAULTS = {"fast_epilogue": 1, "small_m_split_k": 1}
MAX_POS = 1024
LDO_PAD = 72         # columns N .. ldo: more than one 64-column chunk, so a stray chunk past N lands on the sentinel


def _split_of(name):
    return int(name[6:]) if name.startswith("splitk") else 1


def _runs(name, K):
    kb = K // 64
    if name == "kps4":
        return kb % 4 == 0
    return kb % _split_of(name) == 0


@contextlib.contextmanager
def _options(gen, opts):
    try:
        for k, v in opts.items():
            gen.set_option(k, v)
        yield
    finally:
        for k in opts:
            gen.set_option(k, OPTION_DEFAULTS[k])


@pytest.fixture(scope="module")
def gen():
    spec = pkg.TINY_SPEC
    return pkg.B200Generator(spec, pkg.init_random_weights(spec, seed=0), device="cuda", max_positions=MAX_POS)


@pytest.fixture(scope="module")
def ratios(request):
    """Largest err / bound per (kernel, mode), printed when the module ends."""
    table = {}
    yield table
    if not table:
        return
    kernels = [k for k, _, _ in KERNELS]
    kernels += sorted({k for k, _ in table} - set(kernels))
    modes = sorted({m for _, m in table})
    lines = ["", "largest err / bound per (kernel, mode):", f"{'mode':<16}" + "".join(f"{k:>13}" for k in kernels)]
    for m in modes:
        cells = (f"{table[(k, m)]:>13.4f}" if (k, m) in table else f"{'-':>13}" for k in kernels)
        lines.append(f"{m:<16}" + "".join(cells))
    lines.append(f"overall max {max(table.values()):.4f}")
    capman = request.config.pluginmanager.get_plugin("capturemanager")
    with capman.global_and_fixture_disabled() if capman is not None else contextlib.nullcontext():
        for line in lines:
            print(line)


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda") * scale


def _sentinel(shape, dtype):
    if dtype == torch.bfloat16:
        return torch.full(shape, SENT_BF16, dtype=torch.int16, device="cuda").view(torch.bfloat16)
    return torch.full(shape, SENT_F32, dtype=torch.int32, device="cuda").view(torch.float32)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _is_sentinel(t):
    return _bits(t) == (SENT_BF16 if t.dtype == torch.bfloat16 else SENT_F32)


def _check_buffer(buf, inside, what, resid=False):
    """Outside the in-range block: sentinel untouched.  Inside: every element written (no sentinel left)."""
    keep = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    keep[inside] = False
    assert bool(_is_sentinel(buf)[keep].all()), f"{what}: wrote outside its output block"
    if not resid:
        assert not bool(_is_sentinel(buf[inside]).any()), f"{what}: left elements of its output block unwritten"


def _record(ratios, key, r):
    ratios[key] = max(ratios.get(key, 0.0), math.inf if math.isnan(r) else r)


def _assert_same_bits(results, M, what):
    """results: kernel name -> {buffer name: tensor}.  Every single-accumulator kernel returns bn64's bits.  The
    automatic choice under small_m_split_k 2 never splits above 256 rows, so there it returns bn64's bits too; below,
    it returns the bits of bn64 or of the split-K kernel it picked."""
    def same(a, b):
        return all(torch.equal(_bits(a[k]), _bits(b[k])) for k in a)

    base = results["bn64"]
    for name in SINGLE_ACC:
        if name in results:
            assert same(results[name], base), f"{name} {what}: not bn64's bits"
    if "auto_sk2" in results:
        picks = ["bn64"] + ([] if M > 256 else [n for n in results if n.startswith("splitk")])
        assert any(same(results["auto_sk2"], results[n]) for n in picks), f"auto_sk2 {what}: bits of none of {picks}"


def _assert_within(got, ref, bound, ratios, key, what):
    bad, r = exceed(got, ref, bound)
    _record(ratios, key, r)
    assert bad == 0, f"{what}: {bad} of {ref.numel()} elements outside the bound, largest err / bound {r:.3f}"


def _fused_call(gen, A, W, bias, out_mode, out, *, act=0, row_stats=None, xb=None, gamma=None, st=None, rope_cols=0,
                rope_period=0, block_n=0):
    """mc_op_gemm_fused with caller-owned (oversized, sentinel-filled) output, xb and statistics buffers."""
    M, K = A.shape
    N = W.shape[0]
    rc = gen._lib.mc_op_gemm_fused(gen._handle, A.data_ptr(), W.data_ptr(), nat.ptr(bias), M, N, K, act, out_mode,
                                   out.data_ptr(), nat.ptr(row_stats), 0 if row_stats is None else row_stats.shape[1],
                                   nat.ptr(xb), nat.ptr(gamma), nat.ptr(st), rope_cols, rope_period, block_n,
                                   gen._stream())
    nat.check(gen._lib, gen._handle, rc, "mc_op_gemm_fused")


# --------------------------------------------------------------------------------------------- GPU: the matrix

MODES = {  # out_mode, act, rope, role
    "f32": (1, 0, False, None), "f32_nobias": (1, 0, False, None), "bf16": (0, 0, False, None),
    "bf16_gelu": (0, 1, False, None), "resid": (2, 0, False, None), "rope_bf16": (0, 0, True, None),
    "rope_f32": (1, 0, True, None), "consumer_gelu": (0, 1, False, "consumer"),
    "consumer_rope": (0, 0, True, "consumer"), "producer": (2, 0, False, "producer"),
}

N_LIST = [16, 64, 192, 320, 384, 448, 576, 1088, 1152, 2304, 1024]   # spec-matrix widths (N % 256: 16, 0, 64, 128, 192)
K_LIST = [64, 192, 320, 448, 1024, 4096]                             # 1, 3, 5, 7 k-blocks; split-K / KPS 4 shapes
M_LIST = [1, 100, 127, 128, 129, 255, 257, 300, 2597]
PERIODS = [100, 37, 300, 7, 1000, 1]                                  # none divides 128 or 256: tiles span windows


def _cases():
    """(mode, M, N, K, rope period), a covering selection (test_covering_selection states what it covers): every mode
    meets every N twice, once with K cycling through K_LIST and once with a K that every split-K and the KPS 4 kernel
    accept, while M cycles through M_LIST; plus one CTA-pair-sized case of 25 600 rows."""
    cases = []
    for mi, mode in enumerate(MODES):
        rope = MODES[mode][2]
        for i, N in enumerate(N_LIST):
            if (rope and N < 64) or (MODES[mode][3] == "producer" and N % 64):
                continue
            p = PERIODS[(i + mi) % len(PERIODS)] if rope else 0
            cases.append((mode, M_LIST[(i + 2 * mi) % len(M_LIST)], N, K_LIST[(i + mi) % len(K_LIST)], p))
            cases.append((mode, M_LIST[(i + 2 * mi + 4) % len(M_LIST)], N, (1024, 4096)[(i + mi) % 2], p))
    return cases + [("rope_bf16", 25600, 1152, 1024, 100), ("producer", 25600, 1088, 1024, 0)]


CASES = _cases()


def test_covering_selection():
    """Every kernel meets every mode at every N % 256 residue the mode accepts; every mode meets partial last M tiles,
    below and above one tile; every listed M, N and K occurs; one case has >= 25 600 rows."""
    for name, _, _ in KERNELS:
        for mode, (_, _, rope, role) in MODES.items():
            want = {0, 64, 128, 192} | (set() if rope or role == "producer" else {16})
            got = {N % 256 if N >= 64 else N for m, M, N, K, _ in CASES if m == mode and _runs(name, K)}
            assert got == want, (name, mode, got)
    for mode in MODES:
        Ms = {M for m, M, _, _, _ in CASES if m == mode}
        assert any(1 < M < 128 for M in Ms) and any(M > 128 and M % 128 for M in Ms), mode
    assert {c[1] for c in CASES} >= set(M_LIST) and {c[2] for c in CASES} == set(N_LIST)
    assert {c[3] for c in CASES} == set(K_LIST) and max(c[1] for c in CASES) >= 25600


def _case_id(c):
    return f"{c[0]}-M{c[1]}-N{c[2]}-K{c[3]}" + (f"-p{c[4]}" if c[4] else "")


@pytest.mark.gpu
@pytest.mark.parametrize("mode,M,N,K,period", CASES, ids=[_case_id(c) for c in CASES])
def test_gemm_kernels_against_float64(gen, ratios, mode, M, N, K, period):
    out_mode, act, has_rope, role = MODES[mode]
    seed = M * 31 + N * 7 + K
    A = _rand((M, K), seed).to(torch.bfloat16)
    W = (_rand((N, K), seed + 1) / math.sqrt(K)).to(torch.bfloat16)
    bias = None if mode == "f32_nobias" else _rand((N,), seed + 2)
    x0 = _rand((M, N), seed + 3) if out_mode == 2 else None
    stats = None
    if role == "consumer":
        g = torch.Generator(device="cuda").manual_seed(seed + 4)
        stats = 64.0 * (0.25 + 2.0 * torch.rand((M, K // 64), generator=g, device="cuda"))
    gamma = 1.0 + 0.1 * _rand((N,), seed + 5) if role == "producer" else None
    rope_cols = rope_cols_for(N) if has_rope else 0
    rope = None
    if has_rope:
        rope = (rope_cols,) + rope_rows(gen._dev["rope.cos"], gen._dev["rope.sin"], M, period)
    odt = torch.bfloat16 if out_mode == 0 else torch.float32
    pad_rows = 5
    ldo = N + LDO_PAD if role is None else N      # the fused entry point writes dense rows

    def run(bn):
        buf = _sentinel((M + pad_rows, ldo), odt)
        if x0 is not None:
            buf[:M, :N] = x0
        res = {"out": buf}
        if role is None:
            gen.op_gemm(A, W, bias=bias, act=act, out_mode=out_mode, out=buf, M=M, ldo=ldo, rope_cols=rope_cols,
                        rope_period=period, block_n=bn)
        elif role == "consumer":
            _fused_call(gen, A, W, bias, out_mode, buf, act=act, row_stats=stats, rope_cols=rope_cols,
                        rope_period=period, block_n=bn)
        else:
            res["xb"] = _sentinel((M + pad_rows, N), torch.bfloat16)
            res["st"] = _sentinel((M + pad_rows, N // 64), torch.float32)
            _fused_call(gen, A, W, bias, out_mode, buf, xb=res["xb"], gamma=gamma, st=res["st"], block_n=bn)
        return res

    results = {}
    refs = {}
    for name, bn, opts in KERNELS:
        if not _runs(name, K):
            continue
        with _options(gen, opts):
            res = run(bn)
            if name not in SINGLE_ACC:
                again = run(bn)
                for k in res:
                    assert torch.equal(_bits(res[k]), _bits(again[k])), f"{name} {mode}: {k} differs from run to run"
        torch.cuda.synchronize()
        what = f"{name} {_case_id((mode, M, N, K, period))}"
        _check_buffer(res["out"], (slice(0, M), slice(0, N)), what, resid=out_mode == 2)
        # a split-K kernel's bound carries its S; the automatic choice may split (by at most 8)
        split = 8 if name == "auto_sk2" else _split_of(name)
        if split not in refs:
            refs[split] = gemm_reference(A, W, bias=bias, act=act, out_mode=out_mode, x0=x0, rope=rope, row_stats=stats,
                                         norm_eps=gen.spec.norm_eps, split=split)
        ref, bound = refs[split]
        out = res["out"][:M, :N]
        _assert_within(out, ref, bound, ratios, (name, mode), what)
        if role == "producer":
            _check_buffer(res["xb"], (slice(0, M), slice(0, N)), what + " xb")
            _check_buffer(res["st"], (slice(0, M), slice(0, N // 64)), what + " stats")
            xb_want = (out * gamma).to(torch.bfloat16)
            assert torch.equal(_bits(res["xb"][:M]), _bits(xb_want)), f"{what}: xb != bf16(x * gamma)"
            sref, sbound = stats_reference(out)
            _assert_within(res["st"][:M], sref, sbound, ratios, (name, "producer_stats"), what + " stats")
        results[name] = res
    _assert_same_bits(results, M, _case_id((mode, M, N, K, period)))


CONV_CASES = [  # groups, frames per group (valid), row block, N
    (3, 100, 128, 192), (2, 63, 512, 1152), (10, 259, 64, 448), (5, 50, 2048, 16), (4, 31, 192, 576),
    (2, 149, 512, 1024),
]


@pytest.mark.gpu
@pytest.mark.parametrize("Bn,T,blk,N", CONV_CASES)
def test_conv_view_kernels_against_float64(gen, ratios, Bn, T, blk, N):
    """Row-block A view (K = 2 row blocks), group remap (one junk row per group dropped), left padding and ldo > N:
    bf16 + GELU, as the convolutions run it."""
    rows, K, pad, extra = Bn * (1 + T), 2 * blk, 4, 2
    ldo = N + LDO_PAD
    seed = Bn * 1000 + T + blk + N
    buf_a = _rand((rows, blk), seed).to(torch.bfloat16)
    W = (_rand((N, K), seed + 1) / math.sqrt(K)).to(torch.bfloat16)
    bias = _rand((N,), seed + 2)
    flat = torch.cat([buf_a.reshape(-1), torch.zeros(blk, device="cuda", dtype=torch.bfloat16)])
    idx = torch.arange(rows, device="cuda")[:, None] * blk + torch.arange(K, device="cuda")[None, :]
    A_eff = flat[idx]
    results, refs = {}, {}
    inside = (slice(None), slice(pad, pad + T), slice(0, N))
    for name, bn, opts in KERNELS:
        if not _runs(name, K):
            continue
        with _options(gen, opts):
            out = _sentinel((Bn, pad + T + extra, ldo), torch.bfloat16)
            gen.op_gemm(buf_a, W, bias=bias, act=1, out_mode=0, out=out, a_k_wrap=blk, M=rows, K=K, grp_in=1 + T,
                        grp_valid=T, grp_stride=(pad + T + extra) * ldo, grp_off=pad * ldo, ldo=ldo, block_n=bn)
        torch.cuda.synchronize()
        what = f"{name} conv B{Bn} T{T} blk{blk} N{N}"
        _check_buffer(out, inside, what)
        split = 8 if name == "auto_sk2" else _split_of(name)
        if split not in refs:
            ref, bound = gemm_reference(A_eff, W, bias=bias, act=1, out_mode=0, split=split)
            refs[split] = (ref.view(Bn, 1 + T, N)[:, :T], bound.view(Bn, 1 + T, N)[:, :T])
        _assert_within(out[inside], *refs[split], ratios, (name, "conv"), what)
        results[name] = {"out": out}
    _assert_same_bits(results, rows, f"conv B{Bn} T{T} blk{blk} N{N}")


# --------------------------------------------------------------------------------------------- GPU: epilogues alone

ID_K, ID_N = 512, 256        # identity in the first k-block, zeros after it: exact for every kernel, split-K included


def _identity_weights():
    W = torch.zeros((ID_N, ID_K), device="cuda")
    W[torch.arange(ID_N), torch.arange(ID_N) % 64] = 1.0
    return W.to(torch.bfloat16)


def _bf16_grid(lo=2.0 ** -60, hi=10.0):
    """Every bf16 value with lo <= |x| <= hi, and zero (no subnormal inputs or results)."""
    v = torch.arange(-32768, 32768, dtype=torch.int32, device="cuda").to(torch.int16).view(torch.bfloat16).float()
    v = v[torch.isfinite(v) & (((v.abs() >= lo) & (v.abs() <= hi)) | (v == 0))]
    return torch.unique(v)


@pytest.mark.gpu
@pytest.mark.parametrize("fn", ["gelu_f32", "gelu_bf16", "rope_f32", "rope_bf16"])
def test_epilogue_functions_alone(gen, ratios, fn):
    """W = rows of the identity and a zero bias: the accumulator equals the chosen inputs exactly, so tanh-GELU over the
    bf16 grid on [-10, 10] and RoPE at every position of the table are measured against float64 with no accumulation
    error, in every kernel."""
    W = _identity_weights()
    bias = torch.zeros((ID_N,), device="cuda")
    out_mode = 0 if fn.endswith("bf16") else 1
    if fn.startswith("gelu"):
        vals = _bf16_grid()
        M = (vals.numel() + 63) // 64
        A64 = torch.zeros(M * 64, device="cuda")
        A64[:vals.numel()] = vals
        A64 = A64.view(M, 64)
        act, rope_cols, period, rope = 1, 0, 0, None
    else:
        M = MAX_POS
        A64 = _rand((M, 64), seed=77, scale=4.0)
        act, rope_cols, period = 0, 128, MAX_POS
        rope = (rope_cols,) + rope_rows(gen._dev["rope.cos"], gen._dev["rope.sin"], M, period)
    A = torch.zeros((M, ID_K), device="cuda", dtype=torch.bfloat16)
    A[:, :64] = A64.to(torch.bfloat16)
    ref, bound = gemm_reference(A, W, bias=bias, act=act, out_mode=out_mode, rope=rope, exact_acc=True)
    odt = torch.bfloat16 if out_mode == 0 else torch.float32
    results = {}
    for name, bn, opts in KERNELS:
        with _options(gen, opts):
            out = _sentinel((M + 3, ID_N + LDO_PAD), odt)
            gen.op_gemm(A, W, bias=bias, act=act, out_mode=out_mode, out=out, M=M, ldo=ID_N + LDO_PAD,
                        rope_cols=rope_cols, rope_period=period, block_n=bn)
        torch.cuda.synchronize()
        _check_buffer(out, (slice(0, M), slice(0, ID_N)), f"{name} {fn}")
        _assert_within(out[:M, :ID_N], ref, bound, ratios, (name, "id_" + fn), f"{name} {fn}")
        results[name] = {"out": out}
    _assert_same_bits(results, M, fn)


# --------------------------------------------------------------------------------------------- GPU: refusals

REFUSALS = {
    "k_not_64": ("multiples of 64", dict(K=96)),
    "n_not_8": ("multiple of 8", dict(N=20)),
    "rope_period_too_long": ("exceeds table rows", dict(rope_period=MAX_POS + 1)),
    "split_k_does_not_divide": ("do not split", dict(K=192, block_n=1002)),
    "split_k_rope_cols": ("64-wide heads", dict(rope_period=10, rope_cols=96, block_n=1004)),
    "producer_bf16_out": ("needs an fp32 output", dict(producer=True, out_mode=0)),
    "producer_n_not_64": ("N % 64 == 0", dict(producer=True, out_mode=1, N=200)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refusals_name_the_rule_and_leave_the_output(gen, case):
    rule, kw = REFUSALS[case]
    M, N, K = 100, kw.get("N", 256), kw.get("K", 256)
    A = _rand((M, K), 90).to(torch.bfloat16)
    W = _rand((N, K), 91).to(torch.bfloat16)
    bias = _rand((N,), 92)
    out_mode = kw.get("out_mode", 0)
    out = _sentinel((M + 2, N), torch.bfloat16 if out_mode == 0 else torch.float32)
    with pytest.raises(nat.McError, match=rule):
        if kw.get("producer"):
            xb = _sentinel((M, N), torch.bfloat16)
            st = _sentinel((M, N // 64 + 1), torch.float32)
            _fused_call(gen, A, W, bias, out_mode, out, xb=xb, gamma=torch.ones(N, device="cuda"), st=st)
        else:
            gen.op_gemm(A, W, bias=bias, out_mode=0, out=out, M=M, rope_cols=kw.get("rope_cols", 0),
                        rope_period=kw.get("rope_period", 0), block_n=kw.get("block_n", 0))
    torch.cuda.synchronize()
    assert bool(_is_sentinel(out).all()), f"{case}: the refused call wrote its output"
    if kw.get("producer"):
        assert bool(_is_sentinel(xb).all()) and bool(_is_sentinel(st).all())


# --------------------------------------------------------------------------------------------- GPU: RMSNorm, rowstats

NORM_DIMS = [192, 320, 448, 576, 128, 256, 512, 1024]   # generic rmsnorm_kernel, then the rows<NV> kernels


@pytest.mark.gpu
@pytest.mark.parametrize("d", NORM_DIMS)
def test_rmsnorm_and_rowstats_against_float64(gen, ratios, d):
    """op_rmsnorm: y = bf16(x * rs * gamma), rs = rsqrtf(sum x^2 / d + eps).  The sum of squares (per-lane fma chains
    and a 5-level tree) is within d u relative; / d and + eps add u each; rsqrtf 2 ulp (2^-22); two products 2 u; then
    the bf16 store 2^-8:  E = |y| ((d + 2) u / 2 + 2^-22 + 2 u) + 2^-8 (|y| + E).
    op_rowstats: xb = bf16(fp32(x * gamma)) bit for bit, statistics within 65 u sum x^2 of float64 (stats_reference)."""
    M = 333
    x = _rand((M, d), seed=d, scale=3.0)
    x[7] *= 1e-3                     # rows of very different scale
    x[8] *= 1e3
    gamma = 1.0 + 0.1 * _rand((d,), seed=d + 1)
    eps = gen.spec.norm_eps
    xd = x.double()
    y = xd * torch.rsqrt(xd.pow(2).mean(-1, keepdim=True) + eps) * gamma.double()
    E = y.abs() * ((d + 2) * U / 2 + 2.0 ** -22 + 2 * U)
    E = E + U_BF16 * (y.abs() + E)
    _assert_within(gen.op_rmsnorm(x, gamma), y, E, ratios, ("rmsnorm", f"d{d}"), f"rmsnorm d={d}")
    xb, st = gen.op_rowstats(x, gamma)
    assert torch.equal(_bits(xb), _bits((x * gamma).to(torch.bfloat16))), f"rowstats d={d}: xb != bf16(x * gamma)"
    sref, sbound = stats_reference(x)
    _assert_within(st, sref, sbound, ratios, ("rowstats", f"d{d}"), f"rowstats d={d}")
