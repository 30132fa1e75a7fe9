"""Stored outputs of call patterns that are otherwise compared live with the reference (tests/golden/golden_host_calls.npz,
written by tests/golden/make_golden_host_calls.py).  A call pattern returns {name: array}; ``to_golden`` turns that into
npz entries under a prefix, ``assert_matches_golden`` checks a fresh run against them."""
import numpy as np

SAMPLE = 256            # stored values per sampled float array
ATOL = 1e-4             # float outputs of the fp32 oracle network on another host (thread count, SIMD width)


def ords(s: str) -> np.ndarray:
    return np.array([ord(c) for c in s], dtype=np.int32)


def to_golden(calls: dict, prefix: str, sample: bool = True) -> dict:
    """With ``sample``, float arrays become shape + a fixed sample of SAMPLE values (compared to ATOL); everything else is
    stored whole and compared exactly."""
    g = {}
    for k, v in calls.items():
        v = np.asarray(v)
        if sample and v.ndim and np.issubdtype(v.dtype, np.floating):
            flat = v.reshape(-1)
            idx = np.sort(np.random.default_rng(flat.size).choice(flat.size, min(flat.size, SAMPLE), replace=False))
            g[f"{prefix}|{k}|shape"] = np.array(v.shape, dtype=np.int64)
            g[f"{prefix}|{k}|sample"] = flat[idx]
        else:
            g[f"{prefix}|{k}"] = v
    return g


def assert_matches_golden(calls: dict, golden, prefix: str, sample: bool = True) -> None:
    got = to_golden(calls, prefix, sample)
    want = sorted(k for k in golden.files if k.startswith(prefix + "|"))
    assert sorted(got) == want
    for k in want:
        if k.endswith("|sample"):
            assert np.allclose(got[k], golden[k], atol=ATOL, rtol=ATOL), k
        else:
            assert got[k].dtype == golden[k].dtype and np.array_equal(got[k], golden[k]), k


def assert_identical(ours: dict, ref: dict) -> None:
    assert sorted(ours) == sorted(ref)
    for k in ref:
        a, b = np.asarray(ours[k]), np.asarray(ref[k])
        assert a.shape == b.shape and np.array_equal(a, b), k
