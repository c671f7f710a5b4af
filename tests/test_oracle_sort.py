"""CPU: pins the oracle (our C restatement, oracle/sort_oracle.c) against
 (1) golden vectors produced by the reference's own compiled sorter (tests/golden/sort_golden.npz), and
 (2) digests of the compiled reference's outputs on the full 20000-splat matrix, including its SIMD spelling
     (tests/golden/sort_ref_digests.npz, written by tests/golden/make_ref_digests.py)."""
import hashlib

import numpy as np
import pytest

import cases

GOLD = np.load(cases.__file__.replace("cases.py", "golden/sort_golden.npz"))
_DIGESTS = np.load(cases.__file__.replace("cases.py", "golden/sort_ref_digests.npz"))
REF_SHA = {str(k): bytes(s) for k, s in zip(_DIGESTS["cref_keys"], _DIGESTS["cref_sha"])}


def _sha(out: np.ndarray) -> bytes:
    return hashlib.sha256(np.ascontiguousarray(out, np.uint32).tobytes()).digest()


def _golden_cases():
    return [str(k) for k in GOLD["names"]]


@pytest.mark.parametrize("key", _golden_cases())
def test_port_matches_reference_golden(oracle_mod, key):
    name, rtag = key.split("|")
    R = int(rtag[1:])
    kw = dict(cases.sort_matrix(n=3000, seeds=(11,)))[name]
    c = cases.sort_case(**kw)
    out, buckets = oracle_mod.port_sort_indexes(*cases.call_args(c, R), want_buckets=True)
    assert np.array_equal(out, GOLD[key + "|out"]), "sorted indexes differ from the reference's output"
    mapped = np.zeros(max(c["render_count"], 1), np.int32)[: c["render_count"]]
    s0 = c["render_count"] - c["sort_count"]
    mapped[s0:] = buckets[s0:]
    sha = np.frombuffer(hashlib.sha256(out.tobytes() + mapped.tobytes()).digest(), np.uint8)
    assert np.array_equal(sha, GOLD[key + "|sha"]), "bucket values (mappedDistances) differ from the reference's"


@pytest.mark.parametrize("name,kw", cases.sort_matrix(n=20000, seeds=(0, 1)))
def test_port_matches_compiled_reference(oracle_mod, name, kw):
    c = cases.sort_case(**kw)
    for R in cases.RANGES:
        b = oracle_mod.port_sort_indexes(*cases.call_args(c, R))
        assert _sha(b) == REF_SHA[f"{name}|R{R}"], f"{name} R={R}"
    if c["integer_sort"]:
        b = oracle_mod.port_sort_indexes(*cases.call_args(c, 1 << 16))
        assert _sha(b) == REF_SHA[f"{name}|simd"], f"{name} simd"


def test_output_is_reverse_stable_by_bucket(oracle_mod):
    """SURVEY Appendix B: out[s0:] == reverse(stable ascending by bucket)."""
    c = cases.sort_case(seed=5, n=30000, ties=True)
    out, buckets = oracle_mod.port_sort_indexes(*cases.call_args(c, 1 << 16), want_buckets=True)
    order = np.argsort(buckets, kind="stable")
    assert np.array_equal(out, c["indexes"][order][::-1])


def test_integer_centers_round_half_up(oracle_mod):
    """Math.round semantics on the f64 product (SplatMesh.js:1919)."""
    x = np.array([[0.0005, -0.0005, 1.2345], [-1.0005, 2.5, -2.5], [1e-7, -1e-7, 123.4565]], np.float32)
    got = oracle_mod.integer_centers(x)
    want = np.floor(x.astype(np.float64) * 1000.0 + 0.5).astype(np.int32)
    assert np.array_equal(got[:, :3], want) and np.all(got[:, 3] == 1000)
