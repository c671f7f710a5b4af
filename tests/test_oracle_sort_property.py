"""Pinning of the sort restatement (oracle/sort_oracle.c) against the reference's own compiled sorter on 400 seeded examples drawn over
random sizes, ranges, partial sorts, index lists and all six distance branches: the reference's outputs are stored as digests
(tests/golden/sort_ref_digests.npz, written by tests/golden/make_ref_digests.py), the ordering properties are checked directly."""
import hashlib

import numpy as np

import cases

GOLD = np.load(cases.__file__.replace("cases.py", "golden/sort_ref_digests.npz"))
FIELDS = ("seed", "n", "integer", "mode", "kind", "frac", "rbits", "ties")


def test_port_equals_compiled_reference(oracle_mod):
    examples = [dict(zip(FIELDS, (v.item() for v in row))) for row in zip(*(GOLD[f"prop_{k}"] for k in FIELDS))]
    assert len(examples) == 400
    for ex, want_sha in zip(examples, GOLD["prop_sha"]):
        c, R = cases.property_case(**ex)
        args = cases.call_args(c, R)
        got, buckets = oracle_mod.port_sort_indexes(*args, want_buckets=True)
        rc, sc = c["render_count"], c["sort_count"]
        s0 = rc - sc
        # stored examples exclude the reference's undefined behaviour (every sorted distance equal: NaN bucket)
        assert sc == 0 or buckets[s0:rc].max() != buckets[s0:rc].min(), ex     # min and max distance always land in buckets 0 and R-1
        assert hashlib.sha256(got.tobytes()).digest() == bytes(want_sha), ex
        assert np.array_equal(np.sort(got), np.sort(c["indexes"][:rc]))           # a permutation of the input window
        assert np.array_equal(got[:s0], c["indexes"][:s0])                          # head copied through (sorter.cpp:158-160)
        if sc > 1:
            b = buckets[s0:rc]
            pos = {int(v): i for i, v in enumerate(c["indexes"][s0:rc])}
            seq = np.array([pos[int(v)] for v in got[s0:rc]])
            bs = b[seq]
            assert (np.diff(bs) <= 0).all(), ex                                     # buckets descending
            assert (np.diff(seq)[np.diff(bs) == 0] < 0).all(), ex                   # ties: later input positions first
