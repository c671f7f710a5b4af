"""Generates tests/golden/sort_ref_digests.npz: SHA-256 digests of what the REFERENCE's own compiled sorter (oracle/_ref, built by
oracle/Makefile from the reference's src/worker/sorter*.cpp) returns on the inputs of tests/test_oracle_sort.py and
tests/test_oracle_sort_property.py, so that those tests compare the C restatement with the reference on machines that cannot build it.
Run where the reference sources are present:   python tests/golden/make_ref_digests.py
Inputs are regenerated from seeds; only the arguments and one digest per output are stored.

  cref_keys, cref_sha  "<name>|R<R>": sortIndexes() output for cases.sort_matrix(n=20000, seeds=(0, 1)) at each of cases.RANGES;
                       "<name>|simd": the SIMD spelling (sorter.cpp) at R = 2^16, integer cases only
  prop_*               PROPERTY_CASES seeded examples over the ranges of the former property-based draw (sizes 2..400, every
                       distance branch, index kind, partial sort and 1..16-bit range), with their output digests in prop_sha"""
import hashlib
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import cases  # noqa: E402
import oracle  # noqa: E402

PROPERTY_CASES = 400
PROPERTY_SEED = 20240917


def digest(out: np.ndarray) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(out, np.uint32).tobytes()).digest(), np.uint8)


def property_examples():
    """Seeded draws over the argument ranges of test_port_equals_compiled_reference; examples whose sorted distances are all equal are
    dropped (the reference's bucket is NaN there: undefined behaviour the restatement defines instead)."""
    rng = np.random.default_rng(PROPERTY_SEED)
    rows = []
    while len(rows) < PROPERTY_CASES:
        row = dict(seed=int(rng.integers(0, 2**31)), n=int(rng.integers(2, 401)), integer=bool(rng.integers(2)),
                   mode=str(rng.choice(["static", "dynamic", "precomputed"])), kind=str(rng.choice(["identity", "shuffled", "octree"])),
                   frac=float(rng.choice([1.0, 0.5, 0.1, 0.0])), rbits=int(rng.integers(1, 17)), ties=bool(rng.integers(2)))
        c, R = cases.property_case(**row)
        _, buckets = oracle.port_sort_indexes(*cases.call_args(c, R), want_buckets=True)
        rc, sc = c["render_count"], c["sort_count"]
        if sc and buckets[rc - sc:rc].max() == buckets[rc - sc:rc].min():
            continue
        row["sha"] = digest(oracle.ref_sort_indexes(*cases.call_args(c, R)))
        rows.append(row)
    return rows


def main():
    oracle.build()
    assert oracle.have_ref(), "oracle/_ref missing: needs the reference sources (oracle/Makefile REF=...)"
    keys, shas = [], []
    for name, kw in cases.sort_matrix(n=20000, seeds=(0, 1)):
        c = cases.sort_case(**kw)
        for R in cases.RANGES:
            keys.append(f"{name}|R{R}")
            shas.append(digest(oracle.ref_sort_indexes(*cases.call_args(c, R))))
        if c["integer_sort"]:
            keys.append(f"{name}|simd")
            shas.append(digest(oracle.ref_sort_indexes(*cases.call_args(c, 1 << 16), simd=True)))
    store = {"cref_keys": np.array(keys), "cref_sha": np.stack(shas)}
    rows = property_examples()
    for k in ("seed", "n", "integer", "mode", "kind", "frac", "rbits", "ties", "sha"):
        store[f"prop_{k}"] = np.array([r[k] for r in rows])
    np.savez_compressed(ROOT / "tests" / "golden" / "sort_ref_digests.npz", **store)
    print(f"wrote {len(keys)} sort_matrix digests and {len(rows)} property examples")


if __name__ == "__main__":
    main()
