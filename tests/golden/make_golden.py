"""Regenerates tests/golden/tiny_expected.json from the CPU oracle.

The reference itself cannot run here (Python 2 + mmh3 + annoy, none installed),
so these are ORACLE outputs on the reference's fixture tests/tiny_intropolis.tsv,
not reference outputs.  The oracle is pinned separately against the reference's
own embedded unit-test vectors (reference_unittest_vectors.json).
It also writes murmur3_sklearn_vectors.json: random keys and the hashes
sklearn.utils.murmurhash3_32 gives them (the reference hashes with mmh3, which
agrees with sklearn), so the hash check runs without scikit-learn installed.
Run:  python tests/golden/make_golden.py   (needs scikit-learn)
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import morna_oracle as mo  # noqa: E402
from oracle import c_oracle  # noqa: E402


def main():
    lines = open(os.path.join(HERE, "tiny_intropolis.tsv")).readlines()
    idx = mo.go_index(lines, features=3000, sample_count=None, sample_threshold=100)
    S = idx.matrix_f32()
    out = {
        "features": 3000, "sample_threshold": 100,
        "count_samples": idx.sample_count,
        "n_kept": idx.new_internal_id,
        "rows": [],
        "id_map_spot": {str(s): idx.internal_id_map[s] for s in (12, 1, 21504)},
        "id_map_sha256": hashlib.sha256(json.dumps(
            sorted(idx.internal_id_map.items())).encode()).hexdigest(),
        "matrix_f32_sha256": hashlib.sha256(np.ascontiguousarray(S).tobytes()).hexdigest(),
        "abs_sum_f64": float(np.abs(idx.matrix_f64()).sum()),
        "nnz_per_row_hist": {str(k): int(v) for k, v in zip(
            *np.unique((S != 0).sum(axis=1), return_counts=True))},
        "queries": [],
    }
    for line, (h, b, s, idf) in zip(lines, idx.row_trace):
        key, samples, _ = mo.tokenize_line(line)
        out["rows"].append({"key": key, "hash": h, "bucket": b, "sign": s,
                            "n_samples": len(samples), "idf": idf})
    for sample_id in (12, 1, 21504, 33, 5000):
        if sample_id not in idx.internal_id_map:
            continue
        internal = idx.internal_id_map[sample_id]
        ids, d = c_oracle.exact_search(S, S[internal].astype(np.float64), 20)
        ids_py, d_py = mo.exact_search_nn(S[:400], S[internal], 20, clamp=True)
        ids_c400, d_c400 = c_oracle.exact_search(S[:400], S[internal].astype(np.float64), 20)
        assert ids_py == ids_c400.tolist() and d_py == d_c400.tolist()
        out["queries"].append({"sample_id": sample_id, "internal_id": internal,
                               "ids": ids.tolist(), "dists": d.tolist()})
    with open(os.path.join(HERE, "tiny_expected.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote tiny_expected.json; n_kept", out["n_kept"], "sha", out["matrix_f32_sha256"])
    write_murmur3_vectors()


def write_murmur3_vectors():
    from sklearn.utils import murmurhash3_32
    rng = np.random.default_rng(5)
    keys = []
    for _ in range(300):
        n = int(rng.integers(0, 40))
        keys.append(bytes(rng.integers(32, 127, size=n, dtype=np.uint8)).decode("ascii"))
    out = {"source": "sklearn.utils.murmurhash3_32(key, seed=0, positive=False) on the ASCII bytes of key",
           "cases": [[key, int(murmurhash3_32(key.encode("ascii"), seed=0, positive=False))] for key in keys]}
    with open(os.path.join(HERE, "murmur3_sklearn_vectors.json"), "w") as fh:
        json.dump(out, fh, indent=0)
    print("wrote murmur3_sklearn_vectors.json;", len(keys), "keys")


if __name__ == "__main__":
    main()
