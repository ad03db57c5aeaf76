"""Pins the CPU oracle: reference unit-test vectors, hash known answers, fixture KATs."""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import c_oracle
from oracle import morna_oracle as mo
from tests.helpers import GOLDEN, check_order_rule, check_topk, load_reference_vectors, tiny_lines


def test_murmur3_known_answers():
    # published / sklearn-verified answers (SURVEY.md 8c)
    kats = {"": 0, "foo": -156908512, "hello": 613153351, "1": -1810453357,
            "21504": 919914018, "chr1 14830 14929": -28859081,
            "chr1 14830 14969": 1028464060, "chr1 15039 15795": 938554306}
    for key, want in kats.items():
        assert mo.murmur3_x86_32(key) == want
        assert c_oracle.murmur3_32(key) == want


def test_murmur3_matches_sklearn_on_random_keys():
    # sklearn.utils.murmurhash3_32's answers on 300 random keys, stored by tests/golden/make_golden.py
    with open(os.path.join(GOLDEN, "murmur3_sklearn_vectors.json")) as fh:
        cases = json.load(fh)["cases"]
    assert len(cases) == 300
    for key, want in cases:
        key = key.encode("ascii")
        assert mo.murmur3_x86_32(key) == want
        assert c_oracle.murmur3_32(key) == want


def test_floor_mod_bucket_and_sign():
    h, b, s = mo.bucket_and_sign("chr1 14830 14929", 3000)
    assert (h, b, s) == (-28859081, 919, -1)
    raw, bucket, sign = c_oracle.hash_rows(["chr1 14830 14929", "chr1 14830 14969"], 3000)
    assert raw.tolist() == [-28859081, 1028464060]
    assert bucket.tolist() == [919, 1060] and sign.tolist() == [-1, 1]


@pytest.mark.parametrize("case_no", [0, 1, 2])
def test_reference_unittest_neighbour_lists(case_no):
    """morna.py:1176-1187 / 1267-1278 / 1312-1323: the oracle's exact kNN order
    reproduces every golden list, ties aside."""
    vec = load_reference_vectors()
    case = vec["cases"][case_no]
    lines = [l + "\n" for l in vec[case["input"]]]
    if "count_samples" in case:
        assert mo.count_samples(lines) == case["count_samples"]      # morna.py:1149
    idx = mo.go_index(lines, features=case["features"], sample_count=case["sample_count"],
                      sample_threshold=case["sample_threshold"])
    S = idx.matrix_f32()
    assert S.shape[0] == case["n_items"]                              # :1174/:1265/:1310
    for i, expected in enumerate(case["expected"]):
        true_d = np.array([mo.cosine_distance(S[j].tolist(), S[i].tolist(), clamp=True)
                           for j in range(S.shape[0])])
        check_topk(true_d, expected, tol=1e-7)       # Annoy's float32 ties == our ties
        ids, d = mo.exact_search_nn(S, S[i], len(expected), clamp=True)
        check_topk(true_d, ids, d, tol=0.0, dist_tol=0.0)
        check_order_rule(ids, d)
        ids_c, d_c = c_oracle.exact_search(S, S[i].astype(np.float64), len(expected))
        assert ids_c.tolist() == ids and d_c.tolist() == d


def test_lossy_id_map_is_first_seen_order():
    vec = load_reference_vectors()
    lines = [l + "\n" for l in vec["lossy_input"]]
    idx = mo.go_index(lines, features=3000, sample_count=10, sample_threshold=4)
    assert idx.internal_id_map == {10: 0, 9: 1, 8: 2, 7: 3, 6: 4, 5: 5, 4: 6, 3: 7, 2: 8, 1: 9}


def test_tie_rule_later_row_first():
    S = np.zeros((6, 8), np.float32)
    S[1, 0] = 1.0; S[3, 0] = 2.0; S[5, 0] = 0.5      # three parallel rows
    S[0, 1] = 1.0; S[2, 2] = 1.0; S[4, 3] = 1.0
    q = np.zeros(8); q[0] = 3.0
    ids, d = mo.exact_search_nn(S, q, 3)
    assert ids == [5, 3, 1] and d == [0.0, 0.0, 0.0]


def test_unclamped_distance_raises_like_reference():
    # a radicand that rounds negative -> math domain error in the reference
    v = np.array([0.1, 0.2, 0.3], np.float32)
    found = False
    rng = np.random.default_rng(0)
    for _ in range(2000):
        v = rng.standard_normal(7).astype(np.float32)
        q = (v.astype(np.float64) * 3.0).tolist()
        try:
            mo.cosine_distance(v.tolist(), q)
        except ValueError:
            found = True
            assert mo.cosine_distance(v.tolist(), q, clamp=True) == 0.0
            break
    assert found


def test_tiny_fixture_kats():
    with open(os.path.join(GOLDEN, "tiny_expected.json")) as fh:
        exp = json.load(fh)
    lines = tiny_lines()
    assert mo.count_samples(lines) == exp["count_samples"] == 6850
    idx = mo.go_index(lines, features=3000, sample_threshold=100)
    assert idx.new_internal_id == exp["n_kept"]
    for row, (h, b, s, idf) in zip(exp["rows"], idx.row_trace):
        assert (row["hash"], row["bucket"], row["sign"], row["idf"]) == (h, b, s, idf)
    for sid, internal in exp["id_map_spot"].items():
        assert idx.internal_id_map[int(sid)] == internal
    S = idx.matrix_f32()
    assert hashlib.sha256(np.ascontiguousarray(S).tobytes()).hexdigest() == exp["matrix_f32_sha256"]
    m64 = idx.matrix_f64()
    assert m64[0, 919] == -1.2112988444180088 and m64[0, 1060] == 0.5885265379724792
    assert m64[2040, 1060] == 0.39235102531498617
    q0 = exp["queries"][0]
    ids, d = c_oracle.exact_search(S, S[q0["internal_id"]].astype(np.float64), 20)
    assert ids.tolist() == q0["ids"] and d.tolist() == q0["dists"]


def test_c_oracle_bit_identical_to_python_oracle():
    rng = np.random.default_rng(11)
    S = rng.standard_normal((300, 257)).astype(np.float32)
    S[7] = S[3]; S[50] = 2 * S[3]; S[9] = 0
    for qi in (3, 9, 100):
        q = S[qi].astype(np.float64)
        ids, d = mo.exact_search_nn(S, q, 25, clamp=True)
        ids_c, d_c = c_oracle.exact_search(S, q, 25)
        assert ids == ids_c.tolist() and d == d_c.tolist()
    q = rng.standard_normal(257)
    full = c_oracle.distances(S, q)
    assert full.tolist() == [mo.cosine_distance(S[i].tolist(), q.tolist(), clamp=True)
                             for i in range(300)]
    np.testing.assert_allclose(mo.distances_np(S, q), full, rtol=0, atol=1e-12)
    ids_b, d_b = c_oracle.exact_search_batch(S, np.stack([S[3].astype(np.float64), q]), 25, 2)
    assert ids_b[1].tolist() == c_oracle.exact_search(S, q, 25)[0].tolist()


def test_c_oracle_index_accumulate_matches_python():
    vec = load_reference_vectors()
    lines = [l + "\n" for l in vec["lossy_input"]] + tiny_lines()[:1]
    idx = mo.go_index(lines, features=97, sample_count=50, sample_threshold=2)
    keys, row_off, samples, covs, passing, idf = [], [0], [], [], [], []
    freq = {}
    for line in lines:
        key, s, c = mo.tokenize_line(line)
        keys.append(key); samples += s; covs += c; row_off.append(len(samples))
        ok = len(s) >= 2
        passing.append(ok)
        if ok:
            freq[key] = freq.get(key, 0) + len(s)
            import math
            idf.append(math.log(50.0 / freq[key]))
        else:
            idf.append(0.0)
    raw, bucket, sign = c_oracle.hash_rows(keys, 97)
    id_of, n_kept, acc = c_oracle.index_accumulate(row_off, passing, bucket, sign, idf,
                                                   samples, covs, 97, max(samples), len(set(samples)))
    assert n_kept == idx.new_internal_id
    assert {s: int(id_of[s]) for s in idx.internal_id_map} == idx.internal_id_map
    assert np.array_equal(acc, idx.matrix_f64())


def test_py2_float_format():
    assert mo.py2_str(0.0) == "0.0" and mo.py2_str(1.0) == "1.0"
    assert mo.py2_str(1.4142135623730951) == "1.41421356237"
    assert mo.py2_str(1e-05) == "1e-05" and mo.py2_str(7) == "7"
    assert mo.format_results(([3, 1], [0.0, 0.5])) == "1.\t3\t0.0\n2.\t1\t0.5\n"
