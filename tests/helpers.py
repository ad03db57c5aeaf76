"""Shared checks for parity tests."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_reference_vectors():
    with open(os.path.join(GOLDEN, "reference_unittest_vectors.json")) as fh:
        return json.load(fh)


def tiny_lines():
    with open(os.path.join(GOLDEN, "tiny_intropolis.tsv")) as fh:
        return fh.readlines()


def check_topk(true_d, ids, dists=None, tol=1e-9, dist_tol=1e-5):
    """"Identical neighbour ids, ties aside": `ids` is a valid exact top-k list
    for the full true-distance array `true_d` if the ids are distinct and the
    r-th returned row's true distance equals the r-th smallest true distance to
    within `tol`.  Reported distances must sit within `dist_tol` of the truth.
    """
    true_d = np.asarray(true_d, dtype=np.float64)
    ids = np.asarray(ids, dtype=np.int64)
    assert len(set(ids.tolist())) == len(ids), "duplicate ids in result"
    assert ids.min() >= 0 and ids.max() < len(true_d)
    want = np.sort(true_d)[: len(ids)]
    got = true_d[ids]
    bad = np.nonzero(np.abs(got - want) > tol)[0]
    assert bad.size == 0, "rank %d: id %d has true distance %r, expected %r" % (
        bad[0], ids[bad[0]], got[bad[0]], want[bad[0]])
    if dists is not None:
        dists = np.asarray(dists, dtype=np.float64)
        err = np.abs(dists - got)
        assert err.max() <= dist_tol, "distance off by %g at rank %d" % (err.max(), err.argmax())


def check_order_rule(ids, dists):
    """Within the returned list: distance ascending, equal distances id descending."""
    ids = np.asarray(ids, dtype=np.int64)
    dists = np.asarray(dists, dtype=np.float64)
    assert np.all(np.diff(dists) >= 0), "distances not ascending"
    same = np.diff(dists) == 0
    assert np.all(np.diff(ids)[same] < 0), "equal distances must be id-descending"


def assert_lists_equal_oracle(S_host, Q_host, ids, dists, k, label):
    """ids/dists: numpy [nq x k] from the CUDA path; the oracle answers the same queries on the host."""
    from oracle import c_oracle
    want_i, want_d = c_oracle.exact_search_batch(S_host, Q_host, k, n_threads=os.cpu_count() or 1)
    strict = 0
    for j in range(Q_host.shape[0]):
        true_d = c_oracle.distances(S_host, Q_host[j])
        check_topk(true_d, ids[j], dists[j], tol=1e-9, dist_tol=1e-9)
        check_order_rule(ids[j], dists[j])
        # positions whose oracle distance is isolated from both neighbours by more than the rounding of a
        # 3000-term FP64 sum must carry the oracle's id
        wd = want_d[j]
        gap_lo = np.concatenate([[np.inf], np.diff(wd)])
        gap_hi = np.concatenate([np.diff(wd), [np.inf]])
        iso = (gap_lo > 1e-9) & (gap_hi > 1e-9)
        iso[-1] = False                      # the k-th place may be contested by the (k+1)-th row
        assert np.array_equal(ids[j][iso], want_i[j][iso]), "%s: query %d ids differ from the oracle's" % (label, j)
        assert np.abs(dists[j] - wd).max() <= 1e-9, "%s: query %d distances differ from the oracle's" % (label, j)
        strict += int(iso.sum())
    return strict
