"""Within-group search (`MornaSearch.within_group_search` / `within_group_range`): both routes against brute force --
FP64 distances of all rows (morna_angular_distances), +inf where a row's label differs from the query's (or the query has
none) and on its excluded row, stably sorted under the reference order (distance ascending, equal distances id
descending) -- with equal ids and distance bits."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import synth
from tests.test_gpu_exclusion import all_distances, assert_csr_same, assert_same

pytestmark = pytest.mark.gpu

N, D = 50000, 3000


def make_search(S):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=S, stats=(S.shape[0], S.shape[0], S.shape[1]))


def S():
    """Rows of the largest group the grouped route takes (its shared-memory sort)."""
    from morna_b200.search import MornaSearch
    return MornaSearch.WITHIN_SEGMENT_ROWS


def P():
    """(queries of a group in one call) x (its rows) up to which the grouped route takes them."""
    from morna_b200.search import MornaSearch
    return MornaSearch.WITHIN_GROUPED_MAX_PAIRS


def grouping(name, n, seed=7):
    """int32 row labels: contiguous groups of 100, scattered groups of 10, or a mixed size distribution (one group of
    20,000 rows, groups of S - 1, S and S + 1 rows, singletons, random sizes, rows labelled -1) under arbitrary label
    values."""
    rng = np.random.default_rng(seed)
    if name == "contiguous100":
        return (np.arange(n) // 100 * 3 + 11).astype(np.int32)
    if name == "scattered10":
        return (rng.permutation(n) % (n // 10)).astype(np.int32)
    sizes = [20000, S() - 1, S(), S() + 1] + [1] * 300 + rng.integers(2, 400, 20).tolist()
    labels = np.full(n, -1, np.int64)
    perm, at = rng.permutation(n), 0
    values = np.arange(1, len(sizes) + 1, dtype=np.int64) * 2654435761 % (2 ** 31 - 1)       # distinct, arbitrary
    for size, v in zip(sizes, values):
        if at + size > n - 500:                           # (the last rows stay unlabelled)
            break
        labels[perm[at:at + size]] = v
        at += size
    return labels.astype(np.int32)


def brute(s, Q, qg, excl=None, member=None):
    """[nq x n] distances with +inf outside the query's group, on its excluded row and (member: bool [n]) off the subset."""
    dist = all_distances(s, Q)
    n = dist.shape[1]
    qg = torch.as_tensor(np.asarray(qg)).to(s.device).long()
    allowed = (s.row_group.long()[None, :] == qg[:, None]) & (qg[:, None] >= 0)
    if excl is not None:
        e = torch.as_tensor(np.asarray(excl)).to(s.device).long()
        allowed &= (torch.arange(n, device=s.device)[None, :] + s.row_lo) != e[:, None]
    if member is not None:
        allowed &= member[None, :]
    dist[~allowed] = float("inf")
    return dist


def ref_topk(dist, k, row_lo=0):
    n = dist.shape[1]
    kk = min(k, n)
    rows = (n - 1) - torch.sort(dist.flip(1), dim=1, stable=True).indices[:, :kk]
    d = dist.gather(1, rows)
    ids = torch.where(torch.isinf(d), -1, rows + row_lo).to(torch.int32)
    out_i = np.full((dist.shape[0], k), -1, np.int32)
    out_d = np.full((dist.shape[0], k), np.inf)
    out_i[:, :kk], out_d[:, :kk] = ids.cpu().numpy(), d.cpu().numpy()
    out_d[out_i < 0] = np.inf
    return out_i, out_d


def ref_range(dist, R, row_lo=0):
    dist = dist.cpu().numpy()
    off, ids, ds = [0], [], []
    for j in range(dist.shape[0]):
        rows = np.nonzero(dist[j] <= R)[0][::-1]
        rows = rows[np.argsort(dist[j][rows], kind="stable")]
        ids.append(rows + row_lo)
        ds.append(dist[j][rows])
        off.append(off[-1] + len(rows))
    return np.array(off), np.concatenate(ids).astype(np.int32), np.concatenate(ds)


@pytest.fixture(scope="module", params=["gauss", "tissue"])
def search(request):
    return make_search(synth.matrix(request.param, N, D, "cuda"))


def _case(s, name, nq=2048, seed=3):
    labels = grouping(name, N)
    s.set_row_groups(labels)
    rng = np.random.default_rng(seed)
    qid = np.sort(rng.choice(N, nq, replace=False)).astype(np.int64)
    excl = np.where(np.arange(nq) % 2 == 1, qid, -1).astype(np.int32)      # every other query leaves itself out
    return labels, qid, labels[qid], excl


@pytest.mark.parametrize("name", ["contiguous100", "scattered10", "mixed"])
@pytest.mark.parametrize("k", [1, 20, 100, 600])
def test_topk_equals_brute_force(search, name, k):
    s = search
    labels, qid, qg, excl = _case(s, name)
    Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
    want = ref_topk(brute(s, Q, qg, excl), k)
    assert_same(s.within_group_search(qid, k, qg, excl), want, "%s k=%d by id" % (name, k))
    grouped, large = s.last_within_routes
    if name == "mixed":                          # (the groups of 8,192 rows and more get hundreds of queries each)
        assert grouped > 0 and large > 0
    else:                                        # small groups: the grouped kernels answer every query
        assert (grouped, large) == (len(qid), 0)
    assert_same(s.within_group_search(Q, k, qg, excl), want, "%s k=%d by vector" % (name, k))


@pytest.mark.parametrize("name", ["contiguous100", "scattered10", "mixed"])
def test_range_equals_brute_force(search, name):
    s = search
    labels, qid, qg, excl = _case(s, name, nq=1024)
    Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
    dist = brute(s, Q, qg, excl)
    first = torch.sort(dist, dim=1).values[:, :100]          # the 100th nearest within the group, or its farthest
    last = torch.where(torch.isfinite(first), first, float("-inf")).max(dim=1).values
    R = float(torch.median(last[torch.isfinite(last)]))
    for r in (R, 0.0, 1.5):
        got = s.within_group_range(qid, r, qg, excl)
        assert_csr_same(got, ref_range(dist, r), "%s R=%r" % (name, r))
    assert_csr_same(s.within_group_range(Q, R, qg, excl), ref_range(dist, R), "%s by vector" % name)


def test_labels_without_rows_give_empty_lists(search):
    s = search
    labels, qid, qg, excl = _case(s, "mixed", nq=256)
    qg = qg.copy()
    qg[::3] = -1                                           # no group
    qg[1::3] = 2 ** 31 - 1 if (labels != 2 ** 31 - 1).all() else -5        # a label no row carries
    Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
    dist = brute(s, Q, qg, excl)
    assert_same(s.within_group_search(qid, 20, qg, excl), ref_topk(dist, 20), "absent labels")
    assert_csr_same(s.within_group_range(qid, 1.5, qg, excl), ref_range(dist, 1.5), "absent labels, range")
    ids, _ = s.within_group_search(qid, 20, qg, excl)
    assert (ids[::3] < 0).all()
    ids, _ = s.within_group_search(qid[:0], 20, qg[:0])
    assert ids.shape == (0, 20)


@pytest.mark.parametrize("m", [1, 7, 8, 9])
def test_group_query_counts_around_a_tile(search, m):
    """Exactly m queries of one group (QB = 8 per work item) in a call, on groups of S rows (the largest segment the
    grouped route sorts), S + 1 rows (the tensor-core route) and about 100 rows."""
    s = search
    labels = grouping("mixed", N)
    s.set_row_groups(labels)
    vals, counts = np.unique(labels[labels >= 0], return_counts=True)
    for size in (S(), S() + 1, 100):
        g = vals[np.argmin(np.abs(counts - size))]
        rows = np.nonzero(labels == g)[0]
        qid = rows[np.linspace(0, len(rows) - 1, m).astype(np.int64)].astype(np.int64)
        qg = labels[qid]
        excl = np.where(np.arange(m) == 0, qid, -1).astype(np.int32)
        Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
        dist = brute(s, Q, qg, excl)
        assert_same(s.within_group_search(qid, 50, qg, excl), ref_topk(dist, 50), "m=%d size=%d" % (m, size))
        assert s.last_within_routes == ((m, 0) if len(rows) <= S() else (0, m)), (m, len(rows), s.last_within_routes)


def test_pair_count_picks_the_route(search):
    """A group's queries in one call go to the grouped route up to P (queries x rows) and to the tensor-core route past
    it, scattered or contiguous, with the same answers."""
    s = search
    g = int(np.sqrt(P())) + 1                          # g * g > P >= (P // g) * g
    rng = np.random.default_rng(4)
    for labels in ((np.arange(N) // g).astype(np.int32), (rng.permutation(N) // g).astype(np.int32)):
        s.set_row_groups(labels)
        rows = np.nonzero(labels == 0)[0]
        for nq, route in ((len(rows), (0, len(rows))), (P() // g, (P() // g, 0))):
            qid = np.sort(rng.choice(rows, nq, replace=False)).astype(np.int64)
            qg, excl = labels[qid], qid.astype(np.int32)
            Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
            dist = brute(s, Q, qg, excl)
            assert_same(s.within_group_search(qid, 30, qg, excl), ref_topk(dist, 30), "nq=%d" % nq)
            assert s.last_within_routes == route
            assert_csr_same(s.within_group_range(qid, 1.4, qg, excl), ref_range(dist, 1.4), "nq=%d range" % nq)
            assert s.last_within_routes == route


def test_filtered_search(search):
    s = search
    labels = grouping("mixed", N)
    s.set_row_groups(labels)
    rng = np.random.default_rng(9)
    keep = np.sort(rng.choice(N, N // 2, replace=False))
    f = s.subset(keep)
    qid = np.sort(rng.choice(N, 1024, replace=False)).astype(np.int64)     # in and out of the subset
    qg = labels[qid]
    excl = qid.astype(np.int32)
    member = torch.zeros(N, dtype=torch.bool, device="cuda")
    member[torch.from_numpy(keep).cuda()] = True
    Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
    dist = brute(s, Q, qg, excl, member)
    for k in (20, 600):
        assert_same(f.within_group_search(qid, k, qg, excl), ref_topk(dist, k), "filtered k=%d" % k)
    assert_csr_same(f.within_group_range(Q, 1.0, qg, excl), ref_range(dist, 1.0), "filtered range")


@pytest.mark.parametrize("dim", [10000, 30000])
def test_wide_features(dim):
    S = synth.gauss(3000, dim, "cuda", seed=5)
    s = make_search(S)
    labels = np.concatenate([np.arange(2000) // 50, np.full(1000, 999)]).astype(np.int32)   # groups of 50 and of 1,000
    s.set_row_groups(labels)
    qid = np.arange(0, 3000, 7, dtype=np.int64)
    qg, excl = labels[qid], np.where(qid % 2 == 0, qid, -1).astype(np.int32)
    Q = s.vectors[torch.from_numpy(qid).cuda(), :dim].double()
    dist = brute(s, Q, qg, excl)
    assert_same(s.within_group_search(qid, 30, qg, excl), ref_topk(dist, 30), "D=%d" % dim)
    assert_csr_same(s.within_group_range(qid, 1.39, qg, excl), ref_range(dist, 1.39), "D=%d range" % dim)


def test_labels_change_with_set_row_groups(search):
    s = search
    qid = np.arange(0, N, 97, dtype=np.int64)
    for name in ("contiguous100", "mixed"):
        labels = grouping(name, N)
        s.set_row_groups(labels)
        Q = s.vectors[torch.from_numpy(qid).cuda(), :D].double()
        assert_same(s.within_group_search(qid, 20, labels[qid]), ref_topk(brute(s, Q, labels[qid]), 20), name)
    s.set_row_groups(None)
    with pytest.raises(ValueError, match="set_row_groups"):
        s.within_group_search(qid, 20, np.zeros(len(qid), np.int32))
