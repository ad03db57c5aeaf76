"""Filtered search (`MornaSearch.subset`, `FilteredSearch`): every route over a chosen subset of the rows equals the
parent's answer restricted to the subset -- top-k against the parent's full ordering (k = n) restricted and cut to k,
range lists against the parent's lists restricted, the approximate mode against an index built from the subset rows --
with equal ids (the parent's), order and distance bits."""
import io

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import synth
from tests.helpers import assert_lists_equal_oracle, tiny_lines

pytestmark = pytest.mark.gpu

K = 10


def make_search(S, **kw):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=S, stats=(S.shape[0], S.shape[0], S.shape[1]), **kw)


def pick_subset(n, which, seed):
    """Unsorted parent ids with repeats, as a user's list may come."""
    rng = np.random.default_rng(seed)
    ids = {"one": rng.choice(n, 1), "1%": rng.choice(n, max(1, n // 100), replace=False),
           "50%": rng.choice(n, n // 2, replace=False), "all_but_one": np.delete(np.arange(n), int(rng.integers(n))),
           "all": np.arange(n)}[which]
    return rng.permutation(np.concatenate([ids, ids[:3]]))


def host(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def restricted(full, members, k):
    """Each query's list of the parent's full ordering kept where the id is in `members`, cut to k, padded -1 / +inf."""
    f_i, f_d = host(full[0]), host(full[1])
    out_i = np.full((f_i.shape[0], k), -1, np.int32)
    out_d = np.full((f_i.shape[0], k), np.inf)
    keep = np.isin(f_i, members)
    for j in range(f_i.shape[0]):
        i, d = f_i[j][keep[j]][:k], f_d[j][keep[j]][:k]
        out_i[j, :len(i)], out_d[j, :len(i)] = i, d
    return out_i, out_d


def assert_same(got, want, label):
    gi, gd = host(got[0]), host(got[1])
    assert np.array_equal(gi, want[0]), "%s: ids differ" % label
    assert np.array_equal(gd.view(np.int64), want[1].view(np.int64)), "%s: distance bits differ" % label


def restrict_csr(csr, members):
    off, ids, d = (host(t) for t in csr)
    keep = np.isin(ids, members)
    query = np.repeat(np.arange(len(off) - 1), np.diff(off))
    new_off = np.zeros_like(off)
    np.cumsum(np.bincount(query[keep], minlength=len(off) - 1), out=new_off[1:])
    return new_off, ids[keep], d[keep]


def assert_csr_same(got, want, label):
    go, gi, gd = (host(t) for t in got)
    assert np.array_equal(go, want[0]), "%s: offsets differ" % label
    assert np.array_equal(gi, want[1]), "%s: ids differ" % label
    assert np.array_equal(gd.view(np.int64), want[2].view(np.int64)), "%s: distance bits differ" % label


def queries_of(S, nq, seed):
    qa, rows = synth.queries(S, nq // 2, seed=seed)
    qb, _ = synth.queries(S, nq - nq // 2, seed=seed + 1, noise=0.3)
    return torch.cat([qa, qb]).contiguous(), rows.cpu().numpy()


@pytest.fixture(scope="module", params=["gauss", "tissue"])
def idx(request):
    S = synth.matrix(request.param, 3000, 256, "cuda", seed=41)
    parent = make_search(S)
    Q, rows = queries_of(S, 96, seed=42)
    full = parent.exact_search_device(Q, S.shape[0])            # every row, in the reference order
    dist = full[1][:, 49]                                         # each query's 50th-nearest distance
    return {"kind": request.param, "S": S, "parent": parent, "Q": Q, "rows": rows, "full": full,
            "R": float(dist.median())}


@pytest.mark.parametrize("which", ["one", "1%", "50%", "all_but_one", "all"])
def test_topk_every_route_equals_the_restricted_full_ordering(idx, which):
    S, parent, Q, full = idx["S"], idx["parent"], idx["Q"], idx["full"]
    f = parent.subset(pick_subset(S.shape[0], which, seed=len(which)))
    members = f.member_ids
    assert np.all(np.diff(members) > 0) and f.inner.row_hi == len(members)
    want = restricted(full, members, K)
    label = "%s %s" % (idx["kind"], which)
    assert_same(f.batched_search_device(Q, K), want, label + " tensor-core batch")
    assert_same(f.exact_search_device(Q, K, allow_single=False), want, label + " FP64 scan")
    assert_same(f.exact_search_batch(host(Q), K), want, label + " host batch")
    assert_same(f.single_search_stream(Q[:6], K), (want[0][:6], want[1][:6]), label + " single-query stream")
    for j in (0, 60):
        one = (want[0][j:j + 1], want[1][j:j + 1])
        assert_same(f.single_search_device(Q[j], K), one, label + " single query, device")
        assert_same(f.exact_search_batch(host(Q[j:j + 1]), K), one, label + " single query, pinned host")
    got = list(f.search_batches([host(Q[:64]), host(Q[64:])], K))
    assert_same((np.concatenate([g[0] for g in got]), np.concatenate([g[1] for g in got])), want, label + " search_batches")
    # internal ids as queries: the stored rows, in or out of the subset
    rows = idx["rows"][:48]
    got = list(f.search_batches([rows[:20], rows[20:].astype(np.int32)], K))
    assert_same((np.concatenate([g[0] for g in got]), np.concatenate([g[1] for g in got])),
                (want[0][:48], want[1][:48]), label + " id batches")


def test_fewer_kept_rows_than_k_pad_like_a_small_index(idx):
    S, parent, Q = idx["S"], idx["parent"], idx["Q"]
    members = np.array([5, 17, 2999])
    f = parent.subset(members)
    small = make_search(S[torch.from_numpy(members).cuda()])
    for got, ref in ((f.batched_search_device(Q, K), small.batched_search_device(Q, K)),
                     (f.single_search_device(Q[3], K), small.single_search_device(Q[3], K))):
        ref_i = host(ref[0])
        assert (ref_i[:, 3:] == -1).all() and np.isinf(host(ref[1])[:, 3:]).all()
        assert_same(got, (np.where(ref_i >= 0, members[np.maximum(ref_i, 0)], -1).astype(np.int32), host(ref[1])), "padding")


def test_range_both_routes_equal_the_restricted_parent_lists(idx):
    S, parent, Q, R = idx["S"], idx["parent"], idx["Q"], idx["R"]
    f = parent.subset(pick_subset(S.shape[0], "50%", seed=3))
    want = restrict_csr(parent.range_search_device(Q, R), f.member_ids)
    assert_csr_same(f.range_search_device(Q, R), want, "tensor route")
    assert f.last_range_route == "tensor" and len(want[1]) > 0
    assert_csr_same(f.range_search_batch(host(Q), R), want, "host entry")
    f.inner.RANGE_TENSOR_MIN_QUERIES = 1 << 30
    assert_csr_same(f.range_search_device(Q, R), want, "FP64 route")
    assert f.last_range_route == "exact"
    groups = list(f.range_search_groups(Q, R, byte_cap=12 * 200))
    assert len(groups) > 1
    assert np.array_equal(np.concatenate([host(g[3]) for g in groups]), want[1])


def test_approximate_mode_equals_an_index_of_the_subset_rows(idx):
    S, parent, Q = idx["S"], idx["parent"], idx["Q"]
    members = np.sort(pick_subset(S.shape[0], "50%", seed=9))
    f = parent.subset(members)
    own = make_search(S[torch.from_numpy(f.member_ids).cuda()])
    ref_i, ref_d = (host(t) for t in own.approx_search_device(Q, K))
    assert (ref_i >= 0).all()
    assert_same(f.approx_search_device(Q, K), (f.member_ids[ref_i].astype(np.int32), ref_d), "approximate")


def test_topk_overflow_fix_up_under_a_filter():
    """A dense cluster of 3000 copies of one row: every list overflows into the exact scan, inside the subset too."""
    S = synth.gauss(8000, 128, "cuda", seed=9)
    S[:3000] = S[0]
    parent = make_search(S)
    Q = torch.cat([S[:40].double(), queries_of(S, 40, seed=4)[0]]).contiguous()
    full = parent.exact_search_device(Q, S.shape[0])
    members = pick_subset(S.shape[0], "50%", seed=11)
    f = parent.subset(members)
    want = restricted(full, f.member_ids, 100)
    assert_same(f.batched_search_device(Q, 100), want, "overflow")
    assert f.last_stats[0] >= 40
    got = list(f.search_batches([host(Q)], 100))
    assert_same(got[0], want, "overflow, search_batches")
    # ties across the map: equal distances come out by parent id descending
    kept_copies = f.member_ids[f.member_ids < 3000]
    assert np.array_equal(want[0][0], kept_copies[::-1][:100]) and not want[1][0].any()


def test_sparse_route_on_the_tiny_fixture():
    from oracle import morna_oracle as mo
    S = mo.go_index(tiny_lines(), features=3000, sample_threshold=100).matrix_f32()
    parent = make_search(S)
    rng = np.random.default_rng(5)
    f = parent.subset(rng.choice(S.shape[0], S.shape[0] // 2, replace=False))
    assert f.inner.csr is not None
    Q = torch.from_numpy(S[[0, 2040, 6595, 5, 4000, 17]].astype(np.float64)).cuda()
    want = restricted(parent.exact_search_device(Q, S.shape[0]), f.member_ids, 20)
    assert_same(f.exact_search_device(Q, 20), want, "sparse exact")
    assert_same(f.batched_search_device(Q, 20), want, "sparse batched")
    want_r = restrict_csr(parent.range_search_device(Q, 0.7), f.member_ids)
    assert_csr_same(f.range_search_device(Q, 0.7), want_r, "sparse range")


def test_query_outside_the_subset(idx):
    S, parent, Q, full = idx["S"], idx["parent"], idx["Q"], idx["full"]
    n = S.shape[0]
    row = int(idx["rows"][0])                                     # Q[0] is this stored row
    named = make_search(S, internal_id_map={1000 + i: i for i in range(n)})
    f = named.subset(np.delete(np.arange(n), [row, 7]))
    want = restricted((host(full[0])[:1], host(full[1])[:1]), f.member_ids, K)
    assert row not in want[0][0]
    got = f.search_member_n(1000 + row, K, out=io.StringIO())
    assert got[0] == want[0][0].tolist() and got[1] == want[1][0].tolist()
    assert_same(list(f.search_batches([np.array([row])], K))[0], want, "id batch outside the subset")
    g = named.subset(np.delete(np.arange(n), [row, 7]), keep_parent_rows=False)
    with pytest.raises(ValueError):
        g.stored_queries([row])
    assert torch.equal(g.stored_queries([8]), S[8:9].double())


def test_refuses_an_empty_or_foreign_subset(idx):
    parent = idx["parent"]
    for bad in ([], [-1], [3000]):
        with pytest.raises(ValueError):
            parent.subset(bad)


def test_50k_rows_half_subset_equals_the_oracle():
    n, d, nq, k = 50000, 3000, 4096, 100
    S = synth.gauss(n, d, "cuda")
    parent = make_search(S)
    Q, rows = queries_of(S, nq, seed=77)
    members = np.random.default_rng(12).choice(n, n // 2, replace=False)
    f = parent.subset(members, keep_parent_rows=False)
    del parent
    ids, dist = (host(t) for t in f.batched_search_device(Q, k))
    local = np.searchsorted(f.member_ids, ids)
    assert np.array_equal(f.member_ids[local], ids)
    inside = np.isin(rows, f.member_ids)                          # in-index queries whose row was kept find it first
    assert np.array_equal(ids[:nq // 2][inside, 0], rows[inside]) and not dist[:nq // 2][inside, 0].any()
    pick = np.concatenate([np.arange(0, nq // 2, 64), nq // 2 + np.arange(0, nq // 2, 64)])
    S_sub = S[torch.from_numpy(f.member_ids).cuda()].cpu().numpy()
    strict = assert_lists_equal_oracle(S_sub, host(Q)[pick], local[pick], dist[pick], k, "50% subset")
    assert strict > len(pick) * k // 2
