"""Group-capped search (`MornaSearch.set_cap_groups` + `max_per_group=`): every route equals the walk over the brute-force
list -- FP64 distances of all rows (morna_angular_distances), excluded pairs at +inf, stably sorted under the reference
order, each row kept iff fewer than N rows of its cap label were kept before it, cut to k -- with equal ids and distance
bits."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import _lib, synth
from tests.helpers import tiny_lines
from tests.test_gpu_exclusion import assert_csr_same, assert_same, host, make_search, masked_distances

pytestmark = pytest.mark.gpu

N, D = 50000, 3000


def walk(rows, d, caps, m, k=None):
    """The capped walk over one list in the reference order (numpy): positions kept."""
    lab = caps[rows]
    order = np.argsort(lab, kind="stable")
    sl = lab[order]
    start = np.r_[0, np.flatnonzero(sl[1:] != sl[:-1]) + 1] if len(sl) else np.zeros(0, np.int64)
    run = np.repeat(start, np.diff(np.r_[start, len(sl)]))
    rank = np.empty(len(rows), np.int64)
    rank[order] = np.arange(len(sl)) - run
    keep = np.flatnonzero((lab < 0) | (rank < m))
    return keep if k is None else keep[:k]


def reference(s, Q, k, m, qg=None, allowed=None):
    """Brute-force capped top-k: host (ids [nq x k], dists [nq x k]).  `allowed`: bool [n] (a subset), else every row."""
    dist = masked_distances(s, Q, qg)
    if allowed is not None:
        dist[:, ~torch.as_tensor(allowed, device=s.device)] = float("inf")
    n = dist.shape[1]
    rows = (n - 1) - torch.sort(dist.flip(1), dim=1, stable=True).indices
    d = dist.gather(1, rows).cpu().numpy()
    rows = rows.cpu().numpy()
    caps = host(s.cap_group)
    out_i = np.full((Q.shape[0], k), -1, np.int32)
    out_d = np.full((Q.shape[0], k), np.inf)
    for j in range(Q.shape[0]):
        fin = np.isfinite(d[j])
        keep = walk(rows[j][fin], d[j][fin], caps, m, k)
        out_i[j, :len(keep)] = rows[j][fin][keep] + s.row_lo
        out_d[j, :len(keep)] = d[j][fin][keep]
    return out_i, out_d


def cap_labels(kind, n, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "ungrouped":
        return np.full(n, -1, np.int32)
    if kind == "all_but_60":
        g = np.full(n, 3, np.int32)
        g[rng.choice(n, 60, replace=False)] = -1
        return g
    if kind == "g10_scattered":
        return rng.permutation(np.arange(n) // 10).astype(np.int32)
    return (np.arange(n) // int(kind[1:])).astype(np.int32)           # "g100", "g1000": contiguous


@pytest.fixture(scope="module", params=["gauss", "tissue"])
def idx(request):
    S = synth.matrix(request.param, N, D, "cuda", seed=7)
    return request.param, make_search(S)


def queries(s, nq, seed):
    """In-index queries, every third one with noise (out of the index)."""
    Q, rows = synth.queries(s.vectors[:, :s.dim], nq, seed=seed)
    Q[::3] += 0.02 * Q[::3].abs().mean() * torch.randn_like(Q[::3])
    return Q.contiguous(), rows


@pytest.mark.parametrize("grouping", ["g100", "g1000", "g10_scattered", "all_but_60"])
def test_capped_top_k_equals_the_walk(idx, grouping):
    """Every case stays on the tensor cores (no query overflows to the FP64 route), also where the pilot block holds fewer
    than k capped entries (N = 1 with groups of 100, groups of 1,000, one huge group): those rows are scored in lead blocks
    with a capped refinement after each."""
    kind, s = idx
    s.set_cap_groups(cap_labels(grouping, N))
    Q, _ = queries(s, 96, seed=3)
    for m in (1, 2, 5):
        for k in (1, 20, 100, 512):
            want = reference(s, Q, k, m)
            label = "%s/%s N=%d k=%d" % (kind, grouping, m, k)
            assert_same(s.batched_search_device(Q, k, max_per_group=m), want, label)
            assert s.last_stats[0] == 0, "%s: %d queries overflowed" % (label, s.last_stats[0])
    assert_same(s.exact_search_device(Q[:3], 20, max_per_group=2), reference(s, Q[:3], 20, 2), "%s/%s -q" % (kind, grouping))


def test_no_cap_equals_the_uncapped_search(idx):
    kind, s = idx
    Q, _ = queries(s, 128, seed=5)
    plain = tuple(host(t) for t in s.batched_search_device(Q, 100))
    s.set_cap_groups(cap_labels("ungrouped", N))
    assert_same(s.batched_search_device(Q, 100, max_per_group=1), plain, "%s ungrouped" % kind)
    s.set_cap_groups(cap_labels("g1000", N))
    assert_same(s.batched_search_device(Q, 100, max_per_group=1000), plain, "%s N >= largest group" % kind)


def test_with_exclusion_and_through_a_filtered_search(idx):
    kind, s = idx
    s.set_cap_groups(cap_labels("g100", N))
    s.set_row_groups(cap_labels("g10_scattered", N, seed=4))
    Q, rows = queries(s, 128, seed=9)
    qg = s.row_group[rows].clone()
    qg[::5] = -1
    assert_same(s.batched_search_device(Q, 50, query_groups=qg, max_per_group=2), reference(s, Q, 50, 2, qg),
                "%s exclusion" % kind)
    members = np.arange(0, N, 3)
    f = s.subset(members)
    allowed = np.zeros(N, bool)
    allowed[members] = True
    assert_same(f.batched_search_device(Q, 50, max_per_group=1), reference(s, Q, 50, 1, allowed=allowed), "%s subset" % kind)
    fq = f.row_groups_of(rows)
    assert_same(f.batched_search_device(Q, 50, query_groups=fq, max_per_group=2),
                reference(s, Q, 50, 2, fq, allowed=allowed), "%s subset + exclusion" % kind)
    s.set_row_groups(None)


def test_small_row_blocks_run_the_capped_refinements(idx):
    kind, s = idx
    s.set_cap_groups(cap_labels("g100", N))
    Q, _ = queries(s, 128, seed=13)
    lib = s.lib
    try:
        # key 9 = 4096 rows per block, and the pilot block is never larger than a block: a 4096-row pilot, then the
        # capped block schedule (2048-row blocks while the prefix holds few capped entries), a refinement after each
        assert lib.morna_debug_set_tuning(9, 4096) == 0
        for m, k in ((1, 100), (2, 512), (5, 20), (2, 100)):
            assert_same(s.batched_search_device(Q, k, max_per_group=m), reference(s, Q, k, m), "%s blocks N=%d" % (kind, m))
            assert s.last_stats[0] == 0, "%s blocks N=%d: %d queries overflowed" % (kind, m, s.last_stats[0])
    finally:
        lib.morna_debug_set_tuning(9, 131072)


def test_block_schedule_does_not_change_results(idx, monkeypatch):
    """The capped block schedule only keeps lists short: with the usual blocks (no ends) the same queries overflow to the
    FP64 route and give the same bits; with 2048-row blocks throughout the tensor route gives them too."""
    kind, s = idx
    s.set_cap_groups(cap_labels("g100", N))
    Q, _ = queries(s, 64, seed=21)
    want = reference(s, Q, 100, 1)
    for ends, over in ((np.zeros(0, np.int64), 64), (np.arange(2048, N + 2048, 2048).clip(max=N), 0)):
        monkeypatch.setattr(s, "_cap_blocks", lambda m, k: ends)
        assert_same(s.batched_search_device(Q, 100, max_per_group=1), want, "%s %d block ends" % (kind, ends.size))
        assert s.last_stats[0] == over, (ends.size, s.last_stats)


def test_search_batches_range_and_fp64_route(idx):
    kind, s = idx
    s.set_cap_groups(cap_labels("g100", N))
    ids = np.random.default_rng(2).choice(N, 600, replace=False)
    got = list(s.search_batches(iter([ids[:300], ids[300:]]), 20, max_per_group=2))
    for b, (gi, gd) in zip((ids[:300], ids[300:]), got):
        Q = s.vectors[torch.from_numpy(b).cuda(), :D].to(torch.float64)
        assert_same((gi, gd), reference(s, Q, 20, 2), "%s search_batches" % kind)
    Q, _ = queries(s, 80, seed=17)
    assert_same(s.exact_search_device(Q[:6], 1500, max_per_group=3), reference(s, Q[:6], 1500, 3), "%s k > 512" % kind)
    R = float(host(s.exact_search_device(Q[:8], 200)[1])[:, 150].mean())
    caps = host(s.cap_group)
    for q, route in ((Q, "tensor"), (Q[:10], "exact")):
        off, ids_, d = (host(t) for t in s.range_search_device(q, R))
        want_off, want_i, want_d = [0], [], []
        for j in range(q.shape[0]):
            li, ld = ids_[off[j]:off[j + 1]], d[off[j]:off[j + 1]]
            keep = walk(li, ld, caps, 2)
            want_i.append(li[keep]); want_d.append(ld[keep]); want_off.append(want_off[-1] + len(keep))
        got = s.range_search_device(q, R, max_per_group=2)
        assert s.last_range_route == route
        assert_csr_same(got, (np.array(want_off), np.concatenate(want_i).astype(np.int32), np.concatenate(want_d)),
                        "%s range %s" % (kind, route))


def test_pruning_keeps_a_near_duplicate_study_short():
    """~3,000 noisy copies of one row in one group: with N = 1 the group's entries more than 2 eps below its best are
    pruned in every pass, so no list overflows."""
    S = synth.gauss(N, D, "cuda", seed=3)
    base = S[100].clone()
    S[20000:23000] = base + 0.35 * base.abs().mean() * torch.randn((3000, D), device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    s = make_search(S)
    g = cap_labels("ungrouped", N)                              # (the pilot block then has k capped entries at once)
    g[20000:23000] = 999999
    s.set_cap_groups(g)
    Q = torch.cat([S[20000:20064].to(torch.float64), S[:64].to(torch.float64)]).contiguous()
    for m, k in ((1, 100), (2, 20)):
        got = s.batched_search_device(Q, k, max_per_group=m)
        assert s.last_stats[0] == 0, "lists overflowed: %r" % (s.last_stats,)
        assert_same(got, reference(s, Q, k, m), "near duplicates N=%d" % m)


def test_an_exact_duplicate_study_goes_to_the_fp64_route():
    S = synth.gauss(N, D, "cuda", seed=5)
    S[10000:15000] = S[10000]                                   # 5,000 equal rows: their scores tie, nothing can be pruned
    s = make_search(S)
    g = cap_labels("g100", N)
    g[10000:15000] = 777777
    s.set_cap_groups(g)
    Q = torch.cat([S[10000:10032].to(torch.float64), S[30000:30032].to(torch.float64)]).contiguous()
    got = s.batched_search_device(Q, 20, max_per_group=2)
    assert s.last_stats[0] >= 32, s.last_stats                # (a random query may reach the duplicates too)
    assert_same(got, reference(s, Q, 20, 2), "duplicates")


def test_sparse_fixture_index():
    from oracle import morna_oracle as mo
    S = mo.go_index(tiny_lines(), features=3000, sample_threshold=100).matrix_f32()
    s = make_search(torch.from_numpy(S).cuda())
    assert s.csr is not None
    s.set_cap_groups((np.arange(S.shape[0]) % 7).astype(np.int32))
    Q = s.vectors[:40, :s.dim].to(torch.float64).contiguous()
    for m, k in ((1, 5), (3, 20), (2, 600)):
        assert_same(s.batched_search_device(Q, k, max_per_group=m), reference(s, Q, k, m), "sparse N=%d k=%d" % (m, k))


def test_walk_primitive_on_hand_made_lists():
    S = synth.gauss(64, 32, "cuda", seed=1)
    s = make_search(S)
    s.set_cap_groups(np.array([0, 0, 1, 1, 1, -1, 2, 2] + [3] * 56, np.int32))
    lists = [[0, 1, 2, 5, 3, 4, 6], [], [7, 6, 5, 63, 62, 61, 2], [-1, 0, -1, 1, 4], list(range(64)) * 20]
    off = np.r_[0, np.cumsum([len(l) for l in lists])].astype(np.int64)
    flat = np.concatenate([np.array(l, np.int32) for l in lists]).astype(np.int32)
    dd = np.arange(len(flat), dtype=np.float64) / 7.0
    caps = host(s.cap_group)
    dev = lambda a: torch.from_numpy(a).cuda()
    for m in (1, 2, 3):
        for limit in (None, 0, 1, 4):
            o, i, d = (host(t) for t in s.cap_sorted_lists(dev(off), dev(flat), dev(dd), m, limit))
            for j, l in enumerate(lists):
                li, ld = flat[off[j]:off[j + 1]], dd[off[j]:off[j + 1]]
                valid = np.flatnonzero(li >= 0)
                keep = valid[walk(li[valid], ld[valid], caps, m, limit)]
                assert np.array_equal(i[o[j]:o[j + 1]], li[keep]) and np.array_equal(d[o[j]:o[j + 1]], ld[keep]), (m, limit, j)
            w = 5 if limit is None else max(limit, 1)
            pi = torch.empty((len(lists), w), dtype=torch.int32, device="cuda")
            pd = torch.empty((len(lists), w), dtype=torch.float64, device="cuda")
            s.cap_sorted_lists(dev(off), dev(flat), dev(dd), m, w if limit is None else limit, out=(pi, pd))
            for j in range(len(lists)):
                row = host(pi)[j]
                cnt = int((o[j + 1] - o[j]) if limit is None else min(o[j + 1] - o[j], limit))
                cnt = min(cnt, w)
                assert np.array_equal(row[:cnt], i[o[j]:o[j] + cnt]) and (row[cnt:] == -1).all(), (m, limit, j)


def test_refusals(idx):
    kind, s = idx
    Q, _ = queries(s, 4, seed=1)
    s.set_cap_groups(None)
    with pytest.raises(ValueError, match="set_cap_groups"):
        s.batched_search_device(Q, 5, max_per_group=1)
    s.set_cap_groups(cap_labels("g100", N))
    for bad in (0, -1, 1.5, True):
        with pytest.raises(ValueError, match="max_per_group"):
            s.exact_search_device(Q, 5, max_per_group=bad)
    with pytest.raises(ValueError, match="approximate"):
        s.approx_search_device(Q, 5, max_per_group=1)
    with pytest.raises(ValueError, match="approximate"):
        s.search_nn(5, max_per_group=1)
    with pytest.raises(ValueError, match="one per resident row"):
        s.set_cap_groups(np.zeros(3, np.int32))
