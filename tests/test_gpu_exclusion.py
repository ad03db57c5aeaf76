"""Per-query exclusion (`MornaSearch.set_row_groups` + `query_groups=`): every route equals the brute-force answer over
the rows a query does not exclude -- FP64 distances of all rows (morna_angular_distances), excluded pairs set to +inf,
stably sorted under the reference order (distance ascending, equal distances id descending), cut to k, +inf -> id -1 --
with equal ids and distance bits."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import _lib, synth
from tests.helpers import tiny_lines

pytestmark = pytest.mark.gpu

N, D, K = 50000, 3000, 100


def make_search(S):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=S, stats=(S.shape[0], S.shape[0], S.shape[1]))


def all_distances(s, Q):
    n = s.row_hi - s.row_lo
    out = torch.empty((Q.shape[0], n), dtype=torch.float64, device=s.device)
    Q = Q.contiguous()
    _lib.check(s.lib.morna_angular_distances(_lib.dev_ptr(s.vectors), _lib.dev_ptr(s.pp), n, s.dim, s.ld, _lib.ptr(Q),
                                             Q.shape[0], s.dim, _lib.dev_ptr(out), n, _lib.stream_ptr()), "distances")
    return out


def masked_distances(s, Q, qg):
    dist = all_distances(s, Q)
    if qg is not None:
        qg = torch.as_tensor(qg).to(s.device, torch.int32)
        dist[(s.row_group[None, :] == qg[:, None]) & (qg[:, None] >= 0)] = float("inf")
    return dist


def reference(s, Q, k, qg):
    """Brute-force top-k over the allowed rows: host (ids [nq x k], dists [nq x k])."""
    dist = masked_distances(s, Q, qg)
    n = dist.shape[1]
    kk = min(k, n)
    rows = (n - 1) - torch.sort(dist.flip(1), dim=1, stable=True).indices[:, :kk]
    d = dist.gather(1, rows)
    ids = torch.where(torch.isinf(d), -1, rows + s.row_lo).to(torch.int32)
    out_i = np.full((Q.shape[0], k), -1, np.int32)
    out_d = np.full((Q.shape[0], k), np.inf)
    out_i[:, :kk], out_d[:, :kk] = ids.cpu().numpy(), d.cpu().numpy()
    out_d[out_i < 0] = np.inf
    return out_i, out_d


def reference_range(s, Q, R, qg):
    dist = masked_distances(s, Q, qg).cpu().numpy()
    n = dist.shape[1]
    off, ids, ds = [0], [], []
    for j in range(dist.shape[0]):
        rows = np.nonzero(dist[j] <= R)[0][::-1]                 # descending ids, then a stable sort by distance
        rows = rows[np.argsort(dist[j][rows], kind="stable")]
        ids.append(rows + s.row_lo)
        ds.append(dist[j][rows])
        off.append(off[-1] + len(rows))
    return np.array(off), np.concatenate(ids).astype(np.int32), np.concatenate(ds)


def host(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def assert_same(got, want, label):
    gi, gd = host(got[0]), host(got[1])
    assert np.array_equal(gi, want[0]), "%s: ids differ (%d places)" % (label, int((gi != want[0]).sum()))
    assert np.array_equal(gd.view(np.int64), want[1].view(np.int64)), "%s: distance bits differ" % label


def assert_csr_same(got, want, label):
    for g, w, name in zip(got, want, ("offsets", "ids", "dists")):
        g = host(g)
        if name == "dists":
            assert np.array_equal(g.view(np.int64), w.view(np.int64)), "%s: %s differ" % (label, name)
        else:
            assert np.array_equal(g, w), "%s: %s differ" % (label, name)


def groups(kind, n, seed=0):
    """int32 row labels: 'self' (every row its own group), groups of 10 or 500 scattered or contiguous, and 'huge' (one
    group of all but 50 rows, so its queries have fewer than K rows left)."""
    rng = np.random.default_rng(seed)
    if kind == "self":
        return np.arange(n, dtype=np.int32)
    if kind == "huge":
        g = np.arange(1, n + 1, dtype=np.int32)
        g[:n - 50] = 0
        return g
    size, layout = int(kind.split("_")[0][1:]), kind.split("_")[1]
    g = np.arange(n, dtype=np.int32) // size
    return rng.permutation(g).astype(np.int32) if layout == "scattered" else g


@pytest.fixture(scope="module", params=["gauss", "tissue"])
def idx(request):
    S = synth.matrix(request.param, N, D, "cuda", seed=7)
    return request.param, S, make_search(S)


def queries_and_labels(s, nq, seed):
    """In-index queries labelled with their rows' labels, a few out-of-index ones and a few labelled -1."""
    Q, rows = synth.queries(s.vectors[:, :s.dim], nq, seed=seed)
    qg = s.row_group[rows].clone()
    qg[::17] = -1
    Q[1::23] += 0.01 * torch.randn_like(Q[1::23])
    return Q.contiguous(), qg


@pytest.mark.parametrize("grouping", ["self", "g10_scattered", "g500_contiguous", "g500_scattered", "huge"])
def test_batched_path_equals_brute_force(idx, grouping):
    kind, S, s = idx
    s.set_row_groups(groups(grouping, N))
    Q, qg = queries_and_labels(s, 1024, seed=3)
    if grouping == "huge":
        qg[:512] = 0                                        # half the queries keep only 50 rows
    want = reference(s, Q, K, qg)
    assert_same(s.batched_search_device(Q, K, query_groups=qg), want, "%s/%s batched" % (kind, grouping))
    if grouping == "self":
        rows_of = host(s.row_group)
        for j in np.nonzero(host(qg) >= 0)[0][:50]:
            assert host(qg)[j] not in rows_of[want[0][j][want[0][j] >= 0]]
    if grouping == "huge":
        assert (want[0][:512, 50:] == -1).all() and (want[0][:512, :50] >= 0).all()


def test_unlabelled_queries_return_the_unmasked_bits(idx):
    kind, S, s = idx
    s.set_row_groups(groups("g10_scattered", N))
    Q, _ = queries_and_labels(s, 256, seed=5)
    none = torch.full((Q.shape[0],), -1, dtype=torch.int32, device=s.device)
    for fn in (s.batched_search_device, s.exact_search_device):
        assert_same(fn(Q, K, query_groups=none), tuple(host(t) for t in fn(Q, K)), "%s %s" % (kind, fn.__name__))
    R = float(host(s.exact_search_device(Q[:8], K)[1])[:, 50].mean())
    assert_csr_same(s.range_search_device(Q, R, query_groups=none), tuple(host(t) for t in s.range_search_device(Q, R)),
                    "%s range" % kind)


def test_several_row_blocks(idx):
    kind, S, s = idx
    s.set_row_groups(groups("g500_scattered", N, seed=1))
    Q, qg = queries_and_labels(s, 512, seed=7)
    blocks = s.BATCH_BLOCK_ROWS
    try:
        s.BATCH_BLOCK_ROWS = 20000                          # three blocks, each given its slice of the labels
        got = s.batched_search_device(Q, K, query_groups=qg)
    finally:
        s.BATCH_BLOCK_ROWS = blocks
    assert_same(got, reference(s, Q, K, qg), "%s blocks" % kind)


def test_search_batches_by_id_replays_the_graph(idx):
    kind, S, s = idx
    s.set_row_groups(groups("g10_contiguous", N))
    ids = np.random.default_rng(2).choice(N, 4 * 512, replace=False)
    batches = [ids[b:b + 512] for b in range(0, len(ids), 512)]
    got = [(i.copy(), d.copy()) for i, d in s.search_batches(iter(batches), K, query_groups=True)]
    pipe = s._pipes[(K, 2)]
    assert any(getattr(sl, "graph_key", None) is not None for sl in pipe.slots), "the captured step never replayed"
    for b, (gi, gd) in zip(batches, got):
        rows = torch.from_numpy(b).cuda()
        Q = s.vectors[rows, :D].to(torch.float64)
        assert_same((gi, gd), reference(s, Q, K, s.row_group[rows]), "%s search_batches" % kind)
    Q, qg = queries_and_labels(s, 600, seed=9)               # vector batches with a parallel iterable of labels
    parts = [(Q[:300], qg[:300]), (Q[300:], qg[300:])]
    for (q, g), (gi, gd) in zip(parts, s.search_batches((p[0] for p in parts), K, query_groups=(p[1] for p in parts))):
        assert_same((gi, gd), reference(s, q, K, g), "%s vector batches" % kind)
    with pytest.raises(ValueError):
        list(s.search_batches(iter(batches[:1]), K, side_job=True, query_groups=True))


def test_fp64_scan_full_sort_and_mostly_excluded(idx):
    kind, S, s = idx
    g = groups("g500_contiguous", N)
    g[100:N - 30] = 7                                        # group 7: all rows but 130
    s.set_row_groups(g)
    Q, qg = queries_and_labels(s, 40, seed=11)
    qg[:10] = 7                                             # select kernels on a huge tie of +inf keys
    assert_same(s.exact_search_device(Q, K, query_groups=qg), reference(s, Q, K, qg), "%s exact" % kind)
    assert_same(s.exact_search_device(Q[:1], 5, query_groups=qg[:1]), reference(s, Q[:1], 5, qg[:1]), "%s one query" % kind)
    assert_same(s.exact_search_device(Q[:4], 3000, query_groups=qg[:4]), reference(s, Q[:4], 3000, qg[:4]),
                "%s full sort" % kind)
    assert_same(s.exact_search_device(Q[:20], 2000, query_groups=qg[:20]), reference(s, Q[:20], 2000, qg[:20]),
                "%s k = 2000" % kind)
    got = s.exact_search_batch(Q.cpu().numpy(), K, query_groups=qg.cpu().numpy())
    assert_same(got, reference(s, Q, K, qg), "%s exact_search_batch" % kind)


def test_range_both_routes(idx):
    kind, S, s = idx
    s.set_row_groups(groups("g10_scattered", N, seed=4))
    Q, qg = queries_and_labels(s, 300, seed=13)
    R = float(np.median(host(s.exact_search_device(Q[:32], K)[1])[:, K - 1]))
    want = reference_range(s, Q, R, qg)
    got = s.range_search_device(Q, R, query_groups=qg)
    assert s.last_range_route == "tensor"
    assert_csr_same(got, want, "%s range tensor" % kind)
    want16 = reference_range(s, Q[:16], R, qg[:16])
    got = s.range_search_device(Q[:16], R, query_groups=qg[:16])
    assert s.last_range_route == "exact"
    assert_csr_same(got, want16, "%s range exact" % kind)


def dense_cluster_search():
    """Gauss rows with 5000 near-copies of one row at rows 20000-24999, one group: their queries fill the first-pass
    lists with excluded rows past the pilot block, overflow and go to the FP64 scan."""
    S = synth.gauss(N, D, "cuda", seed=3)
    g = torch.Generator(device="cuda").manual_seed(4)
    S[20000:25000] = S[20000] + 1e-3 * torch.randn((5000, D), generator=g, device="cuda")
    s = make_search(S)
    lab = np.arange(N, dtype=np.int32)
    lab[20000:25000] = N
    s.set_row_groups(lab)
    return s


def test_overflowing_group_goes_to_the_fp64_scan():
    s = dense_cluster_search()
    rows = torch.cat([torch.arange(20000, 20064), torch.arange(0, 64)]).cuda()
    Q = s.vectors[rows, :D].to(torch.float64).contiguous()
    qg = s.row_group[rows]
    assert_same(s.batched_search_device(Q, K, query_groups=qg), reference(s, Q, K, qg), "cluster batched")
    assert s.last_stats[0] >= 64, s.last_stats
    R = 0.9 * float(host(s.exact_search_device(Q[64:80], K)[1])[:, K - 1].min())
    want = reference_range(s, Q, R, qg)
    assert_csr_same(s.range_search_device(Q, R, query_groups=qg), want, "cluster range")
    assert s.last_stats[0] >= 64


def test_filtered_search_with_groups(idx):
    kind, S, s = idx
    s.set_row_groups(groups("g10_scattered", N, seed=6))
    members = np.random.default_rng(8).choice(N, N // 2, replace=False)
    f = s.subset(members)
    rows = torch.from_numpy(np.concatenate([np.sort(members)[:100], np.setdiff1d(np.arange(N), members)[:28]])).cuda()
    Q = s.vectors[rows, :D].to(torch.float64).contiguous()
    qg = s.row_group[rows]
    full = reference(s, Q, N, qg)
    keep = np.isin(full[0], members)
    want_i, want_d = np.full((Q.shape[0], K), -1, np.int32), np.full((Q.shape[0], K), np.inf)
    for j in range(Q.shape[0]):
        i, d = full[0][j][keep[j]][:K], full[1][j][keep[j]][:K]
        want_i[j, :len(i)], want_d[j, :len(i)] = i, d
    assert_same(f.batched_search_device(Q, K, query_groups=qg), (want_i, want_d), "%s filtered batched" % kind)
    assert_same(f.exact_search_device(Q, K, query_groups=qg), (want_i, want_d), "%s filtered exact" % kind)
    got = [(i.copy(), d.copy()) for i, d in f.search_batches(iter([rows.cpu().numpy()]), K, query_groups=True)]
    assert_same(got[0], (want_i, want_d), "%s filtered search_batches" % kind)


def test_sparse_path_on_the_tiny_fixture():
    from oracle import morna_oracle as mo
    S = mo.go_index(tiny_lines(), features=3000, sample_threshold=100).matrix_f32()
    s = make_search(S)
    assert s.csr is not None
    n = S.shape[0]
    lab = (np.arange(n) // 40).astype(np.int32)
    lab[: n - 20] = 0                                        # group 0 covers all but 20 rows: a huge tie of +inf keys
    s.set_row_groups(lab)
    rows = torch.tensor([0, 2040, 6595 % n, 5, 4000 % n, 17, n - 1, n - 5]).cuda()
    Q = torch.from_numpy(S[rows.cpu().numpy()].astype(np.float64)).cuda()
    qg = s.row_group[rows].clone()
    qg[1] = 3
    for k in (20, 100):
        assert_same(s.exact_search_device(Q, k, query_groups=qg), reference(s, Q, k, qg), "sparse k=%d" % k)
    assert_same(s.batched_search_device(Q, 20, query_groups=qg), reference(s, Q, 20, qg), "sparse batched")
    assert_csr_same(s.range_search_device(Q, 0.7, query_groups=qg), reference_range(s, Q, 0.7, qg), "sparse range")


def test_refusals(idx):
    from morna_b200 import dist
    kind, S, s = idx
    Q = s.vectors[:4, :D].to(torch.float64).contiguous()
    s.set_row_groups(None)
    with pytest.raises(ValueError):
        s.exact_search_device(Q, K, query_groups=[0, 1, 2, 3])
    s.set_row_groups(groups("self", N))
    with pytest.raises(ValueError):
        s.approx_search_device(Q, K, query_groups=[0, 1, 2, 3])
    with pytest.raises(ValueError):
        dist.sharded_batched_search(s, Q, K, query_groups=[0, 1, 2, 3])
    with pytest.raises(ValueError):
        dist.sharded_range_search(s, Q, 0.5, query_groups=[0, 1, 2, 3])
    with pytest.raises(ValueError):
        s.exact_search_device(Q, K, query_groups=[0, 1])


def test_relabelling_a_search_does_not_replay_a_stale_graph(idx):
    """set_row_groups between two search_batches runs: the captured step of the first run must not be replayed with the
    first run's row labels."""
    kind, S, s = idx
    ids = np.random.default_rng(12).choice(N, 4 * 256, replace=False)
    batches = [ids[b:b + 256] for b in range(0, len(ids), 256)]
    for grouping in ("g500_contiguous", "g10_scattered"):
        s.set_row_groups(groups(grouping, N, seed=3))
        got = [(i.copy(), d.copy()) for i, d in s.search_batches(iter(batches), K, query_groups=True)]
        assert any(getattr(sl, "graph_key", None) is not None for sl in s._pipes[(K, 2)].slots)
        for b, (gi, gd) in zip(batches, got):
            rows = torch.from_numpy(b).cuda()
            Q = s.vectors[rows, :D].to(torch.float64)
            assert_same((gi, gd), reference(s, Q, K, s.row_group[rows]), "%s %s after relabelling" % (kind, grouping))


@pytest.mark.parametrize("block_rows", [512, 2048])
def test_fewer_allowed_rows_than_k_in_the_tensor_lists(block_rows):
    """Short lists built by the tensor-core kernels themselves: a 10,240-row index scored in small row blocks (pilot and
    blocks of `block_rows`), all rows but 60 in one group.  Its queries see fewer than k allowed entries in the pilot and
    in every refinement (threshold -inf), yet each block adds fewer entries than the lists hold, so nothing overflows and
    the pilot, refine and final passes emit every allowed entry themselves (512: lane lists without a pivot; 2048: the
    bisection fallback counting allowed entries)."""
    n, d = 10240, 1024
    S = synth.gauss(n, d, "cuda", seed=17)
    s = make_search(S)
    lab = np.arange(1, n + 1, dtype=np.int32)
    keep = np.linspace(0, n - 1, 60).astype(np.int64)
    group0 = np.setdiff1d(np.arange(n), keep)
    lab[group0] = 0
    s.set_row_groups(lab)
    rng = np.random.default_rng(5)
    rows = torch.from_numpy(np.concatenate([rng.choice(group0, 96, replace=False), rng.choice(n, 32, replace=False)])).cuda()
    Q = s.vectors[rows, :d].to(torch.float64).contiguous()
    qg = s.row_group[rows]
    lib = s.lib
    try:
        assert lib.morna_debug_set_tuning(9, block_rows) == 0
        got = s.batched_search_device(Q, K, query_groups=qg)
        stats = list(s.last_stats)
    finally:
        lib.morna_debug_set_tuning(9, 131072)
    want = reference(s, Q, K, qg)
    assert_same(got, want, "block rows %d" % block_rows)
    assert stats[0] == 0, stats
    assert (want[0][:96, 60:] == -1).all() and (want[0][:96, :60] >= 0).all()
