"""Range search (`MornaSearch.range_search_device`, `search --max-distance`): every row within a distance R, on the
tensor-core route (filter GEMM + FP64 check) and the FP64 route (distance scan), against a brute-force list built from
morna_angular_distances over all rows -- equal ids, order and distance bits."""
import io
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import cli

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KNOB_DEFAULTS = {9: 131072, 10: 8192, 11: 0, 36: 1}


@pytest.fixture
def knobs():
    """set(key, value) for the batched path's block and pilot keys; all back at their defaults after the test."""
    from morna_b200 import _lib
    lib = _lib.load()

    def set_knob(key, value):
        assert key in KNOB_DEFAULTS
        assert lib.morna_debug_set_tuning(key, value) == 0

    try:
        yield set_knob
    finally:
        for key, value in KNOB_DEFAULTS.items():
            lib.morna_debug_set_tuning(key, value)


def make_search(S, **kw):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=S, stats=(S.shape[0], S.shape[0], S.shape[1]), **kw)


def distances(srch, Q):
    """FP64 distances [nq x local rows] from the exact scan."""
    from morna_b200 import _lib
    n = srch.row_hi - srch.row_lo
    Q = Q.contiguous()
    out = torch.empty((Q.shape[0], n), dtype=torch.float64, device=srch.device)
    _lib.check(srch.lib.morna_angular_distances(_lib.dev_ptr(srch.vectors), _lib.dev_ptr(srch.pp), n, srch.dim, srch.ld,
                                                _lib.ptr(Q), Q.shape[0], srch.dim, _lib.dev_ptr(out), n, _lib.stream_ptr()),
               "morna_angular_distances")
    return out


def brute(srch, Q, R, chunk=256, dist=None):
    """CSR (offsets, ids, dists) numpy: rows with d <= R, distance ascending, equal distances id descending."""
    offs, ids, ds = [np.zeros(1, np.int64)], [], []
    base = 0
    for q0 in range(0, Q.shape[0], chunk):
        d = distances(srch, Q[q0:q0 + chunk]) if dist is None else dist[q0:q0 + chunk]
        q, row = torch.nonzero(d <= R, as_tuple=True)               # (query, row) ascending
        q, row = q.flip(0), row.flip(0)                              # query descending, row descending
        dv = d[q, row]
        o = torch.sort(dv, stable=True).indices
        q, row, dv = q[o], row[o], dv[o]
        o = torch.sort(q, stable=True).indices                       # query ascending, then distance, then row descending
        q, row, dv = q[o], row[o], dv[o]
        cnt = torch.bincount(q, minlength=d.shape[0]).cpu().numpy()
        offs.append(base + np.cumsum(cnt))
        base += int(cnt.sum())
        ids.append((row + srch.row_lo).to(torch.int32).cpu().numpy())
        ds.append(dv.cpu().numpy())
    return np.concatenate(offs), np.concatenate(ids) if ids else np.zeros(0, np.int32), \
        np.concatenate(ds) if ds else np.zeros(0, np.float64)


def host(csr):
    return tuple(t.cpu().numpy() for t in csr)


def assert_csr_equal(got, want, label=""):
    go, gi, gd = got
    wo, wi, wd = want
    assert np.array_equal(go, wo), "%s: offsets differ (first at query %d)" % (label, int(np.nonzero(go != wo)[0][0]) - 1)
    assert np.array_equal(gi, wi), "%s: ids differ" % label
    assert np.array_equal(gd.view(np.int64), wd.view(np.int64)), "%s: distance bits differ" % label


def check(srch, Q, R, route, dist=None, label=""):
    got = host(srch.range_search_device(Q, R))
    assert srch.last_range_route == route, label
    assert_csr_equal(got, brute(srch, Q, R, dist=dist), label)
    return got


def median_kth(dist, k):
    return float(torch.kthvalue(dist, k, dim=1).values.median())


# ------------------------------------------------------------------ 50,000 x 3000, 4096 queries, both routes
@pytest.fixture(scope="module", params=["gauss", "tissue"])
def big(request):
    from morna_b200 import synth
    S = synth.matrix(request.param, 50000, 3000, "cuda")
    srch = make_search(S)
    qa, _ = synth.queries(S, 2048, seed=5)
    qb, _ = synth.queries(S, 2048, seed=6, noise=0.3)
    Q = torch.cat([qa, qb]).contiguous()
    dist = torch.cat([distances(srch, Q[i:i + 512]) for i in range(0, Q.shape[0], 512)])
    return {"kind": request.param, "S": S, "srch": srch, "Q": Q, "dist": dist,
            "R": [median_kth(dist, 100), median_kth(dist, 1000)]}


@pytest.mark.parametrize("level", [0, 1])
def test_tensor_route_equals_brute_force(big, level):
    srch, Q, R = big["srch"], big["Q"], big["R"][level]
    got = check(srch, Q, R, "tensor", dist=big["dist"], label="%s R=%r" % (big["kind"], R))
    over, first, matches = srch.last_stats
    assert matches == got[0][-1] and first > 0
    assert over < Q.shape[0] // 2                                 # the filter answered most queries


@pytest.mark.parametrize("level", [0, 1])
def test_exact_route_equals_brute_force(big, level):
    srch, R = big["srch"], big["R"][level]
    Q = big["Q"][::16].contiguous()                               # 256 queries, forced onto the FP64 scan
    srch.RANGE_TENSOR_MIN_QUERIES = 1 << 30
    try:
        check(srch, Q, R, "exact", dist=big["dist"][::16], label="%s R=%r" % (big["kind"], R))
    finally:
        del srch.RANGE_TENSOR_MIN_QUERIES


def test_small_batch_goes_to_the_exact_route(big):
    srch, R = big["srch"], big["R"][1]
    check(srch, big["Q"][:40], R, "exact", dist=big["dist"][:40])


def test_consistent_with_topk(big):
    srch, Q, R = big["srch"], big["Q"], big["R"][0]
    off, ids, d = host(srch.range_search_device(Q, R))
    for j in list(range(0, 4096, 257)) + [4095]:
        cnt = int(off[j + 1] - off[j])
        t_i, t_d = srch.exact_search_device(Q[j:j + 1], cnt)
        assert np.array_equal(t_i.cpu().numpy()[0], ids[off[j]:off[j + 1]])
        assert np.array_equal(t_d.cpu().numpy()[0].view(np.int64), d[off[j]:off[j + 1]].view(np.int64))


def test_oracle_agrees(big):
    from oracle import c_oracle
    srch, R = big["srch"], big["R"][0]
    S_host = big["S"].cpu().numpy()
    Q = big["Q"][::128][:32].contiguous()
    off, ids, d = host(srch.range_search_device(Q, R))
    Q_host = Q.cpu().numpy()
    for j in range(Q.shape[0]):
        true_d = c_oracle.distances(S_host, Q_host[j])
        mine = set(ids[off[j]:off[j + 1]].tolist())
        assert set(np.nonzero(true_d <= R - 1e-9)[0].tolist()) <= mine
        assert not (mine & set(np.nonzero(true_d > R + 1e-9)[0].tolist()))
        assert np.abs(d[off[j]:off[j + 1]] - true_d[ids[off[j]:off[j + 1]]]).max(initial=0.0) <= 1e-9


# ------------------------------------------------------------------ smaller indexes: boundaries, shards, regimes
@pytest.fixture(scope="module")
def small():
    from morna_b200 import synth
    S = synth.gauss(20000, 256, "cuda", seed=7)
    S[100] = 0.0                                                  # a zero row
    S[200:210] = S[5]                                             # ten copies of row 5 (11 equal rows)
    return S, make_search(S)


def small_queries(S, nq, seed=3):
    from morna_b200 import synth
    qa, _ = synth.queries(S, nq // 2, seed=seed)
    qb, _ = synth.queries(S, nq - nq // 2, seed=seed + 10, noise=0.2)
    return torch.cat([qa, qb]).contiguous()


@pytest.mark.parametrize("nq", [200, 10])
def test_boundaries(small, nq):
    S, srch = small
    route = "tensor" if nq >= 64 else "exact"
    Q = small_queries(S, nq)
    Q[0] = S[5].double()                                          # duplicated rows: id descending at distance 0
    Q[1] = 0.0                                                    # the zero query
    off, ids, d = check(srch, Q, 0.0, route, label="R = 0")
    assert ids[off[0]:off[1]].tolist() == [209, 208, 207, 206, 205, 204, 203, 202, 201, 200, 5]
    assert not d[off[0]:off[1]].any()
    # R equal to a row's exact distance includes the row; the next double below excludes it
    dist = distances(srch, Q[2:3])[0]
    row = int(torch.argsort(dist)[37])
    R = float(dist[row])
    off, ids, _ = check(srch, Q, R, route, label="R = d")
    assert srch.row_lo + row in ids[off[2]:off[3]].tolist()
    off, ids, _ = check(srch, Q, float(np.nextafter(R, 0.0)), route, label="R below d")
    assert srch.row_lo + row not in ids[off[2]:off[3]].tolist()
    # zero query and zero row sit at sqrt(2): in range exactly when R >= sqrt(2)
    for R, inside in ((math.sqrt(2.0), True), (float(np.nextafter(math.sqrt(2.0), 0.0)), False)):
        off, ids, _ = check(srch, Q, R, route, label="R = %r" % R)
        assert (off[2] - off[1] == S.shape[0]) == inside
        assert (100 in ids[off[2]:off[3]].tolist()) == inside
    off, ids, _ = check(srch, Q, 2.0, route, label="R = 2")      # every row (the tensor route overflows to the scan)
    assert np.array_equal(np.diff(off), np.full(nq, S.shape[0]))


def test_overflow_of_a_dense_cluster(knobs):
    from morna_b200 import synth
    S = synth.gauss(30000, 128, "cuda", seed=9)
    S[:6000] = S[0] + 1e-3 * synth.gauss(6000, 128, "cuda", seed=10)      # > 4096 rows within reach of each other
    srch = make_search(S)
    Q = torch.cat([S[:100].double(), small_queries(S, 100, seed=4)]).contiguous()
    check(srch, Q, 0.05, "tensor", label="cluster")
    over, first, matches = srch.last_stats
    assert over >= 100 and first > 4096 * 100 and matches >= 6000 * 100


def test_huge_query_value_goes_to_the_exact_scan(small):
    S, srch = small
    Q = small_queries(S, 100)
    Q[7] = Q[7] * 0.0
    Q[7, 3] = 2.0 ** 127
    Q[8, 0] = -(2.0 ** 130)
    check(srch, Q, 1.3, "tensor")
    assert srch.last_stats[0] >= 2


def test_shard_ids_are_global(small):
    S, _ = small
    srch = make_search(S, shard=(1, 2))
    assert srch.row_lo == 10000
    Q = small_queries(S, 128, seed=12)
    off, ids, _ = check(srch, Q, 1.25, "tensor")
    assert ids.min(initial=10000) >= 10000 and len(ids) > 0
    check(srch, Q[:20], 1.25, "exact")


@pytest.mark.parametrize("dim", [10000, 30000])
def test_wide_features(dim):
    from morna_b200 import synth
    S = synth.tissue(3000, dim, "cuda", seed=dim)
    srch = make_search(S)
    Q = small_queries(S, 96, seed=2)
    R = median_kth(distances(srch, Q), 50)
    check(srch, Q, R, "tensor", label="D=%d" % dim)
    check(srch, Q[:16], R, "exact", label="D=%d" % dim)


def test_sparse_index_uses_the_exact_route():
    from morna_b200 import synth
    S = synth.sparse_fixture(20000, 3000, "cuda")
    srch = make_search(S)
    assert srch.csr is not None and srch.sparse_exact
    Q = small_queries(S, 200, seed=8)
    check(srch, Q, 0.0, "exact")
    check(srch, Q, 0.5, "exact")


def test_block_and_pilot_keys_change_nothing(small, knobs):
    S, srch = small
    Q = small_queries(S, 300, seed=21)
    want = host(srch.range_search_device(Q, 1.3))
    for key, value in ((9, 256), (10, 256), (11, 512), (36, 2)):
        knobs(key, value)
        assert_csr_equal(host(srch.range_search_device(Q, 1.3)), want, "key %d" % key)


def test_byte_cap_splits_a_batch_into_groups(small):
    S, srch = small
    Q = small_queries(S, 300, seed=22)
    want = host(srch.range_search_device(Q, 1.35))
    groups = list(srch.range_search_groups(Q, 1.35, byte_cap=12 * 500))
    assert len(groups) > 1 and groups[0][0] == 0 and groups[-1][1] == 300
    off = [np.zeros(1, np.int64)]
    for lo, hi, o, i, d in groups:
        assert o.numel() == hi - lo + 1 and (lo == groups[0][0] or lo == prev_hi)
        prev_hi = hi
        off.append(o[1:].cpu().numpy() + off[-1][-1])
    assert np.array_equal(np.concatenate(off), want[0])
    assert np.array_equal(np.concatenate([g[3].cpu().numpy() for g in groups]), want[1])


def test_bad_radius_is_refused(small):
    _, srch = small
    Q = torch.zeros((1, srch.dim), dtype=torch.float64, device="cuda")
    for R in (-1e-300, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            srch.range_search_device(Q, R)


# ------------------------------------------------------------------ CLI
def _cli(argv, stdin=None):
    out = io.StringIO()
    assert cli.main(argv, stdin=stdin, stdout=out, stderr=io.StringIO()) == 0
    return out.getvalue().splitlines()


def _cut(lines, R, prefix=False):
    """Lines of a `-r <all> -e -d` run kept where the distance is <= R (ranks are unchanged: lists are sorted)."""
    return [l for l in lines if float(l.split("\t")[3 if prefix else 2]) <= R]


@pytest.fixture(scope="module")
def synth_index(tmp_path_factory):
    import gzip
    tmp = tmp_path_factory.mktemp("range_cli")
    rng = np.random.default_rng(17)
    lines = []
    for i in range(300):
        key = "chr%d\t%d\t%d" % (1 + i % 5, 1000 + 37 * i, 1000 + 37 * i + int(rng.integers(50, 5000)))
        n = int(rng.integers(1, 60))
        s = np.sort(rng.choice(400, n, replace=False)) + 1
        lines.append("%s\t+\tGT\tAG\t%s\t%s\n" % (key, ",".join(map(str, s)), ",".join(map(str, rng.integers(1, 40, n)))))
    path = str(tmp / "index.tsv.gz")
    with gzip.open(path, "wt") as fh:
        fh.write("".join(lines))
    meta = tmp / "meta.tsv"
    meta.write_text("".join("%d\tsample_%d tissue\n" % (s, s) for s in range(1, 401, 3)))
    base = str(tmp / "idx")
    assert cli.main(["index", "--intropolis", path, "-x", base, "--features", "512", "-t", "8", "-m", str(meta)],
                    stdout=io.StringIO()) == 0
    qpath = str(tmp / "query.tsv")
    with open(qpath, "w") as fh:
        fh.write("".join(lines[::3]))
    from morna_b200 import files
    return {"base": base, "qpath": qpath, "lines": lines, "size": files.read_stats(base)[1]}


@pytest.mark.parametrize("R", [0.9, 1.2])
def test_cli_every_mode_equals_a_full_list_cut_at_R(synth_index, R):
    base, size, qpath = synth_index["base"], str(synth_index["size"]), synth_index["qpath"]
    # stdin
    raw = "".join("%s\t%d\n" % ("\t".join(l.split("\t")[:3]), 5) for l in synth_index["lines"][:40:2])
    full = _cli(["search", "-x", base, "-f", "raw", "-e", "-d", "-r", size], stdin=io.StringIO(raw))
    for r in (R, float(full[4].split("\t")[2]) + 1e-9):          # (the second radius: at least five samples in range)
        got = _cli(["search", "-x", base, "-f", "raw", "--max-distance", repr(r), "-e", "-d"], stdin=io.StringIO(raw))
        assert got == _cut(full, r)
    assert len(got) >= 5
    assert _cli(["search", "-x", base, "-f", "raw", "--max-distance", repr(r), "-d", "-r", "3"], stdin=io.StringIO(raw)) == got[:3]
    # -q
    from morna_b200 import files
    sid = sorted(files.read_map(base))[7]
    full = _cli(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", size])
    got = _cli(["search", "-x", base, "-q", str(sid), "--max-distance", str(R), "-e", "-d"])
    assert got[:2] == full[:2] and got[2:] == _cut(full[2:], R)
    # --query-intropolis and --all-samples (-m too)
    for mode in (["--query-intropolis", qpath], ["--all-samples"]):
        full = _cli(["search", "-x", base] + mode + ["-e", "-d", "-m", "-r", size])
        got = _cli(["search", "-x", base] + mode + ["--max-distance", str(R), "-e", "-d", "-m"])
        assert got == _cut(full, R, prefix=True) and len(got) > 0
        capped = _cli(["search", "-x", base] + mode + ["--max-distance", str(R), "-d", "-r", "2"])
        per = {}
        want = []
        for l in _cut(_cli(["search", "-x", base] + mode + ["-e", "-d", "-r", size]), R, prefix=True):
            sid_, rest = l.split("\t", 1)
            per[sid_] = per.get(sid_, 0) + 1
            if per[sid_] <= 2:
                want.append(l)
        assert capped == want


def test_cli_tiny_intropolis_goes_through_the_sparse_route(tmp_path):
    from morna_b200.search import MornaSearch
    base = str(tmp_path / "tiny")
    tsv = os.path.join(GOLDEN, "tiny_intropolis.tsv")
    assert cli.main(["index", "--intropolis", tsv, "-x", base], stdout=io.StringIO()) == 0
    srch = MornaSearch(basename=base)
    assert srch.csr is not None and srch.sparse_exact
    size = str(srch.index_size)
    for R in (0.0, 0.7):
        full = _cli(["search", "-x", base, "--query-intropolis", tsv, "-e", "-d", "-r", size])
        got = _cli(["search", "-x", base, "--query-intropolis", tsv, "--max-distance", str(R), "-d"])
        assert got == _cut(full, R, prefix=True) and len(got) > 0
