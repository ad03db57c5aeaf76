"""Batch queries (`search --query-intropolis`, `search --all-samples`): the device junction table, query vectors from an
intropolis file bit for bit against the oracle's finalize_query, the batch search against the exact search, and the
output lines against single-query `search`."""
import io
import os

import numpy as np
import pytest

from morna_b200 import cli
from oracle import morna_oracle as mo

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIM = 512


# ------------------------------------------------------------------ CPU: flags and the host merge
def test_batch_flags_leave_the_parser_defaults_alone():
    p = cli.build_parser()
    s = p.parse_args(["search", "-x", "idx", "--query-intropolis", "q.tsv.gz"])
    assert (s.query_intropolis, s.all_samples, s.format, s.results, s.exact, s.query_id) == ("q.tsv.gz", False, "sam", 20, False, None)
    s = p.parse_args(["search", "-x", "idx", "--all-samples", "-e", "-d", "-m"])
    assert (s.query_intropolis, s.all_samples, s.distances, s.metadata) == (None, True, True, True)


@pytest.mark.parametrize("argv", [
    ["--query-intropolis", "q.tsv", "-q", "12"],
    ["--query-intropolis", "q.tsv", "-rl"],
    ["--query-intropolis", "q.tsv", "-f", "raw"],
    ["--all-samples", "-f", "sam"],                 # also the default's value: given is what counts
    ["--all-samples", "-q", "3"],
    ["--query-intropolis", "q.tsv", "--all-samples"],
])
def test_batch_flags_refuse_other_query_sources(argv):
    err = io.StringIO()
    assert cli.main(["search", "-x", "no_such_index"] + argv, stdout=io.StringIO(), stderr=err) == 2
    assert "cannot be combined" in err.getvalue()


def _merge_by_dict(row_off, sample, cov, rows, match):
    """The reference's rule on the flagged rows: per (key, sample) the coverages summed at the first position."""
    first, new = {}, {}
    for r, m in zip(rows, match):
        for p in range(row_off[r], row_off[r + 1]):
            kp = (int(m), int(sample[p]))
            if kp in first:
                q = first[kp]
                new[q] = new.get(q, int(cov[q])) + int(cov[p])
                new[p] = 0
            else:
                first[kp] = p
    return new


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_merge_repeated_pairs_matches_a_dict(seed):
    from morna_b200.batch_query import merge_repeated_pairs
    rng = np.random.default_rng(seed)
    n_rows = 300
    lens = rng.integers(0, 12, n_rows)
    row_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    sample = rng.integers(0, 15, int(row_off[-1])).astype(np.int32)
    cov = rng.integers(0, 1000, int(row_off[-1])).astype(np.int32)
    rows = np.sort(rng.choice(n_rows, 120, replace=False))
    match = rng.integers(0, 10, len(rows))
    pos, new = merge_repeated_pairs(row_off, sample, cov, rows, match)
    want = _merge_by_dict(row_off, sample, cov, rows, match)
    assert dict(zip(pos.tolist(), new.tolist())) == {p: v for p, v in want.items()}
    assert len(pos) > 0
    none = merge_repeated_pairs(row_off, sample, cov, np.zeros(0, np.int64), np.zeros(0, np.int64))
    assert len(none[0]) == 0


def test_merge_repeated_pairs_refuses_int32_overflow():
    from morna_b200.batch_query import merge_repeated_pairs
    row_off = np.array([0, 1, 2], np.int64)
    with pytest.raises(ValueError):
        merge_repeated_pairs(row_off, np.array([4, 4], np.int32), np.array([2 ** 31 - 1, 5], np.int32), [0, 1], [7, 7])


@pytest.mark.parametrize("gz", [False, True])
def test_read_rows_equals_the_python_tokenizer(tmp_path, gz):
    import gzip
    from morna_b200 import parse
    from morna_b200.batch_query import read_rows
    lines = ["chr1\t5\t9\t+\tGT\tAG\t1,2,3\t4,5,6\n", "chr1\t5\t9\t+\tGT\tAG\t007,8\t5,6\n",
             "chr2\t5\t9\t+\tGT\tAG\t9,5,2\t1,1,1 \n", "chr3\t1\t2\t+\tGT\tAG\t4\t3\n", "chr3\t1\t20\t+\tGT\tAG\t4,6\t3\n"]
    path = str(tmp_path / ("q.tsv.gz" if gz else "q.tsv"))
    with (gzip.open(path, "wt") if gz else open(path, "w")) as fh:
        fh.write("".join(lines))
    packed, key_off, row_off, sample, cov = read_rows(path)
    kb = packed.tobytes()
    got = [(kb[key_off[i]:key_off[i + 1]].decode(), sample[row_off[i]:row_off[i + 1]].tolist(),
            cov[row_off[i]:row_off[i + 1]].tolist()) for i in range(len(key_off) - 1)]
    want = [parse.tokenize_line(line) for line in lines]
    assert got == [(k, s[:len(c)], c[:len(s)]) for k, s, c in want]


# ------------------------------------------------------------------ synthetic index and query files
def _row(key, samples, covs):
    return "%s\t+\tGT\tAG\t%s\t%s\n" % (key.replace(" ", "\t"), ",".join(map(str, samples)), ",".join(map(str, covs)))


def _index_lines(rng, n_rows=300, n_samples=400):
    lines, keys = [], []
    for i in range(n_rows):
        key = "chr%d %d %d" % (1 + i % 5, 1000 + 37 * i, 1000 + 37 * i + int(rng.integers(50, 5000)))
        n = int(rng.integers(1, 60))
        s = np.sort(rng.choice(n_samples, n, replace=False)) + 1
        lines.append(_row(key, s.tolist(), rng.integers(1, 40, n).tolist()))
        keys.append(key)
    return lines, keys


def _query_lines(rng, keys, freq):
    """Every case the pipeline has to get right, in one file."""
    passing = [k for k in keys if k in freq]
    under = [k for k in keys if k not in freq]
    lines = []
    for i in range(40):                                   # indexed keys; samples inside (1..400) and outside the index
        n = int(rng.integers(1, 25))
        s = np.sort(rng.choice(450, n, replace=False)) + 1
        lines.append(_row(passing[i], s.tolist(), rng.integers(1, 30, n).tolist()))
    lines.append(_row("chr9 1 2", [3, 9001, 5], [4, 4, 4]))                     # absent from the index
    lines.append(_row(under[0], [3, 9001, 7], [2, 2, 2]))                      # in the input, under the threshold
    lines.append(_row(passing[3], [5, 9, 12, 300], [1, 2, 3, 4]))             # a key on a second row
    lines.append(_row(passing[50], [5, 9, 5, 11], [6, 7, 8, 9]))              # a sample twice in one row
    lines.append(_row(passing[51], [30, 20, 10], [3, 2, 1]))                  # descending sample list
    lines.append("%s\t+\tGT\tAG\t007,8,44\t5,6,7\n" % passing[52].replace(" ", "\t"))   # Python tokenizer (leading zero)
    lines.append(_row(passing[3], [12, 77], [10, 11]))                        # the key a third time
    lines.append(_row("chr9 1 20", [8801], [5]))                               # 8801: no indexed junction at all
    lines.append(_row("chr9 1 2", [8801, 8802], [1, 1]))                       # (and a prefix of the key above)
    lines.append(_row(passing[60], [8802, 5], [1, 1]))
    return lines


def oracle_queries(lines, freq, sample_count, dim):
    """Per sample in first-seen order: finalize_query of its (key, coverage) stream in file order, keeping indexed keys."""
    from morna_b200 import parse
    order, streams = [], {}
    for line in lines:
        key, samples, covs = parse.tokenize_line(line)
        for s, c in zip(samples, covs):
            if s not in streams:
                streams[s] = {}
                order.append(s)
            if key in freq:
                streams[s][(key,)] = streams[s].get((key,), 0) + c
    Q = np.array([mo.finalize_query(streams[s], freq, sample_count, dim) for s in order], dtype=np.float64).reshape(len(order), dim)
    return np.array(order, dtype=np.int64), Q


@pytest.fixture(scope="module")
def synth(tmp_path_factory):
    import gzip
    from morna_b200 import files
    tmp = tmp_path_factory.mktemp("batch_query")
    rng = np.random.default_rng(11)
    lines, keys = _index_lines(rng)
    path = str(tmp / "index.tsv.gz")
    with gzip.open(path, "wt") as fh:
        fh.write("".join(lines))
    meta = tmp / "meta.tsv"
    meta.write_text("".join("%d\tsample_%d tissue\n" % (s, s) for s in range(1, 401, 3)))
    base = str(tmp / "idx")
    assert cli.main(["index", "--intropolis", path, "-x", base, "--features", str(DIM), "-t", "8", "-m", str(meta)],
                    stdout=io.StringIO()) == 0
    freq = files.read_freq(base)
    assert 100 < len(freq) < len(keys)
    qlines = _query_lines(rng, keys, freq)
    qpath = str(tmp / "query.tsv")
    with open(qpath, "w") as fh:
        fh.write("".join(qlines))
    return {"base": base, "freq": freq, "keys": keys, "qlines": qlines, "qpath": qpath, "tmp": tmp,
            "sample_count": files.read_stats(base)[0], "rng": rng}


def _search(base):
    from morna_b200.search import MornaSearch
    return MornaSearch(basename=base)


# ------------------------------------------------------------------ GPU: the junction table
def _lookup(search, table, keys):
    import torch
    from morna_b200 import _lib
    from morna_b200.batch_query import _hash
    blobs = [k.encode() for k in keys]
    off = np.zeros(len(blobs) + 1, np.int32)
    off[1:] = np.cumsum([len(b) for b in blobs])
    d_keys = torch.from_numpy(np.frombuffer(b"".join(blobs) + b"\0", np.uint8).copy()).cuda()
    d_off = torch.from_numpy(off).cuda()
    raw = _hash(search, d_keys, d_off, len(keys))[0]
    row_off = torch.zeros(len(keys) + 1, dtype=torch.int64, device="cuda")       # no pairs: bit 1 never set
    sample = torch.zeros(1, dtype=torch.int32, device="cuda")
    match, passing, idf, flags, n_flagged = table.lookup(search, d_keys, d_off, raw, row_off, sample, len(keys))
    n = len(keys)
    return match[:n].cpu().numpy(), passing[:n].cpu().numpy(), idf[:n].cpu().numpy(), flags[:n].cpu().numpy(), n_flagged


def _table_search(freq, sample_count=10 ** 6):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=np.ones((1, 8), np.float32), stats=(sample_count, 1, 8), sample_frequencies=freq)


@pytest.mark.gpu
@pytest.mark.parametrize("n_keys", [0, 1, 1000, 1 << 20])
def test_junction_table_matches_a_dict(n_keys):
    import math
    from morna_b200.batch_query import junction_table
    rng = np.random.default_rng(n_keys)
    starts = rng.integers(1, 10 ** 8, n_keys)
    keys = ["chr%d %d %d" % (c, s, s + 1 + d) for c, s, d in zip(rng.integers(1, 23, n_keys), starts, rng.integers(0, 10 ** 5, n_keys))]
    freq = {}
    for i, k in enumerate(keys):
        freq.setdefault(k, 1 + i % 977)
    search = _table_search(freq)
    table = junction_table(search)
    assert junction_table(search) is table                       # built once per index
    index_of = {k: i for i, k in enumerate(k for k, f in freq.items() if f > 0)}
    present = list(freq)[:min(len(freq), 200000)]
    queries = present + ["chr1 1 2", "chr1 1 20", "chr1 1 200", "", "chrX 5 6"]
    queries += [k + "0" for k in present[:1000]] + [k[:-1] for k in present[:1000]]          # prefixes of each other
    queries += ["chr1 1 2"]                                                                    # a key twice
    match, passing, idf, flags, n_flagged = _lookup(search, table, queries)
    want = np.array([index_of.get(q, -1) for q in queries])
    assert np.array_equal(match, want)
    assert np.array_equal(passing, (want >= 0).astype(np.uint8))
    want_idf = np.array([math.log(float(10 ** 6) / freq[q]) if q in index_of else 0.0 for q in queries])
    assert np.array_equal(idf.view(np.int64), want_idf.view(np.int64))
    assert not flags.any() and n_flagged == 0                   # "chr1 1 2" twice, but not in the table
    if n_keys:
        match, _, _, flags, n_flagged = _lookup(search, table, [present[0], "chr1 1 2", present[0]])
        assert match.tolist() == [0, -1, 0] and flags.tolist() == [1, 0, 1] and n_flagged == 2


# ------------------------------------------------------------------ GPU: query vectors bit for bit
@pytest.mark.gpu
@pytest.mark.parametrize("cap", [None, DIM * 16 * 7])
def test_query_vectors_equal_finalize_query_bit_for_bit(synth, cap):
    from morna_b200.batch_query import QueryFile
    search = _search(synth["base"])
    qf = QueryFile(search, synth["qpath"])
    order, Q = oracle_queries(synth["qlines"], synth["freq"], synth["sample_count"], DIM)
    assert np.array_equal(qf.sample_ids, order)
    assert qf.n_merged > 0
    if cap is not None:
        assert len(qf.slices(cap)) > 1
    got = qf.all_vectors(cap)
    assert got.shape == Q.shape
    assert np.array_equal(got.view(np.int64), Q.view(np.int64)), "rows differ: %s" % np.nonzero((got != Q).any(1))[0][:10]
    zero = order.tolist().index(8801)
    assert not Q[zero].any() and Q[order.tolist().index(5)].any()


def _many_sample_lines(rng, keys, freq, n_samples):
    passing = [k for k in keys if k in freq]
    lines = []
    for i in range(250):
        n = min(int(rng.integers(50, 400)), n_samples)
        s = np.sort(rng.choice(n_samples, n, replace=False)) + 1
        key = passing[i % len(passing)] if i % 7 else "chr20 %d %d" % (i, i + 9)
        lines.append(_row(key, s.tolist(), rng.integers(1, 50, n).tolist()))
    return lines


@pytest.mark.gpu
@pytest.mark.parametrize("n_samples", [40, 6000])
def test_batch_exact_search_equals_exact_search_device(synth, n_samples):
    import torch
    from morna_b200.batch_query import QueryFile, search_query_file
    rng = np.random.default_rng(n_samples)
    lines = _many_sample_lines(rng, synth["keys"], synth["freq"], n_samples)
    path = str(synth["tmp"] / ("many_%d.tsv" % n_samples))
    with open(path, "w") as fh:
        fh.write("".join(lines))
    search = _search(synth["base"])
    order, Q = oracle_queries(lines, synth["freq"], synth["sample_count"], DIM)
    assert (len(order) > 4096) if n_samples > 4096 else (len(order) < 64)   # (a sample may be drawn by no row)
    assert np.array_equal(QueryFile(search, path).all_vectors().view(np.int64), Q.view(np.int64))
    k = 15
    want_i, want_d = search.exact_search_device(torch.from_numpy(Q).cuda(), k)
    want_i, want_d = want_i.cpu().numpy(), want_d.cpu().numpy()
    for cap in (None, DIM * 16 * 1500):
        got = list(search_query_file(search, path, k, exact=True, cap=cap))
        if n_samples > 4096:
            assert len(got) > 1
        sid = np.concatenate([g[0] for g in got])
        ids = np.concatenate([g[1] for g in got])
        d = np.concatenate([g[2] for g in got])
        assert np.array_equal(sid, order)
        assert np.array_equal(ids, want_i)
        assert np.array_equal(d.view(np.int64), want_d.view(np.int64))
    approx = list(search_query_file(search, path, k, exact=False))           # the fp16 pass without the re-rank
    assert np.array_equal(np.concatenate([g[0] for g in approx]), order)
    a_d = np.concatenate([g[2] for g in approx])
    assert np.abs(a_d - want_d).max() < 2e-3                                 # sqrt(2 - 2 score): off by ~1e-4


def _cli(argv, stdin=None):
    out = io.StringIO()
    assert cli.main(argv, stdin=stdin, stdout=out, stderr=io.StringIO()) == 0
    return out.getvalue().splitlines()


def _by_query(lines):
    groups = {}
    for line in lines:
        sid, rest = line.split("\t", 1)
        groups.setdefault(int(sid), []).append(rest)
    return groups


@pytest.mark.gpu
def test_cli_query_file_lines_equal_single_query_search(synth):
    from morna_b200 import parse
    base, k = synth["base"], 12
    lines = _cli(["search", "-x", base, "--query-intropolis", synth["qpath"], "-e", "-d", "-r", str(k)])
    groups = _by_query(lines)
    order, _ = oracle_queries(synth["qlines"], synth["freq"], synth["sample_count"], DIM)
    assert list(groups) == order.tolist()                       # first-seen order, each query's lines together
    picks = [8801, 5, 12, 7, 9001] + order[::9].tolist()       # the all-zero query, merged pairs, outside the index
    for sid in picks:
        raw = []
        for line in synth["qlines"]:
            key, samples, covs = parse.tokenize_line(line)
            for s, c in zip(samples, covs):
                if s == sid:
                    raw.append("%s\t%d\n" % (key.replace(" ", "\t"), c))
        single = _cli(["search", "-x", base, "-f", "raw", "-e", "-d", "-r", str(k)], stdin=io.StringIO("".join(raw)))
        assert groups[sid] == single, "sample %d" % sid


@pytest.mark.gpu
def test_cli_tiny_intropolis_as_index_and_query_goes_through_the_sparse_path(tmp_path):
    import torch
    from morna_b200 import files
    base = str(tmp_path / "tiny")
    tsv = os.path.join(GOLDEN, "tiny_intropolis.tsv")
    assert cli.main(["index", "--intropolis", tsv, "-x", base], stdout=io.StringIO()) == 0
    search = _search(base)
    assert search.csr is not None and search.sparse_exact
    with open(tsv) as fh:
        qlines = fh.readlines()
    order, Q = oracle_queries(qlines, files.read_freq(base), files.read_stats(base)[0], 3000)
    lines = _cli(["search", "-x", base, "--query-intropolis", tsv, "-e", "-d", "-r", "5"])
    groups = _by_query(lines)
    assert list(groups) == order.tolist()
    want_i, want_d = search.exact_search_device(torch.from_numpy(Q).cuda(), 5)
    want_i, want_d = want_i.cpu().numpy(), want_d.cpu().numpy()
    for j in range(0, len(order), 97):
        assert groups[int(order[j])] == ["%d.\t%d\t%s" % (r + 1, want_i[j, r], cli.py2_str(float(want_d[j, r]))) for r in range(5)]


@pytest.mark.gpu
def test_cli_all_samples_lines_equal_search_by_id(synth):
    from morna_b200 import files
    base, k = synth["base"], 10
    id_map = files.read_map(base)
    inv = {v: s for s, v in id_map.items()}
    for flags, n_meta in ((["-e", "-d"], 0), (["-d", "-m"], 1)):
        lines = _cli(["search", "-x", base, "--all-samples", "-r", str(k)] + flags)
        groups = _by_query(lines)
        assert list(groups) == [inv[i] for i in range(len(id_map))]          # internal-id order
        for sid in list(groups)[::23] + [inv[len(id_map) - 1]]:
            single = _cli(["search", "-x", base, "-q", str(sid), "-e", "-r", str(k)] + flags)
            assert single[:2] == ["querying by sample id %d" % sid, "this is internal id %d" % id_map[sid]]
            assert groups[sid] == single[2:], "sample %d" % sid
        if n_meta:
            assert any(l.split("\t")[-1] != "None" for l in lines)
