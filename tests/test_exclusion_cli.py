"""`search --exclude-self` / `--exclude-group FILE`: the refusals (exit 2, one message, before any GPU work) on the CPU,
and on the GPU every sample query mode against the unexcluded run's full lists with the query's group removed and the
ranks renumbered."""
import argparse
import io

import numpy as np
import pytest

from morna_b200 import cli, files
from tests.test_filtered_search_cli import _lines, _run, synth_index  # noqa: F401  (synth_index: a module fixture)


@pytest.fixture
def mapped(tmp_path, monkeypatch):
    """A basename with only a .map.mor (sample ids 10, 20, 30, 40 -> internal ids 0..3); opening the index fails the
    test, so a refusal provably comes before any GPU work."""
    base = str(tmp_path / "idx")
    files.write_map(base, {10: 0, 20: 1, 30: 2, 40: 3})

    def no_gpu(*args, **kw):
        raise AssertionError("the index was opened")
    monkeypatch.setattr(cli, "open_search", no_gpu)
    return base, tmp_path


MODES = [["-q", "10", "-e"], ["--all-samples"], ["--query-intropolis", "q.tsv", "-e"], ["-q", "10", "--max-distance", "0.5"],
         ["--all-samples", "--max-distance", "0.5"], ["--query-intropolis", "q.tsv", "-e", "--max-distance", "0.5"]]


def _refused(argv, stdin=None):
    code, out, err = _run(argv, stdin=stdin or io.StringIO(""))
    assert code == 2 and out == "" and len(err.strip().splitlines()) == 1, (code, out, err)
    return err


@pytest.mark.parametrize("mode", MODES)
def test_both_flags_are_refused(mapped, mode):
    base, tmp = mapped
    (tmp / "groups").write_text("10\tA\n")
    err = _refused(["search", "-x", base, "--exclude-self", "--exclude-group", str(tmp / "groups")] + mode)
    assert "--exclude-self cannot be combined with --exclude-group" in err


@pytest.mark.parametrize("fmt", [[], ["-f", "sam"], ["-f", "bed"], ["-f", "raw"], ["-e", "--max-distance", "0.5"]])
def test_a_stdin_query_is_refused(mapped, fmt):
    base, tmp = mapped
    (tmp / "groups").write_text("10\tA\n")
    for flag in (["--exclude-self"], ["--exclude-group", str(tmp / "groups")]):
        assert "no sample id" in _refused(["search", "-x", base] + flag + fmt, io.StringIO("chr1\t10\t20\t3\n"))


def test_query_intropolis_without_exact_is_refused(mapped):
    base, tmp = mapped
    for extra in ([], ["--max-distance", "0.5"]):
        assert "needs -e" in _refused(["search", "-x", base, "--exclude-self", "--query-intropolis", "q.tsv"] + extra)


@pytest.mark.parametrize("mode", MODES)
def test_unreadable_file_is_refused(mapped, mode):
    base, tmp = mapped
    (tmp / "binary").write_bytes(b"\xff\xfe\x00\x81\n")
    for path in (str(tmp / "missing"), str(tmp), str(tmp / "binary")):
        assert "cannot read" in _refused(["search", "-x", base, "--exclude-group", path] + mode)


@pytest.mark.parametrize("mode", MODES)
def test_malformed_lines_are_refused_by_number(mapped, mode):
    base, tmp = mapped
    cases = (("10\tA\n\n20\n", 3, "not 'sample_id<TAB>group'"), ("10\tA\n20\tB\tC\n", 2, "not 'sample_id<TAB>group'"),
             ("10\tA\n20\t \n", 2, "not 'sample_id<TAB>group'"), ("s7\tA\n", 1, "integer sample id"),
             ("2.5\tA\n", 1, "integer sample id"), ("10 A\n", 1, "not 'sample_id<TAB>group'"))
    for text, line, what in cases:
        (tmp / "groups").write_text(text)
        err = _refused(["search", "-x", base, "--exclude-group", str(tmp / "groups")] + mode)
        assert "line %d" % line in err and what in err, (text, err)


@pytest.mark.parametrize("mode", MODES)
def test_one_sample_in_two_groups_is_refused(mapped, mode):
    base, tmp = mapped
    (tmp / "groups").write_text("10\tA\n20\tA\n 10 \tB\n")
    err = _refused(["search", "-x", base, "--exclude-group", str(tmp / "groups")] + mode)
    assert "sample id 10" in err and "two different groups" in err and "lines 1 and 3" in err


def test_labels_of_a_group_file(tmp_path):
    base = str(tmp_path / "idx")
    files.write_map(base, {10: 0, 20: 1, 30: 2, 40: 3})
    files.write_stats(base, 4, 4, 8)
    (tmp_path / "groups").write_text("\n  30\tSRP1 \n10\tSRP2\n99\tSRP1\n30\tSRP1\n")

    def ns(**kw):
        base_kw = dict(basename=base, query_id=10, all_samples=False, query_intropolis=None, exact=True,
                       exclude_self=False, exclude_group=None)
        base_kw.update(kw)
        return argparse.Namespace(**base_kw)
    assert cli.exclusion(ns()) is None
    ex = cli.exclusion(ns(exclude_group=str(tmp_path / "groups")))
    # SRP1 = 0, SRP2 = 1; samples 20 and 40 are groups of their own: n_groups + internal id
    assert ex.row_labels.tolist() == [1, 2 + 1, 0, 2 + 3]
    # a listed sample outside the index still names its group; an unknown sample excludes nothing
    assert ex.labels_of_samples([99, 20, 30, 55]).tolist() == [0, 3, 0, -1]
    ex = cli.exclusion(ns(exclude_self=True))
    assert ex.row_labels.tolist() == [0, 1, 2, 3]


# ------------------------------------------------------------------ GPU: every sample query mode
def drop_group(lines, excluded, prefixed, header=0, limit=None):
    """Result lines without the ids `excluded(query)` names, renumbered from 1 per query and cut to `limit`."""
    out, rank = list(lines[:header]), {}
    for line in lines[header:]:
        f = line.split("\t")
        query, rest = (f[0], f[1:]) if prefixed else ("", f)
        if int(rest[1]) in excluded(query):
            continue
        rank[query] = rank.get(query, 0) + 1
        if limit is not None and rank[query] > limit:
            continue
        out.append("\t".join(([query] if prefixed else []) + ["%d." % rank[query]] + rest[1:]))
    return out


@pytest.mark.gpu
def test_all_samples_exclude_self_equals_k_plus_one_without_the_self_line(synth_index):  # noqa: F811
    base, id_map = synth_index["base"], synth_index["map"]
    k = 7
    got = _lines(["search", "-x", base, "--all-samples", "-d", "-r", str(k), "--exclude-self"])
    assert not any(id_map[int(l.split("\t")[0])] == int(l.split("\t")[2]) for l in got)
    wider = _lines(["search", "-x", base, "--all-samples", "-d", "-r", str(k + 1)])
    assert got == drop_group(wider, lambda q: {id_map[int(q)]}, True, limit=k) and len(got) == k * len(id_map)


@pytest.mark.gpu
def test_every_sample_mode_with_a_group_file_equals_the_full_lists_without_the_group(synth_index, tmp_path):  # noqa: F811
    base, size, id_map = synth_index["base"], synth_index["size"], synth_index["map"]
    sids = sorted(id_map)
    rng = np.random.default_rng(11)
    study = {s: "SRP%d" % rng.integers(0, 12) for s in rng.choice(sids, len(sids) * 2 // 3, replace=False).tolist()}
    study[999999] = "SRP3"                                   # listed, not indexed
    path = tmp_path / "groups"
    path.write_text("".join("%d\t%s\n" % kv for kv in study.items()))
    members = {}
    for s, g in study.items():
        members.setdefault(g, set()).add(id_map.get(s, -1))

    def excluded(q):
        s = int(q)
        return members[study[s]] if s in study else {id_map[s]} if s in id_map else set()
    flag = ["--exclude-group", str(path)]
    # -q: top-k and range
    for sid in (sids[0], sids[len(sids) // 2], max(s for s in sids if s not in study)):
        full = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", size])
        got = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", "9"] + flag)
        assert got == drop_group(full, lambda q: excluded(sid), False, header=2, limit=9) and len(got) > 2
        R = float(full[len(full) // 3].split("\t")[2]) + 1e-9
        got = _lines(["search", "-x", base, "-q", str(sid), "-d", "--max-distance", repr(R)] + flag)
        want = drop_group(full, lambda q: excluded(sid), False, header=2)
        assert got == want[:2] + [l for l in want[2:] if float(l.split("\t")[2]) <= R]
    # --all-samples and --query-intropolis -e: top-k and range
    for mode in (["--all-samples"], ["--query-intropolis", synth_index["qpath"]]):
        full = _lines(["search", "-x", base] + mode + ["-e", "-d", "-r", size])
        got = _lines(["search", "-x", base] + mode + ["-e", "-d", "-r", "5"] + flag)
        assert got == drop_group(full, excluded, True, limit=5) and len(got) > 0, mode
        # (the median 5th-nearest distance: every query keeps a few samples in range)
        R = float(np.median([float(l.split("\t")[3]) for l in full if l.split("\t")[1] == "5."])) + 1e-9
        got = _lines(["search", "-x", base] + mode + ["-e", "-d", "--max-distance", repr(R)] + flag)
        assert got == [l for l in drop_group(full, excluded, True) if float(l.split("\t")[3]) <= R] and len(got) > 0
    # with a subset: the group leaves the subset's lists too
    keep_file = tmp_path / "keep"
    keep_file.write_text("".join("%d\n" % s for s in sids[::2]))
    keep = {id_map[s] for s in sids[::2]}
    full = _lines(["search", "-x", base, "--all-samples", "-e", "-d", "-r", size])
    got = _lines(["search", "-x", base, "--all-samples", "-e", "-d", "-r", "4", "--samples", str(keep_file)] + flag)
    want = drop_group([l for l in full if int(l.split("\t")[0]) in set(sids[::2])],
                      lambda q: excluded(q) | (set(id_map.values()) - keep), True, limit=4)
    assert got == want and len(got) > 0


def test_rows_sharded_search_refuses_an_exclusion():
    from morna_b200 import dist
    for call in (lambda: dist.sharded_exact_search(None, None, 10, query_groups=[0]),
                 lambda: dist.sharded_batched_search(None, None, 10, query_groups=[0]),
                 lambda: dist.sharded_range_search(None, None, 0.5, query_groups=[0]),
                 lambda: list(dist.sharded_range_search_groups(None, None, 0.5, query_groups=[0]))):
        with pytest.raises(ValueError, match="no per-query exclusion"):
            call()
