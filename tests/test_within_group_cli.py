"""`search --within-group FILE`: the refusals (exit 2, one message, before any GPU work) on the CPU, and on the GPU every
sample query mode x {top-k, --max-distance} x {plain, --exclude-self, --samples} against the unrestricted run's full
lists with every sample outside the query's group removed and the ranks renumbered."""
import io

import numpy as np
import pytest

from tests.test_exclusion_cli import MODES, _refused, drop_group, mapped  # noqa: F401  (mapped: a fixture)
from tests.test_filtered_search_cli import _lines, synth_index  # noqa: F401  (synth_index: a module fixture)


def _groups(tmp, text="10\tA\n"):
    (tmp / "groups").write_text(text)
    return ["--within-group", str(tmp / "groups")]


@pytest.mark.parametrize("mode", MODES)
def test_other_group_flags_are_refused(mapped, mode):  # noqa: F811
    base, tmp = mapped
    flag = _groups(tmp)
    err = _refused(["search", "-x", base] + flag + ["--exclude-group", str(tmp / "groups")] + mode)
    assert "--within-group cannot be combined with --exclude-group" in err
    for cap in (["--max-per-group", "2"], ["--max-per-group", "2", "--groups", str(tmp / "groups")]):
        err = _refused(["search", "-x", base] + flag + cap + mode)
        assert "--within-group cannot be combined with --max-per-group" in err


@pytest.mark.parametrize("fmt", [[], ["-f", "sam"], ["-f", "bed"], ["-f", "raw"], ["-e", "--max-distance", "0.5"],
                                 ["--exclude-self"]])
def test_a_stdin_query_is_refused(mapped, fmt):  # noqa: F811
    base, tmp = mapped
    err = _refused(["search", "-x", base] + _groups(tmp) + fmt, io.StringIO("chr1\t10\t20\t3\n"))
    assert "--within-group" in err and "no sample id" in err


def test_query_intropolis_without_exact_is_refused(mapped):  # noqa: F811
    base, tmp = mapped
    for extra in ([], ["--max-distance", "0.5"], ["--exclude-self"]):
        err = _refused(["search", "-x", base] + _groups(tmp) + ["--query-intropolis", "q.tsv"] + extra)
        assert "needs -e" in err


@pytest.mark.parametrize("mode", MODES)
def test_unreadable_file_is_refused(mapped, mode):  # noqa: F811
    base, tmp = mapped
    (tmp / "binary").write_bytes(b"\xff\xfe\x00\x81\n")
    for path in (str(tmp / "missing"), str(tmp), str(tmp / "binary")):
        err = _refused(["search", "-x", base, "--within-group", path] + mode)
        assert "--within-group" in err and "cannot read" in err


@pytest.mark.parametrize("mode", MODES)
def test_malformed_lines_are_refused_by_number(mapped, mode):  # noqa: F811
    base, tmp = mapped
    cases = (("10\tA\n\n20\n", 3, "not 'sample_id<TAB>group'"), ("10\tA\n20\tB\tC\n", 2, "not 'sample_id<TAB>group'"),
             ("s7\tA\n", 1, "integer sample id"), ("10 A\n", 1, "not 'sample_id<TAB>group'"))
    for text, line, what in cases:
        err = _refused(["search", "-x", base] + _groups(tmp, text) + mode)
        assert "line %d" % line in err and what in err, (text, err)


@pytest.mark.parametrize("mode", MODES)
def test_one_sample_in_two_groups_is_refused(mapped, mode):  # noqa: F811
    base, tmp = mapped
    err = _refused(["search", "-x", base] + _groups(tmp, "10\tA\n20\tA\n10\tB\n") + mode)
    assert "sample id 10" in err and "two different groups" in err and "lines 1 and 3" in err


def test_the_flag_belongs_to_search_only():
    from morna_b200 import cli
    with pytest.raises(SystemExit):
        cli.build_parser().parse_args(["index", "--intropolis", "f", "--within-group", "g"])


# ------------------------------------------------------------------ GPU: every sample query mode
@pytest.mark.gpu
def test_every_sample_mode_equals_the_full_lists_inside_the_group(synth_index, tmp_path):  # noqa: F811
    base, size, id_map = synth_index["base"], synth_index["size"], synth_index["map"]
    sids = sorted(id_map)
    rng = np.random.default_rng(5)
    study = {s: "SRP%d" % rng.integers(0, 9) for s in rng.choice(sids, len(sids) * 2 // 3, replace=False).tolist()}
    study[999999] = "SRP2"                                   # listed, not indexed
    path = tmp_path / "groups"
    path.write_text("".join("%d\t%s\n" % kv for kv in study.items()))
    members = {}
    for s, g in study.items():
        if s in id_map:
            members.setdefault(g, set()).add(id_map[s])
    every = set(id_map.values())
    keep_sids = set(sids[::2])
    keep = {id_map[s] for s in keep_sids}
    keep_file = tmp_path / "keep"
    keep_file.write_text("".join("%d\n" % s for s in sorted(keep_sids)))

    def outside(self_too, subset):
        def excluded(q):
            s = int(q)
            inside = members[study[s]] if s in study else {id_map[s]} if s in id_map else set()
            if self_too and s in id_map:
                inside = inside - {id_map[s]}
            if subset:
                inside = inside & keep
            return every - inside
        return excluded
    flag = ["--within-group", str(path)]
    variants = [([], False, False), (["--exclude-self"], True, False), (["--samples", str(keep_file)], False, True),
                (["--exclude-self", "--samples", str(keep_file)], True, True)]
    # -q: a sample in a large group, one of its own (not listed) and, with a filter, one outside the subset
    unlisted = min(s for s in sids if s not in study)
    for sid in (sids[0], sids[len(sids) // 2], unlisted, min(set(sids) - keep_sids)):
        full = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", size])
        for extra, self_too, subset in variants:
            excluded = outside(self_too, subset)
            got = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", "6"] + flag + extra)
            assert got == drop_group(full, lambda q: excluded(sid), False, header=2, limit=6), (sid, extra)
            want = drop_group(full, lambda q: excluded(sid), False, header=2)
            R = float(want[len(want) // 2 + 1].split("\t")[2]) + 1e-9 if len(want) > 3 else 0.5
            got = _lines(["search", "-x", base, "-q", str(sid), "-d", "--max-distance", repr(R)] + flag + extra)
            assert got == want[:2] + [l for l in want[2:] if float(l.split("\t")[2]) <= R], (sid, extra)
    # --all-samples and --query-intropolis -e: top-k, range, range with -r
    for mode in (["--all-samples"], ["--query-intropolis", synth_index["qpath"]]):
        full = _lines(["search", "-x", base] + mode + ["-e", "-d", "-r", size])
        for extra, self_too, subset in variants:
            excluded = outside(self_too, subset)
            lines = full
            if subset and mode == ["--all-samples"]:              # (the subset's samples are the queries)
                lines = [l for l in full if int(l.split("\t")[0]) in keep_sids]
            want = drop_group(lines, excluded, True)
            got = _lines(["search", "-x", base] + mode + ["-e", "-d", "-r", "5"] + flag + extra)
            assert got == drop_group(lines, excluded, True, limit=5) and len(got) > 0, (mode, extra)
            R = float(np.median([float(l.split("\t")[3]) for l in want if l.split("\t")[1] == "3."])) + 1e-9
            got = _lines(["search", "-x", base] + mode + ["-e", "-d", "--max-distance", repr(R)] + flag + extra)
            assert got == [l for l in want if float(l.split("\t")[3]) <= R] and len(got) > 0, (mode, extra)
            got = _lines(["search", "-x", base] + mode + ["-e", "-d", "--max-distance", repr(R), "-r", "2"] + flag + extra)
            assert got == [l for l in drop_group(lines, excluded, True, limit=2) if float(l.split("\t")[3]) <= R]
