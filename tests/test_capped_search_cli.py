"""`search --max-per-group N --groups FILE`: the refusals (exit 2, one message, before any GPU work) on the CPU, and on the
GPU every query mode against the uncapped run's full lists, walked (a sample kept iff fewer than N of its group were kept
before it) and renumbered."""
import io

import numpy as np
import pytest

from tests.test_exclusion_cli import _refused, drop_group, mapped  # noqa: F401  (mapped: a fixture)
from tests.test_filtered_search_cli import _lines, synth_index  # noqa: F401  (synth_index: a module fixture)

MODES = [["-q", "10", "-e"], ["--all-samples"], ["--query-intropolis", "q.tsv", "-e"], ["-q", "10", "--max-distance", "0.5"],
         ["--all-samples", "--max-distance", "0.5"], ["--query-intropolis", "q.tsv", "--max-distance", "0.5"],
         ["-e"], ["--max-distance", "0.5"]]


def _cap(tmp, n="2", text="10\tA\n20\tA\n"):
    (tmp / "groups").write_text(text)
    return ["--max-per-group", n, "--groups", str(tmp / "groups")]


@pytest.mark.parametrize("mode", MODES)
def test_bad_caps_are_refused(mapped, mode):
    base, tmp = mapped
    for n in ("0", "-3"):
        assert "--max-per-group must be at least 1" in _refused(["search", "-x", base] + _cap(tmp, n) + mode)
    assert "--max-per-group needs --groups" in _refused(["search", "-x", base, "--max-per-group", "2"] + mode)
    assert "--groups needs --max-per-group" in _refused(["search", "-x", base, "--groups", str(tmp / "groups")] + mode)


def test_rawlist_and_approximate_mode_are_refused(mapped):
    base, tmp = mapped
    assert "-rl cannot be combined" in _refused(["search", "-x", base, "-rl"] + _cap(tmp), io.StringIO("chr1\t10\t20\t3\n"))
    for mode in ([], ["-f", "bed"], ["--query-intropolis", "q.tsv"]):
        err = _refused(["search", "-x", base] + _cap(tmp) + mode, io.StringIO("chr1\t10\t20\t3\n"))
        assert "needs -e or --max-distance" in err, (mode, err)


@pytest.mark.parametrize("mode", MODES)
def test_group_file_errors_are_refused(mapped, mode):
    base, tmp = mapped
    (tmp / "binary").write_bytes(b"\xff\xfe\x00\x81\n")
    for path in (str(tmp / "missing"), str(tmp), str(tmp / "binary")):
        assert "cannot read" in _refused(["search", "-x", base, "--max-per-group", "1", "--groups", path] + mode)
    for text, line in (("10\tA\n\n20\n", 3), ("s7\tA\n", 1), ("10\tA\n20\tB\tC\n", 2)):
        err = _refused(["search", "-x", base] + _cap(tmp, "1", text) + mode)
        assert "--groups" in err and "line %d" % line in err, (text, err)
    err = _refused(["search", "-x", base] + _cap(tmp, "1", "10\tA\n20\tA\n 10 \tB\n") + mode)
    assert "sample id 10" in err and "two different groups" in err and "lines 1 and 3" in err


# ------------------------------------------------------------------ GPU: every query mode
def capped(lines, group_of, m, prefixed, header=0, limit=None, dropped=lambda q: set()):
    """Full result lines walked per query: a line kept iff fewer than m lines of its group were kept before it (ids
    `dropped(query)` names are left out first), renumbered from 1 and cut to `limit`."""
    out, kept, seen = list(lines[:header]), {}, {}
    for line in lines[header:]:
        f = line.split("\t")
        query, rest = (f[0], f[1:]) if prefixed else ("", f)
        iid = int(rest[1])
        if iid in dropped(query):
            continue
        g = group_of.get(iid)
        if g is not None:
            if seen.get((query, g), 0) >= m:
                continue
            seen[(query, g)] = seen.get((query, g), 0) + 1
        kept[query] = kept.get(query, 0) + 1
        if limit is not None and kept[query] > limit:
            continue
        out.append("\t".join(([query] if prefixed else []) + ["%d." % kept[query]] + rest[1:]))
    return out


@pytest.mark.gpu
def test_every_query_mode_equals_the_walked_full_lists(synth_index, tmp_path):  # noqa: F811
    base, size, id_map = synth_index["base"], synth_index["size"], synth_index["map"]
    sids = sorted(id_map)
    rng = np.random.default_rng(5)
    study = {s: "SRP%d" % rng.integers(0, 6) for s in rng.choice(sids, len(sids) * 3 // 4, replace=False).tolist()}
    study[999999] = "SRP1"                                    # listed, not indexed
    path = tmp_path / "groups"
    path.write_text("".join("%d\t%s\n" % kv for kv in study.items()))
    group_of = {id_map[s]: g for s, g in study.items() if s in id_map}
    for m in (1, 2):
        flag = ["--max-per-group", str(m), "--groups", str(path)]
        for sid in (sids[0], sids[len(sids) // 2]):
            full = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", size])
            got = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", "6"] + flag)
            assert got == capped(full, group_of, m, False, header=2, limit=6) and len(got) > 2
            R = float(full[len(full) // 2].split("\t")[2]) + 1e-9
            got = _lines(["search", "-x", base, "-q", str(sid), "-d", "--max-distance", repr(R), "-r", "4"] + flag)
            want = capped(full, group_of, m, False, header=2)
            assert got == (want[:2] + [l for l in want[2:] if float(l.split("\t")[2]) <= R])[:6]
        for mode in (["--all-samples"], ["--query-intropolis", synth_index["qpath"]]):
            full = _lines(["search", "-x", base] + mode + ["-e", "-d", "-r", size])
            got = _lines(["search", "-x", base] + mode + ["-e", "-d", "-r", "5"] + flag)
            assert got == capped(full, group_of, m, True, limit=5) and len(got) > 0, mode
            R = float(np.median([float(l.split("\t")[3]) for l in full if l.split("\t")[1] == "8."])) + 1e-9
            got = _lines(["search", "-x", base] + mode + ["-e", "-d", "--max-distance", repr(R)] + flag)
            assert got == [l for l in capped(full, group_of, m, True) if float(l.split("\t")[3]) <= R] and len(got) > 0
    # with --samples and --exclude-group: the cap walks what the filter and the exclusion leave
    keep_file = tmp_path / "keep"
    keep_file.write_text("".join("%d\n" % s for s in sids[::2]))
    keep = {id_map[s] for s in sids[::2]}
    members = {}
    for s, g in study.items():
        members.setdefault(g, set()).add(id_map.get(s, -1))

    def dropped(q):
        s = int(q)
        out = members[study[s]] if s in study else {id_map[s]}
        return out | (set(id_map.values()) - keep)
    full = _lines(["search", "-x", base, "--all-samples", "-e", "-d", "-r", size])
    got = _lines(["search", "-x", base, "--all-samples", "-e", "-d", "-r", "4", "--samples", str(keep_file),
                  "--exclude-group", str(path), "--max-per-group", "1", "--groups", str(path)])
    want = capped([l for l in full if int(l.split("\t")[0]) in set(sids[::2])], group_of, 1, True, limit=4, dropped=dropped)
    assert got == want and len(got) > 0
