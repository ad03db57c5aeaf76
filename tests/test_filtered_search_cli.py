"""`search --samples` / `--exclude-samples`: the refusals (exit 2, one message, before any GPU work) on the CPU, and on
the GPU every query mode x {top-k, --max-distance} x {--samples, --exclude-samples} against the unfiltered run's full
lists restricted to the subset and renumbered."""
import argparse
import gzip
import io

import numpy as np
import pytest

from morna_b200 import cli, files


def _run(argv, stdin=None):
    out, err = io.StringIO(), io.StringIO()
    code = cli.main(argv, stdin=stdin, stdout=out, stderr=err)
    return code, out.getvalue(), err.getvalue()


@pytest.fixture
def mapped(tmp_path):
    """A basename with only a .map.mor (sample ids 10, 20, 30, 40 -> internal ids 0..3): enough for the refusals."""
    base = str(tmp_path / "idx")
    files.write_map(base, {10: 0, 20: 1, 30: 2, 40: 3})
    return base, tmp_path


MODES = [[], ["-q", "10"], ["--all-samples"], ["--query-intropolis", "q.tsv"], ["--max-distance", "0.5"],
         ["--all-samples", "--max-distance", "0.5"]]


def _refused(argv, stdin=None):
    code, out, err = _run(argv, stdin=stdin or io.StringIO(""))
    assert code == 2 and out == "" and len(err.strip().splitlines()) == 1, (code, out, err)
    return err


@pytest.mark.parametrize("mode", MODES)
def test_both_flags_are_refused(mapped, mode):
    base, tmp = mapped
    (tmp / "ids").write_text("10\n")
    err = _refused(["search", "-x", base, "--samples", str(tmp / "ids"), "--exclude-samples", str(tmp / "ids")] + mode)
    assert "--samples cannot be combined with --exclude-samples" in err


@pytest.mark.parametrize("flag", ["--samples", "--exclude-samples"])
@pytest.mark.parametrize("mode", MODES)
def test_unreadable_file_is_refused(mapped, flag, mode):
    base, tmp = mapped
    for path in (str(tmp / "missing"), str(tmp)):                # no such file; a directory
        assert "cannot read" in _refused(["search", "-x", base, flag, path] + mode)
    (tmp / "binary").write_bytes(b"\xff\xfe\x00\x81\n")
    assert "cannot read" in _refused(["search", "-x", base, flag, str(tmp / "binary")] + mode)


@pytest.mark.parametrize("flag", ["--samples", "--exclude-samples"])
@pytest.mark.parametrize("mode", MODES)
def test_a_line_that_is_not_an_integer_is_refused_by_number(mapped, flag, mode):
    base, tmp = mapped
    for text, line in (("10\n\n  sample7 \n", 3), ("10\n2.5\n", 2), ("10 20\n", 1)):
        (tmp / "ids").write_text(text)
        err = _refused(["search", "-x", base, flag, str(tmp / "ids")] + mode)
        assert "line %d" % line in err and "not an integer" in err


@pytest.mark.parametrize("flag", ["--samples", "--exclude-samples"])
@pytest.mark.parametrize("mode", MODES)
def test_a_sample_id_not_in_the_index_is_refused_by_name(mapped, flag, mode):
    base, tmp = mapped
    (tmp / "ids").write_text("10\n 20 \n77\n30\n")
    err = _refused(["search", "-x", base, flag, str(tmp / "ids")] + mode)
    assert "sample id 77" in err and "line 3" in err


@pytest.mark.parametrize("mode", MODES)
def test_an_empty_subset_is_refused(mapped, mode):
    base, tmp = mapped
    (tmp / "none").write_text("\n  \n")
    (tmp / "all").write_text("40\n30\n20\n10\n10\n")
    for argv in (["--samples", str(tmp / "none")], ["--exclude-samples", str(tmp / "all")]):
        assert "no sample is left" in _refused(["search", "-x", base] + argv + mode)


def test_sample_filter_reads_ids_with_whitespace_blank_lines_and_repeats(mapped):
    base, tmp = mapped
    (tmp / "ids").write_text("  30\n\n10\t\n30\n")

    def ns(**kw):
        return argparse.Namespace(basename=base, **kw)
    assert cli.sample_filter(ns()) is None
    assert cli.sample_filter(ns(samples=str(tmp / "ids"), exclude_samples=None)).tolist() == [0, 2]
    assert cli.sample_filter(ns(samples=None, exclude_samples=str(tmp / "ids"))).tolist() == [1, 3]


def test_parser_flags_belong_to_search_only():
    p = cli.build_parser()
    s = p.parse_args(["search", "-x", "idx"])
    assert s.samples is None and s.exclude_samples is None
    assert p.parse_args(["search", "-x", "idx", "--exclude-samples", "f"]).exclude_samples == "f"
    with pytest.raises(SystemExit):
        p.parse_args(["junctions", "-x", "i", "-i", "a", "--junction-file", "b", "-sf", "c", "--samples", "f"])


# ------------------------------------------------------------------ GPU: every query mode against the restricted full lists
def _lines(argv, stdin=None):
    code, out, err = _run(argv, stdin)
    assert code == 0, err
    return out.splitlines()


def restrict(lines, keep_iids, prefixed, header=0, keep_queries=None, limit=None):
    """Result lines kept where the internal id is in `keep_iids` (and, prefixed, the query's sample id is in
    `keep_queries` when given), renumbered from 1 per query and cut to `limit` per query."""
    out, rank = list(lines[:header]), {}
    for line in lines[header:]:
        f = line.split("\t")
        query, rest = (f[0], f[1:]) if prefixed else ("", f)
        if int(rest[1]) not in keep_iids or (keep_queries is not None and int(query) not in keep_queries):
            continue
        rank[query] = rank.get(query, 0) + 1
        if limit is not None and rank[query] > limit:
            continue
        out.append("\t".join(([query] if prefixed else []) + ["%d." % rank[query]] + rest[1:]))
    return out


def _sam(junctions):
    """SAM lines with one spliced read per unit of coverage (10M<gap>N10M covers start..end)."""
    lines = []
    for chrom, start, end, cov in junctions:
        read = "r\t0\t%s\t%d\t60\t10M%dN10M\t*\t0\t0\t%s\t%s\n" % (chrom, start - 10, end - start + 1, "A" * 20, "I" * 20)
        lines += [read] * cov
    return "".join(lines)


def _bed(junctions):
    """One BED12 line with two 10-base blocks per junction (start..end between them)."""
    return "".join("%s\t%d\t%d\tj\t%d\t+\t0\t0\t0\t2\t10,10\t0,%d\n" % (c, s - 11, e + 10, cov, e - s + 11)
                   for c, s, e, cov in junctions)


@pytest.fixture(scope="module")
def synth_index(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("filtered_cli")
    rng = np.random.default_rng(23)
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
    id_map = files.read_map(base)
    sids = np.array(sorted(id_map))
    picked = np.random.default_rng(3).choice(sids, len(sids) // 3, replace=False)
    (tmp / "picked").write_text("".join("  %d \n\n" % s for s in np.concatenate([picked, picked[:5]])))
    junctions = [tuple(l.split("\t")[:3]) + (5,) for l in lines[:40:2]]
    junctions = [(c, int(s), int(e), cov) for c, s, e, cov in junctions]
    return {"base": base, "qpath": qpath, "size": str(files.read_stats(base)[1]), "map": id_map,
            "picked": set(int(s) for s in picked), "file": str(tmp / "picked"), "junctions": junctions}


@pytest.mark.gpu
@pytest.mark.parametrize("flag", ["--samples", "--exclude-samples"])
def test_every_query_mode_equals_the_restricted_full_lists(synth_index, flag):
    base, size, id_map = synth_index["base"], synth_index["size"], synth_index["map"]
    kept_sids = {s for s in id_map if (s in synth_index["picked"]) == (flag == "--samples")}
    keep = {id_map[s] for s in kept_sids}
    filt = [flag, synth_index["file"]]
    full_raw = "".join("%s\t%d\t%d\t%d\n" % j for j in synth_index["junctions"])
    full = _lines(["search", "-x", base, "-f", "raw", "-e", "-d", "-r", size], io.StringIO(full_raw))
    # (just above a printed distance: the lines carry 12 significant digits, so a radius equal to a printed value could
    # fall between a row's true distance and its rounding)
    R = float(full[len(full) // 4].split("\t")[2]) + 1e-9
    stdin = {"raw": full_raw, "bed": _bed(synth_index["junctions"]), "sam": _sam(synth_index["junctions"])}
    for fmt, text in stdin.items():
        for exact in (["-e"], []):
            # (-r beyond the subset's size: the approximate mode answers such a k exactly)
            got = _lines(["search", "-x", base, "-f", fmt, "-d", "-r", size] + exact + filt, io.StringIO(text))
            assert got == restrict(full, keep, False) and len(got) > 0, (fmt, exact)
        got = _lines(["search", "-x", base, "-f", fmt, "-d", "-e", "-r", "7", "-m"] + filt, io.StringIO(text))
        with_meta = _lines(["search", "-x", base, "-f", fmt, "-e", "-d", "-m", "-r", size], io.StringIO(text))
        assert got == restrict(with_meta, keep, False, limit=7)
        got = _lines(["search", "-x", base, "-f", fmt, "-d", "--max-distance", repr(R)] + filt, io.StringIO(text))
        want = [l for l in restrict(full, keep, False) if float(l.split("\t")[2]) <= R]
        assert got == want and len(got) > 0, fmt
    # -q: a sample inside the subset and one outside it (which cannot return itself)
    inside, outside = min(kept_sids), min(set(id_map) - kept_sids)
    for sid in (inside, outside):
        full_q = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", size])
        got = _lines(["search", "-x", base, "-q", str(sid), "-e", "-d", "-r", "9"] + filt)
        assert got == restrict(full_q, keep, False, header=2, limit=9) and len(got) > 2
        want = restrict(full_q, keep, False, header=2)
        got = _lines(["search", "-x", base, "-q", str(sid), "-d", "--max-distance", repr(R)] + filt)
        assert got == want[:2] + [l for l in want[2:] if float(l.split("\t")[2]) <= R]
    assert str(id_map[outside]) not in [l.split("\t")[1] for l in got[2:]]
    # --query-intropolis (with and without -e) and --all-samples (only the subset's samples query), -m too
    for mode, queries in ((["--query-intropolis", synth_index["qpath"]], None), (["--all-samples"], kept_sids)):
        full_b = _lines(["search", "-x", base] + mode + ["-e", "-d", "-m", "-r", size])
        for exact in (["-e"], []):
            got = _lines(["search", "-x", base] + mode + exact + ["-d", "-m", "-r", size] + filt)
            assert got == restrict(full_b, keep, True, keep_queries=queries) and len(got) > 0, (mode, exact)
            if queries is not None:
                assert {int(l.split("\t")[0]) for l in got} == kept_sids
        got = _lines(["search", "-x", base] + mode + ["-e", "-d", "-m", "-r", "3"] + filt)
        assert got == restrict(full_b, keep, True, keep_queries=queries, limit=3)
        got = _lines(["search", "-x", base] + mode + ["-d", "-m", "--max-distance", repr(R)] + filt)
        want = [l for l in restrict(full_b, keep, True, keep_queries=queries) if float(l.split("\t")[3]) <= R]
        assert got == want and len(got) > 0, mode
        # an explicit -r caps each range list (lists are sorted, so the first two within R are the first two, if in R)
        got = _lines(["search", "-x", base] + mode + ["-d", "--max-distance", repr(R), "-r", "2"] + filt)
        assert got == ["\t".join(l.split("\t")[:4]) for l in restrict(full_b, keep, True, keep_queries=queries, limit=2)
                       if float(l.split("\t")[3]) <= R]
