"""`search --max-distance` on the command line, without a GPU: the radius and flag checks, and the parsers it leaves alone."""
import io

import numpy as np
import pytest

from morna_b200 import cli


@pytest.mark.parametrize("argv", [
    ["--max-distance", "-1"],
    ["--max-distance", "-0.000001"],
    ["--max-distance", "nan"],
    ["--max-distance", "inf"],
    ["--max-distance=-inf"],
    ["--max-distance", "0.5", "-rl"],
    ["--max-distance", "0.5", "-rl", "-q", "3"],
])
def test_bad_radius_and_rawlist_exit_2(argv):
    err = io.StringIO()
    assert cli.main(["search", "-x", "no_such_index"] + argv, stdout=io.StringIO(), stderr=err) == 2
    assert "--max-distance" in err.getvalue()


def test_batch_modes_with_max_distance_still_refuse_other_query_sources():
    err = io.StringIO()
    argv = ["search", "-x", "no_such_index", "--max-distance", "1", "--all-samples", "-q", "3"]
    assert cli.main(argv, stdout=io.StringIO(), stderr=err) == 2
    assert "cannot be combined" in err.getvalue()


def test_junctions_has_no_max_distance():
    p = cli.build_parser()
    with pytest.raises(SystemExit) as exc:
        p.parse_args(["junctions", "-x", "i", "-i", "a", "--junction-file", "b", "-sf", "c", "--max-distance", "1"])
    assert exc.value.code == 2


def test_parser_defaults_unchanged():
    p = cli.build_parser()
    s = p.parse_args(["search", "-x", "idx"])
    assert (s.results, s.max_distance, s.exact, s.format, s.rawlist) == (20, None, False, "sam", False)
    assert "results" not in getattr(s, "given", ())
    s = p.parse_args(["search", "-x", "idx", "--max-distance", "0.25", "-r", "7"])
    assert (s.max_distance, s.results) == (0.25, 7) and "results" in s.given
    j = p.parse_args(["junctions", "-x", "i", "-i", "a", "--junction-file", "b", "-sf", "c"])
    assert j.results == 20 and not hasattr(j, "max_distance")


def test_cut_lists_keeps_the_first_entries_of_each_list():
    from morna_b200.batch_query import cut_lists
    off = np.array([0, 3, 3, 8], np.int64)
    ids = np.arange(8, dtype=np.int32)
    d = np.arange(8, dtype=np.float64) / 10
    o, i, dd = cut_lists(off, ids, d, 2)
    assert o.tolist() == [0, 2, 2, 4] and i.tolist() == [0, 1, 3, 4] and dd.tolist() == [0.0, 0.1, 0.3, 0.4]
    assert cut_lists(off, ids, d, None)[1] is ids


def test_write_results_prints_csr_batches():
    from morna_b200.batch_query import write_results
    out = io.StringIO()
    write_results(out, np.array([11, 12, 13]), np.array([4, 2, 7], np.int32), np.array([0.0, 0.5, 1.25]), True, None, None,
                  offsets=np.array([0, 2, 2, 3], np.int64))
    assert out.getvalue().splitlines() == ["11\t1.\t4\t0.0", "11\t2.\t2\t0.5", "13\t1.\t7\t1.25"]


def test_check_radius():
    from morna_b200.search import check_radius
    assert check_radius(0) == 0.0 and check_radius("1.5") == 1.5
    for bad in (-1e-300, float("nan"), float("inf"), float("-inf")):
        with pytest.raises(ValueError):
            check_radius(bad)
