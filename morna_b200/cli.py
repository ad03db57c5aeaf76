"""`morna.py index` / `morna.py search` command line of the reference
(morna.py:876-1054, dispatch :1338-1484) in front of the B200 kernels.

Kept: every flag of the two subcommands, stdin for the query, the
"rank.<TAB>id[<TAB>distance][<TAB>metadata]" result lines with Python 2's float
formatting, progress messages, the two extra stdout lines of -q.
Different on purpose: without -e the reference asks Annoy for approximate
neighbours; there is no forest here -- the approximate mode is the tensor-core
scoring pass without the exact re-rank (MornaSearch.search_nn; --search-k,
--n-trees, -b are accepted and ignored), -e is the exact search.  `-q ID -e` runs the exact
search with the stored row as the query (the reference ignores -e after -q).
-m works as in the reference (index: metadata file -> <basename>.meta.mor; search: keywords joined to the results).
The `junctions` subcommand and the convergence back-off loop are outside the hot path and exit with a message.
"""
import argparse
import math
import sys

import numpy as np

_help_intro = "morna (B200-native hot path): index and exactly search junction feature vectors"


def py2_str(v):
    """Python 2 str(): floats print 12 significant digits (morna.py:126 uses str())."""
    if isinstance(v, float):
        s = "%.12g" % v
        if s.lstrip("-").isdigit():
            s += ".0"
        return s
    if isinstance(v, tuple) and len(v) == 1 and isinstance(v[0], str):
        return "(u" + repr(v[0]) + ",)"          # a metadata row as Python 2 prints the sqlite tuple of one unicode string
    return str(v)


def results_output(results, out=None):
    """morna.py:116-127."""
    out = out or sys.stdout
    for i in range(len(results[0])):
        out.write(str(i + 1) + ".")
        for column in results:
            out.write("\t" + py2_str(column[i]))
        out.write("\n")


class _StoreGiven(argparse._StoreAction):
    """A store action that also records that the flag was given (its default cannot tell)."""

    def __call__(self, parser, namespace, values, option_string=None):
        super().__call__(parser, namespace, values, option_string)
        namespace.given = getattr(namespace, "given", frozenset()) | {self.dest}


def add_search_parameters(sub):
    sub.add_argument("-x", "--basename", metavar="<idx>", type=str, required=True,
                     help="path to junction index basename for search")
    sub.add_argument("-v", "--verbose", action="store_const", const=True, default=False, help="be talkative")
    sub.add_argument("--search-k", metavar="<int>", type=int, required=False, default=100,
                     help="accepted for compatibility; the exact search ignores it")
    sub.add_argument("-f", "--format", metavar="<choice>", type=str, required=False, default="sam", action=_StoreGiven,
                     help="one of {sam, bed, raw}")
    sub.add_argument("-d", "--distances", action="store_const", const=True, default=False,
                     help="include distances to nearest neighbors")
    sub.add_argument("-m", "--metadata", action="store_const", const=True, default=False,
                     help="display results mapped to metadata")
    sub.add_argument("-c", "--convergence-backoff", metavar="<int>", type=int, required=False, default=None,
                     help="not supported (the reference calls it non-functional)")
    sub.add_argument("-ch", "--checkpoint", metavar="<int>", type=int, required=False, default=0,
                     help="not supported")
    sub.add_argument("-q", "--query-id", metavar="<int>", type=int, required=False, default=None,
                     help="search for nearest neighbors of the indexed sample with this sample id")
    sub.add_argument("-e", "--exact", action="store_const", const=True, default=False,
                     help="exact nearest neighbor search (always on in this implementation)")
    sub.add_argument("-r", "--results", metavar="<int>", type=int, required=False, default=20, action=_StoreGiven,
                     help="the number of nearest neighbor results to return (with --max-distance: given, at most this "
                          "many per query)")
    sub.add_argument("-rl", "--rawlist", action="store_const", const=True, default=False,
                     help="regurgitate junction list for input sample instead of performing search")


def build_parser():
    parser = argparse.ArgumentParser(description=_help_intro)
    subs = parser.add_subparsers(dest="subparser_name",
                                 help='subcommands; add "-h" or "--help" after a subcommand for its parameters')
    index_parser = subs.add_parser("index", help="creates a morna index")
    search_parser = subs.add_parser("search", help="searches a morna index")
    index_parser.add_argument("--intropolis", metavar="<file>", type=str, required=True,
                              help="path to (gzipped) file recording junctions across samples in intropolis format")
    index_parser.add_argument("-x", "--basename", metavar="<str>", type=str, required=False, default="morna",
                              help="basename path of junction index files to create")
    index_parser.add_argument("--features", metavar="<int>", type=int, required=False, default=3000,
                              help="dimension of feature space")
    index_parser.add_argument("--n-trees", metavar="<int>", type=int, required=False, default=200,
                              help="accepted for compatibility; no Annoy forest is built")
    index_parser.add_argument("-s", "--sample-count", metavar="<int>", type=int, required=False, default=None,
                              help="optionally specify number of unique samples to speed indexing")
    index_parser.add_argument("-t", "--sample-threshold", metavar="<int>", type=int, required=False, default=100,
                              help="minimum number of samples in which a junction should appear")
    index_parser.add_argument("-b", "--buffer-size", metavar="<int>", type=int, required=False, default=1024,
                              help="accepted for compatibility (junction database buffer)")
    index_parser.add_argument("-v", "--verbose", action="store_const", const=True, default=False,
                              help="be talkative")
    index_parser.add_argument("-m", "--metafile", metavar="<file>", type=str, required=False, default=None,
                              help="metadata file: sample id then keywords per line; stored in <basename>.meta.mor for search -m")
    index_parser.add_argument("--no-junction-shards", action="store_const", const=True, default=False,
                              help="do not write the <basename>.shXX.junc.mor shards (only `junctions` reads them)")
    add_search_parameters(search_parser)
    search_parser.add_argument("--query-intropolis", metavar="<file>", type=str, required=False, default=None,
                               help="(gzipped) intropolis-format file: search for every sample it lists, one line per "
                                    "result prefixed by the sample id and a tab")
    search_parser.add_argument("--all-samples", action="store_const", const=True, default=False,
                               help="search for every indexed sample (as -q for each sample id), one line per result "
                                    "prefixed by the sample id and a tab; with --samples / --exclude-samples, for every "
                                    "sample of the subset (the k-NN or range graph of the subset)")
    search_parser.add_argument("--samples", metavar="<file>", type=str, required=False, default=None,
                               help="search only among these indexed samples: a file with one sample id per line")
    search_parser.add_argument("--exclude-samples", metavar="<file>", type=str, required=False, default=None,
                               help="search among every indexed sample except these: a file with one sample id per line")
    search_parser.add_argument("--exclude-self", action="store_const", const=True, default=False,
                               help="leave each query's own sample out of its results (-q, --all-samples, "
                                    "--query-intropolis -e): the most similar OTHER samples")
    search_parser.add_argument("--exclude-group", metavar="<file>", type=str, required=False, default=None,
                               help="a file of 'sample_id<TAB>group' lines (a group is any string, e.g. a study "
                                    "accession): leave each query's own sample and every sample of its group out of its "
                                    "results (-q, --all-samples, --query-intropolis -e)")
    search_parser.add_argument("--max-distance", metavar="<float>", type=float, required=False, default=None,
                               help="return every sample within this angular distance of the query (exact; -r N, if "
                                    "given, keeps the first N per query)")
    search_parser.add_argument("--max-per-group", metavar="<int>", type=int, required=False, default=None,
                               help="return at most this many samples of any one group (--groups) per query: the nearest "
                                    "samples, skipping a sample once this many of its group are listed (exact only)")
    search_parser.add_argument("--groups", metavar="<file>", type=str, required=False, default=None,
                               help="the groups --max-per-group caps: a file of 'sample_id<TAB>group' lines, as for "
                                    "--exclude-group; a sample not listed is a group of its own")
    search_parser.add_argument("--within-group", metavar="<file>", type=str, required=False, default=None,
                               help="a file of 'sample_id<TAB>group' lines, as for --exclude-group: each query searches "
                                    "only the samples of its own group (-q, --all-samples, --query-intropolis -e); a "
                                    "sample not listed is a group of its own")
    junctions_parser = subs.add_parser("junctions", help="extracts the junctions of a query's nearest neighbors")
    add_search_parameters(junctions_parser)                      # morna.py:1023-1054
    junctions_parser.add_argument("-i", "--index", metavar="<idx>", type=str, required=True,
                                  help="index basename or directory of the aligner (kept for compatibility)")
    junctions_parser.add_argument("-p1", "--pass1-sam", metavar="<sam>", type=str, required=False, default="pass1.sam",
                                  help="filename for first pass alignment file output by aligner")
    junctions_parser.add_argument("--junction-filter", type=str, required=False, default=".05,5",
                                  help="retain junctions found in at least {first part} of the result samples, or "
                                       "with at least {second part} coverage in any one result sample")
    junctions_parser.add_argument("--junction-file", type=str, metavar="<gz>", required=True,
                                  help="gzipped file with junction rows in the order of the file the index was made from")
    junctions_parser.add_argument("-sf", "--splicefile", type=str, metavar="<file>", required=True,
                                  help="output intropolis-like file with the retained junctions")
    return parser


def sample_filter(args):
    """--samples / --exclude-samples: the internal ids of the samples to search among (numpy int64, ascending), or None
    without either flag.  Raises ValueError with the message for the user when the flags or the file are not usable."""
    given = [(flag, path) for flag, path in (("--samples", getattr(args, "samples", None)),
                                             ("--exclude-samples", getattr(args, "exclude_samples", None))) if path is not None]
    if not given:
        return None
    if len(given) > 1:
        raise ValueError("--samples cannot be combined with --exclude-samples")
    flag, path = given[0]
    try:
        with open(path) as fh:
            lines = fh.read().splitlines()
    except (OSError, UnicodeDecodeError) as exc:
        raise ValueError("%s: cannot read %s: %s" % (flag, path, exc))
    listed = {}
    for number, line in enumerate(lines, 1):
        text = line.strip()
        if not text:
            continue
        try:
            listed.setdefault(int(text), number)
        except ValueError:
            raise ValueError("%s: line %d of %s is not an integer sample id: %r" % (flag, number, path, text))
    import numpy as np
    from . import files
    id_map = files.read_map(args.basename)
    for sample_id, number in listed.items():
        if sample_id not in id_map:
            raise ValueError("%s: sample id %d (line %d of %s) is not in the index: no internal id is mapped to that "
                             "sample id" % (flag, sample_id, number, path))
    keep = flag == "--samples"
    ids = np.array(sorted(iid for sid, iid in id_map.items() if (sid in listed) == keep), dtype=np.int64)
    if ids.size == 0:
        raise ValueError("%s: no sample is left to search among" % flag)
    return ids


class Exclusion(object):
    """--exclude-self / --exclude-group: every indexed sample carries a label, and a query leaves out every sample whose
    label equals its own.  Listed groups are numbered densely (0 .. n_groups-1, in order of first appearance); a sample
    not listed is a group of its own, labelled n_groups + its internal id.  So a query's own sample is always left out."""

    def __init__(self, group_of, id_map, index_size):
        self.group_of, self.id_map = group_of, id_map           # sample id -> group number; sample id -> internal id
        n_groups = len(set(group_of.values()))
        self.row_labels = np.arange(n_groups, n_groups + index_size, dtype=np.int64)
        for sample_id, g in group_of.items():
            iid = id_map.get(sample_id)
            if iid is not None:
                self.row_labels[iid] = g
        if self.row_labels.size and self.row_labels.max() > np.iinfo(np.int32).max:
            raise ValueError("too many exclusion groups for int32 labels")
        self.row_labels = self.row_labels.astype(np.int32)

    def labels_of_samples(self, sample_ids):
        """Labels of queries named by sample id (--query-intropolis): the group of a listed or indexed sample, else -1
        (nothing left out)."""
        out = np.full(len(sample_ids), -1, dtype=np.int32)
        for j, sid in enumerate(np.asarray(sample_ids).tolist()):
            if sid in self.group_of:
                out[j] = self.group_of[sid]
            elif sid in self.id_map:
                out[j] = self.row_labels[self.id_map[sid]]
        return out


def read_group_file(flag, path):
    """A file of 'sample_id<TAB>group' lines -> {sample id: group number} (groups numbered densely in order of first
    appearance; whitespace stripped, blank lines skipped).  Raises ValueError with the message for the user."""
    group_of = {}
    try:
        with open(path) as fh:
            lines = fh.read().splitlines()
    except (OSError, UnicodeDecodeError) as exc:
        raise ValueError("%s: cannot read %s: %s" % (flag, path, exc))
    numbers, first_line = {}, {}
    for number, line in enumerate(lines, 1):
        text = line.strip()
        if not text:
            continue
        fields = text.split("\t")
        if len(fields) != 2 or not fields[1].strip():
            raise ValueError("%s: line %d of %s is not 'sample_id<TAB>group': %r" % (flag, number, path, text))
        try:
            sample_id = int(fields[0].strip())
        except ValueError:
            raise ValueError("%s: line %d of %s does not start with an integer sample id: %r" % (flag, number, path, text))
        g = numbers.setdefault(fields[1].strip(), len(numbers))
        if group_of.setdefault(sample_id, g) != g:
            raise ValueError("%s: sample id %d is listed with two different groups (lines %d and %d of %s)"
                             % (flag, sample_id, first_line[sample_id], number, path))
        first_line.setdefault(sample_id, number)
    return group_of


def cap_groups(args):
    """--max-per-group N --groups FILE: (N, int32 cap label per internal id -- the group number of a listed sample, -1
    for one not listed, which is never capped), or None without either flag.  Raises ValueError with the message for
    the user when the flags, the query mode or the file are not usable (before any GPU work)."""
    n, path = getattr(args, "max_per_group", None), getattr(args, "groups", None)
    if n is None and path is None:
        return None
    if n is None:
        raise ValueError("--groups needs --max-per-group")
    if path is None:
        raise ValueError("--max-per-group needs --groups")
    if n < 1:
        raise ValueError("--max-per-group must be at least 1")
    if args.rawlist:
        raise ValueError("-rl cannot be combined with --max-per-group")
    if args.query_id is None and not args.all_samples and not args.exact and args.max_distance is None:
        raise ValueError("--max-per-group needs -e or --max-distance: the approximate mode has no cap per group")
    group_of = read_group_file("--groups", path)
    from . import files
    labels = np.full(files.read_stats(args.basename)[1], -1, dtype=np.int32)
    for sample_id, iid in files.read_map(args.basename).items():
        labels[iid] = group_of.get(sample_id, -1)
    return n, labels


def exclusion(args):
    """--exclude-self / --exclude-group: an Exclusion, or None without either flag.  Raises ValueError with the message
    for the user when the flags, the query mode or the file are not usable (before any GPU work)."""
    self_only, path = getattr(args, "exclude_self", False), getattr(args, "exclude_group", None)
    if not self_only and path is None:
        return None
    flag = "--exclude-self" if self_only else "--exclude-group"
    if self_only and path is not None:
        raise ValueError("--exclude-self cannot be combined with --exclude-group")
    if args.query_id is None and not args.all_samples and args.query_intropolis is None:
        raise ValueError("%s needs queries that are samples (-q, --all-samples or --query-intropolis): a query read "
                         "from stdin has no sample id" % flag)
    if args.query_intropolis is not None and not args.exact:
        raise ValueError("%s with --query-intropolis needs -e: the approximate mode has no exclusion" % flag)
    group_of = read_group_file(flag, path) if path is not None else {}
    from . import files
    index_size = files.read_stats(args.basename)[1]
    return Exclusion(group_of, files.read_map(args.basename), index_size)


def within_group(args):
    """--within-group FILE: an Exclusion whose labels are the groups each query searches within, or None without the
    flag.  Raises ValueError with the message for the user when the flags, the query mode or the file are not usable
    (before any GPU work)."""
    path = getattr(args, "within_group", None)
    if path is None:
        return None
    for other, flag in (("exclude_group", "--exclude-group"), ("max_per_group", "--max-per-group")):
        if getattr(args, other, None) is not None:
            raise ValueError("--within-group cannot be combined with %s" % flag)
    if args.query_id is None and not args.all_samples and args.query_intropolis is None:
        raise ValueError("--within-group needs queries that are samples (-q, --all-samples or --query-intropolis): a "
                         "query read from stdin has no sample id")
    if args.query_intropolis is not None and not args.exact:
        raise ValueError("--within-group with --query-intropolis needs -e: the approximate mode has no within-group "
                         "search")
    group_of = read_group_file("--within-group", path)
    from . import files
    return Exclusion(group_of, files.read_map(args.basename), files.read_stats(args.basename)[1])


def within_member(searcher, args, within, exclude_self, max_distance, limit, out):
    """-q --within-group: the result columns of the queried sample against the samples of its own group."""
    from .batch_query import inverse_map
    from .search import _member_internal_id
    from . import files
    internal_id = _member_internal_id(searcher.internal_id_map, args.query_id, out)
    ids = np.array([internal_id], dtype=np.int64)
    groups = within.labels_of_samples([args.query_id])
    exclude = ids.astype(np.int32) if exclude_self else None
    if max_distance is None:
        r_ids, r_d = (t.cpu().numpy()[0] for t in searcher.within_group_search(ids, args.results, groups, exclude))
        r_ids, r_d = r_ids[r_ids >= 0], r_d[r_ids >= 0]
    else:
        _, r_ids, r_d = (t.cpu().numpy() for t in searcher.within_group_range(ids, max_distance, groups, exclude))
        if limit is not None:
            r_ids, r_d = r_ids[:max(limit, 0)], r_d[:max(limit, 0)]
    results = (r_ids.tolist(),)
    if args.distances:
        results += (r_d.tolist(),)
    if args.metadata:
        results += (files.read_meta(args.basename, inverse_map(searcher)[r_ids].tolist()),)
    return results


def open_search(basename, keep, keep_parent_rows, excl=None, cap=None):
    """The index's MornaSearch, or with `keep` (sample_filter's ids) a FilteredSearch over those samples; with `excl`
    (an Exclusion) every row carries its label, with `cap` (cap_groups' result) its cap label."""
    from .search import MornaSearch
    searcher = MornaSearch(basename=basename)
    if excl is not None:
        searcher.set_row_groups(excl.row_labels)
    if cap is not None:
        searcher.set_cap_groups(cap[1])
    return searcher if keep is None else searcher.subset(keep, keep_parent_rows)


def main(argv=None, stdin=None, stdout=None, stderr=None):
    stdin, stdout, stderr = stdin or sys.stdin, stdout or sys.stdout, stderr or sys.stderr
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.subparser_name is None:
        parser.print_help(stderr)
        return 2
    if args.subparser_name == "index":
        from .index import go_index
        go_index(args.intropolis, args.basename, args.features, args.n_trees, args.sample_count,
                 args.sample_threshold, args.buffer_size, args.verbose, args.metafile, out=stdout,
                 junction_shards=not args.no_junction_shards)
        return 0

    from . import parse
    if args.convergence_backoff:
        stderr.write("convergence back-off is not supported (see README of the reference: non-functional)\n")
        return 2
    max_distance = getattr(args, "max_distance", None)
    if max_distance is not None:
        if not (math.isfinite(max_distance) and max_distance >= 0.0):
            stderr.write("--max-distance must be a finite number >= 0\n")
            return 2
        if args.rawlist:
            stderr.write("-rl cannot be combined with --max-distance\n")
            return 2
    # a range search lists everything within the radius; an explicit -r caps each list
    limit = args.results if max_distance is not None and "results" in getattr(args, "given", ()) else None
    try:
        keep = sample_filter(args)
        within = within_group(args) if args.subparser_name == "search" else None
        excl = exclusion(args) if args.subparser_name == "search" else None
        cap = cap_groups(args) if args.subparser_name == "search" else None
    except ValueError as exc:
        stderr.write(str(exc) + "\n")
        return 2
    per_group = cap[0] if cap is not None else None
    if getattr(args, "query_intropolis", None) is not None or getattr(args, "all_samples", False):
        return batch_search(args, stdout, stderr, max_distance, limit, keep, excl, cap, within)
    opened = None
    if args.subparser_name == "junctions":                      # morna.py:1351-1353
        args.format = "sam"
        stdin = opened = open(args.pass1_sam)
    # (a filter keeps the whole index's rows only for -q, whose sample may lie outside the subset)
    # (with --within-group the rows carry its labels; --exclude-self then leaves out the query's own row only)
    searcher = open_search(args.basename, keep, keep_parent_rows=args.query_id is not None, excl=within or excl, cap=cap)
    if args.query_id is not None:                               # morna.py:1358-1365
        if within is not None:
            results = within_member(searcher, args, within, excl is not None, max_distance, limit, stdout)
        elif max_distance is not None:
            results = searcher.search_member_n(args.query_id, limit, include_distances=args.distances,
                                               meta_db=args.metadata, out=stdout, max_distance=max_distance,
                                               exclude=excl is not None, max_per_group=per_group)
        else:
            results = searcher.search_member_n(args.query_id, args.results, args.search_k,
                                               include_distances=args.distances, meta_db=args.metadata, out=stdout,
                                               exclude=excl is not None, max_per_group=per_group)
        results_output(results, stdout)
        return 0
    if args.format == "sam":                                    # :1367-1373
        junctions = parse.junctions_from_sam_stream(stdin)
    elif args.format == "bed":
        junctions = parse.junctions_from_bed_stream(stdin)
    else:
        assert args.format == "raw"
        junctions = parse.junctions_from_raw_stream(stdin)
    if args.rawlist:                                            # :1374-1377
        for junction in junctions:
            stdout.write(str(junction) + "\n")
        return 0
    for i, junction in enumerate(junctions):                    # :1456-1473
        if args.verbose and i % 1000 == 0:
            stderr.write(str(i) + " junctions into query sample\r")
            stderr.flush()
        if " ".join(str(t) for t in junction[:3]) in searcher.sample_frequencies:
            searcher.update_query(junction)
    searcher.finalize_query()
    if args.verbose:
        stderr.write("\n")
    if max_distance is not None:                                # always exact: -e changes nothing
        results = searcher.range_search_nn(max_distance, include_distances=args.distances, meta_db=args.metadata,
                                           num_neighbors=limit, max_per_group=per_group)
    elif args.exact:                                            # :1477-1483
        results = searcher.exact_search_nn(args.results, include_distances=args.distances, meta_db=args.metadata,
                                           max_per_group=per_group)
    else:
        results = searcher.search_nn(args.results, args.search_k, include_distances=args.distances, meta_db=args.metadata)
    results_output(results, stdout)
    if args.subparser_name == "junctions":                      # :1486-1632
        from .junctions import go_junctions
        go_junctions(args, searcher, results, stdout, stderr)
        opened.close()
    return 0


def batch_search(args, stdout, stderr, max_distance=None, limit=None, keep=None, excl=None, cap=None, within=None):
    """--query-intropolis / --all-samples: many queries in one run, results streamed in 4096-query batches.  With
    `max_distance`, every sample within it per query (CSR batches), each list cut to `limit` entries if given.  With
    `keep` (sample_filter's ids), the search runs over those samples only.  With `excl` (an Exclusion), each query
    leaves out the samples of its group.  With `cap` (cap_groups' result), at most N samples per group.  With `within`
    (within_group's Exclusion), each query searches the samples of its own group only, and `excl` (--exclude-self) leaves
    out its own sample."""
    from . import batch_query
    named = [name for name, on in (("--query-intropolis", args.query_intropolis is not None),
                                   ("--all-samples", args.all_samples), ("-q", args.query_id is not None),
                                   ("-rl", args.rawlist), ("-f", "format" in getattr(args, "given", ()))) if on]
    if len(named) > 1:
        stderr.write("%s cannot be combined with %s\n" % (named[0], ", ".join(named[1:])))
        return 2
    # (with an exclusion, --all-samples over a subset takes its labels from the whole index's rows)
    searcher = open_search(args.basename, keep, keep_parent_rows=False, excl=within or excl, cap=cap)
    per_group = cap[0] if cap is not None else None
    inverse = batch_query.inverse_map(searcher)
    meta = args.basename if args.metadata else None
    if within is not None:
        k = None if max_distance is not None else args.results
        if args.all_samples:
            results = batch_query.search_all_samples_within(searcher, inverse, within.row_labels, k, max_distance,
                                                            exclude_self=excl is not None)
        else:
            own = (lambda sids: np.array([within.id_map.get(s, -1) for s in sids.tolist()], dtype=np.int32)) \
                if excl is not None else None
            results = batch_query.search_query_file_within(searcher, args.query_intropolis, within.labels_of_samples, own,
                                                           k, max_distance)
        for batch in results:
            offsets = batch[1] if max_distance is not None else None
            batch_query.write_results(stdout, batch[0], batch[-2], batch[-1], args.distances, meta, inverse,
                                      offsets=offsets, limit=limit)
        return 0
    exclude = excl is not None
    query_labels = excl.labels_of_samples if exclude else None
    if max_distance is not None:
        if args.all_samples:
            results = batch_query.search_all_samples_range(searcher, max_distance, inverse, exclude=exclude,
                                                           max_per_group=per_group)
        else:
            results = batch_query.search_query_file_range(searcher, args.query_intropolis, max_distance,
                                                          query_labels=query_labels, max_per_group=per_group)
        for sample_ids, offsets, ids, dists in results:
            batch_query.write_results(stdout, sample_ids, ids, dists, args.distances, meta, inverse, offsets=offsets, limit=limit)
        return 0
    if args.all_samples:                       # the stored rows as queries: exact, as -q is
        results = batch_query.search_all_samples(searcher, args.results, inverse, exclude=exclude, max_per_group=per_group)
    else:
        results = batch_query.search_query_file(searcher, args.query_intropolis, args.results, exact=args.exact,
                                                query_labels=query_labels, max_per_group=per_group)
    for sample_ids, ids, dists in results:
        batch_query.write_results(stdout, sample_ids, ids, dists, args.distances, meta, inverse)
    return 0


if __name__ == "__main__":
    sys.exit(main())
