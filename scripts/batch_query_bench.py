"""`morna search --query-intropolis` end to end on synthetic gzipped intropolis files: an index of --samples samples at
--features, then a query file of --queries new samples, timed per phase (each phase ends in a device synchronise),
next to the route that exists for one query: MornaSearch.finalize_query per sample plus exact_search_nn, on a slice of
the same samples.  Also times the host-dict join that the device junction table replaces."""
import argparse, gzip, io, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--samples", type=int, default=50000)
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--index-pairs", type=float, default=20e6)
ap.add_argument("--queries", type=int, default=8192)
ap.add_argument("--query-pairs", type=float, default=20e6)
ap.add_argument("--k", type=int, default=20)
ap.add_argument("--baseline-queries", type=int, default=32)
args = ap.parse_args()

import torch
print("device: %s" % torch.cuda.get_device_name(0), flush=True)
try:
    print("nvidia-smi: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                          capture_output=True, text=True, timeout=60).stdout.strip(), flush=True)
except (OSError, subprocess.SubprocessError) as exc:
    print("nvidia-smi: not available (%s)" % exc, flush=True)

rng = np.random.default_rng(7)
tmp = tempfile.mkdtemp()


def write_file(path, n_pairs, n_samples, sample_base, keys=None, new_key_share=0.0):
    """Rows as index_e2e_bench.py makes them: lognormal row lengths, ascending sample lists, geometric coverages."""
    rows, out_keys, total = [], [], 0
    order = iter(rng.permutation(len(keys)).tolist() if keys is not None else [])
    while total < n_pairs:
        n = int(min(n_samples, max(1, rng.lognormal(5.0, 1.5))))
        s = np.sort(rng.choice(n_samples, size=n, replace=False)) + sample_base
        c = 1 + rng.geometric(0.5, size=n)
        pick = next(order, None) if rng.random() >= new_key_share else None
        if pick is not None:
            key = keys[pick]
        else:
            key = "chr%d\t%d\t%d" % (rng.integers(1, 23), rng.integers(10000, 240000000), rng.integers(10000, 240000000))
        rows.append("%s\t+\tGT\tAG\t%s\t%s\n" % (key, ",".join(map(str, s.tolist())), ",".join(map(str, c.tolist()))))
        out_keys.append(key)
        total += n
    with gzip.open(path, "wb", compresslevel=1) as fh:
        fh.write("".join(rows).encode())
    return out_keys, total


t0 = time.perf_counter()
index_path, query_path = os.path.join(tmp, "index.tsv.gz"), os.path.join(tmp, "query.tsv.gz")
index_keys, index_pairs = write_file(index_path, args.index_pairs, args.samples, 1)
# query rows: each junction once, as in an intropolis file; four fifths of them junctions of the index
query_keys, query_pairs = write_file(query_path, args.query_pairs, args.queries, 10 ** 6, keys=index_keys, new_key_share=0.2)
print("synthetic files: index %d rows / %d pairs over %d samples, query %d rows / %d pairs over %d samples (%.0f s)" % (
    len(index_keys), index_pairs, args.samples, len(query_keys), query_pairs, args.queries, time.perf_counter() - t0), flush=True)

from morna_b200 import batch_query, parse
from morna_b200.index import go_index
from morna_b200.search import MornaSearch
base = os.path.join(tmp, "idx")
go_index(index_path, base, args.features, 0, None, 100, 1024, False, None, out=io.StringIO(), junction_shards=False)
search = MornaSearch(basename=base)
print("index: %d samples kept, %d junctions in .freq.mor, dim %d" % (search.index_size, len(search.sample_frequencies), search.dim), flush=True)
inverse = batch_query.inverse_map(search)

for run in range(2):                      # run 0 builds the junction table; run 1 finds it on the object
    times, last = {}, [time.perf_counter()]

    def mark(name):
        torch.cuda.synchronize()
        now = time.perf_counter()
        times[name] = now - last[0]
        last[0] = now

    start = last[0]
    qf = batch_query.QueryFile(search, query_path, on_phase=mark)
    mark("ids")
    vecs = [qf.query_vectors(lo, hi) for lo, hi in qf.slices()]
    mark("accumulate_transpose")
    results = []
    for v in vecs:
        for ids, d in search.search_batches((v[b:b + batch_query.BATCH_QUERIES] for b in range(0, v.shape[0], batch_query.BATCH_QUERIES)), args.k):
            results.append((ids.copy(), d.copy()))
    mark("search_and_d2h")
    out, lo = io.StringIO(), 0
    for ids, d in results:
        batch_query.write_results(out, qf.sample_ids[lo:lo + ids.shape[0]], ids, d, True, None, inverse)
        lo += ids.shape[0]
    mark("output_format")
    total = time.perf_counter() - start
    print("run %d: %d queries from %d rows / %d pairs (%d pairs merged on the host), %d output lines" % (
        run, qf.nq, qf.n_rows, qf.nnz, qf.n_merged, out.getvalue().count("\n")), flush=True)
    for name in ("read_tokenize", "h2d", "hash", "table_build", "lookup", "ids", "accumulate_transpose", "search_and_d2h", "output_format"):
        print("  %-22s %9.2f ms" % (name, 1e3 * times[name]), flush=True)
    print("  end to end             %9.2f ms  -> %.0f queries/s" % (1e3 * total, qf.nq / total), flush=True)

# the host-dict join the device table replaces: one key decode + dict test per row
packed, key_off, row_off, sample, cov = batch_query.read_rows(query_path)
kb = packed.tobytes()
freq = search.sample_frequencies
t0 = time.perf_counter()
hits = sum(1 for i in range(len(key_off) - 1) if kb[key_off[i]:key_off[i + 1]].decode() in freq)
t_dict = time.perf_counter() - t0
print("host dict join of the same %d rows: %.2f ms (%d hits)" % (len(key_off) - 1, 1e3 * t_dict, hits), flush=True)

# the existing route for one query: finalize_query per sample (per-junction Python) + exact_search_nn, on a slice
lens = np.diff(row_off)
row_of_pair = np.repeat(np.arange(len(lens)), lens)
keys = [kb[key_off[i]:key_off[i + 1]].decode() for i in range(len(key_off) - 1)]
slice_ids = qf.sample_ids[:args.baseline_queries]
t_total = 0.0
for sid in slice_ids.tolist():
    where = np.nonzero(sample == sid)[0]
    junctions = [tuple(keys[row_of_pair[p]].split(" ")) + (int(cov[p]),) for p in where.tolist()]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    search.query.clear()
    for j in junctions:
        if " ".join(j[:3]) in freq:
            search.update_query(j)
    search.finalize_query()
    search.exact_search_nn(args.k, include_distances=True)
    torch.cuda.synchronize()
    t_total += time.perf_counter() - t0
print("single-query route on %d of the samples (index already loaded, no process start): %.2f ms per query -> %.0f queries/s" % (
    len(slice_ids), 1e3 * t_total / len(slice_ids), len(slice_ids) / t_total), flush=True)
