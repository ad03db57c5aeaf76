"""Range search (MornaSearch.range_search_device) on 50,000 x 3000 rows, 4096-query batches: the tensor-core route, the
FP64 route on the same queries, and the top-100 batched_search_device step next to them.  Datasets gauss and tissue
(synth.py); queries half in-index rows, half rows with 0.3 relative noise (out of index).  R per dataset is the median
over the first --sample-queries queries of the 100th-nearest distance, and once more of the 1000th.  Times are CUDA events
around whole calls (host reads of the counts included), after a warm-up call, with a synchronise; the 600 MB matrix
exceeds L2.  The FP64 route is an HBM-bound scan (4*n*ld bytes per four queries, twice: count and fill) and is timed on
the first --exact-queries queries only, once, after the scan kernels were warmed by the R estimate; its time grows
linearly with the number of queries."""
import argparse, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=50000)
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--queries", type=int, default=4096)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--exact-queries", type=int, default=256)
ap.add_argument("--sample-queries", type=int, default=512)
args = ap.parse_args()

import numpy as np
import torch
from morna_b200 import _lib, synth
from morna_b200.search import MornaSearch

print("device: %s" % torch.cuda.get_device_name(0), flush=True)
try:
    print("nvidia-smi: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                          capture_output=True, text=True, timeout=60).stdout.strip(), flush=True)
except (OSError, subprocess.SubprocessError) as exc:
    print("nvidia-smi: not available (%s)" % exc, flush=True)


def timed(fn, reps, warm=True):
    if warm:
        fn()                                                 # warm-up: module loads, workspaces
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out


def distances(srch, Q):
    n = srch.row_hi - srch.row_lo
    out = torch.empty((Q.shape[0], n), dtype=torch.float64, device=srch.device)
    _lib.check(srch.lib.morna_angular_distances(_lib.dev_ptr(srch.vectors), _lib.dev_ptr(srch.pp), n, srch.dim, srch.ld,
                                                _lib.ptr(Q), Q.shape[0], srch.dim, _lib.dev_ptr(out), n, _lib.stream_ptr()),
               "morna_angular_distances")
    return out


for kind in ("gauss", "tissue"):
    S = synth.matrix(kind, args.rows, args.features, "cuda")
    srch = MornaSearch(vectors=S, stats=(args.rows, args.rows, args.features))
    qa, _ = synth.queries(S, args.queries // 2, seed=5)
    qb, _ = synth.queries(S, args.queries - args.queries // 2, seed=6, noise=0.3)
    Q = torch.cat([qa, qb]).contiguous()
    kth = {}
    for k in (100, 1000):
        kth[k] = float(torch.kthvalue(distances(srch, Q[:args.sample_queries]), k, dim=1).values.median())
    t_topk, (ti, td) = timed(lambda: srch.batched_search_device(Q, 100), args.reps)
    print("%s: top-100 batched_search_device  %.3f ms per %d-query batch" % (kind, t_topk, Q.shape[0]), flush=True)
    for k in (100, 1000):
        R = kth[k]
        t_a, res_a = timed(lambda: srch.range_search_device(Q, R), args.reps)
        route, stats = srch.last_range_route, list(srch.last_stats)
        assert route == "tensor"
        m = args.exact_queries
        srch.RANGE_TENSOR_MIN_QUERIES = 1 << 30                 # the FP64 route on the first m of the same queries
        t_b, res_b = timed(lambda: srch.range_search_device(Q[:m], R), 1, warm=False)
        assert srch.last_range_route == "exact"
        del srch.RANGE_TENSOR_MIN_QUERIES
        off_a, ids_a, d_a = res_a
        end = int(off_a[m])
        same = (torch.equal(off_a[:m + 1], res_b[0]) and torch.equal(ids_a[:end], res_b[1]) and
                torch.equal(d_a[:end].view(torch.int64), res_b[2].view(torch.int64)))
        print("%s: R = %.6f (median %dth-nearest)  tensor route %.3f ms per %d-query batch  FP64 route %.1f ms per %d queries "
              "(%.1f ms per %d scaled linearly)" % (kind, R, k, t_a, Q.shape[0], t_b, m, t_b * Q.shape[0] / m, Q.shape[0]), flush=True)
        print("%s:   matches/query %.1f  first-pass survivors/query %.1f  overflowed queries %d  routes agree bit for bit on the FP64 route's queries: %s" % (
            kind, stats[2] / Q.shape[0], stats[1] / Q.shape[0], stats[0], same), flush=True)
    del srch, S
    torch.cuda.empty_cache()
