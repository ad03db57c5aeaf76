"""Filtered search (MornaSearch.subset) on 50,000 x 3000 rows (gauss and tissue) and 1,000,000 x 3000 rows (gauss):
the time to build the subset's compacted index, and per 4096-query batch the exact top-100 step (batched_search_device)
and the range step (range_search_device, R = the median 100th-nearest distance of the whole index over the first
--sample-queries queries), each next to the unfiltered step of the same index in the same run.  Subsets keep 1 %, 10 %,
50 % and all but 100 of the rows, drawn from a fixed seed.  Queries: half in-index rows, half rows with 0.3 relative
noise.  Build time: host clock around subset() and a device synchronise, median of --reps builds after one warm-up
build (the gather, the norms copy and the sparse-row check that every index load runs).  Step times: CUDA events
around --reps whole calls after a warm-up call, with a synchronise; every matrix here exceeds L2."""
import argparse, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ap = argparse.ArgumentParser()
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--queries", type=int, default=4096)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--sample-queries", type=int, default=256)
ap.add_argument("--shapes", default="gauss:50000,tissue:50000,gauss:1000000")
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


def timed(fn, reps):
    fn()                                                     # warm-up: module loads, workspaces
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out


def build_ms(parent, ids, reps):
    parent.subset(ids)                                       # warm-up
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        f = parent.subset(ids)
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
        del f
    return float(np.median(times))


def median_kth(srch, Q, k):
    n = srch.row_hi - srch.row_lo
    out = torch.empty((Q.shape[0], n), dtype=torch.float64, device=srch.device)
    _lib.check(srch.lib.morna_angular_distances(_lib.dev_ptr(srch.vectors), _lib.dev_ptr(srch.pp), n, srch.dim, srch.ld,
                                                _lib.ptr(Q), Q.shape[0], srch.dim, _lib.dev_ptr(out), n, _lib.stream_ptr()),
               "morna_angular_distances")
    return float(torch.kthvalue(out, k, dim=1).values.median())


def step_line(label, srch, Q, R):
    t_topk, _ = timed(lambda: srch.batched_search_device(Q, 100), args.reps)
    over = srch.last_stats[0]
    t_range, (off, _, _) = timed(lambda: srch.range_search_device(Q, R), args.reps)
    print("  %-34s top-100 %8.3f ms (%d overflowed)   range %8.3f ms (%s route, %.1f matches/query, %d overflowed)"
          % (label, t_topk, over, t_range, srch.last_range_route, int(off[-1]) / Q.shape[0], srch.last_stats[0]), flush=True)


for shape in args.shapes.split(","):
    kind, rows = shape.split(":")
    n = int(rows)
    S = synth.matrix(kind, n, args.features, "cuda")
    parent = MornaSearch(vectors=S, stats=(n, n, args.features))
    del S
    qa, _ = synth.queries(parent.vectors[:, :args.features], args.queries // 2, seed=5)
    qb, _ = synth.queries(parent.vectors[:, :args.features], args.queries - args.queries // 2, seed=6, noise=0.3)
    Q = torch.cat([qa, qb]).contiguous()
    R = median_kth(parent, Q[:args.sample_queries], 100)
    print("%s %d x %d, %d-query batches, R = %.6f (median 100th-nearest of the whole index)"
          % (kind, n, args.features, Q.shape[0], R), flush=True)
    step_line("unfiltered (%d rows)" % n, parent, Q, R)
    rng = np.random.default_rng(2026)
    for label, m in (("1 %", n // 100), ("10 %", n // 10), ("50 %", n // 2), ("all but 100", n - 100)):
        ids = np.sort(rng.choice(n, m, replace=False))
        t_build = build_ms(parent, ids, args.reps)
        f = parent.subset(ids)
        print("  subset %-11s %8d rows  build %8.3f ms (%.1f GB/s of kept rows read and written)"
              % (label, m, t_build, 2 * m * parent.ld * 4 / t_build / 1e6), flush=True)
        step_line("filtered %s" % label, f, Q, R)
        del f
        torch.cuda.empty_cache()
    del parent, Q, qa, qb
    torch.cuda.empty_cache()
