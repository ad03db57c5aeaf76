"""Per-query exclusion on the batched top-100 step: 4096-query steps by internal id (the stored rows as queries, as
`search --all-samples`) on 50,000 x 3000 and 1,000,000 x 3000 rows (gauss and tissue), each without an exclusion, with
`--exclude-self` labels (every row its own group) and with contiguous groups of 100 and 1,000 rows, all in the same run.
Per case: the step time (CUDA events around --reps whole batched_search_device calls after a warm-up call, with a
synchronise; every matrix exceeds L2), the queries that overflowed to the FP64 scan and the first-pass survivors per
query (last_stats).  With --baseline-lib (the library built from the parent commit), the unexcluded scoring + re-rank
call (morna_knn_batched) of the two libraries alternates --ab-rounds times on the same buffers, to show what the new
exclusion branch in kth_warp_kernel costs a search without one.  The card's name and power limit are read in the same
run."""
import argparse, ctypes, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ap = argparse.ArgumentParser()
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--queries", type=int, default=4096)
ap.add_argument("--k", type=int, default=100)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--ab-rounds", type=int, default=6)
ap.add_argument("--baseline-lib", default=None)
ap.add_argument("--shapes", default="gauss:50000,tissue:50000,gauss:1000000,tissue:1000000")
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
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def raw_step(lib, s, Q, k, bufs):
    """One morna_knn_batched call of `lib` (a ctypes library) on the search's rows."""
    n = s.row_hi - s.row_lo
    ids, d, over, stats, ws = bufs
    f = lib.morna_knn_batched
    f.restype = ctypes.c_int
    f.argtypes = _lib._SIGNATURES["morna_knn_batched"][1]
    _lib.check(f(_lib.dev_ptr(s.vectors), _lib.dev_ptr(s.pp), _lib.dev_ptr(s.hs), s.ld_h, _lib.dev_ptr(s.rho_max), n, s.dim,
                 s.ld, s.row_lo, _lib.ptr(Q), Q.shape[0], s.dim, k, _lib.dev_ptr(ids), _lib.dev_ptr(d), _lib.dev_ptr(over),
                 _lib.dev_ptr(stats), _lib.dev_ptr(ws), ws.numel(), None, _lib.stream_ptr()), "morna_knn_batched")


baseline = ctypes.CDLL(os.path.abspath(args.baseline_lib)) if args.baseline_lib else None
k, nq = args.k, args.queries
for shape in args.shapes.split(","):
    kind, n = shape.split(":")
    n = int(n)
    S = synth.matrix(kind, n, args.features, "cuda", seed=5)
    s = MornaSearch(vectors=S, stats=(n, n, args.features))
    del S
    s.enable_tensor_path()
    rows = torch.from_numpy(np.random.default_rng(1).choice(n, nq, replace=False)).cuda()
    Q = s.vectors[rows, :s.dim].to(torch.float64).contiguous()
    labels = {"self": torch.arange(n, dtype=torch.int32, device="cuda"),
              "groups of 100": torch.arange(n, dtype=torch.int32, device="cuda") // 100,
              "groups of 1000": torch.arange(n, dtype=torch.int32, device="cuda") // 1000}
    ms = timed(lambda: s.batched_search_device(Q, k), args.reps)
    st = s.last_stats
    print("%s %d x %d, %d queries by id, top-%d: unmasked %.3f ms/batch, overflowed %d, first-pass survivors/query %.1f"
          % (kind, n, args.features, nq, k, ms, st[0], st[1] / nq), flush=True)
    for name, lab in labels.items():
        s.set_row_groups(lab)
        qg = s.row_group[rows]
        ms = timed(lambda: s.batched_search_device(Q, k, query_groups=qg), args.reps)
        st = s.last_stats
        print("  exclusion %-15s %.3f ms/batch, overflowed %d, first-pass survivors/query %.1f"
              % (name, ms, st[0], st[1] / nq), flush=True)
    s.set_row_groups(None)
    if baseline is not None:
        bufs = (torch.empty((nq, k), dtype=torch.int32, device="cuda"), torch.empty((nq, k), dtype=torch.float64, device="cuda"),
                torch.empty(nq, dtype=torch.uint8, device="cuda"), torch.empty(4, dtype=torch.int32, device="cuda"),
                _lib.workspace(s.lib.morna_knn_batched_workspace_bytes(n, nq, s.dim, k), s.device))
        times = {"parent": [], "this change": []}
        for r in range(args.ab_rounds):
            for name, lib in ((("parent", baseline), ("this change", s.lib)) if r % 2 == 0 else
                              (("this change", s.lib), ("parent", baseline))):
                times[name].append(timed(lambda: raw_step(lib, s, Q, k, bufs), args.reps))
        print("  A/B unmasked morna_knn_batched, %d alternating rounds of %d calls: parent %s ms, this change %s ms"
              % (args.ab_rounds, args.reps, " ".join("%.3f" % t for t in times["parent"]),
                 " ".join("%.3f" % t for t in times["this change"])), flush=True)
        print("    medians: parent %.3f ms, this change %.3f ms" % (np.median(times["parent"]), np.median(times["this change"])),
              flush=True)
    del s, Q
    torch.cuda.empty_cache()
