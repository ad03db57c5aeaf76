"""Within-group search (`within_group_search` / `within_group_range`) with every row as a query by internal id, each
leaving out its own row (the `search --all-samples --within-group --exclude-self` shape), in 4096-query batches:
50,000 and 1,000,000 x 3000 rows (gauss and tissue).  Groupings: scattered groups of 10, contiguous groups of 100 and
1,000, scattered groups of 1,000, a tissue-like labelling (30 scattered groups of about 33,000 rows, which the grouped
kernels cannot sort) and a heavy-tailed contiguous mix; top-20 and range (R = the median 10th-nearest distance within the
group).  Per case: ms per 4096 queries and for all rows (host clock around the whole run, ending in a synchronise), then
the queries each route took in every batch run on their own (the same routes: a group's queries in a batch all go one
way).  Then the sweep that sets WITHIN_GROUPED_MAX_PAIRS: groups of g rows, contiguous (a group's queries arrive
together: g x g pairs per group and call) and scattered (a few queries per group and call), every query through each
route.  Then the achieved FP64 rate and bytes/s of group_distances_kernel (kernel time from torch.profiler in a run of
its own; FMA and byte counts computed here from the grouping), and next to all of it the unrestricted top-20 run of
--all-samples (search_batches over the same 4096-id batches).  The card's name and power limit are read in the same
run."""
import argparse, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ap = argparse.ArgumentParser()
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--shapes", default="gauss:50000,tissue:50000,gauss:1000000,tissue:1000000")
ap.add_argument("--sweep-rows", type=int, default=200000)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import numpy as np
import torch
from morna_b200.search import MornaSearch
from morna_b200 import synth

out = open(args.out, "w") if args.out else None


def say(line):
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


say("device: %s" % torch.cuda.get_device_name(0))
try:
    say("nvidia-smi: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                        capture_output=True, text=True, timeout=60).stdout.strip())
except (OSError, subprocess.SubprocessError) as exc:
    say("nvidia-smi: not available (%s)" % exc)
B = 4096


def grouping(name, n, rng):
    if name == "mixed":
        # sizes from a heavy-tailed distribution (most groups small, a few of up to 20,000 rows), 2% unlabelled
        labels = np.full(n, -1, np.int64)
        at, g = 0, 0
        while at < n * 49 // 50:
            size = int(min(20000, max(1, rng.pareto(1.2) * 20)))
            labels[at:at + size] = g
            at, g = at + size, g + 1
        return labels[:n].astype(np.int32)
    if name == "tissue-like":
        return (rng.permutation(n) % 30).astype(np.int32)
    size = int(name.split()[-1])
    return ((rng.permutation(n) if name.startswith("scattered") else np.arange(n)) // size).astype(np.int32)


def batches_of(ids):
    return [ids[b:b + B] for b in range(0, len(ids), B)]


def run(s, batches, labels, k=None, r=None):
    """Seconds for these batches of query ids (top-k, or range with r), matches per query, queries per route."""
    torch.cuda.synchronize()
    t, matches, routes, nq = time.perf_counter(), 0, np.zeros(2, np.int64), 0
    for q in batches:
        if not len(q):
            continue
        nq += len(q)
        if r is None:
            s.within_group_search(q, k, labels[q], q.astype(np.int32))
        else:
            matches += s.within_group_range(q, r, labels[q], q.astype(np.int32))[1].numel()
        routes += s.last_within_routes
    torch.cuda.synchronize()
    return time.perf_counter() - t, matches / max(nq, 1), routes


def route_batches(s, batches, labels):
    """Each batch's queries split as the search routes them: (grouped-route batches, tensor-core-route batches)."""
    grouped, large = [], []
    for q in batches:
        plan = s._within_plan(q, labels[q], None)
        grouped.append(q[plan["grouped"]])
        large.append(q[plan["large"]])
    return grouped, large


def work(labels, ld):
    """(FMAs, bytes read) of group_distances_kernel when every row queries its group and every group takes the grouped
    route: each query against every row of its group (D FMAs a pair), each row read once per tile of up to 8 queries (ld
    floats) and each item's queries staged (ld doubles each; items of up to 128 rows)."""
    _, g = np.unique(labels[labels >= 0], return_counts=True)
    g = g.astype(np.float64)
    tiles = np.ceil(g / 8)
    return (float((g * g).sum()) * args.features,
            float((tiles * g).sum()) * ld * 4 + float((g * np.ceil(g / 128)).sum()) * ld * 8)


for shape in args.shapes.split(","):
    kind, n = shape.split(":")
    n = int(n)
    S = synth.matrix(kind, n, args.features, "cuda", seed=5)
    s = MornaSearch(vectors=S, stats=(n, n, args.features))
    del S
    all_ids = np.arange(n, dtype=np.int64)
    batches = batches_of(all_ids)
    # the unrestricted --all-samples top-20 run, for scale
    s.search_batches([all_ids[:B]], 20).__next__()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in s.search_batches(iter(batches), 20):
        pass
    torch.cuda.synchronize()
    t = time.perf_counter() - t
    say("%s %d x %d: unrestricted --all-samples top-20: %.1f ms per 4096 queries, %.1f ms for all rows"
        % (kind, n, args.features, 1e3 * t * B / n, 1e3 * t))
    rng = np.random.default_rng(1)
    for name in ("scattered groups of 10", "groups of 100", "groups of 1000", "scattered groups of 1000", "tissue-like",
                 "mixed"):
        labels = grouping(name, n, rng)
        s.set_row_groups(labels)
        gb, lb = route_batches(s, batches, labels)
        run(s, batches[:1], labels, k=20)                                  # warm-up
        run(s, [np.concatenate(lb)[:B]], labels, k=20)                     # (builds the grouped copy if a route needs it)
        t, _, routes = run(s, batches, labels, k=20)
        tg, tl = run(s, gb, labels, k=20)[0], run(s, lb, labels, k=20)[0]
        say("  %-24s top-20: %8.2f ms per 4096, %9.1f ms all rows | grouped route %7d queries %9.1f ms | tensor-core "
            "route %7d queries %9.1f ms" % (name, 1e3 * t * B / n, 1e3 * t, routes[0], 1e3 * tg, routes[1], 1e3 * tl))
        R = float(np.median(s.within_group_search(all_ids[:B], 10, labels[:B])[1][:, 9].cpu().numpy()))
        if not np.isfinite(R):
            R = 1.0
        t, per, routes = run(s, batches, labels, r=R)
        tg, tl = run(s, gb, labels, r=R)[0], run(s, lb, labels, r=R)[0]
        say("  %-24s range R=%.4f (%.1f matches/query): %8.2f ms per 4096, %9.1f ms all rows | grouped %9.1f ms | "
            "tensor-core %9.1f ms" % (name, R, per, 1e3 * t * B / n, 1e3 * t, 1e3 * tg, 1e3 * tl))
        if name == "groups of 100" and n >= 1000000:
            from torch.profiler import profile, ProfilerActivity
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run(s, batches, labels, k=20)
            kt = sum(e.device_time_total for e in prof.key_averages() if "group_distances_kernel" in e.key) * 1e-6
            st = sum(e.device_time_total for e in prof.key_averages() if "group_select_kernel" in e.key) * 1e-6
            fma, nbytes = work(labels, s.ld)
            say("  group_distances_kernel, groups of 100, all rows: %.1f ms kernel time, %.2e FMA -> %.1f TFLOP/s FP64, "
                "%.2e bytes row + query reads -> %.2f TB/s; group_select_kernel %.1f ms"
                % (1e3 * kt, fma, 2 * fma / kt / 1e12, nbytes, nbytes / kt / 1e12, 1e3 * st))
    del s
    torch.cuda.empty_cache()

# the sweep that sets WITHIN_GROUPED_MAX_PAIRS: every group through each route
n = args.sweep_rows
S = synth.gauss(n, args.features, "cuda", seed=5)
s = MornaSearch(vectors=S, stats=(n, n, args.features))
del S
all_ids = np.arange(n, dtype=np.int64)
batches = batches_of(all_ids)
say("route sweep (WITHIN_GROUPED_MAX_PAIRS = %d): gauss %d x %d, groups of g rows, all rows as queries, top-20; pairs = "
    "mean (queries of a group in a batch) x g" % (MornaSearch.WITHIN_GROUPED_MAX_PAIRS, n, args.features))
rng = np.random.default_rng(2)
for layout, sizes in (("contiguous", (256, 512, 640, 768, 1024, 2048)), ("scattered", (1024, 2048, 4096, 8192))):
    for g in sizes:
        labels = ((rng.permutation(n) if layout == "scattered" else all_ids) // g).astype(np.int32)
        pairs = np.mean([np.unique(labels[q], return_counts=True)[1].mean() for q in batches]) * g
        res = []
        for p in (1 << 62, 0):                # every group on the grouped route / on the tensor-core route
            s.WITHIN_GROUPED_MAX_PAIRS = p
            s.set_row_groups(labels)
            run(s, batches[:1], labels, k=20)
            res.append(run(s, batches, labels, k=20)[0])
        say("  %-10s g = %5d (%9.0f pairs): grouped route %8.2f ms per 4096 queries, tensor-core route %8.2f -> %s"
            % (layout, g, pairs, 1e3 * res[0] * B / n, 1e3 * res[1] * B / n, "grouped" if res[0] < res[1] else "tensor-core"))
