"""Rows-sharded group-capped search (dist.sharded_batched_search / sharded_range_search with max_per_group) on
1,000,000 x 3000 rows, one process per GPU over NCCL, for world sizes 1, 2, 4 and 8 up to the GPUs present.  The same
matrix at every world size (synth.matrix: every rank draws all rows and keeps its block); 4096 queries by internal id
(stored rows, as `search --all-samples`); contiguous groups of 100 rows; N = 1, 2, 5.

Per line: ms per 4096-query batch of the whole call (CUDA events around --reps calls after a warm-up call, then a
synchronise), each capped top-100 next to the uncapped sharded top-100 of the same run, and the capped range search (R =
the median 100th-nearest distance, from the uncapped top-100) next to the uncapped one.  A phase breakdown of the capped
top-100 is taken in separate calls that run the protocol's steps one by one with a synchronise and a barrier at each
boundary: header + label all-gather, local capped search, pack + list all-gather, merge, walk; rank 0's times, with the
rows each rank re-ranked per query in its local search (last_stats).  The card's name and power limit are read in the same
run.  With one process (world 1), the per-rank steps of 2, 4 and 8 ranks are also timed on the one GPU, without the
collectives (emulated())."""
import argparse, os, socket, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=1000000)
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--queries", type=int, default=4096)
ap.add_argument("--k", type=int, default=100)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--worlds", default="1,2,4,8")
ap.add_argument("--kinds", default="gauss")
args = ap.parse_args()

import numpy as np
import torch
import torch.distributed as td
import torch.multiprocessing as mp


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


def phases(srch, Q, k, m, world):
    """The steps of dist.sharded_capped_search timed one by one, in ms (world > 1)."""
    from morna_b200 import dist as mdist
    t, marks = time.perf_counter(), []

    def mark():
        nonlocal t
        torch.cuda.synchronize()
        td.barrier()
        now = time.perf_counter()
        marks.append((now - t) * 1e3)
        t = time.perf_counter()
    mark()
    fields = mdist._cap_fields(srch, m, None, world)
    mdist._agree([Q.shape[0], Q.shape[1], k] + fields, ("queries", "dim", "k") + mdist.CAP_FIELD_NAMES, Q.device, None,
                 world, "bench")
    labels = mdist.all_gather_cap_labels(srch)
    mark()
    ids, d = srch.batched_search_device(Q, k, max_per_group=m)
    mark()
    mine = mdist.pack_topk_lists(ids, d)
    every = torch.empty(world * mine.numel(), dtype=torch.uint8, device=Q.device)
    td.all_gather_into_tensor(every, mine)
    mark()
    every = every.view(world, -1)
    mi, md = mdist.merge_packed_lists(every, Q.shape[0], k, world * k)
    mark()
    offsets = torch.arange(Q.shape[0] + 1, dtype=torch.int64, device=Q.device) * (world * k)
    out = (torch.empty((Q.shape[0], k), dtype=torch.int32, device=Q.device),
           torch.empty((Q.shape[0], k), dtype=torch.float64, device=Q.device))
    srch.cap_sorted_lists(offsets, mi, md, m, k, out=out, cap_group=labels)
    mark()
    return marks[1:]


def emulated(S, whole, Q, opts):
    """One GPU: the G ranks' row blocks searched one after another (no collectives), then the merge and the walk of
    dist.merge_capped_topk on their stacked lists, each timed alone; the result is checked against one process."""
    from morna_b200 import dist as mdist
    from morna_b200.search import MornaSearch
    k, n, nq = opts.k, opts.rows, Q.shape[0]
    for G in (2, 4, 8):
        shards = [MornaSearch(vectors=S, stats=(n, n, opts.features), shard=(r, G), device=Q.device) for r in range(G)]
        for sh in shards:
            sh.set_cap_groups(torch.arange(sh.row_lo, sh.row_hi, dtype=torch.int32, device=Q.device) // 100)
        labels = torch.cat([mdist.cap_label_block(sh, G) for sh in shards])[:n]
        t_plain = [timed(lambda: sh.batched_search_device(Q, k), opts.reps) for sh in shards]
        print("emulated %d ranks on one GPU (%d rows each): uncapped local top-%d %.3f ms/batch (max over ranks)"
              % (G, shards[0].row_hi, k, max(t_plain)), flush=True)
        for m in (1, 2, 5):
            t_local = [timed(lambda: sh.batched_search_device(Q, k, max_per_group=m), opts.reps) for sh in shards]
            every = torch.stack([mdist.pack_topk_lists(*sh.batched_search_device(Q, k, max_per_group=m)) for sh in shards])
            t_merge = timed(lambda: mdist.merge_packed_lists(every, nq, k, G * k), opts.reps)
            mi, md = mdist.merge_packed_lists(every, nq, k, G * k)
            offsets = torch.arange(nq + 1, dtype=torch.int64, device=Q.device) * (G * k)
            out = (torch.empty((nq, k), dtype=torch.int32, device=Q.device), torch.empty((nq, k), dtype=torch.float64, device=Q.device))
            t_walk = timed(lambda: whole.cap_sorted_lists(offsets, mi, md, m, k, out=out, cap_group=labels), opts.reps)
            got = mdist.merge_capped_topk(whole, every, labels, nq, k, m)
            want = whole.batched_search_device(Q, k, max_per_group=m)
            same = bool(torch.equal(got[0], want[0]) and torch.equal(got[1].view(torch.int64), want[1].view(torch.int64)))
            print("  N = %d: local capped top-%d %.3f ms/batch (max over ranks; %.2f x uncapped local)  merge of %d x %d "
                  "entries/query %.3f ms  walk %.3f ms  equal to one process: %s"
                  % (m, k, max(t_local), max(t_local) / max(t_plain), G, k, t_merge, t_walk, same), flush=True)
        del shards, every, mi, md
        torch.cuda.empty_cache()


def worker(rank, world, port, opts):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    td.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from morna_b200 import dist as mdist, synth
    from morna_b200.search import MornaSearch
    k, n = opts.k, opts.rows
    for kind in opts.kinds.split(","):
        S = synth.matrix(kind, n, opts.features, dev, seed=5)
        srch = MornaSearch(vectors=S, stats=(n, n, opts.features), shard=(rank, world), device=dev)
        rows = torch.from_numpy(np.random.default_rng(1).choice(n, opts.queries, replace=False)).to(dev)
        Q = S[rows].to(torch.float64).contiguous()
        srch.set_cap_groups((torch.arange(srch.row_lo, srch.row_hi, dtype=torch.int32, device=dev) // 100))
        if world == 1 and rank == 0:
            emulated(S, srch, Q, opts)
        del S
        torch.cuda.empty_cache()
        t_plain = timed(lambda: mdist.sharded_batched_search(srch, Q, k), opts.reps)
        _, d = mdist.sharded_batched_search(srch, Q, k)
        R = float(d[:, k - 1].median())
        lines = ["%s %d x %d, world %d, %d queries by id, groups of 100: uncapped sharded top-%d %.3f ms/batch"
                 % (kind, n, opts.features, world, Q.shape[0], k, t_plain)]
        for m in (1, 2, 5):
            t_cap = timed(lambda: mdist.sharded_batched_search(srch, Q, k, max_per_group=m), opts.reps)
            srch.batched_search_device(Q, k, max_per_group=m)
            st = torch.tensor(srch.last_stats, dtype=torch.int64, device=dev)
            every = torch.empty(world * st.numel(), dtype=torch.int64, device=dev)
            td.all_gather_into_tensor(every, st)
            per_rank = every.view(world, -1).cpu().tolist()
            lines.append("  N = %d: capped sharded top-%d %.3f ms/batch (%.2f x uncapped); local re-ranked rows/query per "
                         "rank %s, to the FP64 route per rank %s"
                         % (m, k, t_cap, t_cap / t_plain, ["%.1f" % (p[2] / Q.shape[0]) for p in per_rank],
                            [p[0] for p in per_rank]))
            if world > 1:
                ms = np.median(np.array([phases(srch, Q, k, m, world) for _ in range(4)][1:]), axis=0)
                lines.append("    phases (ms, synchronised): header + label gather %.3f (%.1f MB per rank)  local capped "
                             "search %.3f  list gather %.3f (%.2f MB per rank)  merge %.3f  walk %.3f"
                             % (ms[0], 4e-6 * -(-n // world), ms[1], ms[2], 12e-6 * Q.shape[0] * k, ms[3], ms[4]))
        t_range = timed(lambda: mdist.sharded_range_search(srch, Q, R), opts.reps)
        matches = int(mdist.sharded_range_search(srch, Q, R)[0][-1]) / Q.shape[0]
        lines.append("  range R = %.6f (median %dth-nearest, %.1f matches/query): uncapped sharded %.3f ms/batch"
                     % (R, k, matches, t_range))
        for m in (1, 2, 5):
            t_cr = timed(lambda: mdist.sharded_range_search(srch, Q, R, max_per_group=m), opts.reps)
            lines.append("    N = %d: capped sharded range %.3f ms/batch (%.2f x uncapped)" % (m, t_cr, t_cr / t_range))
        if rank == 0:
            print("\n".join(lines), flush=True)
        del srch, Q
        torch.cuda.empty_cache()
    td.destroy_process_group()


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


if __name__ == "__main__":
    n_gpu = torch.cuda.device_count()
    if n_gpu == 0:
        sys.exit("needs a CUDA device")
    print("device: %s  x%d" % (torch.cuda.get_device_name(0), n_gpu), flush=True)
    try:
        print("nvidia-smi: " + subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                              capture_output=True, text=True, timeout=60).stdout.strip().replace("\n", " | "),
              flush=True)
    except (OSError, subprocess.SubprocessError) as exc:
        print("nvidia-smi: not available (%s)" % exc, flush=True)
    for w in map(int, args.worlds.split(",")):
        if w > n_gpu:
            print("world %d: not measured (%d GPUs present)" % (w, n_gpu), flush=True)
            continue
        mp.spawn(worker, args=(w, free_port(), args), nprocs=w, join=True)
