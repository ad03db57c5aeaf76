"""Rows-sharded range search (dist.sharded_range_search) on 1,000,000 x 3000 rows, one process per GPU over NCCL, for
world sizes 1, 2, 4 and 8 up to the GPUs present.  Datasets gauss and tissue (synth.matrix, the same matrix at every
world size: every rank draws all rows and keeps its block); 4096-query batches, half in-index rows and half rows with
0.3 relative noise, as scripts/range_search_bench.py.  R per dataset is the median over the first --sample-queries
queries of the 100th- and of the 1000th-nearest distance, from sharded_exact_search with k = 1000 at the largest world
size (k = 1000 takes the FP64 scan), and is reused at the smaller ones.

Per line: ms per batch of the whole call (CUDA events after warm-up, then a synchronise), the sharded top-100 step
(sharded_batched_search) of the same run, matches per query and overflowed queries per rank, and a phase breakdown
taken in separate calls that run the protocol's steps one by one with a synchronise (and a barrier) at each boundary:
local count, header and counts all-gather, local emit and pack, list all-gather, merge.  Phase times are rank 0's."""
import argparse, os, socket, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=1000000)
ap.add_argument("--features", type=int, default=3000)
ap.add_argument("--queries", type=int, default=4096)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--sample-queries", type=int, default=512)
ap.add_argument("--worlds", default="1,2,4,8")
ap.add_argument("--kinds", default="gauss,tissue")
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


def phases(srch, Q, R, world):
    """The steps of sharded_range_search_groups (one batch, one group) timed one by one, in ms."""
    from morna_b200 import dist as mdist
    from morna_b200.search import _range_groups
    t, marks = time.perf_counter(), []

    def mark():
        nonlocal t
        torch.cuda.synchronize()
        td.barrier()
        now = time.perf_counter()
        marks.append((now - t) * 1e3)
        t = time.perf_counter()
    mark()
    dev = Q.device
    b0, st = next(iter(srch.range_count_batches(Q, R)))
    mark()
    head = torch.tensor([Q.shape[0], Q.shape[1], 0, -1], dtype=torch.int64, device=dev)
    every = torch.empty(world * 4, dtype=torch.int64, device=dev)
    td.all_gather_into_tensor(every, head)
    every.cpu()
    counts = torch.from_numpy(st["counts"]).to(dev)
    every = torch.empty(world * counts.numel(), dtype=torch.int64, device=dev)
    td.all_gather_into_tensor(every, counts)
    rank_counts = every.cpu().numpy().reshape(world, -1)
    (lo, hi), = _range_groups(rank_counts.sum(axis=0) * (world + 1), None)
    cap = int(rank_counts.sum(axis=1).max())
    cap += cap & 1
    mark()
    _, ids, d = srch.range_emit(st, lo, hi)
    mine = mdist.pack_range_lists(ids, d, cap)
    mark()
    gathered = torch.empty(world * mine.numel(), dtype=torch.uint8, device=dev)
    td.all_gather_into_tensor(gathered, mine)
    mark()
    mdist.merge_gathered_csr(gathered, rank_counts, cap)
    mark()
    return marks[1:], cap * 12


def worker(rank, world, port, opts, shared):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    td.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from morna_b200 import dist as mdist, synth
    from morna_b200.search import MornaSearch
    for kind in opts.kinds.split(","):
        S = synth.matrix(kind, opts.rows, opts.features, dev)
        srch = MornaSearch(vectors=S, stats=(opts.rows, opts.rows, opts.features), shard=(rank, world), device=dev)
        qa, _ = synth.queries(S, opts.queries // 2, seed=5)
        qb, _ = synth.queries(S, opts.queries - opts.queries // 2, seed=6, noise=0.3)
        Q = torch.cat([qa, qb]).contiguous()
        del S, qa, qb
        torch.cuda.empty_cache()
        if kind not in shared:
            t0 = time.perf_counter()
            _, d = mdist.sharded_exact_search(lambda q, k: srch.exact_search_device(q, k), Q[:opts.sample_queries], 1000)
            R = {k: float(d[:, k - 1].median()) for k in (100, 1000)}
            if rank == 0:
                shared[kind] = R
                print("%s: R from %d sample queries at world %d (%.1f s): %s" % (
                    kind, opts.sample_queries, world, time.perf_counter() - t0, R), flush=True)
            td.barrier()
        R = shared[kind]
        t_topk = timed(lambda: mdist.sharded_batched_search(srch, Q, 100), opts.reps)
        for k in (100, 1000):
            t_range = timed(lambda: mdist.sharded_range_search(srch, Q, R[k]), opts.reps)
            off, ids, dd = mdist.sharded_range_search(srch, Q, R[k])
            stats = torch.tensor(srch.last_stats, dtype=torch.int64, device=dev)
            every = torch.empty(world * 3, dtype=torch.int64, device=dev)
            td.all_gather_into_tensor(every, stats)
            per_rank = every.view(world, 3).cpu().tolist()
            ph = [phases(srch, Q, R[k], world) for _ in range(3)][1:]
            ms = np.median(np.array([p[0] for p in ph]), axis=0)
            if rank == 0:
                print("%s world %d: R = %.6f (median %dth-nearest)  sharded range %.3f ms per %d-query batch  sharded top-100 "
                      "%.3f ms  ratio %.2f" % (kind, world, R[k], k, t_range, Q.shape[0], t_topk, t_range / t_topk), flush=True)
                print("%s world %d:   matches/query %.1f  overflowed queries per rank %s  first-pass survivors/query per rank %s"
                      % (kind, world, int(off[-1]) / Q.shape[0], [p[0] for p in per_rank],
                         ["%.1f" % (p[1] / Q.shape[0]) for p in per_rank]), flush=True)
                print("%s world %d:   phases (ms, synchronised): count %.3f  header+counts gather %.3f  emit+pack %.3f  "
                      "list gather %.3f (%.2f MB per rank)  merge %.3f" % ((kind, world) + tuple(ms[:4]) + (ph[-1][1] / 1e6, ms[4])),
                      flush=True)
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
    worlds = [w for w in map(int, args.worlds.split(",")) if w <= n_gpu]
    for w in map(int, args.worlds.split(",")):
        if w > n_gpu:
            print("world %d: not measured (%d GPUs present)" % (w, n_gpu), flush=True)
    shared = mp.Manager().dict()
    for world in sorted(worlds, reverse=True):              # the largest world first: it computes R fastest
        mp.spawn(worker, args=(world, free_port(), args, shared), nprocs=world, join=True)
