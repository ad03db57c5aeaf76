#!/usr/bin/env python
"""Headline benchmark: exact top-100 angular kNN queries/s over 50,000 samples x 3000
features, 4096-query batches (BASELINE.json configs[2]) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step = one batch of 4096 queries answered exactly (ids + distances) against the
HBM-resident sample matrix.  N > 1 (torchrun, one rank per GPU): every rank holds the
50k-row matrix and answers its own 4096-query batch -- queries are independent, so
there is no data-path collective; per-GPU work is fixed (weak scaling) and `value`
is all ranks' queries / max-over-ranks device time.

The same run also measures, and reports as extra keys of the ONE JSON line rank 0 prints:
  rows_sharded   BASELINE configs[3]: 1,000,000 x 3000 rows split over the N ranks, the queries replicated, one NCCL
                 all-gather of score bounds and one all-gather of the top-k lists + merge INSIDE the timed region (N = 1:
                 the whole matrix on the one GPU, so strong scaling is computable from the per-N lines)
  datasets       the headline step on clustered ("tissue") and intropolis-like sparse, tie-heavy rows
  single_query   BASELINE configs[1]: 21,504 x 3000, one query, HBM roofline, and its end-to-end latency
  index_build    BASELINE configs[4]: scatter-add of 500 M (sample, coverage) pairs, --features swept
  cpu_baseline   the C port of the reference's loop on all host cores, the literal Python loop, a strong CPU
                 baseline (torch FP32 GEMM + top-k + FP64 re-rank on all cores), Annoy "n/a"
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SAMPLES, DIM, N_QUERIES, K = 50000, 3000, 4096, 100
N_SHARDED = 1000000
METRIC = "exact kNN queries/s (50k samples x 3000 feats, k=100)"
DUMP_BYTES = 60 * 10 ** 6          # --dump-outputs: array bytes in all, below 64 MB with the .npy headers


def dump_outputs(out_dir, ids, dists):
    """--dump-outputs: one step's results as out_dir/ids.npy and out_dir/distances.npy, float64 (the int32 ids are exact
    in it), one row per query.  Above DUMP_BYTES in all, the same seeded sample of queries is written on every run, with
    its row numbers as out_dir/query_rows.npy."""
    arrays = {"ids": np.asarray(ids, dtype=np.float64), "distances": np.asarray(dists, dtype=np.float64)}
    nq = arrays["ids"].shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values()) if nq else 0
    if nq * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(nq, size=DUMP_BYTES // (row_bytes + 8), replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["query_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons through NVML from before the warm-up on; `window()`
    keeps the samples that fall inside the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.max_mhz, self.error, self._stop_evt = index, [], None, None, threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            while not self._stop_evt.is_set():
                self.rows.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(h), nv.nvmlDeviceGetPowerUsage(h) / 1000.0))
                time.sleep(0.005)
        except Exception as exc:      # NVML absent: report that instead of clocks
            self.error = "nvml_unavailable:%s" % type(exc).__name__

    def window(self, t0, t1):
        self._stop_evt.set()
        self.join(timeout=2)
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80, "sync_boost": 0x10}
        rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows[-3:]
        reasons = sorted({n for r in rows for n, bit in names.items() if r[2] & bit})
        if self.error:
            reasons.append(self.error)
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(rows),
                "power_w": float(np.mean([r[3] for r in rows])) if rows else None}


# ---------------------------------------------------------------------------------------------- CPU baselines
def cpu_baseline_run(n_samples, dim, k, n_queries, threads, seed=1234):
    """Times the C port of exact_search_nn (oracle/oracle.c) on `n_queries` queries of the
    same workload, queries split over `threads` host threads.  Returns (queries/s, seconds, (ids, distances)).
    The C oracle is the one build() compiled: nothing is compiled here, the tree may be read-only."""
    from oracle import c_oracle
    rng = np.random.default_rng(seed)
    S = rng.standard_normal((n_samples, dim), dtype=np.float32)
    rows = rng.permutation(n_samples)[:n_queries]
    Q = S[rows].astype(np.float64)
    t0 = time.perf_counter()
    ids, dists = c_oracle.exact_search_batch(S, Q, k, n_threads=threads)
    dt = time.perf_counter() - t0
    assert np.array_equal(ids[:, 0], rows.astype(np.int32))      # each query finds itself first
    return n_queries / dt, dt, (ids, dists)


def literal_reference_qps(dim, n_samples, rows=300, seed=1):
    """The reference as written (pure-Python exact_search_nn, morna.py:681-712, through the literal oracle) on one
    core: `rows` rows timed, extrapolated linearly to n_samples rows (the loop is one pass over the rows)."""
    from oracle import morna_oracle as mo
    rng = np.random.default_rng(seed)
    S = rng.standard_normal((rows, dim)).astype(np.float32)
    t0 = time.perf_counter()
    mo.exact_search_nn(S, S[0].astype(np.float64), 10, clamp=True)
    dt = time.perf_counter() - t0
    return 1.0 / (dt * n_samples / rows)


def strong_cpu_qps(n_samples, dim, k, n_queries, seed=1234):
    """SURVEY 8(d)(ii): what a CPU can do with the same idea -- torch FP32 S @ Q^T on all cores, top-(k+32) per query,
    FP64 re-rank of those candidates.  Not the reference's algorithm and not exact by construction; context only."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(seed)
    S = torch.randn((n_samples, dim), generator=g)
    rows = torch.randperm(n_samples, generator=g)[:n_queries]
    Q = S[rows]
    Sn = S / S.norm(dim=1, keepdim=True)
    t0 = time.perf_counter()
    Qn = Q / Q.norm(dim=1, keepdim=True)
    scores = Qn @ Sn.t()
    cand = scores.topk(k + 32, dim=1).indices
    S64 = S.double()
    out = torch.empty((n_queries, k), dtype=torch.int64)
    for j in range(n_queries):
        c = cand[j]
        rowsj = S64[c]
        qj = Q[j].double()
        cos = (rowsj @ qj) / (rowsj.norm(dim=1) * qj.norm())
        d = (2 - 2 * cos).clamp_min(0).sqrt()
        out[j] = c[torch.argsort(d, stable=True)[:k]]
    dt = time.perf_counter() - t0
    assert bool((out[:, 0] == rows).all())
    return n_queries / dt, dt, cores


def workload_config(n_samples, nq, world):
    return {"workload": "%d samples x %d features (gaussian, seed 1234), %d in-index queries per GPU per step, "
                        "exact top-%d ids+distances" % (n_samples, DIM, nq, K),
            "parallelism": "replicated index, queries sharded x%d" % world,
            "l2": "inputs larger than L2 (sample matrix %.0f MB)" % (n_samples * DIM * 4 / 1e6)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (C port of morna.py:681-712, the
    reference itself is Python 2 and cannot run here) on all host cores."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = 2 * cores
    for _ in range(args.warmup):
        cpu_baseline_run(N_SAMPLES, DIM, K, min(per_step, cores), cores)
    t_total, q_total = 0.0, 0
    for _ in range(args.steps):
        _, dt, last = cpu_baseline_run(N_SAMPLES, DIM, K, per_step, cores)
        t_total += dt
        q_total += per_step
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last)
    value = q_total / t_total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(N_SAMPLES, N_QUERIES, 1),
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port",
                             "sample": "%d of the 4096 queries per step x %d steps, C port of exact_search_nn (morna.py:681-712; the "
                                       "reference itself is Python 2 + annoy and cannot run here), one thread per core" % (per_step, args.steps)},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- GPU arm
def pipeline_ms(torch, srch, batches, k, depth=2):
    """`len(batches)` batches through MornaSearch.search_batches; device time per batch (CUDA events on the current
    stream, which waits for the pipeline's streams)."""
    dev = srch.device
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    got, last = 0, None
    for ids, d in srch.search_batches(iter(batches), k, depth=depth):
        got, last = got + 1, (ids, d)
    pipe = srch._pipes[(k, depth)]
    cur = torch.cuda.current_stream(dev)
    for sl in pipe.slots:
        cur.wait_stream(sl.compute)
        cur.wait_stream(sl.stream)
    e1.record()
    torch.cuda.synchronize(dev)
    assert got == len(batches)
    return e0.elapsed_time(e1) / len(batches), last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=N_SAMPLES)
    ap.add_argument("--queries", type=int, default=N_QUERIES)
    ap.add_argument("--sharded-rows", type=int, default=N_SHARDED, help="rows of the rows-sharded section (0 = skip it)")
    ap.add_argument("--index-pairs", type=float, default=500e6, help="pairs of the index-build section (0 = skip it)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only-headline", action="store_true", help="skip every extra section")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the ids and distances of the last timed step (rank 0's "
                                                          "batch) to DIR as float64 .npy files, to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as td
    from morna_b200 import _lib, synth
    from morna_b200.search import MornaSearch
    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        td.init_process_group("nccl", device_id=device)
    lib = _lib.load()
    n_samples, nq = args.samples, args.queries
    peaks = measured_peaks()

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    t_start = time.perf_counter()

    def note(what):
        if rank == 0:
            sys.stderr.write("[bench %6.1f s] %s\n" % (time.perf_counter() - t_start, what))
            sys.stderr.flush()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic index, resident in HBM; every rank its own queries
    S = synth.gauss(n_samples, DIM, device, 1234)
    srch = MornaSearch(vectors=S, stats=(n_samples, n_samples, DIM), device=device)
    queries64, rows = synth.queries(S, nq, seed=99 + rank)          # in-index queries (float32-valued)
    del S
    host_q = queries64.to(torch.float32).cpu().pin_memory()          # the queries are float32-valued rows
    srch.enable_tensor_path()

    note("index resident")
    sampler = ClockSampler(local_rank); sampler.start()
    for _ in range(args.warmup):
        ids, d = srch.batched_search_device(queries64, K)
    pipeline_ms(torch, srch, [queries64] * max(args.warmup, 6), K)      # both pipeline slots have captured their CUDA graph
    torch.cuda.synchronize()
    assert torch.equal(ids[:, 0].long(), rows), "every in-index query must find itself first"
    assert float(d[:, 0].abs().max()) == 0.0

    # ---- dominant kernel alone: CUDA events on the launching stream at the phase boundaries of single, synchronised steps,
    # taken after the warm-up and before the timed region.  (Taken after the timed region the same synchronised launches
    # read 10-15 % longer once it has been 40 steps long -- filter GEMM 0.88 instead of 0.79 ms -- while the pipelined step
    # itself is unchanged, 1.873 vs 1.881 ms, and the late phase times no longer add up to it: an artefact of launching
    # single steps after a long burst, not the kernels' duration inside the timed steps.)
    roofline = dominant_kernel_roofline(torch, lib, _lib, srch, queries64, peaks)

    # ---- timed region: K steps, inputs resident, CUDA events, max over ranks.  The streaming API on HBM-resident
    # queries: batch i+1 is enqueued before batch i's overflow counters are read, so the host never stalls the device
    launches0 = _lib.launch_count()
    barrier()
    wall0 = time.perf_counter()
    ms_step, (last_ids, last_d) = pipeline_ms(torch, srch, [queries64] * args.steps, K)
    barrier()
    wall1 = time.perf_counter()
    assert int(last_ids[0, 0]) == int(rows[0])
    # copied now: the pipeline hands out views of its pinned buffers, which the sections below overwrite
    last_outputs = (last_ids.copy(), last_d.copy()) if args.dump_outputs and rank == 0 else None
    launches = _lib.launch_count() - launches0
    clocks = sampler.window(wall0, wall1)
    ms_step = max_over_ranks(ms_step)
    value = nq * world / (ms_step / 1e3)

    note("headline timed: %.3f ms per step" % ms_step)
    # ---- end to end through the host API: pinned host queries in, host results out, copies inside the timed region
    pipeline_ms(torch, srch, [host_q] * 6, K)            # (both slots have captured their step by now)
    barrier()
    t0 = time.perf_counter()
    pipeline_ms(torch, srch, [host_q] * args.steps, K)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = nq * world * args.steps / e2e_s

    # ---- the same batches given as sample ids (`search -q`: the queries are stored rows): 4 bytes per query cross PCIe
    host_rows = rows.to(torch.int64).cpu().pin_memory()
    pipeline_ms(torch, srch, [host_rows] * 6, K)
    barrier()
    t0 = time.perf_counter()
    pipeline_ms(torch, srch, [host_rows] * args.steps, K)
    barrier()
    e2e_ids_value = nq * world * args.steps / max_over_ranks(time.perf_counter() - t0)

    # ---- the step's own fraction beside the dominant kernel's
    step_flops = 2.0 * nq * n_samples * DIM
    roofline["step_frac"] = step_flops / (ms_step / 1e3) / 1e12 / peaks["bf16_tflops"]
    roofline["step_frac_of_sustained"] = step_flops / (ms_step / 1e3) / 1e12 / peaks["bf16_tflops_sustained"]
    roofline["step_algorithmic"] = "2*Q*N*D flops / ms_per_step (prep, thresholds, top-k and re-rank included), Q=%d N=%d D=%d" % (nq, n_samples, DIM)

    note("end to end and phases timed")
    # ---- approximate mode (the tensor-core pass without the exact re-rank): throughput and recall@k against the exact lists
    approx = None
    if rank == 0:
        exact_ids, _ = srch.batched_search_device(queries64, K)
        for _ in range(3):
            a_ids, _a_d = srch.approx_search_device(queries64, K)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            a_ids, _a_d = srch.approx_search_device(queries64, K)
        e1.record(); torch.cuda.synchronize()
        both = torch.cat([exact_ids, a_ids], dim=1).sort(dim=1).values
        recall = float((both[:, 1:] == both[:, :-1]).sum()) / float(nq * K)
        approx = {"queries_per_s": nq / (e0.elapsed_time(e1) / 10 / 1e3), "ms_per_step": e0.elapsed_time(e1) / 10,
                  "recall_at_k": recall, "k": K,
                  "what": "MornaSearch.approx_search_device: top-k by fp16 tensor-core score, no FP64 re-rank; recall against the exact lists "
                          "of the same queries (the reference's approximate mode is Annoy, n/a here)"}
    extras = {}
    if approx is not None:
        extras["approximate"] = approx
    full = not args.only_headline and n_samples == N_SAMPLES and nq == N_QUERIES
    if full:
        extras["datasets"] = dataset_lines(torch, synth, MornaSearch, device, rank, max_over_ranks, world)
    note("datasets done")
    del srch
    torch.cuda.empty_cache()
    if full and args.sharded_rows > 0:
        extras["rows_sharded"] = rows_sharded_line(torch, td, synth, MornaSearch, device, rank, world, args.sharded_rows,
                                                   max(5, min(args.steps, 10)), barrier, max_over_ranks)
        torch.cuda.empty_cache()
        rs = extras["rows_sharded"]
        rs["step_frac"] = rs["tensor_frac"]
        roofline["step_frac_1M_rows"] = {
            "value": rs["tensor_frac"], "n_gpus": world, "ms_per_step": rs["ms_per_step"],
            "what": "the same whole-step fraction (2*Q*N*D flops / step time / GPUs / measured bf16 peak; thresholds, top-k, "
                    "FP64 re-rank%s included) on north_star's target shape, %d x %d rows: the per-query costs of the "
                    "exact answer (k-th selection, 100 x 12 KB of rows re-read in FP64) do not grow with N, the contraction does"
                    % (" and the NCCL exchange" if world > 1 else "", args.sharded_rows, DIM)}
    note("rows-sharded done")
    single = index = None
    if rank == 0 and full:
        single = single_query_line(torch, lib, _lib, synth, device, peaks)
        if args.index_pairs > 0:
            torch.cuda.empty_cache()
            index = index_build_line(torch, lib, _lib, device, peaks, args.index_pairs)
    note("single query and index build done")
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            nq_cpu = min(N_QUERIES, 96 * cores)          # ~10 s of work on all host cores
            v, dt, _ = cpu_baseline_run(N_SAMPLES, DIM, K, nq_cpu, cores)
            sv, sdt, _ = strong_cpu_qps(N_SAMPLES, DIM, K, 1024)
            cpu = {"value": v, "unit": "queries/s", "cores": cores, "kind": "port",
                   "sample": "%d of the 4096 queries, C port of exact_search_nn (morna.py:681-712), %d threads, %.1f s"
                             % (nq_cpu, cores, dt),
                   "reference_as_written_qps": literal_reference_qps(DIM, N_SAMPLES),
                   "reference_as_written": "the literal pure-Python loop on one core, 300 rows timed and extrapolated to "
                                           "50000 (the reference itself is Python 2 + annoy + mmh3 and cannot run here)",
                   "strong_cpu": {"value": sv, "unit": "queries/s", "cores": cores, "sample": "1024 queries, %.1f s" % sdt,
                                  "what": "torch FP32 S @ Q^T on all cores + top-(k+32) + FP64 re-rank of those candidates "
                                          "(not the reference's algorithm, not exact by construction; context only)"},
                   "annoy": "n/a (the annoy wheel is not installed and there is no network; the reference's approximate "
                            "mode cannot be timed here)"}
        line = {"metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": roofline.pop("dtype"), "data": "synthetic",
                "config": workload_config(n_samples, nq, world),
                "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": int(host_q.numel() * host_q.element_size()),
                        "d2h_bytes_per_step": int(nq * K * 4 + nq * K * 8)},
                "e2e_queries_by_sample_id": {"value": e2e_ids_value, "unit": "queries/s", "h2d_bytes_per_step": int(nq * 8),
                                             "d2h_bytes_per_step": int(nq * K * 4 + nq * K * 8),
                                             "what": "the same step with the queries named by internal id (stored rows, `search -q`): "
                                                     "ids in, host ids + distances out; PCIe no longer carries 49 MB of vectors per step"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "single_query": single,
                "cpu_baseline": cpu, "peaks": peaks["source"]}
        line.update(extras)
        line["index_build"] = index
        if last_outputs is not None:
            dump_outputs(args.dump_outputs, *last_outputs)
        print(json.dumps(line))
    if world > 1:
        td.destroy_process_group()


def dataset_lines(torch, synth, MornaSearch, device, rank, max_over_ranks, world, steps=8):
    """The headline step on the other SURVEY 8(d) inputs: clustered rows with in- and out-of-index queries, and
    intropolis-like sparse rows where thousands of rows tie (what the reference's own fixture looks like)."""
    out = {}
    for kind, noise in (("tissue", 0.0), ("tissue", 0.05), ("gauss", 0.05), ("sparse", 0.0), ("sparse_fixture", 0.0)):
        S = synth.matrix(kind, N_SAMPLES, DIM, device)
        srch = MornaSearch(vectors=S, stats=(N_SAMPLES, N_SAMPLES, DIM), device=device)
        q, _rows = synth.queries(S, N_QUERIES, seed=99 + rank, noise=noise)
        del S
        srch.enable_tensor_path()
        pipeline_ms(torch, srch, [q] * 6, K)
        ms, _ = pipeline_ms(torch, srch, [q] * steps, K)
        ms = max_over_ranks(ms)
        name = kind + ("_out_of_index" if noise else "_in_index")
        if srch.csr is not None:
            out[name] = {"queries_per_s": N_QUERIES * world / (ms / 1e3), "ms_per_step": ms,
                         "path": "sparse index: CSR exact distances + exact selection (morna_knn_exact_sparse), no tensor pass",
                         "nnz_per_row": float(srch.csr[1].numel()) / N_SAMPLES}
        else:
            out[name] = {"queries_per_s": N_QUERIES * world / (ms / 1e3), "ms_per_step": ms, "path": "tensor cores + FP64 re-rank",
                         "overflowed_queries": int(srch.last_stats[0]), "reranked_per_query": srch.last_stats[2] / N_QUERIES}
        del srch, q
        torch.cuda.empty_cache()
    return out


def rows_sharded_line(torch, td, synth, MornaSearch, device, rank, world, n_rows, steps, barrier, max_over_ranks):
    """BASELINE configs[3]: n_rows x 3000 split into contiguous row blocks over the ranks (rank r draws its block from
    seed 1234 + r), 4096 replicated queries per step, exact global top-100; the all-gather of the score bounds, the
    all-gather of the lists and the merge are inside the timed region.  Strong scaling: the total work is fixed."""
    from morna_b200 import dist as mdist
    lo, hi = mdist.shard_bounds(n_rows, rank, world)
    S = synth.gauss(hi - lo, DIM, device, 1234 + rank)
    srch = MornaSearch(vectors=S, stats=(n_rows, hi - lo, DIM), device=device)
    srch.row_lo, srch.row_hi = lo, hi                     # global ids of this block
    del S
    srch.enable_tensor_path()
    q = synth.gauss(N_QUERIES, DIM, device, 99).to(torch.float64)       # the same out-of-index queries on every rank
    host_q = q.to(torch.float32).cpu().pin_memory()
    host_ids = torch.empty((N_QUERIES, K), dtype=torch.int32).pin_memory()
    host_d = torch.empty((N_QUERIES, K), dtype=torch.float64).pin_memory()

    def step(queries):
        return mdist.sharded_batched_search(srch, queries, K, check_overflow=False)

    copy_stream = torch.cuda.Stream(device=device)
    stage = [torch.empty((N_QUERIES, DIM), dtype=torch.float32, device=device) for _ in range(2)]
    staged, consumed = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]

    def run_e2e(count):
        """`count` steps from pinned host queries to host results: step i+1's host->device copy runs on a copy stream under
        step i's kernels (two device staging buffers); rank 0 copies every step's ids + distances back."""
        cur = torch.cuda.current_stream(device)

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[i & 1])
                stage[i & 1].copy_(host_q, non_blocking=True)
                staged[i & 1].record(copy_stream)
        for ev in consumed:
            ev.record(cur)
        prefetch(0)
        for i in range(count):
            cur.wait_event(staged[i & 1])
            qd = stage[i & 1].to(torch.float64)
            consumed[i & 1].record(cur)
            if i + 1 < count:
                prefetch(i + 1)
            ids, d = step(qd)
            if rank == 0:
                host_ids.copy_(ids, non_blocking=True)
                host_d.copy_(d, non_blocking=True)
        cur.synchronize()

    for _ in range(3):
        ids, d = step(q)
    torch.cuda.synchronize()
    assert int(srch.last_stats[0]) == 0 if srch.last_stats else True
    assert bool((d[:, 1:] >= d[:, :-1]).all()) and int(ids.min()) >= 0 and int(ids.max()) < n_rows
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        step(q)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / steps)
    run_e2e(2)
    barrier()
    t0 = time.perf_counter()
    run_e2e(steps)
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) / steps * 1e3)
    # phases of one step on this rank (CUDA events around the calls of the sharded search)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ev[0].record()
    vals = srch.batched_score_bound(q, K); ev[1].record()
    every = vals[None]
    if world > 1:
        every = torch.empty((world,) + tuple(vals.shape), dtype=vals.dtype, device=device)
        td.all_gather_into_tensor(every, vals)
    bound = srch.union_kth_bound(every, K)
    ev[2].record()
    li, ld_ = srch.batched_finish_bound(bound, check_overflow=False); ev[3].record()
    if world > 1:
        mdist.gather_merge_packed(li, ld_, K)
    ev[4].record()
    torch.cuda.synchronize()
    phase = {n: round(ev[i].elapsed_time(ev[i + 1]), 4) for i, n in
             enumerate(("score_to_local_bounds", "all_gather_bounds_kth", "final_lists_rerank_order", "all_gather_lists_merge"))}
    stats = srch.last_stats
    return {"workload": "%d samples x %d features in %d row blocks, %d replicated out-of-index queries per step, exact global top-%d"
                        % (n_rows, DIM, world, N_QUERIES, K),
            "value": N_QUERIES / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms, "steps": steps, "scaling": "strong",
            "e2e": {"value": N_QUERIES / (e2e_ms / 1e3), "unit": "queries/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(host_q.numel() * 4), "d2h_bytes_per_step": int(N_QUERIES * K * 12)},
            "collectives": ("all_gather of %d B (score bounds) + all_gather of %d B (top-k lists) per rank, NCCL"
                            % (4 * N_QUERIES * K, 12 * N_QUERIES * K)) if world > 1 else "none (one rank)",
            "rows_per_rank": hi - lo, "phase_ms": phase,
            "tensor_frac": 2.0 * N_QUERIES * n_rows * DIM / (ms / 1e3) / 1e12 / world / measured_peaks()["bf16_tflops"]}


def single_query_line(torch, lib, _lib, synth, device, peaks):
    """BASELINE configs[1]: exact top-100 single queries over 21,504 x 3000 rows (the single-query kernel, HBM-bound:
    4*N*D algorithmic bytes per query).  Every figure is device time (CUDA events on the launching stream) of CUDA-graph
    replays holding 32 kernels each, so the host's launch rate does not enter."""
    from morna_b200.search import MornaSearch
    n, m = 21504, 32
    S = synth.gauss(n, DIM, device, 4321)
    srch = MornaSearch(vectors=S, stats=(n, n, DIM), device=device)
    QS = S[torch.arange(m, device=device) * 600 + 7].to(torch.float64).contiguous()      # 32 distinct in-index queries
    side, other = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    algo = 4.0 * n * DIM

    def entry(us):
        return {"us_per_query": us, "queries_per_s": 1e6 / us, "achieved": algo / (us * 1e-6) / 1e9,
                "frac": algo / (us * 1e-6) / 1e9 / peaks["hbm_gbs"]}

    class Arm:
        """One stream's buffers and its captured graph of one morna_knn_single_stream call over `queries`."""
        def __init__(self, stream, queries):
            self.stream, self.q = stream, queries
            with torch.cuda.stream(stream):
                self.want_i, self.want_d = srch.single_search_stream(queries, K)
                self.ws = srch._single_stream_workspace(n)
                self.flags = torch.zeros(queries.shape[0], dtype=torch.int32, device=device)
                self.ids, self.d = torch.empty_like(self.want_i), torch.empty_like(self.want_d)
            stream.synchronize()

        def call(self):
            q = self.q
            _lib.check(lib.morna_knn_single_stream(_lib.dev_ptr(srch.vectors), _lib.dev_ptr(srch.pp), n, DIM, srch.ld, 0, _lib.dev_ptr(q), DIM,
                                                   q.shape[0], K, _lib.dev_ptr(self.ids), _lib.dev_ptr(self.d), _lib.dev_ptr(self.flags),
                                                   _lib.dev_ptr(self.ws), self.ws.numel(), _lib.stream_ptr()), "morna_knn_single_stream")

        def capture(self):
            with torch.cuda.stream(self.stream):
                for _ in range(2):
                    self.call()
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph, stream=self.stream):
                    self.call()
                for _ in range(3):
                    self.graph.replay()
            self.stream.synchronize()

        def check(self):
            assert torch.equal(self.ids, self.want_i) and torch.equal(self.d, self.want_d) and int(self.flags.sum()) == 0

    main_arm = Arm(side, QS)
    for j in (0, 13, 31):                                          # the stream call answers like the one-query call
        one_i, one_d = srch.single_search_device(QS[j], K)
        assert torch.equal(main_arm.want_i[j], one_i[0]) and torch.equal(main_arm.want_d[j], one_d[0])
        assert int(one_i[0, 0]) == j * 600 + 7 and float(one_d[0, 0]) == 0.0
    # hand-over 0: plain launches, every kernel starts after the previous one has drained (one query at a time);
    # 1: programmatic dependent launch, the next kernel begins when every CTA of the current one has finished its scan --
    #    consecutive scans do not overlap, only the one-CTA selection tail and the launch gap are hidden;
    # 2 (library default): ... has finished its first row pass -- consecutive scans overlap by about half
    res = {}
    for mode, name in ((0, "plain_launches"), (1, "handover_after_scan"), (2, "handover_after_first_pass")):
        lib.morna_debug_set_tuning(29, mode)
        main_arm.capture()
        with torch.cuda.stream(side):
            e0.record(side)
            for _ in range(10):
                main_arm.graph.replay()
            e1.record(side)
        side.synchronize()
        main_arm.check()
        res[name] = entry(e0.elapsed_time(e1) * 1e3 / (10 * m))
    # two CUDA streams, each with its own workspaces, plain launches: two queries in flight
    lib.morna_debug_set_tuning(29, 0)
    arm_a, arm_b = Arm(side, QS[:m // 2].contiguous()), Arm(other, QS[m // 2:].contiguous())
    arm_a.capture(); arm_b.capture()
    torch.cuda.synchronize(device)
    e0.record(side)
    other.wait_event(e0)
    for _ in range(10):
        with torch.cuda.stream(side):
            arm_a.graph.replay()
        with torch.cuda.stream(other):
            arm_b.graph.replay()
    e1.record(side); e2.record(other)
    torch.cuda.synchronize(device)
    arm_a.check(); arm_b.check()
    two = entry(max(e0.elapsed_time(e1), e0.elapsed_time(e2)) * 1e3 / (10 * m))
    two["what"] = "plain launches on two CUDA streams, each with its own workspaces: two independent queries in flight"
    lib.morna_debug_set_tuning(29, 2)
    # end to end: host query in (pinned), host ids + distances out, one query at a time through the public call
    hq = QS[5].cpu().pin_memory()
    for _ in range(5):
        srch.exact_search_batch(hq.numpy()[None, :], K)
    t0 = time.perf_counter()
    for _ in range(50):
        hi_, hd_ = srch.exact_search_batch(hq.numpy()[None, :], K)
    e2e_us = (time.perf_counter() - t0) / 50 * 1e6
    assert int(hi_[0, 0]) == 5 * 600 + 7
    traffic = None
    prof = os.path.join(ROOT, "profiles", "r01_step_summary.json")     # dram bytes per launch from the committed ncu capture
    if os.path.exists(prof):
        with open(prof) as fh:
            traffic = json.load(fh).get("scan64_dram_bytes_21504x3000")
    head = res["handover_after_scan"]
    return {"workload": "21504 samples x 3000 features, single queries, exact top-100 (the 258 MB matrix exceeds L2)",
            "us_per_query": head["us_per_query"], "queries_per_s": head["queries_per_s"],
            "kernel": "scan64_select_kernel (one launch per query)",
            "what": "a stream of single queries on one CUDA stream (morna_knn_single_stream, 32 distinct queries per call, CUDA-graph replay), "
                    "every query its own kernel and its own full pass over the matrix; query j+1's kernel is launched with programmatic stream "
                    "serialisation and begins when every CTA of query j has finished its scan, so consecutive scans do not overlap: only the "
                    "one-CTA selection tail and the launch gap are hidden (`stream.handover_after_scan`).  `stream.plain_launches` is one query "
                    "at a time with nothing hidden; `stream.handover_after_first_pass` is the library default (consecutive scans overlap)",
            "stream": res, "two_in_flight": two,
            "e2e": {"us_per_query": e2e_us, "queries_per_s": 1e6 / e2e_us, "h2d_bytes": DIM * 8, "d2h_bytes": K * 12,
                    "what": "MornaSearch.exact_search_batch with one host query: pinned copy in, kernel, ids + distances copied out, synchronous"},
            "roofline": {"bound": "hbm", "achieved": head["achieved"], "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": head["frac"],
                         "frac_plain_launches": res["plain_launches"]["frac"], "frac_overlapping_scans": res["handover_after_first_pass"]["frac"],
                         "traffic": traffic, "traffic_source": "static: dram__bytes_read+write of one launch in the committed ncu capture (profiles/), not measured in this run",
                         "algorithmic": "4*N*D bytes per query"}}


def index_build_line(torch, lib, _lib, device, peaks, pairs):
    """BASELINE configs[4] through scripts/index_bench.py's generator: device time of id assignment, hashing, scatter-add
    and float32 store for each --features value, against 8*nnz + 40*J + 4*N*D algorithmic bytes."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("index_bench", os.path.join(ROOT, "scripts", "index_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.run(pairs=pairs, dims=(500, 1000, 3000, 10000, 30000), peak=peaks["hbm_gbs"], quiet=True)


def dominant_kernel_roofline(torch, lib, _lib, srch, queries64, peaks):
    """Times the kernels of one step with CUDA events recorded on the launching stream at the
    phase boundaries of morna_knn_batched; the dominant one is the tcgen05 GEMM's filter pass."""
    from morna_b200.search import PHASE_NAMES, make_phase_events
    events, arr = make_phase_events()
    reps, acc = 5, [0.0] * 6
    for _ in range(2):
        srch.batched_search_device(queries64, K, phase_events=arr)
    torch.cuda.synchronize()
    for _ in range(reps):
        srch.batched_search_device(queries64, K, phase_events=arr)
        torch.cuda.synchronize()
        for i in range(6):
            acc[i] += events[i].elapsed_time(events[i + 1]) / reps
    n_all = srch.row_hi - srch.row_lo
    n = n_all - (n_all - 1) // srch.BATCH_BLOCK_ROWS * srch.BATCH_BLOCK_ROWS     # the phase events time the last row block
    nq = queries64.shape[0]
    n0 = min(n, 8192)
    ld_h = srch.ld_h
    ms = acc[3] if n > n0 else acc[1]
    rows = (n - n0) if n > n0 else n0
    flops = 2.0 * nq * rows * srch.dim
    achieved = flops / (ms / 1e3) / 1e12
    # SM clocks stay at their maximum during these short GEMM launches (see "clocks": no power-cap reason), so the
    # denominator is the burst cuBLAS bf16 figure; the sustained (power-capped, seconds-long) one is given beside it
    peak = peaks["bf16_tflops"]
    peak_sustained = peaks["bf16_tflops_sustained"]
    traffic = rr_traffic = None
    prof = os.path.join(ROOT, "profiles", "r01_step_summary.json")     # dram bytes per launch from the committed ncu capture
    if os.path.exists(prof) and n_all == N_SAMPLES and nq == N_QUERIES:          # the capture was taken at the headline shape
        with open(prof) as fh:
            summary = json.load(fh)
        traffic, rr_traffic = summary.get("knn_gemm2_filter_dram_bytes"), summary.get("rerank_dist_dram_bytes")
    # second kernel of the step by time: the exact FP64 re-rank, an HBM/L2 gather of candidates*4*ld bytes per query
    blocks = (n_all + srch.BATCH_BLOCK_ROWS - 1) // srch.BATCH_BLOCK_ROWS
    rr_bytes = float(srch.last_stats[2]) / blocks * srch.ld * 4                  # (candidates of one row block)
    rr_gbs = rr_bytes / (acc[5] / 1e3) / 1e9
    rerank = {"bound": "hbm", "kernel": "rerank_dist_kernel<8> + rerank_order_kernel (FP64 canonical sums over the candidate rows)",
              "achieved": rr_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": rr_gbs / peaks["hbm_gbs"],
              "traffic": rr_traffic, "launch_ms": acc[5],
              "algorithmic": "candidates * 4 * ld bytes gathered per batch (%d candidates x %d B); rows re-ranked by several "
                             "queries hit in L2, so achieved can exceed the DRAM traffic rate" % (srch.last_stats[2] // blocks, srch.ld * 4)}
    # context only (not on the product path): the same contraction through cuBLAS, fp16 in / fp16 out
    lib_ms = None
    try:
        a16 = torch.randn((nq, ld_h), device=queries64.device, dtype=torch.float16)
        b16 = srch.hs[n_all - rows:n_all]
        out16 = torch.empty((nq, rows), device=queries64.device, dtype=torch.float16)
        for _ in range(3):
            torch.matmul(a16, b16.t(), out=out16)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tot = 0.0
        for _ in range(10):
            e0.record(); torch.matmul(a16, b16.t(), out=out16); e1.record(); torch.cuda.synchronize()
            tot += e0.elapsed_time(e1) / 10
        lib_ms = tot
        del a16, out16
    except Exception:
        pass
    return {"bound": "tensor", "kernel": "knn_gemm2_kernel<4> (tcgen05 cta_group::2 fp16 UMMA, filter pass over %d rows)" % rows,
            "cublas_same_shape": None if lib_ms is None else {"ms": lib_ms, "tflops": 2.0 * nq * rows * ld_h / (lib_ms / 1e3) / 1e12,
                                                              "what": "torch.matmul fp16 %d x %d x %d, one launch at a time" % (nq, rows, ld_h)},
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
            "traffic_source": "static: dram__bytes_read+write of one launch in the committed ncu capture (profiles/), not measured in this run",
            "algorithmic": "2*Q*N*D flops per launch, Q=%d N=%d D=%d" % (nq, rows, srch.dim),
            "launch_ms": ms, "peak_source": peaks["source"] + " cuBLAS bf16 burst (fp16 runs on the same kind::f16 pipe)",
            "peak_sustained": peak_sustained, "frac_of_sustained": achieved / peak_sustained,
            "phase_ms": {name: round(v, 4) for name, v in zip(PHASE_NAMES, acc)},
            "second_kernel": rerank,
            "candidates_per_query": {"first_pass": srch.last_stats[1] / nq, "reranked": srch.last_stats[2] / nq,
                                     "overflowed_queries": srch.last_stats[0]},
            "dtype": "fp16 first pass (fp32 accumulate), f64 re-rank"}


if __name__ == "__main__":
    main()
