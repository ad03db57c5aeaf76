"""Rows-sharded range search over gloo (CPU, world sizes 2 and 3): the header check, the counts exchange, the query
groups every rank derives from the gathered counts, the list all-gather and the step after it.  The local search is a
stand-in with the two methods the protocol calls (range_count_batches, range_emit), its lists built from the C
oracle's distances with global ids; the merge is a numpy reference (the CUDA kernel is checked in
test_gpu_sharded_range.py).  Every rank must hold the same groups and lists, equal to one process's brute force."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

from morna_b200 import dist as mdist
from morna_b200.search import check_radius


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _ordered(ids, d):
    """Reference order: distance ascending, equal distances id descending."""
    o = np.lexsort((-ids.astype(np.int64), d))
    return ids[o].astype(np.int32), d[o]


def brute_csr(S, Q, R):
    from oracle import c_oracle
    off, ids, ds = [0], [], []
    for q in Q:
        d = c_oracle.distances(S, q)
        keep = np.nonzero(d <= R)[0]
        i, dd = _ordered(keep, d[keep])
        ids.append(i); ds.append(dd); off.append(off[-1] + len(i))
    return (np.array(off, np.int64), np.concatenate(ids) if ids else np.zeros(0, np.int32),
            np.concatenate(ds) if ds else np.zeros(0, np.float64))


class OracleShard(object):
    """This rank's row block [lo, hi) of S with range_count_batches / range_emit, as MornaSearch has them."""
    RANGE_BATCH_QUERIES = 7                          # several batches per call

    def __init__(self, S, lo, hi):
        self.S, self.lo, self.hi = S, lo, hi

    def range_count_batches(self, queries, max_distance):
        from oracle import c_oracle
        r = check_radius(max_distance)
        for b0 in range(0, queries.shape[0], self.RANGE_BATCH_QUERIES):
            qb = queries[b0:b0 + self.RANGE_BATCH_QUERIES]
            lists = []
            for q in qb.numpy():
                d = c_oracle.distances(self.S[self.lo:self.hi], q) if self.hi > self.lo else np.zeros(0)
                keep = np.nonzero(d <= r)[0]
                lists.append(_ordered(keep + self.lo, d[keep]))
            yield b0, {"queries": qb, "lists": lists, "counts": np.array([len(l[0]) for l in lists], np.int64)}

    def range_emit(self, st, lo, hi):
        part = st["lists"][lo:hi]
        off = np.zeros(hi - lo + 1, np.int64)
        np.cumsum([len(p[0]) for p in part], out=off[1:])
        ids = np.concatenate([p[0] for p in part]) if part else np.zeros(0, np.int32)
        d = np.concatenate([p[1] for p in part]) if part else np.zeros(0)
        return torch.from_numpy(off), torch.from_numpy(ids.astype(np.int32)), torch.from_numpy(d.astype(np.float64))


def numpy_merge(gathered, n_lists, nq, cap, rank_offsets, out_offsets, total):
    """Reference for morna_merge_sorted_csr: per query, every rank's entries concatenated and ordered."""
    raw = gathered.numpy().reshape(n_lists, cap * 12)
    dists = [raw[g, :cap * 8].view(np.float64) for g in range(n_lists)]
    ids = [raw[g, cap * 8:].view(np.int32) for g in range(n_lists)]
    roff = rank_offsets.numpy().reshape(n_lists, nq + 1)
    out_i, out_d = [], []
    for j in range(nq):
        i = np.concatenate([ids[g][roff[g, j]:roff[g, j + 1]] for g in range(n_lists)])
        d = np.concatenate([dists[g][roff[g, j]:roff[g, j + 1]] for g in range(n_lists)])
        i, d = _ordered(i, d)
        out_i.append(i); out_d.append(d)
    out_i = np.concatenate(out_i) if out_i else np.zeros(0, np.int32)
    out_d = np.concatenate(out_d) if out_d else np.zeros(0)
    assert len(out_i) == total == int(out_offsets[-1])
    return torch.from_numpy(out_i), torch.from_numpy(out_d)


def _worker(rank, world, port, cases, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    td.init_process_group("gloo", rank=rank, world_size=world)
    for name, (S, Q, R, byte_cap, bad) in cases.items():
        lo, hi = mdist.shard_bounds(S.shape[0], rank, world)
        r = float(np.nextafter(R, 3.0)) if (bad and rank == world - 1) else R
        try:
            groups = list(mdist.sharded_range_search_groups(OracleShard(S, lo, hi), torch.from_numpy(Q), r,
                                                            byte_cap=byte_cap, merge=numpy_merge))
        except ValueError as exc:
            out[(name, rank)] = ("ValueError", str(exc))
            continue
        out[(name, rank)] = ("ok", [(g[0], g[1], g[2].numpy(), g[3].numpy(), g[4].numpy()) for g in groups])
    td.destroy_process_group()


def _cases(world):
    from oracle import c_oracle
    rng = np.random.default_rng(world)
    S = rng.standard_normal((101, 24)).astype(np.float32)
    S[60] = S[3]; S[100] = S[3]; S[90] = 2 * S[3]            # ties across the shard boundaries (and inside a shard)
    Q = np.concatenate([S[[3, 70, 99]].astype(np.float64), rng.standard_normal((20, 24))])
    d_all = np.stack([np.sort(c_oracle.distances(S, q)) for q in Q])
    R = float(np.median(d_all[:, 10]))
    # rank 0 holds every match: queries are rank 0's rows, each with two copies inside rank 0, and R below the gaps
    T = rng.standard_normal((12 * world, 16)).astype(np.float32)
    T[1] = T[0]; T[2] = T[0]; T[4] = T[3]; T[5] = T[3]
    QT = np.concatenate([T[[0, 3, 6, 7, 8, 9]].astype(np.float64)] * 2)
    tiny = rng.standard_normal((2, 8)).astype(np.float32)     # world 3: the last rank has no rows
    return {
        "ties": (S, Q, R, None, False),
        "ties_r0": (S, Q, 0.0, None, False),
        "one_rank": (T, QT, 1e-6, 12 * (world + 1) * 4, False),
        "empty_rank": (tiny, rng.standard_normal((9, 8)), 1.2, None, False),
        "no_queries": (S, Q[:0], R, None, False),
        "bad_radius": (S, Q, R, None, True),
    }


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_range_search_equals_single_process(world):
    cases = _cases(world)
    manager = mp.Manager()
    out = manager.dict()
    mp.spawn(_worker, args=(world, _free_port(), cases, out), nprocs=world, join=True)
    for name, (S, Q, R, byte_cap, bad) in cases.items():
        if bad:
            for rank in range(world):
                assert out[(name, rank)][0] == "ValueError", (name, rank)
            continue
        want = brute_csr(S, Q, R)
        per_rank = []
        for rank in range(world):
            status, groups = out[(name, rank)]
            assert status == "ok", (name, rank, groups)
            per_rank.append(groups)
            spans = [(g[0], g[1]) for g in groups]
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            if Q.shape[0] == 0:
                assert groups == []
                continue
            assert spans[0][0] == 0 and spans[-1][1] == Q.shape[0]
            off = np.concatenate([[0]] + [g[2][1:] + sum(len(h[3]) for h in groups[:k]) for k, g in enumerate(groups)])
            got = (off, np.concatenate([g[3] for g in groups]), np.concatenate([g[4] for g in groups]))
            assert np.array_equal(got[0], want[0]), (name, rank)
            assert np.array_equal(got[1], want[1]), (name, rank)
            assert np.array_equal(got[2].view(np.int64), want[2].view(np.int64)), (name, rank)
        for groups in per_rank[1:]:                               # the same groups on every rank
            assert [(g[0], g[1]) for g in groups] == [(g[0], g[1]) for g in per_rank[0]]
        if name == "one_rank":
            assert len(per_rank[0]) > 1 and want[0][-1] == 20           # 3 + 3 + 1 + 1 + 1 + 1 matches, twice
        if name == "ties_r0":
            assert {3, 60, 100} <= set(want[1][want[0][0]:want[0][1]].tolist())
