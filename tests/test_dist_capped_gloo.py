"""Rows-sharded group-capped search over gloo (CPU, world sizes 2 and 3): the header check, the cap-label all-gather, and
the step after the list all-gather (the merge of every rank's lists and the walk over the merged order), for top-k and
range.  The local search is a stand-in built on the C oracle's distances with global ids, its capped top-k walked in
numpy; the merge and the walk are numpy references passed through the `merge` / `walk` hooks (the CUDA kernels are
checked in test_gpu_sharded_capped.py).  Every rank must hold the same lists, equal to one process's brute force, and a
rank whose arguments differ makes every rank raise ValueError."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

from morna_b200 import dist as mdist
from tests.test_dist_range_gloo import OracleShard, _free_port, _ordered, brute_csr, numpy_merge


def walk_keep(ids, labels, m, limit=None):
    """Positions of a list (reference order) the capped walk keeps; ids < 0 are padding and skipped."""
    seen, keep = {}, []
    for p, i in enumerate(ids.tolist()):
        if i < 0:
            continue
        g = int(labels[i])
        if g >= 0:
            if seen.get(g, 0) >= m:
                continue
            seen[g] = seen.get(g, 0) + 1
        keep.append(p)
        if limit is not None and len(keep) == limit:
            break
    return np.array(keep, np.int64)


def numpy_walk(offsets, ids, dists, max_per_group, limit=None, out=None, cap_group=None):
    """Reference for MornaSearch.cap_sorted_lists(..., cap_group=labels): the CSR, or `out` filled and padded."""
    off, i, d, lab = offsets.numpy(), ids.numpy().reshape(-1), dists.numpy().reshape(-1), cap_group.numpy()
    lists = []
    for j in range(len(off) - 1):
        li, ld = i[off[j]:off[j + 1]], d[off[j]:off[j + 1]]
        keep = walk_keep(li, lab, max_per_group, limit)
        lists.append((li[keep], ld[keep]))
    if out is not None:
        out[0].fill_(-1)
        out[1].fill_(float("inf"))
        for j, (li, ld) in enumerate(lists):
            out[0][j, :len(li)] = torch.from_numpy(li.astype(np.int32))
            out[1][j, :len(ld)] = torch.from_numpy(ld)
        return out
    new_off = np.zeros(len(lists) + 1, np.int64)
    np.cumsum([len(l[0]) for l in lists], out=new_off[1:])
    return (torch.from_numpy(new_off), torch.from_numpy(np.concatenate([l[0] for l in lists] + [np.zeros(0, np.int32)])),
            torch.from_numpy(np.concatenate([l[1] for l in lists] + [np.zeros(0)])))


def numpy_packed_merge(every, nq, k_in, k):
    """Reference for merge_packed_lists: per query every rank's entries ordered, the first k, padded with -1 / +inf."""
    world = every.shape[0]
    raw = every.numpy()
    d = [raw[g, :nq * k_in * 8].view(np.float64).reshape(nq, k_in) for g in range(world)]
    i = [raw[g, nq * k_in * 8:].view(np.int32).reshape(nq, k_in) for g in range(world)]
    out_i = np.full((nq, k), -1, np.int32)
    out_d = np.full((nq, k), np.inf)
    for j in range(nq):
        ai = np.concatenate([x[j] for x in i])
        ad = np.concatenate([x[j] for x in d])
        ai, ad = _ordered(ai[ai >= 0], ad[ai >= 0])
        out_i[j, :min(k, len(ai))], out_d[j, :min(k, len(ai))] = ai[:k], ad[:k]
    return torch.from_numpy(out_i), torch.from_numpy(out_d)


def brute_topk(S, Q, labels, k, m):
    from oracle import c_oracle
    out_i = np.full((len(Q), k), -1, np.int32)
    out_d = np.full((len(Q), k), np.inf)
    for j, q in enumerate(Q):
        d = c_oracle.distances(S, q)
        i, dd = _ordered(np.arange(len(d)), d)
        keep = walk_keep(i, labels, m, k)
        out_i[j, :len(keep)], out_d[j, :len(keep)] = i[keep], dd[keep]
    return out_i, out_d


class CappedOracleShard(OracleShard):
    """OracleShard with cap labels and the capped top-k of its rows, as MornaSearch has them."""

    def __init__(self, S, lo, hi, labels):
        super(CappedOracleShard, self).__init__(S, lo, hi)
        self.index_size, self.row_lo, self.row_hi = S.shape[0], lo, hi
        self.cap_group = None if labels is None else torch.from_numpy(labels[lo:hi].astype(np.int32))

    def batched_search_device(self, queries, k, max_per_group=None):
        ids = np.full((queries.shape[0], k), -1, np.int32)
        d = np.full((queries.shape[0], k), np.inf)
        if self.hi > self.lo:
            i, d = brute_topk(self.S[self.lo:self.hi], queries.numpy(), self.cap_group.numpy(), k, max_per_group)
            ids = np.where(i >= 0, i + self.lo, -1).astype(np.int32)
        return torch.from_numpy(ids), torch.from_numpy(d)


def _worker(rank, world, port, cases, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    td.init_process_group("gloo", rank=rank, world_size=world)
    for name, c in cases.items():
        S, labels = c["S"], c["labels"]
        lo, hi = mdist.shard_bounds(S.shape[0], rank, world)
        last = rank == world - 1
        shard = CappedOracleShard(S, lo, hi, None if (c.get("bad") == "no_labels" and last) else labels)
        m = c["m"] + 1 if (c.get("bad") == "other_n" and last) else c["m"]
        Q = torch.from_numpy(c["Q"])
        try:
            if c["what"] == "labels":
                res = mdist.all_gather_cap_labels(shard).numpy()
            elif c["what"] == "topk":
                res = tuple(t.numpy() for t in mdist.sharded_batched_search(
                    shard, Q, c["k"], max_per_group=m, merge=numpy_packed_merge, walk=numpy_walk))
            else:
                groups = list(mdist.sharded_range_search_groups(shard, Q, c["R"], byte_cap=c["byte_cap"], merge=numpy_merge,
                                                                max_per_group=m, walk=numpy_walk))
                res = ([(g[0], g[1]) for g in groups],
                       tuple(t.numpy() for t in mdist.concat_range_groups(groups, Q.device)))
        except ValueError as exc:
            out[(name, rank)] = ("ValueError", str(exc))
            continue
        out[(name, rank)] = ("ok", res)
    td.destroy_process_group()


def _labels(kind, n, rng):
    if kind == "ungrouped":
        return np.full(n, -1, np.int32)
    if kind == "scattered":
        return rng.permutation(np.arange(n) // 5).astype(np.int32)
    if kind == "one_big":
        g = np.full(n, 3, np.int32)
        g[rng.choice(n, 9, replace=False)] = -1
        return g
    return (np.arange(n) // int(kind[1:])).astype(np.int32)               # "g7", "g40": contiguous, across shard borders


def _cases(world):
    from oracle import c_oracle
    rng = np.random.default_rng(10 + world)
    n = 101                                                               # uneven last shard at world 2 and 3
    S = rng.standard_normal((n, 24)).astype(np.float32)
    S[60] = S[3]; S[100] = S[3]; S[90] = 2 * S[3]                         # ties across the shard boundaries
    Q = np.concatenate([S[[3, 70, 99]].astype(np.float64), rng.standard_normal((14, 24))])
    R = float(np.median(np.stack([np.sort(c_oracle.distances(S, q)) for q in Q])[:, 25]))
    cases = {}
    for kind in ("g7", "g40", "scattered", "one_big", "ungrouped"):
        labels = _labels(kind, n, rng)
        cases["labels_" + kind] = dict(what="labels", S=S, labels=labels, Q=Q, m=1)
        for m in (1, 2):
            for k in (1, 5, 12):
                cases["topk_%s_%d_%d" % (kind, m, k)] = dict(what="topk", S=S, labels=labels, Q=Q, m=m, k=k)
            cases["range_%s_%d" % (kind, m)] = dict(what="range", S=S, labels=labels, Q=Q, m=m, R=R, byte_cap=None)
        cases["range_%s_small_cap" % kind] = dict(what="range", S=S, labels=labels, Q=Q, m=2, R=R,
                                                  byte_cap=12 * (world + 1) * 60)
    # one group's two nearest rows of query 0 on the first and the last rank: each rank's walk keeps its own
    P = S.copy()
    P[n - 1] = P[0] + 1e-3 * rng.standard_normal(24).astype(np.float32)
    planted = _labels("ungrouped", n, rng)
    planted[[0, n - 1]] = 5
    cases["planted"] = dict(what="topk", S=P, labels=planted, Q=P[[0]].astype(np.float64), m=1, k=3)
    cases["planted_range"] = dict(what="range", S=P, labels=planted, Q=P[[0]].astype(np.float64), m=1, R=0.01, byte_cap=None)
    tiny = rng.standard_normal((2, 8)).astype(np.float32)                # world 3: the last rank has no rows
    tiny_labels = np.array([4, 4], np.int32)
    tq = rng.standard_normal((5, 8))
    cases["empty_rank_labels"] = dict(what="labels", S=tiny, labels=tiny_labels, Q=tq, m=1)
    cases["empty_rank_topk"] = dict(what="topk", S=tiny, labels=tiny_labels, Q=tq, m=1, k=2)
    cases["empty_rank_range"] = dict(what="range", S=tiny, labels=tiny_labels, Q=tq, m=1, R=2.0, byte_cap=None)
    g7 = _labels("g7", n, rng)
    for what in ("topk", "range"):
        for bad in ("other_n", "no_labels"):
            cases["bad_%s_%s" % (what, bad)] = dict(what=what, S=S, labels=g7, Q=Q, m=2, k=5, R=R, byte_cap=None, bad=bad)
    return cases


def _brute_range(S, Q, R, labels, m):
    off, ids, d = brute_csr(S, Q, R)
    new_off, ni, nd = [0], [], []
    for j in range(len(Q)):
        li, ld = ids[off[j]:off[j + 1]], d[off[j]:off[j + 1]]
        keep = walk_keep(li, labels, m)
        ni.append(li[keep]); nd.append(ld[keep]); new_off.append(new_off[-1] + len(keep))
    return np.array(new_off, np.int64), np.concatenate(ni).astype(np.int32), np.concatenate(nd)


def _same(got, want):
    return all(np.array_equal(g, w) if g.dtype != np.float64 else np.array_equal(g.view(np.int64), w.view(np.int64))
               for g, w in zip(got, want))


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_capped_search_equals_single_process(world):
    cases = _cases(world)
    manager = mp.Manager()
    out = manager.dict()
    mp.spawn(_worker, args=(world, _free_port(), cases, out), nprocs=world, join=True)
    for name, c in cases.items():
        results = [out[(name, rank)] for rank in range(world)]
        if "bad" in c:
            assert all(r[0] == "ValueError" for r in results), (name, results)
            continue
        assert all(r[0] == "ok" for r in results), (name, results)
        if c["what"] == "labels":
            for _, got in results:
                assert np.array_equal(got, c["labels"]), name
            continue
        if c["what"] == "topk":
            want = brute_topk(c["S"], c["Q"], c["labels"], c["k"], c["m"])
            for rank, (_, got) in enumerate(results):
                assert _same(got, want), (name, rank)
            if name == "planted":
                assert results[0][1][0][0, 0] == 0 and c["S"].shape[0] - 1 not in results[0][1][0][0].tolist()
            continue
        want = _brute_range(c["S"], c["Q"], c["R"], c["labels"], c["m"])
        for rank, (_, (spans, got)) in enumerate(results):
            assert _same(got, want), (name, rank)
            assert spans == results[0][1][0], (name, rank)                     # the same groups on every rank
        if name.endswith("small_cap"):
            assert len(results[0][1][0]) > 1, name
        if name == "planted_range":
            assert want[1].tolist() == [0]
