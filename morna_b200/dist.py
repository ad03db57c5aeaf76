"""Multi-GPU exact search: the sample matrix is row-sharded (row = internal id) in
contiguous blocks, one process per GPU; every rank answers the replicated queries
on its block, the per-rank top-k lists are all-gathered (NCCL over NVLink; gloo in
CPU tests) and merged under the reference order.  The union of per-shard exact
top-k lists contains the global top-k, so the result equals one process scanning
all rows (morna.py:697-712).  This is the only exchange step on the path.

Range search (every row within a distance) runs over the same row blocks: sharded_range_search_groups below.
"""
import struct

import numpy as np
import torch

from . import _lib
from .search import _range_groups, check_radius, concat_range_groups


def shard_bounds(n_rows, rank, world):
    """Contiguous block [lo, hi) of rank `rank`: ceil(n/world) rows per rank."""
    per = -(-n_rows // world)
    lo = min(rank * per, n_rows)
    return lo, min(lo + per, n_rows)


def merge_topk(ids, dists, k, stream=None):
    """Exact top-k of concatenated candidate lists.  ids int32 [nq x m], dists float64
    [nq x m] on the GPU; entries with id < 0 are padding.  Order: distance ascending,
    equal distances id descending (morna.py:705-712)."""
    lib = _lib.load()
    assert ids.is_cuda and dists.is_cuda and ids.shape == dists.shape
    ids = ids.contiguous().to(torch.int32)
    dists = dists.contiguous().to(torch.float64)
    nq, m = ids.shape
    out_i = torch.empty((nq, k), dtype=torch.int32, device=ids.device)
    out_d = torch.empty((nq, k), dtype=torch.float64, device=ids.device)
    if nq == 0:
        return out_i, out_d
    with torch.cuda.device(ids.device):
        ws = _lib.workspace(lib.morna_select_topk_workspace_bytes(m, nq, k), ids.device)
        done = 0
        while done < nq:                     # grid.y limit of the select kernel
            cnt = min(nq - done, 65535)
            _lib.check(lib.morna_select_topk(_lib.dev_ptr(dists[done:]), _lib.dev_ptr(ids[done:]), m, m, 0, cnt, k,
                                             _lib.dev_ptr(out_i[done:]), _lib.dev_ptr(out_d[done:]),
                                             _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr(stream)),
                       "morna_select_topk")
            done += cnt
    return out_i, out_d


def merge_sorted_lists(ids, dists, k, stream=None):
    """Exact top-k of G sorted lists per query.  ids int32 / dists float64 [G x nq x k_in] on the GPU, every
    list sorted under the reference order (what each shard's search returns), padding id -1 / +inf."""
    lib = _lib.load()
    assert ids.is_cuda and dists.is_cuda and ids.shape == dists.shape and ids.dim() == 3
    ids = ids.contiguous().to(torch.int32)
    dists = dists.contiguous().to(torch.float64)
    g, nq, k_in = ids.shape
    out_i = torch.empty((nq, k), dtype=torch.int32, device=ids.device)
    out_d = torch.empty((nq, k), dtype=torch.float64, device=ids.device)
    with torch.cuda.device(ids.device):
        _lib.check(lib.morna_merge_sorted_topk(_lib.dev_ptr(dists), _lib.dev_ptr(ids), g, nq, k_in, k,
                                               _lib.dev_ptr(out_i), _lib.dev_ptr(out_d), _lib.stream_ptr(stream)),
                   "morna_merge_sorted_topk")
    return out_i, out_d


def all_gather_sorted(ids, dists, group=None):
    """Every rank's [nq x k] lists -> [world x nq x k] (one collective per tensor, no concatenation)."""
    import torch.distributed as td
    world = td.get_world_size(group)
    gi = torch.empty((world,) + tuple(ids.shape), dtype=ids.dtype, device=ids.device)
    gd = torch.empty((world,) + tuple(dists.shape), dtype=dists.dtype, device=dists.device)
    td.all_gather_into_tensor(gi, ids.contiguous(), group=group)
    td.all_gather_into_tensor(gd, dists.contiguous(), group=group)
    return gi, gd


def all_gather_topk(ids, dists, group=None):
    """Gather every rank's [nq x k] lists -> [nq x world*k], rank-major along dim 1."""
    import torch.distributed as td
    world = td.get_world_size(group)
    if world == 1:
        return ids, dists
    gi = [torch.empty_like(ids) for _ in range(world)]
    gd = [torch.empty_like(dists) for _ in range(world)]
    td.all_gather(gi, ids.contiguous(), group=group)
    td.all_gather(gd, dists.contiguous(), group=group)
    return torch.cat(gi, dim=1), torch.cat(gd, dim=1)


def _no_exclusion(query_groups):
    if query_groups is not None:
        raise ValueError("rows-sharded search has no per-query exclusion (query_groups); search one GPU's index instead")


def sharded_exact_search(local_search, queries, k, group=None, merge=None, query_groups=None):
    """`local_search(queries, k)` -> this rank's (ids, dists) with GLOBAL internal ids, sorted under the
    reference order.  Returns the merged global (ids, dists), identical on every rank.  On the GPU the
    lists are gathered as [world x nq x k] and merged by rank counting (morna_merge_sorted_topk); a
    `merge(ids [nq x world*k], dists, k)` callable replaces that (the CPU tests pass their own reference rule).
    ``query_groups`` (per-query exclusion) is not supported here: ValueError."""
    _no_exclusion(query_groups)
    import torch.distributed as td
    ids, dists = local_search(queries, k)
    if not (td.is_available() and td.is_initialized() and td.get_world_size(group) > 1):
        return ids, dists
    if merge is None and ids.is_cuda:
        gi, gd = all_gather_sorted(ids, dists, group)
        return merge_sorted_lists(gi, gd, k)
    ids, dists = all_gather_topk(ids, dists, group)
    return (merge or merge_topk)(ids, dists, k)


def sharded_batched_search(search, queries, k, group=None, check_overflow=True, query_groups=None):
    """Rows-sharded exact search of a query batch on the tensor-core path, one process per GPU.  `search` holds this
    rank's row block (MornaSearch(..., shard=(rank, world))), `queries` (CUDA float64 [nq x dim]) are replicated.

      1. every rank scores the queries against its rows and writes, per query, lower bounds of the true cosines of
         its k best rows (fp16 score minus the rank's rigorous error bound);
      2. ONE all-gather (4 * nq * k bytes per rank) and a k-th-largest over the world * k values per query give a bound
         that at least k rows over ALL shards reach -- so the ranks together re-rank about k rows per query instead of
         k rows each;
      3. every rank re-ranks (exact FP64) and orders its surviving rows; ONE more all-gather moves the [nq x k] lists
         (ids and distances packed in one buffer) and every rank merges them by rank counting.

    Returns (ids, dists), identical on every rank and identical to one process scanning all rows.  ``query_groups``
    (per-query exclusion) is not supported here: ValueError."""
    _no_exclusion(query_groups)
    import torch.distributed as td
    world = td.get_world_size(group) if (td.is_available() and td.is_initialized()) else 1
    if world == 1:
        return search.batched_search_device(queries, k, check_overflow=check_overflow)
    vals = search.batched_score_bound(queries, k)
    every = torch.empty((world,) + tuple(vals.shape), dtype=vals.dtype, device=vals.device)
    td.all_gather_into_tensor(every, vals, group=group)
    bound = search.union_kth_bound(every, k)
    nq = queries.shape[0]
    mine = torch.empty(nq * k * 12, dtype=torch.uint8, device=queries.device)      # the send buffer: the lists are written into it
    views = (mine[nq * k * 8:].view(torch.int32).view(nq, k), mine[:nq * k * 8].view(torch.float64).view(nq, k))
    search.batched_finish_bound(bound, check_overflow=check_overflow, out=views)
    return gather_merge_packed(views[0], views[1], k, group, packed=mine)


def gather_merge_packed(ids, dists, k, group=None, packed=None):
    """All-gather of every rank's sorted [nq x k] lists in ONE collective (distances and ids packed into one byte
    buffer per rank: `packed`, or packed here), then the rank-counting merge."""
    import torch.distributed as td
    world = td.get_world_size(group)
    nq, k_in = ids.shape
    nd, ni = nq * k_in * 8, nq * k_in * 4
    mine = packed
    if mine is None:
        mine = torch.empty(nd + ni, dtype=torch.uint8, device=ids.device)
        mine[:nd].view(torch.float64).copy_(dists.reshape(-1))
        mine[nd:].view(torch.int32).copy_(ids.reshape(-1))
    every = torch.empty((world, nd + ni), dtype=torch.uint8, device=ids.device)
    td.all_gather_into_tensor(every, mine, group=group)
    if (nq * k_in) % 2:                       # odd element count: the packed ids would not be 8-byte aligned per rank
        gd = every[:, :nd].contiguous().view(torch.float64).view(world, nq, k_in)
        gi = every[:, nd:].contiguous().view(torch.int32).view(world, nq, k_in)
        return merge_sorted_lists(gi, gd, k)
    lib = _lib.load()
    out_i = torch.empty((nq, k), dtype=torch.int32, device=ids.device)
    out_d = torch.empty((nq, k), dtype=torch.float64, device=ids.device)
    with torch.cuda.device(ids.device):
        _lib.check(lib.morna_merge_packed_topk(_lib.dev_ptr(every), world, nq, k_in, k, _lib.dev_ptr(out_i), _lib.dev_ptr(out_d),
                                               _lib.stream_ptr()), "morna_merge_packed_topk")
    return out_i, out_d


# ------------------------------------------------------------------ range search over a rows-sharded index
# A range list has no fixed length, so the ranks first agree on sizes: every size of a later collective (the query
# groups, each group's buffer) is computed from all-gathered counts, never from one rank's own counts.

def _world_size(group):
    import torch.distributed as td
    return td.get_world_size(group) if (td.is_available() and td.is_initialized()) else 1


def pack_range_lists(ids, dists, cap):
    """One rank's send buffer of the list all-gather: `cap` doubles (distances), then `cap` int32 (ids), as uint8
    [12 * cap] on the lists' device; slots past the lists are padding.  cap is even so every rank's buffer in the
    gathered tensor stays 8-byte aligned."""
    assert cap % 2 == 0 and ids.numel() == dists.numel() <= cap
    buf = torch.empty(cap * 12, dtype=torch.uint8, device=ids.device)
    m = ids.numel()
    buf[:cap * 8].view(torch.float64)[:m].copy_(dists)
    buf[cap * 8:].view(torch.int32)[:m].copy_(ids)
    return buf


def merge_sorted_csr(gathered, n_lists, nq, cap, rank_offsets, out_offsets, total, stream=None):
    """morna_merge_sorted_csr: the merged (ids, dists) [total] of n_lists packed buffers (pack_range_lists) back to back
    in `gathered`; rank_offsets int64 [n_lists * (nq + 1)] and out_offsets int64 [nq + 1] on the GPU."""
    lib = _lib.load()
    dev = gathered.device
    out_i = torch.empty(total, dtype=torch.int32, device=dev)
    out_d = torch.empty(total, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.morna_merge_sorted_csr(_lib.dev_ptr(gathered), n_lists, nq, cap, _lib.dev_ptr(rank_offsets),
                                              _lib.dev_ptr(out_offsets), total, _lib.dev_ptr(out_i), _lib.dev_ptr(out_d),
                                              _lib.stream_ptr(stream)), "morna_merge_sorted_csr")
    return out_i, out_d


def merge_gathered_csr(gathered, counts, cap, merge=None):
    """The step after the list all-gather: `gathered` (flat uint8, world buffers of pack_range_lists(.., cap)) and
    `counts` (host int64 [world x nq], every rank's matches per query of the group) -> the merged device CSR
    (offsets [nq + 1], ids, dists).  `merge` replaces morna_merge_sorted_csr (same arguments as merge_sorted_csr)."""
    counts = np.asarray(counts, dtype=np.int64)
    world, nq = counts.shape
    rank_off = np.zeros((world, nq + 1), dtype=np.int64)
    np.cumsum(counts, axis=1, out=rank_off[:, 1:])
    out_off = np.zeros(nq + 1, dtype=np.int64)
    np.cumsum(counts.sum(axis=0), out=out_off[1:])
    dev = gathered.device
    rank_off_t = torch.from_numpy(rank_off.reshape(-1)).to(dev)
    out_off_t = torch.from_numpy(out_off).to(dev)
    ids, dists = (merge or merge_sorted_csr)(gathered, world, nq, cap, rank_off_t, out_off_t, int(out_off[-1]))
    return out_off_t, ids, dists


def _range_group_exchange(search, st, lo, hi, counts, group, merge):
    """Queries [lo, hi) of a counted batch: this rank's lists, one all-gather, the merge.  counts: host [world x (hi-lo)]."""
    import torch.distributed as td
    dev = st["queries"].device
    cap = int(counts.sum(axis=1).max())
    cap += cap & 1
    if cap == 0:                                      # no rank has a match: every rank skips the list collective
        return (torch.zeros(hi - lo + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev),
                torch.zeros(0, dtype=torch.float64, device=dev))
    _, ids, dists = search.range_emit(st, lo, hi)
    mine = pack_range_lists(ids, dists, cap)
    every = torch.empty(counts.shape[0] * mine.numel(), dtype=torch.uint8, device=dev)
    td.all_gather_into_tensor(every, mine, group=group)
    return merge_gathered_csr(every, counts, cap, merge)


def sharded_range_search_groups(search, queries, max_distance, group=None, byte_cap=None, merge=None, query_groups=None):
    """Range search over a rows-sharded index, one process per GPU: generator over (lo, hi, offsets, ids, dists), the
    device CSR of queries [lo, hi) in query order, as MornaSearch.range_search_groups.  `search` holds this rank's row
    block (MornaSearch(..., shard=(rank, world))); `queries` (CUDA float64 [nq x dim]) and every argument are the same
    on every rank.  Every rank yields the same groups and lists, equal bit for bit to one process holding all rows.

      1. one all-gather of a header (nq, dim, radius bits, byte cap): ValueError on every rank if they differ;
      2. per batch of RANGE_BATCH_QUERIES queries every rank counts its matches (its own route, overflow handling and
         last_stats) and the counts are all-gathered; the query groups follow from the global counts alone, so the
         gathered lists plus the merged ones stay under byte_cap (one query per group at least);
      3. per group every rank writes its lists, ONE all-gather of the packed lists (skipped when no rank has a
         match), and morna_merge_sorted_csr (or `merge`) puts every entry in its place.
    Collectives use flat 1-D tensors on the queries' device (NCCL with CUDA tensors, gloo with CPU tensors).
    ``query_groups`` (per-query exclusion) is not supported here: ValueError."""
    _no_exclusion(query_groups)
    import torch.distributed as td
    world = _world_size(group)
    if world == 1:
        yield from search.range_search_groups(queries, max_distance, byte_cap)
        return
    dev = queries.device
    nq = int(queries.shape[0])
    r = float(max_distance)
    head = torch.tensor([nq, int(queries.shape[1]), struct.unpack("<q", struct.pack("<d", r))[0],
                         -1 if byte_cap is None else int(byte_cap)], dtype=torch.int64, device=dev)
    every = torch.empty(world * head.numel(), dtype=torch.int64, device=dev)
    td.all_gather_into_tensor(every, head, group=group)
    rows = every.view(world, -1).cpu()
    if not bool((rows == rows[0]).all()):
        raise ValueError("sharded range search: the ranks' (queries, dim, radius bits, byte cap) differ: %s" % rows.tolist())
    if nq == 0:
        check_radius(r)
        return
    for b0, st in search.range_count_batches(queries, r):
        counts = torch.from_numpy(np.ascontiguousarray(st["counts"], dtype=np.int64)).to(dev)
        every = torch.empty(world * counts.numel(), dtype=torch.int64, device=dev)
        td.all_gather_into_tensor(every, counts, group=group)
        rank_counts = every.cpu().numpy().reshape(world, -1)
        for lo, hi in _range_groups(rank_counts.sum(axis=0) * (world + 1), byte_cap):
            yield (b0 + lo, b0 + hi) + tuple(_range_group_exchange(search, st, lo, hi, rank_counts[:, lo:hi], group, merge))


def sharded_range_search(search, queries, max_distance, group=None, merge=None, query_groups=None):
    """The whole device CSR (offsets, ids, dists) of sharded_range_search_groups, as MornaSearch.range_search_device."""
    _no_exclusion(query_groups)
    if _world_size(group) == 1:
        return search.range_search_device(queries, max_distance)
    return concat_range_groups(list(sharded_range_search_groups(search, queries, max_distance, group, merge=merge)),
                               queries.device)
