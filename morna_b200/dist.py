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
from .search import _range_groups, check_max_per_group, check_radius, concat_range_groups


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


def sharded_batched_search(search, queries, k, group=None, check_overflow=True, query_groups=None, max_per_group=None,
                           merge=None, walk=None):
    """Rows-sharded exact search of a query batch on the tensor-core path, one process per GPU.  `search` holds this
    rank's row block (MornaSearch(..., shard=(rank, world))), `queries` (CUDA float64 [nq x dim]) are replicated.
    ``max_per_group``: a group-capped search (sharded_capped_search below; `merge` and `walk` are its hooks).

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
    if max_per_group is not None:
        return sharded_capped_search(search, queries, k, max_per_group, group, merge, walk)
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
    mine = packed if packed is not None else pack_topk_lists(ids, dists)
    every = torch.empty((world, mine.numel()), dtype=torch.uint8, device=ids.device)
    td.all_gather_into_tensor(every, mine, group=group)
    return merge_packed_lists(every, nq, k_in, k)


def pack_topk_lists(ids, dists):
    """One rank's send buffer of the packed list all-gather: nq * k doubles (distances), then nq * k int32 (ids)."""
    nd = ids.numel() * 8
    mine = torch.empty(nd + ids.numel() * 4, dtype=torch.uint8, device=ids.device)
    mine[:nd].view(torch.float64).copy_(dists.reshape(-1))
    mine[nd:].view(torch.int32).copy_(ids.reshape(-1))
    return mine


def merge_packed_lists(every, nq, k_in, k):
    """The rank-counting merge of an all-gather of packed lists: `every` uint8 [world x nq * k_in * 12], one
    pack_topk_lists buffer per rank -> the top-k (ids, dists) [nq x k]."""
    world = every.shape[0]
    nd = nq * k_in * 8
    if (nq * k_in) % 2:                       # odd element count: the packed ids would not be 8-byte aligned per rank
        gd = every[:, :nd].contiguous().view(torch.float64).view(world, nq, k_in)
        gi = every[:, nd:].contiguous().view(torch.int32).view(world, nq, k_in)
        return merge_sorted_lists(gi, gd, k)
    lib = _lib.load()
    out_i = torch.empty((nq, k), dtype=torch.int32, device=every.device)
    out_d = torch.empty((nq, k), dtype=torch.float64, device=every.device)
    with torch.cuda.device(every.device):
        _lib.check(lib.morna_merge_packed_topk(_lib.dev_ptr(every), world, nq, k_in, k, _lib.dev_ptr(out_i), _lib.dev_ptr(out_d),
                                               _lib.stream_ptr()), "morna_merge_packed_topk")
    return out_i, out_d


# ------------------------------------------------------------------ group-capped search over a rows-sharded index
# A group can have rows on several ranks, so a row one rank's walk kept can lose its place to another rank's rows of the
# same group: the per-rank lists are merged and the merged order is walked again, with every row's cap label.  Exact
# because every row of the global capped top-k is in its own rank's capped top-k (DESIGN.md section 6).

MERGE_MAX_ENTRIES = 200 * 1024 // 12      # world * k entries per query morna_merge_packed_topk stages in shared memory


def _cap_fields(search, max_per_group, group, world):
    """The capped header's fields: (N or -1 if malformed, index size, 1 if this rank has cap labels, 1 if its row block is
    shard_bounds' block of its rank).  Nothing here raises: a rank that raised on its own before a collective would
    leave the others waiting in it."""
    import torch.distributed as td
    try:
        m = check_max_per_group(max_per_group)
    except (TypeError, ValueError):
        m = -1
    block = (search.row_lo, search.row_hi) == shard_bounds(search.index_size, td.get_rank(group), world)
    return [m, int(search.index_size), int(search.cap_group is not None), int(block)]


def _agree(fields, names, dev, group, world, what):
    """One all-gather of an int64 header; ValueError on every rank unless every rank sent the same fields."""
    import torch.distributed as td
    head = torch.tensor(fields, dtype=torch.int64, device=dev)
    every = torch.empty(world * head.numel(), dtype=torch.int64, device=dev)
    td.all_gather_into_tensor(every, head, group=group)
    rows = every.view(world, -1).cpu()
    if not bool((rows == rows[0]).all()):
        raise ValueError("%s: the ranks' (%s) differ: %s" % (what, ", ".join(names), rows.tolist()))


def _check_cap_fields(max_per_group, fields):
    """After the header agreed: the cap as an int, or the same ValueError on every rank."""
    m = check_max_per_group(max_per_group)
    if not fields[2]:
        raise ValueError("max_per_group needs cap labels on every rank: call set_cap_groups first")
    if not fields[3]:
        raise ValueError("group-capped sharded search: the row blocks are not shard_bounds(%d, rank, world)" % fields[1])
    return m


CAP_FIELD_NAMES = ("max_per_group", "index size", "has cap labels", "row block of its rank")


def cap_label_block(search, world):
    """This rank's send buffer of the cap-label all-gather: its block's labels (set_cap_groups) padded with -1 to
    ceil(index_size / world) rows, so that the gathered blocks sit at their rows (shard_bounds blocks are contiguous)."""
    per = -(-search.index_size // world)
    mine = torch.full((per,), -1, dtype=torch.int32, device=search.cap_group.device)
    mine[:search.row_hi - search.row_lo] = search.cap_group
    return mine


def all_gather_cap_labels(search, group=None):
    """Every row's cap label, int32 [index_size] on this rank's device, in ONE all-gather of cap_label_block."""
    import torch.distributed as td
    world = td.get_world_size(group)
    mine = cap_label_block(search, world)
    every = torch.empty(world * mine.numel(), dtype=torch.int32, device=mine.device)
    td.all_gather_into_tensor(every, mine, group=group)
    return every[:search.index_size]


def merge_capped_topk(search, every, labels, nq, k, max_per_group, merge=None, walk=None):
    """The step after the list all-gather of a capped top-k: `every` (uint8 [world x nq * k * 12], each rank's capped
    [nq x k] lists as pack_topk_lists) merged whole, world * k entries per query (merge_packed_lists, or `merge` with its
    arguments), then the merged order walked with every row's label `labels` (int32 [index_size]) and cut to k
    (search.cap_sorted_lists, or `walk` with its arguments).  Returns (ids, dists) [nq x k], padded with -1 / +inf."""
    world = every.shape[0]
    ids, dists = (merge or merge_packed_lists)(every, nq, k, world * k)
    offsets = torch.arange(nq + 1, dtype=torch.int64, device=ids.device) * (world * k)
    out = (torch.empty((nq, k), dtype=torch.int32, device=ids.device), torch.empty((nq, k), dtype=torch.float64, device=ids.device))
    return (walk or search.cap_sorted_lists)(offsets, ids, dists, max_per_group, k, out=out, cap_group=labels)


def sharded_capped_search(search, queries, k, max_per_group, group=None, merge=None, walk=None):
    """Group-capped top-k over a rows-sharded index (sharded_batched_search(..., max_per_group=N)): per query the nearest
    rows with at most N of any one cap label, identical on every rank and to one process holding all rows.  Every rank
    labels its block (set_cap_groups(global_labels[lo:hi])) and passes the same arguments, max_per_group included.

      1. one all-gather of a header (nq, dim, k, N, index size, has cap labels, row block): ValueError on every rank if
         the ranks differ, or if N is malformed or no rank has labels;
      2. one all-gather of every row's cap label (all_gather_cap_labels; every call, 4 bytes per row);
      3. every rank's capped top-k of its rows (batched_search_device(..., max_per_group=N): the tensor cores, or the FP64
         route), ONE all-gather of the packed lists, the merge of all world * k entries and the walk over the merged
         order, cut to k (merge_capped_topk)."""
    world = _world_size(group)
    if world == 1:
        return search.batched_search_device(queries, k, max_per_group=max_per_group)
    nq, k = int(queries.shape[0]), int(k)
    fields = _cap_fields(search, max_per_group, group, world)
    _agree([nq, int(queries.shape[1]), k] + fields, ("queries", "dim", "k") + CAP_FIELD_NAMES, queries.device, group, world,
           "group-capped sharded search")
    m = _check_cap_fields(max_per_group, fields)
    if world * k > MERGE_MAX_ENTRIES:
        raise ValueError("group-capped sharded search: world size x k = %d exceeds %d" % (world * k, MERGE_MAX_ENTRIES))
    labels = all_gather_cap_labels(search, group)
    ids, dists = search.batched_search_device(queries, k, max_per_group=m)
    if nq == 0 or k <= 0:                 # the same on every rank: no list collective
        return ids, dists
    import torch.distributed as td
    mine = pack_topk_lists(ids, dists)
    every = torch.empty(world * mine.numel(), dtype=torch.uint8, device=mine.device)     # (flat: gloo takes 1-D only)
    td.all_gather_into_tensor(every, mine, group=group)
    return merge_capped_topk(search, every.view(world, -1), labels, nq, k, m, merge, walk)


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


def sharded_range_search_groups(search, queries, max_distance, group=None, byte_cap=None, merge=None, query_groups=None,
                                max_per_group=None, walk=None):
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
    ``max_per_group`` (every rank labelled as for sharded_capped_search): the header also carries N, the index size and
    the label checks, every row's cap label is all-gathered once, and each group's merged lists (the union of the ranks'
    uncapped lists: the global in-range lists) are walked (search.cap_sorted_lists, or `walk` with its arguments);
    byte_cap bounds the lists before the walk.  ``query_groups`` (per-query exclusion) is not supported here: ValueError."""
    _no_exclusion(query_groups)
    import torch.distributed as td
    world = _world_size(group)
    if world == 1:
        yield from search.range_search_groups(queries, max_distance, byte_cap, max_per_group=max_per_group)
        return
    dev = queries.device
    nq = int(queries.shape[0])
    r = float(max_distance)
    fields = [nq, int(queries.shape[1]), struct.unpack("<q", struct.pack("<d", r))[0], -1 if byte_cap is None else int(byte_cap)]
    if max_per_group is None:
        head = torch.tensor(fields, dtype=torch.int64, device=dev)
        every = torch.empty(world * head.numel(), dtype=torch.int64, device=dev)
        td.all_gather_into_tensor(every, head, group=group)
        rows = every.view(world, -1).cpu()
        if not bool((rows == rows[0]).all()):
            raise ValueError("sharded range search: the ranks' (queries, dim, radius bits, byte cap) differ: %s" % rows.tolist())
        m = labels = None
    else:
        cap_fields = _cap_fields(search, max_per_group, group, world)
        _agree(fields + cap_fields, ("queries", "dim", "radius bits", "byte cap") + CAP_FIELD_NAMES, dev, group, world,
               "sharded range search")
        m = _check_cap_fields(max_per_group, cap_fields)
    if nq == 0:
        check_radius(r)
        return
    if m is not None:
        labels = all_gather_cap_labels(search, group)
    for b0, st in search.range_count_batches(queries, r):
        counts = torch.from_numpy(np.ascontiguousarray(st["counts"], dtype=np.int64)).to(dev)
        every = torch.empty(world * counts.numel(), dtype=torch.int64, device=dev)
        td.all_gather_into_tensor(every, counts, group=group)
        rank_counts = every.cpu().numpy().reshape(world, -1)
        for lo, hi in _range_groups(rank_counts.sum(axis=0) * (world + 1), byte_cap):
            csr = _range_group_exchange(search, st, lo, hi, rank_counts[:, lo:hi], group, merge)
            if m is not None:
                csr = (walk or search.cap_sorted_lists)(*csr, m, cap_group=labels)
            yield (b0 + lo, b0 + hi) + tuple(csr)


def sharded_range_search(search, queries, max_distance, group=None, merge=None, query_groups=None, max_per_group=None,
                         walk=None):
    """The whole device CSR (offsets, ids, dists) of sharded_range_search_groups, as MornaSearch.range_search_device."""
    _no_exclusion(query_groups)
    if _world_size(group) == 1:
        return search.range_search_device(queries, max_distance, max_per_group=max_per_group)
    return concat_range_groups(list(sharded_range_search_groups(search, queries, max_distance, group, merge=merge,
                                                                max_per_group=max_per_group, walk=walk)), queries.device)
