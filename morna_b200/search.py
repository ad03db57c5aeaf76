"""MornaSearch -- host-side mirror of the reference class (morna.py:522-787) with the
exact scan running on the B200.  Loads basename.stats/.freq/.map.mor and the vector
store, keeps the float32 sample matrix resident in HBM, and answers exact angular
top-k queries under the reference's order (distance ascending, ties id-descending).
"""
import ctypes
import gc
import math
import os
from collections import defaultdict

import numpy as np
import torch

from . import _lib, files
from .index import round_up


PHASE_NAMES = ("prep_queries", "gemm_pilot", "kth_pilot", "gemm_filter", "kth_final", "rerank_select")


def check_radius(max_distance):
    """A range search radius as a float: finite and >= 0, else ValueError."""
    r = float(max_distance)
    if not (math.isfinite(r) and r >= 0.0):
        raise ValueError("max_distance must be a finite number >= 0, got %r" % (max_distance,))
    return r


def check_max_per_group(max_per_group):
    """A group cap as an int: an integer >= 1, else ValueError."""
    if isinstance(max_per_group, bool) or int(max_per_group) != max_per_group or max_per_group < 1:
        raise ValueError("max_per_group must be an integer >= 1, got %r" % (max_per_group,))
    return int(max_per_group)


def _range_groups(counts, byte_cap):
    """[lo, hi) runs of consecutive queries whose lists (12 bytes per match) fit byte_cap; one run without a cap."""
    nq = len(counts)
    if byte_cap is None:
        return [(0, nq)] if nq else []
    groups, lo, size = [], 0, 0
    for j, c in enumerate(np.asarray(counts, dtype=np.int64).tolist()):
        if j > lo and size + 12 * c > byte_cap:
            groups.append((lo, j))
            lo, size = j, 0
        size += 12 * c
    if nq:
        groups.append((lo, nq))
    return groups


def concat_range_groups(parts, device):
    """One CSR (offsets, ids, dists) from consecutive (lo, hi, offsets, ids, dists) groups of a range search."""
    if not parts:
        return (torch.zeros(1, dtype=torch.int64, device=device), torch.zeros(0, dtype=torch.int32, device=device),
                torch.zeros(0, dtype=torch.float64, device=device))
    offsets, base = [parts[0][2][:1]], 0
    for p in parts:
        offsets.append(p[2][1:] + base)
        base += p[3].numel()
    return torch.cat(offsets), torch.cat([p[3] for p in parts]), torch.cat([p[4] for p in parts])


def _member_internal_id(internal_id_map, query_id, out=None):
    """search -q: the internal id of sample `query_id`, with the two progress lines the reference prints (morna.py:733-745)."""
    import sys
    out = out or sys.stdout
    out.write("querying by sample id " + str(query_id) + "\n")
    try:
        internal_id = internal_id_map[query_id]
    except KeyError:
        raise ValueError("Querying sample id " + str(query_id) + " is not possible because no internal "
                         "id is mapped to that sample id. Likely no sample with that id was included "
                         "in the index.")
    out.write("this is internal id " + str(internal_id) + "\n")
    return internal_id


def make_phase_events():
    """Seven CUDA events for morna_knn_batched's phase boundaries: (events, ctypes array)."""
    import ctypes
    events = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
    for e in events:
        e.record()                      # creates the underlying cudaEvent_t
    return events, (ctypes.c_void_p * 7)(*[e.cuda_event for e in events])


class MornaSearch(object):
    def __init__(self, basename=None, device=None, shard=None, vectors=None, stats=None,
                 sample_frequencies=None, internal_id_map=None):
        """``basename``: index files to load (morna.py:530-550).  ``shard=(rank, world)``
        keeps only this rank's contiguous block of rows (row = internal id).
        Alternatively pass ``vectors`` (numpy/torch [n x dim] float32) and ``stats``
        = (sample_count, index_size, dim) directly."""
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.basename = basename
        if basename is not None:
            self.sample_count, self.index_size, self.dim = files.read_stats(basename)
            self.sample_frequencies = files.read_freq(basename)
            self.internal_id_map = files.read_map(basename)
            if os.path.exists(basename + ".vec.mor"):
                host = files.read_vectors(basename)
            elif os.path.exists(basename + ".annoy.mor"):
                host = files.read_annoy_item_vectors(basename + ".annoy.mor", self.index_size, self.dim)
            else:
                raise IOError("no vector store for index " + basename)
        else:
            self.sample_count, self.index_size, self.dim = stats
            self.sample_frequencies = sample_frequencies if sample_frequencies is not None else defaultdict(int)
            self.internal_id_map = internal_id_map if internal_id_map is not None else {}
            host = vectors
        if host.shape != (self.index_size, self.dim):
            raise ValueError("vector store shape %r does not match stats %r"
                             % (tuple(host.shape), (self.index_size, self.dim)))
        rank, world = shard if shard is not None else (0, 1)
        per = -(-self.index_size // world)
        self.row_lo = min(rank * per, self.index_size)
        self.row_hi = min(self.row_lo + per, self.index_size)
        self.ld = round_up(self.dim, 4)
        self._load_rows(host)
        self.query = defaultdict(int)                      # morna.py:540
        self.query_sample = [0.0] * self.dim               # :541

    def _load_rows(self, host):
        n = self.row_hi - self.row_lo
        dev = self.device
        self.vectors = torch.zeros((n, self.ld), dtype=torch.float32, device=dev)
        if n:
            if isinstance(host, torch.Tensor):
                block = host[self.row_lo:self.row_hi].to(torch.float32)
            else:
                block = torch.from_numpy(np.array(host[self.row_lo:self.row_hi], dtype=np.float32, order="C"))
            self.vectors[:, :self.dim].copy_(block, non_blocking=False)
        self.pp = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            if n:                                          # (a rank of a rows-sharded index may hold no rows)
                _lib.check(self.lib.morna_row_norms(_lib.dev_ptr(self.vectors), n, self.dim, self.ld,
                                                    _lib.dev_ptr(self.pp), _lib.stream_ptr()), "morna_row_norms")
        self._build_csr()

    def _summation_plans(self, counts, row_off, cols):
        """int32 per row for morna_knn_exact_sparse (layout in include/morna_b200.h): how a row of <= 3 non-zeros reproduces
        the dense kernels' summation tree with three accumulators; bit 30 for longer rows (generic emulation)."""
        n, dev = counts.shape[0], self.device
        c = torch.full((n, 3), -1, dtype=torch.int64, device=dev)
        for e in range(3):
            have = counts > e
            c[have, e] = cols[(row_off[:-1][have] + e).clamp_max(cols.numel() - 1)].to(torch.int64)
        lane = (c >> 2) & 31
        l0, l1, l2 = lane[:, 0], lane[:, 1], lane[:, 2]

        def lowbit(x):
            return x & (-x)
        lab, lac, lbc = lowbit(l0 ^ l1), lowbit(l0 ^ l2), lowbit(l1 ^ l2)
        m = torch.maximum(torch.maximum(lab, lac), lbc)
        zero, one, two = (torch.full((n,), v, dtype=torch.int64, device=dev) for v in (0, 1, 2))
        t1 = torch.where(l0 == l1, zero, one)
        # three entries: equal lanes share an accumulator; of three distinct lanes the pair that meets first in the butterfly
        # (largest lowest-differing bit) takes accumulators 0 and 1
        t1_3 = torch.where(l0 == l1, zero, torch.where(l0 == l2, one, torch.where(l1 == l2, one,
                           torch.where(lab == m, one, torch.where(lac == m, two, zero)))))
        t2_3 = torch.where((l0 == l1) & (l1 == l2), zero, torch.where(l0 == l1, one, torch.where(l0 == l2, zero,
                           torch.where(l1 == l2, one, torch.where(lab == m, two, one)))))
        t0_3 = torch.where((l0 != l1) & (l0 != l2) & (l1 != l2) & (lab != m) & (lac != m), two, zero)
        three = counts == 3
        t0 = torch.where(three, t0_3, zero)
        t1 = torch.where(three, t1_3, torch.where(counts == 2, t1, zero))
        t2 = torch.where(three, t2_3, zero)
        plan = t0 | (t1 << 2) | (t2 << 4) | (counts.to(torch.int64) << 8)
        plan = torch.where(counts > 3, torch.full_like(plan, 1 << 30), plan)
        return plan.to(torch.int32).contiguous()

    def _build_csr(self):
        """A sparse index (every row has at most morna_sparse_max_nnz() non-zero buckets -- an index built from a handful
        of junctions, like the reference's fixture) also keeps its rows in CSR form: exact search then costs nnz(row)
        multiply-adds per (query, row) instead of D, with the same bits (morna_knn_exact_sparse).  Index-load time,
        not the hot path: plain torch ops."""
        self.csr = None
        n = self.row_hi - self.row_lo
        if n == 0:
            return
        nz = self.vectors != 0
        counts = nz.sum(dim=1)
        if int(counts.max()) > int(self.lib.morna_sparse_max_nnz()):
            return
        where = nz.nonzero()                               # row-major: columns ascending within a row
        row_off = torch.zeros(n + 1, dtype=torch.int64, device=self.device)
        row_off[1:] = counts.cumsum(0)
        cols = where[:, 1].to(torch.int32).contiguous()
        vals = self.vectors[where[:, 0], where[:, 1]].contiguous()
        if cols.numel() == 0:                              # all-zero index: keep valid pointers
            cols = torch.zeros(1, dtype=torch.int32, device=self.device)
            vals = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.csr = (row_off, cols, vals, self._summation_plans(counts, row_off, cols))
        # Which path answers a batch.  Rows with the same non-zero buckets can be parallel to each other (one bucket:
        # always), i.e. tie from every query's point of view; when the largest such group is wider than the tensor
        # path's candidate lists, its queries would all overflow into the exact scan -- then the CSR exact path answers
        # directly.  Otherwise the tensor-core path is faster even on sparse rows.
        pos = torch.arange(where.shape[0], device=self.device) - row_off[where[:, 0]]
        sig = torch.zeros(n, dtype=torch.int64, device=self.device)
        sig.index_add_(0, where[:, 0], (where[:, 1] + 1) * torch.pow(torch.tensor(1000003, device=self.device), pos))
        self.largest_tie_group = int(torch.unique(sig, return_counts=True)[1].max())
        self.sparse_exact = self.largest_tie_group >= self.TIE_GROUP_FOR_SPARSE_PATH

    # ------------------------------------------------------------------ query construction
    def inverse_lookup(self, internal_id):
        """morna.py:554-572."""
        match, found = None, False
        for sample_id, iid in self.internal_id_map.items():
            if iid == internal_id:
                if found:
                    raise RuntimeError(str(internal_id) + " does not have unique mapping in self.internal_id_map.")
                match, found = sample_id, True
        return match

    def update_query(self, junction):
        """morna.py:597-607."""
        self.query[tuple(junction[:3])] += int(junction[3])

    def hash_keys(self, keys):
        """Device feature hashing of a list of key strings -> (raw, bucket, sign) numpy."""
        blobs = [k.encode("utf-8") for k in keys]
        n = len(blobs)
        if n == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int8)
        off = np.zeros(n + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(b) for b in blobs])
        packed = np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8).copy()
        dev = self.device
        with torch.cuda.device(dev):
            d_keys, d_off = torch.from_numpy(packed).to(dev), torch.from_numpy(off).to(dev)
            raw = torch.empty(n, dtype=torch.int32, device=dev)
            bucket = torch.empty(n, dtype=torch.int32, device=dev)
            sign = torch.empty(n, dtype=torch.int8, device=dev)
            _lib.check(self.lib.morna_hash_junctions(_lib.dev_ptr(d_keys), _lib.dev_ptr(d_off), n, self.dim,
                                                     _lib.dev_ptr(raw), _lib.dev_ptr(bucket), _lib.dev_ptr(sign),
                                                     _lib.stream_ptr()), "morna_hash_junctions")
            return raw.cpu().numpy(), bucket.cpu().numpy(), sign.cpu().numpy()

    def finalize_query(self):
        """morna.py:609-629: hashed, idf-weighted, signed accumulation of the query
        junctions into ``query_sample`` (Python floats, dictionary order)."""
        self.query_sample = [0.0] * self.dim
        junctions = list(self.query.keys())
        keys = [" ".join(str(t) for t in j) for j in junctions]
        _, bucket, sign = self.hash_keys(keys)
        for j, key, b, s in zip(junctions, keys, bucket.tolist(), sign.tolist()):
            freq = self.sample_frequencies[key]             # defaultdict: inserts 0 like the reference (:619)
            idf = 0 if freq == 0 else math.log(float(self.sample_count) / freq)
            self.query_sample[b] += s * (self.query[j] * idf)

    # ------------------------------------------------------------------ exact search
    def _workspace(self, nbytes, kind="exact"):
        """Scratch of the CURRENT stream: calls in flight on different streams never share a workspace."""
        pool = self.__dict__.setdefault("_ws_pool", {})
        key = (kind, torch.cuda.current_stream(self.device).cuda_stream)
        ws = pool.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = pool[key] = _lib.workspace(nbytes, self.device)
            if kind == "single":
                _lib.check(self.lib.morna_knn_single_workspace_init(_lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()),
                           "morna_knn_single_workspace_init")
                pool[("single_flag", key[1])] = torch.zeros(1, dtype=torch.int32, device=self.device)
        return ws

    def single_search_device(self, query, k, stream=None):
        """One query (CUDA float64 [dim]) through the HBM-bound single-query kernel.  Same results as the
        FP64 scan; falls back to it when ties overflow the candidate list.  Everything (allocations, kernels,
        the read of the fallback flag) happens on ``stream`` (default: the current stream)."""
        assert query.is_cuda and query.dtype == torch.float64 and query.numel() == self.dim
        if stream is not None and stream != torch.cuda.current_stream(self.device):
            with torch.cuda.stream(stream):
                return self.single_search_device(query, k)
        query = query.contiguous()
        n, dev = self.row_hi - self.row_lo, self.device
        k_eff = min(int(k), n)
        if n == 0 or k_eff <= 0 or k_eff > 512:
            return self.exact_search_device(query.view(1, -1), k, allow_single=False)
        out_ids = torch.full((1, k), -1, dtype=torch.int32, device=dev)
        out_d = torch.full((1, k), float("inf"), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            sws = self._workspace(self.lib.morna_knn_single_workspace_bytes(n), "single")
            flag = self._ws_pool[("single_flag", torch.cuda.current_stream(dev).cuda_stream)]
            self._sws, self._sfallback = sws, flag            # (kept for callers that replay the call, e.g. bench.py)
            _lib.check(self.lib.morna_knn_single(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, self.row_lo,
                _lib.ptr(query), k_eff, _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d), _lib.dev_ptr(flag),
                _lib.dev_ptr(sws), sws.numel(), _lib.stream_ptr()), "morna_knn_single")
            if int(flag.item()):
                return self.exact_search_device(query.view(1, -1), k, allow_single=False)
        return out_ids, out_d

    def single_search_stream(self, queries, k):
        """A stream of single queries (CUDA float64 [m x dim]), each answered by its own full pass of the
        single-query kernel, launched back to back so that query j+1's scan runs under query j's selection tail
        (morna_knn_single_stream; programmatic dependent launch, two alternating workspaces).  Same results as
        single_search_device per query; queries whose ties overflow the lists are answered by the FP64 scan."""
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.dim() == 2 and queries.shape[1] == self.dim
        queries = queries.contiguous()
        m, n, dev = queries.shape[0], self.row_hi - self.row_lo, self.device
        k_eff = min(int(k), n)
        if m == 0 or n == 0 or k_eff <= 0 or k_eff > 512 or self.csr is not None:
            return self.exact_search_device(queries, k, allow_single=False)
        out_ids = torch.full((m, k), -1, dtype=torch.int32, device=dev)
        out_d = torch.full((m, k), float("inf"), dtype=torch.float64, device=dev)
        ids_k = out_ids if k_eff == k else torch.empty((m, k_eff), dtype=torch.int32, device=dev)
        d_k = out_d if k_eff == k else torch.empty((m, k_eff), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            ws = self._single_stream_workspace(n)
            flags = torch.zeros(m, dtype=torch.int32, device=dev)
            _lib.check(self.lib.morna_knn_single_stream(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, self.row_lo,
                _lib.ptr(queries), self.dim, m, k_eff, _lib.dev_ptr(ids_k), _lib.dev_ptr(d_k), _lib.dev_ptr(flags),
                _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_knn_single_stream")
            if k_eff != k:
                out_ids[:, :k_eff] = ids_k
                out_d[:, :k_eff] = d_k
            redo = torch.nonzero(flags).flatten()
            if redo.numel():
                e_ids, e_d = self.exact_search_device(queries[redo], k, allow_single=False)
                out_ids[redo] = e_ids
                out_d[redo] = e_d
        return out_ids, out_d

    def _single_stream_workspace(self, n):
        """Two single-query workspaces back to back (the halves alternate between consecutive queries), per stream."""
        half = self.lib.morna_knn_single_workspace_bytes(n)
        pool = self.__dict__.setdefault("_ws_pool", {})
        key = ("single_stream", torch.cuda.current_stream(self.device).cuda_stream)
        ws = pool.get(key)
        if ws is None or ws.numel() < 2 * half:
            ws = pool[key] = _lib.workspace(2 * half, self.device)
            for h in (0, 1):
                _lib.check(self.lib.morna_knn_single_workspace_init(ctypes.c_void_p(ws.data_ptr() + h * half), half, _lib.stream_ptr()),
                           "morna_knn_single_workspace_init")
        return ws

    row_group = None                 # device int32 [n]: label of every resident row (set_row_groups), or None

    def set_row_groups(self, labels):
        """Labels for per-query exclusion: int32 [n], one per resident row (None clears them).  A search given
        ``query_groups`` then leaves out, for query q, every row whose label equals query_groups[q] (a label < 0 excludes
        nothing): with every row its own label and a query's label its row's, a stored row no longer finds itself."""
        self._within = None                                # (the within-group layout of the old labels)
        if labels is None:
            self.row_group = None
            return
        t = torch.as_tensor(labels).to(device=self.device, dtype=torch.int32).contiguous()
        if t.shape != (self.row_hi - self.row_lo,):
            raise ValueError("row labels must be one per resident row (%d), got shape %r" % (self.row_hi - self.row_lo, tuple(t.shape)))
        self.row_group = t

    def _query_groups(self, query_groups, nq):
        """Query labels as device int32 [nq], or None without an exclusion."""
        if query_groups is None:
            return None
        if self.row_group is None:
            raise ValueError("query_groups need row labels: call set_row_groups first")
        qg = torch.as_tensor(query_groups).to(device=self.device, dtype=torch.int32).contiguous()
        if qg.shape != (nq,):
            raise ValueError("query_groups must hold one label per query (%d), got shape %r" % (nq, tuple(qg.shape)))
        return qg

    def _excl_args(self, qg, rows=slice(None)):
        """The (row_group, query_group) pointers an *_excl entry point takes."""
        return (_lib.dev_ptr(self.row_group[rows]), _lib.dev_ptr(qg))

    cap_group = None                 # device int32 [n]: cap label of every resident row (set_cap_groups), or None

    def set_cap_groups(self, labels):
        """Labels for group-capped search: int32 [n], one per resident row (None clears them); a label < 0 leaves the row
        ungrouped (a group of its own, never capped).  A search given ``max_per_group=N`` then returns, per query, the
        nearest rows with at most N rows of any one label.  Independent of set_row_groups: "leave out my own study, at
        most N per other study" takes both."""
        self._cap_prefix = {}
        if labels is None:
            self.cap_group = None
            return
        t = torch.as_tensor(labels).to(device=self.device, dtype=torch.int32).contiguous()
        if t.shape != (self.row_hi - self.row_lo,):
            raise ValueError("cap labels must be one per resident row (%d), got shape %r" % (self.row_hi - self.row_lo, tuple(t.shape)))
        self.cap_group = t

    CAP_BLOCK = 2048                 # rows a capped block may add to a candidate list (of 4096) above a weak threshold

    def _cap_blocks(self, m, k):
        """Block ends (host int64) for the capped tensor route (morna_knn_batched_capped's block_ends), from the labels
        alone.  c(b), the capped entries the first b rows hold (a label counted at most m times, an ungrouped row once),
        bounds how selective a threshold after b rows can be: below k + m there may be none (the extra m covers a query
        that excludes one group), and above it about k + m of c(b) representatives pass, so a block of
        CAP_BLOCK * c(b) / (k + m) rows adds about CAP_BLOCK entries.  Ends are multiples of CAP_BLOCK while below that,
        so that any pilot size that is a multiple of it lands on one; the usual blocks take over at BATCH_BLOCK_ROWS ...
        131072 rows per block.  Cached per (m, k)."""
        cache = self.__dict__.setdefault("_cap_prefix", {})
        if (m, k) in cache:
            return cache[(m, k)]
        counts = cache.get(m)
        if counts is None:
            g = self.cap_group.long()
            n = g.numel()
            order = torch.sort(g, stable=True).indices
            sg = g[order]
            head = torch.ones(n, dtype=torch.bool, device=g.device)
            head[1:] = sg[1:] != sg[:-1]
            pos = torch.arange(n, device=g.device)
            rank = torch.empty_like(pos)
            rank[order] = pos - torch.cummax(torch.where(head, pos, torch.zeros_like(pos)), 0).values
            counts = cache[m] = ((g < 0) | (rank < m)).to(torch.int64).cumsum(0).cpu().numpy()
        n, need, ends, b = counts.size, k + m, [], 0
        while b < n:
            c = int(counts[b - 1]) if b else 0
            step = self.CAP_BLOCK if c < need else min(131072, max(self.CAP_BLOCK, self.CAP_BLOCK * c // need))
            b = min(n, b + step)
            ends.append(b)
            if step == 131072:
                break
        cache[(m, k)] = out = np.array(ends, dtype=np.int64)
        return out

    def _cap(self, max_per_group):
        """max_per_group as an int >= 1, or None for an uncapped search."""
        if max_per_group is None:
            return None
        m = check_max_per_group(max_per_group)
        if self.cap_group is None:
            raise ValueError("max_per_group needs cap labels: call set_cap_groups first")
        return m

    def cap_sorted_lists(self, offsets, ids, dists, max_per_group, limit=None, out=None, cap_group=None):
        """The walk of a capped search (morna_cap_sorted_lists) over device lists already in the reference order: offsets
        int64 [L+1], ids int32 (global; -1 is padding), dists float64.  Each entry is kept iff fewer than max_per_group
        entries of its cap label were kept before it in its list, and at most ``limit`` per list (None: no limit).  Returns
        the capped CSR (offsets, ids, dists), or with ``out`` = (ids [L x w], dists [L x w]) fills those, padded.
        ``cap_group``: device int32 labels indexed from id 0 (every row of a rows-sharded index) in place of this
        block's own."""
        L, total = offsets.numel() - 1, ids.numel()
        dev = self.device
        lim = -1 if limit is None else max(int(limit), 0)
        if cap_group is None:
            labels = (self.cap_group, self.row_lo, self.row_hi - self.row_lo)
        else:
            labels = (cap_group, 0, cap_group.numel())
        with torch.cuda.device(dev):
            ws = self._workspace(self.lib.morna_cap_sorted_lists_workspace_bytes(L, total), "cap_walk")
            args = (_lib.dev_ptr(offsets), L, _lib.ptr(ids), _lib.ptr(dists), total, _lib.dev_ptr(labels[0]), labels[1],
                    labels[2], max_per_group, lim)
            if out is not None:
                _lib.check(self.lib.morna_cap_sorted_lists(*args, None, _lib.ptr(out[0]), _lib.ptr(out[1]), out[0].shape[1],
                                                           _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_cap_sorted_lists")
                return out
            out_off = torch.empty(L + 1, dtype=torch.int64, device=dev)
            out_ids = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
            out_d = torch.empty(max(total, 1), dtype=torch.float64, device=dev)
            _lib.check(self.lib.morna_cap_sorted_lists(*args, _lib.dev_ptr(out_off), _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d), 0,
                                                       _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_cap_sorted_lists")
            kept = int(out_off[-1].item())
            return out_off, out_ids[:kept], out_d[:kept]

    CAPPED_SORT_ENTRIES = 1 << 24    # distances sorted at once by the capped FP64 route (queries x rows)

    def _capped_search(self, queries, k, qg, m):
        """Top-k with at most m rows per cap label (see set_cap_groups): the tensor-core route (morna_knn_batched_capped)
        for a dense index of one row block and k <= 512, its overflowed queries and everything else by the FP64 route."""
        nq, n, dev = queries.shape[0], self.row_hi - self.row_lo, self.device
        k = max(int(k), 0)
        if n == 0 or nq == 0 or k == 0:
            return (torch.full((nq, k), -1, dtype=torch.int32, device=dev),
                    torch.full((nq, k), float("inf"), dtype=torch.float64, device=dev))
        if k > 512 or n > self.BATCH_BLOCK_ROWS or (self.csr is not None and self.sparse_exact):
            return self._capped_full_sort(queries, k, qg, m)
        self.enable_tensor_path()
        with torch.cuda.device(dev):
            out_ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
            out_d = torch.empty((nq, k), dtype=torch.float64, device=dev)
            overflow = torch.empty(nq, dtype=torch.uint8, device=dev)
            stats = torch.empty(4, dtype=torch.int32, device=dev)
            ws = self._workspace(self.lib.morna_knn_batched_capped_workspace_bytes(n, nq, self.dim, k), "capped")
            excl = (None, None) if qg is None else self._excl_args(qg)
            blocks = self._cap_blocks(m, k)
            _lib.check(self.lib.morna_knn_batched_capped(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), _lib.dev_ptr(self.hs), self.ld_h, _lib.dev_ptr(self.rho_max),
                n, self.dim, self.ld, self.row_lo, _lib.ptr(queries), nq, self.dim, k, _lib.dev_ptr(self.cap_group), m,
                blocks.ctypes.data_as(ctypes.c_void_p), blocks.size, *excl,
                _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d), _lib.dev_ptr(overflow), _lib.dev_ptr(stats), _lib.dev_ptr(ws),
                ws.numel(), _lib.stream_ptr()), "morna_knn_batched_capped")
            st = stats.cpu()
            self.last_stats = st.to(torch.int64).tolist()
            if int(st[0]) > 0:
                idx = overflow.nonzero().flatten()
                e_ids, e_d = self._capped_full_sort(queries[idx], k, None if qg is None else qg[idx], m)
                out_ids[idx] = e_ids
                out_d[idx] = e_d
        return out_ids, out_d

    def _capped_full_sort(self, queries, k, qg, m):
        """The capped FP64 route: every row's canonical FP64 distance (morna_angular_distances), excluded pairs at +inf, a
        full sort per query under the reference order (torch's; rare), then the walk.  Any k, any number of rows."""
        nq, n, dev = queries.shape[0], self.row_hi - self.row_lo, self.device
        out_ids = torch.full((nq, k), -1, dtype=torch.int32, device=dev)
        out_d = torch.full((nq, k), float("inf"), dtype=torch.float64, device=dev)
        if n == 0 or nq == 0 or k == 0:
            return out_ids, out_d
        per = max(1, self.CAPPED_SORT_ENTRIES // n)
        with torch.cuda.device(dev):
            for j0 in range(0, nq, per):
                q = queries[j0:j0 + per].contiguous()
                b = q.shape[0]
                dist = torch.empty((b, n), dtype=torch.float64, device=dev)
                _lib.check(self.lib.morna_angular_distances(
                    _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, _lib.ptr(q), b, self.dim,
                    _lib.dev_ptr(dist), n, _lib.stream_ptr()), "morna_angular_distances")
                if qg is not None:
                    g = qg[j0:j0 + b, None]
                    dist.masked_fill_((self.row_group[None, :] == g) & (g >= 0), float("inf"))
                # distance ascending, equal distances id descending: stable sort of the id-reversed rows
                rows = (n - 1) - torch.sort(dist.flip(1), dim=1, stable=True).indices
                d = dist.gather(1, rows)
                del dist
                ids = torch.where(torch.isinf(d), -1, rows + self.row_lo).to(torch.int32)
                del rows
                offsets = torch.arange(b + 1, dtype=torch.int64, device=dev) * n
                self.cap_sorted_lists(offsets, ids, d, m, k, out=(out_ids[j0:j0 + b], out_d[j0:j0 + b]))
        return out_ids, out_d

    MAX_SELECT_K = 2048              # kSelMaxK of morna_select_topk
    sparse_exact = False             # set at load for a sparse index whose tie groups would overflow the tensor path's lists
    TIE_GROUP_FOR_SPARSE_PATH = 512  # (the final candidate lists hold 1024 rows; a query usually sees two or more such groups)

    def exact_search_device(self, queries, k, stream=None, allow_single=True, query_groups=None, max_per_group=None):
        """queries: CUDA float64 [nq x dim].  Returns device (ids int32 [nq x k], dists float64 [nq x k]); ids are
        global internal ids (row_lo + local row); short lists are padded with id -1 / +inf.  Like the reference's
        exact_search_nn (morna.py:681-712) any k is served: k above the number of rows returns every row, k <= 0
        an empty list.  ``query_groups`` (int32 [nq], see set_row_groups): query q leaves out the rows labelled
        query_groups[q]; the lists are the brute-force lists of the remaining rows.  ``max_per_group`` (see
        set_cap_groups): the brute-force list walked in order, a row kept iff fewer than that many rows of its cap label
        were kept before it, until k are kept."""
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.dim() == 2
        if stream is not None and stream != torch.cuda.current_stream(self.device):
            with torch.cuda.stream(stream):
                return self.exact_search_device(queries, k, allow_single=allow_single, query_groups=query_groups,
                                                max_per_group=max_per_group)
        queries = queries.contiguous()
        nq = queries.shape[0]
        q_ld = queries.shape[1]            # (a size-1 leading dimension may report stride 0)
        assert q_ld == self.dim, "queries must be [nq x dim]"
        n = self.row_hi - self.row_lo
        dev = self.device
        k = max(int(k), 0)
        out_ids = torch.full((nq, k), -1, dtype=torch.int32, device=dev)
        out_d = torch.full((nq, k), float("inf"), dtype=torch.float64, device=dev)
        k_eff = min(k, n)
        qg = self._query_groups(query_groups, nq)
        m = self._cap(max_per_group)
        if n == 0 or nq == 0 or k_eff == 0:
            return out_ids, out_d
        if m is not None:
            return self._capped_search(queries, k, qg, m)
        if nq == 1 and allow_single and k_eff <= 512 and self.csr is None and qg is None:
            return self.single_search_device(queries[0], k)
        excl = () if qg is None else self._excl_args(qg)
        with torch.cuda.device(dev):
            if k_eff > self.MAX_SELECT_K:
                return self._full_sort_search(queries, k, out_ids, out_d, qg)
            ids_k = out_ids if k_eff == k else torch.empty((nq, k_eff), dtype=torch.int32, device=dev)
            d_k = out_d if k_eff == k else torch.empty((nq, k_eff), dtype=torch.float64, device=dev)
            if self.csr is not None and bool(torch.isfinite(queries).all()):
                row_off, cols, vals, plan = self.csr
                ws = self._workspace(self.lib.morna_knn_exact_sparse_workspace_bytes(n, nq, k_eff), "sparse")
                _lib.check((self.lib.morna_knn_exact_sparse_excl if excl else self.lib.morna_knn_exact_sparse)(
                    _lib.dev_ptr(row_off), _lib.dev_ptr(cols), _lib.dev_ptr(vals), _lib.dev_ptr(plan), _lib.dev_ptr(self.pp), n,
                    self.dim, self.row_lo,
                    _lib.ptr(queries), nq, q_ld, k_eff, _lib.dev_ptr(ids_k), _lib.dev_ptr(d_k), _lib.dev_ptr(ws), ws.numel(),
                    *excl, _lib.stream_ptr()), "morna_knn_exact_sparse")
                if k_eff != k:
                    out_ids[:, :k_eff] = ids_k
                    out_d[:, :k_eff] = d_k
                return out_ids, out_d
            ws = self._workspace(self.lib.morna_knn_exact_workspace_bytes(n, nq, k_eff))
            _lib.check((self.lib.morna_knn_exact_excl if excl else self.lib.morna_knn_exact)(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, self.row_lo,
                _lib.ptr(queries), nq, q_ld, k_eff, _lib.dev_ptr(ids_k), _lib.dev_ptr(d_k),
                _lib.dev_ptr(ws), ws.numel(), *excl, _lib.stream_ptr()), "morna_knn_exact")
            if k_eff != k:
                out_ids[:, :k_eff] = ids_k
                out_d[:, :k_eff] = d_k
        return out_ids, out_d

    def _full_sort_search(self, queries, k, out_ids, out_d, qg=None):
        """k beyond the select kernel's list size (2048): all distances (morna_angular_distances, the canonical FP64
        sums) and a full device sort per query under the reference order -- rare (a user asking for thousands of
        neighbours), so the sort is torch's.  With query labels `qg`, excluded rows sit at +inf and end as padding."""
        n, dev = self.row_hi - self.row_lo, self.device
        k_eff = min(k, n)
        dist = torch.empty(n, dtype=torch.float64, device=dev)
        for j in range(queries.shape[0]):
            _lib.check(self.lib.morna_angular_distances(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, _lib.ptr(queries[j]), 1, self.dim,
                _lib.dev_ptr(dist), n, _lib.stream_ptr()), "morna_angular_distances")
            if qg is not None:
                dist.masked_fill_((self.row_group == qg[j]) & (qg[j] >= 0), float("inf"))
            # distance ascending, equal distances id descending: stable sort of the id-reversed array
            order = torch.sort(dist.flip(0), stable=True).indices[:k_eff]
            rows = (n - 1) - order
            d = dist[rows]
            out_ids[j, :k_eff] = torch.where(torch.isinf(d), -1, rows + self.row_lo).to(torch.int32)
            out_d[j, :k_eff] = d
        return out_ids, out_d

    # ------------------------------------------------------------------ batched search (tensor cores)
    BATCH_BLOCK_ROWS = 1 << 24       # rows per morna_knn_batched call (the call itself walks 131072-row blocks)

    def enable_tensor_path(self):
        """Builds the fp16 tensor-core operand of the resident rows (once)."""
        if getattr(self, "hs", None) is not None:
            return
        n, dev = self.row_hi - self.row_lo, self.device
        self.ld_h = int(self.lib.morna_tensor_operand_ld(self.dim))
        self.hs = torch.empty((max(n, 1), self.ld_h), dtype=torch.float16, device=dev)
        self.rho_max = torch.zeros(1, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            if n:                                          # (no rows: nothing to prepare, and no row pointer to pass)
                _lib.check(self.lib.morna_prepare_tensor_operand(
                    _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, _lib.dev_ptr(self.hs),
                    self.ld_h, _lib.dev_ptr(self.rho_max), _lib.stream_ptr()), "morna_prepare_tensor_operand")
        self._bws = {}
        self.last_stats = None

    def _batched_launch(self, queries, k, stream=None, phase_events=None, qg=None):
        """Enqueues morna_knn_batched for every row block; no host synchronisation.  Returns the
        per-block (b0, b1, ids, dists, overflow, stats) device tensors.  With query labels `qg`: the scoring half with
        the exclusion (each block given its slice of row_group), then the usual re-rank."""
        nq, dev = queries.shape[0], self.device
        n = self.row_hi - self.row_lo
        sid = (stream if stream is not None else torch.cuda.current_stream(dev)).cuda_stream
        parts = []
        with torch.cuda.device(dev):
            for b0 in range(0, n, self.BATCH_BLOCK_ROWS):
                b1 = min(n, b0 + self.BATCH_BLOCK_ROWS)
                out_ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
                out_d = torch.empty((nq, k), dtype=torch.float64, device=dev)
                overflow = torch.empty(nq, dtype=torch.uint8, device=dev)
                stats = torch.empty(4, dtype=torch.int32, device=dev)
                need = self.lib.morna_knn_batched_workspace_bytes(b1 - b0, nq, self.dim, k)
                ws = self._bws.get(sid)                # one workspace per stream: batches in flight do not share
                if ws is None or ws.numel() < need:
                    ws = self._bws[sid] = _lib.workspace(need, dev)
                if qg is None:
                    _lib.check(self.lib.morna_knn_batched(
                        _lib.dev_ptr(self.vectors[b0:b1]), _lib.dev_ptr(self.pp[b0:b1]), _lib.dev_ptr(self.hs[b0:b1]),
                        self.ld_h, _lib.dev_ptr(self.rho_max), b1 - b0, self.dim, self.ld, self.row_lo + b0,
                        _lib.ptr(queries), nq, self.dim, k, _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d),
                        _lib.dev_ptr(overflow), _lib.dev_ptr(stats), _lib.dev_ptr(ws), ws.numel(),
                        phase_events, _lib.stream_ptr(stream)), "morna_knn_batched")
                else:
                    _lib.check(self.lib.morna_knn_batched_score_excl(
                        _lib.dev_ptr(self.hs[b0:b1]), self.ld_h, _lib.dev_ptr(self.rho_max), b1 - b0, self.dim, self.row_lo + b0,
                        _lib.ptr(queries), nq, self.dim, k, _lib.dev_ptr(overflow), _lib.dev_ptr(stats), _lib.dev_ptr(ws),
                        ws.numel(), phase_events, None, None, *self._excl_args(qg, slice(b0, b1)), _lib.stream_ptr(stream)),
                        "morna_knn_batched_score_excl")
                    _lib.check(self.lib.morna_knn_batched_rerank(
                        _lib.dev_ptr(self.vectors[b0:b1]), _lib.dev_ptr(self.pp[b0:b1]), b1 - b0, self.dim, self.ld,
                        self.row_lo + b0, _lib.ptr(queries), nq, self.dim, k, _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d),
                        _lib.dev_ptr(overflow), _lib.dev_ptr(ws), ws.numel(), 0, _lib.stream_ptr(stream)),
                        "morna_knn_batched_rerank")
                parts.append((b0, b1, out_ids, out_d, overflow, stats))
        return parts

    def _batched_finish(self, parts, queries, k, stream=None, host_stats=None, qg=None):
        """Host half: queries whose candidate lists overflowed (ties wider than the lists) are answered
        by the exact scan, then the row blocks' lists are merged.  `host_stats`: stats already copied
        to the host, one [4] int tensor per block; otherwise they are read here (synchronises).  `qg`: the
        query labels of an excluded search (the scan then masks the same rows)."""
        from . import dist as mdist
        stats_total = torch.zeros(4, dtype=torch.int64)
        for i, (b0, b1, out_ids, out_d, overflow, stats) in enumerate(parts):
            st = host_stats[i] if host_stats is not None else stats.cpu()
            stats_total += st.to(torch.int64)
            if int(st[0]) > 0:
                idx = overflow.nonzero().flatten()
                sub = MornaSearch.__new__(MornaSearch)
                sub.__dict__.update(self.__dict__)
                sub.vectors, sub.pp = self.vectors[b0:b1], self.pp[b0:b1]
                sub.row_lo, sub.row_hi, sub._ws_pool = self.row_lo + b0, self.row_lo + b1, {}
                if (b0, b1) != (0, self.row_hi - self.row_lo):
                    sub.csr = None                          # (the CSR form covers the whole resident block)
                if qg is not None:
                    sub.row_group = self.row_group[b0:b1]
                e_ids, e_d = sub.exact_search_device(queries[idx], k, stream, allow_single=False,
                                                     query_groups=None if qg is None else qg[idx])
                out_ids[idx] = e_ids
                out_d[idx] = e_d
        self.last_stats = stats_total.tolist()
        if len(parts) == 1:
            return parts[0][2], parts[0][3]
        return mdist.merge_topk(torch.cat([p[2] for p in parts], 1), torch.cat([p[3] for p in parts], 1), k, stream)

    def batched_search_device(self, queries, k, stream=None, check_overflow=True, phase_events=None, query_groups=None,
                              max_per_group=None):
        """Same contract and same results as exact_search_device, with the N x D
        contraction on the tensor cores (fp16 first pass with a rigorous error bound,
        FP64 re-rank).  Queries whose candidate lists overflow (massive ties) are
        answered by the exact scan.  ``query_groups``: per-query exclusion, as in exact_search_device.
        ``max_per_group``: a group-capped search, as in exact_search_device (one call at a time, no phase events)."""
        from . import dist as mdist
        self.enable_tensor_path()
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.dim() == 2
        queries = queries.contiguous()
        nq = queries.shape[0]
        n = self.row_hi - self.row_lo
        assert queries.shape[1] == self.dim
        qg = self._query_groups(query_groups, nq)
        m = self._cap(max_per_group)
        if m is not None:
            with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream(self.device)):
                return self._capped_search(queries, k, qg, m)
        if n == 0 or nq == 0 or k > 512 or k <= 0 or k > n or (self.csr is not None and self.sparse_exact):
            return self.exact_search_device(queries, k, stream, query_groups=qg)   # (a sparse index: its ties would overflow every list)
        parts = self._batched_launch(queries, k, stream, phase_events, qg)
        if check_overflow:
            return self._batched_finish(parts, queries, k, stream, qg=qg)
        if len(parts) == 1:
            return parts[0][2], parts[0][3]
        return mdist.merge_topk(torch.cat([p[2] for p in parts], 1), torch.cat([p[3] for p in parts], 1), k, stream)

    # rows-sharded search: scoring up to this rank's bound on the k-th best cosine, then -- once the caller has
    # all-reduced the bounds -- final lists, re-rank and order (see dist.sharded_batched_search)
    def batched_score_bound(self, queries, k):
        """First half on this rank's rows: returns float32 [nq x k] lower bounds of the true cosines of its k best
        rows per query (-inf: nothing from this rank).  The candidate state stays in this object until
        batched_finish_bound."""
        self.enable_tensor_path()
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.dim() == 2 and queries.shape[1] == self.dim
        queries = queries.contiguous()
        nq, dev = queries.shape[0], self.device
        n = self.row_hi - self.row_lo
        bound = torch.full((nq, max(k, 1)), float("-inf"), dtype=torch.float32, device=dev)
        tensor = 0 < k <= min(n, 512) and n <= self.BATCH_BLOCK_ROWS and nq > 0
        self._bound_state = (queries, k, tensor, None)
        if not tensor:
            return bound                     # tiny shard or huge k: the exact scan answers locally, nothing to prune with
        with torch.cuda.device(dev):
            overflow = torch.empty(nq, dtype=torch.uint8, device=dev)
            stats = torch.empty(4, dtype=torch.int32, device=dev)
            need = self.lib.morna_knn_batched_workspace_bytes(n, nq, self.dim, k)
            sid = torch.cuda.current_stream(dev).cuda_stream
            ws = self._bws.get(sid)
            if ws is None or ws.numel() < need:
                ws = self._bws[sid] = _lib.workspace(need, dev)
            _lib.check(self.lib.morna_knn_batched_score(
                _lib.dev_ptr(self.hs), self.ld_h, _lib.dev_ptr(self.rho_max), n, self.dim, self.row_lo, _lib.ptr(queries), nq,
                self.dim, k, _lib.dev_ptr(overflow), _lib.dev_ptr(stats), _lib.dev_ptr(ws), ws.numel(), None, None,
                _lib.dev_ptr(bound), _lib.stream_ptr()), "morna_knn_batched_score")
        self._bound_state = (queries, k, tensor, (overflow, stats, ws))
        return bound

    def union_kth_bound(self, gathered, k):
        """gathered: float32 [lists x nq x k] (the all-gathered batched_score_bound results) -> float32 [nq], per query a
        value that at least k rows over all shards reach or exceed in true cosine."""
        lists, nq = gathered.shape[0], gathered.shape[1]
        out = torch.empty(nq, dtype=torch.float32, device=gathered.device)
        gathered = gathered.contiguous()
        with torch.cuda.device(gathered.device):
            _lib.check(self.lib.morna_union_kth_bound(_lib.dev_ptr(gathered), lists, nq, k, _lib.dev_ptr(out), _lib.stream_ptr()),
                       "morna_union_kth_bound")
        return out

    def batched_finish_bound(self, bound, check_overflow=True, out=None):
        """Second half: `bound` float32 [nq] = union_kth_bound of every rank's batched_score_bound result.  Returns this
        rank's (ids, dists), sorted under the reference order with GLOBAL ids; together the ranks' lists hold the global
        top-k (each rank re-ranks only its rows whose score can still reach the global k-th place)."""
        queries, k, tensor, st = self._bound_state
        self._bound_state = None
        if not tensor:
            ids, d = self.exact_search_device(queries, k, allow_single=False)
            if out is not None:
                out[0].copy_(ids); out[1].copy_(d)
                return out
            return ids, d
        overflow, stats, ws = st
        nq, dev = queries.shape[0], self.device
        n = self.row_hi - self.row_lo
        # `out`: caller-provided (ids int32 [nq x k], dists float64 [nq x k]) -- e.g. views of a packed send buffer
        out_ids = out[0] if out is not None else torch.empty((nq, k), dtype=torch.int32, device=dev)
        out_d = out[1] if out is not None else torch.empty((nq, k), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            _lib.check(self.lib.morna_knn_batched_finalize(n, nq, self.dim, k, _lib.dev_ptr(bound), _lib.dev_ptr(overflow),
                                                           _lib.dev_ptr(stats), _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()),
                       "morna_knn_batched_finalize")
            _lib.check(self.lib.morna_knn_batched_rerank(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, self.row_lo, _lib.ptr(queries), nq,
                self.dim, k, _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d), _lib.dev_ptr(overflow), _lib.dev_ptr(ws), ws.numel(), 0,
                _lib.stream_ptr()), "morna_knn_batched_rerank")
        parts = [(0, n, out_ids, out_d, overflow, stats)]
        if check_overflow:
            return self._batched_finish(parts, queries, k)
        return out_ids, out_d

    def search_batches(self, batches, k, depth=2, side_job=False, query_groups=None, max_per_group=None):
        """Streams query batches through the GPU: generator over ``batches`` (each a numpy or torch
        [nq x dim] float32/float64 array, or a 1-D integer array of INTERNAL IDS whose stored rows are the queries, as
        ``search -q``) yielding ``(ids, dists)`` numpy arrays in order -- the same
        results as ``exact_search_batch`` per batch.  ``depth`` batches are in flight, each on its own
        CUDA stream with its own pinned staging buffers and workspace, so batch i+1's host->device
        copy and batch i-1's device->host copy overlap batch i's kernels.
        ``query_groups`` (per-query exclusion, see set_row_groups): True -- every batch is internal ids and takes its
        labels from row_group[ids] (a stored row then never finds itself); or an iterable of int32 label arrays, one per
        batch, in step with ``batches``.  Not with ``side_job``.  ``max_per_group`` (see set_cap_groups): each batch is a
        capped batched_search_device call, one at a time (no pipelining, no graph replay)."""
        if max_per_group is not None:
            if side_job:
                raise ValueError("side_job cannot be combined with max_per_group")
            yield from self._capped_batches(batches, k, query_groups, self._cap(max_per_group))
            return
        if query_groups is not None and side_job:
            raise ValueError("side_job cannot be combined with query_groups")
        if query_groups is not None and self.row_group is None:
            raise ValueError("query_groups need row labels: call set_row_groups first")
        pipes = self.__dict__.setdefault("_pipes", {})
        pipe = pipes.get((k, depth))           # slots (streams, pinned buffers, workspaces) are kept between calls
        if pipe is None or pipe.head != pipe.tail or pipe.side_job != (bool(side_job) and depth > 1):
            pipe = pipes[(k, depth)] = BatchPipeline(self, k, depth, side_job)
        labels = iter(query_groups) if query_groups is not None and query_groups is not True else None
        pending = 0
        for q in batches:
            if pending == depth:
                yield pipe.collect()
                pending -= 1
            pipe.submit(q, query_groups=next(labels) if labels is not None else query_groups)
            pending += 1
        while pending:
            yield pipe.collect()
            pending -= 1

    def _capped_batches(self, batches, k, query_groups, m):
        if query_groups is not None and self.row_group is None:
            raise ValueError("query_groups need row labels: call set_row_groups first")
        labels = iter(query_groups) if query_groups is not None and query_groups is not True else None
        for q in batches:
            t = torch.from_numpy(np.ascontiguousarray(q)) if isinstance(q, np.ndarray) else q
            by_id = t.dim() == 1 and t.dtype in (torch.int32, torch.int64)
            if query_groups is True and not by_id:
                raise ValueError("query_groups=True needs a batch of internal ids")
            if by_id:
                if t.numel():
                    lo, hi = (int(v) for v in (t.min(), t.max()))
                    if lo < self.row_lo or hi >= self.row_hi:
                        raise ValueError("internal ids %d..%d are not all resident on this shard (rows %d..%d)"
                                         % (lo, hi, self.row_lo, self.row_hi - 1))
                rows = t.to(self.device).long() - self.row_lo
                qd = self.vectors[rows, :self.dim].to(torch.float64).contiguous()
            else:
                qd = t.to(self.device).to(torch.float64).contiguous()
            qg = self.row_group[rows] if query_groups is True else next(labels) if labels is not None else None
            ids, d = self.batched_search_device(qd, k, query_groups=qg, max_per_group=m)
            yield ids.cpu().numpy(), d.cpu().numpy()

    def _single_query_host(self, query, k):
        """One host query through the single-query kernel with persistent pinned staging: one host->device copy (the
        query), one launch, one device->host copy (distances, ids and the fallback flag packed in one buffer), one stream
        synchronisation.  Returns numpy (ids [1 x k], dists [1 x k]) or None when the generic path must answer."""
        n, dev = self.row_hi - self.row_lo, self.device
        if n == 0 or k <= 0 or min(k, n) > 512 or self.csr is not None:
            return None
        state = self.__dict__.setdefault("_single_host", {})
        st = state.get(k)
        with torch.cuda.device(dev):
            if st is None:
                nbytes = 8 * k + 4 * k + 8
                st = state[k] = {"h_q": torch.empty(self.dim, dtype=torch.float64).pin_memory(),
                                 "d_q": torch.empty(self.dim, dtype=torch.float64, device=dev),
                                 "d_out": torch.zeros(nbytes, dtype=torch.uint8, device=dev),
                                 "h_out": torch.empty(nbytes, dtype=torch.uint8).pin_memory()}
            st["h_q"].numpy()[:] = query
            st["d_q"].copy_(st["h_q"], non_blocking=True)
            d_out = st["d_out"]
            dist_v, ids_v, flag_v = d_out[:8 * k].view(torch.float64), d_out[8 * k:12 * k].view(torch.int32), d_out[12 * k:12 * k + 4].view(torch.int32)
            k_eff = min(k, n)
            if k_eff < k:
                ids_v.fill_(-1); dist_v.fill_(float("inf"))
            sws = self._workspace(self.lib.morna_knn_single_workspace_bytes(n), "single")
            _lib.check(self.lib.morna_knn_single(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, self.row_lo, _lib.dev_ptr(st["d_q"]), k_eff,
                _lib.dev_ptr(ids_v), _lib.dev_ptr(dist_v), _lib.dev_ptr(flag_v), _lib.dev_ptr(sws), sws.numel(), _lib.stream_ptr()),
                "morna_knn_single")
            st["h_out"].copy_(d_out, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        out = st["h_out"].numpy()
        if int(out[12 * k:12 * k + 4].view(np.int32)[0]):
            return None
        return out[8 * k:12 * k].view(np.int32).reshape(1, k).copy(), out[:8 * k].view(np.float64).reshape(1, k).copy()

    def exact_search_batch(self, queries, k, tensor_cores=None, query_groups=None, max_per_group=None):
        """Host entry: queries numpy [nq x dim] (float32 or float64) -> numpy (ids, dists).
        float32 queries cross PCIe as float32 and are widened (exactly) on the device.  Batches of 64+
        queries use the tensor-core path, which returns the same bits as the scan.  ``query_groups``: per-query
        exclusion, ``max_per_group``: a group-capped search, as in exact_search_device."""
        queries = np.ascontiguousarray(queries)
        if queries.dtype != np.float32:
            queries = queries.astype(np.float64, copy=False)
        if max_per_group is not None:
            self._cap(max_per_group)
        if queries.shape[0] == 1 and not tensor_cores and query_groups is None and max_per_group is None:
            got = self._single_query_host(queries[0], k)
            if got is not None:
                return got
        q = torch.from_numpy(queries)
        if q.numel():
            q = q.pin_memory()
        qd = q.to(self.device, non_blocking=True).to(torch.float64)
        if tensor_cores is None:
            tensor_cores = qd.shape[0] >= 64
        ids, d = (self.batched_search_device if tensor_cores else self.exact_search_device)(qd, k, query_groups=query_groups,
                                                                                            max_per_group=max_per_group)
        return ids.cpu().numpy(), d.cpu().numpy()

    def exact_search_nn(self, num_neighbors, include_distances=True, meta_db=False, query_groups=None, max_per_group=None):
        """morna.py:681-730 for the current ``query_sample``; ``query_groups``: its label ([1]), ``max_per_group``: a
        group-capped search, as in exact_search_device."""
        ids, d = self.exact_search_batch(np.asarray(self.query_sample, dtype=np.float64)[None, :], num_neighbors,
                                         query_groups=query_groups, max_per_group=max_per_group)
        keep = ids[0] >= 0
        results = (ids[0][keep].tolist(),)
        if include_distances:
            results += (d[0][keep].tolist(),)
        if meta_db:
            results += (self._metadata(results[0]),)
        return results

    # ------------------------------------------------------------------ approximate mode
    def approx_search_device(self, queries, k, query_groups=None, max_per_group=None):
        """The k best rows by fp16 tensor-core score, no exact re-rank (morna_knn_batched_approx): the approximate mode
        that stands where the reference asks Annoy (morna.py:632-678).  Same contract as batched_search_device; queries
        whose lists overflow, tiny shards and sparse indexes are answered exactly.  There is no per-query exclusion in
        this mode, nor a cap: ``query_groups`` and ``max_per_group`` raise ValueError."""
        if query_groups is not None:
            raise ValueError("the approximate mode has no per-query exclusion; use an exact search")
        if max_per_group is not None:
            raise ValueError("the approximate mode has no cap per group; use an exact search")
        self.enable_tensor_path()
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.dim() == 2 and queries.shape[1] == self.dim
        queries = queries.contiguous()
        nq, dev = queries.shape[0], self.device
        n = self.row_hi - self.row_lo
        if n == 0 or nq == 0 or k > 512 or k <= 0 or k > n or n > self.BATCH_BLOCK_ROWS or (self.csr is not None and self.sparse_exact):
            return self.exact_search_device(queries, k)
        with torch.cuda.device(dev):
            out_ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
            out_d = torch.empty((nq, k), dtype=torch.float64, device=dev)
            overflow = torch.empty(nq, dtype=torch.uint8, device=dev)
            stats = torch.empty(4, dtype=torch.int32, device=dev)
            need = self.lib.morna_knn_batched_workspace_bytes(n, nq, self.dim, k)
            sid = torch.cuda.current_stream(dev).cuda_stream
            ws = self._bws.get(sid)
            if ws is None or ws.numel() < need:
                ws = self._bws[sid] = _lib.workspace(need, dev)
            _lib.check(self.lib.morna_knn_batched_approx(
                _lib.dev_ptr(self.hs), self.ld_h, _lib.dev_ptr(self.rho_max), n, self.dim, self.row_lo, _lib.ptr(queries), nq,
                self.dim, k, _lib.dev_ptr(out_ids), _lib.dev_ptr(out_d), _lib.dev_ptr(overflow), _lib.dev_ptr(stats),
                _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_knn_batched_approx")
        return self._batched_finish([(0, n, out_ids, out_d, overflow, stats)], queries, k)

    def search_nn(self, num_neighbors, search_k=None, include_distances=True, meta_db=False, max_per_group=None):
        """morna.py:632-678 for the current ``query_sample``: the reference's default (approximate) mode.  Annoy's
        forest is not rebuilt here; the approximate answer is the tensor-core pass without the exact re-rank
        (``search_k`` has no counterpart and is ignored).  ``exact_search_nn`` (-e) is the exact mode.  There is no cap
        per group in this mode: ``max_per_group`` raises ValueError."""
        if max_per_group is not None:
            raise ValueError("the approximate mode has no cap per group; use an exact search")
        q = torch.tensor(self.query_sample, dtype=torch.float64)[None, :].to(self.device)
        ids, d = self.approx_search_device(q, num_neighbors)
        ids, d = ids.cpu().numpy(), d.cpu().numpy()
        keep = ids[0] >= 0
        results = (ids[0][keep].tolist(),)
        if include_distances:
            results += (d[0][keep].tolist(),)
        if meta_db:
            results += (self._metadata(results[0]),)
        return results

    def search_member_n(self, query_id, num_neighbors, search_k=None, include_distances=True,
                        meta_db=False, out=None, max_distance=None, exclude=False, max_per_group=None):
        """morna.py:733-787 with the stored row as the query (float32 values), run
        through the exact scan.  With ``max_distance``: every sample within it (range_search_nn), the first
        ``num_neighbors`` of them when that is not None.  ``exclude``: the query takes its row's label (set_row_groups),
        so its own sample and every sample of its group are left out.  ``max_per_group``: at most that many results per
        cap label (set_cap_groups)."""
        internal_id = _member_internal_id(self.internal_id_map, query_id, out)
        if not (self.row_lo <= internal_id < self.row_hi):
            raise ValueError("internal id %d is not resident on this shard" % internal_id)
        self.query_sample = self.vectors[internal_id - self.row_lo, :self.dim].to(torch.float64).cpu().tolist()
        qg = None
        if exclude:
            if self.row_group is None:
                raise ValueError("exclude needs row labels: call set_row_groups first")
            qg = self.row_group[internal_id - self.row_lo:internal_id - self.row_lo + 1]
        if max_distance is not None:
            return self.range_search_nn(max_distance, include_distances, meta_db, num_neighbors, query_groups=qg,
                                        max_per_group=max_per_group)
        return self.exact_search_nn(num_neighbors, include_distances, meta_db, query_groups=qg, max_per_group=max_per_group)

    def _metadata(self, internal_ids):
        """morna.py:666-676: keywords of every result's sample id from basename.meta.mor."""
        return files.read_meta(self.basename, [self.inverse_lookup(iid) for iid in internal_ids])

    def subset(self, internal_ids, keep_parent_rows=True):
        """A search over only the rows of these internal ids (any order, repeats allowed; resident on this object): a
        FilteredSearch whose results carry this object's internal ids.  ``keep_parent_rows=False``: the result does not
        hold this object's device rows, so dropping this object frees them; queries by internal id must then name rows of
        the subset."""
        return FilteredSearch(self, internal_ids, keep_parent_rows)

    # ------------------------------------------------------------------ range search
    RANGE_BATCH_QUERIES = 4096        # queries per morna_range_batched call (its candidate lists: 4096 x 4096 entries)
    RANGE_TENSOR_MIN_QUERIES = 64     # smaller batches go to the FP64 scan, as top-k batches do

    def range_search_device(self, queries, max_distance, query_groups=None, max_per_group=None):
        """Every row within ``max_distance`` of each query: queries CUDA float64 [nq x dim] -> device CSR (offsets int64
        [nq+1], ids int32 [total], dists float64 [total]); query j's list is ids/dists[offsets[j]:offsets[j+1]], ordered as
        the reference orders results (distance ascending, equal distances id descending), ids global.  The distance is
        exactly exact_search_device's and the comparison inclusive; a query with nothing in range has an empty list.
        Sets ``last_stats`` = [overflowed queries, first-pass survivors, matches] and ``last_range_route`` ("tensor":
        the tensor-core filter with an FP64 check, overflowed queries answered by the scan; "exact": the FP64 scan).
        ``query_groups``: per-query exclusion, as in exact_search_device.  ``max_per_group`` (see set_cap_groups): each
        list walked in its order, an entry kept iff fewer than that many entries of its cap label were kept before it."""
        return concat_range_groups(list(self.range_search_groups(queries, max_distance, query_groups=query_groups,
                                                                 max_per_group=max_per_group)), self.device)

    def range_search_groups(self, queries, max_distance, byte_cap=None, query_groups=None, max_per_group=None):
        """Generator over (lo, hi, offsets, ids, dists): the range_search_device CSR of queries [lo, hi), in query order.
        Batches of RANGE_BATCH_QUERIES are counted first (one small read back); with ``byte_cap``, a batch whose lists
        would take more than that many bytes (12 per match) is emitted in groups of consecutive queries that fit it (one
        query per group at least), so no more than that is allocated at once.  With ``max_per_group`` each group's lists are then walked
        (cap_sorted_lists); the byte cap applies to the lists before the walk."""
        m = self._cap(max_per_group)
        for b0, st in self.range_count_batches(queries, max_distance, query_groups):
            for lo, hi in _range_groups(st["counts"], byte_cap):
                off, ids, d = self.range_emit(st, lo, hi)
                if m is not None:
                    off, ids, d = self.cap_sorted_lists(off, ids, d, m)
                yield b0 + lo, b0 + hi, off, ids, d

    def range_count_batches(self, queries, max_distance, query_groups=None):
        """The counting half of range_search_groups: generator over (b0, st), one per batch of RANGE_BATCH_QUERIES
        queries starting at query b0, where st["counts"] (host int64) holds the batch's matches per query and st is what
        range_emit needs to write any run of its lists.  Updates last_range_route and last_stats as the batches go."""
        r = check_radius(max_distance)
        assert queries.is_cuda and queries.dtype == torch.float64 and queries.dim() == 2 and queries.shape[1] == self.dim
        queries = queries.contiguous()
        nq = queries.shape[0]
        qg = self._query_groups(query_groups, nq)
        route = self._range_route(nq)
        stats = [0, 0, 0]
        self.last_range_route, self.last_stats = route, list(stats)
        for b0 in range(0, nq, self.RANGE_BATCH_QUERIES):
            st = self._range_counts(queries[b0:b0 + self.RANGE_BATCH_QUERIES], r, route,
                                    None if qg is None else qg[b0:b0 + self.RANGE_BATCH_QUERIES])
            stats = [a + b for a, b in zip(stats, st["stats"])]
            self.last_stats = list(stats)
            yield b0, st

    def range_search_batch(self, queries, max_distance, query_groups=None, max_per_group=None):
        """Host entry: queries numpy [nq x dim] -> numpy CSR (offsets, ids, dists) of range_search_device."""
        queries = np.ascontiguousarray(queries)
        if queries.dtype != np.float32:
            queries = queries.astype(np.float64, copy=False)
        q = torch.from_numpy(queries)
        if q.numel():
            q = q.pin_memory()
        qd = q.to(self.device, non_blocking=True).to(torch.float64)
        return tuple(t.cpu().numpy() for t in self.range_search_device(qd, max_distance, query_groups, max_per_group))

    def range_search_nn(self, max_distance, include_distances=True, meta_db=False, num_neighbors=None, query_groups=None,
                        max_per_group=None):
        """Every indexed sample within ``max_distance`` of the current ``query_sample``, as exact_search_nn returns its
        results; ``num_neighbors``: keep only the first that many (after the cap, with ``max_per_group``)."""
        _, ids, d = self.range_search_batch(np.asarray(self.query_sample, dtype=np.float64)[None, :], max_distance,
                                            query_groups, max_per_group)
        if num_neighbors is not None:
            ids, d = ids[:max(int(num_neighbors), 0)], d[:max(int(num_neighbors), 0)]
        results = (ids.tolist(),)
        if include_distances:
            results += (d.tolist(),)
        if meta_db:
            results += (self._metadata(results[0]),)
        return results

    def _range_route(self, nq):
        n = self.row_hi - self.row_lo
        sparse_ties = self.csr is not None and self.sparse_exact         # its parallel rows would overflow every list
        tensor = 0 < n <= self.BATCH_BLOCK_ROWS and nq >= self.RANGE_TENSOR_MIN_QUERIES and not sparse_ties
        return "tensor" if tensor else "exact"

    def _range_counts(self, queries, r, route, qg=None):
        """Matches per query of one batch (host int64) and what range_emit needs; on the tensor route the counts,
        overflow flags and stats come back in one copy, and overflowed queries are counted again by the scan."""
        nq, n, dev = queries.shape[0], self.row_hi - self.row_lo, self.device
        st = {"queries": queries, "r": r, "route": route, "over": np.zeros(0, np.int64), "stats": [0, 0, 0],
              "counts": np.zeros(nq, np.int64), "qg": qg}
        if n == 0 or nq == 0:
            return st
        excl = () if qg is None else self._excl_args(qg)
        with torch.cuda.device(dev):
            if route == "exact":
                st["counts"] = self._range_exact_counts(queries, r, qg)
            else:
                self.enable_tensor_path()
                counts = torch.empty(nq, dtype=torch.int32, device=dev)
                overflow = torch.empty(nq, dtype=torch.uint8, device=dev)
                stats = torch.empty(4, dtype=torch.int64, device=dev)
                ws = self._workspace(self.lib.morna_range_batched_workspace_bytes(n, nq, self.dim), "range")
                _lib.check((self.lib.morna_range_batched_excl if excl else self.lib.morna_range_batched)(
                    _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), _lib.dev_ptr(self.hs), self.ld_h, _lib.dev_ptr(self.rho_max),
                    n, self.dim, self.ld, self.row_lo, _lib.ptr(queries), nq, self.dim, r, _lib.dev_ptr(counts),
                    _lib.dev_ptr(overflow), _lib.dev_ptr(stats), _lib.dev_ptr(ws), ws.numel(), *excl, _lib.stream_ptr()),
                    "morna_range_batched")
                host = torch.cat([counts.to(torch.int64), overflow.to(torch.int64), stats]).cpu().numpy()
                c, over = host[:nq].copy(), np.nonzero(host[nq:2 * nq])[0]
                if len(over):
                    over_dev = torch.from_numpy(over).to(dev)
                    c[over] = self._range_exact_counts(queries[over_dev], r, None if qg is None else qg[over_dev])
                st.update(counts=c, over=over, ws=ws, overflow=overflow)
                st["stats"] = [int(host[2 * nq]), int(host[2 * nq + 1]), 0]
        st["stats"][2] = int(st["counts"].sum())
        return st

    def _range_exact_counts(self, queries, r, qg=None):
        nq, n = queries.shape[0], self.row_hi - self.row_lo
        counts = torch.empty(nq, dtype=torch.int32, device=self.device)
        ws = self._workspace(self.lib.morna_range_exact_workspace_bytes(n, nq, 0), "range_exact")
        excl = () if qg is None else self._excl_args(qg)
        _lib.check((self.lib.morna_range_exact_count_excl if excl else self.lib.morna_range_exact_count)(
            _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, _lib.ptr(queries), nq, self.dim, r,
            _lib.dev_ptr(counts), _lib.dev_ptr(ws), ws.numel(), *excl, _lib.stream_ptr()), "morna_range_exact_count")
        return counts.cpu().numpy().astype(np.int64)

    def _range_exact_fill(self, queries, r, counts, qg=None):
        """FP64 route's lists of `queries` given their counts: device (offsets, ids, dists)."""
        nq, n, dev = queries.shape[0], self.row_hi - self.row_lo, self.device
        off = np.zeros(nq + 1, dtype=np.int64)
        np.cumsum(counts, out=off[1:])
        total = int(off[-1])
        offsets = torch.from_numpy(off).to(dev)
        ids = torch.empty(total, dtype=torch.int32, device=dev)
        d = torch.empty(total, dtype=torch.float64, device=dev)
        if total:
            ws = self._workspace(self.lib.morna_range_exact_workspace_bytes(n, nq, total), "range_exact")
            excl = () if qg is None else self._excl_args(qg)
            _lib.check((self.lib.morna_range_exact_fill_excl if excl else self.lib.morna_range_exact_fill)(
                _lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), n, self.dim, self.ld, self.row_lo, _lib.ptr(queries), nq,
                self.dim, r, _lib.dev_ptr(offsets), total, _lib.dev_ptr(ids), _lib.dev_ptr(d), _lib.dev_ptr(ws), ws.numel(),
                *excl, _lib.stream_ptr()), "morna_range_exact_fill")
        return offsets, ids, d

    def range_emit(self, st, lo, hi):
        """Device CSR (offsets [hi - lo + 1] from 0, ids, dists) of queries [lo, hi) of a batch range_count_batches
        counted."""
        dev, n = self.device, self.row_hi - self.row_lo
        with torch.cuda.device(dev):
            qg = st["qg"]
            if st["route"] == "exact" or n == 0:
                return self._range_exact_fill(st["queries"][lo:hi], st["r"], st["counts"][lo:hi], None if qg is None else qg[lo:hi])
            nq = st["queries"].shape[0]
            counts = st["counts"]
            full = np.zeros(nq + 1, dtype=np.int64)              # queries outside [lo, hi) get empty ranges
            np.cumsum(counts[lo:hi], out=full[lo + 1:hi + 1])
            full[hi + 1:] = full[hi]
            total = int(full[hi])
            offsets = torch.from_numpy(full).to(dev)
            ids = torch.empty(total, dtype=torch.int32, device=dev)
            d = torch.empty(total, dtype=torch.float64, device=dev)
            if total:
                ws = st["ws"]
                _lib.check(self.lib.morna_range_batched_emit(
                    n, nq, self.dim, _lib.dev_ptr(offsets), _lib.dev_ptr(st["overflow"]), _lib.dev_ptr(ids), _lib.dev_ptr(d),
                    _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_range_batched_emit")
            over = st["over"][(st["over"] >= lo) & (st["over"] < hi)]
            if len(over):                                        # the scan's lists spliced into their places
                over_dev = torch.from_numpy(over).to(dev)
                sub_off, sub_ids, sub_d = self._range_exact_fill(st["queries"][over_dev], st["r"], counts[over],
                                                                 None if qg is None else qg[over_dev])
                sub_total = sub_ids.numel()
                if sub_total:
                    lens = torch.from_numpy(counts[over]).to(dev)
                    shift = offsets[torch.from_numpy(over).to(dev)] - sub_off[:-1]
                    dst = torch.repeat_interleave(shift, lens, output_size=sub_total) + torch.arange(sub_total, device=dev)
                    ids[dst] = sub_ids
                    d[dst] = sub_d
            return offsets[lo:hi + 1], ids, d

    # ------------------------------------------------------------------ within-group search
    # The queries of one group in one call take the grouped FP64 route (morna_within_group_*) when the group has at most
    # WITHIN_SEGMENT_ROWS rows (the selection's shared-memory sort) and (queries x rows) is at most WITHIN_GROUPED_MAX_PAIRS;
    # otherwise the tensor-core path searches the group as a row range of the grouped copy (_within_copy).  The grouped
    # route costs about the same per (query, row) pair whatever the group, the tensor-core route a fixed cost per group
    # and call and far less per pair, so the crossing is a pair count.  The sweep of profiles/r10_within_group.log (B200,
    # top-20) puts it near 250,000 pairs for contiguous and scattered groups alike: grouped faster at 65,000 / 85,000
    # pairs (2.6 vs 7.5, 17.4 vs 44.3 ms per 4096 queries), slower at 262,000 / 341,000 (4.5 vs 4.1, 32.5 vs 23.2).
    WITHIN_SEGMENT_ROWS = 8192
    WITHIN_GROUPED_MAX_PAIRS = 250000
    WITHIN_QB = 8                    # queries per work item (kWithinQB of search_within.cu)
    WITHIN_CHUNK_ROWS = 128          # rows per work item
    WITHIN_SCRATCH_ENTRIES = 1 << 25 # distances of one grouped call (256 MB)

    def _within_layout(self):
        """The rows sorted by (label, id), labels < 0 left out: (device int32 local rows, host labels ascending, host
        starts, host counts, {"copy": _within_copy's index once built}).  Cached until set_row_groups."""
        st = self.__dict__.get("_within")
        if st is not None:
            return st
        if self.row_group is None:
            raise ValueError("a within-group search needs row labels: call set_row_groups first")
        g = self.row_group.long()
        order = torch.sort(g, stable=True).indices
        keep = g[order] >= 0
        rows = order[keep].to(torch.int32).contiguous()
        labels, counts = torch.unique(g[order][keep], return_counts=True)
        labels, counts = labels.cpu().numpy(), counts.cpu().numpy().astype(np.int64)
        starts = np.zeros(len(counts), np.int64)
        np.cumsum(counts[:-1], out=starts[1:])
        if rows.numel() == 0:
            rows = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._within = st = (rows, labels, starts, counts, {})
        return st

    def _within_queries(self, queries):
        """(device float64 [nq x dim] or None, device int64 local rows or None): the queries as vectors or stored rows."""
        t = torch.from_numpy(np.ascontiguousarray(queries)) if isinstance(queries, np.ndarray) else torch.as_tensor(queries)
        if t.dim() == 1 and t.dtype in (torch.int32, torch.int64):
            if t.numel():
                lo, hi = (int(v) for v in (torch.aminmax(t) if t.is_cuda else (t.min(), t.max())))
                if lo < self.row_lo or hi >= self.row_hi:
                    raise ValueError("internal ids %d..%d are not all resident (rows %d..%d)"
                                     % (lo, hi, self.row_lo, self.row_hi - 1))
            return None, t.to(self.device).long() - self.row_lo
        assert t.is_cuda and t.dtype == torch.float64 and t.dim() == 2 and t.shape[1] == self.dim, \
            "queries must be CUDA float64 [nq x dim] or 1-D internal ids"
        return t, None

    def _within_plan(self, queries, query_groups, exclude_rows):
        """Per query (host): group index, row count of its group and local excluded row (-1: none)."""
        rows, labels, starts, counts, _ = self._within_layout()
        vecs, qrows = self._within_queries(queries)
        nq = qrows.numel() if qrows is not None else vecs.shape[0]
        qg = torch.as_tensor(query_groups).cpu().numpy().astype(np.int64).reshape(-1)
        if qg.shape != (nq,):
            raise ValueError("query_groups must hold one label per query (%d), got %d" % (nq, qg.size))
        gi = np.minimum(np.searchsorted(labels, qg), max(len(labels) - 1, 0))
        present = (qg >= 0) & (labels[gi] == qg) if len(labels) else np.zeros(nq, bool)
        size = np.where(present, counts[gi] if len(labels) else 0, 0)
        in_call = np.bincount(gi[present], minlength=len(labels))[gi] if len(labels) else size
        grouped = present & (size <= self.WITHIN_SEGMENT_ROWS) & (size * in_call <= self.WITHIN_GROUPED_MAX_PAIRS)
        excl = np.full(nq, -1, np.int64)
        if exclude_rows is not None:
            e = torch.as_tensor(exclude_rows).cpu().numpy().astype(np.int64).reshape(-1)
            if e.shape != (nq,):
                raise ValueError("exclude_rows must hold one internal id per query (%d), got %d" % (nq, e.size))
            inside = (e >= self.row_lo) & (e < self.row_hi)
            excl[inside] = e[inside] - self.row_lo
        self.last_within_routes = (int(grouped.sum()), int((present & ~grouped).sum()))
        return {"vecs": vecs, "qrows": qrows, "nq": nq, "gi": gi, "size": size, "excl": excl,
                "grouped": np.nonzero(grouped)[0], "large": np.nonzero(present & ~grouped)[0]}

    def _within_rows(self, plan, idx):
        """Float64 device query vectors of queries idx (host int64), in that order."""
        if plan["qrows"] is not None:
            return self.vectors[plan["qrows"][torch.from_numpy(idx).to(self.device)], :self.dim].to(torch.float64).contiguous()
        return plan["vecs"][torch.from_numpy(idx).to(self.device)].contiguous()

    def _within_grouped_calls(self, plan, slots):
        """Generator over the grouped route's calls: (kwargs of morna_within_group_*, original query indices).  The
        grouped queries are sorted stably by group and cut where the summed segment lengths would pass the scratch
        budget; each call's work items are tiles of up to WITHIN_QB queries of one group x chunks of its rows.  `slots`:
        "query" -- out_slot is the query's index in the whole call, "local" -- its index in this grouped call."""
        rows, labels, starts, counts, _ = self._within_layout()
        idx = plan["grouped"]
        idx = idx[np.argsort(plan["gi"][idx], kind="stable")]
        lens = plan["size"][idx]
        cum = np.cumsum(lens)
        a, dev, QB, CH = 0, self.device, self.WITHIN_QB, self.WITHIN_CHUNK_ROWS
        while a < len(idx):
            b = max(a + 1, int(np.searchsorted(cum, (cum[a - 1] if a else 0) + self.WITHIN_SCRATCH_ENTRIES, side="right")))
            o, g, ln = idx[a:b], plan["gi"][idx[a:b]], lens[a:b]
            n = b - a
            seg_off = np.zeros(n + 1, np.int64)
            np.cumsum(ln, out=seg_off[1:])
            pos = np.arange(n)
            head_run = np.r_[True, g[1:] != g[:-1]]
            run_start = np.maximum.accumulate(np.where(head_run, pos, 0))
            run_end = np.r_[np.nonzero(head_run)[0][1:], n][np.cumsum(head_run) - 1]
            t0 = np.nonzero((pos - run_start) % QB == 0)[0]
            qn = np.minimum(QB, run_end[t0] - t0)
            nch = (ln[t0] + CH - 1) // CH
            rep = np.repeat(np.arange(len(t0)), nch)
            c = np.arange(rep.size) - np.repeat(np.cumsum(nch) - nch, nch)
            items = np.stack([t0[rep], qn[rep], starts[g[t0]][rep] + c * CH, np.minimum(CH, ln[t0][rep] - c * CH)], 1)
            up = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x, dtype=dt)).to(dev)
            excl = plan["excl"][o]
            yield {"queries": self._within_rows(plan, o), "items": up(items, np.int32), "seg_off": up(seg_off, np.int64),
                   "total": int(seg_off[-1]), "row_begin": up(starts[g], np.int32), "max_segment": int(ln.max()),
                   "exclude": up(excl, np.int32) if (excl >= 0).any() else None,
                   "out_slot": up(o if slots == "query" else pos, np.int32)}, o
            a = b

    def _within_call_args(self, c):
        rows = self._within_layout()[0]
        return (_lib.dev_ptr(self.vectors), _lib.dev_ptr(self.pp), self.row_hi - self.row_lo, self.dim, self.ld), \
               (_lib.dev_ptr(rows), _lib.ptr(c["queries"]), c["queries"].shape[0], self.dim, _lib.dev_ptr(c["items"]),
                c["items"].shape[0], _lib.dev_ptr(c["seg_off"]), c["total"], _lib.dev_ptr(c["row_begin"]), c["max_segment"],
                _lib.dev_ptr(c["exclude"]), _lib.dev_ptr(c["out_slot"]))

    def _within_copy(self):
        """Every labelled row copied once in the layout's order, so that each group is a contiguous row range, with its
        norms and fp16 tensor-core operand; row i carries as exclusion label its position within its group.  Built on
        the first call that sends a group to the tensor-core route and kept until set_row_groups: one more copy of the
        labelled rows (and their fp16 operand) instead of a sub-index per group and call."""
        rows, labels, starts, counts, cache = self._within_layout()
        cp = cache.get("copy")
        if cp is None:
            m = int(counts.sum())
            r = rows[:m].long()
            cp = MornaSearch.__new__(MornaSearch)
            cp.lib, cp.device, cp.basename, cp.dim, cp.ld = self.lib, self.device, self.basename, self.dim, self.ld
            cp.sample_count, cp.index_size = self.sample_count, m
            cp.sample_frequencies, cp.internal_id_map = self.sample_frequencies, self.internal_id_map
            cp.row_lo, cp.row_hi = 0, m
            cp.vectors, cp.pp = self.vectors.index_select(0, r), self.pp.index_select(0, r)
            cp.csr = None                      # (a sparse index's tie groups only overflow to the exact scan here)
            first = torch.from_numpy(np.repeat(starts, counts)).to(self.device)
            cp.row_group = (torch.arange(m, device=self.device) - first).to(torch.int32)
            cp.query, cp.query_sample = defaultdict(int), [0.0] * self.dim
            cp.enable_tensor_path()
            cache["copy"] = cp
        return cp

    def _within_large(self, plan):
        """Generator over the tensor-core route, one group at a time: (search, queries idx (host), their float64 queries,
        exclusion labels or None, local -> internal id map).  The search is the group's row range of _within_copy (a view:
        its rows, norms and fp16 operand sliced, ids local to the range and ascending with the internal ids); an excluded
        row is the existing per-query exclusion on it, the query labelled with that row's position in the group."""
        rows, labels, starts, counts, _ = self._within_layout()
        idx = plan["large"]
        if not len(idx):
            return
        cp = self._within_copy()
        for gval in np.unique(plan["gi"][idx]).tolist():
            sel = idx[plan["gi"][idx] == gval]
            a, L = int(starts[gval]), int(counts[gval])
            view = MornaSearch.__new__(MornaSearch)
            view.__dict__.update(cp.__dict__)
            view.vectors, view.pp, view.hs = cp.vectors[a:a + L], cp.pp[a:a + L], cp.hs[a:a + L]
            view.row_group, view.row_lo, view.row_hi = cp.row_group[a:a + L], 0, L
            view._ws_pool = {}                 # (the single-query workspace is laid out for one row count)
            member = rows[a:a + L]
            excl = plan["excl"][sel]
            qlab = None
            if (excl >= 0).any():
                m = member.cpu().numpy()
                at = np.minimum(np.searchsorted(m, excl), L - 1)
                qlab = torch.from_numpy(np.where((excl >= 0) & (m[at] == excl), at, -1).astype(np.int32)).to(self.device)
            yield view, sel, self._within_rows(plan, sel), qlab, member

    def _within_ids(self, ids, member):
        """Ids local to a group's row range -> internal ids; -1 padding stays."""
        return torch.where(ids >= 0, member[ids.long().clamp(min=0)] + self.row_lo, ids).to(torch.int32)

    def within_group_search(self, queries, k, query_groups, exclude_rows=None):
        """Top-k within each query's own group: the brute-force answer over the rows labelled query_groups[q] (labels of
        set_row_groups; a row labelled < 0 is in no group), without the row exclude_rows[q] (an internal id; -1: none).
        ``queries``: CUDA float64 [nq x dim], or 1-D internal ids whose stored rows are the queries (as ``search -q``).
        ``query_groups``: int32 [nq]; a label < 0 or one no row carries gives an empty list.  Returns device (ids int32
        [nq x k], dists float64 [nq x k]) in the reference order, ids global, padded with -1 / +inf.  A group's queries
        take the grouped FP64 route or the tensor-core route over the group's rows (see WITHIN_GROUPED_MAX_PAIRS); both
        give the brute-force bits.  Sets ``last_within_routes`` = (queries on the grouped route, on the tensor-core
        route)."""
        plan = self._within_plan(queries, query_groups, exclude_rows)
        nq, dev, k = plan["nq"], self.device, max(int(k), 0)
        out_ids = torch.full((nq, k), -1, dtype=torch.int32, device=dev)
        out_d = torch.full((nq, k), float("inf"), dtype=torch.float64, device=dev)
        if nq == 0 or k == 0:
            return out_ids, out_d
        with torch.cuda.device(dev):
            for c, _ in self._within_grouped_calls(plan, "query"):
                ws = self._workspace(self.lib.morna_within_group_workspace_bytes(c["total"]), "within")
                head, tail = self._within_call_args(c)
                _lib.check(self.lib.morna_within_group_topk(*head, self.row_lo, *tail, k, _lib.dev_ptr(out_ids),
                                                            _lib.dev_ptr(out_d), _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()),
                           "morna_within_group_topk")
            for view, sel, q, qlab, member in self._within_large(plan):
                ids, d = view.batched_search_device(q, k, query_groups=qlab)
                at = torch.from_numpy(sel).to(dev)
                out_ids[at] = self._within_ids(ids, member)
                out_d[at] = d
        return out_ids, out_d

    def within_group_range(self, queries, max_distance, query_groups, exclude_rows=None):
        """Every row of each query's own group within ``max_distance``: the within_group_search rows (same arguments),
        as the device CSR (offsets int64 [nq+1], ids int32, dists float64) that range_search_device returns."""
        r = check_radius(max_distance)
        plan = self._within_plan(queries, query_groups, exclude_rows)
        nq, dev = plan["nq"], self.device
        pieces = []
        with torch.cuda.device(dev):
            for c, o in self._within_grouped_calls(plan, "local"):
                ws = self._workspace(self.lib.morna_within_group_workspace_bytes(c["total"]), "within")
                head, tail = self._within_call_args(c)
                n = len(o)
                counts = torch.empty(n, dtype=torch.int64, device=dev)
                _lib.check(self.lib.morna_within_group_range_count(*head, *tail, r, _lib.dev_ptr(counts), _lib.dev_ptr(ws),
                                                                   ws.numel(), _lib.stream_ptr()), "morna_within_group_range_count")
                off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
                torch.cumsum(counts, 0, out=off[1:])
                total = int(off[-1].item())
                ids = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
                d = torch.empty(max(total, 1), dtype=torch.float64, device=dev)
                _lib.check(self.lib.morna_within_group_range_fill(
                    n, tail[0], self.row_lo, _lib.dev_ptr(c["seg_off"]), c["total"], _lib.dev_ptr(c["row_begin"]),
                    c["max_segment"], _lib.dev_ptr(c["out_slot"]), _lib.dev_ptr(off), _lib.dev_ptr(ids), _lib.dev_ptr(d),
                    _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_within_group_range_fill")
                pieces.append((o, off, ids[:total], d[:total]))
            for view, sel, q, qlab, member in self._within_large(plan):
                off, ids, d = view.range_search_device(q, r, query_groups=qlab)
                pieces.append((sel, off - off[:1], self._within_ids(ids, member), d))
            return splice_csr(nq, pieces, dev)


def splice_csr(nq, pieces, device):
    """One CSR over queries 0..nq-1 from pieces (query indices host int64 [m], offsets [m+1] from 0, ids, dists); a query
    in no piece has an empty list."""
    counts = torch.zeros(nq, dtype=torch.int64, device=device)
    for idx, off, _, _ in pieces:
        counts[torch.from_numpy(idx).to(device)] = off[1:] - off[:-1]
    offsets = torch.zeros(nq + 1, dtype=torch.int64, device=device)
    torch.cumsum(counts, 0, out=offsets[1:])
    total = int(offsets[-1].item())
    ids = torch.empty(total, dtype=torch.int32, device=device)
    d = torch.empty(total, dtype=torch.float64, device=device)
    for idx, off, p_ids, p_d in pieces:
        if p_ids.numel():
            shift = offsets[torch.from_numpy(idx).to(device)] - off[:-1]
            dst = torch.repeat_interleave(shift, off[1:] - off[:-1], output_size=p_ids.numel()) + \
                torch.arange(p_ids.numel(), device=device)
            ids[dst] = p_ids
            d[dst] = p_d
    return offsets, ids, d


class FilteredSearch(object):
    """The searches of a MornaSearch over a chosen subset of its rows (MornaSearch.subset), with results under the
    parent's internal ids.

    The subset is a compacted index of its own, ``inner``: a MornaSearch over the chosen rows gathered on the device in
    ascending id order, with their norms copied; it builds its CSR form and tensor-core operand from them as any index
    does.  Every route runs unchanged on ``inner``, which only ever sees its own row numbers; each entry point below maps
    the ids back once, where the results leave.  The results are those of a brute-force search over the subset rows, bit
    for bit: a row's distance is the same canonical FP64 sum wherever the row sits, and local row -> parent id is strictly
    increasing, so the reference order (distance ascending, equal distances id descending) survives the map.

    ``member_ids``: the subset's parent internal ids (numpy int64, ascending).  ``index_size``, ``sample_count``,
    ``internal_id_map``, ``sample_frequencies`` and ``basename`` are the parent's, so query vectors and metadata are
    built exactly as on the whole index."""

    def __init__(self, parent, internal_ids, keep_parent_rows=True):
        ids = np.unique(np.asarray(internal_ids, dtype=np.int64).reshape(-1))
        if ids.size == 0:
            raise ValueError("a filtered search needs at least one row")
        if ids[0] < parent.row_lo or ids[-1] >= parent.row_hi:
            raise ValueError("internal ids %d..%d are not all resident (rows %d..%d)"
                             % (ids[0], ids[-1], parent.row_lo, parent.row_hi - 1))
        dev = parent.device
        self.lib, self.device, self.dim, self.basename = parent.lib, dev, parent.dim, parent.basename
        self.sample_count, self.index_size = parent.sample_count, parent.index_size
        self.sample_frequencies, self.internal_id_map = parent.sample_frequencies, parent.internal_id_map
        self.row_lo, self.row_hi = parent.row_lo, parent.row_hi
        self.member_ids = ids
        self._ids32 = ids.astype(np.int32)
        m = int(ids.size)
        with torch.cuda.device(dev):
            rows = torch.from_numpy(ids - parent.row_lo).to(dev)
            self._ids_dev = torch.from_numpy(self._ids32).to(dev)
            self._local = torch.full((parent.row_hi - parent.row_lo,), -1, dtype=torch.int64, device=dev)
            self._local[rows] = torch.arange(m, device=dev)
            inner = MornaSearch.__new__(MornaSearch)
            inner.lib, inner.device, inner.basename = parent.lib, dev, parent.basename
            inner.sample_count, inner.index_size, inner.dim, inner.ld = parent.sample_count, m, parent.dim, parent.ld
            # (the parent's map: inner._metadata is only ever given parent ids)
            inner.sample_frequencies, inner.internal_id_map = parent.sample_frequencies, parent.internal_id_map
            inner.row_lo, inner.row_hi = 0, m
            inner.vectors = parent.vectors.index_select(0, rows)
            inner.pp = parent.pp.index_select(0, rows)
            if parent.row_group is not None:        # the subset rows keep their labels; queries keep theirs
                inner.row_group = parent.row_group.index_select(0, rows)
            if parent.cap_group is not None:        # and their cap labels
                inner.set_cap_groups(parent.cap_group.index_select(0, rows))
            inner._build_csr()
            inner.query, inner.query_sample = defaultdict(int), [0.0] * parent.dim
        self.inner = inner
        self._parent_rows = parent.vectors if keep_parent_rows else None
        self._parent_row_group = parent.row_group

    def _to_parent(self, ids):
        """Result ids of `inner` (torch on the current stream, or numpy) -> parent internal ids (int32); -1 padding stays."""
        top = self.member_ids.size - 1
        if isinstance(ids, torch.Tensor):
            return torch.where(ids >= 0, self._ids_dev[ids.long().clamp(0, top)], ids)
        ids = np.asarray(ids)
        return np.where(ids >= 0, self._ids32[np.clip(ids, 0, top)], ids).astype(np.int32)

    def _nn(self, results, meta_db):
        ids = self.member_ids[np.asarray(results[0], dtype=np.int64)].tolist()
        out = (ids,) + tuple(results[1:])
        if meta_db:
            out += (self.inner._metadata(ids),)
        return out

    @property
    def last_stats(self):
        return self.inner.last_stats

    @property
    def last_range_route(self):
        return self.inner.last_range_route

    @property
    def query_sample(self):
        return self.inner.query_sample

    @query_sample.setter
    def query_sample(self, value):
        self.inner.query_sample = value

    def update_query(self, junction):
        self.inner.update_query(junction)

    def finalize_query(self):
        self.inner.finalize_query()

    def stored_queries(self, internal_ids):
        """The stored rows of these parent internal ids as float64 device queries [len x dim], as ``search -q`` uses them.
        Rows outside the subset are legal queries (they cannot return themselves) when the parent's rows were kept;
        otherwise every id must be in the subset.  (The subset's rows are bit copies of the parent's: either source gives
        the same queries.)"""
        ids = torch.as_tensor(internal_ids).to(torch.int64).reshape(-1)
        if ids.numel():
            lo, hi = (int(v) for v in torch.aminmax(ids))
            if lo < self.row_lo or hi >= self.row_hi:
                raise ValueError("internal ids %d..%d are not all resident (rows %d..%d)" % (lo, hi, self.row_lo, self.row_hi - 1))
        rows = ids.to(self.device) - self.row_lo
        if self._parent_rows is not None:
            return self._parent_rows[rows, :self.dim].to(torch.float64).contiguous()
        local = self._local[rows]
        if ids.numel() and bool((local < 0).any()):
            raise ValueError("internal ids outside the subset are queries only with keep_parent_rows=True")
        return self.inner.vectors[local, :self.dim].to(torch.float64).contiguous()

    # ------------------------------------------------------------------ top-k (MornaSearch's entry points, ids mapped)
    def row_groups_of(self, internal_ids):
        """Exclusion labels of these parent internal ids (any resident row, in the subset or not), as the parent holds them."""
        if self._parent_row_group is None:
            raise ValueError("query_groups need row labels: call set_row_groups on the parent before subset()")
        return self._parent_row_group[torch.as_tensor(internal_ids).to(self.device).long() - self.row_lo]

    def exact_search_device(self, queries, k, stream=None, allow_single=True, query_groups=None, max_per_group=None):
        ids, d = self.inner.exact_search_device(queries, k, stream, allow_single, query_groups, max_per_group)
        with torch.cuda.stream(stream):
            return self._to_parent(ids), d

    def batched_search_device(self, queries, k, stream=None, check_overflow=True, phase_events=None, query_groups=None,
                              max_per_group=None):
        ids, d = self.inner.batched_search_device(queries, k, stream, check_overflow, phase_events, query_groups, max_per_group)
        with torch.cuda.stream(stream):
            return self._to_parent(ids), d

    def single_search_device(self, query, k, stream=None):
        ids, d = self.inner.single_search_device(query, k, stream)
        with torch.cuda.stream(stream):
            return self._to_parent(ids), d

    def single_search_stream(self, queries, k):
        ids, d = self.inner.single_search_stream(queries, k)
        return self._to_parent(ids), d

    def approx_search_device(self, queries, k, query_groups=None, max_per_group=None):
        ids, d = self.inner.approx_search_device(queries, k, query_groups, max_per_group)
        return self._to_parent(ids), d

    def exact_search_batch(self, queries, k, tensor_cores=None, query_groups=None, max_per_group=None):
        ids, d = self.inner.exact_search_batch(queries, k, tensor_cores, query_groups, max_per_group)
        return self._to_parent(ids), d

    def search_batches(self, batches, k, depth=2, side_job=False, query_groups=None, max_per_group=None):
        """MornaSearch.search_batches over the subset; a batch of internal ids becomes the stored rows of those ids
        (stored_queries) on the device, and with ``query_groups=True`` takes the parent's labels of those ids (a query
        outside the subset too).  The distances are views of pinned buffers, as there."""
        by_rows = query_groups is True
        labels = iter(query_groups) if query_groups is not None and not by_rows else None
        pairs = []

        def queries():
            for q in batches:
                t = torch.from_numpy(np.ascontiguousarray(q)) if isinstance(q, np.ndarray) else q
                by_id = t.dim() == 1 and t.dtype in (torch.int32, torch.int64)
                if by_rows and not by_id:
                    raise ValueError("query_groups=True needs batches of internal ids")
                pairs.append(self.row_groups_of(t) if by_rows else next(labels) if labels is not None else None)
                yield self.stored_queries(t) if by_id else t
        def groups():
            while True:
                yield pairs.pop(0)          # the labels of the batch queries() has just yielded

        for ids, d in self.inner.search_batches(queries(), k, depth, side_job, None if query_groups is None else groups(),
                                                max_per_group):
            yield self._to_parent(ids), d

    def exact_search_nn(self, num_neighbors, include_distances=True, meta_db=False, query_groups=None, max_per_group=None):
        return self._nn(self.inner.exact_search_nn(num_neighbors, include_distances, query_groups=query_groups,
                                                   max_per_group=max_per_group), meta_db)

    def search_nn(self, num_neighbors, search_k=None, include_distances=True, meta_db=False, max_per_group=None):
        return self._nn(self.inner.search_nn(num_neighbors, search_k, include_distances, max_per_group=max_per_group), meta_db)

    def search_member_n(self, query_id, num_neighbors, search_k=None, include_distances=True,
                        meta_db=False, out=None, max_distance=None, exclude=False, max_per_group=None):
        """MornaSearch.search_member_n over the subset; the queried sample may lie outside it (with ``exclude`` it takes
        its label from the parent's rows)."""
        internal_id = _member_internal_id(self.internal_id_map, query_id, out)
        self.query_sample = self.stored_queries([internal_id])[0].cpu().tolist()
        qg = self.row_groups_of([internal_id]) if exclude else None
        if max_distance is not None:
            return self.range_search_nn(max_distance, include_distances, meta_db, num_neighbors, query_groups=qg,
                                        max_per_group=max_per_group)
        return self.exact_search_nn(num_neighbors, include_distances, meta_db, query_groups=qg, max_per_group=max_per_group)

    # ------------------------------------------------------------------ range search
    def range_search_device(self, queries, max_distance, query_groups=None, max_per_group=None):
        offsets, ids, d = self.inner.range_search_device(queries, max_distance, query_groups, max_per_group)
        return offsets, self._to_parent(ids), d

    def range_search_groups(self, queries, max_distance, byte_cap=None, query_groups=None, max_per_group=None):
        for lo, hi, offsets, ids, d in self.inner.range_search_groups(queries, max_distance, byte_cap, query_groups,
                                                                      max_per_group):
            yield lo, hi, offsets, self._to_parent(ids), d

    def range_search_batch(self, queries, max_distance, query_groups=None, max_per_group=None):
        offsets, ids, d = self.inner.range_search_batch(queries, max_distance, query_groups, max_per_group)
        return offsets, self._to_parent(ids), d

    def range_search_nn(self, max_distance, include_distances=True, meta_db=False, num_neighbors=None, query_groups=None,
                        max_per_group=None):
        return self._nn(self.inner.range_search_nn(max_distance, include_distances, False, num_neighbors, query_groups,
                                                   max_per_group), meta_db)

    # ------------------------------------------------------------------ within-group search (parent ids in and out)
    def _within_args(self, queries, exclude_rows):
        """Queries (parent internal ids -> their stored rows) and excluded parent ids -> subset rows (-1: none)."""
        t = torch.from_numpy(np.ascontiguousarray(queries)) if isinstance(queries, np.ndarray) else torch.as_tensor(queries)
        if t.dim() == 1 and t.dtype in (torch.int32, torch.int64):
            t = self.stored_queries(t)
        if exclude_rows is None:
            return t, None
        e = torch.as_tensor(exclude_rows).to(self.device).long().reshape(-1)
        inside = (e >= self.row_lo) & (e < self.row_hi)
        return t, torch.where(inside, self._local[(e - self.row_lo).clamp(0, self.row_hi - self.row_lo - 1)], -1)

    def within_group_search(self, queries, k, query_groups, exclude_rows=None):
        """MornaSearch.within_group_search over the subset: the rows keep the parent's labels, so each list is the subset
        rows of the query's group."""
        q, e = self._within_args(queries, exclude_rows)
        ids, d = self.inner.within_group_search(q, k, query_groups, e)
        return self._to_parent(ids), d

    def within_group_range(self, queries, max_distance, query_groups, exclude_rows=None):
        q, e = self._within_args(queries, exclude_rows)
        offsets, ids, d = self.inner.within_group_range(q, max_distance, query_groups, e)
        return offsets, self._to_parent(ids), d


class _PipeSlot(object):
    pass


class BatchPipeline(object):
    """``depth`` query batches in flight on one MornaSearch (see MornaSearch.search_batches).

    All kernels run on ONE compute stream; every slot has a copy stream for its pinned-host -> device and
    device -> pinned-host transfers, which overlap the other batches' kernels.  The scoring call of batch
    i+1 carries the re-rank of batch i as its side job (helper warps inside the tcgen05 GEMM kernels, see
    morna_knn_batched_score), so a batch's results are completed when the next batch is submitted -- or at
    collect() if nothing followed.  submit() returns at once; collect() waits for the oldest batch and returns
    host arrays (views of the slot's pinned buffers, valid until the slot is reused ``depth`` submits later)."""

    def __init__(self, search, k, depth=2, side_job=False):
        self.search, self.k, self.depth = search, k, depth
        self.side_job = bool(side_job) and depth > 1
        search.enable_tensor_path()
        dev = search.device
        self.compute = torch.cuda.Stream(device=dev)
        self.slots = []
        for _ in range(depth):
            sl = _PipeSlot()
            sl.stream = torch.cuda.Stream(device=dev)        # this slot's copies
            # kernels: one shared stream when a batch's re-rank rides in the next batch's scoring call, else a stream per
            # slot (consecutive batches then overlap a little at their edges)
            sl.compute = self.compute if self.side_job else torch.cuda.Stream(device=dev)
            sl.h2d, sl.scored, sl.ranked, sl.done = (torch.cuda.Event() for _ in range(4))
            sl.nq = -1
            sl.host_q = sl.ws = sl.job = sl.parts = sl.qg = None
            self.slots.append(sl)
        self.head = self.tail = 0           # next slot to submit into / to collect from
        self.unranked = None                # the slot whose candidate lists wait for their re-rank

    def _size(self, sl, nq, dtype, staging):
        s, k = self.search, self.k
        if staging and (sl.host_q is None or sl.host_q.shape[0] != nq or sl.host_q.dtype != dtype):
            sl.host_q = torch.empty((nq, s.dim), dtype=dtype).pin_memory()      # page-locking is slow: only when needed
        if sl.nq == nq:
            return
        sl.nq = nq
        dev = s.device
        sl.host_ids = torch.empty((nq, k), dtype=torch.int32).pin_memory()
        sl.host_d = torch.empty((nq, k), dtype=torch.float64).pin_memory()
        sl.host_stats = torch.empty((1 + max(s.row_hi - s.row_lo - 1, 0) // s.BATCH_BLOCK_ROWS, 4), dtype=torch.int32).pin_memory()
        sl.ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
        sl.d = torch.empty((nq, k), dtype=torch.float64, device=dev)
        sl.overflow = torch.empty(max(nq, 1), dtype=torch.uint8, device=dev)
        sl.stats = torch.empty(4, dtype=torch.int32, device=dev)

    def _score(self, sl, side):
        """Scoring half of the slot's batch on the compute stream (current); `side`: slot whose re-rank rides along."""
        s, k, lib = self.search, self.k, self.search.lib
        n = s.row_hi - s.row_lo
        need = lib.morna_knn_batched_workspace_bytes(n, sl.nq, s.dim, k)
        if sl.ws is None or sl.ws.numel() < need:
            sl.ws = _lib.workspace(need, s.device)
        job = ctypes.byref(side.job) if side is not None else None
        if sl.qg is None:
            _lib.check(lib.morna_knn_batched_score(
                _lib.dev_ptr(s.hs), s.ld_h, _lib.dev_ptr(s.rho_max), n, s.dim, s.row_lo, _lib.ptr(sl.qd), sl.nq, s.dim, k,
                _lib.dev_ptr(sl.overflow), _lib.dev_ptr(sl.stats), _lib.dev_ptr(sl.ws), sl.ws.numel(), None, job, None,
                _lib.stream_ptr()), "morna_knn_batched_score")
        else:
            _lib.check(lib.morna_knn_batched_score_excl(
                _lib.dev_ptr(s.hs), s.ld_h, _lib.dev_ptr(s.rho_max), n, s.dim, s.row_lo, _lib.ptr(sl.qd), sl.nq, s.dim, k,
                _lib.dev_ptr(sl.overflow), _lib.dev_ptr(sl.stats), _lib.dev_ptr(sl.ws), sl.ws.numel(), None, job, None,
                *s._excl_args(sl.qg), _lib.stream_ptr()), "morna_knn_batched_score_excl")
        sl.job = _lib.RerankJob(s.vectors.data_ptr(), s.pp.data_ptr(), n, s.dim, s.ld, s.row_lo, sl.qd.data_ptr(), sl.nq, s.dim, k,
                                sl.overflow.data_ptr(), sl.ws.data_ptr(), sl.ws.numel())

    use_graphs = True        # replay a slot's kernels from a CUDA graph once its buffers are stable

    def _run_step(self, sl):
        """Scoring + re-rank of the slot's batch on its compute stream (current).  The dozen launches and memsets of a step
        are captured into a CUDA graph per slot the second time the slot sees the same query buffer and batch size, and
        replayed from then on: one launch per batch instead of twelve (no gaps between the kernels, a tenth of the host
        time).  Any change of buffer or size falls back to plain launches."""
        def buffers():
            # (with an exclusion the captured scoring call also reads the row labels: set_row_groups may replace them)
            labels = (sl.qg.data_ptr(), self.search.row_group.data_ptr()) if sl.qg is not None else 0
            return (sl.nq, sl.qd.data_ptr(), sl.ws.data_ptr() if sl.ws is not None else 0, sl.ids.data_ptr(), sl.d.data_ptr(),
                    sl.overflow.data_ptr(), sl.stats.data_ptr(), labels)
        key = buffers()
        if self.use_graphs and getattr(sl, "graph_key", None) == key:
            sl.graph.replay()
            self.search.lib.morna_note_graph_replay(sl.graph_launches)     # the library's launch counter counts kernels that ran
        else:
            seen = getattr(sl, "seen_key", None)
            sl.graph_key = None
            if self.use_graphs and seen == key and sl.ws is not None:
                # capture_begin / capture_end directly: the torch.cuda.graph context would synchronise the device, run the
                # garbage collector and empty the allocator cache first -- a stall of several batch times.  Nothing is
                # allocated between the two calls (every buffer of the step already exists).  The cyclic garbage collector
                # is off while capturing: a MornaSearch and its pipelines form a reference cycle, so a dropped search can
                # be collected at any allocation, and destroying its graphs, events and pinned buffers makes CUDA calls
                # (event queries among them) that invalidate a capture running on this thread.
                graph = torch.cuda.CUDAGraph()
                launches0 = _lib.launch_count()
                gc_on = gc.isenabled()
                gc.disable()
                try:
                    graph.capture_begin(capture_error_mode="thread_local")
                    try:
                        self._score(sl, None)
                        self._rerank_kernels(sl, resume=False)
                    finally:
                        graph.capture_end()
                finally:
                    if gc_on:
                        gc.enable()
                sl.graph, sl.graph_key = graph, key
                sl.graph_launches = _lib.launch_count() - launches0      # counted once while capturing: stands for the replay below
                graph.replay()
            else:
                self._score(sl, None)
                self._rerank_kernels(sl, resume=False)
                sl.seen_key = buffers()
        sl.ranked.record()
        self._copy_back(sl, sl.ids, sl.d, [sl.stats])

    def _rerank_kernels(self, sl, resume):
        s, k, lib = self.search, self.k, self.search.lib
        j = sl.job
        _lib.check(lib.morna_knn_batched_rerank(
            j.vectors, j.pp, j.n, j.dim, j.ld, j.id_base, j.queries, j.nq, j.q_ld, j.k, _lib.dev_ptr(sl.ids),
            _lib.dev_ptr(sl.d), j.overflow, j.workspace, j.workspace_bytes, 1 if resume else 0, _lib.stream_ptr()),
            "morna_knn_batched_rerank")

    def _rerank(self, sl, resume):
        """Re-rank half (what the helper warps left of it when `resume`) on the compute stream, then the slot's
        device -> host copies on its copy stream."""
        s, k, lib = self.search, self.k, self.search.lib
        j = sl.job
        _lib.check(lib.morna_knn_batched_rerank(
            j.vectors, j.pp, j.n, j.dim, j.ld, j.id_base, j.queries, j.nq, j.q_ld, j.k, _lib.dev_ptr(sl.ids),
            _lib.dev_ptr(sl.d), j.overflow, j.workspace, j.workspace_bytes, 1 if resume else 0, _lib.stream_ptr()),
            "morna_knn_batched_rerank")
        sl.ranked.record()
        self._copy_back(sl, sl.ids, sl.d, [sl.stats])

    def _copy_back(self, sl, ids, d, stats):
        sl.stream.wait_event(sl.ranked)
        with torch.cuda.stream(sl.stream):
            for i, st in enumerate(stats):
                sl.host_stats[i].copy_(st, non_blocking=True)
            if ids is not None:
                sl.host_ids.copy_(ids, non_blocking=True)
                sl.host_d.copy_(d, non_blocking=True)
            sl.done.record(sl.stream)

    def _check_resident_ids(self, q):
        """Internal ids given as queries must name rows of this shard: outside [row_lo, row_hi) the row index would be
        negative (torch wraps it: a silently wrong query row) or past the block."""
        s = self.search
        if q.numel() == 0:
            return
        lo, hi = (int(v) for v in (torch.aminmax(q) if q.is_cuda else (q.min(), q.max())))    # (one reduction on the device)
        if lo < s.row_lo or hi >= s.row_hi:
            raise ValueError("internal ids %d..%d are not all resident on this shard (rows %d..%d)"
                             % (lo, hi, s.row_lo, s.row_hi - 1))

    def _stage_groups(self, sl, labels):
        """The batch's query labels in the slot's own device buffer (a stable address for the captured step), or None."""
        if labels is None:
            sl.qg = None
            return
        if getattr(sl, "qgbuf", None) is None or sl.qgbuf.shape[0] != sl.nq:
            sl.qgbuf = torch.empty(max(sl.nq, 1), dtype=torch.int32, device=self.search.device)
        sl.qgbuf[:sl.nq].copy_(torch.as_tensor(labels).reshape(-1).to(device=self.search.device, dtype=torch.int32),
                               non_blocking=True)
        sl.qg = sl.qgbuf[:sl.nq]

    def submit(self, queries, query_groups=None):
        """``query_groups``: None, True (a batch of internal ids takes the labels row_group[ids]) or int32 labels [nq]."""
        s, k = self.search, self.k
        sl = self.slots[self.head % self.depth]
        assert self.head - self.tail < self.depth, "collect() before submitting more than `depth` batches"
        q = torch.from_numpy(np.ascontiguousarray(queries)) if isinstance(queries, np.ndarray) else queries
        by_id = q.dim() == 1 and q.dtype in (torch.int32, torch.int64)      # stored rows as queries (search -q): only ids cross PCIe
        if by_id:
            self._check_resident_ids(q)      # before the slot is taken: the pipeline stays usable after the error
        if query_groups is not None:
            if self.side_job:
                raise ValueError("side_job cannot be combined with query_groups")
            if query_groups is True and not by_id:
                raise ValueError("query_groups=True needs a batch of internal ids")
            if len(torch.as_tensor(q if query_groups is True else query_groups).reshape(-1)) != q.shape[0]:
                raise ValueError("query_groups must hold one label per query")
        self.head += 1
        if by_id:
            self._size(sl, q.shape[0], torch.float64, staging=False)
            with torch.cuda.stream(sl.stream):
                if q.is_cuda:
                    sl.stream.wait_stream(torch.cuda.current_stream(s.device))
                rows = q.to(s.device, non_blocking=True).long() - s.row_lo
                if query_groups is None:
                    sl.qd = s.vectors[rows, :s.dim].to(torch.float64).contiguous()
                else:
                    # an excluded batch by ids goes to the slot's own buffer: with its labels also in a slot buffer, the
                    # step's addresses stay the same from batch to batch, so it is captured and replayed as a vector
                    # batch's is (a search without an exclusion takes the line above, as it always has)
                    if getattr(sl, "qbuf", None) is None or sl.qbuf.shape[0] != sl.nq:
                        sl.qbuf = torch.empty((sl.nq, s.dim), dtype=torch.float64, device=s.device)
                    sl.qbuf.copy_(s.vectors[rows, :s.dim])
                    sl.qd = sl.qbuf
                self._stage_groups(sl, s.row_group[rows] if query_groups is True else query_groups)
                sl.h2d.record(sl.stream)
            self._launch(sl)
            return
        if q.dtype != torch.float32:
            q = q.to(torch.float64)
        resident = q.is_cuda                 # queries already in HBM: no host->device copy
        direct = resident or (q.is_pinned() and q.is_contiguous())
        self._size(sl, q.shape[0], q.dtype, staging=not direct)
        if direct:
            src = q                          # already page-locked: copied straight from the caller's buffer,
        else:                                # which must stay untouched until collect()
            sl.host_q.copy_(q)               # pageable source -> the slot's pinned staging buffer
            src = sl.host_q
        if resident:
            sl.stream.wait_stream(torch.cuda.current_stream(s.device))             # the caller's writes to q are done
        with torch.cuda.stream(sl.stream):
            if resident:
                sl.qd = src.to(torch.float64).contiguous()       # (no copy when already float64 and contiguous)
            else:                            # float32 widens exactly; a per-slot device buffer keeps the address stable
                if getattr(sl, "qbuf", None) is None or sl.qbuf.shape[0] != sl.nq:
                    sl.qbuf = torch.empty((sl.nq, s.dim), dtype=torch.float64, device=s.device)
                sl.qbuf.copy_(src.to(s.device, non_blocking=True))
                sl.qd = sl.qbuf
            self._stage_groups(sl, query_groups)
            sl.h2d.record(sl.stream)
        self._launch(sl)

    def _launch(self, sl):
        """Kernels of the slot's batch (queries in sl.qd once sl.h2d fires) on its compute stream."""
        s, k = self.search, self.k
        n = s.row_hi - s.row_lo
        sl.compute.wait_event(sl.h2d)
        with torch.cuda.stream(sl.compute):
            prev, self.unranked = self.unranked, None
            sl.parts = sl.job = None
            sl.mode = "plain"
            if n == 0 or sl.nq == 0 or k > 512 or k <= 0 or k > n or (s.csr is not None and s.sparse_exact):
                if prev is not None:
                    self._rerank(prev, resume=False)
                ids, d = s.exact_search_device(sl.qd, k, query_groups=sl.qg)
                sl.keep = (ids, d)
                sl.ranked.record()
                self._copy_back(sl, ids, d, [])
            elif n > s.BATCH_BLOCK_ROWS:     # several row blocks: every block is scored and re-ranked here, merged at collect()
                if prev is not None:
                    self._rerank(prev, resume=False)
                sl.mode = "blocks"
                sl.parts = s._batched_launch(sl.qd, k, qg=sl.qg)
                sl.ranked.record()
                self._copy_back(sl, None, None, [part[5] for part in sl.parts])
            elif not self.side_job:
                sl.mode = "pipelined"
                self._run_step(sl)
            else:                            # the previous batch's re-rank rides in this batch's GEMM kernels
                sl.mode = "pipelined"
                self._score(sl, prev)
                if prev is not None:
                    self._rerank(prev, resume=True)
                self.unranked = sl

    def collect(self):
        s, k = self.search, self.k
        assert self.tail < self.head, "nothing in flight"
        sl = self.slots[self.tail % self.depth]
        self.tail += 1
        if self.unranked is sl:              # nothing was submitted after it: its re-rank runs on its own
            self.unranked = None
            with torch.cuda.stream(sl.compute):
                self._rerank(sl, resume=False)
        sl.done.synchronize()
        if sl.mode == "plain":
            return sl.host_ids.numpy(), sl.host_d.numpy()
        if sl.mode == "pipelined":
            sl.parts = [(0, s.row_hi - s.row_lo, sl.ids, sl.d, sl.overflow, sl.stats)]
        nparts = len(sl.parts)
        overflowed = int(sl.host_stats[:nparts, 0].sum()) > 0
        if overflowed or nparts > 1:         # rare: exact-scan fix-up and/or merge of row blocks, then copy again
            with torch.cuda.stream(sl.compute):
                ids, d = s._batched_finish(sl.parts, sl.qd, k, host_stats=[sl.host_stats[i] for i in range(nparts)], qg=sl.qg)
                sl.host_ids.copy_(ids, non_blocking=True)
                sl.host_d.copy_(d, non_blocking=True)
            sl.compute.synchronize()
        else:
            s.last_stats = sl.host_stats[0].to(torch.int64).tolist()
        return sl.host_ids.numpy(), sl.host_d.numpy()
