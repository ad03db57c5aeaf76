"""Batch queries: the query vector of every sample of an intropolis-format file, built on the device, and the batch
search behind `morna search --query-intropolis` / `--all-samples`.

A query file is turned into vectors the way the index build turns its input into rows (index.py), with three
differences: a row's idf comes from the index's .freq.mor table and .stats.mor sample count (one device join per row,
csrc/query_build.cu), every row passes, and the sums stay in doubles.  Query j is the j-th distinct sample of the file
in first-seen order.  The vectors equal, bit for bit, what finalize_query (morna.py:609-629) builds from the
(key, coverage) pairs of the rows that list the sample, in file order, keeping only keys present in .freq.mor
(cli.py's `key in sample_frequencies` test).
"""
import numpy as np
import torch

from . import _lib, files, parse
from .index import round_up
from .parse import RowBatch
from .search import FilteredSearch

# Above this many bytes of query vectors in flight (nq * dim * 16: the bucket-major accumulator and its transpose), the
# vectors are built and searched in slices of query ids.
SLICE_BYTES_CAP = 8 << 30
BATCH_QUERIES = 4096


def read_rows(path):
    """Rows of a (gzipped) intropolis file as the binary CSR of RowBatch.finish(): the native tokenizer, and
    parse.tokenize_line for the rows it flags, as the index build reads its input (MornaIndex.add_text)."""
    rows = RowBatch()
    with parse.open_intropolis_binary(path) as fh:
        for block in parse.read_blocks(fh):
            keys, key_off, row_off, sample, cov, line_off, needs = parse.tokenize_buffer(block)
            n = len(needs)
            start = 0
            for stop in np.nonzero(needs)[0].tolist() + [n]:
                if stop > start:
                    k0, k1, p0, p1 = int(key_off[start]), int(key_off[stop]), int(row_off[start]), int(row_off[stop])
                    rows.add_block(keys[k0:k1], np.diff(key_off[start:stop + 1]), np.diff(row_off[start:stop + 1]),
                                   sample[p0:p1], cov[p0:p1])
                if stop < n:
                    rows.add(*parse.tokenize_line(bytes(block[line_off[stop]:line_off[stop + 1]]).decode("utf-8")))
                start = stop + 1
    return rows.finish()


def _hash(search, d_keys, d_key_off, n):
    dev = search.device
    raw = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    bucket = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    sign = torch.empty(max(n, 1), dtype=torch.int8, device=dev)
    _lib.check(search.lib.morna_hash_junctions(_lib.dev_ptr(d_keys), _lib.dev_ptr(d_key_off), n, search.dim, _lib.dev_ptr(raw),
                                               _lib.dev_ptr(bucket), _lib.dev_ptr(sign), _lib.stream_ptr()), "morna_hash_junctions")
    return raw, bucket, sign


class JunctionTable(object):
    """The index's junction keys (every key of .freq.mor with a positive frequency) in a device hash table, with each
    key's idf computed once on the host by morna_idf_host: log(sample_count / freq), the C library's log that CPython's
    math.log calls.  Keys of frequency 0 would contribute +-0.0 and are left out."""

    def __init__(self, search):
        lib, dev = search.lib, search.device
        keys = [k for k, f in search.sample_frequencies.items() if f > 0]
        self.n = n = len(keys)
        freq = np.fromiter((search.sample_frequencies[k] for k in keys), dtype=np.int64, count=n)
        blobs = [k.encode("utf-8") for k in keys]
        off = np.zeros(n + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(b) for b in blobs], dtype=np.int64)
        packed = np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8)
        idf = np.zeros(max(n, 1), dtype=np.float64)
        _lib.check(lib.morna_idf_host(freq.ctypes.data, np.ones(n, np.uint8).ctypes.data, n, int(search.sample_count),
                                      idf.ctypes.data), "morna_idf_host")
        with torch.cuda.device(dev):
            self.keys = torch.from_numpy(packed.copy()).to(dev)
            self.key_off = torch.from_numpy(off).to(dev)
            self.idf = torch.from_numpy(idf).to(dev)
            self.raw = _hash(search, self.keys, self.key_off, n)[0]
            self.table = _lib.workspace(lib.morna_junction_table_bytes(n), dev)
            _lib.check(lib.morna_junction_table_build(_lib.dev_ptr(self.keys), _lib.dev_ptr(self.key_off), _lib.dev_ptr(self.raw),
                                                      n, _lib.dev_ptr(self.table), self.table.numel(), _lib.stream_ptr()),
                       "morna_junction_table_build")

    def lookup(self, search, d_keys, d_key_off, d_raw, d_row_off, d_sample, n_rows):
        """-> device (match int32, pass uint8, idf float64, flags uint8) per row and the number of flagged rows (an int:
        the one value read back)."""
        lib, dev = search.lib, search.device
        match = torch.empty(max(n_rows, 1), dtype=torch.int32, device=dev)
        passing = torch.empty(max(n_rows, 1), dtype=torch.uint8, device=dev)
        idf = torch.empty(max(n_rows, 1), dtype=torch.float64, device=dev)
        flags = torch.empty(max(n_rows, 1), dtype=torch.uint8, device=dev)
        n_flagged = torch.empty(1, dtype=torch.int32, device=dev)
        ws = _lib.workspace(lib.morna_junction_lookup_workspace_bytes(self.n), dev)
        _lib.check(lib.morna_junction_lookup(
            _lib.dev_ptr(self.table), self.table.numel(), _lib.dev_ptr(self.keys), _lib.dev_ptr(self.key_off),
            _lib.dev_ptr(self.raw), _lib.dev_ptr(self.idf), self.n, _lib.dev_ptr(d_keys), _lib.dev_ptr(d_key_off),
            _lib.dev_ptr(d_raw), _lib.dev_ptr(d_row_off), _lib.dev_ptr(d_sample), n_rows, _lib.dev_ptr(match),
            _lib.dev_ptr(passing), _lib.dev_ptr(idf), _lib.dev_ptr(flags), _lib.dev_ptr(n_flagged), _lib.dev_ptr(ws),
            ws.numel(), _lib.stream_ptr()), "morna_junction_lookup")
        return match, passing, idf, flags, int(n_flagged.item())


def junction_table(search):
    """The device junction table of `search`'s index, built on first use and kept on the object."""
    table = getattr(search, "_junction_table", None)
    if table is None:
        table = search._junction_table = JunctionTable(search)
    return table


def merge_repeated_pairs(row_off, sample, cov, rows, match):
    """Coverage fix-ups that make the row-by-row scatter-add equal the reference's per-sample dict of summed coverages.
    `rows`: the flagged rows (ascending), `match`: their key indices.  Every (key, sample) pair met more than once among
    them keeps its first position, which takes the sum of the coverages; the later positions get coverage 0, so they
    add sign * (0 * idf) = +-0.0 to a cell that the reference's sum leaves as it is (x + +-0.0 == x for every x this
    sum can hold: the cells start at +0.0).  Returns (positions int64, new coverages int32)."""
    rows = np.asarray(rows, dtype=np.int64)
    starts = row_off[rows]
    lens = row_off[rows + 1] - starts
    total = int(lens.sum())
    if total == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int32)
    pos = np.repeat(starts - np.concatenate([[0], np.cumsum(lens)[:-1]]), lens) + np.arange(total)
    key = np.repeat(np.asarray(match, dtype=np.int64), lens)
    smp = sample[pos].astype(np.int64)
    order = np.lexsort((pos, smp, key))                # by key, then sample, then file position
    pos, key, smp = pos[order], key[order], smp[order]
    head = np.ones(total, dtype=bool)
    head[1:] = (key[1:] != key[:-1]) | (smp[1:] != smp[:-1])
    group = np.cumsum(head) - 1
    size = np.bincount(group)
    sums = np.add.reduceat(cov[pos].astype(np.int64), np.nonzero(head)[0])
    repeated = size[group] > 1
    if not repeated.any():
        return np.zeros(0, np.int64), np.zeros(0, np.int32)
    new = np.where(head, sums[group], 0)[repeated]
    if new.max() > np.iinfo(np.int32).max or new.min() < np.iinfo(np.int32).min:
        raise ValueError("a summed coverage of a repeated (junction, sample) pair exceeds the int32 range")
    return pos[repeated], new.astype(np.int32)


class QueryFile(object):
    """The rows of a query file on the device, joined against the index: query_vectors(lo, hi) builds the float64
    vectors of queries [lo, hi).  `sample_ids` (numpy int64 [nq]) is the sample id of each query.  `on_phase(name)`, if
    given, is called after each phase (the measurement script synchronises and reads a clock there)."""

    def __init__(self, search, path, on_phase=None):
        mark = on_phase or (lambda name: None)
        self.search = search
        lib, dev = search.lib, search.device
        packed, key_off, row_off, sample, cov = read_rows(path)
        n_rows, nnz = len(key_off) - 1, int(row_off[-1])
        self.n_rows, self.nnz = n_rows, nnz
        if nnz and sample.min() < 0:
            raise ValueError("negative sample id in " + path)
        self.max_sample_id = int(sample.max()) if nnz else 0
        mark("read_tokenize")
        with torch.cuda.device(dev):
            up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt) if len(a) else np.zeros(1, dt)).pin_memory().to(dev, non_blocking=True)
            d_keys = up(np.concatenate([packed, np.zeros(1, np.uint8)]), np.uint8)
            d_key_off, self.row_off = up(key_off, np.int32), up(row_off, np.int64)
            self.sample, self.cov = up(sample, np.int32), up(cov, np.int32)
            mark("h2d")
            d_raw, self.bucket, self.sign = _hash(search, d_keys, d_key_off, n_rows)
            mark("hash")
            table = junction_table(search)
            mark("table_build")
            match, self.passing, self.idf, flags, n_flagged = table.lookup(search, d_keys, d_key_off, d_raw, self.row_off,
                                                                           self.sample, n_rows)
            self.n_merged = 0
            if n_flagged:                                  # rare: a key on several rows, or a row listing a sample twice
                rows = torch.nonzero(flags[:n_rows]).flatten()
                pos, new = merge_repeated_pairs(row_off, sample, cov, rows.cpu().numpy(), match[rows].cpu().numpy())
                if len(pos):
                    self.cov[torch.from_numpy(pos).to(dev)] = torch.from_numpy(new).to(dev)
                self.n_merged = len(pos)
            mark("lookup")
            # every sample of the file is a query, also one none of whose junctions is in the index
            self.id_of = torch.empty(self.max_sample_id + 1, dtype=torch.int32, device=dev)
            n_kept = torch.zeros(1, dtype=torch.int32, device=dev)
            all_pass = torch.ones(max(n_rows, 1), dtype=torch.uint8, device=dev)
            ws = _lib.workspace(lib.morna_assign_internal_ids_workspace_bytes(n_rows, nnz, self.max_sample_id), dev)
            _lib.check(lib.morna_assign_internal_ids(
                _lib.dev_ptr(self.row_off), _lib.dev_ptr(all_pass), n_rows, _lib.dev_ptr(self.sample), nnz, self.max_sample_id,
                0, _lib.dev_ptr(self.id_of), _lib.dev_ptr(n_kept), _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()),
                "morna_assign_internal_ids")
            self.nq = int(n_kept.item()) if nnz else 0
            seen = torch.nonzero(self.id_of >= 0).flatten()
            sample_of = torch.empty(max(self.nq, 1), dtype=torch.int64, device=dev)
            sample_of[self.id_of[seen].long()] = seen
            self.sample_ids = sample_of[:self.nq].cpu().numpy()
            self._acc_ws = None

    def query_vectors(self, lo, hi):
        """float64 [hi - lo x dim] device vectors of queries [lo, hi): morna_index_accumulate over the id range, then
        the bucket-major sums transposed (no float32 rounding)."""
        s, lib, dev = self.search, self.search.lib, self.search.device
        width = hi - lo
        acc_ld = max(round_up(width, 32), 32)
        with torch.cuda.device(dev):
            acc = torch.empty(s.dim * acc_ld, dtype=torch.float64, device=dev)
            need = lib.morna_index_accumulate_workspace_bytes(self.n_rows, self.nnz, s.dim)
            if self._acc_ws is None or self._acc_ws.numel() < need:
                self._acc_ws = _lib.workspace(need, dev)
            _lib.check(lib.morna_index_accumulate(
                _lib.dev_ptr(self.row_off), _lib.dev_ptr(self.passing), _lib.dev_ptr(self.bucket), _lib.dev_ptr(self.sign),
                _lib.dev_ptr(self.idf), self.n_rows, _lib.dev_ptr(self.sample), _lib.dev_ptr(self.cov), self.nnz,
                _lib.dev_ptr(self.id_of), self.max_sample_id, lo, hi, s.dim, _lib.dev_ptr(acc), acc_ld,
                _lib.dev_ptr(self._acc_ws), self._acc_ws.numel(), _lib.stream_ptr()), "morna_index_accumulate")
            return acc.view(s.dim, acc_ld)[:, :width].t().contiguous()

    def slices(self, cap=None):
        """(lo, hi) id slices whose vectors fit the cap (SLICE_BYTES_CAP by default): one slice unless nq*dim*16 exceeds it."""
        cap = SLICE_BYTES_CAP if cap is None else cap
        width = max(1, int(cap) // (self.search.dim * 16))
        return [(lo, min(self.nq, lo + width)) for lo in range(0, self.nq, width)]

    def all_vectors(self, cap=None):
        """Host float64 [nq x dim] of every query (tests, small files)."""
        out = np.zeros((self.nq, self.search.dim), dtype=np.float64)
        for lo, hi in self.slices(cap):
            out[lo:hi] = self.query_vectors(lo, hi).cpu().numpy()
        return out


def search_query_file(search, path, k, exact=True, cap=None, query_labels=None):
    """Generator of (sample ids [b], ids [b x k], dists [b x k]) numpy arrays, batch by batch in query order.  The arrays
    are the caller's (search_batches' own are views of pinned buffers that the pipeline reuses two batches later).
    `query_labels(sample_ids)` -> int32 labels: per-query exclusion (exact only; the search's rows carry labels)."""
    qf = QueryFile(search, path)
    for lo, hi in qf.slices(cap):
        vecs = qf.query_vectors(lo, hi)
        starts = range(0, hi - lo, BATCH_QUERIES)
        if exact:
            groups = None if query_labels is None else \
                (query_labels(qf.sample_ids[lo + b:min(hi, lo + b + BATCH_QUERIES)]) for b in starts)
            results = search.search_batches((vecs[b:b + BATCH_QUERIES] for b in starts), k, query_groups=groups)
        else:
            results = (tuple(t.cpu().numpy() for t in search.approx_search_device(vecs[b:b + BATCH_QUERIES], k)) for b in starts)
        for b, (ids, d) in zip(starts, results):
            yield qf.sample_ids[lo + b:lo + b + ids.shape[0]], ids.copy(), d.copy()


def all_sample_ids(search):
    """Internal ids of the samples --all-samples queries: every indexed sample, or every sample of a FilteredSearch's
    subset (its k-NN or range graph)."""
    if isinstance(search, FilteredSearch):
        return search.member_ids
    return np.arange(search.index_size, dtype=np.int64)


def search_all_samples(search, k, inverse, exclude=False):
    """Every indexed sample by internal id (the stored rows as queries, as `search -q`), exactly; only ids cross PCIe.
    Yields (sample ids, ids, dists) numpy arrays as search_query_file does.  `exclude`: each query takes its row's label
    (the search's rows carry labels), so it leaves out its own sample and its group."""
    members = all_sample_ids(search)
    starts = range(0, len(members), BATCH_QUERIES)
    batches = (members[b:b + BATCH_QUERIES] for b in starts)
    for b, (ids, d) in zip(starts, search.search_batches(batches, k, query_groups=True if exclude else None)):
        yield inverse[members[b:b + ids.shape[0]]], ids.copy(), d.copy()


def search_query_file_range(search, path, max_distance, cap=None, result_cap=None, query_labels=None):
    """Range variant of search_query_file (always exact): every indexed sample within `max_distance` of each query.
    Yields (sample ids [b], offsets int64 [b+1], ids, dists) numpy CSR batches in query order; query j's list is
    ids/dists[offsets[j]:offsets[j+1]].  The lists of a 4096-query batch are counted first, and a batch whose lists
    would take more than `result_cap` bytes (SLICE_BYTES_CAP by default) comes in smaller groups of queries."""
    qf = QueryFile(search, path)
    result_cap = SLICE_BYTES_CAP if result_cap is None else result_cap
    for lo, hi in qf.slices(cap):
        vecs = qf.query_vectors(lo, hi)
        for b in range(0, hi - lo, BATCH_QUERIES):
            groups = None if query_labels is None else query_labels(qf.sample_ids[lo + b:min(hi, lo + b + BATCH_QUERIES)])
            for g0, g1, off, ids, d in search.range_search_groups(vecs[b:b + BATCH_QUERIES], max_distance, result_cap, groups):
                yield qf.sample_ids[lo + b + g0:lo + b + g1], off.cpu().numpy(), ids.cpu().numpy(), d.cpu().numpy()


def search_all_samples_range(search, max_distance, inverse, result_cap=None, exclude=False):
    """Range variant of search_all_samples: the stored rows as queries, built on the device from their ids.  Yields
    (sample ids, offsets, ids, dists) numpy CSR batches as search_query_file_range does."""
    members = all_sample_ids(search)
    result_cap = SLICE_BYTES_CAP if result_cap is None else result_cap
    for b in range(0, len(members), BATCH_QUERIES):
        batch = members[b:b + BATCH_QUERIES]
        groups = None
        if isinstance(search, FilteredSearch):
            q = search.stored_queries(batch)
            if exclude:
                groups = search.row_groups_of(batch)
        else:
            rows = torch.arange(b, b + len(batch), device=search.device) - search.row_lo
            q = search.vectors[rows, :search.dim].to(torch.float64).contiguous()
            if exclude:
                groups = search.row_group[rows]
        for g0, g1, off, ids, d in search.range_search_groups(q, max_distance, result_cap, groups):
            yield inverse[batch[g0:g1]], off.cpu().numpy(), ids.cpu().numpy(), d.cpu().numpy()


def cut_lists(offsets, ids, dists, limit):
    """CSR lists cut to their first `limit` entries (numpy; None: unchanged)."""
    if limit is None:
        return offsets, ids, dists
    lens = np.diff(offsets)
    keep_len = np.minimum(lens, max(int(limit), 0))
    rank = np.arange(len(ids)) - np.repeat(offsets[:-1], lens)
    keep = rank < np.repeat(keep_len, lens)
    out = np.zeros_like(offsets)
    np.cumsum(keep_len, out=out[1:])
    return out, ids[keep], dists[keep]


def write_results(out, sample_ids, ids, dists, include_distances, meta_basename, inverse, offsets=None, limit=None):
    """One batch of results.  Each line: the query's sample id, a tab, then exactly the line cli.results_output prints for
    that query (rank, internal id, distance with -d, metadata tuple with -m).  With `offsets`, the batch is CSR (query j's
    list is ids/dists[offsets[j]:offsets[j+1]]) and each list is cut to its first `limit` entries."""
    from .cli import py2_str
    if offsets is None:
        kept = ids[ids >= 0]
        queries = zip(sample_ids.tolist(), ids.tolist(), dists.tolist())
    else:
        offsets, ids, dists = cut_lists(offsets, ids, dists, limit)
        kept, o, il, dl = ids, offsets.tolist(), ids.tolist(), dists.tolist()
        queries = ((sid, il[o[j]:o[j + 1]], dl[o[j]:o[j + 1]]) for j, sid in enumerate(sample_ids.tolist()))
    meta = None
    if meta_basename is not None:
        meta = iter(files.read_meta(meta_basename, inverse[kept].tolist()))
    lines = []
    for sid, row_ids, row_d in queries:
        prefix = str(sid) + "\t"
        rank = 0
        for iid, dist in zip(row_ids, row_d):
            if iid < 0:
                continue
            rank += 1
            line = prefix + str(rank) + ".\t" + str(iid)
            if include_distances:
                line += "\t" + py2_str(dist)
            if meta is not None:
                line += "\t" + py2_str(next(meta))
            lines.append(line)
    if lines:
        out.write("\n".join(lines) + "\n")


def inverse_map(search):
    """internal id -> sample id as a numpy array, built once per run (inverse_lookup scans the map per id)."""
    inv = np.full(search.index_size, -1, dtype=np.int64)
    for sample_id, iid in search.internal_id_map.items():
        inv[iid] = sample_id
    return inv
