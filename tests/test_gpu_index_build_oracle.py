"""The index build through the C ABI (morna_assign_internal_ids, morna_index_accumulate, morna_round_store) against the
C oracle's sequential scatter-add (oracle.c: oracle_index_accumulate, the order of morna.py:376-388), bit for bit, on
every variant of csrc/index_build.cu and at the sizes where its kernels change shape:

  id pass          first_position_smem_kernel while max_sample_id + 1 <= 49,152, first_position_kernel above that
  warp-per-range   index_accumulate3_kernel: every row strictly ascending, ids in at most 32 ranges of 2^shift
                   (shift 10, 11 or 12); above 131,071 ids its slice would not fit in shared memory
  barrier-per-row  index_accumulate2_kernel, plain (every passing row monotonic) or atomic (a row that is neither), in
                   id tiles of 22,528 and metadata windows of 512 rows; it answers for rows that do not ascend, for ids
                   above 131,071 and for wide --features (>= 4096 rows and fewer than 64 rows a bucket)
  simple           index_accumulate_kernel (tuning key 4 = 0), id tiles of 24,576

The CSR is built here, with bucket, sign and idf chosen per row, so bucket depths, id layouts and the one unsorted pair
of a row sit exactly at a threshold.  The accumulator and the float32 rows are pre-filled with NaN, so a cell the
kernels skip shows, and a cell they must not touch has to stay NaN.  Which variant answered follows from the launch
count of the call and from how the data was built (see `answered`)."""
import math
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import c_oracle

NAN_BITS = np.float64("nan").view(np.int64)
TUNING_DEFAULTS = {8: 3, 4: 1, 7: 1, 12: 10, 25: 1}     # morna_debug_set_tuning keys of the index build, with defaults
FIRST_POS_SMEM_IDS = 49152                               # index_build.cu kFirstPosSmemIds
ACC2_TILE = 22528                                        # kAcc2Tile


@pytest.fixture(scope="module")
def lib():
    from morna_b200 import _lib
    assert torch.cuda.is_available(), "these tests need the B200"
    return _lib.load()


@pytest.fixture
def knobs(lib):
    """Sets index-build tuning keys for one test; they are process-wide, so every default comes back afterwards."""
    def set_(key, value):
        assert lib.morna_debug_set_tuning(key, value) == 0
    for k, v in TUNING_DEFAULTS.items():
        set_(k, v)
    try:
        yield set_
    finally:
        for k, v in TUNING_DEFAULTS.items():
            lib.morna_debug_set_tuning(k, v)


# ------------------------------------------------------------------ inputs
def make(rows, dim, rng, bucket=None, sign=None, idf=None, passing=None, cov=None, max_sample_id=None):
    """CSR of `rows` (one int array of sample ids per row) with per-row bucket / sign / idf / pass; unset ones random."""
    n = len(rows)
    lens = np.array([len(r) for r in rows], np.int64)
    row_off = np.zeros(n + 1, np.int64)
    row_off[1:] = np.cumsum(lens)
    sample = np.concatenate([np.asarray(r, np.int64) for r in rows]).astype(np.int32) if n else np.zeros(0, np.int32)
    nnz = int(row_off[-1])
    d = types.SimpleNamespace(
        dim=dim, row_off=row_off, sample=sample,
        bucket=np.asarray(bucket if bucket is not None else rng.integers(0, dim, n), np.int32),
        sign=np.asarray(sign if sign is not None else rng.choice([-1, 1], n), np.int8),
        idf=np.asarray(idf if idf is not None else rng.uniform(0.01, 9.0, n), np.float64),
        passing=np.asarray(passing if passing is not None else np.ones(n), np.uint8),
        cov=np.asarray(cov if cov is not None else 1 + rng.geometric(0.3, nnz) * rng.integers(1, 40, nnz), np.int32),
        max_sample_id=int(max_sample_id if max_sample_id is not None else sample.max()))
    assert d.sample.max() <= d.max_sample_id and d.sample.min() >= 0
    return d


def random_rows(rng, n_rows, universe, mean_len, max_len=None):
    """Strictly ascending rows drawn from the sorted id array `universe`."""
    lens = np.clip(rng.lognormal(math.log(mean_len), 0.9, n_rows).astype(np.int64), 1, max_len or len(universe))
    return [universe[np.unique(rng.integers(0, len(universe), int(k)))] for k in lens]


def cover(rng, rows, passing, universe, first_row, last_row=None):
    """Adds every id of `universe` that no passing row of [first_row, last_row) lists to random passing rows there."""
    hosts = [j for j in range(first_row, last_row or len(rows)) if passing[j]]
    missing = np.setdiff1d(universe, np.concatenate([rows[j] for j in hosts]))
    for j, part in zip(rng.choice(hosts, size=len(hosts), replace=False), np.array_split(missing, len(hosts))):
        if len(part):
            rows[j] = np.union1d(rows[j], part)


def id_pass_data(m, holes, layout, n_rows=6400, dim=16, seed=1):
    """Rows over an id space of m ids (a sparse subset of it with `holes`).  The id pass reads the rows in three stretches
    and, between them, stops once `distinct_samples` ids have been met.  Every id but A and B is met in passing rows
    before n_rows/64.  With layout 'late', A is first listed by a passing row at n_rows/64 (the first row of the second
    stretch) and B at n_rows/8 (the first row of the third), so at both checks the count is exactly one id short; with
    'early', A and B are also met before n_rows/64, so the count is reached at the first check.  A and B appear in a
    failing row before either cut; X is listed by failing rows only, so it never gets an id.  Every row ascends."""
    rng = np.random.default_rng(seed + m)
    universe = np.arange(m) if not holes else np.union1d(rng.choice(m - 1, size=m // 7, replace=False), [m - 1])
    a, b, x = rng.choice(universe[:-1], size=3, replace=False)
    base = np.setdiff1d(universe, [a, b, x])
    passing = (np.arange(n_rows) % 9 != 4).astype(np.uint8)
    c1, c2, last_failing = n_rows // 64, n_rows // 8, n_rows - 1 - (n_rows - 5) % 9
    rows = random_rows(rng, n_rows, base, 60)
    cover(rng, rows, passing, base, 0, c1)
    assert passing[c1] and passing[c2] and not passing[4] | passing[13] | passing[last_failing]
    placed = [(c1, a), (c2, b), (c2 + 7, a), (n_rows - 1, b), (4, a), (4, b), (4, x), (13, x), (last_failing, x)]
    if layout == "early":
        placed += [(1, a), (2, b)]
    for j, s in placed:
        rows[j] = np.union1d(rows[j], [s])
    d = make(rows, dim, rng, passing=passing, max_sample_id=m - 1)
    d.distinct = len(base) + 2
    met = lambda k: len(np.unique(np.concatenate([r for r, p in zip(rows[:k], passing[:k]) if p])))
    assert (met(c1), met(c2)) == ((d.distinct, d.distinct) if layout == "early" else (d.distinct - 2, d.distinct - 1))
    return d


def warp_data(max_id, n_rows=3000, deep=2400, dim=24, long_row=6000, seed=2):
    """Ascending rows over [0, max_id] for the warp-per-range variant at the shift the default picks: one bucket with
    `deep` rows, buckets 5 and 17 empty, one row listing `long_row` consecutive ids (every segment of it many 32-pair
    chunks), single-pair rows at q * 2^shift - 1 and q * 2^shift for every range boundary q, and short rows straddling
    each boundary."""
    rng = np.random.default_rng(seed + max_id)
    shift = 10
    while (max_id >> shift) + 1 > 32:
        shift += 1
    universe = np.arange(max_id + 1)
    rows = random_rows(rng, n_rows, universe, 150)
    extra = [np.arange(s0, s0 + long_row) for s0 in [int(rng.integers(0, max_id + 2 - long_row))]] + [np.array([max_id])]
    for q in range(1, (max_id >> shift) + 1):
        e = q << shift
        extra += [np.array([e - 1]), np.array([e]), np.arange(e - 3, min(e + 3, max_id + 1))]
    for r in extra:
        rows.insert(int(rng.integers(0, len(rows) + 1)), r)
    n = len(rows)
    bucket = rng.choice(np.setdiff1d(np.arange(dim), [0, 5, 17]), size=n)
    bucket[rng.choice(n, size=deep, replace=False)] = 0
    passing = (rng.random(n) < 0.9).astype(np.uint8)
    passing[[j for j, r in enumerate(rows) if len(r) <= 6 or len(r) == long_row]] = 1
    d = make(rows, dim, rng, bucket=bucket, passing=passing)
    d.shift = shift
    return d


def ascending_violation_data(where, kind, n_rows=300, dim=16, seed=3):
    """Rows over ids [0, 3000) (three sample-id ranges of 1,024) that ascend everywhere except at one position p:
    sample[p] equal to sample[p - 1] ('equal') or the two swapped ('descending').  p is a multiple of 4 inside a passing
    row ('group', the ascending check compares it with the previous 16-byte group's last element), the last pair of the
    array with nnz = 1, 2, 3 mod 4 ('tail1'..'tail3', the scalar tail) or inside a failing row ('failing').  The row
    lists ids below 1,024 up to p - 1 and ids from 1,024 on from p, so a swapped pair puts an id of the second range
    before one of the first: a warp that took the row would get wrong segment bounds.  p - 1 and p are in the same
    32-pair chunk of the row, so a warp that took a row with an equal pair would add both in one step."""
    rng = np.random.default_rng(seed)
    rows = random_rows(rng, n_rows, np.arange(3000), 60, 300)
    passing = (rng.random(n_rows) < 0.85).astype(np.uint8)
    long_rows = [j for j in range(n_rows // 4, n_rows - 1) if len(rows[j]) >= 48]
    if where.startswith("tail"):
        r = int(where[4:])
        nnz_before = sum(len(x) for x in rows[:-1])
        k = 70
        while (nnz_before + k) % 4 != r or (k - 1) % 32 == 0:
            k -= 1
        j, off, passing[-1] = n_rows - 1, k - 1, 1
    else:
        j = [q for q in long_rows if bool(passing[q]) == (where == "group")][0]
        start = sum(len(x) for x in rows[:j])
        off = (start + 12) // 4 * 4 - start                # 9..12 pairs into the row: a multiple of 4 in the array
        k = len(rows[j])
    row = np.concatenate([np.sort(rng.choice(1024, size=off, replace=False)),
                          np.sort(rng.choice(np.arange(1024, 3000), size=k - off, replace=False))])
    if kind == "equal":
        row[off] = row[off - 1]
    else:
        row[off - 1], row[off] = row[off], row[off - 1]
    rows[j] = row
    d = make(rows, dim, rng, passing=passing)
    p = int(d.row_off[j]) + off
    assert where != "group" or p % 4 == 0
    assert kind == "equal" or d.sample[p] < 1024 <= d.sample[p - 1]
    assert not where.startswith("tail") or (p == len(d.sample) - 1 and len(d.sample) % 4 == int(where[4:]))
    return d


def tile_data(kept, n_rows=4096, dim=128, seed=4):
    """Exactly `kept` distinct sample ids (a sparse subset of [0, 1.25 kept)) over n_rows ascending rows in dim buckets,
    buckets 7 and 100 empty: 4096 <= n_rows < 64 * dim, the wide-features shape where the barrier variant answers."""
    rng = np.random.default_rng(seed + kept)
    universe = np.sort(rng.choice(kept + kept // 4, size=kept, replace=False))
    passing = (rng.random(n_rows) < 0.9).astype(np.uint8)
    rows = random_rows(rng, n_rows, universe, 140)
    cover(rng, rows, passing, universe, n_rows // 2)
    bucket = rng.choice(np.setdiff1d(np.arange(dim), [7, 100]), size=n_rows)
    return make(rows, dim, rng, bucket=bucket, passing=passing)


def high_id_data(max_id, n_rows=2000, n_ids=20000, dim=8, seed=5):
    """Ascending rows over n_ids ids spread up to max_id > 131,071: the warp variant's pre-pass runs, its slice would
    need more than 200 KB, and the barrier variant answers."""
    rng = np.random.default_rng(seed + max_id)
    universe = np.union1d(rng.choice(max_id, size=n_ids - 1, replace=False), [max_id])
    rows = random_rows(rng, n_rows, universe, 80)
    rows[n_rows // 3] = np.union1d(rows[n_rows // 3], [max_id])
    return make(rows, dim, rng, passing=(rng.random(n_rows) < 0.9).astype(np.uint8))


def deep_bucket_data(depth, kind, others=400, dim=6, seed=6):
    """`depth` passing rows in bucket 2 (several 512-row metadata windows of the barrier variant; failing rows in the
    same bucket between them), `others` rows elsewhere, random signs.  One row of bucket 2, past its 1,024th row where
    the bucket is that deep, does not ascend: strictly descending ('plain': the plain instantiation answers) or listing
    a sample twice, out of order ('atomic')."""
    rng = np.random.default_rng(seed + depth)
    n_fail = depth // 5
    n = depth + n_fail + others
    rows = random_rows(rng, n, np.arange(3000), 40, 200)
    bucket = rng.choice([0, 1, 3, 4, 5][:dim - 1], size=n)
    passing = np.ones(n, np.uint8)
    deep_rows = np.sort(rng.choice(n, size=depth + n_fail, replace=False))
    bucket[deep_rows] = 2
    passing[rng.choice(deep_rows, size=n_fail, replace=False)] = 0
    in_bucket = [j for j in deep_rows if passing[j]]
    j = in_bucket[min(1030, depth - 3)]
    r = rows[j] if len(rows[j]) >= 3 else np.array([10, 20, 30])
    rows[j] = r[::-1].copy() if kind == "plain" else np.concatenate([r[1:], r[:1], r[1:2]])
    return make(rows, dim, rng, bucket=bucket, passing=passing)


def values_data(descending_row, n_rows=600, dim=16, sample_count=3000, seed=7):
    """Coverages of 1 and 2^31 - 1 next to ordinary ones; idf = log(N / freq) with freq == N on some rows (idf 0; with a
    negative sign every addend of the row is -0.0), freq > N on others (negative idf).  Sample 2999 is listed only by
    idf-0 rows of negative sign, bucket 9 by no row.  `descending_row` makes one row strictly descending, so the
    barrier variant answers instead of the warp variant."""
    rng = np.random.default_rng(seed)
    rows = random_rows(rng, n_rows, np.arange(sample_count - 1), 50)
    freq = rng.integers(1, 2 * sample_count, n_rows)
    freq[rng.random(n_rows) < 0.15] = sample_count
    zero_rows = np.nonzero(freq == sample_count)[0]
    sign = rng.choice([-1, 1], n_rows)
    sign[zero_rows[::2]] = -1
    for j in zero_rows[::2][:20]:
        rows[j] = np.union1d(rows[j], [sample_count - 1])
    if descending_row:
        j = [q for q in range(n_rows // 2, n_rows) if len(rows[q]) >= 3][0]
        rows[j] = rows[j][::-1].copy()
    idf = np.array([math.log(float(sample_count) / f) for f in freq])     # what morna_idf_host computes
    bucket = rng.choice(np.setdiff1d(np.arange(dim), [9]), size=n_rows)
    nnz = sum(len(r) for r in rows)
    cov = np.where(rng.random(nnz) < 0.2, 2 ** 31 - 1, np.where(rng.random(nnz) < 0.3, 1, rng.integers(1, 5000, nnz)))
    return make(rows, dim, rng, bucket=bucket, sign=sign, idf=idf, cov=cov)


# ------------------------------------------------------------------ what the data asks of the kernels
def _steps(d):
    lens = np.diff(d.row_off)
    rid = np.repeat(np.arange(len(lens)), lens)
    start = np.zeros(len(d.sample), bool)
    start[d.row_off[:-1][lens > 0]] = True
    return rid, start


def ascending(d, passing_only):
    """Every row (every passing row) lists strictly ascending ids: what the warp variant needs."""
    rid, start = _steps(d)
    s = d.sample
    ok = s >= 0
    ok[1:] &= start[1:] | (s[1:] > s[:-1])
    if passing_only:
        ok |= d.passing[rid] == 0
    return bool(ok.all())


def some_row_neither(d):
    """Some passing row is neither strictly ascending nor strictly descending: the barrier variant's atomic form."""
    rid, start = _steps(d)
    idx = np.nonzero(~start)[0]
    idx = idx[idx > 0]
    r, s = rid[idx], d.sample
    n = len(d.passing)
    not_up = np.bincount(r, weights=s[idx] <= s[idx - 1], minlength=n) > 0
    not_down = np.bincount(r, weights=s[idx] >= s[idx - 1], minlength=n) > 0
    return bool((not_up & not_down & (d.passing != 0)).any())


def answered(d, launches, unaligned, pipelined=True):
    """(variant, pre-pass launches) of one morna_index_accumulate call.  Its launches (kernels and CUB passes): 5 for the
    bucket sort; 3 for the warp variant's pre-pass (row-start bits, ascending check, row segments); 5 for its chunk lists
    and index_accumulate3_kernel; 6 for the barrier tail (row lengths, scan, rows_monotonic, both instantiations) or 1
    for the simple kernel.  index_accumulate3_kernel returns at once unless every row ascends (every passing row when the
    sample pointer is not 16-byte aligned), and the barrier kernels return at once when it answered."""
    extra = launches - 5 - (6 if pipelined else 1)
    assert extra in (0, 3, 8), "unexpected launch count %d" % launches
    if extra == 8 and ascending(d, passing_only=unaligned):
        return "warp", extra
    if not pipelined:
        return "simple", extra
    return ("barrier-atomic" if some_row_neither(d) else "barrier"), extra


# ------------------------------------------------------------------ references
def oracle(d):
    lens = np.diff(d.row_off)
    listed = d.sample[np.repeat(d.passing != 0, lens)]
    capacity = max(len(np.unique(listed)), 1)
    id_of, n_kept, acc = c_oracle.index_accumulate(d.row_off, d.passing, d.bucket, d.sign, d.idf, d.sample, d.cov,
                                                   d.dim, d.max_sample_id, capacity)
    return id_of, n_kept, acc


def python_loop(d):
    """morna.py:376-388 written out: first-seen ids, then vector[bucket] += sign * (coverage * idf) with Python floats."""
    id_of, vectors = {}, []
    for j in range(len(d.passing)):
        if not d.passing[j]:
            continue
        idf, sign, b = float(d.idf[j]), int(d.sign[j]), int(d.bucket[j])
        for p in range(int(d.row_off[j]), int(d.row_off[j + 1])):
            s = int(d.sample[p])
            if s not in id_of:
                id_of[s] = len(vectors)
                vectors.append([0.0] * d.dim)
            tfidf = int(d.cov[p]) * idf
            vectors[id_of[s]][b] += sign * tfidf
    return id_of, np.array(vectors, np.float64).reshape(len(vectors), d.dim)


def repeated_cells(d, id_of, n_kept):
    """Cells that get two addends from one row (a row listing a sample twice, in any order: the header leaves their
    order free), and each such cell's sum of |addends| (the scale of a last-ulp difference)."""
    lens = np.diff(d.row_off)
    rid = np.repeat(np.arange(len(lens)), lens)
    keep = d.passing[rid] != 0
    m = d.max_sample_id + 1
    key = rid[keep].astype(np.int64) * m + d.sample[keep]
    u, c = np.unique(key, return_counts=True)
    mask = np.zeros((n_kept, d.dim), bool)
    absum = np.zeros((n_kept, d.dim))
    if not (c > 1).any():
        return mask, absum
    rep = u[c > 1]
    mask[id_of[rep % m], d.bucket[rep // m]] = True
    ids, b = id_of[d.sample[keep]], d.bucket[rid[keep]]
    sel = mask[ids, b]
    np.add.at(absum, (ids[sel], b[sel]), np.abs(d.cov[keep][sel] * d.idf[rid[keep]][sel]))
    return mask, absum


def assert_bits(got, want, what, loose=None, absum=None):
    """got == want bit for bit (+0.0 and -0.0 differ); cells in `loose` may differ by 1e-15 of their sum of |addends|."""
    bad = got.view(np.int64) != want.view(np.int64)
    if loose is not None and loose.any():
        near = bad & loose
        assert np.all(np.abs(got[near] - want[near]) <= 1e-15 * absum[near]), what + ": a repeated-sample cell is off"
        bad &= ~loose
    if bad.any():
        first = [tuple(int(v) for v in c) for c in np.argwhere(bad)[:4]]
        raise AssertionError("%s: %d cells differ, first %s: got %s, want %s" % (
            what, int(bad.sum()), first, [got[c] for c in first], [want[c] for c in first]))


# ------------------------------------------------------------------ the device side
def to_device(d, unaligned=False):
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    g = types.SimpleNamespace(row_off=dev(d.row_off), passing=dev(d.passing), bucket=dev(d.bucket), sign=dev(d.sign),
                              idf=dev(d.idf), cov=dev(d.cov))
    if unaligned:               # a contiguous view 4 bytes into its allocation: the ascending check's unaligned route
        buf = torch.zeros(len(d.sample) + 1, dtype=torch.int32, device="cuda")
        buf[1:] = torch.from_numpy(d.sample)
        g.sample = buf[1:]
        assert g.sample.data_ptr() % 16 == 4
    else:
        g.sample = dev(d.sample if len(d.sample) else np.zeros(1, np.int32))
        assert g.sample.data_ptr() % 16 == 0
    return g


def gpu_ids(lib, d, g, distinct):
    from morna_b200 import _lib
    J, nnz = len(d.passing), len(d.sample)
    id_of = torch.full((d.max_sample_id + 1,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
    n_kept = torch.full((1,), -3, dtype=torch.int32, device="cuda")
    ws = _lib.workspace(lib.morna_assign_internal_ids_workspace_bytes(J, nnz, d.max_sample_id), "cuda")
    _lib.check(lib.morna_assign_internal_ids(_lib.dev_ptr(g.row_off), _lib.dev_ptr(g.passing), J, _lib.dev_ptr(g.sample),
                                             nnz, d.max_sample_id, distinct, _lib.dev_ptr(id_of), _lib.dev_ptr(n_kept),
                                             _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_assign_internal_ids")
    return id_of, int(n_kept.item())


def gpu_accumulate(lib, d, g, id_of, lo, hi, pad=5):
    """The accumulator of ids [lo, hi) in a NaN-filled [dim x (hi - lo + pad)] buffer, and the call's launch count."""
    from morna_b200 import _lib
    J, nnz = len(d.passing), len(d.sample)
    acc_ld = hi - lo + pad
    acc = torch.full((d.dim * acc_ld,), float("nan"), dtype=torch.float64, device="cuda")
    ws = _lib.workspace(lib.morna_index_accumulate_workspace_bytes(J, nnz, d.dim), "cuda")
    l0 = _lib.launch_count()
    _lib.check(lib.morna_index_accumulate(
        _lib.dev_ptr(g.row_off), _lib.dev_ptr(g.passing), _lib.dev_ptr(g.bucket), _lib.dev_ptr(g.sign),
        _lib.dev_ptr(g.idf), J, _lib.dev_ptr(g.sample), _lib.dev_ptr(g.cov), nnz, _lib.dev_ptr(id_of), d.max_sample_id,
        lo, hi, d.dim, _lib.dev_ptr(acc), acc_ld, _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_index_accumulate")
    launches = _lib.launch_count() - l0
    return acc, acc_ld, launches


def check_round_store(lib, acc, acc_ld, width, dim, want32):
    from morna_b200 import _lib
    ld4 = (dim + 3) // 4 * 4
    for ld in (ld4, ld4 + 36):
        vec = torch.full((max(width, 1), ld), float("nan"), dtype=torch.float32, device="cuda")
        _lib.check(lib.morna_round_store(_lib.dev_ptr(acc), acc_ld, width, dim, _lib.dev_ptr(vec), ld, _lib.stream_ptr()),
                   "morna_round_store")
        v = vec[:width].cpu().numpy()
        assert np.array_equal(v[:, :dim].view(np.int32), want32.view(np.int32)), "float32 rows differ (ld %d)" % ld
        assert not v[:, dim:].view(np.int32).any(), "pad columns [dim, ld) are not +0.0 (ld %d)" % ld


def check_build(lib, d, ranges=None, distinct=(0,), unaligned=False, pipelined=True):
    """Runs the three calls on `d` and compares everything with the C oracle; returns answered(...) of the calls."""
    id_o, n_kept_o, acc_o = oracle(d)
    g = to_device(d, unaligned)
    for dc in distinct:
        id_of, n_kept = gpu_ids(lib, d, g, dc)
        assert n_kept == n_kept_o, "n_kept %d, oracle %d (distinct_samples %d)" % (n_kept, n_kept_o, dc)
        assert np.array_equal(id_of.cpu().numpy(), id_o), "id_of_sample differs (distinct_samples %d)" % dc
    loose, absum = repeated_cells(d, id_o, n_kept_o)
    variants = set()
    for lo, hi in ranges or [(0, n_kept_o)]:
        w = hi - lo
        want = np.ascontiguousarray(acc_o[lo:hi].T)
        runs = []
        for _ in range(2):                                   # the same call twice: the same bits
            acc, acc_ld, launches = gpu_accumulate(lib, d, g, id_of, lo, hi)
            variants.add(answered(d, launches, unaligned, pipelined))
            a = acc.view(d.dim, acc_ld).cpu().numpy()
            what = "ids [%d, %d)" % (lo, hi)
            assert_bits(a[:, :w], want, what, loose[lo:hi].T, absum[lo:hi].T)
            assert (a[:, w:].view(np.int64) == NAN_BITS).all(), what + ": a cell past id_hi - id_lo was written"
            runs.append(a[:, :w])
        assert_bits(runs[1], runs[0], "second run of ids [%d, %d)" % (lo, hi), loose[lo:hi].T, absum[lo:hi].T)
        want32 = np.where(loose[lo:hi], runs[0].T, acc_o[lo:hi]).astype(np.float32)
        check_round_store(lib, acc, acc_ld, w, d.dim, want32)
    assert len(variants) == 1, variants
    return variants.pop()


# ------------------------------------------------------------------ 1. the id pass
@pytest.mark.gpu
@pytest.mark.parametrize("early_exit", [1, 0])
@pytest.mark.parametrize("layout", ["late", "early"], ids=["first_seen_after_both_cuts", "all_seen_before_first_cut"])
@pytest.mark.parametrize("m,holes", [(FIRST_POS_SMEM_IDS, False), (FIRST_POS_SMEM_IDS + 1, False), (200000, True)],
                         ids=["smem_table_49152_ids", "global_table_49153_ids", "global_table_200000_ids_with_holes"])
def test_id_pass_first_seen_order(lib, knobs, m, holes, layout, early_exit):
    """first_position_smem_kernel up to 49,152 ids, first_position_kernel above; distinct_samples exact, an over-estimate
    and 0.  With the exact count and key 25 on, the early exit is one id short at both checks ('late': a gate that
    stops one id early loses B) or is met at the first check and skips the later stretches ('early').  A sample listed
    by failing rows only stays -1."""
    knobs(25, early_exit)
    d = id_pass_data(m, holes, layout)
    check_build(lib, d, distinct=(d.distinct, d.distinct + 1, 0))


# ------------------------------------------------------------------ 2. warp-per-range variant
@pytest.mark.gpu
@pytest.mark.parametrize("max_id,shift", [(32767, 10), (32768, 11), (65535, 11), (65536, 12), (131071, 12)])
def test_warp_variant_at_each_range_width(lib, knobs, max_id, shift):
    d = warp_data(max_id)
    assert d.shift == shift and int(((d.bucket == 0) & (d.passing != 0)).sum()) > 2048
    assert check_build(lib, d) == ("warp", 8)


@pytest.mark.gpu
@pytest.mark.parametrize("key12", [10, 11, 12])
def test_warp_variant_range_width_knob(lib, knobs, key12):
    knobs(12, key12)
    assert check_build(lib, warp_data(20000, long_row=3000)) == ("warp", 8)


# ------------------------------------------------------------------ 3. the ascending check
@pytest.mark.gpu
@pytest.mark.parametrize("route", ["aligned", "unaligned"])
@pytest.mark.parametrize("kind", ["equal", "descending"])
@pytest.mark.parametrize("where", ["group", "tail1", "tail2", "tail3", "failing"])
def test_ascending_check_one_violation(lib, knobs, where, kind, route):
    """pairs_ascending_kernel (aligned sample pointer) or rows_monotonic_kernel (4 bytes off) must send a passing row
    with one equal or descending neighbour pair to the barrier variant.  A failing row does not matter to the values:
    the aligned check still counts it (barrier answers), the unaligned one looks at passing rows only (warp answers)."""
    d = ascending_violation_data(where, kind)
    variant, _ = check_build(lib, d, unaligned=route == "unaligned")
    if where == "failing":
        assert variant == ("warp" if route == "unaligned" else "barrier")
    else:
        assert variant == "barrier-atomic"


# ------------------------------------------------------------------ 4. barrier-per-row variants
@pytest.mark.gpu
@pytest.mark.parametrize("kept,tiles", [(ACC2_TILE, 1), (ACC2_TILE + 1, 2), (2 * ACC2_TILE, 2), (2 * ACC2_TILE + 1, 3)])
def test_barrier_variant_id_tiles(lib, knobs, kept, tiles):
    d = tile_data(kept)
    assert oracle(d)[1] == kept and -(-kept // ACC2_TILE) == tiles and 4096 <= len(d.passing) < 64 * d.dim
    assert check_build(lib, d) == ("barrier", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("max_id", [131072, 400000])
def test_barrier_variant_above_131071_ids(lib, knobs, max_id):
    assert check_build(lib, high_id_data(max_id)) == ("barrier", 3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["plain", "atomic"])
@pytest.mark.parametrize("depth", [600, 1100])
def test_barrier_variant_deep_bucket_windows(lib, knobs, depth, kind):
    d = deep_bucket_data(depth, kind)
    assert int(((d.bucket == 2) & (d.passing != 0)).sum()) == depth
    assert check_build(lib, d) == ("barrier" if kind == "plain" else "barrier-atomic", 8)


@pytest.mark.gpu
@pytest.mark.parametrize("key,value,kept,tile,variant", [(4, 0, 2 * ACC2_TILE + 1, 24576, "simple"),
                                                          (7, 2, 30000, 15000, "barrier"), (7, 3, 30000, 10000, "barrier")],
                         ids=["simple_kernel_24576_tiles", "split_2_tiles_of_15000", "split_3_tiles_of_10000"])
def test_barrier_knobs_multi_tile(lib, knobs, key, value, kept, tile, variant):
    """Tuning key 4 = 0 (the simple kernel) and key 7 (id tiles per bucket column), each at a shape where the tile it
    gives differs from the default one (22,528 ids) and there are two or three tiles."""
    if key == 7:          # index_build.cu: tile = min(range, 22528, ceil(range / split))
        assert min(kept, ACC2_TILE, -(-kept // value)) == tile < ACC2_TILE
    knobs(key, value)
    d = tile_data(kept)
    assert oracle(d)[1] == kept and -(-kept // tile) == (value if key == 7 else 2)
    assert check_build(lib, d, pipelined=key != 4) == (variant, 0)


# ------------------------------------------------------------------ 5. id ranges
EDGES = [0, 1, 1023, 1024, 1025, 22527, 22528, 22529]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["warp", "barrier"])
def test_id_ranges_concatenate(lib, knobs, variant):
    """Pieces of the id space with edges at 0, 1, 1023..1025, 22527..22529, n - 1 and n, as multi-GPU shards and query
    slices take them (buckets without rows in every piece), each equal to its slice of the oracle, nothing past it
    written."""
    d = warp_data(30000, long_row=3000) if variant == "warp" else tile_data(30000)
    n = oracle(d)[1]
    edges = sorted(set(EDGES + [n - 1, n]))
    assert check_build(lib, d, ranges=list(zip(edges[:-1], edges[1:])))[0] == variant


@pytest.mark.gpu
def test_empty_id_range_and_no_rows_touch_nothing_past_the_range(lib, knobs):
    from morna_b200 import _lib
    d = warp_data(5000, n_rows=200, deep=50, long_row=1000)
    g = to_device(d)
    id_of, n_kept = gpu_ids(lib, d, g, 0)
    acc, acc_ld, _ = gpu_accumulate(lib, d, g, id_of, 700, 700, pad=9)
    assert (acc.cpu().numpy().view(np.int64) == NAN_BITS).all(), "an empty id range wrote cells"
    acc = torch.full((d.dim * 12,), float("nan"), dtype=torch.float64, device="cuda")
    ws = _lib.workspace(lib.morna_index_accumulate_workspace_bytes(0, 0, d.dim), "cuda")
    _lib.check(lib.morna_index_accumulate(
        _lib.dev_ptr(g.row_off), _lib.dev_ptr(g.passing), _lib.dev_ptr(g.bucket), _lib.dev_ptr(g.sign),
        _lib.dev_ptr(g.idf), 0, _lib.dev_ptr(g.sample), _lib.dev_ptr(g.cov), 0, _lib.dev_ptr(id_of), d.max_sample_id,
        3, 10, d.dim, _lib.dev_ptr(acc), 12, _lib.dev_ptr(ws), ws.numel(), _lib.stream_ptr()), "morna_index_accumulate")
    a = acc.view(d.dim, 12).cpu().numpy()
    assert not a[:, :7].view(np.int64).any(), "no rows: cells [0, id_hi - id_lo) must be +0.0"
    assert (a[:, 7:].view(np.int64) == NAN_BITS).all(), "no rows: a cell past id_hi - id_lo was written"


# ------------------------------------------------------------------ 6. values
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["warp", "barrier"])
def test_extreme_values_and_signed_zeros(lib, knobs, variant):
    d = values_data(descending_row=variant == "barrier")
    assert (d.idf == 0).any() and (d.idf < 0).any() and (d.cov == 2 ** 31 - 1).any() and (d.cov == 1).any()
    assert check_build(lib, d)[0] == variant


# ------------------------------------------------------------------ 7. determinism
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["warp", "barrier-atomic"])
def test_default_path_repeats_bit_for_bit(lib, knobs, variant):
    """Three more runs of a default-path case give the first run's bits (check_build already runs every case twice);
    for the atomic form only cells without a repeated sample are fixed."""
    d = warp_data(40000, long_row=3000) if variant == "warp" else deep_bucket_data(1100, "atomic")
    assert check_build(lib, d)[0] == variant
    id_o, n_kept, _ = oracle(d)
    loose, _ = repeated_cells(d, id_o, n_kept)
    g = to_device(d)
    id_of, _ = gpu_ids(lib, d, g, 0)
    runs = [gpu_accumulate(lib, d, g, id_of, 0, n_kept)[0].cpu().numpy() for _ in range(3)]
    keep = np.pad(~loose.T, ((0, 0), (0, 5)), constant_values=True).ravel()
    for r in runs[1:]:
        assert np.array_equal(r.view(np.int64)[keep], runs[0].view(np.int64)[keep])


# ------------------------------------------------------------------ 8. end to end through MornaIndex
@pytest.mark.gpu
@pytest.mark.parametrize("features,n_samples,n_rows,mean_len", [(3000, 21504, 4000, 700), (30000, 3000, 6000, 450)],
                         ids=["features_3000_21504_samples", "features_30000_3000_samples"])
def test_morna_index_build_equals_c_oracle(lib, knobs, features, n_samples, n_rows, mean_len):
    """A few million pairs through MornaIndex.build (hash, idf, ids, scatter-add, float32 store).  At 3,000 features and
    fewer than 4,096 rows the warp variant answers; at 30,000 features (fewer than 64 rows a bucket) the barrier one."""
    from morna_b200 import _lib
    from morna_b200.index import MornaIndex
    rng = np.random.default_rng(features)
    threshold = 100
    idx = MornaIndex(n_samples, "unused", dim=features, sample_threshold=threshold)
    keys, rows, covs, passing, running, freq = [], [], [], [], [], {}
    universe = np.arange(1, n_samples + 1)
    for j, row in enumerate(random_rows(rng, n_rows, universe, mean_len)):
        key = keys[int(rng.integers(0, j))] if j > 10 and j % 7 == 3 else "chr%d %d %d" % (j % 22 + 1, 1000 + 7 * j, 1900 + 7 * j)
        cov = 1 + rng.geometric(0.4, len(row)) * rng.integers(1, 30, len(row))
        ok = len(row) >= threshold
        if ok:
            freq[key] = freq.get(key, 0) + len(row)           # morna.py:365
        idx._rows.add(key, row, cov)
        idx._pass.append(int(ok)); idx._running_freq.append(freq[key] if ok else 0)
        keys.append(key); rows.append(row); covs.append(cov); passing.append(ok); running.append(freq[key] if ok else 0)
    idx.build()
    assert (n_rows < 4096) == (features == 3000) and n_rows // features < 64
    idf = np.empty(n_rows)
    pas, running = np.array(passing, np.uint8), np.array(running, np.int64)      # (held: the call takes raw pointers)
    _lib.check(lib.morna_idf_host(running.ctypes.data, pas.ctypes.data, n_rows, n_samples, idf.ctypes.data),
               "morna_idf_host")
    _, bucket, sign = c_oracle.hash_rows(keys, features)
    d = make(rows, features, rng, bucket=bucket, sign=sign, idf=idf, passing=pas, cov=np.concatenate(covs))
    assert d.row_off[-1] > 2_000_000
    id_o, n_kept, acc_o = oracle(d)
    assert idx.internal_id_map == {int(s): int(id_o[s]) for s in np.nonzero(id_o >= 0)[0]}
    assert_bits(idx.accumulator_f64(), acc_o, "accumulator_f64")
    assert np.array_equal(idx.matrix_f32().view(np.int32), acc_o.astype(np.float32).view(np.int32))


# ------------------------------------------------------------------ the reference itself (host only)
SMALL_CASES = {
    "id_pass_late": lambda: id_pass_data(600, False, "late", n_rows=640),
    "id_pass_early": lambda: id_pass_data(600, False, "early", n_rows=640),
    "id_pass_holes": lambda: id_pass_data(20000, True, "late", n_rows=640),
    "warp": lambda: warp_data(5000, n_rows=200, deep=60, long_row=1500),
    "ascending_equal_tail3": lambda: ascending_violation_data("tail3", "equal", n_rows=120),
    "ascending_descending_group": lambda: ascending_violation_data("group", "descending", n_rows=120),
    "ascending_equal_failing": lambda: ascending_violation_data("failing", "equal", n_rows=120),
    "tiles": lambda: tile_data(700, n_rows=150, dim=12),
    "high_ids": lambda: high_id_data(400000, n_rows=60, n_ids=900),
    "deep_bucket_plain": lambda: deep_bucket_data(600, "plain", others=40),
    "deep_bucket_atomic": lambda: deep_bucket_data(1100, "atomic", others=40),
    "values": lambda: values_data(False, n_rows=200),
}


@pytest.mark.parametrize("case", sorted(SMALL_CASES))
def test_c_oracle_matches_python_loop_on_the_edge_inputs(case):
    """The C oracle that the GPU tests above trust, against morna.py's loop written out in Python, on a small instance of
    each input generator (repeated samples, idf 0 with negative signs, 2^31 - 1 coverages, ids in failing rows only)."""
    d = SMALL_CASES[case]()
    id_o, n_kept, acc_o = oracle(d)
    ids, vectors = python_loop(d)
    assert n_kept == len(ids)
    assert {int(s): int(id_o[s]) for s in np.nonzero(id_o >= 0)[0]} == ids
    assert_bits(acc_o, vectors, case)
