"""Steady-state CUDA-graph replay of the query pipeline, and every branch of the batched path's candidate selection
(kth_warp_kernel), against the exact FP64 scan (ids and distance bits) and the C oracle.

Part A drives MornaSearch.search_batches / BatchPipeline past its first two batches per slot, into the replay-only state
that the benchmark times.  Part B builds inputs that push the k-th selection off its fast path: a lane's survivor list
overflowing, a pivot that misses, a cut below the pivot, candidate lists longer than their caps, the best rows scored
last, exact ties at the cut, and row shards smaller than k.  Where a case exists to reach a regime, it also checks that
the regime was reached, from the search's stats or from the fp16 scores themselves.
"""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests.helpers import assert_lists_equal_oracle

pytestmark = pytest.mark.gpu

# morna_debug_set_tuning keys this file changes, with their defaults: rows per block between two refinements (9), pilot
# rows (10), rows up to the first refinement (11, 0 = key 9), growth factor of the blocks after the first (36)
KNOB_DEFAULTS = {9: 131072, 10: 8192, 11: 0, 36: 1}
CAND_CAP, FIN_CAP, LANE_SLOTS = 4096, 1024, 32       # kCandCap, kFinCap, kKwSlots of search_batched.cu


@pytest.fixture
def knobs():
    """set(key, value) for the knobs above; every one of them is back at its default after the test, pass or fail (they
    are process-wide)."""
    from morna_b200 import _lib
    lib = _lib.load()

    def set_knob(key, value):
        assert key in KNOB_DEFAULTS
        assert lib.morna_debug_set_tuning(key, value) == 0

    try:
        yield set_knob
    finally:
        for key, value in KNOB_DEFAULTS.items():
            lib.morna_debug_set_tuning(key, value)


@pytest.fixture
def replays(monkeypatch):
    """Counts torch.cuda.CUDAGraph.replay calls (a list that grows by one per replay)."""
    calls = []
    original = torch.cuda.CUDAGraph.replay

    def counted(self):
        calls.append(1)
        return original(self)

    monkeypatch.setattr(torch.cuda.CUDAGraph, "replay", counted)
    return calls


def make_search(S, **kw):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=S, stats=(S.shape[0], S.shape[0], S.shape[1]), **kw)


def exact(srch, Q, k):
    """The FP64 scan's answer for host queries (float32 widens exactly), as numpy."""
    ids, d = srch.exact_search_device(torch.from_numpy(np.asarray(Q, dtype=np.float64)).cuda(), k, allow_single=False)
    return ids.cpu().numpy(), d.cpu().numpy()


def check_batched(srch, S, Q, k, label, oracle_rows=(0,)):
    """batched_search_device == exact scan bit for bit, the given queries also == the oracle; returns last_stats
    = [overflowed queries, first-pass survivors, re-ranked sum, re-ranked max]."""
    q = torch.from_numpy(Q).cuda()
    ids, d = srch.batched_search_device(q, k)
    stats = list(srch.last_stats)
    e_ids, e_d = srch.exact_search_device(q, k, allow_single=False)
    assert torch.equal(ids, e_ids), "%s: ids differ from the exact scan" % label
    assert torch.equal(d, e_d), "%s: distances differ from the exact scan" % label
    pick = np.asarray(oracle_rows)
    assert_lists_equal_oracle(S, Q[pick], ids.cpu().numpy()[pick], d.cpu().numpy()[pick], k, label)
    return stats


def unit(v):
    return v / np.linalg.norm(v)


def rows_at_cosines(u, cos, rng):
    """float32 rows whose cosine to the unit vector u is `cos` (each row: cos * u + sqrt(1 - cos^2) * a random unit
    vector orthogonal to u, times a random scale)."""
    w = rng.standard_normal((len(cos), u.shape[0]))
    w -= (w @ u)[:, None] * u[None, :]
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    rows = cos[:, None] * u[None, :] + np.sqrt(1.0 - cos ** 2)[:, None] * w
    return (rows * np.exp(0.3 * rng.standard_normal((len(cos), 1)))).astype(np.float32)


def near(u, m, rng, noise=1e-4):
    """m queries within `noise` (relative) of the direction u."""
    return u[None, :] + noise * rng.standard_normal((m, u.shape[0])) / math.sqrt(u.shape[0])


def tensor_scores(srch, Q):
    """The fp16 first pass's scores (float32 [nq x n]) and error bounds eps (float32 [nq]) of host queries Q."""
    from morna_b200 import _lib
    lib = _lib.load()
    srch.enable_tensor_path()
    n, d = srch.row_hi - srch.row_lo, srch.dim
    q = torch.from_numpy(np.asarray(Q, dtype=np.float64)).cuda()
    nq, ld_s = q.shape[0], (n + 3) // 4 * 4
    scores = torch.zeros((nq, ld_s), dtype=torch.float32, device="cuda")
    eps = torch.zeros(nq, dtype=torch.float32, device="cuda")
    ws = _lib.workspace(lib.morna_knn_batched_workspace_bytes(n, nq, d, 10), "cuda")
    assert lib.morna_debug_tensor_scores(_lib.dev_ptr(srch.hs), srch.ld_h, _lib.dev_ptr(srch.rho_max), n, d, _lib.dev_ptr(q),
                                         nq, d, _lib.dev_ptr(scores), ld_s, _lib.dev_ptr(eps), _lib.dev_ptr(ws), ws.numel(),
                                         _lib.stream_ptr()) == 0
    return scores.cpu().numpy()[:, :n], eps.cpu().numpy()


def pilot_pass(scores, eps, k, n0=8192):
    """What kth_warp_kernel's pilot pass sees for one query: the pivot from its 512 strided samples, the survivors per
    lane (lane of entry i = (i // 4) % 32), the k-th largest score a_k and the cut a_k - 2 eps."""
    s = scores[:n0].astype(np.float32)
    kk = min(k, n0)
    assert n0 > 32 * LANE_SLOTS, "no pivot below 1025 entries"
    stride = n0 >> 9
    want = np.float32(kk) * np.float32(512.0) / np.float32(n0)
    r = int(want + np.float32(4.0) * np.sqrt(want) + np.float32(4.0))
    pivot = np.sort(s[np.arange(512) * stride])[::-1][r - 1]
    surv = s >= pivot
    per_lane = np.bincount(((np.arange(n0) // 4) % 32)[surv], minlength=32)
    a_k = float(np.sort(s)[::-1][kk - 1])
    return dict(pivot=float(pivot), survivors=int(surv.sum()), lane_max=int(per_lane.max()), kk=kk, a_k=a_k,
                cut=a_k - 2.0 * float(eps))


# ================================================================== A. the query pipeline and its graph replay
N_A, D_A, K_A, NQ_A = 6000, 96, 20, 300


@pytest.fixture(scope="module")
def pipe_data():
    rng = np.random.default_rng(2024)
    S = rng.standard_normal((N_A, D_A)).astype(np.float32)
    S[10:13] = S[9]                                          # a few exact ties
    batches = []
    for b in range(10):
        Q = S[rng.permutation(N_A)[:NQ_A]] + np.float32(0.03) * rng.standard_normal((NQ_A, D_A)).astype(np.float32)
        Q[b] = S[9]
        batches.append(Q)
    return S, batches


def run_pipeline(srch, batches, k, depth):
    return [(i.copy(), d.copy(), list(srch.last_stats or [])) for i, d in srch.search_batches(iter(batches), k, depth=depth)]


def assert_batches_exact(srch, batches, got, k, label):
    assert len(got) == len(batches)
    for j, (B, (gi, gd, _)) in enumerate(zip(batches, got)):
        wi, wd = exact(srch, np.asarray(B.cpu() if isinstance(B, torch.Tensor) else B), k)
        assert np.array_equal(gi, wi), "%s: batch %d ids differ from the exact scan" % (label, j)
        assert np.array_equal(gd, wd), "%s: batch %d distances differ from the exact scan" % (label, j)


@pytest.mark.parametrize("source", ["pageable", "pinned", "mixed_dtypes"])
@pytest.mark.parametrize("depth", [1, 2, 3])
def test_steady_state_replay_answers_every_batch(pipe_data, replays, depth, source):
    """Ten batches of one size with different contents: each slot runs plain launches, then captures its graph, then
    only replays it.  The replay must read the slot's new queries and hand back its new lists every time.  Sources:
    pageable numpy, caller-pinned torch tensors (copied straight from the caller's buffer) and float32 / float64 batches
    mixed within each slot (the dtype is not part of the graph key)."""
    S, batches = pipe_data
    if source == "pinned":
        batches = [torch.from_numpy(B).pin_memory() for B in batches]
    elif source == "mixed_dtypes":
        batches = [B.astype(np.float64) if (j // depth) % 2 else B for j, B in enumerate(batches)]
    srch = make_search(S)
    got = run_pipeline(srch, batches, K_A, depth)
    assert len(replays) >= len(batches) - 2 * depth, "only %d graph replays" % len(replays)
    assert all(st[0] == 0 for _, _, st in got)
    assert_batches_exact(srch, batches, got, K_A, "%s depth %d" % (source, depth))
    assert_lists_equal_oracle(S, np.asarray(batches[-1], dtype=np.float64)[:4], got[-1][0][:4], got[-1][1][:4], K_A,
                              "last replayed batch")


def test_device_resident_batches_in_distinct_buffers(pipe_data):
    """Queries already in HBM are used in place: batches of one size in different device buffers must not be answered
    by a graph captured on another buffer's address."""
    S, batches = pipe_data
    srch = make_search(S)
    dev = [torch.from_numpy(B.astype(np.float64)).cuda() for B in batches]
    got = run_pipeline(srch, dev, K_A, 2)
    assert_batches_exact(srch, batches, got, K_A, "device-resident")


def test_graphs_on_and_off_give_the_same_bits_and_launch_count(pipe_data, replays, monkeypatch):
    """The same batches with graphs (captured once per slot, replayed after) and with plain launches: identical lists,
    and the library's launch counter (kernels that ran, replays included) moves by the same amount."""
    from morna_b200 import _lib
    from morna_b200.search import BatchPipeline
    S, batches = pipe_data
    srch = make_search(S)
    srch.enable_tensor_path()
    monkeypatch.setattr(BatchPipeline, "use_graphs", False)
    run_pipeline(srch, batches[:2], K_A, 2)          # one-time set-up of the batched path happens before counting
    runs = []
    for graphs in (True, False):
        monkeypatch.setattr(BatchPipeline, "use_graphs", graphs)
        srch._pipes = {}                             # pipelines are kept per (k, depth): start from a fresh one
        launches0 = _lib.launch_count()
        got = run_pipeline(srch, batches, K_A, 2)
        runs.append((got, _lib.launch_count() - launches0, len(replays)))
    (g_on, l_on, r_on), (g_off, l_off, r_off) = runs
    assert r_on >= len(batches) - 4 and r_off == r_on, "graphs off must not replay (%d / %d)" % (r_on, r_off)
    for (ai, ad, _), (bi, bd, _) in zip(g_on, g_off):
        assert np.array_equal(ai, bi) and np.array_equal(ad, bd)
    assert l_on == l_off and l_on > 0, "launch count with graphs %d, without %d" % (l_on, l_off)
    assert_batches_exact(srch, batches, g_on, K_A, "graphs on")


def test_overflow_fix_up_in_a_replayed_batch(pipe_data, replays):
    """A replay-only batch with an all-zero query and one whose values exceed 2^127 (both overflow: every row ties / the
    scaled re-rank would overflow): collect() patches them with the exact scan.  The next replay of that slot must
    overwrite the patched rows again."""
    S, batches = pipe_data
    batches = [B.astype(np.float64) for B in batches]
    batches[6][3] = 0.0                              # depth 2: batches 4, 6 and 8 of slot 0 are replay-only
    batches[6][7, 5] = 3e38
    srch = make_search(S)
    got = run_pipeline(srch, batches, K_A, 2)
    assert len(replays) >= len(batches) - 4
    assert [st[0] for _, _, st in got] == [0] * 6 + [2] + [0] * 3
    assert_batches_exact(srch, batches, got, K_A, "overflow fix-up")


def test_pipelines_reused_across_calls(pipe_data, replays):
    """A second search_batches call reuses the first call's pipeline, whose slots already hold their graphs: its first
    batches go straight to replay -- after a direct batched_search_device call has run on another workspace."""
    S, batches = pipe_data
    srch = make_search(S)
    first = run_pipeline(srch, batches[:6], K_A, 2)
    n_first = len(replays)
    assert n_first >= 2
    q = torch.from_numpy(batches[9].astype(np.float64)).cuda()
    b_ids, b_d = srch.batched_search_device(q, K_A)
    e_ids, e_d = srch.exact_search_device(q, K_A, allow_single=False)
    assert torch.equal(b_ids, e_ids) and torch.equal(b_d, e_d)
    second = run_pipeline(srch, batches[4:], K_A, 2)
    assert len(replays) - n_first == len(batches[4:]), "the second call's batches must all be replays"
    assert_batches_exact(srch, batches[:6], first, K_A, "first call")
    assert_batches_exact(srch, batches[4:], second, K_A, "second call")


@pytest.mark.parametrize("shard", [None, (1, 2)])
def test_queries_by_id_resident_and_not(pipe_data, shard):
    """search -q: stored rows named by internal id are the queries.  Resident ids are answered like their rows; ids
    outside this shard's rows are refused (host and device ids), before they could index the wrong row."""
    S, _ = pipe_data
    srch = make_search(S, shard=shard)
    lo, hi = srch.row_lo, srch.row_hi
    rng = np.random.default_rng(5)
    ids = [np.concatenate([[lo, hi - 1], rng.integers(lo, hi, size=62)]).astype(np.int64) for _ in range(5)]
    batches = [ids[0], ids[1].astype(np.int32), torch.from_numpy(ids[2]).cuda(), ids[3], ids[4]]
    got = run_pipeline(srch, batches, K_A, 2)
    for j, (i_, (gi, gd, _)) in enumerate(zip(ids, got)):
        wi, wd = exact(srch, S[i_], K_A)
        assert np.array_equal(gi, wi) and np.array_equal(gd, wd), "by-id batch %d" % j
    bad = [np.array([hi], np.int64), np.array([lo, hi + 5], np.int64)]
    if lo > 0:
        bad += [np.array([lo - 1], np.int64), np.array([0, lo + 3], np.int64)]
    bad += [torch.from_numpy(b).cuda() for b in bad]
    for b in bad:
        with pytest.raises(ValueError, match="not all resident"):
            run_pipeline(srch, [ids[0], b], K_A, 2)
    got = run_pipeline(srch, [ids[0]], K_A, 2)       # a refused batch leaves nothing broken behind
    assert np.array_equal(got[0][0], exact(srch, S[ids[0]], K_A)[0])


# ================================================================== B. candidate selection on adversarial inputs
def background(n, d, rng):
    return rng.standard_normal((n, d)).astype(np.float32)


def test_lane_list_overflow_takes_the_bisection():
    """48 near-copies of query 0 in the pilot block, all at entries of lane 1 ((i // 4) % 32 == 1) that the pivot never
    samples (the samples are every 16th entry): the pivot stays at the Gaussian background's level, lane 1 collects more
    than its 32 list slots, and the k-th largest must come from the streaming bisection over all entries."""
    rng = np.random.default_rng(101)
    n, d, k = 20000, 64, 64
    S = background(n, d, rng)
    Q = rng.standard_normal((16, d))
    at = (4 + 128 * np.arange(12)[:, None] + np.arange(4)[None, :]).ravel()
    assert np.all((at // 4) % 32 == 1) and np.all(at % 16 != 0) and at.max() < 8192
    S[at] = (Q[0][None, :] + 1e-3 * rng.standard_normal((len(at), d))).astype(np.float32)
    srch = make_search(S)
    scores, eps = tensor_scores(srch, Q[:1])
    pp = pilot_pass(scores[0], eps[0], k)
    assert pp["lane_max"] > LANE_SLOTS and pp["survivors"] >= k, pp
    assert pp["cut"] >= pp["pivot"], pp            # a list-based emit would be taken, were the lists complete
    stats = check_batched(srch, S, Q, k, "lane overflow", oracle_rows=(0, 5))
    assert stats[0] == 0
    ids = exact(srch, Q[:1], k)[0][0]
    assert set(at.tolist()) <= set(ids.tolist())   # every planted copy is among query 0's neighbours


def test_pivot_miss_takes_the_bisection():
    """Every sampled pilot entry (i % 16 == 0, 512 rows) is planted with a cosine in [0.90, 0.99] to query 0, the rest is
    Gaussian background: the pivot (about the 20th sample) lets only ~20 entries through, fewer than k = 100, and the
    k-th largest must come from the bisection.  The planted cosines are graded, so a cut taken from the survivors alone
    would sit above the 100th planted row and lose rows."""
    rng = np.random.default_rng(202)
    n, d, k = 20000, 64, 100
    S = background(n, d, rng)
    Q = rng.standard_normal((16, d))
    at = np.arange(0, 8192, 16)
    S[at] = rows_at_cosines(unit(Q[0]), rng.permutation(np.linspace(0.99, 0.90, len(at))), rng)
    srch = make_search(S)
    scores, eps = tensor_scores(srch, Q[:1])
    pp = pilot_pass(scores[0], eps[0], k)
    assert pp["survivors"] < k and pp["lane_max"] <= LANE_SLOTS, pp
    stats = check_batched(srch, S, Q, k, "pivot miss", oracle_rows=(0, 3))
    assert stats[0] == 0


def dense_cluster(n, d, m, width, rng, top=0.9):
    """n rows: m of them (at random positions) with cosines uniform in [top - width, top] to a direction u, the rest
    Gaussian-like around it (cosines uniform in [-0.5, 0.5]).  Returns rows, u."""
    u = unit(rng.standard_normal(d))
    cos = rng.uniform(-0.5, 0.5, n)
    cos[rng.permutation(n)[:m]] = top - width * rng.random(m)
    return rows_at_cosines(u, cos, rng), u


def eps_of(d, seed):
    """The first pass's error bound for queries near a direction, on a probe of the same construction."""
    rng = np.random.default_rng(seed)
    S, u = dense_cluster(2048, d, 512, 0.01, rng)
    return float(tensor_scores(make_search(S), near(u, 1, rng))[1][0])


def test_cut_below_the_pivot_re_streams_the_pilot():
    """2000 of 9000 rows within ~7 eps of each other in cosine: about 500 pilot entries lie within 2 eps below the k-th,
    more than pass the pivot (~320), so the pilot's emit re-streams every entry; the final lists stay under their cap
    of 1024 with 400+ re-ranked rows (no overflow)."""
    rng = np.random.default_rng(303)
    n, d, k, m = 9000, 128, 100, 2000
    e = eps_of(d, 1)
    S, u = dense_cluster(n, d, m, m * 2 * e / 550, rng)
    Q = np.concatenate([near(u, 8, rng), rng.standard_normal((8, d))])
    srch = make_search(S)
    scores, eps = tensor_scores(srch, Q[:1])
    pp = pilot_pass(scores[0], eps[0], k)
    assert pp["cut"] < pp["pivot"] and pp["survivors"] >= k and pp["lane_max"] <= LANE_SLOTS, pp
    stats = check_batched(srch, S, Q, k, "cut below pivot", oracle_rows=(0, 7, 8))
    assert stats[0] == 0 and 400 <= stats[3] <= FIN_CAP, stats


def test_final_list_overflow_goes_to_the_exact_scan():
    """3000 of 9000 rows within ~3 eps of each other: ~2000 rows lie within 2 eps of the k-th score, more than the final
    list's 1024 slots but fewer than the first-pass cap of 4096 -- the final pass marks the query overflowed and the
    exact scan answers it."""
    rng = np.random.default_rng(404)
    n, d, k, m = 9000, 128, 100, 3000
    e = eps_of(d, 2)
    S, u = dense_cluster(n, d, m, m * 2 * e / 1900, rng)
    Q = np.concatenate([near(u, 8, rng), rng.standard_normal((8, d))])
    srch = make_search(S)
    scores, eps = tensor_scores(srch, Q[:1])
    s = scores[0]
    a_k = float(np.sort(s)[::-1][k - 1])
    pp = pilot_pass(s, eps[0], k)
    assert (s >= a_k - 2 * eps[0]).sum() > FIN_CAP and (s >= pp["cut"]).sum() < CAND_CAP
    stats = check_batched(srch, S, Q, k, "final overflow", oracle_rows=(0, 9))
    assert stats[0] == 8, stats                      # every query near u, none of the Gaussian ones


def tied_cluster(n, d, rng, spread):
    """n rows whose cosines to u all lie within `spread` of 0.9."""
    u = unit(rng.standard_normal(d))
    return rows_at_cosines(u, 0.9 - spread * rng.random(n), rng), u


@pytest.mark.parametrize("block_rows", [256, 1024, 131072])
def test_first_pass_cap_overflow_at_pilot_and_refine(knobs, block_rows):
    """20,000 rows whose cosines to the queries all lie within eps / 4 of each other: every entry survives every cut.
    With the default blocks the pilot's 8192 survivors exceed the first-pass cap (4096); with 256- or 1024-row blocks
    the list grows by a block per refinement until a refine pass finds it over the cap.  Either way the query is
    marked overflowed and answered by the exact scan -- and only those queries: blocks no longer than the pilot used to
    skip every refinement, so the Gaussian queries' lists were filtered by the threshold of 256 rows alone and some of
    them overflowed too."""
    knobs(9, block_rows)
    rng = np.random.default_rng(505)
    n, d, k = 20000, 64, 50
    e = eps_of(d, 3)
    S, u = tied_cluster(n, d, rng, e / 4)
    Q = np.concatenate([rng.standard_normal((16, d)), near(u, 16, rng, 1e-5)])       # (overflowing queries last)
    srch = make_search(S)
    stats = check_batched(srch, S, Q, k, "cap overflow", oracle_rows=(0, 16))
    assert stats[0] == 16, stats


def test_refine_pass_cap_overflow_with_spread_scores(knobs):
    """A pilot of 256 far rows gives a loose threshold; the next 5744 rows (the first refine block) all pass it, so the
    refine pass finds more entries than the cap kept -- and the true neighbours are among them, spread over the block.
    The query must go to the exact scan rather than be answered from the part of the list that was kept."""
    knobs(10, 256)
    knobs(11, 6000)
    rng = np.random.default_rng(606)
    n, d, k = 12000, 64, 50
    u = unit(rng.standard_normal(d))
    cos = np.concatenate([rng.uniform(-0.2, 0.0, 256), rng.uniform(0.3, 0.95, 6000 - 256), rng.uniform(-0.2, 0.2, n - 6000)])
    S = rows_at_cosines(u, cos, rng)
    Q = np.concatenate([rng.standard_normal((16, d)), near(u, 16, rng, 1e-3)])       # (overflowing queries last)
    srch = make_search(S)
    stats = check_batched(srch, S, Q, k, "refine cap overflow", oracle_rows=(0, 16, 31))
    assert stats[0] >= 16, stats


# key 9 (block rows), key 11 (rows before the first refinement), key 36 (block growth), key 10 (pilot rows), k: a pruned
# product in which every pair of settings of two different knobs meets; the last two have a pilot shorter than k
BEST_LAST = [(256, 0, 1, 256, 50), (256, 300, 2, 1000, 50), (256, 5000, 8, 8192, 50),
             (1024, 0, 2, 8192, 50), (1024, 300, 8, 256, 50), (1024, 5000, 1, 1000, 50),
             (131072, 0, 8, 1000, 50), (131072, 300, 1, 8192, 50), (131072, 5000, 2, 256, 50),
             (256, 0, 1, 256, 512), (256, 300, 2, 256, 512)]


@pytest.mark.parametrize("block_rows,first_block,growth,pilot_rows,k", BEST_LAST)
def test_best_rows_last(knobs, block_rows, first_block, growth, pilot_rows, k):
    """Rows in increasing cosine to the queries' direction: the pilot holds only the far rows and every later block
    beats everything before it, so each refinement must tighten the threshold again.  Block sizes, the first block,
    block growth and pilot size change no bit."""
    for key, val in ((9, block_rows), (11, first_block), (36, growth), (10, pilot_rows)):
        knobs(key, val)
    rng = np.random.default_rng(707)
    n, d = 16000, 64
    u = unit(rng.standard_normal(d))
    S = rows_at_cosines(u, np.sort(rng.uniform(-0.5, 0.95, n)), rng)
    Q = np.concatenate([rng.standard_normal((8, d)), near(u, 8, rng, 3e-2)])
    srch = make_search(S)
    check_batched(srch, S, Q, k, "best rows last %r" % ((block_rows, first_block, growth, pilot_rows, k),),
                  oracle_rows=(0, 8))


@pytest.mark.parametrize("where", ["inside_a_block", "across_blocks", "across_the_pilot"])
def test_exact_ties_at_the_kth_place(knobs, where):
    """k - 1 rows clearly closest to the query, then a row and its exact copies: the k-th and (k+1)-th candidates have
    the same fp16 score and the same distance.  Both must survive to the re-rank, which puts the larger id first --
    copies next to each other in one block, on both sides of a block boundary, and on both sides of the pilot's end."""
    knobs(9, 1024)
    knobs(10, 1024)
    rng = np.random.default_rng({"inside_a_block": 1, "across_blocks": 2, "across_the_pilot": 3}[where])
    n, d, k = 12000, 64, 50
    S = background(n, d, rng)
    Q = rng.standard_normal((8, d))
    copies = {"inside_a_block": [5000, 5001], "across_blocks": [6143, 6144, 6145], "across_the_pilot": [1023, 1024]}[where]
    u = unit(Q[0])
    better = rng.permutation(np.setdiff1d(np.arange(n), copies))[:k - 1]
    S[better] = rows_at_cosines(u, np.linspace(0.95, 0.9, k - 1), rng)
    S[copies] = rows_at_cosines(u, np.array([0.85]), rng)[0]
    srch = make_search(S)
    scores, _ = tensor_scores(srch, Q[:1])
    assert len(set(scores[0][copies].tolist())) == 1 and np.sort(scores[0])[::-1][k - 1] == scores[0][copies[0]]
    check_batched(srch, S, Q, k, "ties " + where, oracle_rows=(0, 1))
    ids = exact(srch, Q[:1], k)[0][0]
    assert ids[k - 1] == max(copies)


def sharded_bound_search(S, q, k, world):
    """The rows-sharded search with its two exchange steps emulated in one process (bounds, union, finish, merge)."""
    from morna_b200 import dist as mdist
    shards = [make_search(S, shard=(r, world)) for r in range(world)]
    vals = torch.stack([sh.batched_score_bound(q, k) for sh in shards])
    bound = shards[0].union_kth_bound(vals, k)
    parts = [sh.batched_finish_bound(bound.clone()) for sh in shards]
    ids, dist = mdist.merge_sorted_lists(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
    return shards, vals, ids, dist


@pytest.mark.parametrize("n,world,k,kind", [(1700, 8, 210, "gauss"), (1500, 8, 200, "gauss"), (20000, 3, 50, "tied")])
def test_sharded_bound_path_with_small_or_overflowing_shards(n, world, k, kind):
    """Rows-sharded bound path: the last shard holds fewer than k rows (1700 / 8, k = 210), every shard does (1500 / 8,
    k = 200) -- such a shard answers by the exact scan and contributes only -inf bounds -- or every shard overflows
    for the queries whose rows all tie within eps.  The merged lists are the unsharded answer and the oracle's."""
    rng = np.random.default_rng(n + world)
    d = 64
    if kind == "tied":
        S, u = tied_cluster(n, d, rng, eps_of(d, 4) / 4)
        Q = np.concatenate([near(u, 8, rng, 1e-5), rng.standard_normal((8, d))])
    else:
        S = background(n, d, rng)
        S[100:103] = S[99]
        S[n - 2] = S[99]                                     # ties inside and across shards
        Q = S[rng.permutation(n)[:40]].astype(np.float64) + 0.05 * rng.standard_normal((40, d))
        Q[0] = S[99]
    q = torch.from_numpy(Q).cuda()
    whole = make_search(S)
    w_ids, w_d = whole.batched_search_device(q, k)
    e_ids, e_d = whole.exact_search_device(q, k, allow_single=False)
    assert torch.equal(w_ids, e_ids) and torch.equal(w_d, e_d)
    shards, vals, ids, dist = sharded_bound_search(S, q, k, world)
    small = [r for r, sh in enumerate(shards) if sh.row_hi - sh.row_lo < k]
    for r in small:
        assert bool(torch.isinf(vals[r]).all() and (vals[r] < 0).all()), "a shard smaller than k must give -inf bounds"
    if kind == "tied":
        assert all(sh.last_stats[0] > 0 for sh in shards), [sh.last_stats for sh in shards]
    else:
        assert small and (len(small) == world) == (n == 1500)
    assert torch.equal(ids, w_ids) and torch.equal(dist, w_d)
    pick = np.array([0, 1, 9])
    assert_lists_equal_oracle(S, Q[pick], ids.cpu().numpy()[pick], dist.cpu().numpy()[pick], k, "sharded %d / %d" % (n, world))
