"""Rows-sharded range search on the GPU: morna_merge_sorted_csr against a numpy merge bit for bit, the whole protocol
emulated in one process over G shards of one matrix (every shard counts and writes its own lists, the step after the
all-gather is fed with their packed buffers), and the NCCL run with two ranks.  Results must equal the unsharded
range_search_device and the brute-force lists of test_gpu_range_search.py, in offsets, ids and distance bits."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import dist as mdist, synth
from morna_b200.search import _range_groups
from tests.test_dist_range_gloo import _ordered, numpy_merge
from tests.test_gpu_range_search import assert_csr_equal, brute, distances, host, make_search, median_kth

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ the merge kernel
def random_lists(G, nq, rng, max_len=20, empty_rank=None, values=None, long_list=None):
    """Per rank: CSR counts [nq] and sorted (ids, dists) with ids distinct over all ranks; `values`: distances drawn from
    that small set (ties across ranks); `long_list` = (rank, query, length)."""
    lens = rng.integers(0, max_len + 1, size=(G, nq))
    lens[rng.random((G, nq)) < 0.3] = 0                       # empty lists
    if empty_rank is not None:
        lens[empty_rank] = 0
    if long_list is not None:
        lens[long_list[0], long_list[1]] = long_list[2]
    ids = rng.permutation(int(lens.sum()) * 3 + 10)[:int(lens.sum())].astype(np.int32)
    per_rank, at = [], 0
    for g in range(G):
        li, ld = [], []
        for j in range(nq):
            i = ids[at:at + lens[g, j]]
            at += lens[g, j]
            d = rng.choice(values, len(i)) if values is not None else rng.random(len(i)) * 2.0
            i, d = _ordered(i, d.astype(np.float64))
            li.append(i); ld.append(d)
        per_rank.append((np.concatenate(li) if li else np.zeros(0, np.int32), np.concatenate(ld) if ld else np.zeros(0)))
    return lens, per_rank


def packed_gather(per_rank, cap):
    return torch.cat([mdist.pack_range_lists(torch.from_numpy(i).cuda(), torch.from_numpy(d).cuda(), cap)
                      for i, d in per_rank])


@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("case", ["random", "ties", "empty_rank", "nq0", "nq1", "odd"])
def test_merge_kernel_equals_numpy(G, case):
    rng = np.random.default_rng(G * 100 + len(case))
    nq = {"nq0": 0, "nq1": 1}.get(case, 300)
    lens, per_rank = random_lists(G, nq, rng, values=np.array([0.0, 0.25, 0.5, 1.0]) if case == "ties" else None,
                                  empty_rank=G - 1 if case == "empty_rank" else None)
    if case == "odd":                                            # an odd largest total, padded to even
        while int(lens.sum(axis=1).max()) % 2 == 0:
            lens, per_rank = random_lists(G, nq, rng)
    cap = int(lens.sum(axis=1).max(initial=0))
    cap += cap & 1
    gathered = packed_gather(per_rank, cap) if cap else torch.zeros(0, dtype=torch.uint8, device="cuda")
    got = host(mdist.merge_gathered_csr(gathered, lens, cap))
    want = mdist.merge_gathered_csr(gathered.cpu(), lens, cap, merge=numpy_merge)
    assert_csr_equal(got, tuple(t.numpy() for t in want), "G=%d %s" % (G, case))
    assert got[0][-1] == lens.sum()


def test_merge_kernel_long_list():
    """One query with 300,000 entries on one rank among short lists: no staging limit."""
    rng = np.random.default_rng(7)
    G, nq = 3, 40
    lens, per_rank = random_lists(G, nq, rng, long_list=(1, 17, 300000))
    cap = int(lens.sum(axis=1).max())
    cap += cap & 1
    gathered = packed_gather(per_rank, cap)
    got = host(mdist.merge_gathered_csr(gathered, lens, cap))
    want = mdist.merge_gathered_csr(gathered.cpu(), lens, cap, merge=numpy_merge)
    assert_csr_equal(got, tuple(t.numpy() for t in want), "long list")


def test_merge_kernel_refuses_bad_arguments():
    from morna_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(64, dtype=torch.uint8, device="cuda")
    off = torch.zeros(4, dtype=torch.int64, device="cuda")
    p = _lib.dev_ptr
    assert lib.morna_merge_sorted_csr(p(buf), 1, 1, 3, p(off), p(off), 1, p(buf), p(buf), None) == _lib.ERR_INVALID_ARGUMENT   # odd cap
    assert lib.morna_merge_sorted_csr(p(buf), 0, 1, 2, p(off), p(off), 1, p(buf), p(buf), None) == _lib.ERR_INVALID_ARGUMENT   # no lists
    assert lib.morna_merge_sorted_csr(p(buf), 1, 1, 2, p(off), p(off), 3, p(buf), p(buf), None) == _lib.ERR_INVALID_ARGUMENT   # total > slots
    assert lib.morna_merge_sorted_csr(None, 1, 0, 0, None, None, 0, None, None, None) == _lib.OK                             # nothing to do


# ------------------------------------------------------------------ the protocol in one process
def emulate(shards, Q, R, byte_cap=None):
    """sharded_range_search_groups with the collectives replaced by concatenation: every shard counts its batches and
    writes its lists; the groups follow from the global counts; the step after the gather gets the packed buffers."""
    world = len(shards)
    parts = []
    for batches in zip(*[sh.range_count_batches(Q, R) for sh in shards]):
        b0 = batches[0][0]
        counts = np.stack([st["counts"] for _, st in batches])
        for lo, hi in _range_groups(counts.sum(axis=0) * (world + 1), byte_cap):
            c = counts[:, lo:hi]
            cap = int(c.sum(axis=1).max())
            cap += cap & 1
            lists = [sh.range_emit(st, lo, hi) for sh, (_, st) in zip(shards, batches)]
            gathered = torch.cat([mdist.pack_range_lists(l[1], l[2], cap) for l in lists]) if cap else \
                torch.zeros(0, dtype=torch.uint8, device="cuda")
            parts.append((b0 + lo, b0 + hi) + tuple(mdist.merge_gathered_csr(gathered, c, cap)))
    from morna_b200.search import concat_range_groups
    return parts, host(concat_range_groups(parts, "cuda"))


N, D = 60000, 1000


@pytest.fixture(scope="module")
def planted():
    S = synth.gauss(N, D, "cuda", seed=31)
    S[:6000] = S[0] + 1e-3 * synth.gauss(6000, D, "cuda", seed=32)     # a dense cluster inside the first shard
    S[20001:20005] = S[20000]                                          # duplicates inside a shard ...
    S[19999] = S[20000]; S[30001] = S[20000]; S[N - 5] = S[20000]      # ... and across shard boundaries (G = 2, 3, 5)
    whole = make_search(S)
    qa, _ = synth.queries(S, 256, seed=41)
    qb, _ = synth.queries(S, 256, seed=42, noise=0.3)
    Q = torch.cat([qa, qb]).contiguous()
    Q[0] = S[20000].double()
    R100 = median_kth(torch.cat([distances(whole, Q[i:i + 128]) for i in range(0, 512, 128)]), 100)
    return {"S": S, "whole": whole, "Q": Q, "R": R100, "shards": {}}


def shards_of(planted, G):
    if G not in planted["shards"]:
        planted["shards"].clear()                                      # one set of shards on the device at a time
        planted["shards"][G] = [make_search(planted["S"], shard=(r, G)) for r in range(G)]
    return planted["shards"][G]


def check_emulated(planted, G, Q, R, route, byte_cap=None, label=""):
    shards = shards_of(planted, G)
    parts, got = emulate(shards, Q, R, byte_cap)
    assert all(sh.last_range_route == route for sh in shards), label
    want = host(planted["whole"].range_search_device(Q, R))
    assert_csr_equal(got, want, label + " vs unsharded")
    assert_csr_equal(got, brute(planted["whole"], Q, R), label + " vs brute force")
    return parts, got


@pytest.mark.parametrize("G", [2, 3, 5])
def test_emulated_tensor_route(planted, G):
    Q, R = planted["Q"], planted["R"]
    _, got = check_emulated(planted, G, Q, R, "tensor", label="G=%d R100" % G)
    assert got[0][-1] >= 50 * Q.shape[0]                            # half the queries have 100 matches or more
    parts, _ = check_emulated(planted, G, Q, R, "tensor", byte_cap=12 * (G + 1) * 20000, label="G=%d capped" % G)
    assert len(parts) > 1                                            # several groups, concatenated to the uncapped result
    _, (off, ids, _) = check_emulated(planted, G, Q, 0.0, "tensor", label="G=%d R=0" % G)
    assert ids[off[0]:off[1]].tolist() == [N - 5, 30001, 20004, 20003, 20002, 20001, 20000, 19999]
    _, none = check_emulated(planted, G, Q[256:], 0.0, "tensor", label="G=%d no match" % G)
    assert none[0][-1] == 0


@pytest.mark.parametrize("G", [2, 3, 5])
def test_emulated_exact_route(planted, G):
    check_emulated(planted, G, planted["Q"][:40], planted["R"], "exact", label="G=%d 40 queries" % G)


@pytest.mark.parametrize("G", [2, 3, 5])
def test_emulated_overflow_in_one_shard(planted, G):
    """Queries inside the dense cluster: only the first shard's first-pass lists overflow to the FP64 scan."""
    S = planted["S"]
    qn, _ = synth.queries(S, 64, seed=43, noise=0.3)
    Q = torch.cat([S[:64].double(), qn]).contiguous()
    check_emulated(planted, G, Q, 0.05, "tensor", label="G=%d cluster" % G)
    shards = shards_of(planted, G)
    assert shards[0].last_stats[0] >= 64
    assert all(sh.last_stats[0] == 0 for sh in shards[1:])


@pytest.mark.parametrize("G", [2, 3, 5])
def test_emulated_every_row_in_range(G):
    S = synth.gauss(3000, D, "cuda", seed=44)
    whole = make_search(S)
    shards = [make_search(S, shard=(r, G)) for r in range(G)]
    Q, _ = synth.queries(S, 128, seed=45, noise=0.3)
    _, got = emulate(shards, Q, 2.0)
    assert_csr_equal(got, host(whole.range_search_device(Q, 2.0)), "R = 2")
    assert_csr_equal(got, brute(whole, Q, 2.0), "R = 2 vs brute force")
    assert np.array_equal(np.diff(got[0]), np.full(128, 3000))


def test_world_size_one_is_the_local_search(planted):
    Q, R = planted["Q"][:100], planted["R"]
    assert_csr_equal(host(mdist.sharded_range_search(planted["whole"], Q, R)),
                     host(planted["whole"].range_search_device(Q, R)), "no process group")


# ------------------------------------------------------------------ NCCL, two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as td
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    td.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    S = synth.gauss(30000, 512, "cuda", seed=51)                   # every rank draws the same matrix, keeps its block
    S[14999] = S[15000]
    srch = make_search(S, shard=(rank, world), device=torch.device("cuda", rank))
    qa, _ = synth.queries(S, 300, seed=52)
    qb, _ = synth.queries(S, 300, seed=53, noise=0.3)
    Q = torch.cat([qa, qb]).contiguous()
    R = float(np.load(os.path.join(out_dir, "R.npy")))
    res = {"whole": mdist.sharded_range_search(srch, Q, R)}
    parts = list(mdist.sharded_range_search_groups(srch, Q, R, byte_cap=12 * (world + 1) * 3000))
    res["ngroups"] = torch.tensor([len(parts)])
    from morna_b200.search import concat_range_groups
    res["capped"] = concat_range_groups(parts, Q.device)
    res["zero"] = mdist.sharded_range_search(srch, Q[300:], 0.0)    # no rank has a match
    for key, val in res.items():
        for i, t in enumerate(val if isinstance(val, tuple) else (val,)):
            np.save(os.path.join(out_dir, "%s%d_%d.npy" % (key, i, rank)), t.cpu().numpy())
    td.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_rank_sharded_range_search(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    S = synth.gauss(30000, 512, "cuda", seed=51)
    S[14999] = S[15000]
    whole = make_search(S)
    qa, _ = synth.queries(S, 300, seed=52)
    qb, _ = synth.queries(S, 300, seed=53, noise=0.3)
    Q = torch.cat([qa, qb]).contiguous()
    R = median_kth(distances(whole, Q), 100)
    np.save(tmp_path / "R.npy", np.float64(R))
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)

    def load(key, rank):
        return tuple(np.load(tmp_path / ("%s%d_%d.npy" % (key, i, rank))) for i in range(3))

    want = host(whole.range_search_device(Q, R))
    for rank in range(world):
        assert_csr_equal(load("whole", rank), want, "rank %d" % rank)
        assert_csr_equal(load("capped", rank), want, "rank %d capped" % rank)
        assert int(np.load(tmp_path / ("ngroups0_%d.npy" % rank))[0]) > 1
        zero = load("zero", rank)
        assert zero[0].tolist() == [0] * 301 and len(zero[1]) == 0
    assert_csr_equal(want, brute(whole, Q, R), "one process vs brute force")
