"""Rows-sharded group-capped search on the GPU: the protocol emulated in one process over G shards of one matrix (every
shard labels its block and runs its own capped search; the collectives are concatenations; the step after the list
all-gather is dist.merge_capped_topk, or merge_gathered_csr and the walk for range), and the NCCL run with two ranks.
Results must equal the unsharded search with the same cap and the brute-force walk of test_gpu_capped_search.py, in ids
and distance bits."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import dist as mdist, synth
from morna_b200.search import concat_range_groups
from tests.test_gpu_capped_search import cap_labels, queries, reference, walk
from tests.test_gpu_exclusion import assert_csr_same, assert_same, host
from tests.test_gpu_range_search import brute, distances, make_search, median_kth
from tests.test_gpu_sharded_range import emulate

pytestmark = pytest.mark.gpu

N, D = 50000, 3000
GROUPINGS = ["g100", "g1000", "g10_scattered", "all_but_60", "ungrouped"]


def labelled_shards(S, labels, G):
    shards = []
    for r in range(G):
        sh = make_search(S, shard=(r, G))
        sh.set_cap_groups(labels[sh.row_lo:sh.row_hi])
        shards.append(sh)
    return shards


def gathered_labels(shards):
    """all_gather_cap_labels with the collective replaced by a concatenation."""
    return torch.cat([mdist.cap_label_block(sh, len(shards)) for sh in shards])[:shards[0].index_size]


def emulate_topk(shards, Q, k, m):
    """sharded_capped_search with its collectives replaced by concatenations."""
    labels = gathered_labels(shards)
    every = torch.stack([mdist.pack_topk_lists(*sh.batched_search_device(Q, k, max_per_group=m)) for sh in shards])
    return mdist.merge_capped_topk(shards[0], every, labels, Q.shape[0], k, m)


def emulate_range(shards, Q, R, m, byte_cap=None):
    """sharded_range_search_groups(..., max_per_group=m) with its collectives replaced by concatenations."""
    labels = gathered_labels(shards)
    parts, _ = emulate(shards, Q, R, byte_cap)
    capped = [p[:2] + shards[0].cap_sorted_lists(*p[2:], m, cap_group=labels) for p in parts]
    return capped, host_all(concat_range_groups(capped, "cuda"))


def host_all(ts):
    return tuple(host(t) for t in ts)


def walked_csr(csr, caps, m):
    off, ids, d = csr
    o, i, dd = [0], [], []
    for j in range(len(off) - 1):
        li, ld = ids[off[j]:off[j + 1]], d[off[j]:off[j + 1]]
        keep = walk(li, ld, caps, m)
        i.append(li[keep]); dd.append(ld[keep]); o.append(o[-1] + len(keep))
    return np.array(o, np.int64), np.concatenate(i).astype(np.int32), np.concatenate(dd)


@pytest.fixture(scope="module", params=["gauss", "tissue"])
def idx(request):
    S = synth.matrix(request.param, N, D, "cuda", seed=7)
    whole = make_search(S)
    Q, _ = queries(whole, 64, seed=3)
    return {"kind": request.param, "S": S, "whole": whole, "Q": Q, "want": {}, "shards": {}}


def shards_of(idx, grouping, G):
    key = (grouping, G)
    if key not in idx["shards"]:
        idx["shards"].clear()                                         # one set of shards on the device at a time
        idx["shards"][key] = labelled_shards(idx["S"], cap_labels(grouping, N), G)
    return idx["shards"][key]


@pytest.mark.parametrize("G", [1, 2, 3, 5])
@pytest.mark.parametrize("grouping", GROUPINGS)
def test_emulated_capped_top_k(idx, grouping, G):
    """k = 600 takes the FP64 route on every shard; the rest run on the tensor cores."""
    whole, Q = idx["whole"], idx["Q"]
    whole.set_cap_groups(cap_labels(grouping, N))
    shards = shards_of(idx, grouping, G)
    for m in (1, 2, 5):
        key = (grouping, m)
        if key not in idx["want"]:                                    # the walk's first k entries are its top-k
            idx["want"][key] = reference(whole, Q, 600, m)
        full = idx["want"][key]
        for k in (1, 20, 100, 600):
            label = "%s/%s G=%d N=%d k=%d" % (idx["kind"], grouping, G, m, k)
            want = (full[0][:, :k], full[1][:, :k])
            got = emulate_topk(shards, Q, k, m)
            assert_same(got, want, label + " vs brute force")
            assert_same(got, host_all(whole.batched_search_device(Q, k, max_per_group=m)), label + " vs unsharded")


@pytest.mark.parametrize("G", [2, 3, 5])
@pytest.mark.parametrize("grouping", ["g100", "g1000", "g10_scattered", "all_but_60"])
def test_emulated_capped_range(idx, grouping, G):
    whole, Q = idx["whole"], idx["Q"]
    labels = cap_labels(grouping, N)
    whole.set_cap_groups(labels)
    shards = shards_of(idx, grouping, G)
    if "R" not in idx:
        idx["R"] = median_kth(distances(whole, Q), 100)
        idx["brute"] = brute(whole, Q, idx["R"])
    R = idx["R"]
    for m in (1, 2, 5):
        label = "%s/%s G=%d N=%d range" % (idx["kind"], grouping, G, m)
        want = walked_csr(idx["brute"], labels, m)
        _, got = emulate_range(shards, Q, R, m)
        assert_csr_same(got, want, label + " vs brute force")
        assert_csr_same(got, host_all(whole.range_search_device(Q, R, max_per_group=m)), label + " vs unsharded")
        parts, got = emulate_range(shards, Q, R, m, byte_cap=12 * (G + 1) * 2000)
        assert len(parts) > 1, label
        assert_csr_same(got, want, label + " byte cap")


def test_planted_group_across_shards():
    """N = 1 and one group's two nearest rows of a query on different shards: each shard's own walk keeps its row, so
    the merged lists hold both, and only the walk over the merged order drops the second."""
    S = synth.gauss(20000, 512, "cuda", seed=61)
    S[15000] = S[100] + 1e-3 * S[100].abs().mean() * torch.randn(512, device="cuda", generator=torch.Generator("cuda").manual_seed(2))
    labels = cap_labels("g100", 20000)
    labels[[100, 15000]] = 999999
    whole = make_search(S)
    whole.set_cap_groups(labels)
    shards = labelled_shards(S, labels, 2)
    Q = torch.cat([S[[100]].double(), synth.queries(S, 63, seed=62)[0]]).contiguous()
    every = torch.stack([mdist.pack_topk_lists(*sh.batched_search_device(Q, 10, max_per_group=1)) for sh in shards])
    merged = host(mdist.merge_packed_lists(every, Q.shape[0], 10, 10)[0])
    assert merged[0, 0] == 100 and merged[0, 1] == 15000                   # the merge alone keeps both
    got = emulate_topk(shards, Q, 10, 1)
    assert host(got[0])[0, 0] == 100 and 15000 not in host(got[0])[0].tolist()
    assert_same(got, reference(whole, Q, 10, 1), "planted")
    off, ids, _ = emulate_range(shards, Q[:1], 0.01, 1)[1]
    assert ids.tolist() == [100]


def test_empty_last_shard():
    """12 rows over 5 shards: 3, 3, 3, 3 and 0 rows; k = 600 is more than every shard and the index hold."""
    S = synth.gauss(12, 64, "cuda", seed=63)
    labels = np.array([0, 0, 1, 1, 1, 2, 2, -1, 3, 3, 3, 3], np.int32)
    whole = make_search(S)
    whole.set_cap_groups(labels)
    shards = labelled_shards(S, labels, 5)
    assert shards[-1].row_hi == shards[-1].row_lo
    Q = torch.cat([S.double(), synth.gauss(8, 64, "cuda", seed=64).double()]).contiguous()
    for m, k in ((1, 2), (2, 3), (1, 600), (2, 600)):
        got = emulate_topk(shards, Q, k, m)
        assert_same(got, reference(whole, Q, k, m), "empty shard N=%d k=%d" % (m, k))
        assert_same(got, host_all(whole.batched_search_device(Q, k, max_per_group=m)), "unsharded")
    _, got = emulate_range(shards, Q, 1.0, 1)
    assert_csr_same(got, host_all(whole.range_search_device(Q, 1.0, max_per_group=1)), "empty shard range")


def test_world_size_one_is_the_local_search(idx):
    whole, Q = idx["whole"], idx["Q"]
    whole.set_cap_groups(cap_labels("g100", N))
    assert_same(mdist.sharded_batched_search(whole, Q, 100, max_per_group=2),
                host_all(whole.batched_search_device(Q, 100, max_per_group=2)), "top-k, no process group")
    R = float(host(whole.exact_search_device(Q[:8], 200)[1])[:, 150].mean())
    assert_csr_same(host_all(mdist.sharded_range_search(whole, Q, R, max_per_group=2)),
                    host_all(whole.range_search_device(Q, R, max_per_group=2)), "range, no process group")


# ------------------------------------------------------------------ NCCL, two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _nccl_setup(world, device):
    S = synth.gauss(30000, 512, device, seed=71)                     # every rank draws the same matrix, keeps its block
    S[20000] = S[5] + 1e-3 * S[5].abs().mean()                        # a group's two nearest rows on different ranks
    labels = cap_labels("g100", 30000)
    labels[[5, 20000]] = 999999
    qa, _ = synth.queries(S, 300, seed=72)
    qb, _ = synth.queries(S, 300, seed=73, noise=0.3)
    return S, labels, torch.cat([S[[5]].double(), qa, qb]).contiguous()


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as td
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    td.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    S, labels, Q = _nccl_setup(world, dev)
    srch = make_search(S, shard=(rank, world), device=dev)
    srch.set_cap_groups(labels[srch.row_lo:srch.row_hi])
    R = float(np.load(os.path.join(out_dir, "R.npy")))
    res = {"top100": mdist.sharded_batched_search(srch, Q, 100, max_per_group=2),
           "top20": mdist.sharded_batched_search(srch, Q, 20, max_per_group=1),
           "range": mdist.sharded_range_search(srch, Q, R, max_per_group=2)}
    parts = list(mdist.sharded_range_search_groups(srch, Q, R, byte_cap=12 * (world + 1) * 3000, max_per_group=1))
    res["ngroups"] = torch.tensor([len(parts)])
    res["range_groups"] = concat_range_groups(parts, Q.device)
    for key, val in res.items():
        for i, t in enumerate(val if isinstance(val, tuple) else (val,)):
            np.save(os.path.join(out_dir, "%s%d_%d.npy" % (key, i, rank)), t.cpu().numpy())
    td.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_rank_sharded_capped_search(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    S, labels, Q = _nccl_setup(world, "cuda")
    whole = make_search(S)
    whole.set_cap_groups(labels)
    R = median_kth(distances(whole, Q), 100)
    np.save(tmp_path / "R.npy", np.float64(R))
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)

    def load(key, rank, n):
        return tuple(np.load(tmp_path / ("%s%d_%d.npy" % (key, i, rank))) for i in range(n))

    want = {"top100": host_all(whole.batched_search_device(Q, 100, max_per_group=2)),
            "top20": host_all(whole.batched_search_device(Q, 20, max_per_group=1)),
            "range": host_all(whole.range_search_device(Q, R, max_per_group=2)),
            "range_groups": host_all(whole.range_search_device(Q, R, max_per_group=1))}
    assert want["top20"][0][0, 0] == 5 and 20000 not in want["top20"][0][0].tolist()
    assert_same(want["top100"], reference(whole, Q, 100, 2), "one process vs brute force")
    for rank in range(world):
        for key in ("top100", "top20"):
            assert_same(load(key, rank, 2), want[key], "rank %d %s" % (rank, key))
        for key in ("range", "range_groups"):
            assert_csr_same(load(key, rank, 3), want[key], "rank %d %s" % (rank, key))
        assert int(np.load(tmp_path / ("ngroups0_%d.npy" % rank))[0]) > 1
