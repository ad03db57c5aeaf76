"""The headline kernels against the ORACLE (oracle/oracle.c, the C twin of morna.py:101-114 + 681-712) at the
BASELINE shapes -- not against the repo's own scan.  Every test draws the matrix on the GPU from a fixed seed, copies
it to the host for the oracle, and compares neighbour ids ("ties aside": a returned list is right when the r-th
returned row's oracle distance equals the r-th smallest oracle distance) and distances (1e-9 here; the bar is 1e-5).
Where the oracle's consecutive distances differ by more than the summation noise the ids must be the oracle's own.
"""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from morna_b200 import synth
from tests.helpers import assert_lists_equal_oracle

pytestmark = pytest.mark.gpu


def make_search(S, **kw):
    from morna_b200.search import MornaSearch
    return MornaSearch(vectors=S, stats=(S.shape[0], S.shape[0], S.shape[1]), **kw)


@pytest.mark.parametrize("kind", ["gauss", "tissue"])
def test_batched_headline_shape_equals_oracle(kind):
    """configs[2]: 50,000 x 3000, one 4096-query batch (half in-index rows, half the same rows + noise), k = 100;
    64 of the answers (32 in-index, 32 out-of-index) are compared with the oracle."""
    n, d, nq, k = 50000, 3000, 4096, 100
    S = synth.matrix(kind, n, d, "cuda")
    srch = make_search(S)
    q_in, rows = synth.queries(S, nq // 2)
    q_out, _ = synth.queries(S, nq // 2, noise=0.05)
    q = torch.cat([q_in, q_out]).contiguous()
    ids, dist = srch.batched_search_device(q, k)
    torch.cuda.synchronize()
    assert srch.last_stats[0] == 0, "no query may overflow on %s data: %r" % (kind, srch.last_stats)
    assert torch.equal(ids[: nq // 2, 0].long(), rows)              # an in-index query finds itself first ...
    assert float(dist[: nq // 2, 0].abs().max()) == 0.0             # ... at distance exactly 0
    pick = np.concatenate([np.arange(0, nq // 2, 64), nq // 2 + np.arange(0, nq // 2, 64)])
    assert len(pick) == 64
    S_host = S.cpu().numpy()
    Q_host = q[torch.from_numpy(pick).cuda()].cpu().numpy()
    strict = assert_lists_equal_oracle(S_host, Q_host, ids.cpu().numpy()[pick], dist.cpu().numpy()[pick], k, kind)
    assert strict > 64 * k // 2
    # the streaming host API returns the same lists
    for gi, gd in srch.search_batches([q.cpu().numpy()], k):
        assert np.array_equal(gi, ids.cpu().numpy()) and np.array_equal(gd, dist.cpu().numpy())


def test_single_query_sra_shape_equals_oracle():
    """configs[1]: 21,504 x 3000, one query at a time through the single-query kernel, k = 100; 16 queries
    (8 stored rows, 8 noisy) against the oracle."""
    n, d, k = 21504, 3000, 100
    S = synth.gauss(n, d, "cuda", seed=4321)
    srch = make_search(S)
    q_in, rows = synth.queries(S, 8)
    q_out, _ = synth.queries(S, 8, noise=0.05)
    q = torch.cat([q_in, q_out]).contiguous()
    got_i, got_d = [], []
    for j in range(q.shape[0]):
        i_, d_ = srch.single_search_device(q[j], k)
        assert int(srch._sfallback.item()) == 0
        got_i.append(i_[0].cpu().numpy()); got_d.append(d_[0].cpu().numpy())
    assert_lists_equal_oracle(S.cpu().numpy(), q.cpu().numpy(), np.stack(got_i), np.stack(got_d), k, "single")
    assert [int(g[0]) for g in got_i[:8]] == rows.tolist()


def test_two_row_shards_merged_equal_oracle_at_100k_rows():
    """The multi-GPU data path without the transport: 100,000 x 3000 rows as two row shards, each answered by the
    batched path with global ids, the two sorted lists merged by morna_merge_sorted_topk; 16 queries vs the oracle."""
    from morna_b200 import dist as mdist
    n, d, nq, k = 100000, 3000, 256, 100
    S = synth.gauss(n, d, "cuda", seed=7)
    q_in, _ = synth.queries(S, nq // 2)
    q_out, _ = synth.queries(S, nq // 2, noise=0.05)
    q = torch.cat([q_in, q_out]).contiguous()
    parts = []
    for r in range(2):
        sh = make_search(S, shard=(r, 2))
        parts.append(sh.batched_search_device(q, k))
        assert sh.last_stats[0] == 0
        del sh
    gi = torch.stack([p[0] for p in parts]); gd = torch.stack([p[1] for p in parts])
    ids, dist = mdist.merge_sorted_lists(gi, gd, k)
    pick = np.arange(0, nq, 16)
    S_host = S.cpu().numpy()
    Q_host = q[torch.from_numpy(pick).cuda()].cpu().numpy()
    assert_lists_equal_oracle(S_host, Q_host, ids.cpu().numpy()[pick], dist.cpu().numpy()[pick], k, "two shards")


@pytest.mark.parametrize("world", [2, 5])
def test_sharded_bound_path_equals_unsharded_and_oracle(world):
    """The rows-sharded search with its two exchange steps emulated in one process: every shard scores up to the lower
    bounds of its k best cosines, the k-th largest of all shards' bounds is taken per query (what follows the
    all-gather), every shard builds its lists from that global bound and re-ranks, the sorted lists are merged.  Together the shards re-rank about k rows per query --
    not k per shard -- and the result is the unsharded one and the oracle's."""
    from morna_b200 import dist as mdist
    n, d, nq, k = 60000, 1000, 512, 100
    S = synth.gauss(n, d, "cuda", seed=3)
    S[1000:1004] = S[999]                         # ties inside a shard ...
    S[n - 5] = S[999]                             # ... and across shards
    q_in, _ = synth.queries(S, nq // 2)
    q_out, _ = synth.queries(S, nq // 2, noise=0.05)
    q = torch.cat([q_in, q_out]).contiguous()
    q[0] = S[999].double()
    whole = make_search(S)
    w_ids, w_d = whole.batched_search_device(q, k)
    shards = [make_search(S, shard=(r, world)) for r in range(world)]
    vals = torch.stack([sh.batched_score_bound(q, k) for sh in shards])          # what the all-gather leaves
    bound = shards[0].union_kth_bound(vals, k)
    want = vals.permute(1, 0, 2).reshape(nq, -1).sort(dim=1, descending=True).values[:, k - 1]
    assert torch.equal(bound, want) and bool((bound > -1).all())
    parts = [sh.batched_finish_bound(bound.clone()) for sh in shards]
    reranked = sum(sh.last_stats[2] for sh in shards) / nq
    assert reranked < 1.6 * k, "the shards together re-ranked %.0f rows per query" % reranked
    ids, dist = mdist.merge_sorted_lists(torch.stack([p_[0] for p_ in parts]), torch.stack([p_[1] for p_ in parts]), k)
    assert torch.equal(ids, w_ids) and torch.equal(dist, w_d)
    pick = np.arange(0, nq, 32)
    assert_lists_equal_oracle(S.cpu().numpy(), q.cpu().numpy()[pick], ids.cpu().numpy()[pick], dist.cpu().numpy()[pick], k,
                              "sharded bound")
    print("rows re-ranked per query over %d shards: %.1f" % (world, reranked))


def test_same_sign_rows_wide_features_stay_within_eps_and_equal_oracle():
    """Adversarial case for the fp32 accumulation term of eps: D = 10,000, every entry positive, so all partial sums
    of a dot product have one sign and grow to ~1 -- each of the D/16 chained tensor-core additions truncates at the
    scale of the full sum.  The fp16 scores must stay inside the rigorous bound and the lists must be the oracle's."""
    from morna_b200 import _lib
    lib = _lib.load()
    n, d, nq, k = 6000, 10000, 192, 50
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    S = torch.rand((n, d), generator=g, device="cuda") + 0.5           # all cosines ~0.96
    srch = make_search(S)
    srch.enable_tensor_path()
    q = torch.cat([S[:96].double(), (torch.rand((96, d), generator=g, device="cuda") + 0.5).double()]).contiguous()
    ld_s = (n + 3) // 4 * 4
    scores = torch.zeros((nq, ld_s), dtype=torch.float32, device="cuda")
    eps = torch.zeros(nq, dtype=torch.float32, device="cuda")
    ws = _lib.workspace(lib.morna_knn_batched_workspace_bytes(n, nq, d, k), "cuda")
    rc = lib.morna_debug_tensor_scores(_lib.dev_ptr(srch.hs), srch.ld_h, _lib.dev_ptr(srch.rho_max), n, d, _lib.dev_ptr(q),
                                       nq, d, _lib.dev_ptr(scores), ld_s, _lib.dev_ptr(eps), _lib.dev_ptr(ws), ws.numel(),
                                       _lib.stream_ptr())
    assert rc == 0
    S64 = S.double()
    cos = (q @ S64.t()) / (q.norm(dim=1, keepdim=True) * S64.norm(dim=1)[None, :])
    err = (scores[:, :n].double() - cos).abs()
    assert bool((err <= eps.double()[:, None]).all()), "error %g above the bound %g" % (float(err.max()), float(eps.min()))
    print("same-sign D=%d: max fp16 score error %.3g, bound %.3g" % (d, float(err.max()), float(eps.min())))
    ids, dist = srch.batched_search_device(q, k)
    pick = np.arange(0, nq, 12)
    assert_lists_equal_oracle(S.cpu().numpy(), q.cpu().numpy()[pick], ids.cpu().numpy()[pick], dist.cpu().numpy()[pick], k,
                              "same-sign")


@pytest.mark.parametrize("d", [10000, 30000])
def test_every_search_path_at_wide_features_equals_oracle(d):
    """--features up to 30,000 (morna.py:982-986; BASELINE configs[4] sweeps that far): the batched tensor-core path,
    the single-query call and the generic FP64 scan all answer an index this wide, and agree with the oracle."""
    n, nq, k = 2500, 96, 40
    S = synth.gauss(n, d, "cuda", seed=d)
    srch = make_search(S)
    q_in, rows = synth.queries(S, nq // 2)
    q_out, _ = synth.queries(S, nq // 2, noise=0.05)
    q = torch.cat([q_in, q_out]).contiguous()
    b_ids, b_d = srch.batched_search_device(q, k)
    assert srch.last_stats[0] == 0
    e_ids, e_d = srch.exact_search_device(q, k, allow_single=False)
    assert torch.equal(b_ids, e_ids) and torch.equal(b_d, e_d)
    for j in (0, nq - 1):
        s_ids, s_d = srch.single_search_device(q[j], k)
        assert torch.equal(s_ids[0], e_ids[j]) and torch.equal(s_d[0], e_d[j])
    pick = np.arange(0, nq, 12)
    assert_lists_equal_oracle(S.cpu().numpy(), q.cpu().numpy()[pick], b_ids.cpu().numpy()[pick], b_d.cpu().numpy()[pick], k,
                              "D=%d" % d)
    assert b_ids[: nq // 2, 0].tolist() == rows.tolist()


# ------------------------------------------------------------------ multi-process NCCL (needs >= 2 GPUs)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as td
    from morna_b200 import dist as mdist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    td.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    n, d, nq, k = 30000, 512, 256, 40
    S = synth.gauss(n, d, "cuda", seed=11)                    # every rank draws the same matrix, keeps its block
    srch = make_search(S, shard=(rank, world), device=torch.device("cuda", rank))
    q, _ = synth.queries(S, nq, noise=0.02)
    ids, dist = mdist.sharded_exact_search(lambda qq, kk: srch.batched_search_device(qq, kk), q, k)
    ids2, dist2 = mdist.sharded_batched_search(srch, q, k)
    assert torch.equal(ids, ids2) and torch.equal(dist, dist2)
    if rank == 0:
        np.save(os.path.join(out_dir, "S.npy"), S.cpu().numpy()); np.save(os.path.join(out_dir, "Q.npy"), q.cpu().numpy())
    np.save(os.path.join(out_dir, "ids%d.npy" % rank), ids.cpu().numpy())
    np.save(os.path.join(out_dir, "dist%d.npy" % rank), dist.cpu().numpy())
    td.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_nccl_two_rank_sharded_search_equals_oracle(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    S, Q = np.load(tmp_path / "S.npy"), np.load(tmp_path / "Q.npy")
    ids = [np.load(tmp_path / ("ids%d.npy" % r)) for r in range(world)]
    dist = [np.load(tmp_path / ("dist%d.npy" % r)) for r in range(world)]
    assert np.array_equal(ids[0], ids[1]) and np.array_equal(dist[0], dist[1])       # every rank holds the merged answer
    pick = np.arange(0, Q.shape[0], 8)
    assert_lists_equal_oracle(S, Q[pick], ids[0][pick], dist[0][pick], 40, "nccl")
