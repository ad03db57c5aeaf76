"""The streaming pipeline's CUDA-graph capture while an earlier MornaSearch waits for the cyclic garbage collector."""
import gc

import numpy as np
import pytest


@pytest.mark.gpu
def test_capture_survives_collection_of_a_dropped_search():
    """A MornaSearch and its pipelines form a reference cycle, so a dropped search (graphs, events, pinned buffers) is
    freed by the cyclic collector, at whatever allocation triggers it.  With the collector running at nearly every
    allocation, the next search's graph capture must still succeed and return the exact scan's answers."""
    import torch
    from morna_b200 import synth
    from morna_b200.search import MornaSearch
    S = synth.gauss(3000, 256, "cuda", seed=21)
    q, _ = synth.queries(S, 256, noise=0.05)
    old = MornaSearch(vectors=S, stats=(3000, 3000, 256))
    for _ in old.search_batches([q] * 3, 10):              # the third batch is captured into a graph
        pass
    assert any(getattr(sl, "graph_key", None) is not None for sl in old._pipes[(10, 2)].slots)
    del old
    thresholds = gc.get_threshold()
    gc.collect()
    gc.set_threshold(1, 1, 1)
    try:
        dropped = MornaSearch(vectors=S, stats=(3000, 3000, 256))
        for _ in dropped.search_batches([q] * 3, 10):
            pass
        del dropped                                        # left to the collector, which now runs all the time
        search = MornaSearch(vectors=S, stats=(3000, 3000, 256))
        got = [(ids.copy(), d.copy()) for ids, d in search.search_batches([q] * 4, 10)]
        assert any(getattr(sl, "graph_key", None) is not None for sl in search._pipes[(10, 2)].slots)
    finally:
        gc.set_threshold(*thresholds)
    want_i, want_d = search.exact_search_device(q, 10)
    for ids, d in got:
        assert np.array_equal(ids, want_i.cpu().numpy())
        assert np.array_equal(d.view(np.int64), want_d.cpu().numpy().view(np.int64))
