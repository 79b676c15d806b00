"""Host-side logic of the multi-GPU path on CPU: the sharding of the clusters over the ranks.
(The pattern exchange itself is the library's pf_exchange_run: tests/test_gpu_exchange_run.py and
tests/test_gpu_multirank.py.)"""
import numpy as np

from panfeed_b200 import dist as pfdist


def test_shard_clusters_balanced_and_complete():
    rng = np.random.default_rng(1)
    w = rng.integers(1, 1000, 200)
    for world in (1, 2, 3, 8):
        shards = pfdist.shard_clusters(w, world)
        assert sorted(c for s in shards for c in s) == list(range(200))
        loads = [int(w[s].sum()) for s in shards]
        assert max(loads) - min(loads) <= int(w.max())
        assert all(s == sorted(s) for s in shards)
