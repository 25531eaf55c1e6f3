"""Queries for the corpora of the re-check redo tests, which hold one document many times (test_gpu_subbatch_and_redo,
test_gpu_sharded_group): the ordinary queries of those tests must not reach the copies, so that only the query drawn
from the repeated document makes the tensor-core pass give up."""
import numpy as np


def ordinary_queries(oracle, ix, pool, copies, n, seed):
    """n queries drawn from `pool` whose candidates, in both variants, hold none of the doc ids in `copies`."""
    cand, _ = oracle.synthetic_queries(pool, 2 * n, nq=32, seed=seed)
    out = []
    for q in cand:
        if all(not np.isin(oracle.search_one(ix, q, oracle.SearchParameters(n_ivf_probe=8, centroid_batch_size=cbs),
                                             trace=True)[1].candidates, copies).any() for cbs in (100_000, 128)):
            out.append(q)
    assert len(out) >= n, len(out)
    return out[:n]
