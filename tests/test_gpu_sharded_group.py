"""The doc-sharded protocol's merge kernels (k_merge_cut, k_merge_topk) on ONE GPU: G shard handles on
device 0 joined into an in-process shard group (pb_shard_group: peer copies behind a host barrier instead of
NCCL), searched together from G host threads.  Every rank's result must be bit-identical to the CPU oracle
searching the UNSHARDED index (SURVEY 8e strict mode; the NCCL transport runs the same kernels on the same
buffers, tests/gpu_sharded_check.py)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sharded_protocol as sp  # noqa: E402
from repeated_doc import ordinary_queries  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def npb():
    import next_plaid_b200 as m
    m.build_library()
    if m.device_count() < 1:
        pytest.fail("GPU tests need a B200; the library has no CPU fallback")
    return m


def _group(npb, oracle, ix, G, bounds=None):
    """G shard handles over the doc ranges [bounds[g], bounds[g + 1]) (default: make_shard's equal split)."""
    D = ix.num_documents
    bounds = bounds or [g * D // G for g in range(G + 1)]
    shards = []
    for g in range(G):
        sh, base = sp.shard_range(oracle, ix, bounds[g], bounds[g + 1])
        shards.append(npb.MmapIndex.from_arrays(sh.centroids, sh.bucket_weights, sh.codes, sh.residuals,
                                                sh.doc_lengths, sh.ivf, sh.ivf_lengths, sh.nbits, device=0,
                                                doc_id_base=base))
    return npb.ShardGroup(shards)


def _check(oracle, ix, grp, qs, pg, po, subset=None):
    res = grp.search_batch(qs, pg, subset=subset)
    for r, per_rank in enumerate(grp.all_results):          # every rank holds the same global answer
        for a, b in zip(per_rank, res):
            assert a.passage_ids.tolist() == b.passage_ids.tolist() and np.array_equal(a.scores, b.scores), r
    for q, got in zip(qs, res):
        want = oracle.search_one(ix, q, po, subset=subset)
        assert got.passage_ids.tolist() == want.passage_ids.tolist()
        assert np.array_equal(got.scores, want.scores)


@pytest.fixture(scope="module")
def corpus(oracle):
    docs = oracle.synthetic_corpus(3000, 40, dim=128, seed=31, ragged=True)
    ix = oracle.create_index(docs, nbits=4, seed=5, num_partitions=512)
    qs, _ = oracle.synthetic_queries(docs, 12, nq=32, seed=6)
    return docs, ix, qs


@pytest.mark.parametrize("G", [2, 3, 8])
def test_group_equals_unsharded_oracle(npb, oracle, corpus, G):
    docs, ix, qs = corpus
    grp = _group(npb, oracle, ix, G)
    try:
        for cbs in (100_000, 128):                               # dense and batched variants
            kw = dict(top_k=10, n_ivf_probe=8, n_full_scores=256, centroid_batch_size=cbs)
            _check(oracle, ix, grp, qs, npb.SearchParameters(**kw), oracle.SearchParameters(**kw))
        kw = dict(top_k=50, n_ivf_probe=4, n_full_scores=64, centroid_batch_size=128)   # top_k > n_full_scores/4
        _check(oracle, ix, grp, qs, npb.SearchParameters(**kw), oracle.SearchParameters(**kw))
        # subset with the batched variant (candidate intersection only, search.rs:542-545)
        kw = dict(top_k=10, n_ivf_probe=8, n_full_scores=256, centroid_batch_size=128)
        _check(oracle, ix, grp, qs, npb.SearchParameters(**kw), oracle.SearchParameters(**kw),
               subset=list(range(0, 3000, 3)))
    finally:
        grp.close()


def test_group_ties_across_shards(npb, oracle):
    """Duplicated documents in different shards tie on the approximate AND the exact score: the global cut
    and the final order must fall back to the global doc id exactly as the unsharded stable sorts do."""
    base = oracle.synthetic_corpus(300, 24, dim=128, seed=41, ragged=False)
    docs = [base[i % 300] for i in range(1200)]                 # every doc four times, one copy per shard of G=4
    ix = oracle.create_index(docs, nbits=4, seed=6, num_partitions=128)
    qs, _ = oracle.synthetic_queries(docs, 8, nq=32, seed=7)
    grp = _group(npb, oracle, ix, 4)
    try:
        for nfs, k in ((64, 10), (32, 20), (400, 40)):
            kw = dict(top_k=k, n_ivf_probe=8, n_full_scores=nfs, centroid_batch_size=64)
            _check(oracle, ix, grp, qs, npb.SearchParameters(**kw), oracle.SearchParameters(**kw))
    finally:
        grp.close()


def test_group_with_an_empty_shard_and_mixed_query_lengths(npb, oracle):
    docs = oracle.synthetic_corpus(900, 30, dim=64, seed=51, ragged=True)
    ix = oracle.create_index(docs, nbits=2, seed=8, num_partitions=128)
    qs = [oracle.synthetic_queries(docs, 1, nq=n, seed=60 + n)[0][0] for n in (1, 7, 32, 33, 48, 64)]
    G = 3
    grp = _group(npb, oracle, ix, G)
    try:
        kw = dict(top_k=10, n_ivf_probe=4, n_full_scores=128, centroid_batch_size=64)
        _check(oracle, ix, grp, qs, npb.SearchParameters(**kw), oracle.SearchParameters(**kw))
        # subset that leaves the middle shard without any eligible doc
        sub = list(range(0, 300)) + list(range(600, 900, 2))
        _check(oracle, ix, grp, qs, npb.SearchParameters(**kw), oracle.SearchParameters(**kw), subset=sub)
    finally:
        grp.close()


# ---- a tensor-core pass that one shard gives up -------------------------------------------------------------------------
# The probe flags are the same on every rank (a2/a3 are replicated), a re-check overflow (more docs inside the certified
# band than rc_cap = 2M + 1024) depends on the shard's own documents.  The redo must be decided by all ranks together:
# a rank redoing alone would wait at the group barrier, or pair its exchanges with its peers' next sub-batch.

@pytest.fixture(scope="module")
def repeated(oracle):
    base = oracle.synthetic_corpus(1200, 30, dim=128, seed=7, ragged=True)
    q_rep = oracle.synthetic_queries([base[600]], 1, nq=32, seed=5)[0][0]
    return base, q_rep


def _repeated_index(oracle, base, first):
    """base[:1200] and 1400 copies of base[600], the copies first or last: at G = 2 the contiguous split puts 1300
    copies in one shard (more than rc_cap) and 101 in the other."""
    copies = [base[600]] * 1400
    docs = copies + base[:1200] if first else base[:1200] + copies
    ix = oracle.create_index(docs, nbits=4, seed=3, num_partitions=256)
    copy_ids = list(range(1400)) + [2000] if first else [600] + list(range(1200, 2600))
    return ix, np.array(copy_ids)


def _ordinary(oracle, ix, base, copy_ids, n, seed):
    """n queries whose candidates, in both variants, hold no copy of the repeated doc."""
    return ordinary_queries(oracle, ix, base[:600] + base[601:1200], copy_ids, n, seed)


@pytest.mark.parametrize("first", [False, True])
def test_a_recheck_overflow_on_one_shard_is_redone_by_every_rank(npb, oracle, repeated, first):
    base, q_rep = repeated
    ix, copy_ids = _repeated_index(oracle, base, first)
    ordinary = _ordinary(oracle, ix, base, copy_ids, 2, seed=17)
    batch = [ordinary[0], q_rep, ordinary[1]]
    heavy = 0 if first else 1
    # the shards searched on their own: only the one holding 1300 copies gives the tensor-core pass up
    alone = [npb.MmapIndex.from_arrays(sh.centroids, sh.bucket_weights, sh.codes, sh.residuals, sh.doc_lengths, sh.ivf,
                                       sh.ivf_lengths, sh.nbits, device=0, doc_id_base=b)
             for sh, b in (sp.make_shard(oracle, ix, g, 2) for g in range(2))]
    grp = _group(npb, oracle, ix, 2)
    try:
        for cbs in (100_000, 128):
            kw = dict(top_k=10, n_ivf_probe=8, n_full_scores=64, centroid_batch_size=cbs)
            for g, h in enumerate(alone):
                h.search_batch(batch, npb.SearchParameters(**kw))
                assert h.last_work_counters()["n_k1_tc_redo"] == (g == heavy), (g, cbs)
            _check(oracle, ix, grp, batch, npb.SearchParameters(**kw), oracle.SearchParameters(**kw))
            assert [c["n_k1_tc_redo"] for c in grp.all_counters] == [1, 1], grp.all_counters
            assert [c["n_k1_tc"] for c in grp.all_counters] == [0, 0], grp.all_counters
    finally:
        grp.close()
        for h in alone:
            h.close()


def test_a_recheck_overflow_in_one_sub_batch_of_one_shard(npb, oracle, repeated, monkeypatch):
    base, q_rep = repeated
    ix, copy_ids = _repeated_index(oracle, base, False)
    ordinary = _ordinary(oracle, ix, base, copy_ids, 48, seed=23)
    monkeypatch.setenv("PB_WS_BUDGET_MB", "1")      # read at open: several sub-batches per call on every shard
    grp = _group(npb, oracle, ix, 2)
    monkeypatch.delenv("PB_WS_BUDGET_MB")
    try:
        for cbs in (100_000, 128):
            kw = dict(top_k=10, n_ivf_probe=8, n_full_scores=64, centroid_batch_size=cbs)
            pg, po = npb.SearchParameters(**kw), oracle.SearchParameters(**kw)
            _check(oracle, ix, grp, ordinary, pg, po)
            n_sub = grp.all_counters[0]["n_k1_tc"]
            assert n_sub >= 3 and all(c["n_k1_tc"] == n_sub and c["n_k1_tc_redo"] == 0 for c in grp.all_counters), \
                grp.all_counters
            qb = -(-len(ordinary) // n_sub)                  # equal sub-batches
            pos = qb * (n_sub // 2) + 1                      # inside a sub-batch that is neither first nor last
            assert 0 < pos // qb < n_sub - 1
            batch = ordinary[:pos] + [q_rep] + ordinary[pos + 1:]
            _check(oracle, ix, grp, batch, pg, po)
            assert all(c["n_k1_tc_redo"] == 1 and c["n_k1_tc"] == n_sub - 1 for c in grp.all_counters), grp.all_counters
    finally:
        grp.close()


def test_a_shard_without_documents_and_unequal_shards_decide_with_the_group(npb, oracle, repeated, monkeypatch):
    """G = 3 over the doc ranges [0, 900), [900, 900) and [900, 2600), the copies in the last one.  The empty shard has no
    tensor-core operands and runs every pass on the exact path; under a 1 MB budget the shards' own sizes would cut the
    call into different sub-batches.  The ranks must still agree on the sub-batches and on every redo."""
    base, q_rep = repeated
    ix, copy_ids = _repeated_index(oracle, base, False)
    ordinary = _ordinary(oracle, ix, base, copy_ids, 48, seed=23)
    for budget in (None, "1"):
        if budget:
            monkeypatch.setenv("PB_WS_BUDGET_MB", budget)
        grp = _group(npb, oracle, ix, 3, bounds=[0, 900, 900, 2600])
        monkeypatch.delenv("PB_WS_BUDGET_MB", raising=False)
        try:
            for cbs in (100_000, 128):
                kw = dict(top_k=10, n_ivf_probe=8, n_full_scores=64, centroid_batch_size=cbs)
                pg, po = npb.SearchParameters(**kw), oracle.SearchParameters(**kw)
                _check(oracle, ix, grp, ordinary, pg, po)
                n_sub = grp.all_counters[0]["n_k1_tc"]
                assert [c["n_k1_tc"] for c in grp.all_counters] == [n_sub, 0, n_sub], grp.all_counters
                assert [c["n_k1_tc_redo"] for c in grp.all_counters] == [0, 0, 0], grp.all_counters
                assert n_sub >= (3 if budget else 1), grp.all_counters
                qb = -(-len(ordinary) // n_sub)
                pos = qb * (n_sub // 2) + 1                  # a middle sub-batch when the call splits
                batch = ordinary[:pos] + [q_rep] + ordinary[pos + 1:]
                _check(oracle, ix, grp, batch, pg, po)
                assert [c["n_k1_tc"] for c in grp.all_counters] == [n_sub - 1, 0, n_sub - 1], grp.all_counters
                assert [c["n_k1_tc_redo"] for c in grp.all_counters] == [1, 1, 1], grp.all_counters
        finally:
            grp.close()
