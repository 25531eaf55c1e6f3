"""Calls that the workspace budget (PB_WS_BUDGET_MB, read at open) splits into several sub-batches, and tensor-core
passes that give up because of the corpus, must give the same bits as one batch and as the CPU oracle.

A split call exercises what a single sub-batch never does: the query and result offsets of later sub-batches, the trace
index, device-resident outputs written at an offset, and one workspace reused by sub-batches of different row widths
(QS = 8, 32 or 64 query tokens: k_approx16<4> and <8>).  The corpus-dependent give-up is the a5 re-check overflowing:
more docs inside the certified band than rc_cap = 2M + 1024 raise the device flag (k_recheck_pairs) and the host
redoes that sub-batch on the exact fp32 path."""
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from repeated_doc import ordinary_queries  # noqa: E402

pytestmark = pytest.mark.gpu

BUDGET_MB = 1


@pytest.fixture(scope="module")
def npb():
    import next_plaid_b200 as m
    m.build_library()
    if m.device_count() < 1:
        pytest.fail("GPU tests need a B200; the library has no CPU fallback")
    return m


def _gpu_index(npb, ix, budget_mb=None, **kw):
    with pytest.MonkeyPatch.context() as mp:
        if budget_mb is not None:
            mp.setenv("PB_WS_BUDGET_MB", str(budget_mb))
        return npb.MmapIndex.from_arrays(ix.centroids, ix.bucket_weights, ix.codes, ix.residuals,
                                         ix.doc_lengths, ix.ivf, ix.ivf_lengths, ix.nbits, **kw)


def _same(a, b):
    return a.passage_ids.tolist() == b.passage_ids.tolist() and np.array_equal(a.scores, b.scores)


def _params(npb, oracle, **kw):
    return npb.SearchParameters(**kw), oracle.SearchParameters(**kw)


# ---- sub-batching ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def corpus(oracle, npb):
    docs = oracle.synthetic_corpus(3000, 48, dim=128, seed=21, ragged=True)
    ix = oracle.create_index(docs, nbits=4, seed=4, num_partitions=512)
    # 40 queries in blocks of 7, the sub-batch size at 1 MB on the tensor-core path (K = 512, QS = 64, D = 3000:
    # 512 * 64 * 2 + 3000 * 24 + ... bytes per query): short blocks (QS <= 32) alternate with long ones (QS = 64), so
    # a narrower sub-batch follows a wider one on the same workspace; one empty query
    lens = [1, 5, 32, 32, 5, 32, 1,
            48, 33, 64, 5, 32, 1, 48,
            32, 5, 32, 1, 32, 5, 32,
            64, 1, 33, 32, 48, 5, 64,
            5, 32, 1, 32, 32, 5, 1,
            33, 0, 5, 64, 32]
    batch = [oracle.synthetic_queries(docs, 1, nq=n, seed=300 + i)[0][0] if n else np.zeros((0, 128), np.float32)
             for i, n in enumerate(lens)]
    whole, split = _gpu_index(npb, ix), _gpu_index(npb, ix, budget_mb=BUDGET_MB)
    yield docs, ix, batch, whole, split
    whole.close()
    split.close()


WORK_SUMS = ("n_queries", "n_query_tokens", "n_candidates", "n_exact_docs")


@pytest.mark.parametrize("kw,half,on_tc", [
    (dict(top_k=10, n_ivf_probe=8, n_full_scores=256), False, True),                            # dense variant
    (dict(top_k=10, n_ivf_probe=8, n_full_scores=256, centroid_batch_size=128), False, True),   # batched variant
    (dict(top_k=10, n_ivf_probe=8, n_full_scores=256, centroid_batch_size=128), True, True),    # subset, batched
    (dict(top_k=50, n_ivf_probe=4, n_full_scores=64, centroid_batch_size=128), False, True),    # top_k > nfs / 4
    (dict(top_k=10, n_ivf_probe=8, n_full_scores=256), True, False),    # subset, dense: eligibility filter, fp32 table
])
def test_sub_batched_calls_equal_one_batch_and_the_oracle(oracle, npb, corpus, kw, half, on_tc):
    docs, ix, batch, whole, split = corpus
    subset = list(range(0, len(docs), 2)) if half else None
    pg, po = _params(npb, oracle, **kw)
    a = split.search_batch(batch, pg, subset=subset)
    wa = split.last_work_counters()
    b = whole.search_batch(batch, pg, subset=subset)
    wb = whole.last_work_counters()
    if on_tc:
        assert wb["n_k1_tc"] == 1 and wa["n_k1_tc"] >= 2 and wa["n_k1_tc_redo"] == 0, (wa, wb)  # the call split
    else:
        # the eligibility filter forces the list-scan probe in every sub-batch (n_probe_list counts them), and a call
        # off the tensor-core path holds the fp32 and the 16-bit score tables: its sub-batches are sized for
        # 6 bytes per (centroid, query token) entry, which is at least this many sub-batches
        K, D, QS_all = ix.num_centroids, ix.num_documents, 64
        need = math.ceil(len(batch) * (K * QS_all * 6 + D * 24) / (BUDGET_MB << 20))
        assert wa["n_k1_tc"] == 0 and wb["n_probe_list"] == 1, (wa, wb)
        assert wa["n_probe_list"] >= need, (wa["n_probe_list"], need)
    for k in WORK_SUMS:
        assert wa[k] == wb[k], (k, wa, wb)
    for i, (q, x, y) in enumerate(zip(batch, a, b)):
        assert x.query_id == i
        assert _same(x, y), i
        assert _same(x, oracle.search_one(ix, q, po, subset=subset)), i


def test_trace_across_sub_batches_matches_the_oracle_stage_by_stage(oracle, npb, corpus):
    docs, ix, batch, whole, split = corpus
    pg, po = _params(npb, oracle, top_k=10, n_ivf_probe=8, n_full_scores=256, centroid_batch_size=128)
    res, tr = split.search_batch(batch, pg, trace=True)
    w = split.last_work_counters()
    # a traced call runs the exact path with the list-scan probe, one count per sub-batch
    assert w["n_k1_tc"] == 0 and w["n_probe_list"] >= 3, w
    for i, q in enumerate(batch):     # every sub-batch, the last one included
        want, wt = oracle.search_one(ix, q, po, trace=True)
        assert tr.cells[i].tolist() == wt.cells.tolist(), f"cells q{i}"
        assert tr.candidates[i].tolist() == wt.candidates.tolist(), f"candidates q{i}"
        assert np.array_equal(tr.approx[i], wt.approx), f"approx q{i}"
        assert tr.kept[i].tolist() == wt.kept.tolist(), f"kept q{i}"
        assert np.array_equal(tr.kept_exact[i], wt.kept_exact), f"exact q{i}"
        assert _same(res[i], want), i


def test_device_resident_outputs_across_sub_batches(oracle, npb, corpus):
    import torch
    docs, ix, batch, whole, split = corpus
    dev = torch.device("cuda", 0)
    offs = np.zeros(len(batch) + 1, np.int64)
    offs[1:] = np.cumsum([q.shape[0] for q in batch])
    dq = torch.from_numpy(np.ascontiguousarray(np.concatenate(batch, 0), np.float32)).to(dev)
    for kw in (dict(top_k=10, n_ivf_probe=8, n_full_scores=256),
               dict(top_k=50, n_ivf_probe=4, n_full_scores=64, centroid_batch_size=128)):
        pg = npb.SearchParameters(**kw)
        k, B = kw["top_k"], len(batch)
        ids = torch.full((B, k), -7, dtype=torch.int64, device=dev)      # sentinels: every row must be written
        sc = torch.full((B, k), float("nan"), dtype=torch.float32, device=dev)
        cn = torch.full((B,), -1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        split.search_batch_device(dq.data_ptr(), offs, pg, ids.data_ptr(), sc.data_ptr(), cn.data_ptr())
        w = split.last_work_counters()
        assert w["n_k1_tc"] >= 2 and w["n_k1_tc_redo"] == 0, w
        torch.cuda.synchronize()
        ids, sc, cn = ids.cpu().numpy(), sc.cpu().numpy(), cn.cpu().numpy()
        host = split.search_batch(batch, pg)
        for i, r in enumerate(host):
            n = int(cn[i])
            assert n == len(r.passage_ids), (kw, i)
            assert ids[i, :n].tolist() == r.passage_ids.tolist(), (kw, i)
            assert np.array_equal(sc[i, :n], r.scores), (kw, i)


def test_lanes_and_sub_batches_together_change_no_bit(oracle, npb, corpus):
    # each lane searches its slice of the batch under half the budget, so with lanes the call splits further
    docs, ix, batch, whole, split = corpus
    for kw in (dict(top_k=10, n_ivf_probe=8, n_full_scores=256),
               dict(top_k=25, n_ivf_probe=8, n_full_scores=512, centroid_batch_size=128)):
        pg, po = _params(npb, oracle, **kw)
        want = whole.search_batch(batch, pg)
        ww = whole.last_work_counters()
        one = split.search_batch(batch, pg)
        w1 = split.last_work_counters()
        split.set_lanes(2)
        try:
            two = split.search_batch(batch, pg)
            w2 = split.last_work_counters()
        finally:
            split.set_lanes(1)
        assert w2["n_k1_tc"] > w1["n_k1_tc"] >= 2 and w2["n_k1_tc_redo"] == 0, (w1, w2)
        for k in WORK_SUMS:
            assert w1[k] == ww[k] and w2[k] == ww[k], (k, ww, w1, w2)
        for i, (x, y, z) in enumerate(zip(want, one, two)):
            assert _same(y, x) and _same(z, x), (kw, i)
        for q, x in zip(batch[-7:], want[-7:]):
            assert _same(x, oracle.search_one(ix, q, po))


# ---- the tensor-core pass giving up because of the corpus -------------------------------------------------------------

def _without_docs(oracle, ix, drop):
    """`ix` without the docs in `drop` (a set of doc ids): same centroids and codec, so a2/a3 are unchanged."""
    keep = [d for d in range(ix.num_documents) if d not in drop]
    tok = np.concatenate([np.arange(ix.doc_offsets[d], ix.doc_offsets[d + 1]) for d in keep])
    dl = ix.doc_lengths[keep]
    ivf, ivf_lengths = oracle.build_ivf(ix.codes[tok], dl, ix.num_centroids)
    return oracle.Index(ix.centroids, ix.bucket_weights, ix.bucket_cutoffs, ix.codes[tok], ix.residuals[tok], dl,
                        ivf, ivf_lengths, ix.nbits)


@pytest.fixture(scope="module")
def repeated_doc(oracle):
    # one document 1400 times: for top_k = 10 and n_full_scores 64 / 256 (M = 16 / 64) a query drawn from it has
    # ~1420 candidates, 1400 of them tied exactly at the top approximate score, against rc_cap = 1056 / 1152
    base = oracle.synthetic_corpus(1200, 30, dim=128, seed=7, ragged=True)
    docs = base[:600] + [base[600]] * 1400 + base[601:1200]
    ix = oracle.create_index(docs, nbits=4, seed=3, num_partitions=256)
    copies = np.arange(600, 2000)
    q_rep = oracle.synthetic_queries([base[600]], 3, nq=32, seed=5)[0]
    ordinary = ordinary_queries(oracle, ix, base[:600] + base[601:1200], copies, 30, seed=17)
    return ix, set(copies[1:].tolist()), q_rep, ordinary


@pytest.mark.parametrize("cbs", [100_000, 128])
def test_recheck_overflow_redoes_the_sub_batch_and_leaves_the_workspace_clean(oracle, npb, repeated_doc, cbs):
    ix, extra_copies, q_rep, ordinary = repeated_doc
    gpu = _gpu_index(npb, ix)
    single = _without_docs(oracle, ix, extra_copies)     # the same doc once, same centroids
    control = _gpu_index(npb, single)
    try:
        for nfs in (64, 256):
            pg, po = _params(npb, oracle, top_k=10, n_ivf_probe=8, n_full_scores=nfs, centroid_batch_size=cbs)
            # the probe alone does not give up on these queries: with the copies gone the pass stays on the tensor cores
            res = control.search_batch(q_rep, pg)
            w = control.last_work_counters()
            assert w["n_k1_tc"] == 1 and w["n_k1_tc_redo"] == 0, (nfs, w)
            for q, r in zip(q_rep, res):
                assert _same(r, oracle.search_one(single, q, po))
            # with the copies the re-check overflows: the sub-batch is redone once on the exact path
            batch = [ordinary[0], q_rep[0], ordinary[1]]
            res = gpu.search_batch(batch, pg)
            w = gpu.last_work_counters()
            assert w["n_k1_tc_redo"] == 1 and w["n_k1_tc"] == 0, (nfs, w)
            for q, r in zip(batch, res):          # includes the doc-id tie-break over 1400 exact ties
                assert _same(r, oracle.search_one(ix, q, po)), nfs
            # the abandoned pass restored the workspace invariants (cleared re-check maxima, zeroed bitmaps): the
            # next call on the same handle stays on the tensor cores and is exact
            res = gpu.search_batch(ordinary[:8], pg)
            w = gpu.last_work_counters()
            assert w["n_k1_tc"] == 1 and w["n_k1_tc_redo"] == 0, (nfs, w)
            for q, r in zip(ordinary[:8], res):
                assert _same(r, oracle.search_one(ix, q, po)), nfs
    finally:
        control.close()
        gpu.close()


def test_recheck_redo_of_a_middle_sub_batch(oracle, npb, repeated_doc):
    ix, extra_copies, q_rep, ordinary = repeated_doc
    split = _gpu_index(npb, ix, budget_mb=BUDGET_MB)
    try:
        for cbs in (100_000, 128):
            pg, po = _params(npb, oracle, top_k=10, n_ivf_probe=8, n_full_scores=64, centroid_batch_size=cbs)
            split.search_batch(ordinary, pg)
            w = split.last_work_counters()
            n_sub = w["n_k1_tc"]
            assert n_sub >= 3 and w["n_k1_tc_redo"] == 0, w
            qb = math.ceil(len(ordinary) / n_sub)            # equal sub-batches
            pos = qb * (n_sub // 2) + 1                      # inside a sub-batch that is neither first nor last
            assert 0 < pos // qb < n_sub - 1
            batch = ordinary[:pos] + [q_rep[0]] + ordinary[pos + 1:]
            res = split.search_batch(batch, pg)
            w = split.last_work_counters()
            assert w["n_k1_tc_redo"] == 1 and w["n_k1_tc"] == n_sub - 1, (n_sub, w)
            for i, (q, r) in enumerate(zip(batch, res)):
                assert _same(r, oracle.search_one(ix, q, po)), (cbs, i)
    finally:
        split.close()
