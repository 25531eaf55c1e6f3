"""Reference implementation of the doc-sharded search protocol (SURVEY.md 8e, DESIGN.md 5) over
torch.distributed, with the CPU oracle as each shard's engine.  The CUDA path implements the same two
exchanges with NCCL all-gathers inside libplaid_b200 (k_cut -> all-gather -> k_merge_cut -> k_exact ->
all-gather -> k_merge_topk); this file is the executable specification the gloo tests run.

The oracle engine never gives a pass up; the CUDA engine's tensor-core pass can, and the redo is collective: each rank's
local fallback flag (0 on a rank that is not on the tensor-core path) is all-gathered before exchange 1, and if any
rank raised it, all ranks redo the sub-batch on the exact path together; the ranks also agree on one sub-batch size per
call.  So every rank issues the same exchanges in the same order."""
import numpy as np


def total_key(scores):
    """search.rs:110-133 as a sortable integer: finite by total_cmp, every non-finite lowest."""
    s = np.asarray(scores, np.float32)
    bits = s.view(np.int32).astype(np.int64)
    key = np.where(bits < 0, bits ^ 0x7FFFFFFF, bits)
    return np.where(np.isfinite(s), key, -(2 ** 40))


def make_shard(oracle, ix, g, G):
    """Shard g of G: the g-th of G contiguous, equal doc ranges of `ix` (shard_range)."""
    D = ix.num_documents
    return shard_range(oracle, ix, g * D // G, (g + 1) * D // G)


def shard_range(oracle, ix, d0, d1):
    """Contiguous doc range [d0, d1) of `ix` as its own index: centroids replicated, IVF restricted."""
    t0, t1 = int(ix.doc_offsets[d0]), int(ix.doc_offsets[d1])
    codes, res, dl = ix.codes[t0:t1], ix.residuals[t0:t1], ix.doc_lengths[d0:d1]
    ivf, ivf_lengths = oracle.build_ivf(codes, dl, ix.num_centroids)
    return oracle.Index(ix.centroids, ix.bucket_weights, ix.bucket_cutoffs, codes, res, dl, ivf, ivf_lengths,
                        ix.nbits), d0


def sharded_search_one(oracle, dist, shard, base, q, p, subset=None):
    """One query on every rank; returns (global ids, scores) identical on all ranks."""
    world = dist.get_world_size()
    M = min(p.n_full_scores, max(p.n_full_scores // 4, p.top_k))
    local_subset = None if subset is None else [int(s) - base for s in subset]
    # a2-a5 on the shard (probe is replicated: same Q, same C => same cells)
    _, tr = oracle.search_one(shard, q, p, subset=local_subset, trace=True)
    gid = tr.candidates + base
    order = np.lexsort((gid, -total_key(tr.approx)))[:M]            # (approx desc, global id asc)
    mine = [(int(total_key(tr.approx)[i]), int(gid[i])) for i in order]
    # exchange 1: every shard's sorted top-M
    allk = [None] * world
    dist.all_gather_object(allk, mine)
    merged = sorted((k for part in allk for k in part), key=lambda k: (-k[0], k[1]))[:M]
    # my members of the global cut, with their global approximate rank
    mine2 = []
    for rank, (_, g) in enumerate(merged):
        if base <= g < base + shard.num_documents:
            ex = oracle.maxsim_score(q, oracle.get_document_embeddings(shard, g - base))
            mine2.append((float(ex), rank, g))
    # exchange 2: exact triples
    alle = [None] * world
    dist.all_gather_object(alle, mine2)
    trip = [t for part in alle for t in part]
    trip.sort(key=lambda t: (-int(total_key([t[0]])[0]), t[1]))     # stable sort by exact desc == tie on approx rank
    trip = trip[:p.top_k]
    return np.array([t[2] for t in trip], np.int64), np.array([t[0] for t in trip], np.float32)
