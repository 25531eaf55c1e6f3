/*
 * plaid_b200.h -- C-ABI of libplaid_b200: the PLAID search hot path of the `next-plaid` crate
 * (centroid scoring -> IVF candidates -> approximate score -> residual decompression -> MaxSim ->
 * top-k) as hand-written sm_100a CUDA, behind the entry points a Rust `extern "C"` block in
 * next-plaid/src/index.rs would bind (INTEGRATION.md shows that shim).
 *
 * The reference has no FFI for this path (search is hard-wired to the CPU, search.rs:85-90), so
 * each export cites the Rust item it replaces.  Paths are relative to next-plaid/src/.
 *
 * Conventions
 *   - plain pointers and sizes, no C++/torch types; every function returns a pb_status (0 = ok);
 *     pb_last_error() gives the thread-local message the shim maps to Error::Search(String)
 *     (error.rs:10-66).
 *   - there is NO CPU fallback: without a usable sm_100 device every entry point fails with
 *     PB_ERR_CUDA (same contract as NEXT_PLAID_FORCE_GPU, lib.rs:71-84, codec.rs:275-288).
 *   - index arrays are copied to the device at open; query / result pointers are never retained
 *     past the call; a handle may be searched from many host threads at once (state.rs:24-47).
 *   - numerics: every contraction uses one pinned fp32 order (DESIGN.md "Numerics"), the same one
 *     oracle/plaid_oracle.c uses, so results are bit-identical to that restatement of the
 *     reference and within 1e-5 of any other sgemm order.
 */
#ifndef PLAID_B200_H
#define PLAID_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define PB_API
#else
#define PB_API __attribute__((visibility("default")))
#endif

#define PB_VERSION_MAJOR 0
#define PB_VERSION_MINOR 1

typedef enum pb_status {
    PB_OK = 0,
    PB_ERR_INVALID = 1,     /* bad argument (shape, nbits not dividing 8 -- codec.rs:161-166, ...) */
    PB_ERR_CUDA = 2,        /* no device / CUDA runtime error (no CPU fallback) */
    PB_ERR_IO = 3,          /* index directory unreadable or malformed -- Error::IndexLoad */
    PB_ERR_UNSUPPORTED = 4, /* valid for the reference, outside this build's limits (stated) */
    PB_ERR_NOMEM = 5,
    PB_ERR_COMM = 6         /* NCCL */
} pb_status;

typedef struct pb_index pb_index; /* opaque; replaces next_plaid::MmapIndex (index.rs:995-1016) */

enum { PB_MEM_HOST = 0, PB_MEM_DEVICE = 1 };

/*
 * The arrays MmapIndex holds after load (index.rs:1026-1139), in the reference's own dtypes.
 * memory_space = PB_MEM_DEVICE means every pointer is a device pointer on `device` (used by the
 * synthetic benchmark to build 10^9-token indices without a host copy); arrays are still copied.
 */
typedef struct pb_index_desc {
    int32_t dim;                   /* embedding_dim (index.rs:1310); multiple of 4, <= 1024 */
    int32_t nbits;                 /* 1, 2, 4 or 8 (codec.rs:161) */
    int64_t num_centroids;         /* K = centroids.nrows() = ivf_lengths.len() */
    int64_t num_documents;         /* D */
    int64_t num_embeddings;        /* N = sum(doc_lengths); padding rows of merged_*.npy excluded */
    const float *centroids;        /* [K][dim]        centroids.npy  <f4 */
    const float *bucket_weights;   /* [2^nbits]       bucket_weights.npy <f4 */
    const int64_t *codes;          /* [N]             merged_codes.npy <i8 */
    const uint8_t *residuals;      /* [N][dim*nbits/8] merged_residuals.npy u1 */
    const int64_t *doc_lengths;    /* [D]             doclens.*.json */
    const int64_t *ivf;            /* [sum ivf_lengths] ivf.npy <i8, per-centroid ascending unique doc ids */
    const int32_t *ivf_lengths;    /* [K]             ivf_lengths.npy <i4 */
    int32_t device;                /* CUDA ordinal */
    int32_t memory_space;          /* PB_MEM_HOST | PB_MEM_DEVICE */
    int64_t doc_id_base;           /* global id of local doc 0 (doc-sharded deployment), else 0 */
    int32_t flags;                 /* PB_OPEN_* below, 0 = none */
} pb_index_desc;
/* pb_index_desc.flags.
 * ADOPT_RESIDUALS: memory_space must be PB_MEM_DEVICE; the packed residuals (the largest array: 19 GB per million
 *   300-token docs at 4 bits) are used in place instead of copied -- the caller keeps them alive until pb_index_close.
 * ivf == NULL && ivf_lengths == NULL (no flag needed): the inverted file is built on the device from the codes,
 *   exactly as index.rs:850-873 does (per centroid the ascending unique doc ids); pb_index_export_ivf returns it. */
enum { PB_OPEN_ADOPT_RESIDUALS = 1 };

/* search.rs:27-69 SearchParameters.  batch_size is accepted and ignored, as in the reference
 * (it is never read there). */
typedef struct pb_search_params {
    int64_t batch_size;
    int64_t n_full_scores;
    int64_t top_k;
    int64_t n_ivf_probe;
    int64_t centroid_batch_size;      /* 0 or >= K selects the dense variant (search.rs:337) */
    int32_t has_centroid_score_threshold; /* Option<f32>: 0 = None */
    float centroid_score_threshold;
} pb_search_params;

/* SearchParameters::default(), search.rs:58-69 */
PB_API void pb_search_params_default(pb_search_params *p);

/* ---- index lifetime ------------------------------------------------------------------- */

/* MmapIndex::load(path) (index.rs:1026): reads the reference's index directory as-is
 * (metadata.json, centroids.npy, bucket_weights.npy, ivf.npy, ivf_lengths.npy, doclens.N.json,
 * N.codes.npy, N.residuals.npy) and uploads it to `device`. */
PB_API pb_status pb_index_load(const char *index_dir, int32_t device, pb_index **out);

/* Same, from arrays already in memory (what a Rust MmapIndex owns after its own load). */
PB_API pb_status pb_index_open(const pb_index_desc *desc, pb_index **out);

/* Drop for the handle. */
PB_API void pb_index_close(pb_index *ix);

/* The inverted file of the handle in the reference's dtypes (ivf.npy <i8, ivf_lengths.npy <i4; index.rs:501-508):
 * what create_index writes after building it (index.rs:850-873).  out_ivf may be NULL to query the total length
 * (returned in *out_total); out_lengths [K] may be NULL. */
PB_API pb_status pb_index_export_ivf(pb_index *ix, int64_t *out_ivf, int32_t *out_lengths, int64_t *out_total);

/* accessors, index.rs:1290-1312 */
PB_API int64_t pb_index_num_documents(const pb_index *ix);
PB_API int64_t pb_index_num_embeddings(const pb_index *ix);
PB_API int64_t pb_index_num_partitions(const pb_index *ix);
PB_API double pb_index_avg_doclen(const pb_index *ix);
PB_API int32_t pb_index_embedding_dim(const pb_index *ix);
PB_API int32_t pb_index_nbits(const pb_index *ix);
PB_API int32_t pb_index_device(const pb_index *ix);

/* ---- search ------------------------------------------------------------------------------ */

/*
 * MmapIndex::search_batch (index.rs:1279 -> search::search_many_mmap, search.rs:643) and, with
 * n_queries = 1, MmapIndex::search (index.rs:1258 -> search_one_mmap, search.rs:327).
 *
 *   queries        [q_tok_offsets[n_queries]][dim] f32 row-major: the Array2<f32> of each query
 *                  concatenated (host memory)
 *   q_tok_offsets  [n_queries+1] row offsets of each query in `queries`
 *   subset         Option<&[i64]>: NULL = None; otherwise n_subset doc ids (may be empty)
 *   out_ids        [n_queries][top_k] passage_ids (i64), descending score      (QueryResult,
 *   out_scores     [n_queries][top_k] scores (f32)                              search.rs:72-80)
 *   out_counts     [n_queries] number of valid entries of each row (<= top_k)
 *
 * query_id of result i is i (search.rs:661).  A query that cannot be searched yields count 0, as
 * the reference's parallel mode does (search.rs:656-660).
 */
PB_API pb_status pb_search_batch(pb_index *ix, const float *queries, const int64_t *q_tok_offsets,
                                 int64_t n_queries, const pb_search_params *params,
                                 const int64_t *subset, int64_t n_subset, int64_t *out_ids,
                                 float *out_scores, int32_t *out_counts);

/* Stage outputs of the last pb_search_batch_traced call, for stage-level parity tests.
 * All arrays are caller-allocated host memory; any may be NULL. */
typedef struct pb_trace {
    int64_t *cells;        /* [n_queries][cells_cap] ascending centroid ids that survive a3 */
    int32_t *n_cells;      /* [n_queries] */
    int64_t cells_cap;
    int64_t *candidates;   /* [n_queries][cand_cap] ascending doc ids (a4) */
    float *approx;         /* [n_queries][cand_cap] approximate score of each candidate (a5) */
    int32_t *n_candidates; /* [n_queries] */
    int64_t cand_cap;
    int64_t *kept;         /* [n_queries][kept_cap] docs sent to exact scoring, approx-rank order (a6) */
    float *kept_exact;     /* [n_queries][kept_cap] their exact MaxSim (a7+a8) */
    int32_t *n_kept;       /* [n_queries] */
    int64_t kept_cap;
} pb_trace;

PB_API pb_status pb_search_batch_traced(pb_index *ix, const float *queries,
                                        const int64_t *q_tok_offsets, int64_t n_queries,
                                        const pb_search_params *params, const int64_t *subset,
                                        int64_t n_subset, int64_t *out_ids, float *out_scores,
                                        int32_t *out_counts, pb_trace *trace);

/* ---- stage entry points (each is one kernel of the path; used by tests, bench and ncu) ---- */

/* Stage 1, S = Q * C^T (search.rs:345).  out: [n_query_tokens][K] row-major f32, host. */
PB_API pb_status pb_centroid_scores(pb_index *ix, const float *query_tokens, int64_t n_query_tokens,
                                    float *out_scores);

/* MmapIndex::decompress_documents (index.rs:1197-1245): embeddings of the listed docs,
 * concatenated.  out_embeddings [sum lengths][dim] f32 host, out_lengths [n_docs]; an id
 * >= num_documents contributes length 0 as in the reference.  Call with out_embeddings = NULL to
 * get the lengths first. */
PB_API pb_status pb_decompress_documents(pb_index *ix, const int64_t *doc_ids, int64_t n_docs,
                                         float *out_embeddings, int64_t *out_lengths);

/* maxsim::maxsim_score (maxsim.rs:270) for n_docs documents given as decompressed f32 tokens
 * (doc i = rows [doc_tok_offsets[i], doc_tok_offsets[i+1]) of doc_tokens), one query.
 * Host pointers; `device` selects the GPU. */
PB_API pb_status pb_maxsim_scores(int32_t device, const float *query, int32_t n_query_tokens,
                                  int32_t dim, const float *doc_tokens,
                                  const int64_t *doc_tok_offsets, int64_t n_docs, float *out_scores);

/* Exact MaxSim of each query against EVERY document of the index through the fused
 * decompress+MaxSim kernel (recall ground truth).  out_scores [n_queries][num_documents] host. */
PB_API pb_status pb_exhaustive_scores(pb_index *ix, const float *queries,
                                      const int64_t *q_tok_offsets, int64_t n_queries,
                                      float *out_scores);

/* ---- timing hooks for bench.py (device-side, CUDA events on the library's own stream) ----- */

/* Stage ids for pb_last_stage_ms */
enum {
    PB_STAGE_H2D = 0,
    PB_STAGE_CENTROID_SCORES = 1, /* a2 */
    PB_STAGE_PROBE = 2,           /* a3 */
    PB_STAGE_CANDIDATES = 3,      /* a4 */
    PB_STAGE_APPROX = 4,          /* a5 */
    PB_STAGE_CUT = 5,             /* a6 */
    PB_STAGE_EXACT = 6,           /* a7+a8 */
    PB_STAGE_TOPK = 7,            /* a9 */
    PB_STAGE_D2H = 8,
    PB_STAGE_COUNT = 9
};

/* Diagnostic switch for the approximate stage (default on): 1 = two-pass (16-bit first pass +
 * exact re-check of the docs that can still make the cut), 0 = single exact pass over every
 * candidate.  Both produce the reference's cut bit for bit; tests compare them. */
PB_API void pb_set_fast_approx(pb_index *ix, int32_t enabled);

/* Diagnostic switch for the exact stage (default on): 1 = an fp16 tcgen05 estimate with a certified error bound
 * first picks the kept docs that can still reach the top_k, and only those are scored exactly; 0 = every kept
 * doc is scored exactly.  Same results bit for bit; tests compare both.  (PB_FAST_EXACT=0 in the environment
 * sets the default.)  The filter applies when dim is 64/96/128, queries have <= 64 tokens and no trace is asked. */
PB_API void pb_set_fast_exact(pb_index *ix, int32_t enabled);

/* Diagnostic switch for a2 (default on): 1 = the score table comes from the tcgen05 split-fp16 GEMM (k_scores16_tc) and
 * the values that decide something are recomputed as pinned-order fp32 dots; 0 = the dense fp32 FFMA2 kernel
 * (k_centroid_scores), which is also the device-gated fallback for flagged queries and shapes outside the tensor-core
 * kernel's (dim not in {64, 96, 128}, eligibility filters, the dense variant's radix-select probe for n_ivf_probe > 64, n_ivf_probe > K/1024).  Same results bit
 * for bit; tests and bench.py compare both.  (PB_K1_TC=0 in the environment sets the default.) */
PB_API void pb_set_scores_tc(pb_index *ix, int32_t enabled);

/* Lanes: a batch of >= 16 queries is cut into `lanes` slices that run the whole pipeline concurrently, each on its own
 * stream and workspace (helper threads inside the library do the launching), so that one slice's latency-bound kernels
 * overlap another's bandwidth-bound ones.  Results are independent of the setting (queries are independent; next-plaid
 * itself searches a batch query by query, search.rs:1136-1160).  Default 1 = off (env PB_LANES): measured on config B a
 * single caller gains 2 % with 2 lanes, while several host threads calling one handle -- the reference's deployment
 * model, which already overlaps whole batches -- lose 10 %.  Doc-sharded handles and traced calls always run one lane. */
PB_API void pb_set_lanes(pb_index *ix, int32_t lanes);

/* Enable per-stage CUDA-event timing for subsequent searches on this handle (adds event
 * records only, no synchronisation inside the path). */
PB_API void pb_set_profiling(pb_index *ix, int32_t enabled);
/* Milliseconds and kernel launches per stage, summed over the sub-batches of the calling thread's
 * last pb_search_batch.  out_ms / out_launches: [PB_STAGE_COUNT]. */
PB_API pb_status pb_last_stage_stats(pb_index *ix, float *out_ms, int32_t *out_launches);
/* Device time of the calling thread's last search call, one CUDA-event pair on the library's stream around the whole
 * call (all sub-batches, their exchanges and the gaps between them); needs pb_set_profiling(ix, 1). */
PB_API pb_status pb_last_call_ms(pb_index *ix, float *out_ms);
/* Device time of the main kernel of each stage alone (CUDA events around that one launch, summed over sub-batches):
 * the `achieved` side of bench.py's roofline blocks. */
enum {
    PB_KERNEL_SCORES = 0,   /* k_scores16_tc (or k_centroid_scores on the exact path) */
    PB_KERNEL_APPROX16 = 1, /* k_approx16, the first approximate pass */
    PB_KERNEL_FILTER = 2,   /* k_exact_tc, the tcgen05 MaxSim estimate of every kept doc */
    PB_KERNEL_EXACT = 3,    /* k_exact, fused decompress + MaxSim of the survivors */
    PB_KERNEL_COUNT = 4
};
PB_API pb_status pb_last_kernel_ms(pb_index *ix, float *out_ms /* [PB_KERNEL_COUNT] */);
/* Work counters of the calling thread's last search: candidates scored, doc tokens gathered by the
 * approximate stage, docs / tokens exact-scored. */
typedef struct pb_work_counters {
    int64_t n_queries;
    int64_t n_query_tokens;
    int64_t n_cells;
    int64_t n_candidates;
    int64_t n_candidate_tokens;
    int64_t n_exact_docs;      /* docs / tokens scored exactly (the filter's survivors when it is on) */
    int64_t n_exact_tokens;
    int64_t n_filter_docs;     /* docs / tokens estimated by the tensor-core filter (0 when off) */
    int64_t n_filter_tokens;
    int64_t k1_tc_max_code_diff; /* PB_K1_TC_DIAG=1 only: largest difference between the exact 16-bit score table and
                                  * its split-fp16 tensor-core twin (diagnostic; 0 otherwise) */
    int64_t k1_rows_mismatch;    /* PB_K1_TC_DIAG=1 only: words of the sparse exact-row kernel (k_exact_rows, on the probe's
                                  * cells) that differ from the dense score table; 0 expected */
    int64_t n_probe_threshold;   /* sub-batches whose a3 ran threshold-first on the 16-bit table (no device fallback) */
    int64_t n_probe_list;        /* sub-batches whose a3 ran the per-lane list scan (fallback, eligibility filter, ...) */
    int64_t n_k1_tc;             /* sub-batches whose score table came from the tcgen05 kernel (k_scores16_tc) */
    int64_t n_recheck_docs;      /* docs that got the exact fp32 approximate score (a5 second pass) */
    int64_t n_k1_tc_redo;        /* sub-batches the tensor-core pass handed back to the exact path (flagged query, list overflow) */
    int64_t n_exact_pairs;       /* (token, query token) similarities the pair form of the exact stage evaluated */
    int64_t n_pair_fallback_queries; /* queries whose pair list overflowed (or that had no estimate): scored by k_exact */
} pb_work_counters;
PB_API pb_status pb_last_work_counters(pb_index *ix, pb_work_counters *out);

/* Search with queries already resident on the device and results left on the device:
 * the kernel-only timing leg of bench.py ("value"); same semantics as pb_search_batch. */
PB_API pb_status pb_search_batch_device(pb_index *ix, const float *d_queries,
                                        const int64_t *q_tok_offsets_host, int64_t n_queries,
                                        const pb_search_params *params, int64_t *d_out_ids,
                                        float *d_out_scores, int32_t *d_out_counts);

/* ---- index-build path (SURVEY 8 a12, secondary) ----------------------------------------------
 *
 * The reference's build-time GPU seams are cuda::compress_into_codes_cuda_batched (cuda.rs:353, called
 * from codec.rs:265-272) and cuda::compress_and_residuals_cuda_batched (cuda.rs:496, called from
 * index.rs:318-323) plus third-party k-means (kmeans.rs:125-130).  Here a pb_codec holds the
 * centroids / cutoffs on the device (ResidualCodec, codec.rs:107-123) and every call is bit-identical
 * to the CPU implementation (compress_into_codes_cpu, quantize_residuals), including its last-maximum
 * tie rule -- the reference's own CUDA kernel picks the FIRST maximum (cuda.rs:202).
 * k-means: fastkmeans-rs is not in the reference tree, so pb_kmeans_fit is parity-unpinned. */
typedef struct pb_codec pb_codec;
typedef struct pb_shard_group pb_shard_group;   /* in-process rank group, see "doc-sharded deployment" below */
PB_API pb_status pb_codec_open(int32_t device, const float *centroids, int64_t num_centroids, int32_t dim,
                               int32_t nbits, const float *bucket_cutoffs /* may be NULL */, pb_codec **out);
PB_API void pb_codec_close(pb_codec *c);
/* How the last compress/encode call found its codes: tokens whose argmax the tcgen05 shortlist certified
 * vs tokens sent through the exact fp32 kernel (all of them when the filter is not in use: dim not in
 * {64, 96, 128}, K < 256, or PB_ASSIGN_EXACT set). */
PB_API pb_status pb_codec_last_assign_stats(pb_codec *c, int64_t *n_tokens, int64_t *n_exact_fallback,
                                            int32_t *used_tensor_cores);
/* ResidualCodec::compress_into_codes (codec.rs:260): out_codes[n] i64 */
PB_API pb_status pb_codec_compress_into_codes(pb_codec *c, const float *embeddings, int64_t n, int64_t *out_codes);
/* compress_and_residuals (index.rs:17-40 / cuda.rs:496): codes + f32 residuals [n][dim] */
PB_API pb_status pb_codec_compress_and_residuals(pb_codec *c, const float *embeddings, int64_t n,
                                                 int64_t *out_codes, float *out_residuals);
/* encode_index_chunk (index.rs:289-371): codes + packed residuals [n][dim*nbits/8] (quantize_residuals,
 * codec.rs:356-411) */
PB_API pb_status pb_codec_encode_chunk(pb_codec *c, const float *embeddings, int64_t n, int64_t *out_codes,
                                       uint8_t *out_residuals_packed);
/* find_outliers (update.rs:490-608, the numeric kernel of update_centroids): ascending row indices whose
 * minimum squared L2 distance to every centroid exceeds threshold_sq, including the f64 re-check of
 * borderline rows.  out_indices must hold n entries. */
PB_API pb_status pb_codec_find_outliers(pb_codec *c, const float *embeddings, int64_t n, float threshold_sq,
                                        int64_t *out_indices, int64_t *out_count);
/* prepare_codec_artifacts' arithmetic (index.rs:228-287) on held-out embeddings the caller sampled (index.rs:195-226
 * is a seeded shuffle on the host): nearest-centroid residuals, then
 *   out_cutoffs [2^nbits - 1]  quantiles i / 2^nbits of the flattened residuals        (index.rs:260-266)
 *   out_weights [2^nbits]      quantiles (i + 1/2) / 2^nbits                             (index.rs:267-270)
 *   out_avg_residual [dim]     mean |residual| per dimension (may be NULL)               (index.rs:255-258)
 *   out_cluster_threshold      quantile 0.75 of the residual L2 norms (may be NULL)      (index.rs:249-253)
 * with utils.rs:125-149's quantile (sort, position q (n - 1) in f64, lo (1 - w) + hi w, w as f32).  The codec keeps
 * the cutoffs, so pb_codec_encode_chunk works afterwards.  n * dim < 2^31. */
PB_API pb_status pb_codec_train(pb_codec *c, const float *heldout_embeddings, int64_t n, float *out_cutoffs,
                                float *out_weights, float *out_avg_residual, float *out_cluster_threshold);
/* the sizing rules around it: compute_kmeans (kmeans.rs:273-312) and prepare_codec_artifacts (index.rs:195-212) */
PB_API int64_t pb_kmeans_num_sample_docs(int64_t num_documents);
PB_API int64_t pb_kmeans_num_partitions(int64_t num_documents, double avg_sample_doclen, int64_t num_sample_tokens);
PB_API int64_t pb_codec_num_sample_docs(int64_t num_documents);
PB_API int64_t pb_codec_heldout_tokens(int64_t num_embeddings);
/* compute_kmeans' inner fit + L2 normalisation (kmeans.rs:319-419): out_centroids [K][dim] */
PB_API pb_status pb_kmeans_fit(int32_t device, const float *samples, int64_t n, int32_t dim, int64_t num_centroids,
                               int32_t niters, uint64_t seed, float *out_centroids);

/* Data-parallel k-means for the multi-GPU build (SURVEY 8e "Build path"): one rank per GPU, each with its shard of
 * the sample points; per iteration one all-reduce of the [K][dim] sums + [K] counts.  A pb_build_comm is an NCCL
 * communicator (one process per GPU; ship pb_comm_unique_id's 128 bytes as for search) or a member of an in-process
 * pb_shard_group (one host thread per rank).  Every rank receives the same L2-normalised centroids.  The encode
 * that follows needs no communication: each rank runs pb_codec_encode_chunk on its own documents. */
typedef struct pb_build_comm pb_build_comm;
PB_API pb_status pb_build_comm_init(const uint8_t *id128, int32_t rank, int32_t world, int32_t device, pb_build_comm **out);
PB_API pb_status pb_build_comm_group(pb_shard_group *g, int32_t rank, int32_t device, pb_build_comm **out);
PB_API void pb_build_comm_destroy(pb_build_comm *c);
PB_API pb_status pb_kmeans_fit_dp(pb_build_comm *c, const float *samples_local, int64_t n_local, int32_t dim,
                                  int64_t num_centroids, int32_t niters, uint64_t seed, float *out_centroids);

/* MmapIndex::create_with_kmeans (index.rs:1392 -> kmeans.rs:261-422 -> index.rs:551-911): from document embeddings to
 * the reference's index directory (file set of index.rs:394-525), every numeric step on the device -- k-means
 * (pb_kmeans_fit), codec training (pb_codec_train), per-chunk encode (pb_codec_encode_chunk), inverted file
 * (index.rs:850-873) -- and the host doing only sampling and file writing.  The directory loads with the reference's
 * MmapIndex::load and with pb_index_load.  Sample membership and the k-means iteration are parity-unpinned (the
 * reference delegates them to rand_chacha / fastkmeans-rs, neither in its tree); everything downstream of the
 * centroids and the held-out sample is bit-identical to the reference's CPU arithmetic.
 *   embeddings   [sum doc_lengths][dim] f32 host, documents concatenated; doc_lengths [n_docs]
 *   out_index    optional: the freshly built index, already open on params->device */
typedef struct pb_create_params {  /* IndexConfig, index.rs:73-102 */
    int32_t nbits;                   /* 4 */
    int32_t kmeans_niters;           /* 4 */
    int32_t max_points_per_centroid; /* 256 */
    int32_t device;
    int64_t num_partitions;          /* 0 = the heuristic of kmeans.rs:304-309 */
    int64_t batch_size;              /* docs per chunk file, 50 000 */
    uint64_t seed;                   /* 42 */
} pb_create_params;
PB_API void pb_create_params_default(pb_create_params *p);
PB_API pb_status pb_create_index(const float *embeddings, const int64_t *doc_lengths, int64_t n_docs, int32_t dim,
                                 const pb_create_params *params, const char *index_dir, pb_index **out_index);

/* ---- doc-sharded deployment (SURVEY 8e; no reference analogue: the reference is single-process) ----
 *
 * One process per GPU; shard g holds a contiguous doc-id range (pb_index_desc.doc_id_base) with the
 * centroids replicated.  After pb_index_comm_init every pb_search_batch on the handle is a collective:
 * all ranks call it with the same queries and parameters and all receive the same global result,
 * bit-identical to searching the unsharded index.  Per sub-batch, an all-gather of the per-shard top-M
 * approximate keys and two of the exact (key, rank) and (id, score) words reproduce the reference's GLOBAL
 * n_full_scores/4 cut (search.rs:460-469) and its stable final sort (search.rs:496).  A fourth
 * all-gather of one 8-byte flag word per rank comes first, so that all ranks redo a sub-batch on the
 * exact path together when any shard's tensor-core pass gives up; and once per call the ranks
 * all-gather their sub-batch sizes and all use the smallest.
 */
PB_API pb_status pb_comm_unique_id(uint8_t *out128);   /* rank 0: 128-byte NCCL unique id */
PB_API pb_status pb_index_comm_init(pb_index *ix, const uint8_t *id128, int32_t rank, int32_t world);
/* The same protocol inside ONE process: one handle per shard (same or different devices), one host thread
 * per handle, all threads call pb_search_batch together.  The exchanges are peer copies behind a host
 * barrier instead of NCCL; a peer that fails or does not arrive within 60 s breaks the group (PB_ERR_COMM).
 * The group must outlive every handle that joined it. */
PB_API pb_status pb_shard_group_create(int32_t world, pb_shard_group **out);
PB_API void pb_shard_group_destroy(pb_shard_group *g);
PB_API pb_status pb_index_group_join(pb_index *ix, pb_shard_group *g, int32_t rank);

/* ---- misc ----------------------------------------------------------------------------- */

PB_API const char *pb_last_error(void);       /* thread-local, never NULL */
PB_API const char *pb_version(void);
PB_API int32_t pb_device_count(void);         /* 0 when no usable device: callers must fail */

#ifdef __cplusplus
}
#endif
#endif /* PLAID_B200_H */
