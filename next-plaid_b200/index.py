"""Host-side mirror of the reference's index/search interface over the C-ABI of libplaid_b200.

Names, argument meaning and error behaviour follow next-plaid/src (paths relative to it):
  MmapIndex.load / search / search_batch / accessors ... index.rs:1026, :1258, :1279, :1290-1312
  SearchParameters, QueryResult ........................ search.rs:27-80
  Error kinds .......................................... error.rs:10-66

This module is a thin ctypes binding: all work happens in hand-written sm_100a kernels behind
include/plaid_b200.h.  There is no CPU path: if the shared library or a B200 is missing every call
raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libplaid_b200.so")

PB_OK, PB_ERR_INVALID, PB_ERR_CUDA, PB_ERR_IO, PB_ERR_UNSUPPORTED, PB_ERR_NOMEM, PB_ERR_COMM = range(7)
STAGES = ["h2d", "centroid_scores", "probe", "candidates", "approx", "cut", "exact", "topk", "d2h"]


class PlaidError(RuntimeError):
    """next_plaid::Error (error.rs:10-66); `.status` is the pb_status code."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[pb_status {status}] {message}")
        self.status = status


class _Desc(C.Structure):
    _fields_ = [
        ("dim", C.c_int32), ("nbits", C.c_int32), ("num_centroids", C.c_int64),
        ("num_documents", C.c_int64), ("num_embeddings", C.c_int64),
        ("centroids", C.c_void_p), ("bucket_weights", C.c_void_p), ("codes", C.c_void_p),
        ("residuals", C.c_void_p), ("doc_lengths", C.c_void_p), ("ivf", C.c_void_p),
        ("ivf_lengths", C.c_void_p), ("device", C.c_int32), ("memory_space", C.c_int32),
        ("doc_id_base", C.c_int64), ("flags", C.c_int32),
    ]


class _Params(C.Structure):
    _fields_ = [
        ("batch_size", C.c_int64), ("n_full_scores", C.c_int64), ("top_k", C.c_int64),
        ("n_ivf_probe", C.c_int64), ("centroid_batch_size", C.c_int64),
        ("has_centroid_score_threshold", C.c_int32), ("centroid_score_threshold", C.c_float),
    ]


class _Trace(C.Structure):
    _fields_ = [
        ("cells", C.c_void_p), ("n_cells", C.c_void_p), ("cells_cap", C.c_int64),
        ("candidates", C.c_void_p), ("approx", C.c_void_p), ("n_candidates", C.c_void_p),
        ("cand_cap", C.c_int64),
        ("kept", C.c_void_p), ("kept_exact", C.c_void_p), ("n_kept", C.c_void_p),
        ("kept_cap", C.c_int64),
    ]


class _Work(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_queries", "n_query_tokens", "n_cells", "n_candidates",
                                         "n_candidate_tokens", "n_exact_docs", "n_exact_tokens",
                                         "n_filter_docs", "n_filter_tokens", "k1_tc_max_code_diff",
                                         "k1_rows_mismatch", "n_probe_threshold", "n_probe_list", "n_k1_tc",
                                         "n_recheck_docs", "n_k1_tc_redo", "n_exact_pairs",
                                         "n_pair_fallback_queries")]


EXPORTS = [
    "pb_search_params_default", "pb_index_load", "pb_index_open", "pb_index_close",
    "pb_index_num_documents", "pb_index_num_embeddings", "pb_index_num_partitions",
    "pb_index_avg_doclen", "pb_index_embedding_dim", "pb_index_nbits", "pb_index_device",
    "pb_search_batch", "pb_search_batch_traced", "pb_centroid_scores", "pb_decompress_documents",
    "pb_maxsim_scores", "pb_exhaustive_scores", "pb_set_profiling", "pb_last_stage_stats",
    "pb_last_work_counters", "pb_search_batch_device", "pb_last_error", "pb_version",
    "pb_device_count", "pb_comm_unique_id", "pb_index_comm_init", "pb_shard_group_create", "pb_shard_group_destroy",
    "pb_index_group_join", "pb_index_export_ivf", "pb_last_call_ms", "pb_last_kernel_ms", "pb_set_fast_approx", "pb_set_fast_exact", "pb_set_scores_tc", "pb_set_lanes",
    "pb_codec_open", "pb_codec_close", "pb_codec_compress_into_codes", "pb_codec_compress_and_residuals",
    "pb_codec_encode_chunk", "pb_kmeans_fit", "pb_codec_train", "pb_kmeans_num_sample_docs",
    "pb_kmeans_num_partitions", "pb_codec_num_sample_docs", "pb_codec_heldout_tokens", "pb_create_index",
    "pb_create_params_default", "pb_build_comm_init", "pb_build_comm_group", "pb_build_comm_destroy", "pb_kmeans_fit_dp", "pb_codec_last_assign_stats", "pb_codec_find_outliers",
]

_lib = None


def load_library():
    """dlopen libplaid_b200.so; raise (never fall back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PlaidError(PB_ERR_CUDA, f"{LIB_PATH} is not built (run __graft_entry__.build()); "
                                          "there is no CPU fallback for the search path")
        L = C.CDLL(LIB_PATH)
        L.pb_last_error.restype = C.c_char_p
        L.pb_version.restype = C.c_char_p
        for f in ("pb_index_num_documents", "pb_index_num_embeddings", "pb_index_num_partitions"):
            getattr(L, f).restype = C.c_int64
            getattr(L, f).argtypes = [C.c_void_p]
        L.pb_index_avg_doclen.restype = C.c_double
        L.pb_index_avg_doclen.argtypes = [C.c_void_p]
        for f in ("pb_index_embedding_dim", "pb_index_nbits", "pb_index_device"):
            getattr(L, f).restype = C.c_int32
            getattr(L, f).argtypes = [C.c_void_p]
        L.pb_index_close.argtypes = [C.c_void_p]
        L.pb_index_close.restype = None
        L.pb_set_profiling.argtypes = [C.c_void_p, C.c_int32]
        L.pb_set_profiling.restype = None
        L.pb_set_fast_approx.argtypes = [C.c_void_p, C.c_int32]
        L.pb_set_fast_approx.restype = None
        L.pb_set_fast_exact.argtypes = [C.c_void_p, C.c_int32]
        L.pb_set_fast_exact.restype = None
        L.pb_set_scores_tc.argtypes = [C.c_void_p, C.c_int32]
        L.pb_set_scores_tc.restype = None
        L.pb_set_lanes.argtypes = [C.c_void_p, C.c_int32]
        L.pb_set_lanes.restype = None
        L.pb_index_load.argtypes = [C.c_char_p, C.c_int32, C.POINTER(C.c_void_p)]
        L.pb_index_open.argtypes = [C.POINTER(_Desc), C.POINTER(C.c_void_p)]
        L.pb_search_batch_traced.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                             C.POINTER(_Params), C.c_void_p, C.c_int64, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p]
        L.pb_search_batch.argtypes = L.pb_search_batch_traced.argtypes[:-1]
        L.pb_search_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                             C.POINTER(_Params), C.c_void_p, C.c_void_p, C.c_void_p]
        L.pb_centroid_scores.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.pb_decompress_documents.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.pb_maxsim_scores.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_int64, C.c_void_p]
        L.pb_exhaustive_scores.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.pb_last_stage_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.pb_last_work_counters.argtypes = [C.c_void_p, C.POINTER(_Work)]
        L.pb_last_call_ms.argtypes = [C.c_void_p, C.c_void_p]
        L.pb_last_kernel_ms.argtypes = [C.c_void_p, C.c_void_p]
        L.pb_index_export_ivf.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pb_codec_open.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                    C.POINTER(C.c_void_p)]
        L.pb_codec_close.argtypes = [C.c_void_p]
        L.pb_codec_close.restype = None
        L.pb_codec_find_outliers.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p]
        L.pb_codec_last_assign_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pb_codec_compress_into_codes.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.pb_codec_compress_and_residuals.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.pb_codec_encode_chunk.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.pb_kmeans_fit.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.c_uint64,
                                    C.c_void_p]
        L.pb_codec_train.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        for f in ("pb_kmeans_num_sample_docs", "pb_codec_num_sample_docs", "pb_codec_heldout_tokens"):
            getattr(L, f).restype = C.c_int64
            getattr(L, f).argtypes = [C.c_int64]
        L.pb_kmeans_num_partitions.restype = C.c_int64
        L.pb_kmeans_num_partitions.argtypes = [C.c_int64, C.c_double, C.c_int64]
        L.pb_create_index.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_char_p, C.c_void_p]
        L.pb_create_params_default.argtypes = [C.c_void_p]
        L.pb_create_params_default.restype = None
        L.pb_build_comm_init.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        L.pb_build_comm_group.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.pb_build_comm_destroy.argtypes = [C.c_void_p]
        L.pb_build_comm_destroy.restype = None
        L.pb_kmeans_fit_dp.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.c_uint64, C.c_void_p]
        L.pb_comm_unique_id.argtypes = [C.c_void_p]
        L.pb_index_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
        L.pb_shard_group_create.argtypes = [C.c_int32, C.c_void_p]
        L.pb_shard_group_destroy.argtypes = [C.c_void_p]
        L.pb_shard_group_destroy.restype = None
        L.pb_index_group_join.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
        _lib = L
    return _lib


def _check(status: int):
    if status != PB_OK:
        raise PlaidError(status, load_library().pb_last_error().decode("utf-8", "replace"))


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class ShardGroup:
    """pb_shard_group: several shard handles of ONE process searched together (one host thread per shard).

    `search_batch` runs the collective from len(shards) threads and returns rank 0's result (every rank's
    result is identical; `all_results` keeps them for the tests).  Work counters are per host thread, so each
    rank's thread also records its `last_work_counters()` in `all_counters`."""

    def __init__(self, shards: Sequence["MmapIndex"]):
        self.shards = list(shards)
        h = C.c_void_p()
        _check(load_library().pb_shard_group_create(len(self.shards), C.byref(h)))
        self._g = h
        for r, s in enumerate(self.shards):
            _check(load_library().pb_index_group_join(s._h, self._g, r))
        self.all_results = None
        self.all_counters = None

    def search_batch(self, queries, params=None, subset=None):
        import threading
        out, err = [None] * len(self.shards), [None] * len(self.shards)
        counters = [None] * len(self.shards)

        def run(r):
            try:
                out[r] = self.shards[r].search_batch(queries, params, subset=subset)
                counters[r] = self.shards[r].last_work_counters()
            except Exception as e:      # noqa: BLE001 - re-raised below
                err[r] = e
        ths = [threading.Thread(target=run, args=(r,)) for r in range(len(self.shards))]
        [t.start() for t in ths]
        [t.join() for t in ths]
        for e in err:
            if e is not None:
                raise e
        self.all_results = out
        self.all_counters = counters
        return out[0]

    def close(self):
        for s in self.shards:
            s.close()
        self.shards = []
        if self._g:
            load_library().pb_shard_group_destroy(self._g)
            self._g = None


def comm_unique_id() -> bytes:
    """pb_comm_unique_id (rank 0); ship the 128 bytes to the other ranks."""
    buf = np.zeros(128, np.uint8)
    _check(load_library().pb_comm_unique_id(_ptr(buf)))
    return buf.tobytes()


def device_count() -> int:
    return int(load_library().pb_device_count())


@dataclass
class SearchParameters:
    """search.rs:27-69; defaults are SearchParameters::default() (search.rs:58-69)."""
    batch_size: int = 2000
    n_full_scores: int = 4096
    top_k: int = 10
    n_ivf_probe: int = 8
    centroid_batch_size: int = 100_000
    centroid_score_threshold: Optional[float] = 0.4

    def _c(self) -> _Params:
        t = self.centroid_score_threshold
        return _Params(self.batch_size, self.n_full_scores, self.top_k, self.n_ivf_probe,
                       self.centroid_batch_size, 0 if t is None else 1, 0.0 if t is None else float(t))


@dataclass
class QueryResult:
    """search.rs:72-80."""
    query_id: int
    passage_ids: np.ndarray
    scores: np.ndarray


@dataclass
class SearchTrace:
    cells: List[np.ndarray]
    candidates: List[np.ndarray]
    approx: List[np.ndarray]
    kept: List[np.ndarray]
    kept_exact: List[np.ndarray]


def _pack_queries(queries: Sequence[np.ndarray], dim: int):
    offs = np.zeros(len(queries) + 1, np.int64)
    for i, q in enumerate(queries):
        q = np.asarray(q)
        if q.ndim != 2 or q.shape[1] != dim:
            raise PlaidError(PB_ERR_INVALID, f"query {i} has shape {q.shape}, expected [tokens, {dim}]")
        offs[i + 1] = offs[i] + q.shape[0]
    flat = np.zeros((int(offs[-1]), dim), np.float32)
    for i, q in enumerate(queries):
        flat[offs[i]:offs[i + 1]] = q
    return flat, offs


class MmapIndex:
    """GPU-resident stand-in for next_plaid::MmapIndex (index.rs:995-1016)."""

    def __init__(self, handle: int, path: str = ""):
        self._h = C.c_void_p(handle)
        self.path = path

    # -- construction ----------------------------------------------------------------------
    @classmethod
    def load(cls, index_path: str, device: int = 0) -> "MmapIndex":
        """MmapIndex::load (index.rs:1026): reads the reference's index directory."""
        L = load_library()
        h = C.c_void_p()
        _check(L.pb_index_load(os.fsencode(index_path), device, C.byref(h)))
        return cls(h.value, index_path)

    @classmethod
    def from_arrays(cls, centroids, bucket_weights, codes, residuals, doc_lengths, ivf, ivf_lengths,
                    nbits: int, device: int = 0, doc_id_base: int = 0) -> "MmapIndex":
        """pb_index_open from host arrays in the reference's dtypes."""
        L = load_library()
        cen = np.ascontiguousarray(centroids, np.float32)
        w = np.ascontiguousarray(bucket_weights, np.float32)
        cd = np.ascontiguousarray(codes, np.int64)
        rs = np.ascontiguousarray(residuals, np.uint8)
        dl = np.ascontiguousarray(doc_lengths, np.int64)
        # ivf = ivf_lengths = None: the inverted file is built on the device from the codes (index.rs:850-873)
        iv = None if ivf is None else np.ascontiguousarray(ivf, np.int64)
        il = None if ivf_lengths is None else np.ascontiguousarray(ivf_lengths, np.int32)
        d = _Desc(cen.shape[1], nbits, cen.shape[0], len(dl), len(cd), _ptr(cen), _ptr(w), _ptr(cd),
                  _ptr(rs), _ptr(dl), _ptr(iv), _ptr(il), device, 0, doc_id_base, 0)
        h = C.c_void_p()
        _check(L.pb_index_open(C.byref(d), C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_device_pointers(cls, dim, nbits, K, D, N, centroids, bucket_weights, codes, residuals,
                             doc_lengths, ivf, ivf_lengths, device: int = 0, doc_id_base: int = 0,
                             adopt_residuals: bool = False):
        """pb_index_open with PB_MEM_DEVICE pointers (integers), e.g. torch tensors' data_ptr().  ivf = ivf_lengths
        = None: the inverted file is built on the device (index.rs:850-873).  adopt_residuals: the packed residuals
        are used in place (keep the array alive until close())."""
        L = load_library()
        d = _Desc(dim, nbits, K, D, N, centroids, bucket_weights, codes, residuals, doc_lengths, ivf,
                  ivf_lengths, device, 1, doc_id_base, 1 if adopt_residuals else 0)
        h = C.c_void_p()
        _check(L.pb_index_open(C.byref(d), C.byref(h)))
        return cls(h.value)

    def close(self):
        if self._h:
            load_library().pb_index_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- accessors (index.rs:1290-1312) ----------------------------------------------------------
    def num_documents(self) -> int:
        return int(load_library().pb_index_num_documents(self._h))

    def num_embeddings(self) -> int:
        return int(load_library().pb_index_num_embeddings(self._h))

    def num_partitions(self) -> int:
        return int(load_library().pb_index_num_partitions(self._h))

    def avg_doclen(self) -> float:
        return float(load_library().pb_index_avg_doclen(self._h))

    def embedding_dim(self) -> int:
        return int(load_library().pb_index_embedding_dim(self._h))

    def nbits(self) -> int:
        return int(load_library().pb_index_nbits(self._h))

    # -- search ------------------------------------------------------------------------------
    def search(self, query: np.ndarray, params: SearchParameters,
               subset: Optional[Sequence[int]] = None) -> QueryResult:
        """MmapIndex::search (index.rs:1258)."""
        r = self.search_batch([query], params, True, subset)[0]
        r.query_id = 0
        return r

    def search_batch(self, queries: Sequence[np.ndarray], params: SearchParameters,
                     parallel: bool = True, subset: Optional[Sequence[int]] = None,
                     trace: bool = False):
        """MmapIndex::search_batch (index.rs:1279).  `parallel` is accepted for signature parity;
        the GPU always processes the batch together."""
        L = load_library()
        flat, offs = _pack_queries(queries, self.embedding_dim())
        B, k = len(queries), max(int(params.top_k), 0)
        ids = np.zeros((B, max(k, 1)), np.int64)
        sc = np.zeros((B, max(k, 1)), np.float32)
        cn = np.zeros(B, np.int32)
        ss = None if subset is None else np.ascontiguousarray(subset, np.int64)
        p = params._c()
        tr, bufs = None, None
        if trace:
            D, K = self.num_documents(), self.num_partitions()
            M = max(min(params.n_full_scores, max(params.n_full_scores // 4, params.top_k)), 1)
            cc = min(K, max(int(offs[-1]) * max(params.n_ivf_probe, 1), 1)) if ss is None else K
            bufs = dict(cells=np.zeros((B, cc), np.int64), n_cells=np.zeros(B, np.int32),
                        cand=np.zeros((B, max(D, 1)), np.int64), approx=np.zeros((B, max(D, 1)), np.float32),
                        n_cand=np.zeros(B, np.int32), kept=np.zeros((B, M), np.int64),
                        kex=np.zeros((B, M), np.float32), n_kept=np.zeros(B, np.int32))
            tr = _Trace(_ptr(bufs["cells"]), _ptr(bufs["n_cells"]), cc, _ptr(bufs["cand"]),
                        _ptr(bufs["approx"]), _ptr(bufs["n_cand"]), max(D, 1), _ptr(bufs["kept"]),
                        _ptr(bufs["kex"]), _ptr(bufs["n_kept"]), M)
        _check(L.pb_search_batch_traced(self._h, _ptr(flat), _ptr(offs), B, C.byref(p), _ptr(ss),
                                        0 if ss is None else len(ss), _ptr(ids), _ptr(sc), _ptr(cn),
                                        None if tr is None else C.cast(C.pointer(tr), C.c_void_p)))
        res = [QueryResult(i, ids[i, :cn[i]].copy(), sc[i, :cn[i]].copy()) for i in range(B)]
        if trace:
            t = SearchTrace(
                [bufs["cells"][i, :bufs["n_cells"][i]].copy() for i in range(B)],
                [bufs["cand"][i, :bufs["n_cand"][i]].copy() for i in range(B)],
                [bufs["approx"][i, :bufs["n_cand"][i]].copy() for i in range(B)],
                [bufs["kept"][i, :bufs["n_kept"][i]].copy() for i in range(B)],
                [bufs["kex"][i, :bufs["n_kept"][i]].copy() for i in range(B)])
            return res, t
        return res

    # -- stage entry points --------------------------------------------------------------------
    def centroid_scores(self, query_tokens: np.ndarray) -> np.ndarray:
        """Stage 1, S = Q.C^T (search.rs:345), [n_tokens, K]."""
        q = np.ascontiguousarray(query_tokens, np.float32)
        out = np.zeros((q.shape[0], self.num_partitions()), np.float32)
        _check(load_library().pb_centroid_scores(self._h, _ptr(q), q.shape[0], _ptr(out)))
        return out

    def decompress_documents(self, doc_ids: Sequence[int]):
        """MmapIndex::decompress_documents (index.rs:1197): (embeddings [sum len, dim], lengths)."""
        L = load_library()
        ids = np.ascontiguousarray(doc_ids, np.int64)
        lens = np.zeros(len(ids), np.int64)
        _check(L.pb_decompress_documents(self._h, _ptr(ids), len(ids), None, _ptr(lens)))
        emb = np.zeros((int(lens.sum()), self.embedding_dim()), np.float32)
        if emb.shape[0]:
            _check(L.pb_decompress_documents(self._h, _ptr(ids), len(ids), _ptr(emb), _ptr(lens)))
        return emb, lens

    def get_document_embeddings(self, doc_id: int) -> np.ndarray:
        """MmapIndex::get_document_embeddings (index.rs:1159)."""
        if not (0 <= doc_id < self.num_documents()):
            raise PlaidError(PB_ERR_INVALID, f"Invalid document ID: {doc_id}")
        return self.decompress_documents([doc_id])[0]

    def exhaustive_scores(self, queries: Sequence[np.ndarray]) -> np.ndarray:
        """Exact MaxSim of each query against every document (recall ground truth)."""
        flat, offs = _pack_queries(queries, self.embedding_dim())
        out = np.zeros((len(queries), self.num_documents()), np.float32)
        _check(load_library().pb_exhaustive_scores(self._h, _ptr(flat), _ptr(offs), len(queries), _ptr(out)))
        return out

    # -- doc-sharded deployment ------------------------------------------------------------------
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        """pb_index_comm_init: after this, search_batch is a collective over `world` ranks."""
        buf = np.frombuffer(bytes(unique_id), np.uint8).copy()
        assert buf.size == 128
        _check(load_library().pb_index_comm_init(self._h, _ptr(buf), rank, world))

    # -- measurement hooks -------------------------------------------------------------------------
    def set_fast_approx(self, mode):
        """0/False = single exact pass over every candidate, 1/True = two-pass (default)."""
        load_library().pb_set_fast_approx(self._h, int(mode))

    def set_scores_tc(self, on: bool):
        """a2 on the tensor cores (default on) vs the dense fp32 kernel; same results either way."""
        load_library().pb_set_scores_tc(self._h, 1 if on else 0)

    def set_fast_exact(self, on: bool):
        """tcgen05 certified filter in front of the exact stage (default on); same results either way."""
        load_library().pb_set_fast_exact(self._h, 1 if on else 0)

    def set_profiling(self, on: bool):
        load_library().pb_set_profiling(self._h, 1 if on else 0)

    def set_lanes(self, lanes: int):
        """Slices of a batch searched concurrently inside one call (pb_set_lanes); 1 = off."""
        load_library().pb_set_lanes(self._h, int(lanes))

    def last_stage_stats(self):
        ms = np.zeros(len(STAGES), np.float32)
        ln = np.zeros(len(STAGES), np.int32)
        _check(load_library().pb_last_stage_stats(self._h, _ptr(ms), _ptr(ln)))
        return dict(zip(STAGES, ms.tolist())), dict(zip(STAGES, ln.tolist()))

    def export_ivf(self):
        """pb_index_export_ivf: (ivf <i8 global doc ids, ivf_lengths <i4), what create_index writes to ivf.npy /
        ivf_lengths.npy (index.rs:501-508)."""
        L = load_library()
        tot = C.c_int64()
        _check(L.pb_index_export_ivf(self._h, None, None, C.byref(tot)))
        ivf = np.zeros(max(tot.value, 1), np.int64)
        lens = np.zeros(self.num_partitions(), np.int32)
        _check(L.pb_index_export_ivf(self._h, _ptr(ivf), _ptr(lens), C.byref(tot)))
        return ivf[:tot.value], lens

    def last_call_ms(self) -> float:
        v = np.zeros(1, np.float32)
        _check(load_library().pb_last_call_ms(self._h, _ptr(v)))
        return float(v[0])

    def last_kernel_ms(self) -> dict:
        v = np.zeros(4, np.float32)
        _check(load_library().pb_last_kernel_ms(self._h, _ptr(v)))
        return dict(zip(("scores", "approx16", "filter", "exact"), v.tolist()))

    def last_work_counters(self) -> dict:
        w = _Work()
        _check(load_library().pb_last_work_counters(self._h, C.byref(w)))
        return {n: int(getattr(w, n)) for n, _ in _Work._fields_}

    def search_batch_device(self, d_queries_ptr: int, q_tok_offsets: np.ndarray, params: SearchParameters,
                            d_ids_ptr: int, d_scores_ptr: int, d_counts_ptr: int):
        """pb_search_batch_device: queries and results stay on the device (kernel-only timing)."""
        offs = np.ascontiguousarray(q_tok_offsets, np.int64)
        p = params._c()
        _check(load_library().pb_search_batch_device(self._h, d_queries_ptr, _ptr(offs), len(offs) - 1,
                                                     C.byref(p), d_ids_ptr, d_scores_ptr, d_counts_ptr))


def maxsim_scores(query: np.ndarray, docs: Sequence[np.ndarray], device: int = 0) -> np.ndarray:
    """maxsim::maxsim_score (maxsim.rs:270) for a list of already-decompressed documents."""
    q = np.ascontiguousarray(query, np.float32)
    offs = np.zeros(len(docs) + 1, np.int64)
    for i, d in enumerate(docs):
        offs[i + 1] = offs[i] + d.shape[0]
    flat = np.zeros((int(offs[-1]), q.shape[1]), np.float32)
    for i, d in enumerate(docs):
        flat[offs[i]:offs[i + 1]] = d
    out = np.zeros(len(docs), np.float32)
    _check(load_library().pb_maxsim_scores(device, _ptr(q), q.shape[0], q.shape[1], _ptr(flat), _ptr(offs),
                                           len(docs), _ptr(out)))
    return out


class _CreateParams(C.Structure):
    _fields_ = [("nbits", C.c_int32), ("kmeans_niters", C.c_int32), ("max_points_per_centroid", C.c_int32),
                ("device", C.c_int32), ("num_partitions", C.c_int64), ("batch_size", C.c_int64), ("seed", C.c_uint64)]


def create_index(embeddings: Sequence[np.ndarray], index_dir: str, nbits: int = 4, kmeans_niters: int = 4,
                 num_partitions: int = 0, batch_size: int = 50_000, seed: int = 42, device: int = 0,
                 max_points_per_centroid: int = 256) -> "MmapIndex":
    """MmapIndex::create_with_kmeans (index.rs:1392): builds the reference's index directory from document embeddings
    on the GPU (pb_create_index) and returns the open index."""
    L = load_library()
    dl = np.array([e.shape[0] for e in embeddings], np.int64)
    flat = np.ascontiguousarray(np.concatenate(embeddings, 0), np.float32)
    p = _CreateParams(nbits, kmeans_niters, max_points_per_centroid, device, num_partitions, batch_size, seed)
    h = C.c_void_p()
    _check(L.pb_create_index(_ptr(flat), _ptr(dl), len(dl), flat.shape[1], C.byref(p), index_dir.encode(), C.byref(h)))
    return MmapIndex(h.value)


def kmeans_fit_dp(shards: Sequence[np.ndarray], K: int, niters: int = 4, seed: int = 42, device: int = 0,
                  nccl: Optional[tuple] = None) -> np.ndarray:
    """pb_kmeans_fit_dp.  Without `nccl`: the shards are fitted by len(shards) host threads of this process through an
    in-process shard group (all on `device`); with nccl = (unique_id, rank, world) the single shard shards[0] is this
    rank's part of an NCCL job.  Returns the centroids (identical on every rank)."""
    L = load_library()
    dim = shards[0].shape[1]
    if nccl is not None:
        uid, rank, world = nccl
        buf = np.frombuffer(bytes(uid), np.uint8).copy()
        h = C.c_void_p()
        _check(L.pb_build_comm_init(_ptr(buf), rank, world, device, C.byref(h)))
        x = np.ascontiguousarray(shards[0], np.float32)
        out = np.zeros((K, dim), np.float32)
        try:
            _check(L.pb_kmeans_fit_dp(h, _ptr(x), x.shape[0], dim, K, niters, seed, _ptr(out)))
        finally:
            L.pb_build_comm_destroy(h)
        return out
    import threading
    G = len(shards)
    g = C.c_void_p()
    _check(L.pb_shard_group_create(G, C.byref(g)))
    outs, errs = [None] * G, [None] * G

    def run(r):
        try:
            h = C.c_void_p()
            _check(L.pb_build_comm_group(g, r, device, C.byref(h)))
            x = np.ascontiguousarray(shards[r], np.float32)
            out = np.zeros((K, dim), np.float32)
            try:
                _check(L.pb_kmeans_fit_dp(h, _ptr(x), x.shape[0], dim, K, niters, seed, _ptr(out)))
            finally:
                L.pb_build_comm_destroy(h)
            outs[r] = out
        except Exception as e:      # noqa: BLE001 - re-raised below
            errs[r] = e
    ths = [threading.Thread(target=run, args=(r,)) for r in range(G)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    L.pb_shard_group_destroy(g)
    for e in errs:
        if e is not None:
            raise e
    for o in outs[1:]:
        assert np.array_equal(o, outs[0]), "ranks disagree on the centroids"
    return outs[0]


def kmeans_sizing(num_documents: int, avg_sample_doclen: float, num_sample_tokens: int, num_embeddings: int) -> dict:
    """The sizing rules of compute_kmeans (kmeans.rs:273-312) and prepare_codec_artifacts (index.rs:195-212)."""
    L = load_library()
    return {"kmeans_sample_docs": int(L.pb_kmeans_num_sample_docs(num_documents)),
            "num_partitions": int(L.pb_kmeans_num_partitions(num_documents, float(avg_sample_doclen), num_sample_tokens)),
            "codec_sample_docs": int(L.pb_codec_num_sample_docs(num_documents)),
            "heldout_tokens": int(L.pb_codec_heldout_tokens(num_embeddings))}


class ResidualCodec:
    """Device-resident next_plaid::ResidualCodec (codec.rs:107-123) for the index-build path."""

    def __init__(self, nbits: int, centroids: np.ndarray, bucket_cutoffs: Optional[np.ndarray] = None,
                 device: int = 0):
        cen = np.ascontiguousarray(centroids, np.float32)
        cut = None if bucket_cutoffs is None else np.ascontiguousarray(bucket_cutoffs, np.float32)
        h = C.c_void_p()
        _check(load_library().pb_codec_open(device, _ptr(cen), cen.shape[0], cen.shape[1], nbits, _ptr(cut),
                                            C.byref(h)))
        self._h, self.nbits, self.dim = h, nbits, cen.shape[1]

    def close(self):
        if self._h:
            load_library().pb_codec_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def last_assign_stats(self) -> dict:
        n, f, tc = C.c_int64(), C.c_int64(), C.c_int32()
        _check(load_library().pb_codec_last_assign_stats(self._h, C.byref(n), C.byref(f), C.byref(tc)))
        return {"tokens": n.value, "exact_fallback": f.value, "tensor_cores": bool(tc.value)}

    def compress_into_codes(self, embeddings: np.ndarray) -> np.ndarray:
        """codec.rs:260."""
        e = np.ascontiguousarray(embeddings, np.float32)
        out = np.zeros(e.shape[0], np.int64)
        _check(load_library().pb_codec_compress_into_codes(self._h, _ptr(e), e.shape[0], _ptr(out)))
        return out

    def compress_and_residuals(self, embeddings: np.ndarray):
        """index.rs:17-40."""
        e = np.ascontiguousarray(embeddings, np.float32)
        codes = np.zeros(e.shape[0], np.int64)
        res = np.zeros_like(e)
        _check(load_library().pb_codec_compress_and_residuals(self._h, _ptr(e), e.shape[0], _ptr(codes), _ptr(res)))
        return codes, res

    def find_outliers(self, embeddings: np.ndarray, threshold_sq: float) -> np.ndarray:
        """update.rs:490: row indices farther than sqrt(threshold_sq) from every centroid."""
        e = np.ascontiguousarray(embeddings, np.float32)
        out = np.zeros(max(e.shape[0], 1), np.int64)
        cnt = C.c_int64()
        _check(load_library().pb_codec_find_outliers(self._h, _ptr(e), e.shape[0], float(threshold_sq), _ptr(out),
                                                     C.byref(cnt)))
        return out[:cnt.value].copy()

    def train(self, heldout: np.ndarray):
        """pb_codec_train (prepare_codec_artifacts, index.rs:228-287, on held-out rows the caller sampled):
        (bucket_cutoffs, bucket_weights, avg_residual, cluster_threshold); the codec keeps the cutoffs."""
        e = np.ascontiguousarray(heldout, np.float32).reshape(-1, self.dim)
        nopt = 1 << self.nbits
        cut, wts, avg = np.zeros(max(nopt - 1, 1), np.float32), np.zeros(nopt, np.float32), np.zeros(self.dim, np.float32)
        thr = C.c_float()
        _check(load_library().pb_codec_train(self._h, _ptr(e), e.shape[0], _ptr(cut), _ptr(wts), _ptr(avg), C.byref(thr)))
        return cut[:nopt - 1], wts, avg, float(thr.value)

    def encode_chunk(self, embeddings: np.ndarray):
        """encode_index_chunk (index.rs:289): (codes i64 [n], packed residuals u8 [n, dim*nbits/8])."""
        e = np.ascontiguousarray(embeddings, np.float32)
        codes = np.zeros(e.shape[0], np.int64)
        packed = np.zeros((e.shape[0], self.dim * self.nbits // 8), np.uint8)
        _check(load_library().pb_codec_encode_chunk(self._h, _ptr(e), e.shape[0], _ptr(codes), _ptr(packed)))
        return codes, packed


def kmeans_fit(samples: np.ndarray, num_centroids: int, niters: int = 4, seed: int = 42, device: int = 0) -> np.ndarray:
    """The fit inside compute_kmeans (kmeans.rs:319-419): Lloyd iterations + L2 normalisation."""
    x = np.ascontiguousarray(samples, np.float32)
    out = np.zeros((num_centroids, x.shape[1]), np.float32)
    _check(load_library().pb_kmeans_fit(device, _ptr(x), x.shape[0], x.shape[1], num_centroids, niters, seed, _ptr(out)))
    return out
