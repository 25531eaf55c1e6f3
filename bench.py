#!/usr/bin/env python
"""bench.py -- queries/sec of the PLAID search hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W                     # the CUDA path (this repo)
    python bench.py --impl reference --gpus N --steps K --warmup W    # the reference's CPU algorithm
    python bench.py ... --dump-outputs DIR     # also write the last timed step's results as DIR/*.npy

The inputs are a function of the arguments alone (seeded), so two builds run with the same arguments can be
compared output for output.  Nothing is written under the repository: the tree may be read-only.

One "step" = one batch of queries searched through the whole path (centroid scoring -> probe -> candidates ->
approximate score -> cut -> decompress + MaxSim -> top-k) against a synthetic index resident in HBM.

  N = 1   BASELINE.json configs[1]: 1M docs x 300 tok x 128-d, 4-bit residuals, K = 2^18, batch 32 queries x 32 tokens,
          top_k = 100 (the largest configuration of `configs` that fits one GPU: 10M docs at 4 bits is 204 GB).
  N > 1   configs[2]: the SAME fixed 10M-doc corpus doc-sharded over the N ranks (N = 8: 1.25M docs per GPU), batch 256,
          queries replicated, results merged by the two exchanges of DESIGN.md section 5 ("scaling": "strong").  The N = 1 line is a
          different workload (1M docs, batch 32), so value_N / value_1 is not an efficiency; the basis of the
          strong-scaling curve is the smallest N that holds the corpus (N = 2 with adopted residuals).

Rank 0 prints ONE JSON line:
  value     whole-job queries/sec with queries already in HBM: one CUDA-event pair on the library's stream around every
            search call (pb_last_call_ms), max over ranks
  e2e       the same metric through the public C-ABI call with HOST buffers (pinned queries in, host results out),
            H2D / D2H inside the timed region, wall clock, max over ranks
  roofline  the dominant kernel by device time (CUDA events around that one launch, pb_last_kernel_ms): algorithmic
            bytes / time against the measured HBM peak of MEASURED_PEAKS.json; roofline_all holds every measured
            kernel, `maxsim` the decompress + MaxSim kernels the BASELINE metric names
  parity    this run's results against the CPU oracle (ids identical, max |score difference|) on a sample, and the
            library against itself over EVERY timed query with the tensor-core paths switched off
  cpu_baseline  the CPU oracle (C restatement of the reference's Rust path, OpenMP) timed on this box's host cores on
            that sample (N = 1 only)

Synthetic corpus (seed 42), generated directly in the codec domain -- centroid code + packed residual per token, so a
token IS normalise(C[code] + w[bucket]) (codec.rs:455-467) -- in chunks of 50 000 docs (the reference's own chunk
size, index.rs:88-102) seeded by chunk index, so the corpus is the same for every N.  Every doc belongs to one of
D/1024 topics, a topic owns a pool of 256 centroids; a token draws its code from the pool (70 %, skewed), uniformly
(20 %) or from 4096 hub centroids (10 %).  A query is 32 tokens of one doc, each perturbed by 0.15 x unit noise.
The library builds the inverted file itself (index.rs:850-873) and uses the residual array in place.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # no __pycache__ in the tree
if "--impl" in sys.argv and "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is a CPU measurement and uses every host thread
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import numpy as np  # noqa: E402

CHUNK_DOCS = int(os.environ.get("PB_BENCH_CHUNK_DOCS", 50_000))
# dry-run hooks for tests/test_bench_harness_cpu.py: a stand-in library module and a CPU torch device
LIB_MODULE = os.environ.get("PB_BENCH_LIB", "next_plaid_b200")
DEVICE_TYPE = os.environ.get("PB_BENCH_DEVICE", "cuda")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--docs-total", type=int, default=0, help="corpus size; 0 = 1M at N=1, 10M at N>1")
    ap.add_argument("--doclen", type=int, default=300)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--nbits", type=int, default=4)
    ap.add_argument("--log2k", type=int, default=18)
    ap.add_argument("--batch", type=int, default=0, help="queries per step; 0 = 32 at N=1, 256 at N>1")
    ap.add_argument("--nq", type=int, default=32)
    ap.add_argument("--top-k", type=int, default=100)
    ap.add_argument("--n-ivf-probe", type=int, default=8)
    ap.add_argument("--n-full-scores", type=int, default=4096)
    ap.add_argument("--threshold", type=float, default=0.4)
    ap.add_argument("--recall-queries", type=int, default=-1, help="-1 = 256 at N=1, 128 at N>1")
    ap.add_argument("--parity-queries", type=int, default=-1, help="oracle-checked queries; -1 = 64 at N=1, 16 at N>1")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU oracle (parity + cpu_baseline)")
    ap.add_argument("--threads", type=int, default=2, help="host threads for the extra concurrent-callers measurement")
    ap.add_argument("--lanes", type=int, default=0, help="pb_set_lanes (0 = the library's default, 1 = off)")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--docs-per-topic", type=int, default=1024)
    ap.add_argument("--pool", type=int, default=256, help="centroids per topic pool")
    ap.add_argument("--res-sigma", type=float, default=0.05, help="per-dimension residual scale")
    ap.add_argument("--query-noise", type=float, default=0.15)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's results as DIR/passage_ids.npy, scores.npy, counts.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", 1))
    if a.docs_total <= 0:
        a.docs_total = 1_000_000 if world == 1 else 10_000_000
    if a.batch <= 0:
        a.batch = 32 if world == 1 else 256
    if a.recall_queries < 0:
        a.recall_queries = 256 if world == 1 else 128
    if a.parity_queries < 0:
        a.parity_queries = 64 if world == 1 else 16
    return a


# ----------------------------------------------------------------------------------------------
# synthetic corpus in the codec domain, generated on the GPU with torch (harness, not product)
# ----------------------------------------------------------------------------------------------
def chunk_layout(args, world):
    """(docs per rank, chunk size, chunks per rank): chunk boundaries do not depend on N for the default sizes."""
    if args.docs_total % world:
        raise SystemExit(f"--docs-total {args.docs_total} is not a multiple of {world} ranks")
    per_rank = args.docs_total // world
    chunk = CHUNK_DOCS if per_rank % CHUNK_DOCS == 0 else per_rank // max(1, -(-per_rank // CHUNK_DOCS))
    if per_rank % chunk:
        raise SystemExit(f"{per_rank} docs per rank do not split into equal chunks of about {CHUNK_DOCS}")
    return per_rank, chunk, per_rank // chunk


def corpus_globals(args, device):
    import torch
    K, dim, nbits = 1 << args.log2k, args.dim, args.nbits
    g = torch.Generator(device=device)
    g.manual_seed(args.seed)
    cent = torch.randn(K, dim, generator=g, device=device, dtype=torch.float32)
    cent /= cent.norm(dim=1, keepdim=True)
    n_topics = max(args.docs_total // args.docs_per_topic, 4)
    P = min(args.pool, K)
    pools = torch.randint(0, K, (n_topics, P), generator=g, device=device, dtype=torch.int32)
    hubs = torch.randint(0, K, (4096,), generator=g, device=device, dtype=torch.int64)   # stop-word-like centroids
    nb = 1 << nbits
    probs = (torch.arange(nb, dtype=torch.float64) + 0.5) / nb
    w = (args.res_sigma * torch.special.ndtri(probs)).to(torch.float32).to(device)   # quantile mid-points of N(0, s^2)
    return dict(centroids=cent, pools=pools, hubs=hubs, bucket_weights=w, n_topics=n_topics, P=P, K=K)


def gen_chunk(args, G, chunk_index: int, n_docs: int, device):
    """codes i64 [n_docs*T], residuals u8 [n_docs*T, packed] of chunk `chunk_index` (a function of seed and index)."""
    import torch
    T, K, P = args.doclen, G["K"], G["P"]
    g = torch.Generator(device=device)
    g.manual_seed(args.seed * 1_000_003 + 7919 * (chunk_index + 1))
    n = n_docs * T
    topic = torch.randint(0, G["n_topics"], (n_docs,), generator=g, device=device, dtype=torch.int64).repeat_interleave(T)
    u = torch.rand(n, generator=g, device=device)
    pidx = (u * u * P).to(torch.int64).clamp_(max=P - 1)
    from_pool = G["pools"][topic, pidx].to(torch.int64)
    rnd = torch.randint(0, K, (n,), generator=g, device=device, dtype=torch.int64)
    sel = torch.rand(n, generator=g, device=device)
    hub = G["hubs"][torch.randint(0, 4096, (n,), generator=g, device=device)]
    codes = torch.where(sel < 0.7, from_pool, torch.where(sel < 0.9, rnd, hub))
    residuals = torch.randint(0, 256, (n, args.dim * args.nbits // 8), generator=g, device=device, dtype=torch.uint8)
    return codes, residuals


def build_shard(args, G, rank, world, device):
    """This rank's contiguous doc range as device tensors (codes i64, residuals u8, doc_lengths i64)."""
    import torch
    per_rank, chunk, n_chunks = chunk_layout(args, world)
    T, packed = args.doclen, args.dim * args.nbits // 8
    N = per_rank * T
    codes = torch.empty(N, dtype=torch.int64, device=device)
    residuals = torch.empty((N, packed), dtype=torch.uint8, device=device)
    for c in range(n_chunks):
        cc, rr = gen_chunk(args, G, rank * n_chunks + c, chunk, device)
        codes[c * chunk * T:(c + 1) * chunk * T] = cc
        residuals[c * chunk * T:(c + 1) * chunk * T] = rr
        del cc, rr
    doc_lengths = torch.full((per_rank,), T, dtype=torch.int64, device=device)
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    return dict(codes=codes, residuals=residuals, doc_lengths=doc_lengths, D=per_rank, N=N)


def open_shard(npb, args, G, sh, device_index, base):
    # the library builds the inverted file from the codes (ivf = None) and uses the residual array in place
    return npb.MmapIndex.from_device_pointers(
        args.dim, args.nbits, G["K"], sh["D"], sh["N"], G["centroids"].data_ptr(), G["bucket_weights"].data_ptr(),
        sh["codes"].data_ptr(), sh["residuals"].data_ptr(), sh["doc_lengths"].data_ptr(), None, None,
        device=device_index, doc_id_base=base, adopt_residuals=True)


def _bitrev(v, nbits):
    r = 0
    for k in range(nbits):
        if v & (1 << k):
            r |= 1 << (nbits - 1 - k)
    return r


def make_queries(args, G, device, n_queries: int, seed: int):
    """Queries from docs of chunk 0: nq tokens of one doc (decoded in the harness from the generator's own arrays:
    normalise(C[code] + w[bucket]), first dim in the high bits, bucket index bit-reversed, codec.rs:389-395 / :449-467),
    each perturbed by query_noise x unit noise.  Both arms call this with the same seed."""
    import torch
    _, chunk, _ = chunk_layout(args, int(os.environ.get("WORLD_SIZE", 1)))
    codes, res = gen_chunk(args, G, 0, chunk, device)
    T, nbits, dim = args.doclen, args.nbits, args.dim
    rng = np.random.default_rng(seed)
    src = rng.integers(0, chunk, size=n_queries)
    shifts = torch.tensor([8 - nbits * (j + 1) for j in range(8 // nbits)], device=device, dtype=torch.int32)
    w = G["bucket_weights"]
    w_rev = torch.stack([w[_bitrev(f, nbits)] for f in range(1 << nbits)])
    out = []
    for d in src.tolist():
        tok = torch.from_numpy(rng.integers(0, T, size=args.nq)).to(device) + d * T
        c = codes[tok]
        fields = ((res[tok].to(torch.int32).unsqueeze(-1) >> shifts) & ((1 << nbits) - 1)).reshape(args.nq, dim)
        v = G["centroids"][c] + w_rev[fields.to(torch.int64)]
        v = (v / v.norm(dim=1, keepdim=True).clamp_min(1e-12)).cpu().numpy()
        noise = rng.standard_normal(v.shape).astype(np.float32)
        noise /= np.linalg.norm(noise, axis=1, keepdims=True)
        q = v + args.query_noise * noise
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        out.append(np.ascontiguousarray(q, np.float32))
    del codes, res
    return out


def host_corpus(oracle, args, G, device, world):
    """The whole corpus in host memory as one oracle.Index per 50 000-doc chunk (each with its own inverted file);
    oracle.search_sharded over them equals a search of the concatenated index."""
    import torch
    per_rank, chunk, n_chunks = chunk_layout(args, world)
    cent = G["centroids"].cpu().numpy()
    w = G["bucket_weights"].cpu().numpy()
    K, T = G["K"], args.doclen
    shards, bases = [], []
    for c in range(n_chunks * world):
        codes, res = gen_chunk(args, G, c, chunk, device)
        doc = torch.arange(chunk, device=device, dtype=torch.int64).repeat_interleave(T)
        keys = torch.unique(codes * chunk + doc)
        ivf = (keys % chunk).cpu().numpy()
        ivf_lengths = torch.bincount(keys // chunk, minlength=K).to(torch.int32).cpu().numpy()
        shards.append(oracle.Index(cent, w, None, codes.cpu().numpy(), res.cpu().numpy(),
                                   np.full(chunk, T, np.int64), ivf, ivf_lengths, args.nbits))
        bases.append(c * chunk)
        del codes, res, doc, keys
    return shards, bases


def host_bytes_needed(args):
    tok = args.docs_total * args.doclen
    return int(tok * (args.dim * args.nbits // 8 + 8 + 6) * 1.1)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return dict(hbm=float(j["hbm_gbs"]), bf16=float(j.get("bf16_tflops_sustained", j.get("bf16_tflops", 1435.1))),
                        src="measured (MEASURED_PEAKS.json)")
        except Exception:
            pass
    return dict(hbm=6650.0, bf16=1400.0, src="fallback (B200_PROFILING.md)")


def workload_config(args, world):
    per_rank = args.docs_total // world
    name = {1_000_000: "BASELINE configs[1]", 10_000_000: "BASELINE configs[2]"}.get(args.docs_total, "custom")
    return {"workload": f"{name}: {args.docs_total // 1000}k docs x {args.doclen} tok x {args.dim}-d, {args.nbits}-bit, "
                        f"K=2^{args.log2k}, batch {args.batch} x {args.nq} query tokens, top_k {args.top_k}",
            "docs_per_gpu": per_rank, "total_docs": args.docs_total, "doclen": args.doclen, "dim": args.dim,
            "nbits": args.nbits, "num_centroids": 1 << args.log2k, "batch_queries": args.batch,
            "query_tokens": args.nq, "top_k": args.top_k, "n_ivf_probe": args.n_ivf_probe,
            "n_full_scores": args.n_full_scores, "centroid_score_threshold": args.threshold,
            "variant": "batched" if (1 << args.log2k) > 100_000 else "dense",
            "parallelism": f"doc-shard x{world} (fixed corpus)" if world > 1 else "single GPU",
            "l2": "index (>= 20 GB/GPU) exceeds the 126 MB L2; a distinct query batch every step"}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, ids, scores, counts):
    """Write what one search call returned, one row per query, so that two builds can be compared output for output:
    passage_ids.npy (f64, exact for any doc id below 2^53), scores.npy (f32) and counts.npy (f64).  Slots past a row's
    count are undefined in the library's output; they are written as id -1 and score 0.  When the arrays exceed 64 MB,
    a fixed, seeded sample of rows is written instead, with the sampled row numbers in rows.npy."""
    ids, scores, counts = np.asarray(ids, np.int64), np.asarray(scores, np.float32), np.asarray(counts, np.int64)
    valid = np.arange(ids.shape[1])[None, :] < counts[:, None]
    out = {"passage_ids": np.where(valid, ids, -1).astype(np.float64),
           "scores": np.where(valid, scores, np.float32(0)).astype(np.float32),
           "counts": counts.astype(np.float64)}
    row_bytes = sum(a[0].nbytes for a in out.values()) + 8
    if len(counts) * row_bytes > DUMP_MAX_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(len(counts), DUMP_MAX_BYTES // row_bytes, replace=False))
        out = {name: a[rows] for name, a in out.items()}
        out["rows"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def same_results(a, b):
    ids = sum(int(x.passage_ids.tolist() == y.passage_ids.tolist()) for x, y in zip(a, b))
    dmax = 0.0
    for x, y in zip(a, b):
        if len(x.scores) != len(y.scores):
            dmax = float("inf")
        elif len(x.scores):
            dmax = max(dmax, float(np.abs(x.scores - y.scores).max()))
    return ids, dmax


# ----------------------------------------------------------------------------------------------
def run_b200(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    import importlib
    npb = importlib.import_module(LIB_MODULE)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(minutes=30))
    on_gpu = DEVICE_TYPE == "cuda"
    dev = torch.device("cuda", local) if on_gpu else torch.device("cpu")
    sync = (lambda: torch.cuda.synchronize(dev)) if on_gpu else (lambda: None)
    if on_gpu:
        torch.cuda.set_device(dev)
    t0 = time.time()
    G = corpus_globals(args, dev)
    sh = build_shard(args, G, rank, world, dev)
    t_gen = time.time() - t0
    per_rank = sh["D"]
    gpu = open_shard(npb, args, G, sh, local, rank * per_rank)
    del sh["codes"]                                   # the library narrowed them to u32; residuals stay (adopted)
    if on_gpu:
        torch.cuda.empty_cache()
    t_build = time.time() - t0
    if world > 1:   # doc-sharded: the library runs its own NCCL all-gathers; torch only ships the unique id
        uid = [npb.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        gpu.comm_init(uid[0], rank, world)
    params = npb.SearchParameters(top_k=args.top_k, n_ivf_probe=args.n_ivf_probe, n_full_scores=args.n_full_scores,
                                  centroid_score_threshold=args.threshold)
    n_batches = min(max(args.steps + args.warmup, 4), 24)
    n_q = max(n_batches * args.batch, args.recall_queries, args.parity_queries)
    queries = make_queries(args, G, dev, n_q, seed=args.seed + 7)      # deterministic: every rank draws the same
    batches = [queries[i * args.batch:(i + 1) * args.batch] for i in range(n_batches)]

    # ---- recall@top_k against exhaustive exact MaxSim over the decompressed corpus (untimed) ----
    rq = queries[:args.recall_queries]
    recall = None
    if rq:
        top = []
        for i0 in range(0, len(rq), 32):                     # 32 queries x docs-per-GPU floats at a time
            part = rq[i0:i0 + 32]
            ex = gpu.exhaustive_scores(part)                 # this shard's docs
            for i in range(len(part)):
                o = np.argpartition(-ex[i], min(args.top_k, ex.shape[1] - 1))[:args.top_k]
                o = o[np.lexsort((o, -ex[i][o]))]
                top.append([(float(ex[i][j]), int(j) + rank * per_rank) for j in o])
            del ex
        res = []
        for i0 in range(0, len(rq), args.batch):
            res += gpu.search_batch(rq[i0:i0 + args.batch], params)       # collective when sharded
        if world > 1:
            alls = [None] * world
            dist.all_gather_object(alls, top)
            top = [sorted((t for part in alls for t in part[i]), key=lambda t: (-t[0], t[1]))[:args.top_k]
                   for i in range(len(rq))]
        hits = [len({t[1] for t in top[i]} & set(r.passage_ids.tolist())) / float(args.top_k)
                for i, r in enumerate(res)]
        recall = float(np.mean(hits))

    # ---- device-resident timing ("value"): one CUDA-event pair per call on the library's stream ----
    flat = [np.concatenate(b, 0) for b in batches]
    offs = np.arange(args.batch + 1, dtype=np.int64) * args.nq
    d_q = [torch.from_numpy(f).to(dev) for f in flat]
    d_ids = torch.empty((args.batch, args.top_k), dtype=torch.int64, device=dev)
    d_sc = torch.empty((args.batch, args.top_k), dtype=torch.float32, device=dev)
    d_cn = torch.empty((args.batch,), dtype=torch.int32, device=dev)
    if args.lanes > 0:
        gpu.set_lanes(args.lanes)
    gpu.set_profiling(True)
    sampler = ClockSampler(local if on_gpu else -1)       # spans warm-up + both timed regions (nvidia-smi needs ~0.2 s to start)
    for i in range(args.warmup):
        gpu.search_batch_device(d_q[i % n_batches].data_ptr(), offs, params, d_ids.data_ptr(), d_sc.data_ptr(),
                                d_cn.data_ptr())
    sync()
    if world > 1:
        dist.barrier()
    def timed_region():
        stage_ms, kern_ms, work = {}, {}, {}
        launches, dev_ms = 0, 0.0
        tw = time.perf_counter()
        for i in range(args.steps):
            gpu.search_batch_device(d_q[(args.warmup + i) % n_batches].data_ptr(), offs, params, d_ids.data_ptr(),
                                    d_sc.data_ptr(), d_cn.data_ptr())
            dev_ms += gpu.last_call_ms()
            ms, ln = gpu.last_stage_stats()
            for k, v in ms.items():
                stage_ms[k] = stage_ms.get(k, 0.0) + v
            for k, v in gpu.last_kernel_ms().items():
                kern_ms[k] = kern_ms.get(k, 0.0) + v
            launches += sum(ln.values())
            for k, v in gpu.last_work_counters().items():
                work[k] = work.get(k, 0) + v
        sync()
        return stage_ms, kern_ms, work, launches, dev_ms, 1e3 * (time.perf_counter() - tw)

    stage_ms, kern_ms, work, launches, dev_ms, wall_ms = timed_region()
    if args.dump_outputs and rank == 0:      # every rank holds the same merged results
        dump_outputs(args.dump_outputs, d_ids.cpu().numpy(), d_sc.cpu().numpy(), d_cn.cpu().numpy())
    # the same steps with the batch searched as one slice (pb_set_lanes(1)): kernels run alone, so these are the
    # per-kernel times that are not stretched by a co-running slice
    one_lane = None
    if world == 1 and args.lanes > 1 and args.batch >= 16:
        gpu.set_lanes(1)
        gpu.search_batch_device(d_q[0].data_ptr(), offs, params, d_ids.data_ptr(), d_sc.data_ptr(), d_cn.data_ptr())
        st1, km1, _, ln1, dm1, _ = timed_region()
        gpu.set_lanes(args.lanes)
        one_lane = {"value": args.batch * args.steps / (dm1 * 1e-3), "unit": "queries/s", "ms_per_step": dm1 / args.steps,
                    "gpu_launches": ln1, "stage_ms_per_step": {k: v / args.steps for k, v in st1.items()},
                    "kernel_ms_per_step": {k: v / args.steps for k, v in km1.items()}}
    if world > 1:
        dist.barrier()
    gpu.set_profiling(False)

    # ---- end-to-end through the public API: pinned host queries in, host results out ----
    pinned = [torch.from_numpy(f).pin_memory() if on_gpu else torch.from_numpy(f) for f in flat]
    L = npb.load_library()
    h_ids = np.zeros((args.batch, args.top_k), np.int64)
    h_sc = np.zeros((args.batch, args.top_k), np.float32)
    h_cn = np.zeros(args.batch, np.int32)
    pc = params._c()

    def e2e_step(i, bufs=None):
        ids, sc, cn = bufs or (h_ids, h_sc, h_cn)
        st = L.pb_search_batch(gpu._h, C.c_void_p(pinned[i % n_batches].data_ptr()), offs.ctypes.data_as(C.c_void_p),
                               args.batch, C.byref(pc), None, 0, ids.ctypes.data_as(C.c_void_p),
                               sc.ctypes.data_as(C.c_void_p), cn.ctypes.data_as(C.c_void_p))
        if st != 0:
            raise RuntimeError(L.pb_last_error().decode())
    for i in range(args.warmup):
        e2e_step(i)
    sync()
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(args.warmup + i)
    sync()
    e2e_s = time.perf_counter() - t1
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()

    # ---- the reference's deployment model: several host threads share one index (state.rs:24-47) ----
    concurrent = None
    if world == 1 and args.threads > 1:
        def worker(tid):
            bufs = (np.zeros_like(h_ids), np.zeros_like(h_sc), np.zeros_like(h_cn))
            for i in range(tid, args.steps, args.threads):
                e2e_step(args.warmup + i, bufs)
        for rep in range(2):          # first repetition creates the extra workspaces
            ths = [threading.Thread(target=worker, args=(t,)) for t in range(args.threads)]
            sync()
            tc0 = time.perf_counter()
            [t.start() for t in ths]
            [t.join() for t in ths]
            sync()
            tc = time.perf_counter() - tc0
        concurrent = {"host_threads": args.threads, "value": args.batch * args.steps / tc, "unit": "queries/s",
                      "ms_per_step": 1e3 * tc / args.steps,
                      "note": "same steps through pb_search_batch (host buffers) from T threads on one handle"}

    # ---- parity 1: the library against itself over EVERY timed query, certified tensor-core paths off ----
    fast = [gpu.search_batch(b, params) for b in batches]
    gpu.set_scores_tc(False)
    gpu.set_fast_exact(False)
    plain = [gpu.search_batch(b, params) for b in batches]
    gpu.set_scores_tc(True)
    gpu.set_fast_exact(True)
    si, sd = 0, 0.0
    for a, b in zip(fast, plain):
        i_, d_ = same_results(a, b)
        si += i_
        sd = max(sd, d_)
    self_parity = {"queries": n_batches * args.batch, "ids_identical": si, "max_abs_score_diff": sd,
                   "what": "default path (tcgen05 score table + tcgen05 MaxSim filter) vs both switched off "
                           "(fp32 FFMA2 centroid scores, every kept doc scored exactly), all timed batches"}

    # ---- parity 2 + CPU baseline: the CPU oracle on a bounded sample (rank 0) ----
    cpu = None
    parity = None
    if not args.no_cpu and args.parity_queries > 0:
        sample = queries[:args.parity_queries]
        gres = []
        for i0 in range(0, len(sample), args.batch):
            gres += gpu.search_batch(sample[i0:i0 + args.batch], params)      # collective when sharded
        if rank == 0:
            import psutil
            need, have = host_bytes_needed(args), psutil.virtual_memory().available
            if need > 0.8 * have:
                parity = {"skipped": f"host corpus needs {need >> 30} GiB, {have >> 30} GiB available"}
            else:
                from oracle import oracle
                shards, bases = host_corpus(oracle, args, G, dev, world)
                po = oracle.SearchParameters(top_k=args.top_k, n_ivf_probe=args.n_ivf_probe,
                                             n_full_scores=args.n_full_scores, centroid_score_threshold=args.threshold)
                oracle.search_sharded(shards, bases, sample[0], po)          # warm the page cache / thread pool
                c0 = time.perf_counter()
                cres = [oracle.search_sharded(shards, bases, q, po) for q in sample]
                c_s = time.perf_counter() - c0
                same_ids, max_ds = same_results(gres, cres)
                parity = {"queries": len(sample), "ids_identical": same_ids, "max_abs_score_diff": max_ds,
                          "against": "CPU oracle (C restatement of search.rs / codec.rs / maxsim.rs) on the whole corpus"}
                if world == 1:
                    cpu = {"value": len(sample) / c_s, "unit": "queries/s", "cores": oracle.lib().po_num_threads(),
                           "kind": "port", "sample": f"{len(sample)} queries of batch 0.., same index and parameters, "
                                                     f"{c_s:.1f} s of wall time (C restatement of the reference, OpenMP)"}
                del shards
        if world > 1:
            dist.barrier()

    # ---- roofline: algorithmic bytes (DESIGN.md section 4) / the kernel's own CUDA-event time ----
    peaks = measured_peaks()
    steps = max(args.steps, 1)
    nq_tot = work.get("n_query_tokens", 0)
    K = 1 << args.log2k
    packed = args.dim * args.nbits // 8
    qs_pad = (args.nq + 7) & ~7
    alg = {
        # hi/lo fp16 centroid tiles read once per launch, the 16-bit table written once
        "scores": steps * K * args.dim * 4 + nq_tot * K * 2,
        # one u32 code per (candidate, distinct code) + each 16-bit table entry once
        "approx16": work.get("n_candidate_tokens", 0) * 4 + nq_tot * K * 2,
        # packed residual + code per token: every kept doc in the tensor-core filter, the survivors again in fp32
        "filter": work.get("n_filter_tokens", 0) * (packed + 4),
        "exact": work.get("n_exact_tokens", 0) * (packed + 4),
    }
    pair_form = work.get("n_exact_pairs", 0) > 0
    names = {"scores": "k_scores16_tc", "approx16": "k_approx16", "filter": "k_maxsim_tc (pass 1: every kept doc)",
             "exact": "k_maxsim_tc (pass 2: survivors) + k_pair_exact" if pair_form else "k_exact"}
    per_kernel = {}
    for k, ms_tot in kern_ms.items():
        ms1 = ms_tot / steps
        gbs = alg[k] / steps / (ms1 * 1e-3) / 1e9 if ms1 > 0 else 0.0
        per_kernel[k] = {"kernel": names[k], "ms_per_launch": ms1, "algorithmic_bytes_per_launch": alg[k] / steps,
                         "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peaks["hbm"]}
    if "scores" in per_kernel and per_kernel["scores"]["ms_per_launch"] > 0:
        fl = 2.0 * nq_tot * K * args.dim / steps
        t = per_kernel["scores"]["ms_per_launch"] * 1e-3
        per_kernel["scores"].update({"algorithmic_tflops": fl / t / 1e12, "issued_tflops_3_split_products": 3 * fl / t / 1e12,
                                     "frac_of_bf16_peak_issued": 3 * fl / t / 1e12 / peaks["bf16"],
                                     "tensor_peak_tflops": peaks["bf16"]})
    if "approx16" in per_kernel and per_kernel["approx16"]["ms_per_launch"] > 0:
        # what actually bounds this kernel: one 2*QS-byte row of the L2-resident table per (candidate, distinct code)
        l2b = work.get("n_candidate_tokens", 0) * qs_pad * 2 / steps
        t = per_kernel["approx16"]["ms_per_launch"] * 1e-3
        sm = (clocks.get("sm_mhz") or 1965.0) * 1e6
        per_kernel["approx16"].update({"l2_gather_bytes_per_launch": l2b, "l2_gather_gbs": l2b / t / 1e9,
                                       "l2_cap_gbs": 6300 * sm / 1e9,
                                       "frac_of_l2_cap": l2b / t / (6300 * sm),
                                       "l2_cap_source": "B300_MICROARCH.md: LTS throughput cap ~6300 B/clk full chip"})
    dom = max(kern_ms, key=kern_ms.get) if kern_ms else None
    roof = None
    if dom:
        d = per_kernel[dom]
        cap = os.path.join(ROOT, "profiles", "r02_traffic.json")
        traffic_cap = None
        if os.path.exists(cap):
            try:
                tr = json.load(open(cap))
                hit = [k for k in tr if k.split("<")[0] == names[dom].split(" ")[0].split("<")[0]]
                traffic_cap = dict(tr[hit[0]], capture_kernel=hit[0]) if hit else None
            except Exception:
                traffic_cap = None
        roof = {"bound": "hbm", "kernel": d["kernel"], "achieved": d["achieved_gbs"], "peak": peaks["hbm"], "unit": "GB/s",
                "frac": d["frac_of_hbm_peak"], "traffic": None, "traffic_from_capture": traffic_cap,
                "peak_source": peaks["src"], "ms_per_launch": d["ms_per_launch"],
                "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"],
                "note": "traffic is not measured in this run (ncu only): traffic_from_capture cites the committed "
                        "ncu --set full capture when one exists for this kernel.  k_approx16 gathers rows of the "
                        "L2-resident 16-bit score table: its limiter is L2 throughput (see roofline_all.approx16), "
                        "the HBM fraction is the contract's number"}
    ms_f = kern_ms.get("filter", 0.0) / steps
    ms_e = kern_ms.get("exact", 0.0) / steps
    maxsim = None
    if ms_f + ms_e > 0:
        b_ = (alg["filter"] + alg["exact"]) / steps
        maxsim = {"kernels": "k_maxsim_tc pass 1 (tcgen05 estimate of every kept doc) + " +
                             ("pass 2 over the survivors (lists the (token, q) pairs inside the certified band) + "
                              "k_pair_exact (pinned-order fp32 similarity of those pairs)" if pair_form else
                              "k_exact (fused decompress + fp32 MaxSim of the survivors)"),
                  "ms_per_step": ms_f + ms_e, "algorithmic_bytes_per_step": b_,
                  "achieved_gbs": b_ / ((ms_f + ms_e) * 1e-3) / 1e9,
                  "frac_of_hbm_peak": b_ / ((ms_f + ms_e) * 1e-3) / 1e9 / peaks["hbm"],
                  "exact_stage_ms_per_step": stage_ms.get("exact", 0.0) / steps,
                  "exact_pairs_per_step": work.get("n_exact_pairs", 0) / steps,
                  "pair_fallback_queries_per_step": work.get("n_pair_fallback_queries", 0) / steps,
                  "fp32_tflops_k_exact": (2.0 * work.get("n_exact_tokens", 0) * args.nq * args.dim / steps / (ms_e * 1e-3) / 1e12)
                  if ms_e > 0 and not pair_form else None}

    if world > 1:
        tt = torch.tensor([dev_ms, e2e_s, wall_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s, wall_ms = float(tt[0]), float(tt[1]), float(tt[2])
    qps = args.batch * args.steps / (dev_ms * 1e-3)
    out = {
        "metric": "queries/sec", "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "wall_ms_per_step": wall_ms / args.steps,
        "higher_is_better": True, "scaling": "strong" if world > 1 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (codec-domain corpus, seed 42, 50k-doc chunks)",
        "config": workload_config(args, world),
        "recall_at_k": recall, "recall_queries": len(rq),
        "e2e": {"value": args.batch * args.steps / e2e_s, "unit": "queries/s",
                "h2d_bytes_per_step": int(flat[0].nbytes + offs.nbytes),
                "d2h_bytes_per_step": int(h_ids.nbytes + h_sc.nbytes + h_cn.nbytes), "ms_per_step": 1e3 * e2e_s / args.steps},
        "lanes": {"count": args.lanes if args.lanes > 1 and world == 1 and args.batch >= 16 else 1,
                  "what": "slices of a batch searched concurrently inside one call, each on its own stream "
                          "(pb_set_lanes); stage / kernel times of the timed region are sums over the slices",
                  "one_lane": one_lane},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "roofline_all": per_kernel, "maxsim": maxsim,
        "cpu_baseline": cpu, "parity": parity, "self_parity": self_parity, "concurrent": concurrent,
        "stage_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
        "kernel_ms_per_step": {k: v / args.steps for k, v in kern_ms.items()},
        "work_per_step": {k: v / args.steps for k, v in work.items()},
        "index_build_s": t_build, "corpus_generation_s": t_gen,
    }
    if rank == 0:
        print(json.dumps(out))
    gpu.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    """The reference's own CPU implementation of the path.  The reference is Rust and this image has no cargo/rustc, so
    oracle/_ref cannot exist; the timed code is the C restatement (oracle/), on all host threads, same corpus
    generator, same queries and parameters as the b200 arm, on a bounded sample per step.  Under torchrun rank 0 alone
    runs; the product library is not loaded."""
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    import torch
    from oracle import oracle
    if DEVICE_TYPE == "cuda":
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
        torch.cuda.set_device(dev)
    else:
        dev = torch.device("cpu")
    G = corpus_globals(args, dev)
    n_batches = min(max(args.steps + args.warmup, 4), 24)
    n_q = max(n_batches * args.batch, args.recall_queries, args.parity_queries)
    queries = make_queries(args, G, dev, n_q, seed=args.seed + 7)
    shards, bases = host_corpus(oracle, args, G, dev, world)
    po = oracle.SearchParameters(top_k=args.top_k, n_ivf_probe=args.n_ivf_probe, n_full_scores=args.n_full_scores,
                                 centroid_score_threshold=args.threshold)
    # bounded sample: CPU work per query grows with the corpus (about 0.3 s per query per million docs on 64 threads)
    per_step = max(1, min(args.batch, round(8e6 / args.docs_total)))
    step_q = lambda i: queries[(i % n_batches) * args.batch:][:per_step]   # noqa: E731
    for i in range(args.warmup):
        for q in step_q(i):
            oracle.search_sharded(shards, bases, q, po)
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = [oracle.search_sharded(shards, bases, q, po) for q in step_q(args.warmup + i)]
    s = time.perf_counter() - t0
    if args.dump_outputs:
        ids = np.full((len(last), args.top_k), -1, np.int64)
        sc = np.zeros((len(last), args.top_k), np.float32)
        for r, res in enumerate(last):
            ids[r, :len(res.passage_ids)], sc[r, :len(res.scores)] = res.passage_ids, res.scores
        dump_outputs(args.dump_outputs, ids, sc, [len(res.passage_ids) for res in last])
    qps = per_step * args.steps / s
    cores = oracle.lib().po_num_threads()
    sample = (f"{per_step} queries per step (the first of each {args.batch}-query batch of the b200 arm), {args.steps} steps; "
              f"ms_per_step is scaled to the full batch")
    print(json.dumps({
        "impl": "reference", "metric": "queries/sec", "value": qps, "unit": "queries/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * s / args.steps * args.batch / per_step,
        "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (codec-domain corpus, seed 42, 50k-doc chunks)",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


if __name__ == "__main__":
    # stdout carries exactly one JSON line: native libraries that print to fd 1 (NCCL's version banner) go to stderr
    _out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _out
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
