// engine.cu -- host side of libplaid_b200: the device-resident index (what MmapIndex holds after
// load, index.rs:995-1016), the search pipeline that replaces search::search_many_mmap
// (search.rs:643) and the C-ABI of include/plaid_b200.h.  No CPU fallback anywhere: every entry
// point needs an sm_100 device.
#include "engine_internal.h"
#include "kernels.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include <dlfcn.h>

// ------------------------------------------------------------------------------------------
// NCCL, bound at run time (dlopen) so single-GPU hosts need no libnccl.  Only the doc-sharded path
// (pb_index_comm_init) touches it.  Types restated from nccl.h 2.27 (stable ABI since 2.x).
// ------------------------------------------------------------------------------------------
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { PB_NCCL_UINT64 = 5, PB_NCCL_FLOAT32 = 7, PB_NCCL_SUM = 0 };
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load() {
        if (h) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) {
            h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) return false;
        GetUniqueId = (int (*)(ncclUniqueId *))dlsym(h, "ncclGetUniqueId");
        CommInitRank = (int (*)(ncclComm_t *, int, ncclUniqueId, int))dlsym(h, "ncclCommInitRank");
        CommDestroy = (int (*)(ncclComm_t))dlsym(h, "ncclCommDestroy");
        AllGather = (int (*)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllGather");
        AllReduce = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllReduce");
        GetErrorString = (const char *(*)(int))dlsym(h, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && CommDestroy && AllGather && AllReduce && GetErrorString;
    }
};
static NcclApi g_nccl;

// ------------------------------------------------------------------------------------------
// In-process shard group: the same two exchanges without NCCL, for ONE process that drives several shards
// from several host threads (any mix of devices, including all shards on one GPU -- which is how the merge
// kernels run under `pytest -m gpu` on a single-GPU box).  An all-gather is a host barrier, one
// cudaMemcpyPeerAsync per peer into the caller's receive buffer, and a second barrier so nobody reuses a
// send buffer that is still being read.
// ------------------------------------------------------------------------------------------
struct pb_shard_group {
    int world = 0;
    std::mutex mu;
    std::condition_variable cv;
    int arrived = 0;
    unsigned long long gen = 0;
    bool broken = false;
    int joined = 0;
    std::vector<const void *> send;
    std::vector<int> dev;
    // false = a peer failed or did not arrive within the timeout; the group stays broken
    bool barrier() {
        std::unique_lock<std::mutex> g(mu);
        if (broken) return false;
        const unsigned long long my = gen;
        if (++arrived == world) {
            arrived = 0;
            ++gen;
            cv.notify_all();
            return true;
        }
        if (!cv.wait_for(g, std::chrono::seconds(60), [&] { return gen != my || broken; })) broken = true;
        if (broken) cv.notify_all();
        return !broken;
    }
    void fail() {
        std::lock_guard<std::mutex> g(mu);
        broken = true;
        cv.notify_all();
    }
};

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;

pb_status pb_fail(pb_status s, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return s;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return pb_fail(PB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                           __FILE__, __LINE__);                                                    \
    } while (0)
#define CKN(call)                                                                                  \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != 0) return pb_fail(PB_ERR_COMM, "%s failed: %s", #call, g_nccl.GetErrorString(r_)); \
    } while (0)
#define CKS(expr)                                                                                  \
    do {                                                                                           \
        pb_status s_ = (expr);                                                                     \
        if (s_ != PB_OK) return s_;                                                                \
    } while (0)

// CUDA-event pair around the main kernel of a stage (profiling mode only); read after the sub-batch's synchronize
#define KEV_BEGIN(k)                                                                               \
    do {                                                                                           \
        if (ix->profiling) CK(cudaEventRecord(ws.kev[2 * (k)], ws.stream));                        \
    } while (0)
#define KEV_END(k)                                                                                 \
    do {                                                                                           \
        if (ix->profiling) {                                                                       \
            CK(cudaEventRecord(ws.kev[2 * (k) + 1], ws.stream));                                   \
            g_stats.kernel_seen[k] = true;                                                         \
        }                                                                                          \
    } while (0)

extern "C" const char *pb_last_error(void) { return g_err.c_str(); }
extern "C" const char *pb_version(void) { return "plaid_b200 0.1 (sm_100a)"; }

extern "C" int32_t pb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

static pb_status check_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return pb_fail(PB_ERR_CUDA, "no CUDA device available (%s); libplaid_b200 has no CPU fallback",
                       e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return pb_fail(PB_ERR_INVALID, "device %d out of range (have %d)", device, n);
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    if (p.major != 10)
        return pb_fail(PB_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, p.major,
                       p.minor);
    CK(cudaSetDevice(device));
    return PB_OK;
}

// ------------------------------------------------------------------------------------------
// device buffers
// ------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool zero_on_grow = false;
    bool owned = true;
    void adopt(void *ptr, size_t bytes) {  // caller-owned device memory, used in place
        if (p && owned) cudaFree(p);
        p = ptr;
        cap = bytes;
        owned = false;
    }
    pb_status ensure(size_t bytes) {
        if (bytes <= cap) return PB_OK;
        if (p && owned) cudaFree(p);
        owned = true;
        p = nullptr;
        cap = 0;
        size_t want = bytes + (bytes >> 3) + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return pb_fail(PB_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        }
        cap = want;
        if (zero_on_grow) {
            e = cudaMemset(p, 0, want);
            if (e != cudaSuccess) return pb_fail(PB_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
        }
        return PB_OK;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    ~DevBuf() {
        if (p && owned) cudaFree(p);
    }
};

struct HostBuf {  // pinned
    void *p = nullptr;
    size_t cap = 0;
    pb_status ensure(size_t bytes) {
        if (bytes <= cap) return PB_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes + 256);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return pb_fail(PB_ERR_NOMEM, "cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
        }
        cap = bytes + 256;
        return PB_OK;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    ~HostBuf() {
        if (p) cudaFreeHost(p);
    }
};

// per-call scratch; a pool of these makes pb_search_batch re-entrant on one handle
struct Workspace {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[PB_STAGE_COUNT + 1] = {};
    cudaEvent_t kev[2 * PB_KERNEL_COUNT] = {};  // begin / end around the main kernel of a stage
    cudaEvent_t call_ev[2] = {};                // around a whole search call
    DevBuf Q, qoff, ST, partial, sel, cells, ncells, bitmap, cand, ncand, approx, keys, kept, nkept, tokp, maxkey,
        exact, fkeys, oids, oscores, ocounts, subset, subset_bits, elig, misc, list, counters, lkeys, ST16, qrange, qflag, lsum, cand2, ncand2,  cellbits,
        gkeys, krank, payload, gfkeys, gpayload, cmax16, tau16, plist, pcount, Qi, Qh16t, Ql16t, ST16b, k1diag, k1rows, ulist, nulist, est, kept2, krank2, nkept2, tokp2, ktok2, qnmax, qexp, qrange_tc, mslot, slicecnt, rcmax, rcpairs, rcn, cellflags, estkey, srcrank, xpairs, xnpairs, needexact, gbase, redoflag;
    HostBuf hq, hres, hcounts, hredo;
    pb_status init() {
        CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        for (auto &e : ev) CK(cudaEventCreate(&e));
        for (auto &e : kev) CK(cudaEventCreate(&e));
        for (auto &e : call_ev) CK(cudaEventCreate(&e));
        bitmap.zero_on_grow = true;
        maxkey.zero_on_grow = true;
        subset_bits.zero_on_grow = true;
        elig.zero_on_grow = true;
        cellbits.zero_on_grow = true;
        rcmax.zero_on_grow = true;
        return PB_OK;
    }
    ~Workspace() {
        for (auto &e : ev)
            if (e) cudaEventDestroy(e);
        for (auto &e : kev)
            if (e) cudaEventDestroy(e);
        for (auto &e : call_ev)
            if (e) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
};

struct Stats {
    float ms[PB_STAGE_COUNT] = {};
    float kernel_ms[PB_KERNEL_COUNT] = {};
    bool kernel_seen[PB_KERNEL_COUNT] = {};
    float call_ms = 0.f;
    int launches[PB_STAGE_COUNT] = {};
    pb_work_counters work = {};
};
static thread_local Stats g_stats;

// One helper thread of a laned search call (search_impl): runs the pipeline of a slice of the batch on its own workspace
// and stream while the caller runs another slice, so that one slice's latency-bound kernels overlap the other's
// bandwidth-bound ones.
struct LaneWorker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, done = false, quit = false;
    LaneWorker() {
        th = std::thread([this] {
            std::unique_lock<std::mutex> lk(m);
            for (;;) {
                cv.wait(lk, [this] { return has_job || quit; });
                if (quit) return;
                lk.unlock();
                job();
                lk.lock();
                has_job = false;
                done = true;
                cv.notify_all();
            }
        });
    }
    void submit(std::function<void()> f) {
        std::lock_guard<std::mutex> lk(m);
        job = std::move(f);
        has_job = true;
        done = false;
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [this] { return done; });
    }
    ~LaneWorker() {
        {
            std::lock_guard<std::mutex> lk(m);
            quit = true;
            cv.notify_all();
        }
        if (th.joinable()) th.join();
    }
};

struct pb_index {
    int device = 0;
    int dim = 0, nbits = 0, packed = 0;
    long long K = 0, D = 0, N = 0, ivf_len = 0, doc_id_base = 0;
    int max_doclen = 0;
    int sm_count = 148;
    DevBuf centroids, w_rev, codes, residuals, doc_off, ivf, ivf_off, ucodes, udoc_off;
    long long n_ucodes = 0;
    bool build_ivf = false;    // no inverted file was given: built from the codes at finalize (index.rs:850-873)
    float cmax = 1.0f;         // largest centroid L2 norm (range of the 16-bit score table)
    bool fast_approx = true;   // two-pass approximate stage (exact cut either way)
    bool k1_tc = true;         // a2 on the tensor cores (k_scores16_tc) with its certified consumers: the default;
                               // PB_K1_TC=0 keeps every sub-batch on the exact fp32 kernel (the device-gated fallback)
    int k1_margin = 1;         // E: code units an estimate-built 16-bit code may differ from the exact one (PB_K1_TC_E widens it)
    int cent_exp = 0;          // centroids enter the tensor-core operands scaled by 2^cent_exp (max norm in [1, 2))
    bool k1_diag = false;      // also run the exact table and report the largest code difference (PB_K1_TC_DIAG=1)
    DevBuf cent_h16t, cent_l16t;  // its centroid operands: fp16 hi / lo, UMMA tile order
    int approx_grid = 8;       // k_approx16 CTAs per SM and query (PB_APPROX_GRID)
    int xtc_grid = 32;         // k_exact_tc CTAs per SM across the batch (PB_XTC_GRID)
    bool probe16 = true;       // a3 threshold-first selection on the 16-bit table (PB_PROBE16=0: per-lane lists only)
    bool fast_exact = true;    // tcgen05 certified filter in front of the exact stage (same results either way)
    float vmin = 0.0f;         // smallest pre-normalisation token norm |c + w| over the index (error bound of the filter)
    float wmax = 0.0f;         // largest residual norm |w| over the index (same)
    DevBuf centroids_f16;      // [K][dim] fp16 copy for the filter (k_exact_tc, the variant without a score table)
    DevBuf tok_inv_norm;       // [N] 1 / |c + w| for the linear estimate (k_maxsim_tc)
    bool filter_v1 = false;    // PB_FILTER_V1=1: always the decompressing filter k_exact_tc (A/B measurement)
    bool pair_exact = true;    // exact stage on the (token, query token) pairs that can hold a maximum (PB_PAIR_EXACT=0: k_exact)
    int ws_grid = 8;           // k_maxsim_tc CTAs per SM across the batch (PB_WS_GRID)
    int ws_grid2 = 8;          // the same for its pass 2 over the filter's survivors (PB_WS_GRID2; 1: 0.54, 2: 0.43, 4 and 8: 0.40 ms)
    int lanes = 1;             // slices of a batch searched concurrently, each on its own stream (pb_set_lanes / PB_LANES; 1 = off)
    std::mutex lane_mu;        // one laned call at a time per handle (a second concurrent caller runs un-laned)
    std::vector<std::unique_ptr<LaneWorker>> lane_workers;
    bool profiling = false;
    size_t st_budget = (size_t)8 << 30;  // workspace budget of one search call (PB_WS_BUDGET_MB)
    ncclComm_t comm = nullptr;  // doc-sharded deployment: one rank per GPU
    pb_shard_group *group = nullptr;  // or one host thread per shard inside this process (pb_index_group_join)
    int rank = 0, world = 1;
    std::mutex mu;
    std::vector<std::unique_ptr<Workspace>> pool;
};

// A workspace of the handle's pool, held for one call.  It goes back to the pool only if the call set `done`: the
// kernels restore its scratch invariants (cleared bitmaps, zeroed maxima) as they go, so after a call that failed half
// way its state is unknown, and it is freed instead once its stream is idle.
struct WorkspaceLease {
    pb_index *ix;
    std::unique_ptr<Workspace> ws;
    bool done = false;
    pb_status acquire() {
        {
            std::lock_guard<std::mutex> g(ix->mu);
            if (!ix->pool.empty()) {
                ws = std::move(ix->pool.back());
                ix->pool.pop_back();
                return PB_OK;
            }
        }
        std::unique_ptr<Workspace> fresh(new Workspace());
        CKS(fresh->init());
        ws = std::move(fresh);
        return PB_OK;
    }
    ~WorkspaceLease() {
        if (!ws) return;
        if (done) {
            std::lock_guard<std::mutex> g(ix->mu);
            ix->pool.push_back(std::move(ws));
        } else {
            cudaStreamSynchronize(ws->stream);
        }
    }
};

// ------------------------------------------------------------------------------------------
// DIM dispatch
// ------------------------------------------------------------------------------------------
#define PB_DIM_SWITCH(dim, ...)                                                                    \
    switch (dim) {                                                                                 \
        case 32: { constexpr int DIM = 32; __VA_ARGS__; } break;                                   \
        case 64: { constexpr int DIM = 64; __VA_ARGS__; } break;                                   \
        case 96: { constexpr int DIM = 96; __VA_ARGS__; } break;                                   \
        case 128: { constexpr int DIM = 128; __VA_ARGS__; } break;                                 \
        case 256: { constexpr int DIM = 256; __VA_ARGS__; } break;                                 \
        default: return pb_fail(PB_ERR_UNSUPPORTED, "embedding_dim %d not built (32/64/96/128/256)", dim); \
    }
// the dims of the tensor-core kernels
#define PB_TC_DIM_SWITCH(dim, ...)                                                                 \
    switch (dim) {                                                                                 \
        case 64: { constexpr int DIM = 64; __VA_ARGS__; } break;                                   \
        case 96: { constexpr int DIM = 96; __VA_ARGS__; } break;                                   \
        case 128: { constexpr int DIM = 128; __VA_ARGS__; } break;                                 \
        default: return pb_fail(PB_ERR_UNSUPPORTED, "tensor-core kernels: embedding_dim %d not built (64/96/128)", dim); \
    }
// bits per residual dimension (a divisor of 8, checked at open)
#define PB_NBITS_SWITCH(nbits, ...)                                                                \
    switch (nbits) {                                                                               \
        case 1: { constexpr int NBITS = 1; __VA_ARGS__; } break;                                   \
        case 2: { constexpr int NBITS = 2; __VA_ARGS__; } break;                                   \
        case 4: { constexpr int NBITS = 4; __VA_ARGS__; } break;                                   \
        default: { constexpr int NBITS = 8; __VA_ARGS__; } break;                                  \
    }

// QS: query tokens per score-table row.  Up to 32 tokens: rounded up to 8 (rows of at most 64 bytes); beyond: to a
// multiple of 64, so that a row is whole 128-byte lines (a 96-byte row straddles lines and costs the first approximate
// pass 2.5x instead of 1.5-2x: profiles/r02_summary.md)
static int query_row_tokens(int nq_max) {
    return nq_max <= 32 ? std::max(8, (nq_max + 7) & ~7) : ((nq_max + 63) & ~63);
}

static bool dim_supported(int d) { return d == 32 || d == 64 || d == 96 || d == 128 || d == 256; }

static size_t smem_scores(int dim) { return (size_t)(PB_TOK_TILE + 2 * PB_Q_TILE) * (dim + 4) * sizeof(float); }
static size_t smem_exact(int dim, int packed) {
    return (size_t)(PB_TOK_TILE + PB_Q_TILE) * (dim + 4) * sizeof(float) + PB_Q_TILE * 129 * sizeof(float) +
           PB_TOK_TILE * sizeof(int) + 256 * sizeof(float) + (size_t)PB_TOK_TILE * packed;
}

template <class Kern> static pb_status set_smem(Kern k, size_t bytes) {
    // a kernel's static shared memory counts towards the 48 KB a launch may use without opting in
    if (bytes > 40 * 1024) CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return PB_OK;
}

// ------------------------------------------------------------------------------------------
// index open / close
// ------------------------------------------------------------------------------------------
static unsigned bitrev_n(unsigned v, int nbits) {
    unsigned r = 0;
    for (int k = 0; k < nbits; ++k)
        if (v & (1u << k)) r |= 1u << (nbits - 1 - k);
    return r;
}

template <class T>
static pb_status fetch_host(std::vector<T> &dst, const T *src, size_t n, int space) {
    dst.resize(n);
    if (n == 0) return PB_OK;
    if (space == PB_MEM_DEVICE) CK(cudaMemcpy(dst.data(), src, n * sizeof(T), cudaMemcpyDeviceToHost));
    else memcpy(dst.data(), src, n * sizeof(T));
    return PB_OK;
}

static pb_status upload(DevBuf &dst, const void *src, size_t bytes, int space) {
    CKS(dst.ensure(std::max<size_t>(bytes, 16)));
    if (bytes == 0) return PB_OK;
    CK(cudaMemcpy(dst.p, src, bytes, space == PB_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    return PB_OK;
}

// i64 -> u32 with a range check, streamed through a bounded staging buffer, into dst[dst_off..]
static pb_status upload_narrow(DevBuf &dst, long long dst_off, const int64_t *src, long long n, long long limit,
                               int space, const char *what) {
    if (n == 0) return PB_OK;
    DevBuf bad;
    CKS(bad.ensure(16));
    CK(cudaMemset(bad.p, 0, 4));
    const long long chunk = 1ll << 26;  // 64M elements = 512 MiB of i64
    DevBuf stage;
    if (space == PB_MEM_HOST) CKS(stage.ensure((size_t)std::min(n, chunk) * 8));
    for (long long o = 0; o < n; o += chunk) {
        long long m = std::min(chunk, n - o);
        const long long *in = reinterpret_cast<const long long *>(src) + o;
        if (space == PB_MEM_HOST) {
            CK(cudaMemcpy(stage.p, in, (size_t)m * 8, cudaMemcpyHostToDevice));
            in = stage.as<long long>();
        }
        k_narrow_i64_u32<<<1184, 256>>>(in, dst.as<uint32_t>() + dst_off + o, m, limit, bad.as<int>());
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
    }
    int hbad = 0;
    CK(cudaMemcpy(&hbad, bad.p, 4, cudaMemcpyDeviceToHost));
    if (hbad) return pb_fail(PB_ERR_INVALID, "%s contains a value outside [0, %lld)", what, limit);
    return PB_OK;
}

// codes + packed residuals of tokens [tok_off, tok_off+n) (one chunk file pair, or everything)
pb_status pb_index_upload_tokens(pb_index *ix, long long tok_off, const int64_t *codes, const uint8_t *residuals,
                                 long long n, int space) {
    if (n == 0) return PB_OK;
    if (tok_off < 0 || tok_off + n > ix->N) return pb_fail(PB_ERR_INVALID, "token range [%lld,+%lld) outside the index", tok_off, n);
    CK(cudaSetDevice(ix->device));
    if (!ix->residuals.owned) {  // PB_OPEN_ADOPT_RESIDUALS: the caller's array is the index
        if (tok_off != 0 || n != ix->N || residuals != ix->residuals.as<uint8_t>())
            return pb_fail(PB_ERR_INVALID, "adopted residuals cover the whole index");
    } else
        CK(cudaMemcpy(ix->residuals.as<uint8_t>() + (size_t)tok_off * ix->packed, residuals, (size_t)n * ix->packed,
                      space == PB_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    return upload_narrow(ix->codes, tok_off, codes, n, ix->K, space, "codes");
}

// Everything except the per-token arrays (d->codes / d->residuals may be NULL here).
pb_status pb_index_open_begin(const pb_index_desc *d, pb_index **out) {
    if (!d || !out) return pb_fail(PB_ERR_INVALID, "null argument");
    *out = nullptr;
    if (d->nbits <= 0 || 8 % d->nbits != 0)  // codec.rs:161-166
        return pb_fail(PB_ERR_INVALID, "nbits must be a divisor of 8, got %d", d->nbits);
    if (d->dim <= 0 || d->dim % 4 != 0) return pb_fail(PB_ERR_INVALID, "embedding_dim %d must be a positive multiple of 4", d->dim);
    if (!dim_supported(d->dim)) return pb_fail(PB_ERR_UNSUPPORTED, "embedding_dim %d not built (32/64/96/128/256)", d->dim);
    if (d->num_centroids <= 0 || d->num_documents < 0 || d->num_embeddings < 0)
        return pb_fail(PB_ERR_INVALID, "bad shapes K=%lld D=%lld N=%lld", (long long)d->num_centroids,
                       (long long)d->num_documents, (long long)d->num_embeddings);
    if (d->num_centroids >= (1ll << 32) - 1 || d->num_documents >= (1ll << 32) - 1)
        return pb_fail(PB_ERR_UNSUPPORTED, "K and D must be below 2^32-1 per shard");
    if (d->doc_id_base < 0 || d->doc_id_base + d->num_documents >= (1ll << 32) - 1)
        return pb_fail(PB_ERR_UNSUPPORTED, "global doc ids must stay below 2^32-1");
    if (!d->centroids || !d->bucket_weights || (!d->doc_lengths && d->num_documents) || (!d->ivf_lengths && d->ivf))
        return pb_fail(PB_ERR_INVALID, "null index array");
    if ((d->flags & PB_OPEN_ADOPT_RESIDUALS) && (d->memory_space != PB_MEM_DEVICE || !d->residuals))
        return pb_fail(PB_ERR_INVALID, "PB_OPEN_ADOPT_RESIDUALS needs device-resident residuals");
    CKS(check_device(d->device));
    std::unique_ptr<pb_index> ix(new pb_index());
    ix->device = d->device;
    ix->dim = d->dim;
    ix->nbits = d->nbits;
    ix->packed = d->dim * d->nbits / 8;
    ix->K = d->num_centroids;
    ix->D = d->num_documents;
    ix->N = d->num_embeddings;
    ix->doc_id_base = d->doc_id_base;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, d->device));
    ix->sm_count = prop.multiProcessorCount;
    for (const char *name : {"PB_ST_BUDGET_MB", "PB_WS_BUDGET_MB"})
        if (const char *e = getenv(name)) {
            long v = atol(e);
            if (v > 0) ix->st_budget = (size_t)v << 20;
        }
    const int sp = d->memory_space;
    // doc offsets (index.rs:1107-1110)
    std::vector<int64_t> dl;
    CKS(fetch_host(dl, d->doc_lengths, (size_t)ix->D, sp));
    std::vector<long long> doff((size_t)ix->D + 1, 0);
    int maxlen = 0;
    for (long long i = 0; i < ix->D; ++i) {
        if (dl[i] < 0 || dl[i] > (1 << 30)) return pb_fail(PB_ERR_INVALID, "doc_lengths[%lld] = %lld", i, (long long)dl[i]);
        doff[i + 1] = doff[i] + dl[i];
        maxlen = std::max<int>(maxlen, (int)dl[i]);
    }
    if (doff[ix->D] != ix->N)
        return pb_fail(PB_ERR_INVALID, "sum(doc_lengths)=%lld != num_embeddings=%lld", doff[ix->D], ix->N);
    ix->max_doclen = maxlen;
    CKS(upload(ix->doc_off, doff.data(), doff.size() * 8, PB_MEM_HOST));
    // ivf offsets (index.rs:1089-1094); without an inverted file it is built from the codes in pb_index_finalize
    ix->build_ivf = d->ivf_lengths == nullptr;
    if (!ix->build_ivf) {
        std::vector<int32_t> il;
        CKS(fetch_host(il, d->ivf_lengths, (size_t)ix->K, sp));
        std::vector<long long> ioff((size_t)ix->K + 1, 0);
        for (long long i = 0; i < ix->K; ++i) {
            if (il[i] < 0) return pb_fail(PB_ERR_INVALID, "ivf_lengths[%lld] < 0", i);
            ioff[i + 1] = ioff[i] + il[i];
        }
        ix->ivf_len = ioff[ix->K];
        if (ix->ivf_len && !d->ivf) return pb_fail(PB_ERR_INVALID, "null ivf");
        CKS(upload(ix->ivf_off, ioff.data(), ioff.size() * 8, PB_MEM_HOST));
    }
    // bucket weights with the packer's bit reversal folded in (codec.rs:168-214, :389-395)
    std::vector<float> w;
    CKS(fetch_host(w, d->bucket_weights, (size_t)1 << ix->nbits, sp));
    std::vector<float> wrev(256, 0.f);
    for (unsigned f = 0; f < (1u << ix->nbits); ++f) wrev[f] = w[bitrev_n(f, ix->nbits)];
    CKS(upload(ix->w_rev, wrev.data(), 256 * sizeof(float), PB_MEM_HOST));
    CKS(upload(ix->centroids, d->centroids, (size_t)ix->K * ix->dim * sizeof(float), sp));
    if (d->flags & PB_OPEN_ADOPT_RESIDUALS)
        ix->residuals.adopt(const_cast<uint8_t *>(d->residuals), (size_t)ix->N * ix->packed);
    else CKS(ix->residuals.ensure(std::max<size_t>((size_t)ix->N * ix->packed, 16)));
    CKS(ix->codes.ensure(std::max<size_t>((size_t)ix->N * 4, 16)));
    if (!ix->build_ivf) {
        CKS(ix->ivf.ensure(std::max<size_t>((size_t)ix->ivf_len * 4, 16)));
        CKS(upload_narrow(ix->ivf, 0, d->ivf, ix->ivf_len, std::max<long long>(ix->D, 1), sp, "ivf"));
    }
    *out = ix.release();
    return PB_OK;
}

// The inverted file of an index opened without one (index.rs:850-873), from the per-doc distinct code lists.
static pb_status build_ivf_on_device(pb_index *ix) {
    CKS(ix->ivf_off.ensure((size_t)(ix->K + 1) * 8));
    const long long cap = std::max<long long>(ix->n_ucodes, 1);
    DevBuf ka, kb, cnt, tmp;
    CKS(ka.ensure((size_t)cap * 8));
    CKS(kb.ensure((size_t)cap * 8));
    CKS(cnt.ensure(16));
    CK(cudaMemset(cnt.p, 0, 16));
    if (ix->D > 0) {
        k_ivf_pairs<<<ix->sm_count * 8, 256>>>(ix->ucodes.as<uint32_t>(), ix->udoc_off.as<long long>(), ix->D, ka.as<u64>(),
                                               cnt.as<unsigned long long>());
        CK(cudaGetLastError());
    }
    unsigned long long m = 0;
    CK(cudaMemcpy(&m, cnt.p, 8, cudaMemcpyDeviceToHost));
    if (m > (1ull << 31) - 2) return pb_fail(PB_ERR_UNSUPPORTED, "more than 2^31 (centroid, doc) pairs per shard");
    int kbits = 1;
    while ((1ll << kbits) < ix->K) ++kbits;
    size_t tb = 0;
    CK(cub::DeviceRadixSort::SortKeys(nullptr, tb, ka.as<u64>(), kb.as<u64>(), (int)m, 0, 32 + kbits));
    size_t tb2 = 0;
    CK(cub::DeviceSelect::Unique(nullptr, tb2, kb.as<u64>(), ka.as<u64>(), cnt.as<int>() + 2, (int)m));
    CKS(tmp.ensure(std::max(tb, tb2) + 16));
    CK(cub::DeviceRadixSort::SortKeys(tmp.p, tb, ka.as<u64>(), kb.as<u64>(), (int)m, 0, 32 + kbits));
    CK(cub::DeviceSelect::Unique(tmp.p, tb2, kb.as<u64>(), ka.as<u64>(), cnt.as<int>() + 2, (int)m));
    int m2 = 0;
    CK(cudaMemcpy(&m2, cnt.as<int>() + 2, 4, cudaMemcpyDeviceToHost));
    ix->ivf_len = m2;
    CKS(ix->ivf.ensure(std::max<size_t>((size_t)m2 * 4, 16)));
    k_ivf_from_keys<<<ix->sm_count * 8, 256>>>(ka.as<u64>(), m2, ix->ivf.as<uint32_t>());
    k_ivf_offsets<<<(unsigned)((ix->K + 256) / 256), 256>>>(ka.as<u64>(), m2, ix->K, ix->ivf_off.as<long long>());
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return PB_OK;
}

// Derived arrays that need every token: the per-doc distinct-code lists k_approx walks.
pb_status pb_index_finalize(pb_index *ix) {
    CK(cudaSetDevice(ix->device));
    if ((unsigned long long)ix->K * 1024ull * 4ull >= (1ull << 40)) return pb_fail(PB_ERR_UNSUPPORTED, "K too large");
    std::vector<long long> uoff((size_t)ix->D + 1, 0);
    if (ix->D > 0) {
        DevBuf counts;
        CKS(counts.ensure((size_t)ix->D * 4));
        const int blocks = (int)std::min<long long>(ix->D, (long long)ix->sm_count * 16);
        k_unique_codes<<<blocks, 128>>>(ix->codes.as<uint32_t>(), ix->doc_off.as<long long>(), ix->D, nullptr, nullptr,
                                        counts.as<int>());
        CK(cudaGetLastError());
        std::vector<int> hc((size_t)ix->D);
        CK(cudaMemcpy(hc.data(), counts.p, hc.size() * 4, cudaMemcpyDeviceToHost));
        for (long long i = 0; i < ix->D; ++i) uoff[i + 1] = uoff[i] + hc[i];
    }
    {
        DevBuf mx;
        CKS(mx.ensure(16));
        CK(cudaMemset(mx.p, 0, 4));
        k_max_row_norm<<<ix->sm_count * 4, 256>>>(ix->centroids.as<float>(), ix->K, ix->dim, mx.as<float>());
        CK(cudaGetLastError());
        float m2 = 0.f;
        CK(cudaMemcpy(&m2, mx.p, 4, cudaMemcpyDeviceToHost));
        ix->cmax = sqrtf(m2);
        if (const char *e = getenv("PB_FAST_APPROX")) ix->fast_approx = atoi(e) != 0;
        if (const char *e = getenv("PB_FAST_EXACT")) ix->fast_exact = atoi(e) != 0;
        if (const char *e = getenv("PB_FILTER_V1")) ix->filter_v1 = atoi(e) != 0;
        if (const char *e = getenv("PB_PAIR_EXACT")) ix->pair_exact = atoi(e) != 0;
        if (const char *e = getenv("PB_WS_GRID")) ix->ws_grid = std::max(1, atoi(e));
        if (const char *e = getenv("PB_WS_GRID2")) ix->ws_grid2 = std::max(1, atoi(e));
        if (const char *e = getenv("PB_LANES")) ix->lanes = std::min(8, std::max(1, atoi(e)));
        if (const char *e = getenv("PB_PROBE16")) ix->probe16 = atoi(e) != 0;
        if (const char *e = getenv("PB_K1_TC_DIAG")) ix->k1_diag = atoi(e) != 0;
        if (const char *e = getenv("PB_K1_TC")) ix->k1_tc = atoi(e) != 0;
        if (const char *e = getenv("PB_K1_TC_E")) ix->k1_margin = std::max(1, atoi(e));
        if (const char *e = getenv("PB_APPROX_GRID")) ix->approx_grid = std::max(1, atoi(e));
        if (const char *e = getenv("PB_XTC_GRID")) ix->xtc_grid = std::max(1, atoi(e));
    }
    if ((ix->dim == 64 || ix->dim == 96 || ix->dim == 128) && ix->N > 0 && ix->K > 0) {
        // operands of the tensor-core filter (k_exact_tc): fp16 centroids and the smallest token norm
        CKS(ix->centroids_f16.ensure((size_t)ix->K * ix->dim * 2));
        k_rows_to_f16_plain<<<ix->sm_count * 8, 256>>>(ix->centroids.as<float>(), ix->K * (long long)ix->dim,
                                                      ix->centroids_f16.as<__half>());
        CK(cudaGetLastError());
        DevBuf mn;
        CKS(mn.ensure(16));
        CKS(ix->tok_inv_norm.ensure((size_t)ix->N * 4));  // 1 / |c + w| per token: operand of the linear estimate (k_maxsim_tc)
        const float init[2] = {3.0e38f, 0.0f};
        CK(cudaMemcpy(mn.p, init, 8, cudaMemcpyHostToDevice));
        PB_TC_DIM_SWITCH(ix->dim, {
            k_min_vnorm<DIM><<<ix->sm_count * 8, 256>>>(ix->centroids.as<float>(), ix->w_rev.as<float>(), ix->nbits,
                                                        ix->codes.as<uint32_t>(), ix->residuals.as<uint8_t>(), ix->N,
                                                        mn.as<float>(), ix->tok_inv_norm.as<float>());
        });
        CK(cudaGetLastError());
        if ((ix->k1_diag || ix->k1_tc) && ix->cmax > 0.0f && ix->cmax < 3.0e38f) {
            // operands of the tensor-core score table: centroids * 2^cent_exp (max norm in [1, 2)), fp16 hi / lo parts
            ix->cent_exp = -ilogbf(ix->cmax);
            const size_t elems = (size_t)((ix->K + 127) / 128) * 128 * ix->dim;
            CKS(ix->cent_h16t.ensure(elems * 2));
            CKS(ix->cent_l16t.ensure(elems * 2));
            CK(cudaMemset(ix->cent_h16t.p, 0, elems * 2));
            CK(cudaMemset(ix->cent_l16t.p, 0, elems * 2));
            k_rows_to_f16_split_tiles<<<ix->sm_count * 8, 256>>>(ix->centroids.as<float>(), ix->K, ix->dim, ix->cent_exp,
                                                                ix->cent_h16t.as<__half>(), ix->cent_l16t.as<__half>());
            CK(cudaGetLastError());
        }
        float got[2] = {0.f, 0.f};
        CK(cudaMemcpy(got, mn.p, 8, cudaMemcpyDeviceToHost));
        ix->vmin = got[0] < 1e30f ? got[0] : 0.0f;
        ix->wmax = got[1];
    }
    ix->n_ucodes = uoff[ix->D];
    CKS(upload(ix->udoc_off, uoff.data(), uoff.size() * 8, PB_MEM_HOST));
    CKS(ix->ucodes.ensure(std::max<size_t>((size_t)ix->n_ucodes * 4, 16)));
    if (ix->D > 0) {
        const int blocks = (int)std::min<long long>(ix->D, (long long)ix->sm_count * 16);
        k_unique_codes<<<blocks, 128>>>(ix->codes.as<uint32_t>(), ix->doc_off.as<long long>(), ix->D,
                                        ix->udoc_off.as<long long>(), ix->ucodes.as<uint32_t>(), nullptr);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
    }
    if (ix->build_ivf) CKS(build_ivf_on_device(ix));
    return PB_OK;
}

extern "C" pb_status pb_index_export_ivf(pb_index *ix, int64_t *out_ivf, int32_t *out_lengths, int64_t *out_total) {
    if (!ix) return pb_fail(PB_ERR_INVALID, "null argument");
    CK(cudaSetDevice(ix->device));
    if (out_total) *out_total = ix->ivf_len;
    if (!out_ivf && !out_lengths) return PB_OK;
    DevBuf di, dl;
    if (out_ivf) CKS(di.ensure(std::max<size_t>((size_t)ix->ivf_len * 8, 16)));
    if (out_lengths) CKS(dl.ensure(std::max<size_t>((size_t)ix->K * 4, 16)));
    k_ivf_export<<<ix->sm_count * 8, 256>>>(ix->ivf.as<uint32_t>(), ix->ivf_off.as<long long>(), ix->ivf_len, ix->K,
                                           ix->doc_id_base, out_ivf ? di.as<long long>() : nullptr,
                                           out_lengths ? dl.as<int>() : nullptr);
    CK(cudaGetLastError());
    if (out_ivf && ix->ivf_len) CK(cudaMemcpy(out_ivf, di.p, (size_t)ix->ivf_len * 8, cudaMemcpyDeviceToHost));
    if (out_lengths) CK(cudaMemcpy(out_lengths, dl.p, (size_t)ix->K * 4, cudaMemcpyDeviceToHost));
    return PB_OK;
}

extern "C" pb_status pb_index_open(const pb_index_desc *d, pb_index **out) {
    if (!d || !out) return pb_fail(PB_ERR_INVALID, "null argument");
    if (d->num_embeddings > 0 && (!d->codes || !d->residuals)) return pb_fail(PB_ERR_INVALID, "null index array");
    pb_index *ix = nullptr;
    CKS(pb_index_open_begin(d, &ix));
    pb_status s = pb_index_upload_tokens(ix, 0, d->codes, d->residuals, d->num_embeddings, d->memory_space);
    if (s == PB_OK) s = pb_index_finalize(ix);
    if (s != PB_OK) {
        pb_index_close(ix);
        return s;
    }
    *out = ix;
    return PB_OK;
}

extern "C" void pb_index_close(pb_index *ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    ix->lane_workers.clear();  // joins the helper threads
    cudaDeviceSynchronize();
    if (ix->comm) g_nccl.CommDestroy(ix->comm);
    delete ix;
}

extern "C" int64_t pb_index_num_documents(const pb_index *ix) { return ix ? ix->D : 0; }
extern "C" int64_t pb_index_num_embeddings(const pb_index *ix) { return ix ? ix->N : 0; }
extern "C" int64_t pb_index_num_partitions(const pb_index *ix) { return ix ? ix->K : 0; }
extern "C" double pb_index_avg_doclen(const pb_index *ix) { return (ix && ix->D) ? (double)ix->N / (double)ix->D : 0.0; }
extern "C" int32_t pb_index_embedding_dim(const pb_index *ix) { return ix ? ix->dim : 0; }
extern "C" int32_t pb_index_nbits(const pb_index *ix) { return ix ? ix->nbits : 0; }
extern "C" int32_t pb_index_device(const pb_index *ix) { return ix ? ix->device : -1; }

extern "C" void pb_search_params_default(pb_search_params *p) {  // search.rs:58-69
    if (!p) return;
    p->batch_size = 2000;
    p->n_full_scores = 4096;
    p->top_k = 10;
    p->n_ivf_probe = 8;
    p->centroid_batch_size = 100000;
    p->has_centroid_score_threshold = 1;
    p->centroid_score_threshold = 0.4f;
}

extern "C" void pb_set_fast_approx(pb_index *ix, int32_t enabled) {
    if (!ix) return;
    ix->fast_approx = enabled != 0;  // 0 = single exact pass over every candidate, otherwise two-pass
}
extern "C" void pb_set_scores_tc(pb_index *ix, int32_t enabled) {
    if (ix) ix->k1_tc = enabled != 0;  // effective when the tensor-core operands were built at open (k1_tc_usable)
}
extern "C" void pb_set_lanes(pb_index *ix, int32_t lanes) {
    if (ix) ix->lanes = std::min(8, std::max(1, (int)lanes));
}
extern "C" void pb_set_fast_exact(pb_index *ix, int32_t enabled) {
    if (ix) ix->fast_exact = enabled != 0;
}
extern "C" void pb_set_profiling(pb_index *ix, int32_t enabled) {
    if (ix) ix->profiling = enabled != 0;
}
extern "C" pb_status pb_last_stage_stats(pb_index *, float *out_ms, int32_t *out_launches) {
    for (int i = 0; i < PB_STAGE_COUNT; ++i) {
        if (out_ms) out_ms[i] = g_stats.ms[i];
        if (out_launches) out_launches[i] = g_stats.launches[i];
    }
    return PB_OK;
}
extern "C" pb_status pb_last_call_ms(pb_index *, float *out_ms) {
    if (!out_ms) return pb_fail(PB_ERR_INVALID, "null argument");
    *out_ms = g_stats.call_ms;
    return PB_OK;
}
extern "C" pb_status pb_last_kernel_ms(pb_index *, float *out_ms) {
    if (!out_ms) return pb_fail(PB_ERR_INVALID, "null argument");
    for (int i = 0; i < PB_KERNEL_COUNT; ++i) out_ms[i] = g_stats.kernel_ms[i];
    return PB_OK;
}
extern "C" pb_status pb_last_work_counters(pb_index *, pb_work_counters *out) {
    if (!out) return pb_fail(PB_ERR_INVALID, "null argument");
    *out = g_stats.work;
    return PB_OK;
}

// ------------------------------------------------------------------------------------------
// kernel launch helpers shared by the search pipeline and the stage entry points
// ------------------------------------------------------------------------------------------
static int pow2_ceil(int n) {
    int P = 1;
    while (P < n) P <<= 1;
    return P;
}

// a2 on the tensor cores (k_scores_tc.cuh).  err = certified bound of |exact - estimate| in 16-bit code units
// (derivation at the top of that file); E = ceil(err) is the largest difference between an estimate-built code and
// the exact-table code, 2E + 1 the code margin of its consumers.
static float k1_err_codes(int dim) {
    const float chain = (float)dim * 5.9604645e-8f;                 // dim * 2^-24: the pinned fp32 FMA chain
    const float tc = (3.0f * (float)(dim / 16) + 3.0f) * 2.3841858e-7f;  // 2^-22 per MMA accumulation + the dropped split terms
    const float sub = 2.0f * 2.9802322e-8f * sqrtf((float)dim);     // fp16 subnormal spacing of the lo parts
    return (chain + tc + sub) * 32768.0f * 1.0001f;
}
static bool k1_tc_usable(const pb_index *ix) {
    return ix->k1_tc && ix->cent_h16t.p && (ix->dim == 64 || ix->dim == 96 || ix->dim == 128) && k1_err_codes(ix->dim) < 1.0f;
}

// the 16-bit score table from the split-fp16 UMMA GEMM (k_scores16_tc) into `table`; `flags` gets the per-query
// out-of-range bits the exact kernel would set in qflag
static pb_status launch_k1_table(pb_index *ix, Workspace &ws, int B, int QS, unsigned short *table, int *flags) {
    const int n_groups = (int)(((long long)B * QS + 127) / 128);
    const size_t qelems = (size_t)n_groups * 128 * ix->dim;
    CKS(ws.Qh16t.ensure(qelems * 2));
    CKS(ws.Ql16t.ensure(qelems * 2));
    CKS(ws.qrange_tc.ensure((size_t)B * 8 + 16));
    k_query_split_tiles<<<ix->sm_count, 256, 0, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), ws.qexp.as<int>(), B, QS,
                                                             ix->dim, ws.Qh16t.as<__half>(), ws.Ql16t.as<__half>());
    k_query_range_tc<<<(B + 127) / 128, 128, 0, ws.stream>>>(ws.qrange.as<float2>(), ws.qexp.as<int>(), ix->cent_exp, B,
                                                            ws.qrange_tc.as<float2>());
    const int tiles = (int)((ix->K + 127) / 128);
    const size_t sm = (size_t)6 * 128 * ix->dim * 2 + 128;
    PB_TC_DIM_SWITCH(ix->dim, {
        auto kern = k_scores16_tc<DIM>;
        CKS(set_smem(kern, sm));
        KEV_BEGIN(PB_KERNEL_SCORES);
        kern<<<tiles, 320, sm, ws.stream>>>(ix->cent_h16t.as<__half>(), ix->cent_l16t.as<__half>(), ix->K,
                                            ws.Qh16t.as<__half>(), ws.Ql16t.as<__half>(), n_groups, B, QS,
                                            ws.qoff.as<int>(), ws.qrange_tc.as<float2>(), table, flags);
        KEV_END(PB_KERNEL_SCORES);
    });
    CK(cudaGetLastError());
    return PB_OK;
}

// diagnostic twin of the score table on the tensor cores, compared code by code with the exact one
static pb_status launch_k1_diag(pb_index *ix, Workspace &ws, int B, int QS) {
    if (!ix->cent_h16t.p || (ix->dim != 64 && ix->dim != 96 && ix->dim != 128)) return PB_OK;
    CKS(ws.ST16b.ensure((size_t)B * ix->K * QS * 2));
    CKS(ws.k1diag.ensure((size_t)(B + 4) * 4));
    CK(cudaMemsetAsync(ws.k1diag.p, 0, (size_t)(B + 4) * 4, ws.stream));
    CKS(launch_k1_table(ix, ws, B, QS, ws.ST16b.as<unsigned short>(), ws.k1diag.as<int>() + 4));
    k_diff16<<<dim3(ix->sm_count, B), 256, 0, ws.stream>>>(ws.ST16.as<unsigned short>(), ws.ST16b.as<unsigned short>(),
                                                          ws.qoff.as<int>(), ix->K, QS, ws.k1diag.as<int>());
    CK(cudaGetLastError());
    return PB_OK;
}

// chunk size of the threshold-first probe: 1024 centroids, fewer for small K so that at least 2n chunks exist (tau is
// the n-th largest chunk maximum); *n_chunks < n means the path cannot run
static int probe_chunk_rows(long long K, int n, int *n_chunks) {
    int rows = 1024;
    while (rows > 32 && (K + rows - 1) / rows < 2ll * n) rows >>= 1;
    *n_chunks = (int)((K + rows - 1) / rows);
    return rows;
}

// The threshold-first probe on the 16-bit table ws.ST16: the largest code of each chunk of centroids per query token,
// tau = the n-th largest of those, every centroid at or above tau into a per-row list, the top n of each list into
// ws.sel.  A row that cannot trust its list raises the returned device flag.  On the tensor-core table (tc) the
// collect settles the codes within the margin around tau by exact dots, and the merge runs whatever the flag says,
// since k_cells_unique reads every row of sel.  On the exact path the collect reads the fp32 table ws.ST, and the merge
// leaves sel to the per-lane list scan when the flag is up.
static pb_status launch_threshold_probe(pb_index *ix, Workspace &ws, int B, int QS, int n, int n_chunks, int chunk_rows,
                                        bool tc, int **d_fallback_out) {
    const int cap = n * std::max(2, 128 / n);
    CKS(ws.cmax16.ensure((size_t)B * n_chunks * QS * 2));
    CKS(ws.tau16.ensure((size_t)B * QS * 4));
    CKS(ws.plist.ensure((size_t)B * QS * cap * 8));
    CKS(ws.pcount.ensure((size_t)B * QS * 4 + 16));
    CK(cudaMemsetAsync(ws.plist.p, 0, (size_t)B * QS * cap * 8, ws.stream));
    CK(cudaMemsetAsync(ws.pcount.p, 0, (size_t)B * QS * 4 + 16, ws.stream));
    int *d_fallback = ws.pcount.as<int>() + (size_t)B * QS;
    const dim3 grid((n_chunks + 3) / 4, B);
    k_chunkmax16<<<grid, 128, 0, ws.stream>>>(ws.ST16.as<unsigned short>(), ix->K, QS, n_chunks, chunk_rows,
                                              ws.cmax16.as<unsigned short>());
    k_tau16<<<dim3(QS, B), 32, 0, ws.stream>>>(ws.cmax16.as<unsigned short>(), ws.qoff.as<int>(), QS, n, n_chunks,
                                              ws.qflag.as<int>(), ws.tau16.as<uint32_t>(), d_fallback);
    if (tc)
        k_collect16_tc<<<grid, 128, 0, ws.stream>>>(ws.ST16.as<unsigned short>(), ws.Q.as<float>(), ws.qoff.as<int>(),
                                                    ix->centroids.as<float>(), ix->dim, 2 * ix->k1_margin + 1, ix->K, QS,
                                                    n_chunks, chunk_rows, ws.tau16.as<uint32_t>(), cap, ws.pcount.as<int>(),
                                                    ws.plist.as<u64>(), d_fallback);
    else
        k_collect16<<<grid, 128, 0, ws.stream>>>(ws.ST16.as<unsigned short>(), ws.ST.as<float>(), ix->K, QS, n_chunks,
                                                 chunk_rows, ws.tau16.as<uint32_t>(), cap, ws.pcount.as<int>(),
                                                 ws.plist.as<u64>(), d_fallback);
    k_topn_merge<<<dim3(QS, B), 32, 0, ws.stream>>>(ws.plist.as<u64>(), ws.qoff.as<int>(), QS, n, cap / n, ws.sel.as<u64>(),
                                                  tc ? nullptr : d_fallback, 0);
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_PROBE] += 4;
    *d_fallback_out = d_fallback;
    return PB_OK;
}

// a2 on the exact fp32 kernel: the table ws.ST and, with16, its 16-bit twin ws.ST16 (under PB_K1_TC_DIAG also the
// tensor-core table, compared with it)
static pb_status launch_centroid_scores(pb_index *ix, Workspace &ws, int B, int QS, int *launches, bool with16) {
    const int tiles = (int)((ix->K + PB_TOK_TILE - 1) / PB_TOK_TILE);
    // enough CTAs to fill the machine twice over; each CTA keeps its centroid tile in smem and walks queries
    int groups = std::max(1, std::min(B, (4 * ix->sm_count + tiles - 1) / tiles));
    // packed fp32 FMA (FFMA2): query rows interleaved pairwise, one instruction advances two dots
    CKS(ws.Qi.ensure((size_t)B * QS * ix->dim * 4));
    k_interleave_query_rows<<<dim3(8, B), 256, 0, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), QS, ix->dim,
                                                               ws.Qi.as<float>());
    PB_DIM_SWITCH(ix->dim, {
        auto kern = k_centroid_scores<DIM, true>;
        CKS(set_smem(kern, smem_scores(DIM)));
        KEV_BEGIN(PB_KERNEL_SCORES);
        kern<<<dim3(tiles, groups), 128, smem_scores(DIM), ws.stream>>>(ws.Qi.as<float>(), ws.qoff.as<int>(), B, QS,
                                                                        ix->centroids.as<float>(), ix->K,
                                                                        ws.ST.as<float>(),
                                                                        with16 ? ws.ST16.as<unsigned short>() : nullptr,
                                                                        ws.qrange.as<float2>(), ws.qflag.as<int>());
        KEV_END(PB_KERNEL_SCORES);
    });
    CK(cudaGetLastError());
    if (launches) *launches += 2;
    if (with16 && ix->k1_diag && ix->cent_h16t.p) CKS(launch_k1_diag(ix, ws, B, QS));
    return PB_OK;
}

// all-gather of `count` 64-bit words per rank over whichever transport the handle joined
static pb_status shard_allgather(pb_index *ix, cudaStream_t stream, const void *send, void *recv, size_t count) {
    if (ix->comm) {
        CKN(g_nccl.AllGather(send, recv, count, PB_NCCL_UINT64, ix->comm, stream));
        return PB_OK;
    }
    pb_shard_group *g = ix->group;
    if (!g) return pb_fail(PB_ERR_COMM, "sharded handle without a transport");
    cudaError_t e = cudaStreamSynchronize(stream);  // my send buffer is complete
    if (e != cudaSuccess) {
        g->fail();
        return pb_fail(PB_ERR_CUDA, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
    }
    g->send[ix->rank] = send;
    if (!g->barrier()) return pb_fail(PB_ERR_COMM, "shard group: a peer failed or timed out");
    for (int p = 0; p < g->world && e == cudaSuccess; ++p)
        e = cudaMemcpyPeerAsync(static_cast<char *>(recv) + (size_t)p * count * 8, ix->device, g->send[p], g->dev[p],
                                count * 8, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);  // peers may reuse their send buffers after the barrier
    if (e != cudaSuccess) {
        g->fail();
        return pb_fail(PB_ERR_CUDA, "shard group copy failed: %s", cudaGetErrorString(e));
    }
    if (!g->barrier()) return pb_fail(PB_ERR_COMM, "shard group: a peer failed or timed out");
    return PB_OK;
}

// A collective decision of a sharded handle: one 64-bit word per rank, all-gathered, read on every rank's host
// (returned in ws.hredo[0 .. world)).  `d_lo`, when given, is a device int copied over the low half of `mine` (a flag
// raised on the device).
static pb_status shard_vote(pb_index *ix, Workspace &ws, u64 mine, const int *d_lo, const u64 **all) {
    const int G = ix->world;
    CKS(ws.redoflag.ensure((size_t)(G + 1) * 8));
    CKS(ws.hredo.ensure((size_t)(G + 1) * 8));
    u64 *h = ws.hredo.as<u64>();
    h[G] = mine;
    CK(cudaMemcpyAsync(ws.redoflag.p, h + G, 8, cudaMemcpyHostToDevice, ws.stream));
    if (d_lo) CK(cudaMemcpyAsync(ws.redoflag.p, d_lo, 4, cudaMemcpyDeviceToDevice, ws.stream));
    CKS(shard_allgather(ix, ws.stream, ws.redoflag.p, ws.redoflag.as<u64>() + 1, 1));
    CK(cudaMemcpyAsync(h, ws.redoflag.as<u64>() + 1, (size_t)G * 8, cudaMemcpyDeviceToHost, ws.stream));
    CK(cudaStreamSynchronize(ws.stream));
    *all = h;
    return PB_OK;
}

struct KeptView {  // the docs the exact stage scores: the cut's output, or the filter's survivors
    uint32_t *kept;
    int *nkept;
    long long *tokp;
    uint32_t *krank;  // global approximate rank (sharded) or nullptr
};

static pb_status launch_exact(pb_index *ix, Workspace &ws, const KeptView &kv, int B, int QS, int Mcap, int kept_shared,
                              long long max_tokens, int *launches, const int *only_flagged = nullptr, bool timed = true) {
    // each CTA owns a contiguous range of chunks; aim for 8 waves of 2 CTAs/SM over the whole grid
    long long chunks = (max_tokens + PB_TOK_TILE - 1) / PB_TOK_TILE;
    long long want = std::max<long long>(1, ((long long)ix->sm_count * 16 + B - 1) / B);
    int gx = (int)std::max<long long>(1, std::min<long long>(chunks, want));
    PB_DIM_SWITCH(ix->dim, {
        auto kern = k_exact<DIM, false>;
        CKS(set_smem(kern, smem_exact(DIM, ix->packed)));
        if (timed) KEV_BEGIN(PB_KERNEL_EXACT);
        kern<<<dim3(gx, B), 128, smem_exact(DIM, ix->packed), ws.stream>>>(
            ws.Q.as<float>(), ws.qoff.as<int>(), QS, ix->centroids.as<float>(), ix->w_rev.as<float>(), ix->nbits,
            ix->codes.as<uint32_t>(), ix->residuals.as<uint8_t>(), ix->doc_off.as<long long>(), nullptr,
            kv.kept, kv.nkept, kv.tokp, Mcap, kept_shared, ws.maxkey.as<uint32_t>(), only_flagged);
        if (timed) KEV_END(PB_KERNEL_EXACT);
    });
    CK(cudaGetLastError());
    if (launches) ++*launches;
    return PB_OK;
}

static size_t smem_exact_tc(int dim, int packed, int nqt) {
    const int nbits = packed * 8 / dim;
    return (size_t)(dim / 8) * PB_XTC_LBO + (size_t)nqt * dim * 2 + (size_t)256 * (8 / nbits) * 2 + 64;
}

// error of one fp16 tensor-core similarity relative to |q| (derivation above k_exact_tc); 0 = filter unusable
static float filter_eps_unit(const pb_index *ix) {
    const float u = 1.0f / 2048.0f;  // fp16 unit roundoff
    const float vmin = ix->vmin * 0.9999f, wmax = ix->wmax * 1.0001f;
    if (!(vmin > 0.0f) || !(ix->cmax < 3.0e4f) || !(wmax < 3.0e4f)) return 0.0f;  // operands must fit fp16
    const float rho = u * ((ix->cmax + wmax) / vmin + 1.0f) * (1.0f + 2.0f * u);  // |v - v~| / |v|
    if (!(rho < 0.25f)) return 0.0f;
    const float sub = 3.0f * sqrtf((float)ix->dim) * 2.98e-8f / vmin;  // fp16 subnormal spacing 2^-25: h(c), h(w), their sum
    return u + (1.0f + u) * rho / (1.0f - 0.5f * rho) + sub + 4e-5f;
}

// the same for the linear filter (derivation above k_maxsim_tc and in DESIGN.md 4c); E = code error of the score table (0 = exact table)
static float filter_eps_unit2(const pb_index *ix, int E) {
    const float u = 1.0f / 2048.0f;
    const float vmin = ix->vmin * 0.9999f, wmax = ix->wmax * 1.0001f;
    if (!(vmin > 0.0f) || !(ix->cmax < 3.0e4f) || !(wmax < 3.0e4f)) return 0.0f;
    const float ds = ((float)E + 1.01f) * 2.0f * ix->cmax * 1.0001f / 65535.0f;
    const float dw = wmax * (2.0f * u + u * u + 3.0517578e-5f);
    // k_maxsim_tc decodes a code with one FFMA whose folded constant (|.| <= 257 R, R = |q| cmax) is rounded once:
    // <= 257 R 2^-24 = 0.503 code units
    const float dfold = 0.53f * 2.0f * ix->cmax * 1.0001f / 65535.0f;
    const float eps = (ds + dw + dfold) / vmin + 8e-6f;
    return eps < 0.05f ? eps : 0.0f;
}

static size_t smem_maxsim_tc(int dim, int packed, int nqt) {
    const int nbits = packed * 8 / dim;
    return (size_t)2 * (dim / 8) * PB_XTC_LBO + (size_t)nqt * dim * 2 + (size_t)256 * (8 / nbits) * 2 * (nbits == 4 ? 4 : 1) +
           4 * 128 * sizeof(MsMeta) +
           12 * 8 + 16;
}

// the warp-specialised linear estimate over the docs of `in`: pass 1 (pairs == nullptr) leaves per (doc, q) maxima in
// `keys`; pass 2 lists the (token, q) pairs within the certified band of the maxima `keys` holds at src_rank
static pb_status launch_maxsim_tc(pb_index *ix, Workspace &ws, const KeptView &in, int B, int QS, int Mcap, long long max_tokens,
                                  int nq_max, uint32_t *keys, const uint32_t *src_rank, float band_unit, u64 *pairs,
                                  int *n_pairs, int pair_cap, int kev) {
    const bool emit = pairs != nullptr;
    // CTAs per SM over the batch: ws_grid for pass 1 (all kept docs), ws_grid2 for pass 2 (the survivors, ~1/10 of the
    // tokens; fewer, longer CTAs measured slower: the pass is latency-bound and wants the parallelism)
    long long chunks = (max_tokens + 127) / 128;
    long long want = std::max<long long>(1, ((long long)ix->sm_count * (emit ? ix->ws_grid2 : ix->ws_grid) + B - 1) / B);
    int gx = (int)std::max<long long>(1, std::min<long long>(chunks, want));
    const int nqt = nq_max <= 32 ? 32 : 64;
    const size_t sm = smem_maxsim_tc(ix->dim, ix->packed, nqt);
    CKS(ws.gbase.ensure((size_t)B * Mcap * 8));
    k_doc_gbase<<<dim3((Mcap + 255) / 256, B), 256, 0, ws.stream>>>(in.kept, in.nkept, in.tokp, ix->doc_off.as<long long>(), Mcap,
                                                                    ws.gbase.as<long long>());
    CK(cudaGetLastError());
    PB_TC_DIM_SWITCH(ix->dim, PB_NBITS_SWITCH(ix->nbits, {
        auto kern = emit ? (nqt == 32 ? k_maxsim_tc<DIM, NBITS, 32, true> : k_maxsim_tc<DIM, NBITS, 64, true>)
                         : (nqt == 32 ? k_maxsim_tc<DIM, NBITS, 32, false> : k_maxsim_tc<DIM, NBITS, 64, false>);
        CKS(set_smem(kern, sm));
        if (kev >= 0) KEV_BEGIN(kev);
        kern<<<dim3(gx, B), 288, sm, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), QS, ws.ST16.as<unsigned short>(),
                                                  ix->K, ws.qrange.as<float2>(), ws.qflag.as<int>(), ix->w_rev.as<float>(),
                                                  ix->codes.as<uint32_t>(), ix->residuals.as<uint8_t>(),
                                                  ix->tok_inv_norm.as<float>(), ws.gbase.as<long long>(),
                                                  in.nkept, in.tokp, Mcap, keys, src_rank, ws.qnmax.as<float>(),
                                                  band_unit, pairs, n_pairs, pair_cap);
        if (kev >= 0) KEV_END(kev);
    }));
    CK(cudaGetLastError());
    return PB_OK;
}

// a7': tensor-core estimate of every kept doc, then the survivors that can still reach the top_k
static pb_status launch_filter(pb_index *ix, Workspace &ws, const KeptView &in, const KeptView &out, int B, int QS, int Mcap,
                               int top_k, long long max_tokens, float eps_unit, int nq_max, bool linear, bool keep_keys,
                               int *launches) {
    long long chunks = (max_tokens + 127) / 128;
    long long want = std::max<long long>(1, ((long long)ix->sm_count * ix->xtc_grid + B - 1) / B);
    int gx = (int)std::max<long long>(1, std::min<long long>(chunks, want));
    const int nqt = nq_max <= 32 ? 32 : 64;
    const size_t sm = smem_exact_tc(ix->dim, ix->packed, nqt);
    // keep_keys: the per (doc, q) maxima go to their own buffer and stay there for the pair pass of the exact stage
    uint32_t *keys = keep_keys ? ws.estkey.as<uint32_t>() : ws.maxkey.as<uint32_t>();
    if (keep_keys) CK(cudaMemsetAsync(keys, 0, (size_t)B * Mcap * QS * 4, ws.stream));
    if (linear) {
        CKS(launch_maxsim_tc(ix, ws, in, B, QS, Mcap, max_tokens, nq_max, keys, nullptr, 0.0f, nullptr, nullptr, 0,
                             PB_KERNEL_FILTER));
    } else {
        PB_TC_DIM_SWITCH(ix->dim, PB_NBITS_SWITCH(ix->nbits, {
            auto kern = nqt == 32 ? k_exact_tc<DIM, NBITS, 32> : k_exact_tc<DIM, NBITS, 64>;
            CKS(set_smem(kern, sm));
            KEV_BEGIN(PB_KERNEL_FILTER);
            kern<<<dim3(gx, B), 128, sm, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), QS,
                                                      ix->centroids_f16.as<__half>(), ix->w_rev.as<float>(),
                                                      ix->codes.as<uint32_t>(), ix->residuals.as<uint8_t>(),
                                                      ix->doc_off.as<long long>(), in.kept, in.nkept, in.tokp, Mcap, keys);
            KEV_END(PB_KERNEL_FILTER);
        }));
        CK(cudaGetLastError());
    }
    k_tc_finalize<<<dim3((Mcap + 7) / 8, B), 256, 0, ws.stream>>>(keys, ws.qoff.as<int>(), QS, in.nkept, Mcap, in.tokp,
                                                                  ws.est.as<float>(), keep_keys ? 0 : 1);
    CK(cudaGetLastError());
    const int Pm = pow2_ceil(Mcap);
    CKS(set_smem(k_tc_select, (size_t)Pm * 8));
    k_tc_select<<<B, 1024, (size_t)Pm * 8, ws.stream>>>(ws.est.as<float>(), in.kept, in.krank, in.nkept, Mcap, top_k,
                                                        ws.qoff.as<int>(), ws.qnmax.as<float>(), eps_unit,
                                                        ix->doc_off.as<long long>(), out.kept, out.krank, out.nkept,
                                                        out.tokp, ws.ktok2.as<long long>(),
                                                        keep_keys ? ws.srcrank.as<uint32_t>() : nullptr);
    CK(cudaGetLastError());
    if (launches) *launches += 3 + (keep_keys ? 1 : 0);
    return PB_OK;
}

// ------------------------------------------------------------------------------------------
// the search pipeline: plan_call decides what holds for the whole call, run_pass runs the stages a2..a9 over one
// sub-batch (stage_* below, in pipeline order), search_impl_inner loops over the sub-batches
// ------------------------------------------------------------------------------------------
struct SearchIO {
    const float *queries;  // host or device
    bool queries_on_device;
    const int64_t *q_off;  // host
    int64_t n_queries;
    const int64_t *subset;  // host
    int64_t n_subset;
    bool has_subset;
    int64_t *out_ids;  // host or device
    float *out_scores;
    int32_t *out_counts;
    bool out_on_device;
    pb_trace *trace;
};

struct CallPlan {
    const pb_search_params *p = nullptr;
    const SearchIO *io = nullptr;
    int64_t Bt = 0;                  // queries of the call
    bool empty = false;              // every result is empty: no sub-batch runs
    int top_k = 0, M = 0, Mcap = 1;  // M: docs the cut keeps, min(n_full_scores, max(n_full_scores / 4, top_k))
    bool batched = false, sharded = false;
    bool fast = false;               // two-pass approximate stage on a 16-bit table
    long long Wd = 0, Wk = 0;        // 32-bit words of a doc / centroid bitmap
    const uint32_t *d_subset_bits = nullptr, *d_elig = nullptr;
    int n_probe = 0;
    long long n_elig = 0;
    bool all_eligible = false, big_probe = false;
    bool tc_call = false;            // a sub-batch whose rows fit (QS / 8 <= 32) takes the tensor-core path
    int QB = 1;                      // queries per sub-batch
};

// how a3 picks the cells of each query token
enum class ProbeMode {
    TensorCore,   // threshold-first on the estimate table, done by run_k1_tc in a2
    Threshold,    // threshold-first on the 16-bit table; the per-lane list scan where the device raises the fallback flag
    List,         // per-lane list scan of the fp32 table
    AllEligible,  // every eligible centroid (a subset whose scaled n_ivf_probe reaches them all)
    BigProbe,     // row-wise radix select (n_ivf_probe beyond the per-lane lists)
};

// The pinned host buffer of one pass (ws.hcounts): the query offsets going to the device, and the per-query counts,
// work counters and flags coming back
struct PassHost {
    int *qoff;                     // [B + 1]
    unsigned long long *counters;  // [B + 2] ws.counters: candidate codes gathered, kept-doc tokens per query, re-check gathers
    long long *surv_tokens;        // [B] tokens of the filter's survivors
    int *n_cells, *n_cand, *n_kept, *survivors, *rechecked, *pairs, *need_exact;  // [B] each
    int *fell;                     // the threshold-first probe gave up
    // lays the fields out from `base`, 16-byte aligned, and returns their size (base == nullptr: only the size)
    size_t carve(char *base, int B) {
        size_t off = 0;
        auto at = [&](size_t bytes) {
            off = (off + 15) & ~(size_t)15;
            char *q = base ? base + off : nullptr;
            off += bytes;
            return q;
        };
        qoff = reinterpret_cast<int *>(at((size_t)(B + 1) * 4));
        counters = reinterpret_cast<unsigned long long *>(at((size_t)(B + 2) * 8));
        surv_tokens = reinterpret_cast<long long *>(at((size_t)B * 8));
        for (int **f : {&n_cells, &n_cand, &n_kept, &survivors, &rechecked, &pairs, &need_exact})
            *f = reinterpret_cast<int *>(at((size_t)B * 4));
        fell = reinterpret_cast<int *>(at(4));
        return off;
    }
};

// One pass over the sub-batch [b0, b0 + B): its shape (H2D), then what each stage decides for the stages after it
struct Pass {
    int64_t b0 = 0, r0 = 0, R = 0;  // first query, its first token, the sub-batch's tokens
    int B = 0, nq_max = 0, QS = 0;
    bool tc = false;                // a2 + a3 on the tensor-core table
    ProbeMode probe = ProbeMode::List;
    int cells_cap = 0;              // a3: cells per query
    int *d_fallback = nullptr;      // a3: device flag of the threshold-first probe (0 = it did the work)
    const uint32_t *cand_list = nullptr;  // a5: the candidates scored, which the cut reads
    const int *cand_n = nullptr;
    KeptView kv = {};               // a6 / a7: the docs the exact stage scores
    bool filt = false;              // a7: the certified filter ran
    bool pairs = false;             // a8: the exact stage ran on (token, query token) pairs
    long long *d_ids = nullptr;     // a9: the results on the device
    float *d_sc = nullptr;
    int *d_cn = nullptr;
    PassHost host = {};
};

// The subset of a call: its doc bitmap and, with the dense variant, the eligible centroids and the scaled n_ivf_probe
// (search.rs:350-382).  No eligible centroid: every per-token pool is empty, so every result is (plan.empty).
static pb_status plan_subset(pb_index *ix, Workspace &ws, const SearchIO &io, CallPlan &plan) {
    const pb_search_params *p = plan.p;
    CKS(ws.subset_bits.ensure((size_t)plan.Wd * 4));
    CK(cudaMemsetAsync(ws.subset_bits.p, 0, (size_t)plan.Wd * 4, ws.stream));
    if (io.n_subset > 0) {
        CKS(ws.subset.ensure((size_t)io.n_subset * 8));
        CK(cudaMemcpyAsync(ws.subset.p, io.subset, (size_t)io.n_subset * 8, cudaMemcpyHostToDevice, ws.stream));
        k_subset_bits<<<296, 256, 0, ws.stream>>>(ws.subset.as<long long>(), io.n_subset, ix->doc_id_base, ix->D,
                                                 ws.subset_bits.as<uint32_t>());
        CK(cudaGetLastError());
    }
    plan.d_subset_bits = ws.subset_bits.as<uint32_t>();
    if (plan.batched) return PB_OK;
    CKS(ws.elig.ensure((size_t)plan.Wk * 4));
    CKS(ws.misc.ensure(64));
    CK(cudaMemsetAsync(ws.elig.p, 0, (size_t)plan.Wk * 4, ws.stream));
    CK(cudaMemsetAsync(ws.misc.p, 0, 64, ws.stream));
    k_eligible_bits<<<ix->sm_count * 8, 256, 0, ws.stream>>>(plan.d_subset_bits, ix->D, ix->doc_off.as<long long>(),
                                                             ix->codes.as<uint32_t>(), ws.elig.as<uint32_t>());
    k_popcount<<<ix->sm_count, 256, 0, ws.stream>>>(ws.elig.as<uint32_t>(), plan.Wk, ws.misc.as<unsigned long long>());
    CK(cudaGetLastError());
    unsigned long long ne = 0;
    CK(cudaMemcpyAsync(&ne, ws.misc.p, 8, cudaMemcpyDeviceToHost, ws.stream));
    CK(cudaStreamSynchronize(ws.stream));
    plan.n_elig = (long long)ne;
    if (plan.n_elig == 0) {
        plan.empty = true;
        return PB_OK;
    }
    unsigned long long scaled = io.n_subset > 0 ? (unsigned long long)p->n_ivf_probe * (unsigned long long)ix->D /
                                                      (unsigned long long)io.n_subset
                                                : (unsigned long long)p->n_ivf_probe;
    scaled = std::max<unsigned long long>(scaled, (unsigned long long)p->n_ivf_probe);
    scaled = std::min<unsigned long long>(scaled, (unsigned long long)plan.n_elig);
    plan.d_elig = ws.elig.as<uint32_t>();
    if ((long long)scaled >= plan.n_elig) plan.all_eligible = true;
    else plan.n_probe = (int)scaled;
    return PB_OK;
}

// Everything a search call decides once: the argument checks, the cut size, the variant, the subset, the probe, whether
// the tensor-core path is open and the sub-batch size.  Takes the call's workspace from the pool (lease) unless the
// call has no queries.  `lanes`: concurrent slices of the caller's batch, which share the workspace budget.
static pb_status plan_call(pb_index *ix, const pb_search_params *p, const SearchIO &io, int lanes, WorkspaceLease &lease,
                           CallPlan &plan) {
    if (!ix || !p) return pb_fail(PB_ERR_INVALID, "null argument");
    if (io.n_queries < 0) return pb_fail(PB_ERR_INVALID, "n_queries < 0");
    if (io.n_queries > 0 && (!io.queries || !io.q_off)) return pb_fail(PB_ERR_INVALID, "null queries");
    if (p->top_k < 0 || p->n_full_scores < 0) return pb_fail(PB_ERR_INVALID, "top_k / n_full_scores must be >= 0");
    if (p->n_ivf_probe < 1) return pb_fail(PB_ERR_INVALID, "n_ivf_probe must be >= 1");
    if (p->top_k > 0 && (!io.out_ids || !io.out_scores)) return pb_fail(PB_ERR_INVALID, "null outputs");
    if (!io.out_counts) return pb_fail(PB_ERR_INVALID, "null out_counts");
    CK(cudaSetDevice(ix->device));
    g_stats = Stats();
    plan.p = p;
    plan.io = &io;
    const int64_t Bt = plan.Bt = io.n_queries;
    if (Bt == 0) return PB_OK;
    for (int64_t b = 0; b < Bt; ++b)
        if (io.q_off[b + 1] < io.q_off[b]) return pb_fail(PB_ERR_INVALID, "q_tok_offsets not monotone");
    plan.top_k = (int)p->top_k;
    const long long n_dec = std::max<long long>(p->n_full_scores / 4, p->top_k);  // search.rs:468
    const long long Mll = std::min<long long>(p->n_full_scores, n_dec);             // take(nfs).take(n_dec)
    if (Mll > 16384)
        return pb_fail(PB_ERR_UNSUPPORTED, "min(n_full_scores, max(n_full_scores/4, top_k)) = %lld exceeds 16384", Mll);
    plan.M = (int)Mll;
    plan.Mcap = std::max(plan.M, 1);
    plan.batched = p->centroid_batch_size > 0 && ix->K > p->centroid_batch_size;  // search.rs:337
    plan.sharded = ix->world > 1;
    if (plan.sharded && io.has_subset && !plan.batched)
        return pb_fail(PB_ERR_UNSUPPORTED, "subset with the dense variant needs the global eligible-centroid set; "
                                            "not built for doc-sharded indices");
    CKS(lease.acquire());
    Workspace &ws = *lease.ws;
    // a shard with no documents still takes part in the exchanges
    plan.empty = plan.M == 0 || plan.top_k == 0 || (ix->D == 0 && !plan.sharded);
    if (plan.empty) return PB_OK;

    plan.Wd = (ix->D + 31) / 32;
    plan.Wk = (ix->K + 31) / 32;
    plan.n_probe = (int)std::min<long long>(p->n_ivf_probe, ix->K);
    if (io.has_subset) {
        CKS(plan_subset(ix, ws, io, plan));
        if (plan.empty) return PB_OK;
    }
    // effective n_ivf_probe beyond 64: the dense variant switches to a row-wise radix select; the batched variant's
    // heap-order threshold rule is tied to the streaming formulation, whose per-lane lists hold up to 192 entries
    const int n_probe = plan.n_probe;
    const int stream_max = plan.batched ? 192 : 64;
    plan.big_probe = !plan.all_eligible && n_probe > stream_max;
    if (plan.big_probe && plan.batched)
        return pb_fail(PB_ERR_UNSUPPORTED, "n_ivf_probe %d > 192 with the batched variant is not built", n_probe);

    // ---- sub-batching: bound the transposed score matrix ----
    int nq_max_all = 0;
    for (int64_t b = 0; b < Bt; ++b) nq_max_all = std::max<int>(nq_max_all, (int)(io.q_off[b + 1] - io.q_off[b]));
    const int QS_all = query_row_tokens(nq_max_all);
    if (!plan.all_eligible && !plan.big_probe && (long long)QS_all * n_probe > 8192)
        return pb_fail(PB_ERR_UNSUPPORTED, "query tokens x n_ivf_probe = %lld exceeds 8192", (long long)QS_all * n_probe);
    size_t per_q = (size_t)ix->K * QS_all * sizeof(float);
    if (per_q >= ((size_t)1 << 32))
        return pb_fail(PB_ERR_UNSUPPORTED, "num_centroids x query tokens x 4 = %zu bytes per query exceeds 2^32", per_q);
    // the score table comes from the tensor cores unless something needs the dense fp32 S (an eligibility filter,
    // the radix-select probe, a trace) or the shape is outside the kernel's (DESIGN.md "a2"); all of that is fixed for
    // the call except the sub-batch's row width QS / 8 <= 32
    plan.fast = ix->fast_approx && !io.trace;  // trace wants every candidate's exact approximate score
    int n_chunks_k = 0;
    probe_chunk_rows(ix->K, n_probe, &n_chunks_k);
    plan.tc_call = k1_tc_usable(ix) && plan.fast && ix->probe16 && !ix->k1_diag && !plan.all_eligible && !plan.big_probe &&
                   !plan.d_elig && n_chunks_k >= n_probe && n_probe <= 192;
    // sub-batch size: the score tables (16-bit on the tensor-core path; fp32 and 16-bit otherwise) and the per-(query,
    // doc) scratch (candidate lists, code sums, approximate scores, cut keys, bitmap: 24.2 bytes per document) share
    // one budget
    const bool tc_all = plan.tc_call && QS_all / 8 <= 32;  // every sub-batch of the call can take the tensor-core path
    const size_t per_q_all = (size_t)ix->K * QS_all * (tc_all ? 2 : 6) + (size_t)ix->D * 24 + (size_t)ix->D / 8 + 4096;
    int QB = (int)std::max<size_t>(1, std::min<size_t>((size_t)Bt, ix->st_budget / lanes / per_q_all));
    QB = std::min(QB, 256);
    if (plan.sharded) {
        // every rank must cut the call into the same sub-batches (each sub-batch is a set of exchanges), but per_q_all
        // depends on the shard's own documents and tensor-core operands: the group takes the smallest size
        const u64 *all = nullptr;
        CKS(shard_vote(ix, ws, (u64)QB, nullptr, &all));
        for (int g = 0; g < ix->world; ++g) QB = std::min<int>(QB, (int)all[g]);
    }
    plan.QB = (int)((Bt + (Bt + QB - 1) / QB - 1) / ((Bt + QB - 1) / QB));  // equal sub-batches
    return PB_OK;
}

static ProbeMode probe_mode(const pb_index *ix, const CallPlan &plan, int QS, bool tc) {
    if (tc) return ProbeMode::TensorCore;
    if (plan.all_eligible) return ProbeMode::AllEligible;
    if (plan.big_probe) return ProbeMode::BigProbe;
    // threshold-first selection needs the 16-bit table and at least n_probe chunk maxima
    const int n = plan.n_probe;
    int n_chunks = 0;
    probe_chunk_rows(ix->K, n, &n_chunks);
    const bool thr = plan.fast && !plan.d_elig && ix->probe16 && QS / 8 <= 32 && n_chunks >= n && n <= 192;
    return thr ? ProbeMode::Threshold : ProbeMode::List;
}

// ---- H2D: the shape of the sub-batch at ps.b0, its query tokens and offsets ----
static pb_status stage_h2d(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const SearchIO &io = *plan.io;
    ps.B = (int)std::min<int64_t>(plan.QB, plan.Bt - ps.b0);
    ps.r0 = io.q_off[ps.b0];
    ps.R = io.q_off[ps.b0 + ps.B] - ps.r0;
    for (int b = 0; b < ps.B; ++b) ps.nq_max = std::max(ps.nq_max, (int)(io.q_off[ps.b0 + b + 1] - io.q_off[ps.b0 + b]));
    ps.QS = query_row_tokens(ps.nq_max);
    const size_t qbytes = (size_t)ps.R * ix->dim * 4;
    CKS(ws.Q.ensure(std::max<size_t>(qbytes, 16)));
    CKS(ws.qoff.ensure((size_t)(ps.B + 1) * 4));
    if (ps.R > 0) {
        const float *src = io.queries + (size_t)ps.r0 * ix->dim;
        if (io.queries_on_device) CK(cudaMemcpyAsync(ws.Q.p, src, qbytes, cudaMemcpyDeviceToDevice, ws.stream));
        else {
            CKS(ws.hq.ensure(qbytes));
            memcpy(ws.hq.p, src, qbytes);
            CK(cudaMemcpyAsync(ws.Q.p, ws.hq.p, qbytes, cudaMemcpyHostToDevice, ws.stream));
        }
    }
    CKS(ws.hcounts.ensure(PassHost().carve(nullptr, ps.B)));
    ps.host.carve(ws.hcounts.as<char>(), ps.B);
    for (int b = 0; b <= ps.B; ++b) ps.host.qoff[b] = (int)(io.q_off[ps.b0 + b] - ps.r0);
    CK(cudaMemcpyAsync(ws.qoff.p, ps.host.qoff, (size_t)(ps.B + 1) * 4, cudaMemcpyHostToDevice, ws.stream));
    return PB_OK;
}

// a2 + a3 on the tensor-core table.  Nothing is read back here: a flagged query or a probe-list overflow raises
// ps.d_fallback on the device, the kernels after it stay memory-safe, and run_pass redoes the sub-batch on the exact
// path once it sees the flag at the end.
static pb_status run_k1_tc(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const pb_search_params *p = plan.p;
    const int B = ps.B, QS = ps.QS, n = plan.n_probe;
    int n_chunks = 0;
    const int chunk_rows = probe_chunk_rows(ix->K, n, &n_chunks);
    const int cm = 2 * ix->k1_margin + 1;
    CKS(ws.Qi.ensure((size_t)B * QS * ix->dim * 4));
    k_interleave_query_rows<<<dim3(8, B), 256, 0, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), QS, ix->dim, ws.Qi.as<float>());
    CKS(launch_k1_table(ix, ws, B, QS, ws.ST16.as<unsigned short>(), ws.qflag.as<int>()));
    g_stats.launches[PB_STAGE_CENTROID_SCORES] += 4;
    const int cells_cap = (int)std::min<long long>((long long)QS * n, ix->K);
    CKS(ws.sel.ensure((size_t)B * QS * n * 8));
    CKS(ws.cells.ensure((size_t)B * cells_cap * 4));
    CKS(ws.ncells.ensure((size_t)B * 4 + 16));
    CKS(ws.ulist.ensure((size_t)B * cells_cap * 4));
    CKS(ws.nulist.ensure((size_t)B * 4 + 16));
    CKS(ws.k1rows.ensure((size_t)B * cells_cap * QS * 4));
    CKS(launch_threshold_probe(ix, ws, B, QS, n, n_chunks, chunk_rows, true, &ps.d_fallback));
    // the selected centroids, their exact rows, the variant's threshold rule
    const int P = pow2_ceil(ps.nq_max * n);
    CKS(set_smem(k_cells_unique, (size_t)P * 8));
    k_cells_unique<<<B, 256, (size_t)P * 8, ws.stream>>>(ws.sel.as<u64>(), ws.qoff.as<int>(), QS, n, cells_cap,
                                                         ws.ulist.as<uint32_t>(), ws.nulist.as<int>());
    const size_t smr = (size_t)(PB_TOK_TILE * (ix->dim + 4) + PB_Q_TILE * ix->dim) * sizeof(float);
    PB_DIM_SWITCH(ix->dim, {
        auto kern = k_exact_rows<DIM>;
        CKS(set_smem(kern, smr));
        kern<<<dim3((cells_cap + PB_TOK_TILE - 1) / PB_TOK_TILE, B), 128, smr, ws.stream>>>(
            ws.Qi.as<float>(), ws.qoff.as<int>(), QS, ix->centroids.as<float>(), ws.ulist.as<uint32_t>(), ws.nulist.as<int>(),
            cells_cap, ws.k1rows.as<float>());
    });
    CKS(ws.cellflags.ensure((size_t)B * cells_cap * 4));
    k_cells_thr<<<dim3(8, B), 256, 0, ws.stream>>>(
        ws.sel.as<u64>(), ws.k1rows.as<float>(), ws.ulist.as<uint32_t>(), ws.nulist.as<int>(), ws.qoff.as<int>(), ix->K, QS, n,
        cells_cap, p->has_centroid_score_threshold, p->centroid_score_threshold, plan.batched ? 1 : 0,
        plan.batched ? (long long)p->centroid_batch_size : ix->K, ws.cellflags.as<int>(), ws.ST16.as<unsigned short>(),
        ws.qrange.as<float2>(), cm, ws.Q.as<float>(), ix->centroids.as<float>(), ix->dim, ws.cmax16.as<unsigned short>(),
        n_chunks, chunk_rows);
    k_cells_emit<<<B, 256, 0, ws.stream>>>(ws.ulist.as<uint32_t>(), ws.nulist.as<int>(), ws.cellflags.as<int>(), cells_cap,
                                           ws.cells.as<uint32_t>(), ws.ncells.as<int>());
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_PROBE] += 4;
    ps.cells_cap = cells_cap;
    return PB_OK;
}

// ---- a2 centroid scores: the query range and flags, then the tensor-core table (with a3) or the fp32 one ----
static pb_status stage_scores(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const int B = ps.B, QS = ps.QS;
    if (!ps.tc) CKS(ws.ST.ensure((size_t)B * ix->K * QS * sizeof(float)));
    if (plan.fast) {
        CKS(ws.ST16.ensure((size_t)B * ix->K * QS * 2));
        CKS(ws.qrange.ensure((size_t)B * 8 + 16));
        CKS(ws.qflag.ensure((size_t)B * 4 + 16));
        CKS(ws.qexp.ensure((size_t)B * 4 + 16));
        CKS(ws.qnmax.ensure((size_t)B * 4 + 16));
        k_query_range<<<B, 256, 0, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), ix->dim, ix->cmax,
                                                ws.qrange.as<float2>(), ws.qflag.as<int>(), ws.qexp.as<int>(),
                                                ws.qnmax.as<float>());
        CK(cudaGetLastError());
        g_stats.launches[PB_STAGE_CENTROID_SCORES] += 1;
    }
    if (ps.tc) return run_k1_tc(ix, ws, plan, ps);
    return launch_centroid_scores(ix, ws, B, QS, &g_stats.launches[PB_STAGE_CENTROID_SCORES], plan.fast);
}

// a3 by per-lane lists: k_topn_partial scans the fp32 table, k_topn_merge keeps the top n per row, k_cells applies the
// variant's threshold rule.  ProbeMode::Threshold runs the threshold-first probe first; the list scan then only does the
// rows whose fallback flag is up.
static pb_status probe_lists(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const pb_search_params *p = plan.p;
    const int B = ps.B, QS = ps.QS, n = plan.n_probe;
    const int n_chunks = (int)((ix->K + 1023) / 1024);
    ps.cells_cap = (int)std::min<long long>((long long)QS * n, ix->K);
    CKS(ws.partial.ensure((size_t)B * QS * n_chunks * n * 8));
    CKS(ws.sel.ensure((size_t)B * QS * n * 8));
    CKS(ws.cells.ensure((size_t)B * ps.cells_cap * 4));
    CKS(ws.ncells.ensure((size_t)B * 4 + 16));
    size_t sm1 = (size_t)4 * n * 32 * 8;
    CKS(set_smem(k_topn_partial, sm1));
    const bool thr = ps.probe == ProbeMode::Threshold;
    int t_chunks = 0;
    const int t_rows = probe_chunk_rows(ix->K, n, &t_chunks);
    if (thr) CKS(launch_threshold_probe(ix, ws, B, QS, n, t_chunks, t_rows, false, &ps.d_fallback));
    k_topn_partial<<<dim3((n_chunks + 3) / 4, B, (QS + 31) / 32), 128, sm1, ws.stream>>>(
        ws.ST.as<float>(), ws.qoff.as<int>(), ix->K, QS, n, plan.d_elig, ws.partial.as<u64>(), n_chunks, ps.d_fallback, 1);
    k_topn_merge<<<dim3(QS, B), 32, 0, ws.stream>>>(ws.partial.as<u64>(), ws.qoff.as<int>(), QS, n, n_chunks,
                                                  ws.sel.as<u64>(), ps.d_fallback, 1);
    const int P = pow2_ceil(ps.nq_max * n);
    size_t sm2 = (size_t)P * 12;
    CKS(set_smem(k_cells, sm2));
    k_cells<<<B, 256, sm2, ws.stream>>>(ws.sel.as<u64>(), ws.ST.as<float>(), ws.qoff.as<int>(), ix->K, QS, n,
                                        ps.cells_cap, p->has_centroid_score_threshold, p->centroid_score_threshold,
                                        plan.batched ? 1 : 0, plan.batched ? (long long)p->centroid_batch_size : ix->K,
                                        ws.cells.as<uint32_t>(), ws.ncells.as<int>(),
                                        thr ? ws.cmax16.as<unsigned short>() : nullptr, t_chunks, t_rows,
                                        ws.qrange.as<float2>(), ps.d_fallback);
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_PROBE] += 3;
    return PB_OK;
}

// ---- a3 probe: the cells (centroids) each query reads ----
static pb_status stage_probe(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const pb_search_params *p = plan.p;
    const int B = ps.B, QS = ps.QS;
    switch (ps.probe) {
        case ProbeMode::TensorCore: return PB_OK;  // the cells are in place (run_k1_tc)
        case ProbeMode::Threshold:
        case ProbeMode::List: return probe_lists(ix, ws, plan, ps);
        case ProbeMode::AllEligible: {
            ps.cells_cap = (int)plan.n_elig;
            CKS(ws.list.ensure((size_t)plan.n_elig * 4 + 16));
            CKS(ws.cells.ensure((size_t)B * ps.cells_cap * 4));
            CKS(ws.ncells.ensure((size_t)B * 4 + 16));
            int *d_listn = reinterpret_cast<int *>(ws.misc.as<char>() + 16);
            k_cells_from_bits<<<1, 1024, 0, ws.stream>>>(plan.d_elig, ix->K, ws.list.as<uint32_t>(), d_listn);
            k_cells_filter_list<<<B, 256, 0, ws.stream>>>(ws.list.as<uint32_t>(), d_listn, ws.ST.as<float>(),
                                                          ws.qoff.as<int>(), ix->K, QS, p->has_centroid_score_threshold,
                                                          p->centroid_score_threshold, ps.cells_cap, ws.cells.as<uint32_t>(),
                                                          ws.ncells.as<int>());
            break;
        }
        case ProbeMode::BigProbe: {
            ps.cells_cap = (int)std::min<long long>((long long)QS * plan.n_probe, ix->K);
            CKS(ws.cellbits.ensure((size_t)B * plan.Wk * 4));
            CKS(ws.cells.ensure((size_t)B * ps.cells_cap * 4));
            CKS(ws.ncells.ensure((size_t)B * 4 + 16));
            k_topn_select_row<<<dim3(QS, B), 256, 0, ws.stream>>>(ws.ST.as<float>(), ws.qoff.as<int>(), ix->K, QS, plan.n_probe,
                                                                  plan.d_elig, ws.cellbits.as<uint32_t>(), plan.Wk);
            k_cells_from_query_bits<<<B, 1024, 0, ws.stream>>>(ws.cellbits.as<uint32_t>(), plan.Wk, ws.ST.as<float>(),
                                                               ws.qoff.as<int>(), ix->K, QS, p->has_centroid_score_threshold,
                                                               p->centroid_score_threshold, ps.cells_cap, ws.cells.as<uint32_t>(),
                                                               ws.ncells.as<int>());
            break;
        }
    }
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_PROBE] += 2;
    return PB_OK;
}

// ---- a4 candidates: the docs of the cells' posting lists, once each ----
static pb_status stage_candidates(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const int B = ps.B;
    const long long Wd = plan.Wd;
    CKS(ws.bitmap.ensure((size_t)B * Wd * 4));
    CKS(ws.cand.ensure((size_t)B * ix->D * 4));
    CKS(ws.ncand.ensure((size_t)B * 4 + 16));
    k_mark<<<dim3(ps.cells_cap, B), 128, 0, ws.stream>>>(ws.cells.as<uint32_t>(), ws.ncells.as<int>(), ps.cells_cap,
                                                         ix->ivf.as<uint32_t>(), ix->ivf_off.as<long long>(), plan.d_subset_bits,
                                                         ws.bitmap.as<uint32_t>(), Wd);
    const int slices = (int)std::max<long long>(1, std::min<long long>(32, (4ll * ix->sm_count + B - 1) / B));
    CKS(ws.slicecnt.ensure((size_t)B * slices * 4));
    k_compact_count<<<dim3(slices, B), 256, 0, ws.stream>>>(ws.bitmap.as<uint32_t>(), Wd, ws.slicecnt.as<int>());
    k_compact_emit<<<dim3(slices, B), 256, 0, ws.stream>>>(ws.bitmap.as<uint32_t>(), Wd, ws.slicecnt.as<int>(),
                                                           ws.cand.as<uint32_t>(), ix->D, ws.ncand.as<int>());
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_CANDIDATES] += 3;
    return PB_OK;
}

// ---- a5 approximate scores: the two-pass approximate stage (with the re-check on the tensor-core path), or k_approx ----
static pb_status stage_approx(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const int B = ps.B, QS = ps.QS;
    int *L = g_stats.launches;
    CKS(ws.counters.ensure((size_t)(B + 2) * 8));  // [0] candidate codes gathered, [1+b] kept-doc tokens, [B+1] re-check gathers
    CK(cudaMemsetAsync(ws.counters.p, 0, (size_t)(B + 2) * 8, ws.stream));
    CKS(ws.approx.ensure((size_t)B * ix->D * 4));
    CKS(ws.keys.ensure((size_t)B * ix->D * 8));
    ps.cand_list = ws.cand.as<uint32_t>();
    ps.cand_n = ws.ncand.as<int>();
    if (plan.fast) {
        CKS(ws.lsum.ensure((size_t)B * ix->D * 4));
        CKS(ws.cand2.ensure((size_t)B * ix->D * 4));
        CKS(ws.ncand2.ensure((size_t)B * 4 + 16));
        const dim3 ga(ix->sm_count * ix->approx_grid, B);
        const uint32_t *list = ws.cand.as<uint32_t>();
        const int *list_n = ws.ncand.as<int>();
        KEV_BEGIN(PB_KERNEL_APPROX16);
        (QS <= 32 ? k_approx16<4> : k_approx16<8>)<<<ga, 256, 0, ws.stream>>>(
            ws.ST16.as<unsigned short>(), ws.qoff.as<int>(), ix->K, QS, ix->ucodes.as<uint32_t>(), ix->udoc_off.as<long long>(),
            list, ix->D, list_n, ws.lsum.as<uint32_t>(), ws.counters.as<unsigned long long>());
        KEV_END(PB_KERNEL_APPROX16);
        // band per query token in code units (W = band * nq + 8).  Exact table: +-1 code of rounding per token and side
        // plus the fp32 summation error -> 4.  Estimate table (k_scores_tc.cuh): W = nq (1.004 + 2 err) + nq^2/256 + 4
        // <= nq (ceil(1.004 + 2 err) + 1) + 8 for nq <= 256.
        const int band_per_q = ps.tc ? (int)ceilf(1.004f + 2.0f * std::max(k1_err_codes(ix->dim), (float)(ix->k1_margin - 1))) + 1 : 4;
        k_select_u32<<<B, 1024, 0, ws.stream>>>(ws.lsum.as<uint32_t>(), list_n, plan.M, band_per_q, ws.lsum.as<uint32_t>(), list,
                                                list_n, ix->D, ws.qoff.as<int>(), ws.qflag.as<int>(),
                                                ws.cand2.as<uint32_t>(), ws.ncand2.as<int>());
        CK(cudaGetLastError());
        L[PB_STAGE_APPROX] += 2;
        ps.cand_list = ws.cand2.as<uint32_t>();
        ps.cand_n = ws.ncand2.as<int>();
    }
    if (ps.tc) {  // the exact approximate score of the docs around the cut from pinned-order dots (no dense fp32 S)
        const int rc_cap = 2 * plan.Mcap + 1024, pair_cap = 64 * rc_cap;
        CKS(ws.rcmax.ensure((size_t)B * rc_cap * QS * 4));
        CKS(ws.rcpairs.ensure((size_t)B * pair_cap * 8));
        CKS(ws.rcn.ensure((size_t)B * 4 + 16));
        CK(cudaMemsetAsync(ws.rcn.p, 0, (size_t)B * 4, ws.stream));
        (QS <= 32 ? k_recheck_pairs<4> : k_recheck_pairs<8>)<<<dim3(ix->sm_count * 2, B), 256, 0, ws.stream>>>(
            ws.ST16.as<unsigned short>(), ws.qoff.as<int>(), ix->K, QS, ix->ucodes.as<uint32_t>(), ix->udoc_off.as<long long>(),
            ps.cand_list, ix->D, ps.cand_n, 2 * ix->k1_margin + 1, rc_cap, pair_cap, ws.rcpairs.as<u64>(), ws.rcn.as<int>(),
            ps.d_fallback, ws.counters.as<unsigned long long>() + B + 1);
        k_recheck_dots<<<dim3(ix->sm_count * 2, B), 128, 0, ws.stream>>>(ws.rcpairs.as<u64>(), ws.rcn.as<int>(), pair_cap,
                                                                         ws.Q.as<float>(), ws.qoff.as<int>(),
                                                                         ix->centroids.as<float>(), ix->dim, rc_cap, QS,
                                                                         ws.rcmax.as<uint32_t>());
        k_recheck_sum<<<dim3(ix->sm_count, B), 256, 0, ws.stream>>>(ws.rcmax.as<uint32_t>(), ws.qoff.as<int>(), QS, ps.cand_list,
                                                                    ix->D, ps.cand_n, rc_cap, ws.approx.as<float>(),
                                                                    ws.keys.as<u64>(), (uint32_t)ix->doc_id_base);
        L[PB_STAGE_APPROX] += 2;
    } else
        k_approx<<<dim3(ix->sm_count * 8, B), 256, 0, ws.stream>>>(
            ws.ST.as<float>(), ws.qoff.as<int>(), ix->K, QS, ix->ucodes.as<uint32_t>(), ix->udoc_off.as<long long>(),
            ps.cand_list, ix->D, ps.cand_n, ws.approx.as<float>(), ws.keys.as<u64>(),
            plan.fast ? ws.counters.as<unsigned long long>() + B + 1 : ws.counters.as<unsigned long long>(),
            (uint32_t)ix->doc_id_base);
    CK(cudaGetLastError());
    L[PB_STAGE_APPROX] += 1;
    return PB_OK;
}

// ---- a6 cut: the top M per query by approximate score; sharded, exchange 1 turns it into this shard's share of the
// global cut ----
static pb_status stage_cut(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const int B = ps.B, M = plan.M, Mcap = plan.Mcap;
    const bool sharded = plan.sharded;
    CKS(ws.kept.ensure((size_t)B * Mcap * 4));
    CKS(ws.nkept.ensure((size_t)B * 4 + 16));
    CKS(ws.tokp.ensure((size_t)B * (Mcap + 1) * 8));
    if (sharded) CKS(ws.lkeys.ensure((size_t)B * Mcap * 8));
    const int Pm = pow2_ceil(Mcap);
    CKS(set_smem(k_cut, (size_t)Pm * 8));
    k_cut<<<B, 1024, (size_t)Pm * 8, ws.stream>>>(ws.keys.as<u64>(), ws.approx.as<float>(), ix->D, ps.cand_n, M,
                                                  Mcap, ix->doc_off.as<long long>(), ws.kept.as<uint32_t>(),
                                                  ws.nkept.as<int>(), ws.tokp.as<long long>(),
                                                  ws.counters.as<long long>() + 1, (uint32_t)ix->doc_id_base,
                                                  sharded ? ws.lkeys.as<u64>() : nullptr);
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_CUT] += 1;
    if (sharded) {
        // exchange 1: every shard's sorted top-M cut keys -> global cut -> my members (SURVEY 8e)
        const int G = ix->world;
        CKS(ws.gkeys.ensure((size_t)G * B * M * 8));
        CKS(ws.krank.ensure((size_t)B * Mcap * 4));
        CKS(shard_allgather(ix, ws.stream, ws.lkeys.p, ws.gkeys.p, (size_t)B * M));
        k_merge_cut<<<B, 1024, 0, ws.stream>>>(ws.gkeys.as<u64>(), G, ix->rank, B, M, (uint32_t)ix->doc_id_base, ix->D,
                                               ix->doc_off.as<long long>(), ws.kept.as<uint32_t>(),
                                               ws.krank.as<uint32_t>(), ws.nkept.as<int>(),
                                               ws.tokp.as<long long>(), ws.counters.as<long long>() + 1);
        CK(cudaGetLastError());
        g_stats.launches[PB_STAGE_CUT] += 2;
    }
    ps.kv = KeptView{ws.kept.as<uint32_t>(), ws.nkept.as<int>(), ws.tokp.as<long long>(),
                     sharded ? ws.krank.as<uint32_t>() : nullptr};
    return PB_OK;
}

// a8 in pair form: pass 2 of the estimate over the filter's survivors lists the (token, q) pairs that can hold a
// per-token maximum, k_pair_exact evaluates them in the pinned order; a query whose list overflows (or that published
// no estimate) goes through k_exact
static pb_status launch_pair_exact(pb_index *ix, Workspace &ws, const CallPlan &plan, const Pass &ps, float eps_unit) {
    const int B = ps.B, QS = ps.QS, Mcap = plan.Mcap;
    const long long max_tokens = (long long)Mcap * std::max(ix->max_doclen, 1);
    const int pair_cap = 16 * Mcap + 4096;  // ~ (top_k + ties) * nq * (1 + a few) pairs per query in practice
    CKS(ws.xpairs.ensure((size_t)B * pair_cap * 8));
    CKS(ws.xnpairs.ensure((size_t)B * 4 + 16));
    CKS(ws.needexact.ensure((size_t)B * 4 + 16));
    CK(cudaMemsetAsync(ws.xnpairs.p, 0, (size_t)B * 4, ws.stream));
    KEV_BEGIN(PB_KERNEL_EXACT);  // pass 2 + pair evaluation + the (normally empty) k_exact of flagged queries
    CKS(launch_maxsim_tc(ix, ws, ps.kv, B, QS, Mcap, max_tokens, ps.nq_max, ws.estkey.as<uint32_t>(),
                         ws.srcrank.as<uint32_t>(), eps_unit, ws.xpairs.as<u64>(), ws.xnpairs.as<int>(), pair_cap, -1));
    k_pair_overflow<<<(B + 255) / 256, 256, 0, ws.stream>>>(ws.xnpairs.as<int>(), pair_cap, ws.qflag.as<int>(), B,
                                                            ws.needexact.as<int>());
    CK(cudaGetLastError());
    const size_t smp = ((size_t)(ps.nq_max + 256) * (ix->dim + 1) + 256) * 4;
    const int pe_ctas = std::max(1, std::min(16, (2 * ix->sm_count + B - 1) / B));  // about one wave over the batch
    PB_TC_DIM_SWITCH(ix->dim, {
        CKS(set_smem(k_pair_exact<DIM>, smp));
        k_pair_exact<DIM><<<dim3(pe_ctas, B), 256, smp, ws.stream>>>(
            ws.xpairs.as<u64>(), ws.xnpairs.as<int>(), pair_cap, ws.Q.as<float>(), ws.qoff.as<int>(), QS,
            ix->centroids.as<float>(), ix->w_rev.as<float>(), ix->nbits, ix->codes.as<uint32_t>(),
            ix->residuals.as<uint8_t>(), Mcap, ws.maxkey.as<uint32_t>());
    });
    CK(cudaGetLastError());
    g_stats.launches[PB_STAGE_EXACT] += 5;
    CKS(launch_exact(ix, ws, ps.kv, B, QS, Mcap, 0, max_tokens, &g_stats.launches[PB_STAGE_EXACT], ws.needexact.as<int>(),
                     false));
    KEV_END(PB_KERNEL_EXACT);
    return PB_OK;
}

// ---- a7 + a8 exact: only the top_k need exact scores, so the certified tensor-core filter drops the kept docs that
// provably cannot reach them; the exact MaxSim of the rest, by pairs or by k_exact ----
static pb_status stage_exact(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const int B = ps.B, QS = ps.QS, Mcap = plan.Mcap;
    const long long max_tokens = (long long)Mcap * std::max(ix->max_doclen, 1);
    int *L = g_stats.launches;
    CKS(ws.maxkey.ensure((size_t)B * Mcap * QS * 4));
    CKS(ws.exact.ensure((size_t)B * Mcap * 4));
    CKS(ws.fkeys.ensure((size_t)B * Mcap * 8));
    // the linear form needs the 16-bit score table of this pass (a flagged query publishes no estimate and keeps
    // every doc); without a table (PB_FAST_APPROX=0) the decompressing form estimates from fp16 centroids
    const bool linear = plan.fast && !ix->filter_v1 && ix->tok_inv_norm.p;
    const float eps_unit = linear ? filter_eps_unit2(ix, ps.tc ? ix->k1_margin : 0) : filter_eps_unit(ix);
    ps.filt = ix->fast_exact && !plan.io->trace && ix->centroids_f16.p && eps_unit > 0.0f && ps.nq_max <= 64 &&
              plan.top_k < Mcap && ix->packed % 4 == 0;
    if (ps.filt) {
        CKS(ws.est.ensure((size_t)B * Mcap * 4));
        CKS(ws.kept2.ensure((size_t)B * Mcap * 4));
        CKS(ws.krank2.ensure((size_t)B * Mcap * 4));
        CKS(ws.nkept2.ensure((size_t)B * 4 + 16));
        CKS(ws.tokp2.ensure((size_t)B * (Mcap + 1) * 8));
        CKS(ws.ktok2.ensure((size_t)B * 8 + 16));
        if (!plan.fast) {  // the two-pass mode computed it with the score range
            CKS(ws.qnmax.ensure((size_t)B * 4 + 16));
            k_query_range<<<B, 256, 0, ws.stream>>>(ws.Q.as<float>(), ws.qoff.as<int>(), ix->dim, ix->cmax, nullptr, nullptr,
                                                    nullptr, ws.qnmax.as<float>());
            CK(cudaGetLastError());
            L[PB_STAGE_EXACT] += 1;
        }
        KeptView kv2{ws.kept2.as<uint32_t>(), ws.nkept2.as<int>(), ws.tokp2.as<long long>(), ws.krank2.as<uint32_t>()};
        ps.pairs = linear && ix->pair_exact && Mcap <= 65535 && QS <= 256;
        if (ps.pairs) {
            CKS(ws.estkey.ensure((size_t)B * Mcap * QS * 4));
            CKS(ws.srcrank.ensure((size_t)B * Mcap * 4));
        }
        CKS(launch_filter(ix, ws, ps.kv, kv2, B, QS, Mcap, plan.top_k, max_tokens, eps_unit, ps.nq_max, linear, ps.pairs,
                          &L[PB_STAGE_EXACT]));
        ps.kv = kv2;
        if (!plan.sharded) ps.kv.krank = nullptr;  // survivors keep their order, so position breaks ties the same way
    }
    if (ps.pairs) CKS(launch_pair_exact(ix, ws, plan, ps, eps_unit));
    else CKS(launch_exact(ix, ws, ps.kv, B, QS, Mcap, 0, max_tokens, &L[PB_STAGE_EXACT]));
    if (plan.sharded) {
        CKS(ws.payload.ensure((size_t)B * Mcap * 8));
        CK(cudaMemsetAsync(ws.fkeys.p, 0xff, (size_t)B * Mcap * 8, ws.stream));  // ~0 = no entry
    }
    k_exact_finalize<<<dim3((Mcap + 7) / 8, B), 256, 0, ws.stream>>>(
        ws.maxkey.as<uint32_t>(), ws.qoff.as<int>(), QS, ps.kv.nkept, Mcap, 0, ws.exact.as<float>(), ws.fkeys.as<u64>(),
        ps.kv.krank, ps.kv.kept, (uint32_t)ix->doc_id_base, plan.sharded ? ws.payload.as<u64>() : nullptr);
    CK(cudaGetLastError());
    L[PB_STAGE_EXACT] += 1;
    return PB_OK;
}

// ---- a9 top-k: into the caller's device arrays at the sub-batch's offset, or into staging for the readback;
// sharded, exchange 2 merges every shard's exact scores ----
static pb_status stage_topk(pb_index *ix, Workspace &ws, const CallPlan &plan, Pass &ps) {
    const SearchIO &io = *plan.io;
    const int B = ps.B, M = plan.M, Mcap = plan.Mcap, top_k = plan.top_k;
    const int Pm = pow2_ceil(Mcap);
    if (io.out_on_device) {
        ps.d_ids = reinterpret_cast<long long *>(io.out_ids) + (size_t)ps.b0 * top_k;
        ps.d_sc = io.out_scores + (size_t)ps.b0 * top_k;
        ps.d_cn = io.out_counts + ps.b0;
    } else {
        CKS(ws.oids.ensure((size_t)B * top_k * 8));
        CKS(ws.oscores.ensure((size_t)B * top_k * 4));
        CKS(ws.ocounts.ensure((size_t)B * 4 + 16));
        ps.d_ids = ws.oids.as<long long>();
        ps.d_sc = ws.oscores.as<float>();
        ps.d_cn = ws.ocounts.as<int>();
    }
    if (plan.sharded) {
        // exchange 2: (exact key | global approx rank) + (doc id | score) of every shard, merged on every rank
        const int G = ix->world;
        CKS(ws.gfkeys.ensure((size_t)G * B * M * 8));
        CKS(ws.gpayload.ensure((size_t)G * B * M * 8));
        CKS(shard_allgather(ix, ws.stream, ws.fkeys.p, ws.gfkeys.p, (size_t)B * M));
        CKS(shard_allgather(ix, ws.stream, ws.payload.p, ws.gpayload.p, (size_t)B * M));
        CKS(ws.mslot.ensure((size_t)B * Mcap * 4));
        CKS(set_smem(k_merge_topk, (size_t)Pm * 8));
        k_merge_topk<<<B, 1024, (size_t)Pm * 8, ws.stream>>>(ws.gfkeys.as<u64>(), ws.gpayload.as<u64>(), G, B, M, top_k,
                                                            ws.mslot.as<uint32_t>(), ps.d_ids, ps.d_sc, ps.d_cn);
        CK(cudaGetLastError());
        g_stats.launches[PB_STAGE_TOPK] += 3;
    } else {
        CKS(set_smem(k_topk, (size_t)Pm * 8));
        k_topk<<<B, 1024, (size_t)Pm * 8, ws.stream>>>(ws.fkeys.as<u64>(), ws.exact.as<float>(), ps.kv.kept, ps.kv.nkept, Mcap,
                                                       top_k, ix->doc_id_base, ps.d_ids, ps.d_sc, ps.d_cn);
        CK(cudaGetLastError());
        g_stats.launches[PB_STAGE_TOPK] += 1;
    }
    return PB_OK;
}

// ---- D2H: the pass's counts and flags into ps.host and, for host outputs, the results into ws.hres ----
static pb_status stage_readback(Workspace &ws, const CallPlan &plan, Pass &ps) {
    const int B = ps.B, top_k = plan.top_k;
    const PassHost &h = ps.host;
    *h.fell = 0;
    CK(cudaMemcpyAsync(h.n_cells, ws.ncells.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    CK(cudaMemcpyAsync(h.n_cand, ws.ncand.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    CK(cudaMemcpyAsync(h.n_kept, ws.nkept.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    CK(cudaMemcpyAsync(h.counters, ws.counters.p, (size_t)(B + 2) * 8, cudaMemcpyDeviceToHost, ws.stream));
    if (ps.filt) {
        CK(cudaMemcpyAsync(h.surv_tokens, ws.ktok2.p, (size_t)B * 8, cudaMemcpyDeviceToHost, ws.stream));
        CK(cudaMemcpyAsync(h.survivors, ws.nkept2.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    }
    if (plan.fast) CK(cudaMemcpyAsync(h.rechecked, ws.ncand2.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    if (ps.pairs) {
        CK(cudaMemcpyAsync(h.pairs, ws.xnpairs.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
        CK(cudaMemcpyAsync(h.need_exact, ws.needexact.p, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    }
    if (ps.d_fallback) CK(cudaMemcpyAsync(h.fell, ps.d_fallback, 4, cudaMemcpyDeviceToHost, ws.stream));
    if (!plan.io->out_on_device) {
        CKS(ws.hres.ensure((size_t)B * top_k * 12 + (size_t)B * 4));
        char *r = ws.hres.as<char>();
        CK(cudaMemcpyAsync(r, ps.d_ids, (size_t)B * top_k * 8, cudaMemcpyDeviceToHost, ws.stream));
        CK(cudaMemcpyAsync(r + (size_t)B * top_k * 8, ps.d_sc, (size_t)B * top_k * 4, cudaMemcpyDeviceToHost, ws.stream));
        CK(cudaMemcpyAsync(r + (size_t)B * top_k * 12, ps.d_cn, (size_t)B * 4, cudaMemcpyDeviceToHost, ws.stream));
    }
    return PB_OK;
}

// ---- the pass's stage and kernel times (profiling) and its work counters, from what the readback brought ----
static pb_status stage_accounting(pb_index *ix, Workspace &ws, const CallPlan &plan, const Pass &ps) {
    const int B = ps.B;
    const PassHost &h = ps.host;
    pb_work_counters &w = g_stats.work;
    if (ix->profiling) {
        for (int s = 0; s < PB_STAGE_COUNT; ++s) {
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, ws.ev[s], ws.ev[s + 1]));
            g_stats.ms[s] += ms;
        }
        for (int k = 0; k < PB_KERNEL_COUNT; ++k)
            if (g_stats.kernel_seen[k]) {
                float ms = 0.f;
                CK(cudaEventElapsedTime(&ms, ws.kev[2 * k], ws.kev[2 * k + 1]));
                g_stats.kernel_ms[k] += ms;
                g_stats.kernel_seen[k] = false;
            }
    }
    if (plan.fast && ix->k1_diag && ws.k1diag.p) {
        int got[2] = {0, 0};
        CK(cudaMemcpy(got, ws.k1diag.p, 8, cudaMemcpyDeviceToHost));
        w.k1_tc_max_code_diff = std::max<long long>(w.k1_tc_max_code_diff, got[0]);
    }
    w.n_queries += B;
    w.n_query_tokens += ps.R;
    switch (ps.probe) {
        case ProbeMode::TensorCore: w.n_k1_tc += 1; break;
        case ProbeMode::Threshold: (*h.fell ? w.n_probe_list : w.n_probe_threshold) += 1; break;
        case ProbeMode::List: w.n_probe_list += 1; break;
        case ProbeMode::AllEligible:
        case ProbeMode::BigProbe: break;
    }
    if (plan.fast)
        for (int b = 0; b < B; ++b) w.n_recheck_docs += h.rechecked[b];
    if (ps.pairs)
        for (int b = 0; b < B; ++b) {
            if (h.need_exact[b]) w.n_pair_fallback_queries += 1;
            else w.n_exact_pairs += h.pairs[b];
        }
    w.n_candidate_tokens += (long long)h.counters[0];
    for (int b = 0; b < B; ++b) {
        w.n_cells += h.n_cells[b];
        w.n_candidates += h.n_cand[b];
        if (ps.filt) {
            w.n_filter_docs += h.n_kept[b];
            w.n_filter_tokens += (long long)h.counters[1 + b];
            w.n_exact_docs += h.survivors[b];
            w.n_exact_tokens += h.surv_tokens[b];
        } else {
            w.n_exact_docs += h.n_kept[b];
            w.n_exact_tokens += (long long)h.counters[1 + b];
        }
    }
    return PB_OK;
}

// ---- the trace of a pass (tests only; synchronous copies) ----
static pb_status stage_trace(pb_index *ix, Workspace &ws, const CallPlan &plan, const Pass &ps) {
    pb_trace *t = plan.io->trace;
    if (!t) return PB_OK;
    const PassHost &h = ps.host;
    for (int b = 0; b < ps.B; ++b) {
        const int64_t gb = ps.b0 + b;
        if (t->n_cells) t->n_cells[gb] = h.n_cells[b];
        if (t->n_candidates) t->n_candidates[gb] = h.n_cand[b];
        if (t->n_kept) t->n_kept[gb] = h.n_kept[b];
        if (t->cells) {
            int n = (int)std::min<int64_t>(h.n_cells[b], t->cells_cap);
            std::vector<uint32_t> tmp(n);
            CK(cudaMemcpy(tmp.data(), ws.cells.as<uint32_t>() + (size_t)b * ps.cells_cap, (size_t)n * 4, cudaMemcpyDeviceToHost));
            for (int i = 0; i < n; ++i) t->cells[gb * t->cells_cap + i] = tmp[i];
        }
        if (t->candidates || t->approx) {
            int n = (int)std::min<int64_t>(h.n_cand[b], t->cand_cap);
            std::vector<uint32_t> tmp(n);
            CK(cudaMemcpy(tmp.data(), ws.cand.as<uint32_t>() + (size_t)b * ix->D, (size_t)n * 4, cudaMemcpyDeviceToHost));
            if (t->candidates)
                for (int i = 0; i < n; ++i) t->candidates[gb * t->cand_cap + i] = (int64_t)tmp[i] + ix->doc_id_base;
            if (t->approx)
                CK(cudaMemcpy(t->approx + gb * t->cand_cap, ws.approx.as<float>() + (size_t)b * ix->D, (size_t)n * 4,
                              cudaMemcpyDeviceToHost));
        }
        if (t->kept || t->kept_exact) {
            int n = (int)std::min<int64_t>(h.n_kept[b], t->kept_cap);
            std::vector<uint32_t> tmp(n);
            CK(cudaMemcpy(tmp.data(), ws.kept.as<uint32_t>() + (size_t)b * plan.Mcap, (size_t)n * 4, cudaMemcpyDeviceToHost));
            if (t->kept)
                for (int i = 0; i < n; ++i) t->kept[gb * t->kept_cap + i] = (int64_t)tmp[i] + ix->doc_id_base;
            if (t->kept_exact)
                CK(cudaMemcpy(t->kept_exact + gb * t->kept_cap, ws.exact.as<float>() + (size_t)b * plan.Mcap, (size_t)n * 4,
                              cudaMemcpyDeviceToHost));
        }
    }
    return PB_OK;
}

// One pass over the sub-batch at b0, stage by stage, with the stage events ws.ev[0..9] between them.  The first pass
// takes the tensor-core path where the call and the sub-batch's rows allow it: a flagged query, a probe-list overflow or
// a re-check overflow raises a device flag instead of being read back mid-way; the pass then finishes on (memory-safe)
// garbage and *redo asks for a second pass, on the exact path.  On a sharded handle every rank votes on its first pass,
// whatever path it takes: the ranks' flags are gathered before the first exchange, so that every rank abandons the
// pass together and the ranks' exchanges stay paired.
static pb_status run_pass(pb_index *ix, Workspace &ws, const CallPlan &plan, int64_t b0, bool first, bool *redo) {
    auto mark = [&](int s) -> pb_status {
        if (ix->profiling) CK(cudaEventRecord(ws.ev[s], ws.stream));
        return PB_OK;
    };
    *redo = false;
    Pass ps;
    ps.b0 = b0;
    CKS(mark(0));
    CKS(stage_h2d(ix, ws, plan, ps));
    CKS(mark(1));
    ps.tc = first && plan.tc_call && ps.QS / 8 <= 32;
    ps.probe = probe_mode(ix, plan, ps.QS, ps.tc);
    CKS(stage_scores(ix, ws, plan, ps));
    CKS(mark(2));
    CKS(stage_probe(ix, ws, plan, ps));
    CKS(mark(3));
    CKS(stage_candidates(ix, ws, plan, ps));
    CKS(mark(4));
    CKS(stage_approx(ix, ws, plan, ps));
    CKS(mark(5));
    if (first && plan.sharded) {
        // The probe flags are the same on every rank (a2/a3 are replicated), a re-check overflow is not: it depends
        // on this shard's documents.  Nor is the path: a rank without tensor-core operands (a shard with no tokens)
        // or with other settings runs the exact pass and votes 0.  Every rank's flag word is gathered here, before
        // exchange 1, and the pass is abandoned on all ranks if any rank raised it; a lone redo would pair its
        // exchanges with the peers' next ones.  The kernels so far have restored their scratch invariants
        // (bitmaps, re-check maxima).
        const u64 *all = nullptr;
        CKS(shard_vote(ix, ws, 0, ps.tc ? ps.d_fallback : nullptr, &all));
        u64 any = 0;
        for (int g = 0; g < ix->world; ++g) any |= all[g];
        if (any) {
            *redo = true;
            return PB_OK;
        }
    }
    CKS(stage_cut(ix, ws, plan, ps));
    CKS(mark(6));
    CKS(stage_exact(ix, ws, plan, ps));
    CKS(mark(7));
    CKS(stage_topk(ix, ws, plan, ps));
    CKS(mark(8));
    CKS(stage_readback(ws, plan, ps));
    CKS(mark(9));
    CK(cudaStreamSynchronize(ws.stream));
    if (ps.tc && *ps.host.fell) {  // the tensor-core pass gave up on the device: same sub-batch again on the exact path
        *redo = true;
        return PB_OK;
    }
    const SearchIO &io = *plan.io;
    if (!io.out_on_device) {
        const size_t n = (size_t)ps.B * plan.top_k;
        const char *r = ws.hres.as<char>();
        memcpy(io.out_ids + (size_t)ps.b0 * plan.top_k, r, n * 8);
        memcpy(io.out_scores + (size_t)ps.b0 * plan.top_k, r + n * 8, n * 4);
        memcpy(io.out_counts + ps.b0, r + n * 12, (size_t)ps.B * 4);
    }
    CKS(stage_accounting(ix, ws, plan, ps));
    return stage_trace(ix, ws, plan, ps);
}

// `lanes`: how many slices of the caller's batch run concurrently (search_impl); they share the workspace budget
static pb_status search_impl_inner(pb_index *ix, const pb_search_params *p, const SearchIO &io, int lanes) {
    WorkspaceLease lease{ix};
    CallPlan plan;
    CKS(plan_call(ix, p, io, lanes, lease, plan));
    if (plan.Bt == 0) return PB_OK;
    Workspace &ws = *lease.ws;
    if (plan.empty) {
        if (io.out_on_device) CK(cudaMemsetAsync(io.out_counts, 0, (size_t)plan.Bt * 4, ws.stream));
        else memset(io.out_counts, 0, (size_t)plan.Bt * 4);
        CK(cudaStreamSynchronize(ws.stream));
        lease.done = true;
        return PB_OK;
    }
    const bool prof = ix->profiling;
    if (prof) CK(cudaEventRecord(ws.call_ev[0], ws.stream));
    for (int64_t b0 = 0; b0 < plan.Bt; b0 += plan.QB) {
        bool redo = false;
        CKS(run_pass(ix, ws, plan, b0, true, &redo));
        if (redo) {
            g_stats.work.n_k1_tc_redo += 1;
            CKS(run_pass(ix, ws, plan, b0, false, &redo));
        }
    }
    if (prof) {
        CK(cudaEventRecord(ws.call_ev[1], ws.stream));
        CK(cudaEventSynchronize(ws.call_ev[1]));
        CK(cudaEventElapsedTime(&g_stats.call_ms, ws.call_ev[0], ws.call_ev[1]));
    }
    lease.done = true;
    return PB_OK;
}

static void merge_stats(Stats &a, const Stats &b) {
    for (int i = 0; i < PB_STAGE_COUNT; ++i) {
        a.ms[i] += b.ms[i];
        a.launches[i] += b.launches[i];
    }
    for (int i = 0; i < PB_KERNEL_COUNT; ++i) a.kernel_ms[i] += b.kernel_ms[i];
    const int64_t *src = reinterpret_cast<const int64_t *>(&b.work);
    int64_t *dst = reinterpret_cast<int64_t *>(&a.work);
    const size_t kdiff = offsetof(pb_work_counters, k1_tc_max_code_diff) / 8;
    for (size_t i = 0; i < sizeof(pb_work_counters) / 8; ++i) dst[i] = i == kdiff ? std::max(dst[i], src[i]) : dst[i] + src[i];
}

// events of the calling thread around a laned call (the lanes' own call events live on different streams)
struct LaneClock {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2] = {};
    int device = -1;
};
static thread_local LaneClock g_lane_clock;

static pb_status search_impl(pb_index *ix, const pb_search_params *p, const SearchIO &io) {
    // Lanes: the queries of a batch are independent, so the batch is cut into `lanes` slices searched concurrently, each
    // through the whole pipeline on its own workspace and stream (helper threads do the launching).  Not with a trace
    // (per-stage dumps), not doc-sharded (the exchanges are collective calls in batch order), not for small batches.
    int lanes = 1;
    if (ix && p && ix->lanes > 1 && !io.trace && ix->world == 1 && io.n_queries >= 16)
        lanes = (int)std::min<int64_t>(ix->lanes, io.n_queries / 8);
    std::unique_lock<std::mutex> lane_lock;
    if (lanes > 1) {
        lane_lock = std::unique_lock<std::mutex>(ix->lane_mu, std::try_to_lock);
        if (!lane_lock.owns_lock()) lanes = 1;  // another host thread is using the helpers: it already provides the overlap
    }
    if (lanes <= 1) {
        const pb_status st = search_impl_inner(ix, p, io, 1);
        if (st != PB_OK && ix && ix->group) ix->group->fail();  // the peers must not wait for a rank that gave up
        return st;
    }
    while ((int)ix->lane_workers.size() < lanes - 1) ix->lane_workers.emplace_back(new LaneWorker());
    const bool prof = ix->profiling;
    LaneClock &clk = g_lane_clock;
    if (prof) {
        CK(cudaSetDevice(ix->device));
        if (clk.device != ix->device) {
            CK(cudaStreamCreateWithFlags(&clk.stream, cudaStreamNonBlocking));
            CK(cudaEventCreate(&clk.ev[0]));
            CK(cudaEventCreate(&clk.ev[1]));
            clk.device = ix->device;
        }
        CK(cudaEventRecord(clk.ev[0], clk.stream));
    }
    std::vector<SearchIO> ios(lanes, io);
    std::vector<pb_status> sts(lanes, PB_OK);
    std::vector<Stats> stats(lanes);
    std::vector<std::string> errs(lanes);
    const int64_t Bt = io.n_queries, top_k = p->top_k;
    for (int l = 0; l < lanes; ++l) {
        const int64_t b0 = Bt * l / lanes, b1 = Bt * (l + 1) / lanes;
        ios[l].q_off = io.q_off + b0;
        ios[l].n_queries = b1 - b0;
        if (io.out_ids) ios[l].out_ids = io.out_ids + b0 * top_k;
        if (io.out_scores) ios[l].out_scores = io.out_scores + b0 * top_k;
        ios[l].out_counts = io.out_counts ? io.out_counts + b0 : nullptr;
    }
    auto run_lane = [&](int l) {
        sts[l] = search_impl_inner(ix, p, ios[l], lanes);
        stats[l] = g_stats;
        if (sts[l] != PB_OK) errs[l] = g_err;
    };
    for (int l = 1; l < lanes; ++l) ix->lane_workers[l - 1]->submit([&, l] { run_lane(l); });
    run_lane(0);
    for (int l = 1; l < lanes; ++l) ix->lane_workers[l - 1]->wait();
    Stats total = stats[0];
    for (int l = 1; l < lanes; ++l) merge_stats(total, stats[l]);
    total.call_ms = 0.f;
    for (int l = 0; l < lanes; ++l) total.call_ms = std::max(total.call_ms, stats[l].call_ms);
    if (prof) {
        CK(cudaEventRecord(clk.ev[1], clk.stream));
        CK(cudaEventSynchronize(clk.ev[1]));
        CK(cudaEventElapsedTime(&total.call_ms, clk.ev[0], clk.ev[1]));
    }
    g_stats = total;
    for (int l = 0; l < lanes; ++l)
        if (sts[l] != PB_OK) {
            g_err = errs[l];
            return sts[l];
        }
    return PB_OK;
}

extern "C" pb_status pb_search_batch_traced(pb_index *ix, const float *queries, const int64_t *q_tok_offsets,
                                            int64_t n_queries, const pb_search_params *params, const int64_t *subset,
                                            int64_t n_subset, int64_t *out_ids, float *out_scores, int32_t *out_counts,
                                            pb_trace *trace) {
    SearchIO io{queries, false, q_tok_offsets, n_queries, subset, subset ? n_subset : 0, subset != nullptr,
                out_ids, out_scores, out_counts, false, trace};
    return search_impl(ix, params, io);
}

extern "C" pb_status pb_search_batch(pb_index *ix, const float *queries, const int64_t *q_tok_offsets, int64_t n_queries,
                                     const pb_search_params *params, const int64_t *subset, int64_t n_subset,
                                     int64_t *out_ids, float *out_scores, int32_t *out_counts) {
    return pb_search_batch_traced(ix, queries, q_tok_offsets, n_queries, params, subset, n_subset, out_ids, out_scores,
                                  out_counts, nullptr);
}

extern "C" pb_status pb_search_batch_device(pb_index *ix, const float *d_queries, const int64_t *q_tok_offsets_host,
                                            int64_t n_queries, const pb_search_params *params, int64_t *d_out_ids,
                                            float *d_out_scores, int32_t *d_out_counts) {
    SearchIO io{d_queries, true, q_tok_offsets_host, n_queries, nullptr, 0, false,
                d_out_ids, d_out_scores, d_out_counts, true, nullptr};
    return search_impl(ix, params, io);
}

// ------------------------------------------------------------------------------------------
// stage entry points
// ------------------------------------------------------------------------------------------
extern "C" pb_status pb_centroid_scores(pb_index *ix, const float *query_tokens, int64_t n, float *out) {
    if (!ix || (!query_tokens && n) || (!out && n)) return pb_fail(PB_ERR_INVALID, "null argument");
    if (n == 0) return PB_OK;
    CK(cudaSetDevice(ix->device));
    WorkspaceLease lease{ix};
    CKS(lease.acquire());
    Workspace &ws = *lease.ws;
    // one pseudo-query per block of <= 64 tokens keeps the per-query transposed layout small
    const int blk = 64;
    DevBuf S;
    CKS(S.ensure((size_t)blk * ix->K * 4));
    for (int64_t r0 = 0; r0 < n; r0 += blk) {
        int nq = (int)std::min<int64_t>(blk, n - r0);
        int QS = std::max(8, (nq + 7) & ~7);
        CKS(ws.Q.ensure((size_t)nq * ix->dim * 4));
        CKS(ws.qoff.ensure(8));
        int qoff[2] = {0, nq};
        CK(cudaMemcpyAsync(ws.Q.p, query_tokens + (size_t)r0 * ix->dim, (size_t)nq * ix->dim * 4, cudaMemcpyHostToDevice, ws.stream));
        CK(cudaMemcpyAsync(ws.qoff.p, qoff, 8, cudaMemcpyHostToDevice, ws.stream));
        CKS(ws.ST.ensure((size_t)ix->K * QS * 4));
        CKS(launch_centroid_scores(ix, ws, 1, QS, nullptr, false));
        k_transpose_scores<<<(unsigned)((ix->K + 255) / 256), 256, 0, ws.stream>>>(ws.ST.as<float>(), ix->K, QS, nq, S.as<float>());
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out + (size_t)r0 * ix->K, S.p, (size_t)nq * ix->K * 4, cudaMemcpyDeviceToHost, ws.stream));
        CK(cudaStreamSynchronize(ws.stream));
    }
    lease.done = true;
    return PB_OK;
}

extern "C" pb_status pb_decompress_documents(pb_index *ix, const int64_t *doc_ids, int64_t n_docs, float *out_embeddings,
                                             int64_t *out_lengths) {
    if (!ix || (!doc_ids && n_docs) || !out_lengths) return pb_fail(PB_ERR_INVALID, "null argument");
    CK(cudaSetDevice(ix->device));
    if (n_docs == 0) return PB_OK;
    std::vector<long long> doff((size_t)ix->D + 1);
    CK(cudaMemcpy(doff.data(), ix->doc_off.p, doff.size() * 8, cudaMemcpyDeviceToHost));
    std::vector<uint32_t> docs;
    std::vector<long long> prefix(1, 0);
    for (int64_t i = 0; i < n_docs; ++i) {
        int64_t d = doc_ids[i] - ix->doc_id_base;
        if (d < 0 || d >= ix->D) {  // index.rs:1202-1204: unknown id -> length 0
            out_lengths[i] = 0;
            continue;
        }
        out_lengths[i] = doff[d + 1] - doff[d];
        docs.push_back((uint32_t)d);
        prefix.push_back(prefix.back() + out_lengths[i]);
    }
    if (!out_embeddings || docs.empty() || prefix.back() == 0) return PB_OK;
    const long long total = prefix.back();
    DevBuf ddocs, dpre, dout;
    CKS(upload(ddocs, docs.data(), docs.size() * 4, PB_MEM_HOST));
    CKS(upload(dpre, prefix.data(), prefix.size() * 8, PB_MEM_HOST));
    const long long chunk_tok = 1ll << 22;  // bound the staging buffer (2 GiB at dim 128)
    CKS(dout.ensure((size_t)std::min(total, chunk_tok + ix->max_doclen) * ix->dim * 4));
    // process doc ranges whose token count fits the staging buffer
    size_t i0 = 0;
    while (i0 < docs.size()) {
        size_t i1 = i0;
        while (i1 < docs.size() && prefix[i1] - prefix[i0] < chunk_tok) ++i1;  // <= chunk_tok + max_doclen tokens
        const int nd = (int)(i1 - i0);
        const long long ntok = prefix[i1] - prefix[i0];
        std::vector<long long> local(nd + 1);
        for (int j = 0; j <= nd; ++j) local[j] = prefix[i0 + j] - prefix[i0];
        CK(cudaMemcpy(dpre.p, local.data(), local.size() * 8, cudaMemcpyHostToDevice));
        int blocks = (int)std::max<long long>(1, std::min<long long>((ntok + 7) / 8, (long long)ix->sm_count * 8));
        PB_DIM_SWITCH(ix->dim, {
            k_decompress<DIM><<<blocks, 256>>>(ix->centroids.as<float>(), ix->w_rev.as<float>(), ix->nbits,
                                               ix->codes.as<uint32_t>(), ix->residuals.as<uint8_t>(),
                                               ix->doc_off.as<long long>(), ddocs.as<uint32_t>() + i0, dpre.as<long long>(),
                                               nd, dout.as<float>());
        });
        CK(cudaGetLastError());
        CK(cudaMemcpy(out_embeddings + (size_t)prefix[i0] * ix->dim, dout.p, (size_t)ntok * ix->dim * 4, cudaMemcpyDeviceToHost));
        i0 = i1;
    }
    return PB_OK;
}

extern "C" pb_status pb_maxsim_scores(int32_t device, const float *query, int32_t nq, int32_t dim, const float *doc_tokens,
                                      const int64_t *doc_tok_offsets, int64_t n_docs, float *out_scores) {
    if ((!query && nq) || (!doc_tok_offsets) || (!out_scores && n_docs)) return pb_fail(PB_ERR_INVALID, "null argument");
    if (!dim_supported(dim)) return pb_fail(PB_ERR_UNSUPPORTED, "embedding_dim %d not built (32/64/96/128/256)", dim);
    if (nq < 0 || n_docs < 0) return pb_fail(PB_ERR_INVALID, "negative size");
    CKS(check_device(device));
    if (n_docs == 0) return PB_OK;
    if (n_docs > (1 << 30)) return pb_fail(PB_ERR_UNSUPPORTED, "too many documents in one call");
    const long long total = doc_tok_offsets[n_docs] - doc_tok_offsets[0];
    const int QS = std::max(8, (nq + 7) & ~7);
    const int Mcap = (int)n_docs;
    DevBuf dQ, dqoff, dtok, dkept, dnk, dtp, dmax, dex;
    dmax.zero_on_grow = true;
    int qoff[2] = {0, nq};
    std::vector<long long> tp(n_docs + 1);
    for (int64_t i = 0; i <= n_docs; ++i) tp[i] = doc_tok_offsets[i] - doc_tok_offsets[0];
    CKS(upload(dQ, query, (size_t)nq * dim * 4, PB_MEM_HOST));
    CKS(upload(dqoff, qoff, 8, PB_MEM_HOST));
    CKS(upload(dtok, doc_tokens + (size_t)doc_tok_offsets[0] * dim, (size_t)total * dim * 4, PB_MEM_HOST));
    CKS(upload(dtp, tp.data(), tp.size() * 8, PB_MEM_HOST));
    CKS(upload(dnk, &Mcap, 4, PB_MEM_HOST));
    CKS(dkept.ensure((size_t)Mcap * 4));
    CKS(dmax.ensure((size_t)Mcap * QS * 4));
    CKS(dex.ensure((size_t)Mcap * 4));
    long long chunks = (total + PB_TOK_TILE - 1) / PB_TOK_TILE;
    int gx = (int)std::max<long long>(1, std::min<long long>(chunks, 148ll * 16));
    PB_DIM_SWITCH(dim, {
        auto kern = k_exact<DIM, true>;
        CKS(set_smem(kern, smem_exact(DIM, 0)));
        kern<<<dim3(gx, 1), 128, smem_exact(DIM, 0)>>>(dQ.as<float>(), dqoff.as<int>(), QS, nullptr, nullptr, 8, nullptr,
                                                    nullptr, nullptr, dtok.as<float>(), dkept.as<uint32_t>(),
                                                    dnk.as<int>(), dtp.as<long long>(), Mcap, 0, dmax.as<uint32_t>(), nullptr);
    });
    CK(cudaGetLastError());
    k_exact_finalize<<<dim3((Mcap + 7) / 8, 1), 256>>>(dmax.as<uint32_t>(), dqoff.as<int>(), QS, dnk.as<int>(), Mcap, 0,
                                                      dex.as<float>(), nullptr, nullptr, nullptr, 0u, nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out_scores, dex.p, (size_t)Mcap * 4, cudaMemcpyDeviceToHost));
    return PB_OK;
}

extern "C" pb_status pb_exhaustive_scores(pb_index *ix, const float *queries, const int64_t *q_off, int64_t n_queries,
                                          float *out_scores) {
    if (!ix || (!queries && n_queries) || !q_off || (!out_scores && n_queries)) return pb_fail(PB_ERR_INVALID, "null argument");
    CK(cudaSetDevice(ix->device));
    if (n_queries == 0 || ix->D == 0) return PB_OK;
    WorkspaceLease lease{ix};
    CKS(lease.acquire());
    Workspace &ws = *lease.ws;
    std::vector<long long> doff((size_t)ix->D + 1);
    CK(cudaMemcpy(doff.data(), ix->doc_off.p, doff.size() * 8, cudaMemcpyDeviceToHost));
    const int QBmax = 32;
    const int Mblk = 1 << 16;
    for (int64_t b0 = 0; b0 < n_queries; b0 += QBmax) {
        const int B = (int)std::min<int64_t>(QBmax, n_queries - b0);
        const int64_t r0 = q_off[b0], R = q_off[b0 + B] - r0;
        std::vector<int> qoff(B + 1);
        int nq_max = 0;
        for (int b = 0; b <= B; ++b) qoff[b] = (int)(q_off[b0 + b] - r0);
        for (int b = 0; b < B; ++b) nq_max = std::max(nq_max, qoff[b + 1] - qoff[b]);
        const int QS = std::max(8, (nq_max + 7) & ~7);
        CKS(ws.Q.ensure(std::max<size_t>((size_t)R * ix->dim * 4, 16)));
        CKS(ws.qoff.ensure((size_t)(B + 1) * 4));
        if (R) CK(cudaMemcpyAsync(ws.Q.p, queries + (size_t)r0 * ix->dim, (size_t)R * ix->dim * 4, cudaMemcpyHostToDevice, ws.stream));
        CK(cudaMemcpyAsync(ws.qoff.p, qoff.data(), (size_t)(B + 1) * 4, cudaMemcpyHostToDevice, ws.stream));
        CK(cudaStreamSynchronize(ws.stream));
        CKS(ws.kept.ensure((size_t)Mblk * 4));
        CKS(ws.nkept.ensure(16));
        CKS(ws.tokp.ensure((size_t)(Mblk + 1) * 8));
        CKS(ws.maxkey.ensure((size_t)B * Mblk * QS * 4));
        CKS(ws.exact.ensure((size_t)B * Mblk * 4));
        // maxkey layout changes with QS/Mcap: rows are reset by finalize, but only those < n_kept
        for (long long d0 = 0; d0 < ix->D; d0 += Mblk) {
            const int nd = (int)std::min<long long>(Mblk, ix->D - d0);
            k_fill_identity<<<64, 256, 0, ws.stream>>>(ws.kept.as<uint32_t>(), nd, (uint32_t)d0);
            k_range_prefix<<<64, 256, 0, ws.stream>>>(ix->doc_off.as<long long>(), d0, nd, ws.tokp.as<long long>());
            CK(cudaMemcpyAsync(ws.nkept.p, &nd, 4, cudaMemcpyHostToDevice, ws.stream));
            const KeptView kv{ws.kept.as<uint32_t>(), ws.nkept.as<int>(), ws.tokp.as<long long>(), nullptr};
            CKS(launch_exact(ix, ws, kv, B, QS, Mblk, 1, doff[d0 + nd] - doff[d0], nullptr));
            k_exact_finalize<<<dim3((Mblk + 7) / 8, B), 256, 0, ws.stream>>>(ws.maxkey.as<uint32_t>(), ws.qoff.as<int>(), QS,
                                                                           ws.nkept.as<int>(), Mblk, 1, ws.exact.as<float>(),
                                                                           nullptr, nullptr, nullptr, 0u, nullptr);
            CK(cudaGetLastError());
            for (int b = 0; b < B; ++b)
                CK(cudaMemcpyAsync(out_scores + (size_t)(b0 + b) * ix->D + d0, ws.exact.as<float>() + (size_t)b * Mblk,
                                   (size_t)nd * 4, cudaMemcpyDeviceToHost, ws.stream));
            CK(cudaStreamSynchronize(ws.stream));
        }
    }
    lease.done = true;
    return PB_OK;
}


// ------------------------------------------------------------------------------------------
// doc-sharded deployment: one process per GPU, NCCL all-gathers of the per-shard top lists.
// The host passes the 128-byte NCCL unique id between ranks however it likes (torch.distributed,
// MPI, a file); nothing else crosses the C-ABI.
// ------------------------------------------------------------------------------------------
extern "C" pb_status pb_comm_unique_id(uint8_t *out128) {
    if (!out128) return pb_fail(PB_ERR_INVALID, "null argument");
    if (!g_nccl.load()) return pb_fail(PB_ERR_COMM, "libnccl.so.2 not found (%s)", dlerror());
    ncclUniqueId id;
    CKN(g_nccl.GetUniqueId(&id));
    memcpy(out128, id.internal, 128);
    return PB_OK;
}

extern "C" pb_status pb_index_comm_init(pb_index *ix, const uint8_t *id128, int32_t rank, int32_t world) {
    if (!ix || !id128) return pb_fail(PB_ERR_INVALID, "null argument");
    if (world < 1 || rank < 0 || rank >= world) return pb_fail(PB_ERR_INVALID, "bad rank %d / world %d", rank, world);
    if (ix->comm) return pb_fail(PB_ERR_INVALID, "communicator already initialised");
    if (world == 1) return PB_OK;
    if (!g_nccl.load()) return pb_fail(PB_ERR_COMM, "libnccl.so.2 not found (%s)", dlerror());
    CK(cudaSetDevice(ix->device));
    ncclUniqueId id;
    memcpy(id.internal, id128, 128);
    CKN(g_nccl.CommInitRank(&ix->comm, world, id, rank));
    ix->rank = rank;
    ix->world = world;
    return PB_OK;
}

// In-process alternative to NCCL: one handle per shard, one host thread per handle (any devices, peer copies)
extern "C" pb_status pb_shard_group_create(int32_t world, pb_shard_group **out) {
    if (!out || world < 1 || world > 64) return pb_fail(PB_ERR_INVALID, "shard group: world must be in [1, 64]");
    pb_shard_group *g = new pb_shard_group();
    g->world = world;
    g->send.assign((size_t)world, nullptr);
    g->dev.assign((size_t)world, 0);
    *out = g;
    return PB_OK;
}
extern "C" void pb_shard_group_destroy(pb_shard_group *g) { delete g; }
extern "C" pb_status pb_index_group_join(pb_index *ix, pb_shard_group *g, int32_t rank) {
    if (!ix || !g) return pb_fail(PB_ERR_INVALID, "null argument");
    if (rank < 0 || rank >= g->world) return pb_fail(PB_ERR_INVALID, "bad rank %d / world %d", rank, g->world);
    if (ix->comm || ix->group) return pb_fail(PB_ERR_INVALID, "communicator already initialised");
    std::lock_guard<std::mutex> lk(g->mu);
    g->dev[rank] = ix->device;
    ++g->joined;
    ix->group = g;
    ix->rank = rank;
    ix->world = g->world;
    return PB_OK;
}

// ------------------------------------------------------------------------------------------
// index-build path (SURVEY 8 a12, secondary): ResidualCodec on the device
// ------------------------------------------------------------------------------------------
struct pb_codec {
    int device = 0, dim = 0, nbits = 0, sm_count = 148;
    long long K = 0;
    DevBuf centroids, cutoffs, cent_bf16, cent_norm;
    bool has_cutoffs = false;
    bool use_tc = false;   // tcgen05 certified filter in front of the exact assignment
    float cmax = 0.f;
    int c_finite = 1;
    long long last_tokens = 0, last_fallback = 0;
};

static size_t smem_assign_tc(int dim) {
    return (size_t)2 * PB_TC_M * dim * 2 + (size_t)PB_TC_STAGES * PB_TC_N * dim * 2 + (2 * PB_TC_STAGES + 5) * 8 + 16;
}

static size_t smem_assign(int dim) { return (size_t)((dim <= 128 ? 2 : 1) * PB_TOK_TILE + 64) * (dim + 4) * sizeof(float); }

static pb_status launch_assign(int dim, int sm_count, const float *dX, long long n, const float *dC, long long K,
                               const float *bias, long long *codes64, uint32_t *codes32, cudaStream_t st) {
    if (n == 0) return PB_OK;
    (void)sm_count;
    const unsigned blocks = (unsigned)((n + 63) / 64);
    PB_DIM_SWITCH(dim, {
        auto kern = k_assign<DIM>;
        CKS(set_smem(kern, smem_assign(DIM)));
        kern<<<blocks, 256, smem_assign(DIM), st>>>(dX, n, dC, K, bias, codes64, codes32);
    });
    CK(cudaGetLastError());
    return PB_OK;
}

extern "C" pb_status pb_codec_open(int32_t device, const float *centroids, int64_t K, int32_t dim, int32_t nbits,
                                   const float *bucket_cutoffs, pb_codec **out) {
    if (!centroids || !out) return pb_fail(PB_ERR_INVALID, "null argument");
    *out = nullptr;
    if (nbits <= 0 || 8 % nbits != 0) return pb_fail(PB_ERR_INVALID, "nbits must be a divisor of 8, got %d", nbits);
    if (K <= 0 || K >= (1ll << 32) - 1) return pb_fail(PB_ERR_INVALID, "bad num_centroids %lld", (long long)K);
    if (!dim_supported(dim)) return pb_fail(PB_ERR_UNSUPPORTED, "embedding_dim %d not built (32/64/96/128/256)", dim);
    CKS(check_device(device));
    std::unique_ptr<pb_codec> c(new pb_codec());
    c->device = device;
    c->dim = dim;
    c->nbits = nbits;
    c->K = K;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    CKS(upload(c->centroids, centroids, (size_t)K * dim * 4, PB_MEM_HOST));
    if (bucket_cutoffs) {
        CKS(upload(c->cutoffs, bucket_cutoffs, (size_t)((1 << nbits) - 1) * 4, PB_MEM_HOST));
        c->has_cutoffs = true;
    }
    // tensor-core filter: fp16 copy of the centroids (tile order), their largest norm, finiteness
    c->use_tc = (dim == 64 || dim == 96 || dim == 128) && K >= 256 && !getenv("PB_ASSIGN_EXACT") &&
                smem_assign_tc(dim) <= 227 * 1024;
    if (c->use_tc) {
        const size_t kpad = (size_t)((K + 127) / 128) * 128;  // tile order, zero padded
        CKS(c->cent_bf16.ensure(kpad * dim * 2));
        CK(cudaMemset(c->cent_bf16.p, 0, kpad * dim * 2));
        CKS(c->cent_norm.ensure((size_t)K * 4));
        k_rows_to_bf16<<<c->sm_count * 8, 256>>>(c->centroids.as<float>(), K, dim, c->cent_bf16.as<__nv_bfloat16>(),
                                                 c->cent_norm.as<float>());
        CK(cudaGetLastError());
        std::vector<float> nr((size_t)K);
        CK(cudaMemcpy(nr.data(), c->cent_norm.p, (size_t)K * 4, cudaMemcpyDeviceToHost));
        float mx = 0.f;
        for (float v : nr) {
            if (!(v < 1e18f)) c->c_finite = 0;
            else mx = std::max(mx, v);
        }
        c->cmax = mx;
    }
    *out = c.release();
    return PB_OK;
}

extern "C" pb_status pb_codec_last_assign_stats(pb_codec *c, int64_t *n_tokens, int64_t *n_exact_fallback, int32_t *used_tensor_cores) {
    if (!c) return pb_fail(PB_ERR_INVALID, "null argument");
    if (n_tokens) *n_tokens = c->last_tokens;
    if (n_exact_fallback) *n_exact_fallback = c->last_fallback;
    if (used_tensor_cores) *used_tensor_cores = c->use_tc ? 1 : 0;
    return PB_OK;
}

// nearest-centroid codes of m device-resident rows: tensor-core shortlist + certified exact re-score,
// exact kernel for whatever cannot be certified
static pb_status assign_codes(pb_codec *c, const float *dX, long long m, long long *dcodes) {
    if (!c->use_tc) {
        c->last_fallback += m;
        return launch_assign(c->dim, c->sm_count, dX, m, c->centroids.as<float>(), c->K, nullptr, dcodes, nullptr, 0);
    }
    DevBuf xb, xn, ts, ti, nfb, fl;
    const size_t mpad = (size_t)((m + 255) / 256) * 256;  // two 128-token tiles per CTA, zero padded
    CKS(xb.ensure(mpad * c->dim * 2));
    CK(cudaMemset(xb.p, 0, mpad * c->dim * 2));
    CKS(xn.ensure((size_t)m * 4));
    CKS(ts.ensure((size_t)m * 16));
    CKS(ti.ensure((size_t)m * 16));
    CKS(nfb.ensure(16));
    CKS(fl.ensure((size_t)m * 8));
    CK(cudaMemset(nfb.p, 0, 4));
    k_rows_to_bf16<<<c->sm_count * 8, 256>>>(dX, m, c->dim, xb.as<__nv_bfloat16>(), xn.as<float>());
    const unsigned blocks = (unsigned)((m + 2 * PB_TC_M - 1) / (2 * PB_TC_M));
    const size_t sm = smem_assign_tc(c->dim);
    switch (c->dim) {
#define PB_TC_CASE(DV)                                                                                     \
    case DV: {                                                                                             \
        auto kern = k_assign_tc<DV, false>;                                                                \
        CKS(set_smem(kern, sm));                                                                           \
        kern<<<blocks, 320, sm>>>(xb.as<__nv_bfloat16>(), m, c->cent_bf16.as<__nv_bfloat16>(), c->K, ts.as<float>(), \
                                  ti.as<uint32_t>(), nullptr);                                             \
    } break;
        PB_TC_CASE(64) PB_TC_CASE(96) PB_TC_CASE(128)
#undef PB_TC_CASE
        default: return pb_fail(PB_ERR_UNSUPPORTED, "tensor-core assignment not built for dim %d", c->dim);
    }
    CK(cudaGetLastError());
    k_assign_certify<<<c->sm_count * 8, 256>>>(dX, m, c->dim, c->centroids.as<float>(), xn.as<float>(), c->cmax, c->c_finite,
                                               ts.as<float>(), ti.as<uint32_t>(), dcodes, nfb.as<int>(), fl.as<long long>());
    CK(cudaGetLastError());
    int nf = 0;
    CK(cudaMemcpy(&nf, nfb.p, 4, cudaMemcpyDeviceToHost));
    c->last_fallback += nf;
    if (nf > 0) {
        DevBuf gx, gc;
        CKS(gx.ensure((size_t)nf * c->dim * 4));
        CKS(gc.ensure((size_t)nf * 8));
        k_gather_rows_i64<<<c->sm_count * 8, 256>>>(dX, fl.as<long long>(), nf, c->dim, gx.as<float>());
        CKS(launch_assign(c->dim, c->sm_count, gx.as<float>(), nf, c->centroids.as<float>(), c->K, nullptr, gc.as<long long>(),
                          nullptr, 0));
        k_scatter_codes<<<(nf + 255) / 256, 256>>>(gc.as<long long>(), fl.as<long long>(), nf, dcodes);
        CK(cudaGetLastError());
    }
    return PB_OK;
}

extern "C" void pb_codec_close(pb_codec *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    delete c;
}

// embeddings are processed in slabs so the staging buffers stay bounded
static pb_status codec_run(pb_codec *c, const float *emb, int64_t n, int64_t *out_codes, uint8_t *out_packed,
                           float *out_residuals) {
    if (!c || (!emb && n) || n < 0) return pb_fail(PB_ERR_INVALID, "null argument");
    if ((out_packed) && !c->has_cutoffs) return pb_fail(PB_ERR_INVALID, "bucket_cutoffs required for quantization");  // codec.rs:359-362
    CK(cudaSetDevice(c->device));
    if (n == 0) return PB_OK;
    const long long slab = 1ll << 20;
    const int packed = c->dim * c->nbits / 8;
    c->last_tokens = n;
    c->last_fallback = 0;
    DevBuf dX, dcodes, dpk, dres;
    CKS(dX.ensure((size_t)std::min<long long>(n, slab) * c->dim * 4));
    CKS(dcodes.ensure((size_t)std::min<long long>(n, slab) * 8));
    if (out_packed) CKS(dpk.ensure((size_t)std::min<long long>(n, slab) * packed));
    if (out_residuals) CKS(dres.ensure((size_t)std::min<long long>(n, slab) * c->dim * 4));
    for (long long o = 0; o < n; o += slab) {
        const long long m = std::min(slab, n - o);
        CK(cudaMemcpy(dX.p, emb + (size_t)o * c->dim, (size_t)m * c->dim * 4, cudaMemcpyHostToDevice));
        CKS(assign_codes(c, dX.as<float>(), m, dcodes.as<long long>()));
        if (out_packed || out_residuals) {
            PB_DIM_SWITCH(c->dim, {
                k_quantize_pack<DIM><<<c->sm_count * 8, 256>>>(dX.as<float>(), m, c->centroids.as<float>(),
                                                                dcodes.as<long long>(), c->cutoffs.as<float>(), c->nbits,
                                                                out_packed ? dpk.as<uint8_t>() : nullptr,
                                                                out_residuals ? dres.as<float>() : nullptr);
            });
            CK(cudaGetLastError());
        }
        if (out_codes) CK(cudaMemcpy(out_codes + o, dcodes.p, (size_t)m * 8, cudaMemcpyDeviceToHost));
        if (out_packed) CK(cudaMemcpy(out_packed + (size_t)o * packed, dpk.p, (size_t)m * packed, cudaMemcpyDeviceToHost));
        if (out_residuals) CK(cudaMemcpy(out_residuals + (size_t)o * c->dim, dres.p, (size_t)m * c->dim * 4, cudaMemcpyDeviceToHost));
    }
    return PB_OK;
}

extern "C" pb_status pb_codec_compress_into_codes(pb_codec *c, const float *embeddings, int64_t n, int64_t *out_codes) {
    if (!out_codes && n) return pb_fail(PB_ERR_INVALID, "null argument");
    return codec_run(c, embeddings, n, out_codes, nullptr, nullptr);
}

extern "C" pb_status pb_codec_encode_chunk(pb_codec *c, const float *embeddings, int64_t n, int64_t *out_codes,
                                           uint8_t *out_residuals_packed) {
    if ((!out_codes || !out_residuals_packed) && n) return pb_fail(PB_ERR_INVALID, "null argument");
    return codec_run(c, embeddings, n, out_codes, out_residuals_packed, nullptr);
}

extern "C" pb_status pb_codec_compress_and_residuals(pb_codec *c, const float *embeddings, int64_t n, int64_t *out_codes,
                                                     float *out_residuals) {
    if ((!out_codes || !out_residuals) && n) return pb_fail(PB_ERR_INVALID, "null argument");
    // residuals only need the subtraction: run the pack kernel without a packed output
    bool had = c && c->has_cutoffs;
    if (c && !had) {  // the kernel reads ncut cutoffs only when packing; give it a valid (unused) pointer
        float zero[255] = {0};
        CKS(upload(c->cutoffs, zero, sizeof zero, PB_MEM_HOST));
    }
    return codec_run(c, embeddings, n, out_codes, nullptr, out_residuals);
}

// prepare_codec_artifacts' arithmetic (index.rs:228-287) for held-out embeddings the caller selected: residuals of
// the nearest centroid, cluster_threshold = quantile 0.75 of their L2 norms, avg_residual = per-dimension mean of
// |residual|, bucket cutoffs / weights = quantiles of the flattened residuals at i/2^b and (i+1/2)/2^b
// (utils.rs:125-149: sort, position q (n-1) in f64, lo (1-w) + hi w with w cast to f32).  The codec keeps the cutoffs.
static float quantile_pick(const std::vector<float> &sorted_at, const std::vector<long long> &pos, long long n, double q) {
    // sorted_at[i] = sorted[pos[i]]; pos holds floor/ceil positions of every requested quantile in order
    const double idx = q * (double)(n - 1);
    const long long lo = (long long)floor(idx), hi = (long long)ceil(idx);
    float vlo = 0.f, vhi = 0.f;
    for (size_t i = 0; i < pos.size(); ++i) {
        if (pos[i] == lo) vlo = sorted_at[i];
        if (pos[i] == hi) vhi = sorted_at[i];
    }
    if (lo == hi) return vlo;
    const float w = (float)(idx - (double)lo);
    return vlo * (1.0f - w) + vhi * w;
}

static pb_status device_quantiles(DevBuf &vals, long long n, const std::vector<double> &qs, std::vector<float> &out) {
    out.assign(qs.size(), 0.0f);
    if (n == 0) return PB_OK;
    DevBuf sorted, tmp;
    CKS(sorted.ensure((size_t)n * 4));
    size_t tb = 0;
    CK(cub::DeviceRadixSort::SortKeys(nullptr, tb, vals.as<float>(), sorted.as<float>(), (int)n));
    CKS(tmp.ensure(tb + 16));
    CK(cub::DeviceRadixSort::SortKeys(tmp.p, tb, vals.as<float>(), sorted.as<float>(), (int)n));
    std::vector<long long> pos;
    for (double q : qs) {
        const double idx = q * (double)(n - 1);
        pos.push_back((long long)floor(idx));
        pos.push_back((long long)ceil(idx));
    }
    std::vector<float> at(pos.size());
    for (size_t i = 0; i < pos.size(); ++i)
        CK(cudaMemcpy(&at[i], sorted.as<float>() + pos[i], 4, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < qs.size(); ++i) out[i] = quantile_pick(at, pos, n, qs[i]);
    return PB_OK;
}

extern "C" pb_status pb_codec_train(pb_codec *c, const float *heldout, int64_t n, float *out_cutoffs, float *out_weights,
                                    float *out_avg_residual, float *out_cluster_threshold) {
    if (!c || (!heldout && n) || n < 0 || !out_cutoffs || !out_weights) return pb_fail(PB_ERR_INVALID, "null argument");
    if ((long long)n * c->dim >= (1ll << 31)) return pb_fail(PB_ERR_UNSUPPORTED, "held-out sample too large");
    CK(cudaSetDevice(c->device));
    const int nopt = 1 << c->nbits;
    DevBuf dX, dcodes, dres, dnorm, davg;
    CKS(dX.ensure(std::max<size_t>((size_t)n * c->dim * 4, 16)));
    CKS(dcodes.ensure(std::max<size_t>((size_t)n * 8, 16)));
    CKS(dres.ensure(std::max<size_t>((size_t)n * c->dim * 4, 16)));
    CKS(dnorm.ensure(std::max<size_t>((size_t)n * 4, 16)));
    CKS(davg.ensure((size_t)c->dim * 4));
    if (n > 0) {
        CK(cudaMemcpy(dX.p, heldout, (size_t)n * c->dim * 4, cudaMemcpyHostToDevice));
        CKS(assign_codes(c, dX.as<float>(), n, dcodes.as<long long>()));
        if (!c->has_cutoffs) {  // the residual kernel takes a cutoff pointer it does not read without a packed output
            float zero[255] = {0};
            CKS(upload(c->cutoffs, zero, sizeof zero, PB_MEM_HOST));
        }
        PB_DIM_SWITCH(c->dim, {
            k_quantize_pack<DIM><<<c->sm_count * 8, 256>>>(dX.as<float>(), n, c->centroids.as<float>(), dcodes.as<long long>(),
                                                            c->cutoffs.as<float>(), c->nbits, nullptr, dres.as<float>());
        });
        k_residual_stats<<<c->sm_count * 4, 256>>>(dres.as<float>(), n, c->dim, dnorm.as<float>());
        k_column_abs_mean<<<(c->dim + 31) / 32, 32>>>(dres.as<float>(), n, c->dim, davg.as<float>());
        CK(cudaGetLastError());
    }
    std::vector<double> q75{0.75}, qc, qw;
    for (int i = 1; i < nopt; ++i) qc.push_back((double)i / (double)nopt);
    for (int i = 0; i < nopt; ++i) qw.push_back(((double)i + 0.5) / (double)nopt);
    std::vector<float> r75, rc, rw;
    CKS(device_quantiles(dnorm, n, q75, r75));
    CKS(device_quantiles(dres, (long long)n * c->dim, qc, rc));
    CKS(device_quantiles(dres, (long long)n * c->dim, qw, rw));
    for (int i = 0; i < nopt - 1; ++i) out_cutoffs[i] = rc[i];
    for (int i = 0; i < nopt; ++i) out_weights[i] = rw[i];
    if (out_cluster_threshold) *out_cluster_threshold = n ? r75[0] : 0.0f;
    if (out_avg_residual) {
        if (n) CK(cudaMemcpy(out_avg_residual, davg.p, (size_t)c->dim * 4, cudaMemcpyDeviceToHost));
        else memset(out_avg_residual, 0, (size_t)c->dim * 4);
    }
    float cut[255] = {0};
    for (int i = 0; i < nopt - 1; ++i) cut[i] = rc[i];
    CKS(upload(c->cutoffs, cut, sizeof cut, PB_MEM_HOST));
    c->has_cutoffs = true;
    return PB_OK;
}

// compute_kmeans' sizing rules (kmeans.rs:273-312) and prepare_codec_artifacts' (index.rs:195-212), as the host
// side needs them to pick its samples
extern "C" int64_t pb_kmeans_num_sample_docs(int64_t num_documents) {  // min(floor(1 + 16 sqrt(120 D)), D)
    const double v = 1.0 + 16.0 * sqrt(120.0 * (double)num_documents);
    return std::min<int64_t>((int64_t)v, num_documents);
}
extern "C" int64_t pb_kmeans_num_partitions(int64_t num_documents, double avg_sample_doclen, int64_t num_sample_tokens) {
    const double est = avg_sample_doclen * (double)num_documents;  // K = 2^floor(log2(16 sqrt(avg_doclen * D)))
    const double k = pow(2.0, floor(log2(16.0 * sqrt(est))));
    return std::max<int64_t>(1, std::min<int64_t>((int64_t)k, num_sample_tokens));
}
extern "C" int64_t pb_codec_num_sample_docs(int64_t num_documents) {  // clamp(floor(16 sqrt(120 D)), 1, D)
    const int64_t v = (int64_t)(16.0 * sqrt(120.0 * (double)num_documents));
    return std::max<int64_t>(1, std::min<int64_t>(v, num_documents));
}
extern "C" int64_t pb_codec_heldout_tokens(int64_t num_embeddings) {  // min(0.05 N, 50 000)
    return (int64_t)std::min(0.05 * (double)num_embeddings, 50000.0);
}

// k-means assignment step.  dims 64 / 96 / 128 with K >= 256: the fp16 tcgen05 GEMM of the encode path with the
// -|c|^2/2 bias added in its epilogue, best shortlist entry taken as is; otherwise the exact fp32 kernel.
struct KmeansAssign {
    DevBuf xb, cb, bias, ts, ti, scratch;
    bool tc = false;
    long long n = 0, K = 0;
    int dim = 0, sms = 0;
    pb_status init(const float *dX, long long n_, int dim_, long long K_, int sms_, cudaStream_t st) {
        n = n_; K = K_; dim = dim_; sms = sms_;
        tc = (dim == 64 || dim == 96 || dim == 128) && K >= 256 && n > 0 && !getenv("PB_KMEANS_EXACT");
        if (!tc) return PB_OK;
        const size_t npad = (size_t)((n + 255) / 256) * 256, kpad = (size_t)((K + 127) / 128) * 128;
        CKS(xb.ensure(npad * dim * 2));
        CKS(cb.ensure(kpad * dim * 2));
        CKS(bias.ensure(kpad * 4));
        CKS(ts.ensure((size_t)n * 16));
        CKS(ti.ensure((size_t)n * 16));
        CKS(scratch.ensure(std::max<size_t>((size_t)std::max(n, K) * 4, 16)));
        CK(cudaMemsetAsync(xb.p, 0, npad * dim * 2, st));
        k_rows_to_bf16<<<sms * 8, 256, 0, st>>>(dX, n, dim, xb.as<__nv_bfloat16>(), scratch.as<float>());
        CK(cudaGetLastError());
        return PB_OK;
    }
    pb_status run(const float *dX, const float *dC, float *dbias_exact, uint32_t *codes, cudaStream_t st) {
        if (!tc) {
            k_half_sqnorm<<<sms * 4, 256, 0, st>>>(dC, K, dim, dbias_exact);
            return launch_assign(dim, sms, dX, n, dC, K, dbias_exact, nullptr, codes, st);
        }
        const size_t kpad = (size_t)((K + 127) / 128) * 128;
        CK(cudaMemsetAsync(cb.p, 0, kpad * dim * 2, st));
        k_rows_to_bf16<<<sms * 8, 256, 0, st>>>(dC, K, dim, cb.as<__nv_bfloat16>(), scratch.as<float>());
        k_half_sqnorm_padded<<<sms * 4, 256, 0, st>>>(dC, K, (long long)kpad, dim, bias.as<float>());
        const unsigned blocks = (unsigned)((n + 2 * PB_TC_M - 1) / (2 * PB_TC_M));
        const size_t sm = (size_t)2 * PB_TC_M * dim * 2 + (size_t)PB_TC_STAGES * PB_TC_N * dim * 2 + (2 * PB_TC_STAGES + 5) * 8 + 16;
        switch (dim) {
#define PB_KM_CASE(DV)                                                                                                 \
    case DV: {                                                                                                         \
        auto kern = k_assign_tc<DV, true>;                                                                             \
        CKS(set_smem(kern, sm));                                                                                       \
        kern<<<blocks, 320, sm, st>>>(xb.as<__nv_bfloat16>(), n, cb.as<__nv_bfloat16>(), K, ts.as<float>(),            \
                                      ti.as<uint32_t>(), bias.as<float>());                                            \
    } break;
            PB_KM_CASE(64) PB_KM_CASE(96) PB_KM_CASE(128)
#undef PB_KM_CASE
            default: return pb_fail(PB_ERR_UNSUPPORTED, "tensor-core k-means assignment not built for dim %d", dim);
        }
        k_take_top1<<<sms * 4, 256, 0, st>>>(ti.as<uint32_t>(), n, codes);
        CK(cudaGetLastError());
        return PB_OK;
    }
};

extern "C" pb_status pb_kmeans_fit(int32_t device, const float *samples, int64_t n, int32_t dim, int64_t K, int32_t niters,
                                   uint64_t seed, float *out_centroids) {
    if (!samples || !out_centroids) return pb_fail(PB_ERR_INVALID, "null argument");
    if (n <= 0 || K <= 0 || K > n) return pb_fail(PB_ERR_INVALID, "need 0 < K <= n (K=%lld, n=%lld)", (long long)K, (long long)n);
    if (!dim_supported(dim)) return pb_fail(PB_ERR_UNSUPPORTED, "embedding_dim %d not built (32/64/96/128/256)", dim);
    CKS(check_device(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    const int sms = prop.multiProcessorCount;
    DevBuf dX, dC, dbias, dcodes, dsums, dcnt, didx;
    CKS(upload(dX, samples, (size_t)n * dim * 4, PB_MEM_HOST));
    CKS(dC.ensure((size_t)K * dim * 4));
    CKS(dbias.ensure((size_t)K * 4));
    CKS(dcodes.ensure((size_t)n * 4));
    CKS(dsums.ensure((size_t)K * dim * 4));
    CKS(dcnt.ensure((size_t)K * 4));
    // initial centroids: K distinct sample points (partial Fisher-Yates with a 64-bit LCG)
    std::vector<long long> perm((size_t)n);
    for (long long i = 0; i < n; ++i) perm[i] = i;
    uint64_t s = seed * 6364136223846793005ull + 1442695040888963407ull;
    for (long long i = 0; i < K; ++i) {
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        long long j = i + (long long)((s >> 11) % (uint64_t)(n - i));
        std::swap(perm[i], perm[j]);
    }
    CKS(upload(didx, perm.data(), (size_t)K * 8, PB_MEM_HOST));
    k_gather_rows<<<sms * 4, 256>>>(dX.as<float>(), didx.as<long long>(), K, dim, dC.as<float>());
    CK(cudaGetLastError());
    KmeansAssign ka;
    CKS(ka.init(dX.as<float>(), n, dim, K, sms, 0));
    for (int it = 0; it < niters; ++it) {
        CKS(ka.run(dX.as<float>(), dC.as<float>(), dbias.as<float>(), dcodes.as<uint32_t>(), 0));
        CK(cudaMemset(dsums.p, 0, (size_t)K * dim * 4));
        CK(cudaMemset(dcnt.p, 0, (size_t)K * 4));
        k_accumulate<<<sms * 8, 256>>>(dX.as<float>(), n, dim, dcodes.as<uint32_t>(), dsums.as<float>(), dcnt.as<float>());
        k_update_centroids<<<sms * 4, 256>>>(dC.as<float>(), K, dim, dsums.as<float>(), dcnt.as<float>());
        CK(cudaGetLastError());
    }
    k_normalize_rows<<<sms * 4, 256>>>(dC.as<float>(), K, dim);  // kmeans.rs:415-419
    CK(cudaGetLastError());
    CK(cudaMemcpy(out_centroids, dC.p, (size_t)K * dim * 4, cudaMemcpyDeviceToHost));
    return PB_OK;
}

// ------------------------------------------------------------------------------------------
// Data-parallel k-means (SURVEY 8e "Build path"): every rank holds a shard of the sample points, the centroids are
// replicated, and one all-reduce per iteration sums the per-rank [K][dim] coordinate sums and [K] counts (135 MB at
// K = 2^18, dim 128) -- over NCCL when the communicator came from pb_build_comm_init, or through the in-process shard
// group (peer copies + a rank-ordered sum, identical on every rank) when it came from pb_build_comm_group.
// ------------------------------------------------------------------------------------------
struct pb_build_comm {
    int device = 0, rank = 0, world = 1;
    ncclComm_t nccl = nullptr;
    pb_shard_group *group = nullptr;
    cudaStream_t stream = nullptr;
    DevBuf stage;
};

extern "C" pb_status pb_build_comm_init(const uint8_t *id128, int32_t rank, int32_t world, int32_t device, pb_build_comm **out) {
    if (!id128 || !out) return pb_fail(PB_ERR_INVALID, "null argument");
    if (world < 1 || rank < 0 || rank >= world) return pb_fail(PB_ERR_INVALID, "bad rank %d / world %d", rank, world);
    CKS(check_device(device));
    std::unique_ptr<pb_build_comm> c(new pb_build_comm());
    c->device = device;
    c->rank = rank;
    c->world = world;
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    if (world > 1) {
        if (!g_nccl.load()) return pb_fail(PB_ERR_COMM, "libnccl.so.2 not found (%s)", dlerror());
        ncclUniqueId id;
        memcpy(id.internal, id128, 128);
        CKN(g_nccl.CommInitRank(&c->nccl, world, id, rank));
    }
    *out = c.release();
    return PB_OK;
}
extern "C" pb_status pb_build_comm_group(pb_shard_group *g, int32_t rank, int32_t device, pb_build_comm **out) {
    if (!g || !out) return pb_fail(PB_ERR_INVALID, "null argument");
    if (rank < 0 || rank >= g->world) return pb_fail(PB_ERR_INVALID, "bad rank %d / world %d", rank, g->world);
    CKS(check_device(device));
    std::unique_ptr<pb_build_comm> c(new pb_build_comm());
    c->device = device;
    c->rank = rank;
    c->world = g->world;
    c->group = g;
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    {
        std::lock_guard<std::mutex> lk(g->mu);
        g->dev[rank] = device;
    }
    *out = c.release();
    return PB_OK;
}
extern "C" void pb_build_comm_destroy(pb_build_comm *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->nccl) g_nccl.CommDestroy(c->nccl);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

// in-place sum of `count` floats over the ranks; the result is bit-identical on every rank
static pb_status build_allreduce(pb_build_comm *c, float *buf, size_t count) {
    if (c->world == 1) return PB_OK;
    if (c->nccl) {
        CKN(g_nccl.AllReduce(buf, buf, count, PB_NCCL_FLOAT32, PB_NCCL_SUM, c->nccl, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        return PB_OK;
    }
    pb_shard_group *g = c->group;
    CKS(c->stage.ensure((size_t)c->world * count * 4));
    cudaError_t e = cudaStreamSynchronize(c->stream);
    g->send[c->rank] = buf;
    if (e != cudaSuccess || !g->barrier()) {
        g->fail();
        return pb_fail(PB_ERR_COMM, "shard group: a peer failed or timed out");
    }
    for (int p = 0; p < g->world && e == cudaSuccess; ++p)
        e = cudaMemcpyPeerAsync(c->stage.as<float>() + (size_t)p * count, c->device, g->send[p], g->dev[p], count * 4, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess || !g->barrier()) {  // everyone has read every buffer: they may be overwritten now
        g->fail();
        return pb_fail(PB_ERR_COMM, "shard group all-reduce failed");
    }
    k_sum_ranks<<<c->stage.cap ? 296 : 1, 256, 0, c->stream>>>(c->stage.as<float>(), c->world, (long long)count, buf);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(c->stream));
    return PB_OK;
}

extern "C" pb_status pb_kmeans_fit_dp(pb_build_comm *c, const float *samples, int64_t n_local, int32_t dim, int64_t K,
                                      int32_t niters, uint64_t seed, float *out_centroids) {
    if (!c || (!samples && n_local) || !out_centroids) return pb_fail(PB_ERR_INVALID, "null argument");
    if (n_local < 0 || K <= 0) return pb_fail(PB_ERR_INVALID, "bad sizes");
    if (!dim_supported(dim)) return pb_fail(PB_ERR_UNSUPPORTED, "embedding_dim %d not built (32/64/96/128/256)", dim);
    CK(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, c->device));
    const int sms = prop.multiProcessorCount;
    const long long n = n_local;
    // rank r seeds centroids [k0, k1) with distinct points of its shard; one all-reduce of the zero-padded table
    // gives every rank the same start
    const long long k0 = K * c->rank / c->world, k1 = K * (c->rank + 1) / c->world, kmine = k1 - k0;
    if (kmine > n) return pb_fail(PB_ERR_INVALID, "rank %d holds %lld points but seeds %lld centroids", c->rank, n, kmine);
    DevBuf dX, dC, dbias, dcodes, dacc, didx;
    CKS(upload(dX, samples, (size_t)std::max<long long>(n, 1) * dim * 4, PB_MEM_HOST));
    CKS(dC.ensure((size_t)K * dim * 4));
    CKS(dbias.ensure((size_t)K * 4));
    CKS(dcodes.ensure((size_t)std::max<long long>(n, 1) * 4));
    CKS(dacc.ensure((size_t)K * (dim + 1) * 4));  // [K][dim] sums followed by [K] counts: one all-reduce
    std::vector<long long> perm((size_t)n);
    for (long long i = 0; i < n; ++i) perm[i] = i;
    uint64_t s = (seed + 0x9e3779b97f4a7c15ull * (uint64_t)(c->rank + 1)) * 6364136223846793005ull + 1442695040888963407ull;
    for (long long i = 0; i < kmine; ++i) {
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        long long j = i + (long long)((s >> 11) % (uint64_t)(n - i));
        std::swap(perm[i], perm[j]);
    }
    CK(cudaMemsetAsync(dC.p, 0, (size_t)K * dim * 4, c->stream));
    if (kmine > 0) {
        CKS(upload(didx, perm.data(), (size_t)kmine * 8, PB_MEM_HOST));
        k_gather_rows<<<sms * 4, 256, 0, c->stream>>>(dX.as<float>(), didx.as<long long>(), kmine, dim, dC.as<float>() + (size_t)k0 * dim);
        CK(cudaGetLastError());
    }
    CKS(build_allreduce(c, dC.as<float>(), (size_t)K * dim));
    float *sums = dacc.as<float>(), *counts = dacc.as<float>() + (size_t)K * dim;
    KmeansAssign ka;
    CKS(ka.init(dX.as<float>(), n, dim, K, sms, c->stream));
    for (int it = 0; it < niters; ++it) {
        CKS(ka.run(dX.as<float>(), dC.as<float>(), dbias.as<float>(), dcodes.as<uint32_t>(), c->stream));
        CK(cudaMemsetAsync(dacc.p, 0, (size_t)K * (dim + 1) * 4, c->stream));
        if (n > 0) k_accumulate<<<sms * 8, 256, 0, c->stream>>>(dX.as<float>(), n, dim, dcodes.as<uint32_t>(), sums, counts);
        CK(cudaGetLastError());
        CKS(build_allreduce(c, dacc.as<float>(), (size_t)K * (dim + 1)));
        k_update_centroids<<<sms * 4, 256, 0, c->stream>>>(dC.as<float>(), K, dim, sums, counts);
        CK(cudaGetLastError());
    }
    k_normalize_rows<<<sms * 4, 256, 0, c->stream>>>(dC.as<float>(), K, dim);  // kmeans.rs:415-419
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out_centroids, dC.p, (size_t)K * dim * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return PB_OK;
}

// find_outliers (update.rs:490-608) on the codec's centroids
extern "C" pb_status pb_codec_find_outliers(pb_codec *c, const float *embeddings, int64_t n, float threshold_sq,
                                            int64_t *out_indices, int64_t *out_count) {
    if (!c || (!embeddings && n) || !out_count || (!out_indices && n)) return pb_fail(PB_ERR_INVALID, "null argument");
    *out_count = 0;
    if (n <= 0) return n == 0 ? PB_OK : pb_fail(PB_ERR_INVALID, "negative size");
    CK(cudaSetDevice(c->device));
    DevBuf cn, dX, xn, md, fl;
    CKS(cn.ensure((size_t)c->K * 4));
    k_squared_norms_ref<<<c->sm_count * 4, 256>>>(c->centroids.as<float>(), c->K, c->dim, cn.as<float>());
    const long long slab = 1ll << 20;
    CKS(dX.ensure((size_t)std::min<long long>(n, slab) * c->dim * 4));
    CKS(xn.ensure((size_t)std::min<long long>(n, slab) * 4));
    CKS(md.ensure((size_t)std::min<long long>(n, slab) * 4));
    CKS(fl.ensure((size_t)std::min<long long>(n, slab)));
    std::vector<uint8_t> hf((size_t)std::min<long long>(n, slab));
    int64_t cnt = 0;
    for (long long o = 0; o < n; o += slab) {
        const long long m = std::min(slab, n - o);
        CK(cudaMemcpy(dX.p, embeddings + (size_t)o * c->dim, (size_t)m * c->dim * 4, cudaMemcpyHostToDevice));
        k_squared_norms_ref<<<c->sm_count * 4, 256>>>(dX.as<float>(), m, c->dim, xn.as<float>());
        const unsigned blocks = (unsigned)((m + 63) / 64);
        PB_DIM_SWITCH(c->dim, {
            auto kern = k_min_dist<DIM>;
            CKS(set_smem(kern, smem_assign(DIM)));
            kern<<<blocks, 256, smem_assign(DIM)>>>(dX.as<float>(), m, xn.as<float>(), c->centroids.as<float>(), c->K,
                                                    cn.as<float>(), md.as<float>());
        });
        k_outlier_decide<<<c->sm_count * 8, 256>>>(dX.as<float>(), m, c->dim, c->centroids.as<float>(), c->K, md.as<float>(),
                                                   threshold_sq, fl.as<uint8_t>());
        CK(cudaGetLastError());
        CK(cudaMemcpy(hf.data(), fl.p, (size_t)m, cudaMemcpyDeviceToHost));
        for (long long i = 0; i < m; ++i)
            if (hf[i]) out_indices[cnt++] = o + i;
    }
    *out_count = cnt;
    return PB_OK;
}
