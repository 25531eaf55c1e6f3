// k_scores_tc.cuh -- a2 on the tensor cores (the default path) and the consumers of its score table.
// Part of kernels.cuh (included from there, in order; not a standalone header).
// ==========================================================================================
// a2 = the one dense contraction of the path (search.rs:345 / :171-174): S = Q C^T for every query token of the
// sub-batch against all K centroids.  k_scores16_tc computes it as a 3-product split-fp16 UMMA GEMM
//     x = xh + xl  (xh = fp16(x), xl = fp16(x - xh));   S~ = qh.ch + qh.cl + ql.ch   (fp32 accumulator in TMEM)
// and writes ONLY the 16-bit fixed-point score table ST16[b][c][QS] the probe (a3) and the first approximate pass
// (a5) stream / gather.  Nothing downstream needs a dense fp32 S: the few values that decide something
//   - the exact selection keys of the probe winners            (k_collect16_tc)
//   - the threshold test of the selected cells                 (k_cells_unique -> k_exact_rows -> k_cells_thr)
//   - the per-token maxima of the docs around the cut          (k_approx_recheck)
// are recomputed as pinned-order fp32 dots (common.cuh), so every decision and every output bit equals the
// exact path's.
//
// Error budget (the certificate).  Both operands are scaled by powers of two (exact) so that max|q'|, max|c'| are
// in [1, 2): kq per query (k_query_range), kc per index (pb_index_finalize).  With e = the pinned-order fp32 dot
// and t = the tensor-core estimate of the same pair, in units of R' = max|q'| max|c'| (1 + 1e-4):
//     |e - q.c|  <= dim 2^-24                     (fp32 FMA chain, |partial sums| <= |q'||c'|)
//     |t - q.c|  <= 3 * 2^-22 + 2^-21             (two dropped split terms + ql.cl; fp32 accumulation of 3 dim/16 MMAs)
//                   + 2^-25 sqrt(dim) (|q'| + |c'|) / R'   (fp16 subnormal spacing of the lo parts)
// => |e - t| * scale <= err_codes(dim) = (dim 2^-24 + 2^-20) * 32768 + 4 * 2^-25 sqrt(dim) * 32768 < 0.34 for
// dim <= 128 (k1_err_codes() in engine.cu), i.e. an estimate-built code differs from the exact-table code by at most
// E = 1.  Consumers use: code margin 2E + 1 = 3 for "could still be the maximum / in the top n", and the band
// W = nq (1.004 + 2 err) + nq^2 / 256 + 4 for the first approximate pass (derivations at each kernel).
// PB_K1_TC_DIAG=1 measures the largest code difference against the exact table (pb_work_counters).
// grid = ceil(K/128) CTAs, 320 threads: warps 0-7 epilogue (warp w: TMEM lanes 32*(w%4).., column half w/4), warp 8
// bulk-copy loader, warp 9 MMA issuer.
// ==========================================================================================

// fp16 hi/lo split of `n` rows, scaled by 2^kexp, into UMMA tile order (128-row tiles, K-major core matrices);
// rows >= n stay zero
__global__ void k_rows_to_f16_split_tiles(const float *__restrict__ X, long long n, int dim, int kexp,
                                          __half *__restrict__ Xh, __half *__restrict__ Xl) {
    const int lane = threadIdx.x & 31;
    const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
    const size_t tile_elems = (size_t)128 * dim;
    const float mul = ldexpf(1.0f, kexp);
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += nw) {
        const size_t tbase = (size_t)(r >> 7) * tile_elems;
        const int rr = (int)(r & 127);
        for (int j = lane; j < dim; j += 32) {
            const float v = X[(size_t)r * dim + j] * mul;
            const __half h = __float2half_rn(v);
            const size_t o = tbase + (size_t)((j >> 3) * 16 + (rr >> 3)) * 64 + (rr & 7) * 8 + (j & 7);
            Xh[o] = h;
            Xl[o] = __float2half_rn(v - __half2float(h));
        }
    }
}

// the same for the query rows in the QS-padded layout (row = b*QS + q, rows q >= nq are zero); query b is scaled by
// 2^qexp[b]
__global__ void k_query_split_tiles(const float *__restrict__ Q, const int *__restrict__ q_off, const int *__restrict__ qexp,
                                    int B, int QS, int dim, __half *__restrict__ Qh, __half *__restrict__ Ql) {
    const int lane = threadIdx.x & 31;
    const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
    const size_t tile_elems = (size_t)128 * dim;
    const long long n = (((long long)B * QS + 127) / 128) * 128;
    for (long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += nw) {
        const long long b = r / QS;
        const int q = (int)(r - b * QS);
        const bool real = b < B && q < q_off[b + 1] - q_off[b];
        const float mul = real ? ldexpf(1.0f, qexp[b]) : 0.0f;
        const size_t tbase = (size_t)(r >> 7) * tile_elems;
        const int rr = (int)(r & 127);
        for (int j = lane; j < dim; j += 32) {
            const float v = real ? Q[(size_t)(q_off[b] + q) * dim + j] * mul : 0.0f;
            const __half h = __float2half_rn(v);
            const size_t o = tbase + (size_t)((j >> 3) * 16 + (rr >> 3)) * 64 + (rr & 7) * 8 + (j & 7);
            Qh[o] = h;
            Ql[o] = __float2half_rn(v - __half2float(h));
        }
    }
}

// qrange_tc[b] = (R*scale, scale * 2^-(qexp[b] + kc)): the code of an accumulator value of the scaled operands
__global__ void k_query_range_tc(const float2 *__restrict__ qrange, const int *__restrict__ qexp, int kc, int B,
                                 float2 *__restrict__ qrange_tc) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float2 rg = qrange[b];
    qrange_tc[b] = make_float2(rg.x, ldexpf(rg.y, -(qexp[b] + kc)));
}

template <int DIM>
__global__ void __launch_bounds__(320, 1)
k_scores16_tc(const __half *__restrict__ Ch, const __half *__restrict__ Cl, long long K, const __half *__restrict__ Qh,
              const __half *__restrict__ Ql, int n_groups, int B, int QS, const int *__restrict__ q_off,
              const float2 *__restrict__ qrange_tc, unsigned short *__restrict__ ST16, int *__restrict__ qflag) {
    extern __shared__ __align__(128) unsigned char smem_k1[];
    constexpr int KSTEPS = DIM / 16;
    constexpr uint32_t T_BYTES = 128 * DIM * 2;  // one 128-row fp16 tile
    constexpr uint32_t LBO = 16 * 128, SBO = 128;
    unsigned char *Ah = smem_k1, *Al = Ah + T_BYTES;  // this CTA's centroid tile, hi and lo
    unsigned char *Bs = Al + T_BYTES;                 // 2 stages x (hi, lo) query-row tiles
    uint64_t *bars = reinterpret_cast<uint64_t *>(Bs + 4 * T_BYTES);
    uint64_t *full = bars, *empty = bars + 2, *tfull = bars + 4, *tempty = bars + 6, *abar = bars + 8;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 9);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long c0 = (long long)blockIdx.x * 128;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
            mbar_init(&tfull[i], 1);
            mbar_init(&tempty[i], 256);
        }
        mbar_init(abar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (w == 9) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (w == 8) {
        // ---------------- loader ----------------
        if (lane == 0) {
            mbar_expect_tx(abar, 2 * T_BYTES);
            bulk_g2s(Ah, reinterpret_cast<const unsigned char *>(Ch) + (size_t)blockIdx.x * T_BYTES, T_BYTES, abar);
            bulk_g2s(Al, reinterpret_cast<const unsigned char *>(Cl) + (size_t)blockIdx.x * T_BYTES, T_BYTES, abar);
            for (int g = 0; g < n_groups; ++g) {
                const int st = g & 1;
                mbar_wait(&empty[st], (uint32_t)(((g >> 1) & 1) ^ 1));
                mbar_expect_tx(&full[st], 2 * T_BYTES);
                bulk_g2s(Bs + (size_t)(2 * st) * T_BYTES, reinterpret_cast<const unsigned char *>(Qh) + (size_t)g * T_BYTES, T_BYTES, &full[st]);
                bulk_g2s(Bs + (size_t)(2 * st + 1) * T_BYTES, reinterpret_cast<const unsigned char *>(Ql) + (size_t)g * T_BYTES, T_BYTES, &full[st]);
            }
        }
    } else if (w == 9) {
        // ---------------- MMA issuer: 3 products per k-step into one fp32 accumulator ----------------
        // instruction descriptor: c = f32, a = b = f16 (format 0), K-major, N = 128, M = 128
        const uint32_t idesc = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        mbar_wait(abar, 0);
        for (int g = 0; g < n_groups; ++g) {
            const int st = g & 1, acc = g & 1;
            mbar_wait(&full[st], (uint32_t)((g >> 1) & 1));
            mbar_wait(&tempty[acc], (uint32_t)(((g >> 1) & 1) ^ 1));
            tc_fence_after();
            if (lane == 0) {
                const uint32_t ah = smem_u32(Ah), al = smem_u32(Al);
                const uint32_t bh = smem_u32(Bs + (size_t)(2 * st) * T_BYTES), bl = smem_u32(Bs + (size_t)(2 * st + 1) * T_BYTES);
#pragma unroll
                for (int s = 0; s < KSTEPS; ++s) {
                    const u64 dah = tc_smem_desc(ah + s * 2 * LBO, LBO, SBO), dal = tc_smem_desc(al + s * 2 * LBO, LBO, SBO);
                    const u64 dbh = tc_smem_desc(bh + s * 2 * LBO, LBO, SBO), dbl = tc_smem_desc(bl + s * 2 * LBO, LBO, SBO);
                    tc_mma_bf16(tmem_base + acc * 128, dah, dbh, idesc, s > 0 ? 1u : 0u);
                    tc_mma_bf16(tmem_base + acc * 128, dah, dbl, idesc, 1u);
                    tc_mma_bf16(tmem_base + acc * 128, dal, dbh, idesc, 1u);
                }
                tc_commit(&empty[st]);   // query tiles consumed
                tc_commit(&tfull[acc]);  // accumulators ready
            }
            __syncwarp();
        }
    } else {
        // ---------------- epilogue: thread = centroid row (TMEM lane), 64 of the 128 padded query rows ----------------
        const int lg = w & 3, ch = w >> 2;
        const long long c = c0 + 32 * lg + lane;
        for (int g = 0; g < n_groups; ++g) {
            const int acc = g & 1;
            mbar_wait(&tfull[acc], (uint32_t)((g >> 1) & 1));
            tc_fence_after();
            // (Both 32-column loads in flight and the accumulator handed back before the conversion and the stores was
            // measured: 0.349 against 0.351 ms -- the TMEM read latency is not what bounds the epilogue.)
#pragma unroll 1
            for (int cb = 2 * ch; cb < 2 * ch + 2; ++cb) {
                uint32_t rr[32];
                tc_ld32(tmem_base + ((uint32_t)(32 * lg) << 16) + acc * 128 + cb * 32, rr);
#pragma unroll
                for (int sub = 0; sub < 4; ++sub) {
                    const int row0 = g * 128 + cb * 32 + sub * 8;  // 8 query rows of one query (QS % 8 == 0)
                    const int b = row0 / QS, q = row0 - b * QS;
                    if (b >= B || c >= K) continue;
                    const float2 rg = qrange_tc[b];  // (R*scale, scale / 2^(kq+kc))
                    uint32_t cd[8];
                    bool ok = true;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        // code = floor(x) clamped to [0, 65535]; x outside [+0, 65536) (NaN, -0 included) raises the
                        // query's flag and the sub-batch is redone on the exact path, so only in-range codes matter.
                        // Padding rows hold a zero accumulator: x = R*scale, in range.
                        const float x = __fmaf_rn(__uint_as_float(rr[sub * 8 + i]), rg.y, rg.x);
                        ok &= __float_as_uint(x) < 0x47800000u;
                        cd[i] = min(__float2uint_rd(x), 65535u);
                    }
                    if (!ok) atomicOr(&qflag[b], 1);
                    *reinterpret_cast<uint4 *>(ST16 + ((size_t)b * K + c) * QS + q) =
                        make_uint4(cd[0] | (cd[1] << 16), cd[2] | (cd[3] << 16), cd[4] | (cd[5] << 16), cd[6] | (cd[7] << 16));
                }
            }
            tc_fence_before();
            mbar_arrive(&tempty[acc]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (w == 9) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
    }
}

// largest |a - b| over the codes of real query tokens (PB_K1_TC_DIAG)
__global__ void k_diff16(const unsigned short *__restrict__ a, const unsigned short *__restrict__ b, const int *__restrict__ q_off,
                         long long K, int QS, int *__restrict__ out_max) {
    const int bq = blockIdx.y, nq = q_off[bq + 1] - q_off[bq];
    int best = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < K * QS; i += (long long)gridDim.x * blockDim.x) {
        const int q = (int)(i % QS);
        if (q >= nq) continue;
        const size_t o = (size_t)bq * K * QS + i;
        best = max(best, abs((int)a[o] - (int)b[o]));
    }
    best = __reduce_max_sync(PB_FULL, best);
    if ((threadIdx.x & 31) == 0 && best) atomicMax(out_max, best);
}

// ------------------------------------------------------------------------------------------
// Exact pinned-order score rows for a LIST of centroids per query: OUT[b][i][QS] = S[q][list[b][i]].
// Same FFMA2 tile as k_centroid_scores<., true>; the centroid rows are gathered with cp.async.
// grid = (ceil(cap/128), B), 128 threads.
// ------------------------------------------------------------------------------------------
template <int DIM>
__global__ void __launch_bounds__(128, 2)
k_exact_rows(const float *__restrict__ Qi, const int *__restrict__ q_off, int QS, const float *__restrict__ C,
             const uint32_t *__restrict__ list, const int *__restrict__ list_n, int cap, float *__restrict__ out) {
    extern __shared__ __align__(16) float smem[];
    constexpr int LD = DIM + 4, G = DIM / 4;
    float *Vs = smem;                      // [128][LD] gathered centroid rows
    float *Qs = smem + PB_TOK_TILE * LD;   // 16 interleaved row pairs
    const int b = blockIdx.y, n = min(list_n[b], cap), i0 = blockIdx.x * PB_TOK_TILE;
    if (i0 >= n) return;
    const int nv = min(PB_TOK_TILE, n - i0);
    const uint32_t *lst = list + (size_t)b * cap + i0;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int idx = threadIdx.x; idx < PB_TOK_TILE * G; idx += blockDim.x) {
        const int r = idx / G, g = idx - r * G;
        if (r < nv) cp_async16(Vs + r * LD + 4 * g, C + (size_t)lst[r] * DIM + 4 * g);
        else *reinterpret_cast<float4 *>(Vs + r * LD + 4 * g) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int nq = q_off[b + 1] - q_off[b];
    for (int qb = 0; qb < nq; qb += PB_Q_TILE) {
        load_pairs_async<DIM>(Qs, Qi + ((size_t)b * QS + qb) * DIM, min(PB_Q_TILE, QS - qb) / 2, PB_Q_TILE / 2);
        cp_async_wait_all();
        __syncthreads();
        if (qb + 8 * w < ((nq + 7) & ~7)) {
            float acc[8][4];
            tile_dots_f2<DIM>(Qs + 4 * w * 2 * DIM, Vs + lane * LD, acc);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = lane + 32 * k;
                if (i < nv) {
                    float4 *dst = reinterpret_cast<float4 *>(out + ((size_t)b * cap + i0 + i) * QS + qb + 8 * w);
                    dst[0] = make_float4(acc[0][k], acc[1][k], acc[2][k], acc[3][k]);
                    dst[1] = make_float4(acc[4][k], acc[5][k], acc[6][k], acc[7][k]);
                }
            }
        }
        __syncthreads();
    }
}

// the pinned-order dot of common.cuh for one (query token, centroid) pair, 128-bit loads
PB_DEV float pinned_dot(const float *__restrict__ q, const float *__restrict__ c, int dim) {
    float s = 0.0f;
    for (int j = 0; j < dim; j += 4) {
        const float4 a = *reinterpret_cast<const float4 *>(q + j), v = *reinterpret_cast<const float4 *>(c + j);
        s = __fmaf_rn(a.x, v.x, s);
        s = __fmaf_rn(a.y, v.y, s);
        s = __fmaf_rn(a.z, v.z, s);
        s = __fmaf_rn(a.w, v.w, s);
    }
    return s;
}

// ------------------------------------------------------------------------------------------
// a3 on the tensor-core table.  k_chunkmax16 / k_tau16 (k_probe.cuh) run unchanged: tau = the n-th largest chunk
// maximum of a token's ESTIMATE codes, so n entries with code >= tau exist (set A).  An entry x of the exact top n
// outside A displaces some a in A with e(x) >= e(a), hence t(x) >= t(a) - 2 delta and code(x) >= code(a) - (2E + 1)
// >= tau - code_margin: k_collect16_tc lowers the thresholds by code_margin and takes the exact selection key of
// every hit from a pinned-order dot, so k_topn_merge ranks exactly the keys the exact path would.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_collect16_tc(const unsigned short *__restrict__ ST16, const float *__restrict__ Q, const int *__restrict__ q_off,
               const float *__restrict__ C, int dim, int code_margin, long long K, int QS, int n_chunks, int chunk_rows,
               const uint32_t *__restrict__ tau, int cap, int *__restrict__ counts, u64 *__restrict__ list,
               int *__restrict__ fallback) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.y;
    const int chunk = blockIdx.x * 4 + w;
    if (chunk >= n_chunks || *fallback) return;
    const int GQ = QS >> 3, L = (32 / GQ) * GQ, g = lane % GQ;  // lane -> query-token group as in k_chunkmax16
    if (lane >= L) return;
    const long long c0 = (long long)chunk * chunk_rows;
    const int rows = (int)min((long long)chunk_rows, K - c0);
    const uint4 *base = reinterpret_cast<const uint4 *>(ST16 + ((size_t)b * K + c0) * QS);
    const int total = rows * GQ;
    // this lane's 8 thresholds as packed halfwords; padding rows (tau = 65536) never match
    uint32_t t2[4], live[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        uint32_t a = tau[(size_t)b * QS + 8 * g + 2 * e], c = tau[(size_t)b * QS + 8 * g + 2 * e + 1];
        if (a < 65536u) a = a > (uint32_t)code_margin ? a - (uint32_t)code_margin : 0u;
        if (c < 65536u) c = c > (uint32_t)code_margin ? c - (uint32_t)code_margin : 0u;
        t2[e] = min(a, 65535u) | (min(c, 65535u) << 16);
        live[e] = (a < 65536u ? 0xffffu : 0u) | (c < 65536u ? 0xffff0000u : 0u);
    }
    for (int i0 = lane; i0 < total; i0 += 8 * L) {
        uint4 v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = (i0 + L * e < total) ? __ldg(base + i0 + L * e) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t hx = __vcmpgeu2(v[e].x, t2[0]) & live[0], hy = __vcmpgeu2(v[e].y, t2[1]) & live[1];
            const uint32_t hz = __vcmpgeu2(v[e].z, t2[2]) & live[2], hw = __vcmpgeu2(v[e].w, t2[3]) & live[3];
            if ((hx | hy | hz | hw) == 0u || i0 + L * e >= total) continue;  // the common case
            const long long c = c0 + (i0 + L * e) / GQ;
            const uint32_t hits[4] = {hx, hy, hz, hw};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (!((hits[j >> 1] >> (16 * (j & 1))) & 1u)) continue;
                const int q = 8 * g + j;
                const int slot = atomicAdd(&counts[(size_t)b * QS + q], 1);
                if (slot < cap) {
                    const float s = pinned_dot(Q + (size_t)(q_off[b] + q) * dim, C + (size_t)c * dim, dim);
                    list[((size_t)b * QS + q) * cap + slot] = ((u64)score_key_asc(s) << 32) | (uint32_t)(~(uint32_t)c);
                } else atomicOr(fallback, 1);
            }
        }
    }
}

// the distinct selected centroids of a query, ascending: ulist[b][0..n_u).  grid = B, 256 threads, smem = P*12.
__global__ void __launch_bounds__(256)
k_cells_unique(const u64 *__restrict__ sel, const int *__restrict__ q_off, int QS, int n, int cap,
               uint32_t *__restrict__ ulist, int *__restrict__ n_u) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x;
    const int nq = q_off[b + 1] - q_off[b];
    const int total = nq * n;
    const int P = next_pow2(max(total, 1));
    u64 *s = reinterpret_cast<u64 *>(smem_raw);  // [P]
    __shared__ int scan_tmp[33];
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        u64 v = ~0ull;
        if (i < total) {
            const u64 k = sel[(size_t)b * QS * n + i];  // rows q < nq are the first nq*n entries
            if (k != 0ull) v = (u64)(uint32_t)(~(uint32_t)k);
        }
        s[i] = v;
    }
    __syncthreads();
    bitonic_sort_u64(s, P);
    int nu = 0;
    for (int base = 0; base < P; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int f = (i < P && s[i] != ~0ull && (i == 0 || s[i - 1] != s[i])) ? 1 : 0;
        int tot;
        const int pos = block_exclusive_scan(f, scan_tmp, &tot);
        if (f && nu + pos < cap) ulist[(size_t)b * cap + nu + pos] = (uint32_t)s[i];
        nu += tot;
    }
    if (threadIdx.x == 0) n_u[b] = min(nu, cap);
}

// the variant's threshold rule (k_cells, k_probe.cuh) on the exact rows of the selected centroids:
// rows[b][u][QS] = S[.][ulist[b][u]].  The batched variant's slab-prefix scan ("did c enter token q's slab heap?")
// ranks the earlier centroids of the slab on the 16-bit estimate table: with kv16 = the code of the exact value v,
// an estimate code >= kv16 + code_margin is certainly not below v, one <= kv16 - code_margin certainly below,
// anything between is settled by a pinned-order dot.  grid = (slices, B), 256 threads: a warp per selected centroid, the
// keep flags go to global memory and k_cells_emit compacts them in order.
__global__ void __launch_bounds__(256)
k_cells_thr(const u64 *__restrict__ sel, const float *__restrict__ rows, const uint32_t *__restrict__ ulist,
            const int *__restrict__ n_u, const int *__restrict__ q_off, long long K, int QS, int n, int cap, int has_thr,
            float thr, int batched, long long slab, int *__restrict__ flags,
            const unsigned short *__restrict__ ST16, const float2 *__restrict__ qrange, int code_margin,
            const float *__restrict__ Q, const float *__restrict__ C, int dim, const unsigned short *__restrict__ cmax16,
            int n_chunks, int chunk_rows) {
    const int b = blockIdx.y;
    const int nq = q_off[b + 1] - q_off[b];
    const int nu = n_u[b];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int u = blockIdx.x * nwarps + w; u < nu; u += gridDim.x * nwarps) {
        const uint32_t c = ulist[(size_t)b * cap + u];
        int keep = 1;
        if (has_thr) {
            const float *row = rows + ((size_t)b * cap + u) * QS;
            if (!batched) {
                uint32_t best = 0u;
                for (int q = lane; q < nq; q += 32) best = max(best, score_key_asc(row[q]));
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) best = max(best, __shfl_xor_sync(PB_FULL, best, m));
                // Iterator::max_by keeps the last maximum: all non-finite -> the last token's value
                const float mval = best ? key_to_score(best) : (nq > 0 ? row[nq - 1] : -INFINITY);
                keep = (mval >= thr);
            } else {
                uint32_t best = 0u;
                for (int q = lane; q < nq; q += 32) {
                    const u64 *sq = sel + ((size_t)b * QS + q) * n;
                    bool is_sel = false;
                    for (int i = 0; i < n; ++i)
                        if (sq[i] != 0ull && (uint32_t)(~(uint32_t)sq[i]) == c) is_sel = true;
                    if (is_sel) best = max(best, score_key_asc(row[q]));
                }
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) best = max(best, __shfl_xor_sync(PB_FULL, best, m));
                const float m1 = best ? key_to_score(best) : -INFINITY;
                keep = (m1 >= thr);
                if (!keep) {
                    // another token may have recorded a score >= thr for c while scanning its slab
                    const long long s0 = (long long)(c / slab) * slab;
                    const float2 rg = qrange[b];
                    for (int q = 0; q < nq && !keep; ++q) {
                        const float v = row[q];
                        const uint32_t kv = score_key_asc(v);
                        if (!(kv != 0u && v >= thr)) continue;  // finite and over the threshold
                        const int kv16 = (int)fminf(fmaxf(floorf(__fmaf_rn(v, rg.y, rg.x)), 0.0f), 65535.0f);
                        const unsigned short *col16 = ST16 + (size_t)b * K * QS + q;
                        const float *qrow = Q + (size_t)(q_off[b] + q) * dim;
                        // the chunk maxima of the probe (k_chunkmax16) rule out almost every chunk of the slab prefix: a
                        // chunk whose largest estimate code is <= kv16 - code_margin holds no entry that could reach v
                        int cnt = 0;
                        const long long ch_lo = s0 / chunk_rows, ch_hi = ((long long)c + chunk_rows - 1) / chunk_rows;
                        for (long long ch0 = ch_lo; ch0 < ch_hi; ch0 += 32) {
                            const long long chl = ch0 + lane;
                            const bool need = chl < ch_hi &&
                                              (int)cmax16[((size_t)b * n_chunks + chl) * QS + q] + code_margin > kv16;
                            unsigned todo = __ballot_sync(PB_FULL, need);
                            while (todo) {
                                const long long ch = ch0 + (__ffs(todo) - 1);
                                todo &= todo - 1;
                                const long long r_lo = max(s0, ch * chunk_rows), r_hi = min((long long)c, (ch + 1) * chunk_rows);
                                for (long long c2 = r_lo + lane; c2 < r_hi; c2 += 128) {  // four strided loads in flight
                                    int cd[4];
#pragma unroll
                                    for (int e = 0; e < 4; ++e) cd[e] = c2 + 32 * e < r_hi ? (int)col16[(size_t)(c2 + 32 * e) * QS] : -1000000;
#pragma unroll
                                    for (int e = 0; e < 4; ++e) {
                                        if (cd[e] >= kv16 + code_margin) ++cnt;
                                        else if (cd[e] + code_margin > kv16)
                                            cnt += (score_key_asc(pinned_dot(qrow, C + (size_t)(c2 + 32 * e) * dim, dim)) >= kv) ? 1 : 0;
                                    }
                                }
                            }
                        }
#pragma unroll
                        for (int m = 16; m >= 1; m >>= 1) cnt += __shfl_xor_sync(PB_FULL, cnt, m);
                        if (cnt < n) keep = 1;
                    }
                }
            }
        }
        if (lane == 0) flags[(size_t)b * cap + u] = keep;
    }
}

// ordered compaction of the kept cells.  grid = B, 256 threads.
__global__ void __launch_bounds__(256)
k_cells_emit(const uint32_t *__restrict__ ulist, const int *__restrict__ n_u, const int *__restrict__ flags, int cap,
             uint32_t *__restrict__ cells, int *__restrict__ n_cells) {
    __shared__ int scan_tmp[33];
    const int b = blockIdx.x;
    const int nu = n_u[b];
    int outn = 0;
    for (int base = 0; base < nu; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int f = (i < nu) ? flags[(size_t)b * cap + i] : 0;
        int tot;
        const int pos = block_exclusive_scan(f, scan_tmp, &tot);
        if (f && outn + pos < cap) cells[(size_t)b * cap + outn + pos] = ulist[(size_t)b * cap + i];
        outn += tot;
    }
    if (threadIdx.x == 0) n_cells[b] = min(outn, cap);
}

// ------------------------------------------------------------------------------------------
// a5 second pass on the tensor-core table: the EXACT approximate score (search.rs:305-324) of the docs that can
// still make the cut, without a dense fp32 S.  For a doc and a query token q, m_q = the largest estimate code over
// the doc's distinct codes; the code c* that attains the exact maximum satisfies code(c*) >= m_q - (2E + 1)
// (e(c*) >= e(c^) for the estimate's argmax c^, so t(c*) >= t(c^) - 2 delta), so the exact per-token maximum is the
// maximum of the pinned-order dots over the (typically one or two) codes within `code_margin` of m_q.  Three kernels,
// each with all the parallelism the work has (a one-kernel form -- warp per doc, dots in place -- ran at 8 warps per
// SM and 1.6 ms):
//   k_recheck_pairs  warp per doc: column maxima, then the (doc slot, q, code) pairs inside the margin appended to the
//                    query's pair list (staged per warp: one atomic per doc and pass)
//   k_recheck_dots   thread per pair: the pinned-order dot, atomicMax of its score key into exactmax[b][slot][q]
//   k_recheck_sum    warp per doc: the q-ordered fp32 sum of the maxima -> approx[b][i] and the cut key (what k_approx
//                    emits); clears the doc's exactmax row for the next call
// More docs than rc_cap or more pairs than pair_cap raise *fallback (the sub-batch is redone on the exact path).  The
// abandoned pass must stay memory-safe: k_recheck_sum still gives every candidate a cut key holding its own doc id
// (score 0 past rc_cap, where no maxima row exists), because k_cut and the exact stage index documents by that id.
// ------------------------------------------------------------------------------------------
// Two passes over the doc's codes with the row-group gather of k_approx16 (16-byte loads of 8 query tokens, packed
// vmaxu2 / vcmpgeu2): pass A the column maxima, pass B (rows now in L1) every (code, query token) whose estimate code is
// within code_margin of its column maximum.  (A one-pass form -- lane = query token, 2-byte loads, the three largest codes
// of every column tracked in registers -- was issue-bound: 0.33 ms against 0.24 ms for 1024 docs x 32 queries.)  Hits go through a per-warp
// shared-memory stage so that the query's pair counter sees one atomic per (doc, pass); a stage overflow (a query token
// whose maximum is inside the margin of zero lists every code) writes the surplus directly.  The padding entries of a
// code list repeat its last code: such repeats are listed again, k_recheck_dots' atomicMax does not care.
template <int LPR>
__global__ void __launch_bounds__(256, LPR == 4 ? 3 : 2)
k_recheck_pairs(const unsigned short *__restrict__ ST16, const int *__restrict__ q_off, long long K, int QS,
                 const uint32_t *__restrict__ ucodes, const long long *__restrict__ udoc_off,
                 const uint32_t *__restrict__ cand, long long cand_cap, const int *__restrict__ n_cand, int code_margin,
                 int rc_cap, int pair_cap, u64 *__restrict__ pairs, int *__restrict__ n_pairs, int *__restrict__ fallback,
                 unsigned long long *__restrict__ tok_counter) {
    constexpr int RG = 32 / LPR;   // row groups of a warp = rows per load instruction
    constexpr int QB = 8 * LPR;    // query tokens covered by one pass
    constexpr int NI = 64 / RG;    // load instructions per 64 codes
    constexpr int STAGE = 128;
    __shared__ u64 stage[8][STAGE];
    __shared__ int stage_n[8];
    const int b = blockIdx.y;
    const int nq = q_off[b + 1] - q_off[b];
    const int n = n_cand[b];
    if (n > rc_cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(fallback, 1);
        return;
    }
    const int lane = threadIdx.x & 31, wv = threadIdx.x >> 5, r = lane / LPR, sl = lane % LPR;
    const int warps_per_grid = gridDim.x * (blockDim.x >> 5);
    const char *STb = reinterpret_cast<const char *>(ST16 + (size_t)b * K * QS);
    const unsigned rowb = (unsigned)QS * 2u;
    u64 *plist = pairs + (size_t)b * pair_cap;
    const uint32_t mg2 = (uint32_t)code_margin | ((uint32_t)code_margin << 16);
    unsigned long long my_tokens = 0;
    for (int i = blockIdx.x * (blockDim.x >> 5) + wv; i < n; i += warps_per_grid) {
        const uint32_t d = cand[(size_t)b * cand_cap + i];
        const long long t0 = udoc_off[d], t1 = udoc_off[d + 1];
        my_tokens += (unsigned long long)(t1 - t0);
        for (int qc = 0; qc < nq; qc += QB) {
            const int q0 = qc + 8 * sl;
            const bool in_row = q0 < QS;  // QS is a multiple of 8: groups past the row are skipped
            const char *col = STb + (in_row ? q0 * 2 : 0);
            // ---- pass A: packed column maxima of query tokens q0 .. q0 + 7 ----
            uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
            for (long long t = t0; t < t1; t += 64) {
                const uint32_t cl0 = ucodes[min(t + lane, t1 - 1)], cl1 = ucodes[min(t + 32 + lane, t1 - 1)];
                if (t + 64 <= t1) {
                    uint4 v[NI];
#pragma unroll
                    for (int e = 0; e < NI; ++e)
                        v[e] = gather16(col + (size_t)__shfl_sync(PB_FULL, e < NI / 2 ? cl0 : cl1, RG * (e % (NI / 2)) + r) * rowb);
#pragma unroll
                    for (int e = 0; e < NI; ++e) {
                        m0 = __vmaxu2(m0, v[e].x);
                        m1 = __vmaxu2(m1, v[e].y);
                        m2 = __vmaxu2(m2, v[e].z);
                        m3 = __vmaxu2(m3, v[e].w);
                    }
                } else {
                    const int ne = (int)((t1 - t + RG - 1) / RG);
                    for (int e = 0; e < ne; ++e) {
                        const uint4 va = gather16(col + (size_t)__shfl_sync(PB_FULL, e < NI / 2 ? cl0 : cl1, RG * (e % (NI / 2)) + r) * rowb);
                        m0 = __vmaxu2(m0, va.x);
                        m1 = __vmaxu2(m1, va.y);
                        m2 = __vmaxu2(m2, va.z);
                        m3 = __vmaxu2(m3, va.w);
                    }
                }
            }
#pragma unroll
            for (int m = LPR; m < 32; m <<= 1) {
                m0 = __vmaxu2(m0, __shfl_xor_sync(PB_FULL, m0, m));
                m1 = __vmaxu2(m1, __shfl_xor_sync(PB_FULL, m1, m));
                m2 = __vmaxu2(m2, __shfl_xor_sync(PB_FULL, m2, m));
                m3 = __vmaxu2(m3, __shfl_xor_sync(PB_FULL, m3, m));
            }
            // thresholds (saturating: a maximum inside the margin of zero admits every code) and the real query tokens
            const uint32_t l0 = __vsubus2(m0, mg2), l1 = __vsubus2(m1, mg2), l2 = __vsubus2(m2, mg2), l3 = __vsubus2(m3, mg2);
            uint32_t vm[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                vm[j] = in_row ? ((q0 + 2 * j < nq ? 0xffffu : 0u) | (q0 + 2 * j + 1 < nq ? 0xffff0000u : 0u)) : 0u;
            if (lane == 0) stage_n[wv] = 0;
            __syncwarp();
            const u64 head = (u64)i << 40;
            // ---- pass B: the (code, query token) pairs inside the margin ----
            for (long long t = t0; t < t1; t += 64) {
                const uint32_t cl0 = ucodes[min(t + lane, t1 - 1)], cl1 = ucodes[min(t + 32 + lane, t1 - 1)];
                const int ne = t + 64 <= t1 ? NI : (int)((t1 - t + RG - 1) / RG);
#pragma unroll 4
                for (int e = 0; e < ne; ++e) {
                    const uint32_t c = __shfl_sync(PB_FULL, e < NI / 2 ? cl0 : cl1, RG * (e % (NI / 2)) + r);
                    const uint4 v = gather16(col + (size_t)c * rowb);
                    const uint32_t h[4] = {__vcmpgeu2(v.x, l0) & vm[0], __vcmpgeu2(v.y, l1) & vm[1], __vcmpgeu2(v.z, l2) & vm[2],
                                           __vcmpgeu2(v.w, l3) & vm[3]};
                    if ((h[0] | h[1] | h[2] | h[3]) && t + (e < NI / 2 ? 0 : 32) + RG * (e % (NI / 2)) + r < t1) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
#pragma unroll
                            for (int hi = 0; hi < 2; ++hi)
                                if (h[j] & (hi ? 0xffff0000u : 0xffffu)) {
                                    const u64 entry = head | ((u64)(q0 + 2 * j + hi) << 32) | c;
                                    const int slot = atomicAdd(&stage_n[wv], 1);
                                    if (slot < STAGE) stage[wv][slot] = entry;
                                    else {
                                        const int pos = atomicAdd(&n_pairs[b], 1);
                                        if (pos < pair_cap) plist[pos] = entry;
                                        else atomicOr(fallback, 1);
                                    }
                                }
                    }
                }
            }
            __syncwarp();
            const int staged = min(stage_n[wv], STAGE);
            if (staged) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&n_pairs[b], staged);
                base = __shfl_sync(PB_FULL, base, 0);
                if (base + staged > pair_cap) {
                    if (lane == 0) atomicOr(fallback, 1);
                } else {
                    for (int k = lane; k < staged; k += 32) plist[base + k] = stage[wv][k];
                }
            }
            __syncwarp();
        }
    }
    if (lane == 0 && my_tokens) atomicAdd(tok_counter, my_tokens);
}

// thread per pair.  (A warp-cooperative form -- rows staged coalesced into a padded shared-memory tile, then a chain per
// lane -- was measured: 0.37 ms against 0.25 ms; staging the query per CTA costs more than the half-used sectors.)
__global__ void __launch_bounds__(128)
k_recheck_dots(const u64 *__restrict__ pairs, const int *__restrict__ n_pairs, int pair_cap, const float *__restrict__ Q,
               const int *__restrict__ q_off, const float *__restrict__ C, int dim, int rc_cap, int QS,
               uint32_t *__restrict__ exactmax) {
    const int b = blockIdx.y;
    const int n = min(n_pairs[b], pair_cap);
    const float *Qb = Q + (size_t)q_off[b] * dim;
    const u64 *plist = pairs + (size_t)b * pair_cap;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const u64 pr = plist[j];
        const uint32_t slot = (uint32_t)(pr >> 40), q = (uint32_t)(pr >> 32) & 255u, c = (uint32_t)pr;
        const float *qr = Qb + (size_t)q * dim, *cr = C + (size_t)c * dim;
        float s = 0.0f;
#pragma unroll 8
        for (int d0 = 0; d0 < dim; d0 += 4) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(qr + d0)), v = __ldg(reinterpret_cast<const float4 *>(cr + d0));
            s = __fmaf_rn(a.x, v.x, s);
            s = __fmaf_rn(a.y, v.y, s);
            s = __fmaf_rn(a.z, v.z, s);
            s = __fmaf_rn(a.w, v.w, s);
        }
        atomicMax(&exactmax[((size_t)b * rc_cap + slot) * QS + q], score_key_asc(s));
    }
}


__global__ void __launch_bounds__(256)
k_recheck_sum(uint32_t *__restrict__ exactmax, const int *__restrict__ q_off, int QS, const uint32_t *__restrict__ cand,
              long long cand_cap, const int *__restrict__ n_cand, int rc_cap, float *__restrict__ approx,
              u64 *__restrict__ keys, uint32_t doc_id_base) {
    const int b = blockIdx.y, lane = threadIdx.x & 31;
    const int nq = q_off[b + 1] - q_off[b];
    const int n = n_cand[b];
    for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += gridDim.x * (blockDim.x >> 5)) {
        uint32_t *row = exactmax + ((size_t)b * rc_cap + i) * QS;
        float score = 0.0f;  // score += max for q ascending, skipping rows without a finite maximum (search.rs:318-320)
        for (int qc = 0; i < rc_cap && qc < QS; qc += 32) {  // past rc_cap the query is flagged: a placeholder key
            const uint32_t mk = qc + lane < QS ? row[qc + lane] : 0u;
            if (qc + lane < QS) row[qc + lane] = 0u;
            const int lim = min(32, nq - qc);
            for (int qq = 0; qq < lim; ++qq) {
                const uint32_t kk = __shfl_sync(PB_FULL, mk, qq);
                if (kk) score = __fadd_rn(score, key_to_score(kk));
            }
        }
        if (lane == 0) {
            const uint32_t d = cand[(size_t)b * cand_cap + i];
            approx[(size_t)b * cand_cap + i] = score;
            keys[(size_t)b * cand_cap + i] = ((u64)(~score_key_asc(score)) << 32) | (d + doc_id_base);
        }
    }
}
