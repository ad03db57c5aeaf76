// Exact angular kNN over a SPARSE index: rows with a handful of non-zero buckets, which is what an index built
// from few junctions looks like (the reference's own fixture tests/tiny_intropolis.tsv: 1-3 non-zeros in 3000
// buckets, and thousands of rows parallel to each other).  On such data the tensor-core path is the wrong tool --
// thousands of rows tie inside any fp16 error band, so every candidate list overflows -- while the exact FP64
// distance of a (query, row) pair costs nnz(row) multiply-adds instead of D.  The distances computed here are
// BIT-IDENTICAL to the dense scan's (morna_angular_distances): skipping a zero entry skips adding +-0 to a sum,
// which never changes it, and the non-zero terms are added in the dense kernels' canonical order -- lane
// (col/4)%32 accumulates its terms by ascending column, then the 32 lane sums meet in the fixed xor-butterfly,
// emulated below on the few lanes that hold anything.  Replaces cosine_distance + the scan of exact_search_nn
// (morna.py:101-114, 697-712) for sparse indexes; the top-k selection is morna_select_topk as in morna_knn_exact.
#include <math.h>

#include "common.cuh"

namespace morna {

constexpr int kSparseMaxNnz = 16;        // rows with more non-zeros keep the index on the dense paths
constexpr int kSparseThreads = 256;

// qq with the canonical tree: one warp per query
__global__ void __launch_bounds__(kSparseThreads)
query_norms_kernel(const double *__restrict__ queries, int64_t nq, int64_t q_ld, int32_t dim, double *__restrict__ qq) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (kSparseThreads / 32) + (threadIdx.x >> 5);
    if (q >= nq) return;
    const double *src = queries + q * q_ld;
    double acc = 0.0;
    for (int c = lane; 4 * c < dim; c += 32) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const double a = 4 * c + t < dim ? src[4 * c + t] : 0.0;
            acc = fma(a, a, acc);
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) qq[q] = acc;
}

// The canonical sum of a row with more than three non-zeros: per-lane partial sums by ascending column, then the
// xor-butterfly emulated on the lanes that hold anything (rare rows; kept out of line so the common path stays lean).
__device__ __noinline__ double sparse_dot_generic(const int32_t *__restrict__ cols, const float *__restrict__ vals, int64_t e0,
                                                  int64_t e1, const double *__restrict__ qv) {
    int lane_of[kSparseMaxNnz];
    double sum_of[kSparseMaxNnz];
    int m = 0;
    for (int64_t e = e0; e < e1; ++e) {                      // ascending columns: each lane's terms in its own order
        const int col = cols[e];
        const int lane = (col >> 2) & 31;
        const double prod_a = (double)vals[e], prod_b = __ldg(qv + col);
        int j = 0;
        while (j < m && lane_of[j] != lane) ++j;
        if (j == m) { lane_of[m] = lane; sum_of[m] = 0.0; ++m; }
        sum_of[j] = fma(prod_a, prod_b, sum_of[j]);
    }
    // the butterfly v += shfl_xor(v, 16), 8, 4, 2, 1: after a step the lanes that differ only in that bit hold the
    // same value, so a lane class is its index with the bit cleared; x + 0 = x for the absent partner
#pragma unroll
    for (int bit = 16; bit > 0; bit >>= 1) {
        for (int i = 0; i < m; ++i) {
            for (int j = i + 1; j < m; ++j) {
                if ((lane_of[i] ^ lane_of[j]) == bit) {                     // processed bits are already cleared in both
                    sum_of[i] = sum_of[i] + sum_of[j];
                    lane_of[j] = lane_of[m - 1]; sum_of[j] = sum_of[m - 1]; --m;
                    break;
                }
            }
            lane_of[i] &= ~bit;
        }
    }
    return m > 0 ? sum_of[0] : 0.0;
}

constexpr int kSparseQT = 4;             // queries per thread: the row's entries are loaded once for all of them

// thread = (row, kSparseQT queries).  Rows with at most three non-zeros -- the common case -- follow a per-row PLAN made
// at index load (MornaSearch._build_csr): every entry adds into one of three accumulators (entries of one summation lane
// share an accumulator, in ascending column order) and the result is (a0 + a1) + a2, the order in which the butterfly
// meets these lanes (the two lanes whose indices differ in the highest "lowest differing bit" meet first).  plan bits:
// 2e..2e+1 = accumulator of entry e, 8..12 = nnz, 30 = generic row.
__global__ void __launch_bounds__(kSparseThreads)
sparse_distances_kernel(const int64_t *__restrict__ row_off, const int32_t *__restrict__ cols, const float *__restrict__ vals,
                        const int32_t *__restrict__ plan, const double *__restrict__ pp, int64_t n,
                        const double *__restrict__ queries, int64_t nq, int64_t q_ld, const double *__restrict__ qq,
                        double *__restrict__ dist, int64_t dist_ld) {
    const int64_t row = (int64_t)blockIdx.x * kSparseThreads + threadIdx.x;
    const int64_t q0 = (int64_t)blockIdx.y * kSparseQT;
    if (row >= n) return;
    const int pl = plan[row];
    const int64_t e0 = row_off[row];
    const double ppr = pp[row];
    if (pl & (1 << 30)) {
        const int64_t e1 = row_off[row + 1];
        for (int t = 0; t < kSparseQT && q0 + t < nq; ++t) {
            const double pq = sparse_dot_generic(cols, vals, e0, e1, queries + (q0 + t) * q_ld);
            dist[(q0 + t) * dist_ld + row] = angular_from_sums(ppr, qq[q0 + t], pq);
        }
        return;
    }
    const int nnz = (pl >> 8) & 31;
    int c[3] = {0, 0, 0};
    double v[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int e = 0; e < 3; ++e)
        if (e < nnz) { c[e] = cols[e0 + e]; v[e] = (double)vals[e0 + e]; }
#pragma unroll
    for (int t = 0; t < kSparseQT; ++t) {
        if (q0 + t >= nq) break;
        const double *qv = queries + (q0 + t) * q_ld;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
#pragma unroll
        for (int e = 0; e < 3; ++e) {
            if (e < nnz) {
                const double qe = __ldg(qv + c[e]);
                const int tgt = (pl >> (2 * e)) & 3;
                if (tgt == 0) a0 = fma(v[e], qe, a0);
                else if (tgt == 1) a1 = fma(v[e], qe, a1);
                else a2 = fma(v[e], qe, a2);
            }
        }
        const double pq = (a0 + a1) + a2;
        // pq == 0: 2 - 2*0/x = 2 whatever the norms are -- skip the division and the first square root
        dist[(q0 + t) * dist_ld + row] = pq == 0.0 ? sqrt(2.0) : angular_from_sums(ppr, qq[q0 + t], pq);
    }
}

// ---- exact top-k under massive ties ------------------------------------------------------------------------------
// One CTA per query over its n distances.  A sparse index has few distinct distance values per query (thousands of
// parallel rows), which defeats pivot-and-sort selection; a radix select does not care: the k-th smallest 64-bit key
// is found digit by digit (11 bits a pass, 2048-bin shared histogram, warp-aggregated increments), then one pass in
// DESCENDING row order keeps everything below it and, among the rows tied with it, the first `quota` met -- the highest
// ids, which is the reference's tie rule (morna.py:705-712: equal distances, later row first).  The k survivors are
// sorted under the full rule in shared memory.  Distances are >= 0 (or +inf), so their bit patterns order like the values.
constexpr int kRsThreads = 1024, kRsWarps = kRsThreads / 32;
constexpr int kRsBits = 11, kRsBins = 1 << kRsBits;
constexpr int kRsMaxK = 2048;

__global__ void __launch_bounds__(kRsThreads)
select_radix_kernel(const double *__restrict__ dist, int64_t n, int64_t dist_ld, int32_t id_base, int32_t k,
                    int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sd = reinterpret_cast<double *>(smem_raw);                 // [P] selected distances
    int *si = reinterpret_cast<int *>(sd + kRsMaxK);                   // [P] selected ids
    __shared__ unsigned int hist[kRsBins];
    __shared__ unsigned int warp_tot[kRsWarps];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_need, s_count, s_ties;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double *row = dist + (int64_t)blockIdx.x * dist_ld;
    int32_t *oi = out_ids + (int64_t)blockIdx.x * k;
    double *od = out_dist + (int64_t)blockIdx.x * k;
    const int kk = (int)min((int64_t)k, n);
    if (kk == 0) {
        for (int i = tid; i < k; i += kRsThreads) { oi[i] = -1; od[i] = INFINITY; }
        return;
    }
    __shared__ unsigned long long s_and, s_or;
    __shared__ int s_bin_count;
    if (tid == 0) { s_prefix = 0ull; s_need = kk; s_count = 0; s_ties = 0; }
    unsigned long long mask = 0ull;
    constexpr int kUnroll = 4;                                         // independent loads in flight per thread (the passes are L2-latency bound)
    for (int shift = 64 - kRsBits; ; shift -= kRsBits) {               // digits at bits 53, 42, 31, 20, 9 and the last 9 bits
        const int width = shift >= 0 ? kRsBits : kRsBits + shift;
        const int sh = shift >= 0 ? shift : 0;
        const unsigned int bins = 1u << width;
        for (int b = tid; b < kRsBins; b += kRsThreads) hist[b] = 0u;
        if (tid == 0) { s_and = ~0ull; s_or = 0ull; }
        __syncthreads();
        const unsigned long long prefix = s_prefix;
        unsigned long long my_and = ~0ull, my_or = 0ull;
        for (int64_t i0 = 0; i0 < n; i0 += kUnroll * kRsThreads) {
            unsigned long long key[kUnroll];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const int64_t i = i0 + u * kRsThreads + tid;
                key[u] = i < n ? (unsigned long long)__double_as_longlong(row[i]) : ~0ull;
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const int64_t i = i0 + u * kRsThreads + tid;
                unsigned int digit = 0xffffffffu;
                if (i < n && (key[u] & mask) == prefix) {
                    digit = (unsigned int)(key[u] >> sh) & (bins - 1u);
                    my_and &= key[u]; my_or |= key[u];
                }
                const unsigned int peers = __match_any_sync(kFull, digit);
                if (digit != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(&hist[digit], (unsigned int)__popc(peers));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            my_and &= __shfl_xor_sync(kFull, my_and, o);
            my_or |= __shfl_xor_sync(kFull, my_or, o);
        }
        if (lane == 0) { atomicAnd(&s_and, my_and); atomicOr(&s_or, my_or); }
        __syncthreads();
        // the bin in which the cumulative count reaches s_need: every thread owns two consecutive bins
        const unsigned int h0 = hist[2 * tid], h1 = hist[2 * tid + 1];
        unsigned int incl = h0 + h1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        unsigned int before = incl - (h0 + h1);
        for (int w = 0; w < warp; ++w) before += warp_tot[w];
        const unsigned int need = (unsigned int)s_need;
        const bool all_equal = s_and == s_or;                          // every key still matching the prefix is the same key
        const unsigned long long the_key = s_or;
        __syncthreads();                                               // everyone has read s_need / warp_tot / s_and / s_or
        if (all_equal) {                                               // thousands of exact ties: no need to walk the lower digits
            if (tid == 0) s_prefix = the_key;                          // (s_need stays: that many of the tied rows belong to the answer)
            mask = ~0ull;
            __syncthreads();
            break;
        }
        if (before < need && need <= before + h0 + h1) {
            const int bin = need <= before + h0 ? 2 * tid : 2 * tid + 1;
            s_need = (int)(need - (bin == 2 * tid ? before : before + h0));
            s_prefix = prefix | ((unsigned long long)bin << sh);
            s_bin_count = (int)(bin == 2 * tid ? h0 : h1);
        }
        mask |= (unsigned long long)(bins - 1u) << sh;
        __syncthreads();
        if (shift <= 0 || s_need == s_bin_count) break;                // every key with this prefix is wanted: lower digits do not matter
    }
    // keys are compared under `mask` from here on: either all 64 bits, or the prefix of a bin that is wanted whole
    const unsigned long long key_k = s_prefix;                         // the kk-th smallest key (under mask)
    const int quota = s_need;                                          // how many of the rows tied with it (under mask) belong to the answer
    // descending row order: everything below key_k, and the first `quota` ties met.  While ties are still wanted every
    // 1024-row step ranks its ties across the CTA (two barriers); thousands of rows tie in a sparse index, so the quota is
    // met within a step or two, and from then on only the (fewer than k) rows below key_k matter: no barriers, four
    // loads in flight.  (ncu of the one-loop version: half of the kernel's samples sat in the per-step prefix over the
    // 32 warp totals, executed for all 49 steps.)
    int64_t top = n;
    for (; top > 0 && s_ties < quota; top -= kRsThreads) {             // (s_ties is read between the barriers that follow its update)
        const int64_t i = top - 1 - tid;
        bool less = false, tie = false;
        double d = 0.0;
        if (i >= 0) {
            d = row[i];
            const unsigned long long key = (unsigned long long)__double_as_longlong(d) & mask;
            less = key < key_k; tie = key == key_k;
        }
        const unsigned int tie_mask = __ballot_sync(kFull, tie);
        if (lane == 0) warp_tot[warp] = __popc(tie_mask);
        __syncthreads();
        int tie_rank = s_ties + __popc(tie_mask & ((1u << lane) - 1u));
        int block_ties = 0;
        for (int w = 0; w < kRsWarps; ++w) { if (w < warp) tie_rank += warp_tot[w]; block_ties += warp_tot[w]; }
        const bool take = less || (tie && tie_rank < quota);
        const unsigned int take_mask = __ballot_sync(kFull, take);
        int base = 0;
        if (lane == 0 && take_mask) base = atomicAdd(&s_count, __popc(take_mask));
        base = __shfl_sync(kFull, base, 0);
        if (take) {
            const int at = base + __popc(take_mask & ((1u << lane) - 1u));
            if (at < kRsMaxK) { sd[at] = d; si[at] = id_base + (int)i; }
        }
        __syncthreads();
        if (tid == 0) s_ties += block_ties;
        __syncthreads();
    }
    for (; top > 0; top -= kUnroll * kRsThreads) {                     // the quota of ties is met: rows below key_k only
        double d[kUnroll];
        int64_t i[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            i[u] = top - 1 - (int64_t)u * kRsThreads - tid;
            d[u] = i[u] >= 0 ? row[i[u]] : INFINITY;
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const bool take = i[u] >= 0 && ((unsigned long long)__double_as_longlong(d[u]) & mask) < key_k;
            const unsigned int take_mask = __ballot_sync(kFull, take);
            if (take_mask == 0u) continue;
            int base = 0;
            if (lane == 0) base = atomicAdd(&s_count, __popc(take_mask));
            base = __shfl_sync(kFull, base, 0);
            if (take) {
                const int at = base + __popc(take_mask & ((1u << lane) - 1u));
                if (at < kRsMaxK) { sd[at] = d[u]; si[at] = id_base + (int)i[u]; }
            }
        }
    }
    __syncthreads();
    const int count = min(s_count, kRsMaxK);                           // == kk
    int P = 32;
    while (P < count) P <<= 1;
    for (int i = count + tid; i < P; i += kRsThreads) { sd[i] = INFINITY; si[i] = -1; }
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = tid; i < (P >> 1); i += kRsThreads) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const double dl = sd[lo], dh = sd[hi];
                const int il = si[lo], ih = si[hi];
                const bool swap = asc ? before(dh, ih, dl, il) : before(dl, il, dh, ih);
                if (swap) { sd[lo] = dh; sd[hi] = dl; si[lo] = ih; si[hi] = il; }
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < k; i += kRsThreads) {
        const bool ok = i < count && si[i] >= 0;
        oi[i] = ok ? si[i] : -1;
        od[i] = ok ? sd[i] : INFINITY;
    }
}

static int g_sparse_tile_mb = 1700;      // morna_debug_set_tuning key 35: MB of distance scratch per query tile
void set_sparse_tile_mb(int v) { g_sparse_tile_mb = v > 0 ? v : 1700; }

static int64_t sparse_query_tile(int64_t n, int64_t nq) {
    // Bytes of distance scratch per tile.  Measured at 50,000 rows x 4096 queries (scripts/sparse_probe.py, fixture-like /
    // 40-junction rows): 96 MB (251 queries, the passes hit in L2) 4.21 / 5.72 ms, 240 MB 3.35 / 4.43, 480 MB 3.07 / 4.00,
    // 960 MB 2.88 / 3.74, all queries in one tile (1.64 GB) 2.79 / 3.62 -- the selection kernel (one 1024-thread CTA per
    // query, two per SM) wants many waves per launch more than it wants L2 hits.  Several tiles are made equal.
    const int64_t budget = (int64_t)g_sparse_tile_mb << 20;
    int64_t t = budget / (8 * (n > 0 ? n : 1));
    if (t < 1) t = 1;
    if (t > 16384) t = 16384;
    if (t >= nq) return nq > 0 ? nq : 1;
    const int64_t tiles = (nq + t - 1) / t;
    return (nq + tiles - 1) / tiles;
}

}  // namespace morna

using namespace morna;

extern "C" int32_t morna_sparse_max_nnz(void) { return kSparseMaxNnz; }

extern "C" size_t morna_knn_exact_sparse_workspace_bytes(int64_t n, int64_t nq, int32_t k) {
    const int64_t tile = sparse_query_tile(n, nq);
    return align_up((size_t)tile * (size_t)(n > 0 ? n : 1) * sizeof(double), 256) + align_up((size_t)(nq > 0 ? nq : 1) * sizeof(double), 256) +
           morna_select_topk_workspace_bytes(n, tile, k) + 256;
}

extern "C" int morna_knn_exact_sparse(const int64_t *row_off, const int32_t *cols, const float *vals, const int32_t *plan,
                                      const double *pp, int64_t n, int32_t dim, int32_t id_base, const double *queries, int64_t nq,
                                      int64_t q_ld, int32_t k, int32_t *out_ids, double *out_dist, void *workspace,
                                      size_t workspace_bytes, void *stream) {
    return morna_knn_exact_sparse_excl(row_off, cols, vals, plan, pp, n, dim, id_base, queries, nq, q_ld, k, out_ids, out_dist,
                                       workspace, workspace_bytes, nullptr, nullptr, stream);
}

extern "C" int morna_knn_exact_sparse_excl(const int64_t *row_off, const int32_t *cols, const float *vals, const int32_t *plan,
                                           const double *pp, int64_t n, int32_t dim, int32_t id_base, const double *queries,
                                           int64_t nq, int64_t q_ld, int32_t k, int32_t *out_ids, double *out_dist, void *workspace,
                                           size_t workspace_bytes, const int32_t *row_group, const int32_t *query_group,
                                           void *stream) {
    if (!row_off || !cols || !vals || !plan || !pp || !queries || !out_ids || !out_dist || n <= 0 || nq < 0 || dim <= 0 || q_ld < dim || k <= 0 ||
        !row_group != !query_group)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (!workspace || workspace_bytes < morna_knn_exact_sparse_workspace_bytes(n, nq, k)) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    if (nq == 0) return MORNA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t tile = sparse_query_tile(n, nq);
    unsigned char *ws = (unsigned char *)workspace;
    double *dist = (double *)ws;
    const size_t dist_bytes = align_up((size_t)tile * (size_t)n * sizeof(double), 256);
    double *qq = (double *)(ws + dist_bytes);
    const size_t qq_bytes = align_up((size_t)nq * sizeof(double), 256);
    void *sel_ws = ws + dist_bytes + qq_bytes;
    const size_t sel_bytes = workspace_bytes - dist_bytes - qq_bytes;
    query_norms_kernel<<<(unsigned)((nq + kSparseThreads / 32 - 1) / (kSparseThreads / 32)), kSparseThreads, 0, s>>>(queries, nq, q_ld, dim, qq);
    MORNA_LAUNCH_CHECK();
    for (int64_t q0 = 0; q0 < nq; q0 += tile) {
        const int64_t cnt = nq - q0 < tile ? nq - q0 : tile;
        {                                                     // cnt <= 16384 queries per tile: grid.y stays small
            dim3 grid((unsigned)((n + kSparseThreads - 1) / kSparseThreads), (unsigned)((cnt + kSparseQT - 1) / kSparseQT));
            sparse_distances_kernel<<<grid, kSparseThreads, 0, s>>>(row_off, cols, vals, plan, pp, n, queries + q0 * q_ld, cnt, q_ld,
                                                                   qq + q0, dist, n);
            MORNA_LAUNCH_CHECK();
        }
        if (row_group) {
            const int rc = launch_mask_excluded(dist, n, n, cnt, row_group, query_group + q0, s);
            if (rc != MORNA_OK) return rc;
        }
        if (k <= kRsMaxK && n <= 0x7fffffff) {
            const size_t smem = (size_t)kRsMaxK * (sizeof(double) + sizeof(int));
            select_radix_kernel<<<(unsigned)cnt, kRsThreads, smem, s>>>(dist, n, n, id_base, k, out_ids + q0 * k, out_dist + q0 * k);
            MORNA_LAUNCH_CHECK();
            if (row_group) {
                const int rc = launch_pad_masked(out_ids + q0 * k, out_dist + q0 * k, cnt * k, s);
                if (rc != MORNA_OK) return rc;
            }
            continue;
        }
        for (int64_t y0 = 0; y0 < cnt; y0 += 65535) {
            const int64_t ny = cnt - y0 < 65535 ? cnt - y0 : 65535;
            int rc = morna_select_topk(dist + y0 * n, nullptr, n, n, id_base, ny, k, out_ids + (q0 + y0) * k, out_dist + (q0 + y0) * k,
                                       sel_ws, sel_bytes, stream);
            if (rc != MORNA_OK) return rc;
        }
        if (row_group) {
            const int rc = launch_pad_masked(out_ids + q0 * k, out_dist + q0 * k, cnt * k, s);
            if (rc != MORNA_OK) return rc;
        }
    }
    return MORNA_OK;
}
