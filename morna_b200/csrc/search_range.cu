// Exact range search, FP64 route: every row within a distance R of each query, from the distance scan of
// morna_knn_exact (morna_angular_distances: the canonical sums, so the distances equal every other path's bit for bit).
// It answers what the tensor-core route (morna_range_batched) does not take: small batches, queries whose first-pass
// lists overflowed or whose values reach 2^127, sparse indexes whose parallel rows tie by the thousand, and blocks of
// more than 2^24 rows.
//
// Cost: the scan is HBM-bound at 4*n*ld bytes per group of four queries, and the fill call runs it a second time
// rather than keep n distances per query between the calls.  Each query tile writes n doubles per query to the
// scratch and reads them back once per call; the fill then sorts 12 bytes per match (segmented radix sort over the
// 64 key bits, about 2x the list in extra scratch).
//
// morna_merge_sorted_csr, at the end, merges the per-rank lists of the rows-sharded range search (morna_b200/dist.py).
#include <math.h>

#include <cub/block/block_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include "common.cuh"

namespace morna {

constexpr int kRangeCountThreads = 256;
constexpr int kRangeCompactThreads = 1024;

// queries per tile: 256 MB of distance scratch, as morna_knn_exact
static int64_t range_query_tile(int64_t n, int64_t nq) {
    const int64_t budget = (int64_t)256 << 20;
    int64_t t = budget / (8 * (n > 0 ? n : 1));
    if (t < 4) t = 4;
    t = t / 4 * 4;
    if (t > 16384) t = 16384;
    if (t > nq) t = nq;
    return t > 0 ? t : 1;
}

// one CTA per query: rows of the tile's distance row with d <= R
__global__ void __launch_bounds__(kRangeCountThreads)
range_count_kernel(const double *__restrict__ dist, int64_t n, double R, int32_t *__restrict__ counts) {
    __shared__ int s_warp[kRangeCountThreads / 32];
    const double *dq = dist + (int64_t)blockIdx.x * n;
    int c = 0;
    for (int64_t i = threadIdx.x; i < n; i += kRangeCountThreads) c += dq[i] <= R;
    c = __reduce_add_sync(kFull, c);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kRangeCountThreads / 32; ++w) t += s_warp[w];
        counts[blockIdx.x] = t;
    }
}

// one CTA per query: its matches in DESCENDING row order, written to [offsets[q], offsets[q+1]) -- the stable sort by
// distance afterwards then leaves equal distances id-descending, the reference order
__global__ void __launch_bounds__(kRangeCompactThreads)
range_compact_kernel(const double *__restrict__ dist, int64_t n, double R, int32_t id_base, const int64_t *__restrict__ offsets,
                     int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    using Scan = cub::BlockScan<int, kRangeCompactThreads>;
    __shared__ typename Scan::TempStorage tmp;
    const double *dq = dist + (int64_t)blockIdx.x * n;
    const int64_t o = offsets[blockIdx.x], room = offsets[blockIdx.x + 1] - o;
    int64_t done = 0;
    for (int64_t base = 0; base < n && done < room; base += kRangeCompactThreads) {
        const int64_t row = n - 1 - (base + threadIdx.x);
        double d = 0.0;
        int flag = 0;
        if (row >= 0) { d = dq[row]; flag = d <= R; }
        int pos, agg;
        Scan(tmp).ExclusiveSum(flag, pos, agg);
        if (flag && done + pos < room) { out_ids[o + done + pos] = id_base + (int32_t)row; out_dist[o + done + pos] = d; }
        done += agg;
        __syncthreads();                                  // tmp is reused by the next chunk's scan
    }
}

struct RangeExactWs { size_t dist, keys, vals, cub, cub_bytes, total; int64_t tile; };

static RangeExactWs range_exact_layout(int64_t n, int64_t nq, int64_t total) {
    RangeExactWs w{};
    w.tile = range_query_tile(n, nq);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off += align_up(bytes, 256); return at; };
    w.dist = take((size_t)w.tile * (size_t)(n > 0 ? n : 1) * sizeof(double));
    if (total > 0) {
        w.keys = take((size_t)total * sizeof(double));
        w.vals = take((size_t)total * sizeof(int32_t));
        cub::DoubleBuffer<double> kb(nullptr, nullptr);
        cub::DoubleBuffer<int32_t> vb(nullptr, nullptr);
        size_t bytes = 0;
        cub::DeviceSegmentedRadixSort::SortPairs(nullptr, bytes, kb, vb, (int)total, (int)(nq > 0 ? nq : 1),
                                                 (const int64_t *)nullptr, (const int64_t *)nullptr);
        w.cub_bytes = bytes;
        w.cub = take(bytes);
    }
    w.total = off + 256;
    return w;
}

static bool range_args_ok(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld, const double *queries,
                          int64_t nq, int64_t q_ld, double R) {
    return vectors && pp && queries && n > 0 && nq >= 0 && dim > 0 && ld >= dim && !(ld & 3) && q_ld >= dim && n <= INT32_MAX &&
           R >= 0.0 && !isinf(R);
}

// Merge of the rows-sharded range search: one thread per slot of the all-gathered buffer.  A slot past its rank's last
// entry is padding.  The entry finds its query by binary search in its rank's offsets, then its output position as its
// index in its own list plus, for every other rank, how many of that rank's entries for the query come before it
// (binary search in global memory).  Lists of any length: nothing is staged in shared memory.
constexpr int kMergeCsrThreads = 256;

__global__ void __launch_bounds__(kMergeCsrThreads)
merge_sorted_csr_kernel(const unsigned char *__restrict__ gathered, int32_t n_lists, int64_t nq, int64_t cap,
                        const int64_t *__restrict__ rank_offsets, const int64_t *__restrict__ out_offsets,
                        int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    const int64_t t = (int64_t)blockIdx.x * kMergeCsrThreads + threadIdx.x;
    if (t >= (int64_t)n_lists * cap) return;
    const int g = (int)(t / cap);
    const int64_t e = t - (int64_t)g * cap;
    const int64_t *off = rank_offsets + (int64_t)g * (nq + 1);
    if (e >= off[nq]) return;
    int64_t lo = 0, hi = nq;                                   // the query j with off[j] <= e < off[j + 1]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (off[mid] <= e) lo = mid; else hi = mid;
    }
    const int64_t j = lo;
    const size_t rank_bytes = (size_t)cap * 12;
    const double *dg = reinterpret_cast<const double *>(gathered + (size_t)g * rank_bytes);
    const int32_t *ig = reinterpret_cast<const int32_t *>(gathered + (size_t)g * rank_bytes + (size_t)cap * 8);
    const double d = dg[e];
    const int32_t id = ig[e];
    int64_t pos = out_offsets[j] + (e - off[j]);
    for (int h = 0; h < n_lists; ++h) {
        if (h == g) continue;
        const int64_t *oh = rank_offsets + (int64_t)h * (nq + 1);
        const double *dh = reinterpret_cast<const double *>(gathered + (size_t)h * rank_bytes);
        const int32_t *ih = reinterpret_cast<const int32_t *>(gathered + (size_t)h * rank_bytes + (size_t)cap * 8);
        int64_t a = oh[j], b = oh[j + 1];                      // first entry of rank h's list that does NOT come before
        const int64_t start = a;
        while (a < b) {
            const int64_t mid = (a + b) >> 1;
            if (before(dh[mid], ih[mid], d, id)) a = mid + 1; else b = mid;
        }
        pos += a - start;
    }
    out_ids[pos] = id;
    out_dist[pos] = d;
}

}  // namespace morna

using namespace morna;

extern "C" size_t morna_range_exact_workspace_bytes(int64_t n, int64_t nq, int64_t total) {
    if (total < 0 || total > INT32_MAX) return 0;
    return range_exact_layout(n, nq, total).total;
}

extern "C" int morna_range_exact_count(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                       const double *queries, int64_t nq, int64_t q_ld, double max_distance, int32_t *counts,
                                       void *workspace, size_t workspace_bytes, void *stream) {
    return morna_range_exact_count_excl(vectors, pp, n, dim, ld, queries, nq, q_ld, max_distance, counts, workspace, workspace_bytes,
                                        nullptr, nullptr, stream);
}

// The count and fill passes run the same mask on the same distances, so counts and lists agree.
extern "C" int morna_range_exact_count_excl(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                            const double *queries, int64_t nq, int64_t q_ld, double max_distance, int32_t *counts,
                                            void *workspace, size_t workspace_bytes, const int32_t *row_group,
                                            const int32_t *query_group, void *stream) {
    if (!range_args_ok(vectors, pp, n, dim, ld, queries, nq, q_ld, max_distance) || !counts || !row_group != !query_group)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    const RangeExactWs w = range_exact_layout(n, nq, 0);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    double *dist = (double *)((unsigned char *)workspace + w.dist);
    for (int64_t q0 = 0; q0 < nq; q0 += w.tile) {
        const int64_t cnt = std::min<int64_t>(w.tile, nq - q0);
        int rc = morna_angular_distances(vectors, pp, n, dim, ld, queries + q0 * q_ld, cnt, q_ld, dist, n, stream);
        if (rc != MORNA_OK) return rc;
        if (row_group && (rc = launch_mask_excluded(dist, n, n, cnt, row_group, query_group + q0, s)) != MORNA_OK) return rc;
        range_count_kernel<<<(unsigned)cnt, kRangeCountThreads, 0, s>>>(dist, n, max_distance, counts + q0);
        MORNA_LAUNCH_CHECK();
    }
    return MORNA_OK;
}

extern "C" int morna_range_exact_fill(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                                      const double *queries, int64_t nq, int64_t q_ld, double max_distance, const int64_t *offsets,
                                      int64_t total, int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                                      void *stream) {
    return morna_range_exact_fill_excl(vectors, pp, n, dim, ld, id_base, queries, nq, q_ld, max_distance, offsets, total, out_ids,
                                       out_dist, workspace, workspace_bytes, nullptr, nullptr, stream);
}

extern "C" int morna_range_exact_fill_excl(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                                           const double *queries, int64_t nq, int64_t q_ld, double max_distance, const int64_t *offsets,
                                           int64_t total, int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                                           const int32_t *row_group, const int32_t *query_group, void *stream) {
    if (!range_args_ok(vectors, pp, n, dim, ld, queries, nq, q_ld, max_distance) || !offsets || !out_ids || !out_dist ||
        total < 0 || total > INT32_MAX || nq > INT32_MAX || !row_group != !query_group)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0 || total == 0) return MORNA_OK;
    const RangeExactWs w = range_exact_layout(n, nq, total);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace;
    double *dist = (double *)(ws + w.dist);
    for (int64_t q0 = 0; q0 < nq; q0 += w.tile) {
        const int64_t cnt = std::min<int64_t>(w.tile, nq - q0);
        int rc = morna_angular_distances(vectors, pp, n, dim, ld, queries + q0 * q_ld, cnt, q_ld, dist, n, stream);
        if (rc != MORNA_OK) return rc;
        if (row_group && (rc = launch_mask_excluded(dist, n, n, cnt, row_group, query_group + q0, s)) != MORNA_OK) return rc;
        range_compact_kernel<<<(unsigned)cnt, kRangeCompactThreads, 0, s>>>(dist, n, max_distance, id_base, offsets + q0,
                                                                           out_ids, out_dist);
        MORNA_LAUNCH_CHECK();
    }
    // distances are >= +0, so the radix order of the keys is their numeric order; the sort is stable
    cub::DoubleBuffer<double> kb(out_dist, (double *)(ws + w.keys));
    cub::DoubleBuffer<int32_t> vb(out_ids, (int32_t *)(ws + w.vals));
    size_t cub_bytes = w.cub_bytes;
    MORNA_CUDA_TRY(cub::DeviceSegmentedRadixSort::SortPairs(ws + w.cub, cub_bytes, kb, vb, (int)total, (int)nq, offsets,
                                                            offsets + 1, 0, 64, s));
    if (kb.Current() != out_dist) {
        MORNA_CUDA_TRY(cudaMemcpyAsync(out_dist, kb.Current(), (size_t)total * sizeof(double), cudaMemcpyDeviceToDevice, s));
        MORNA_CUDA_TRY(cudaMemcpyAsync(out_ids, vb.Current(), (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    }
    return MORNA_OK;
}

extern "C" int morna_merge_sorted_csr(const void *gathered, int32_t n_lists, int64_t nq, int64_t cap, const int64_t *rank_offsets,
                                      const int64_t *out_offsets, int64_t total, int32_t *out_ids, double *out_dist,
                                      void *stream) {
    if (n_lists <= 0 || nq < 0 || cap < 0 || (cap & 1) || total < 0 || total > (int64_t)n_lists * cap)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0 || total == 0) return MORNA_OK;
    if (!gathered || ((uintptr_t)gathered & 7) || !rank_offsets || !out_offsets || !out_ids || !out_dist)
        return MORNA_ERR_INVALID_ARGUMENT;
    const int64_t slots = (int64_t)n_lists * cap;
    const int64_t blocks = (slots + kMergeCsrThreads - 1) / kMergeCsrThreads;
    if (blocks > INT32_MAX) return MORNA_ERR_INVALID_ARGUMENT;
    merge_sorted_csr_kernel<<<(unsigned)blocks, kMergeCsrThreads, 0, (cudaStream_t)stream>>>(
        (const unsigned char *)gathered, n_lists, nq, cap, rank_offsets, out_offsets, out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}
