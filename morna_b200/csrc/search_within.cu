// Within-group search, grouped FP64 route: each query's distances to the rows of its own group only, then one sort per
// query.  The rows are gathered through an id list (every group's rows contiguous in it), so many small per-query
// subsets are served in one pass instead of one full scan each.  Distances are the canonical sums of common.cuh (the
// lane/chunk order, FMA chain and butterfly of angular_distances_kernel), so every distance has the bits
// morna_angular_distances gives the same (row, query) pair.
#include <math.h>

#include "common.cuh"

namespace morna {

constexpr int kWithinQB = 8;                       // queries of one group per work item
constexpr int kWithinThreads = 512;
constexpr int kWithinWarps = kWithinThreads / kWarp;
constexpr int kWithinMaxSegment = 8192;            // rows of a group the selection sorts in shared memory
constexpr int kWithinSelectThreads = 256;

// Element e..e+3 of query t of the item: staged in shared memory (doubles, zero past dim), or read from global memory
// for wide --features (bounds-checked against dim, as angular_distances_wide_kernel does).  Same values either way.
template <bool kSmemQ>
__device__ __forceinline__ void query4(const double *qs, int64_t ld, const double *qsrc, int32_t dim, int e, double &x0,
                                       double &x1, double &x2, double &x3) {
    if (kSmemQ) {
        const double2 a = *reinterpret_cast<const double2 *>(qs + e), b = *reinterpret_cast<const double2 *>(qs + e + 2);
        x0 = a.x; x1 = a.y; x2 = b.x; x3 = b.y;
    } else {
        x0 = e < dim ? __ldg(qsrc + e) : 0.0; x1 = e + 1 < dim ? __ldg(qsrc + e + 1) : 0.0;
        x2 = e + 2 < dim ? __ldg(qsrc + e + 2) : 0.0; x3 = e + 3 < dim ? __ldg(qsrc + e + 3) : 0.0;
    }
}

// One CTA per work item {first query, query count (1..kWithinQB), first row, row count}: the item's queries (all of one
// group, consecutive in the call) against rows group_rows[first row ..+ row count) of that group, one warp per row.
// Query q's distances go to dist[seg_off[q] + (position in group_rows - row_begin[q])]; the row exclude_rows[q] (if
// any) gets +inf.
template <bool kSmemQ>
__global__ void __launch_bounds__(kWithinThreads, 1)
group_distances_kernel(const float *__restrict__ vectors, const double *__restrict__ pp, int64_t ld, int32_t dim,
                       const int32_t *__restrict__ group_rows, const double *__restrict__ queries, int64_t q_ld,
                       const int4 *__restrict__ items, const int64_t *__restrict__ seg_off,
                       const int32_t *__restrict__ row_begin, const int32_t *__restrict__ exclude_rows,
                       double *__restrict__ dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *qs = reinterpret_cast<double *>(smem_raw);          // [kWithinQB][ld] (kSmemQ)
    __shared__ double qq_s[kWithinQB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int4 it = items[blockIdx.x];
    const int q0 = it.x, qn = it.y, r0 = it.z, rn = it.w;
    const int chunks = (int)(ld >> 2);

    if (kSmemQ) {
        // only the item's qn queries: the slots past them feed accumulators that are never written out
        for (int64_t i = threadIdx.x; i < (int64_t)qn * ld; i += kWithinThreads) {
            const int qi = (int)(i / ld), c = (int)(i % ld);
            qs[i] = c < dim ? queries[(int64_t)(q0 + qi) * q_ld + c] : 0.0;
        }
        __syncthreads();
    }
    if (warp < qn) {          // qq with the canonical tree
        const double *qsrc = queries + (int64_t)(q0 + min(warp, qn - 1)) * q_ld;
        double acc = 0.0;
        for (int c = lane; c < chunks; c += 32) {
            double a0, a1, a2, a3;
            query4<kSmemQ>(qs + (int64_t)warp * ld, ld, qsrc, dim, 4 * c, a0, a1, a2, a3);
            acc = fma(a0, a0, acc); acc = fma(a1, a1, acc);
            acc = fma(a2, a2, acc); acc = fma(a3, a3, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) qq_s[warp] = acc;
    }
    __syncthreads();

    for (int i = warp; i < rn; i += kWithinWarps) {
        const int32_t row = group_rows[r0 + i];
        const float4 *src = reinterpret_cast<const float4 *>(vectors + (int64_t)row * ld);
        double acc[kWithinQB];
#pragma unroll
        for (int t = 0; t < kWithinQB; ++t) acc[t] = 0.0;
        int c = lane;
        // 4 independent 16-byte loads in flight per lane; per lane the chunks are still taken in increasing order (the
        // wide variant, whose query operands come from global memory as well, takes them one at a time: no spills)
        for (; kSmemQ && c + 96 < chunks; c += 128) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = ldg_stream_f4(src + c + 32 * u);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double a0 = v[u].x, a1 = v[u].y, a2 = v[u].z, a3 = v[u].w;
#pragma unroll
                for (int t = 0; t < kWithinQB; ++t) {
                    double x0, x1, x2, x3;
                    query4<kSmemQ>(qs + (int64_t)t * ld, ld, queries + (int64_t)(q0 + min(t, qn - 1)) * q_ld, dim,
                                   4 * (c + 32 * u), x0, x1, x2, x3);
                    acc[t] = fma(a0, x0, acc[t]); acc[t] = fma(a1, x1, acc[t]);
                    acc[t] = fma(a2, x2, acc[t]); acc[t] = fma(a3, x3, acc[t]);
                }
            }
        }
        for (; c < chunks; c += 32) {
            const float4 v = ldg_stream_f4(src + c);
            const double a0 = v.x, a1 = v.y, a2 = v.z, a3 = v.w;
#pragma unroll
            for (int t = 0; t < kWithinQB; ++t) {
                double x0, x1, x2, x3;
                query4<kSmemQ>(qs + (int64_t)t * ld, ld, queries + (int64_t)(q0 + min(t, qn - 1)) * q_ld, dim, 4 * c,
                               x0, x1, x2, x3);
                acc[t] = fma(a0, x0, acc[t]); acc[t] = fma(a1, x1, acc[t]);
                acc[t] = fma(a2, x2, acc[t]); acc[t] = fma(a3, x3, acc[t]);
            }
        }
        const double ppr = pp[row];
#pragma unroll
        for (int t = 0; t < kWithinQB; ++t) {
            const double pq = warp_sum(acc[t]);
            if (lane == 0 && t < qn) {
                const int q = q0 + t;
                const bool excluded = exclude_rows != nullptr && exclude_rows[q] == row;
                dist[seg_off[q] + (r0 + i - row_begin[q])] = excluded ? INFINITY : angular_from_sums(ppr, qq_s[t], pq);
            }
        }
    }
}

// One CTA per query j of the call, writing the result of output row out_slot[j].  Its segment (the distances to the
// rows of its group, at most kWithinMaxSegment) is sorted in shared memory under `before` with the row ids.
//   kMode 0: top-k -- the first k entries, +inf (excluded) and missing entries as id -1 / +inf
//   kMode 1: count -- entries with d <= r into counts[out_slot[j]] (no sort)
//   kMode 2: fill  -- the first out_offsets[s + 1] - out_offsets[s] sorted entries (the count pass's d <= r prefix)
template <int kMode>
__global__ void __launch_bounds__(kWithinSelectThreads)
group_select_kernel(const double *__restrict__ dist, const int64_t *__restrict__ seg_off,
                    const int32_t *__restrict__ row_begin, const int32_t *__restrict__ group_rows, int32_t id_base,
                    const int32_t *__restrict__ out_slot, int32_t k, double r, int64_t *__restrict__ counts,
                    const int64_t *__restrict__ out_offsets, int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int64_t j = blockIdx.x;
    const int64_t s0 = seg_off[j];
    const int L = (int)(seg_off[j + 1] - s0);
    const int64_t slot = out_slot[j];
    const double *dj = dist + s0;
    if (kMode == 1) {
        __shared__ int s_count;
        if (threadIdx.x == 0) s_count = 0;
        __syncthreads();
        int mine = 0;
        for (int i = threadIdx.x; i < L; i += kWithinSelectThreads) mine += dj[i] <= r ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(kFull, mine, o);
        if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&s_count, mine);
        __syncthreads();
        if (threadIdx.x == 0) counts[slot] = s_count;
        return;
    }
    int P = 1;
    while (P < L) P <<= 1;
    double *sd = reinterpret_cast<double *>(smem_raw);           // [P]
    int *si = reinterpret_cast<int *>(sd + P);                   // [P]
    const int32_t *rows = group_rows + row_begin[j];
    for (int i = threadIdx.x; i < P; i += kWithinSelectThreads) {
        sd[i] = i < L ? dj[i] : INFINITY;
        si[i] = i < L ? rows[i] : -1;
    }
    bitonic_sort_smem<true>(sd, si, P);
    if (kMode == 0) {
        for (int i = threadIdx.x; i < k; i += kWithinSelectThreads) {
            const bool ok = i < L && !isinf(sd[i]);
            out_ids[slot * k + i] = ok ? si[i] + id_base : -1;
            out_dist[slot * k + i] = ok ? sd[i] : INFINITY;
        }
    } else {
        const int64_t o = out_offsets[slot];
        const int cnt = (int)(out_offsets[slot + 1] - o);
        for (int i = threadIdx.x; i < cnt; i += kWithinSelectThreads) {
            out_ids[o + i] = si[i] + id_base;
            out_dist[o + i] = sd[i];
        }
    }
}

static int launch_group_distances(const float *vectors, const double *pp, int32_t dim, int64_t ld,
                                  const int32_t *group_rows, const double *queries, int64_t q_ld, const int32_t *items,
                                  int64_t n_items, const int64_t *seg_off, const int32_t *row_begin,
                                  const int32_t *exclude_rows, double *dist, cudaStream_t s) {
    if (n_items <= 0) return MORNA_OK;
    if (n_items > 0x7fffffff) return MORNA_ERR_INVALID_ARGUMENT;
    const size_t smem = (size_t)kWithinQB * ld * sizeof(double);
    const int4 *it = reinterpret_cast<const int4 *>(items);
    if (smem <= 200 * 1024) {
        auto kern = group_distances_kernel<true>;
        int rca = ensure_dynamic_smem((const void *)kern, smem);
        if (rca != MORNA_OK) return rca;
        kern<<<(unsigned)n_items, kWithinThreads, smem, s>>>(vectors, pp, ld, dim, group_rows, queries, q_ld, it, seg_off,
                                                            row_begin, exclude_rows, dist);
    } else {
        group_distances_kernel<false><<<(unsigned)n_items, kWithinThreads, 0, s>>>(
            vectors, pp, ld, dim, group_rows, queries, q_ld, it, seg_off, row_begin, exclude_rows, dist);
    }
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

template <int kMode>
static int launch_group_select(int64_t nq, int32_t max_segment, const double *dist, const int64_t *seg_off,
                               const int32_t *row_begin, const int32_t *group_rows, int32_t id_base,
                               const int32_t *out_slot, int32_t k, double r, int64_t *counts, const int64_t *out_offsets,
                               int32_t *out_ids, double *out_dist, cudaStream_t s) {
    if (nq <= 0) return MORNA_OK;
    if (nq > 0x7fffffff) return MORNA_ERR_INVALID_ARGUMENT;
    int P = 1;
    while (P < max_segment) P <<= 1;
    const size_t smem = kMode == 1 ? 0 : (size_t)P * (sizeof(double) + sizeof(int));
    auto kern = group_select_kernel<kMode>;
    if (smem > 48 * 1024) {
        int rca = ensure_dynamic_smem((const void *)kern, smem);
        if (rca != MORNA_OK) return rca;
    }
    kern<<<(unsigned)nq, kWithinSelectThreads, smem, s>>>(dist, seg_off, row_begin, group_rows, id_base, out_slot, k, r,
                                                          counts, out_offsets, out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

static bool within_args_ok(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                           const int32_t *group_rows, const double *queries, int64_t nq, int64_t q_ld, const int32_t *items,
                           int64_t n_items, const int64_t *seg_off, const int32_t *row_begin, int32_t max_segment,
                           const int32_t *out_slot) {
    return vectors && pp && group_rows && queries && items && seg_off && row_begin && out_slot && n > 0 && nq >= 0 &&
           n_items >= 0 && dim > 0 && ld >= dim && !(ld & 3) && q_ld >= dim && max_segment >= 0 &&
           max_segment <= kWithinMaxSegment;
}

}  // namespace morna

using namespace morna;

extern "C" size_t morna_within_group_workspace_bytes(int64_t total) {
    return align_up((size_t)(total > 0 ? total : 1) * sizeof(double), 256);
}

extern "C" int morna_within_group_topk(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                       int32_t id_base, const int32_t *group_rows, const double *queries, int64_t nq,
                                       int64_t q_ld, const int32_t *items, int64_t n_items, const int64_t *seg_off,
                                       int64_t total, const int32_t *row_begin, int32_t max_segment,
                                       const int32_t *exclude_rows, const int32_t *out_slot, int32_t k, int32_t *out_ids, double *out_dist,
                                       void *workspace, size_t workspace_bytes, void *stream) {
    if (!within_args_ok(vectors, pp, n, dim, ld, group_rows, queries, nq, q_ld, items, n_items, seg_off, row_begin,
                        max_segment, out_slot) || total < 0 || k <= 0 || !out_ids || !out_dist || !workspace)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (workspace_bytes < morna_within_group_workspace_bytes(total)) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    double *dist = (double *)workspace;
    int rc = launch_group_distances(vectors, pp, dim, ld, group_rows, queries, q_ld, items, n_items, seg_off, row_begin,
                                    exclude_rows, dist, s);
    if (rc != MORNA_OK) return rc;
    return launch_group_select<0>(nq, max_segment, dist, seg_off, row_begin, group_rows, id_base, out_slot, k, 0.0,
                                  nullptr, nullptr, out_ids, out_dist, s);
}

extern "C" int morna_within_group_range_count(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                              const int32_t *group_rows, const double *queries, int64_t nq, int64_t q_ld,
                                              const int32_t *items, int64_t n_items, const int64_t *seg_off,
                                              int64_t total, const int32_t *row_begin, int32_t max_segment,
                                              const int32_t *exclude_rows,
                                              const int32_t *out_slot, double max_distance, int64_t *counts,
                                              void *workspace, size_t workspace_bytes, void *stream) {
    if (!within_args_ok(vectors, pp, n, dim, ld, group_rows, queries, nq, q_ld, items, n_items, seg_off, row_begin,
                        max_segment, out_slot) || total < 0 || !counts || !workspace || !(max_distance >= 0.0) || isinf(max_distance))
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (workspace_bytes < morna_within_group_workspace_bytes(total)) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    double *dist = (double *)workspace;
    int rc = launch_group_distances(vectors, pp, dim, ld, group_rows, queries, q_ld, items, n_items, seg_off, row_begin,
                                    exclude_rows, dist, s);
    if (rc != MORNA_OK) return rc;
    return launch_group_select<1>(nq, max_segment, dist, seg_off, row_begin, group_rows, 0, out_slot, 0, max_distance,
                                  counts, nullptr, nullptr, nullptr, s);
}

extern "C" int morna_within_group_range_fill(int64_t nq, const int32_t *group_rows, int32_t id_base,
                                             const int64_t *seg_off, int64_t total, const int32_t *row_begin,
                                             int32_t max_segment, const int32_t *out_slot, const int64_t *out_offsets, int32_t *out_ids,
                                             double *out_dist, const void *workspace, size_t workspace_bytes,
                                             void *stream) {
    if (!group_rows || !seg_off || !row_begin || !out_slot || !out_offsets || !out_ids || !out_dist || !workspace ||
        nq < 0 || max_segment < 0 || max_segment > kWithinMaxSegment)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < morna_within_group_workspace_bytes(total)) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    return launch_group_select<2>(nq, max_segment, (const double *)workspace, seg_off, row_begin, group_rows, id_base,
                                  out_slot, 0, 0.0, nullptr, out_offsets, out_ids, out_dist, (cudaStream_t)stream);
}
