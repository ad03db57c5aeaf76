// Exact angular kNN: row norms, FP64-accumulated distance scan, exact top-k select.
// Replaces cosine_distance (morna.py:101-114) and the scan/insert loop of
// exact_search_nn (morna.py:697-712).
#include <math.h>

#include "common.cuh"

namespace morna {

// ------------------------------------------------------------------ row norms
constexpr int kScanThreads = 256;
constexpr int kScanWarps = kScanThreads / kWarp;

__global__ void __launch_bounds__(kScanThreads)
row_norms_kernel(const float *__restrict__ vectors, int64_t n, int64_t ld, double *__restrict__ pp) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * kScanWarps;
    const int chunks = (int)(ld >> 2);
    for (int64_t row = (int64_t)blockIdx.x * kScanWarps + (threadIdx.x >> 5); row < n; row += warps_total) {
        const float4 *src = reinterpret_cast<const float4 *>(vectors + row * ld);
        double acc = 0.0;
        for (int c = lane; c < chunks; c += 32) {
            float4 v = ldg_stream_f4(src + c);
            double a0 = v.x, a1 = v.y, a2 = v.z, a3 = v.w;
            acc = fma(a0, a0, acc); acc = fma(a1, a1, acc);
            acc = fma(a2, a2, acc); acc = fma(a3, a3, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) pp[row] = acc;
    }
}

// ------------------------------------------------------------------ distance scan
// One warp per stored row, QB queries per CTA held in shared memory as doubles.
// HBM-bound for QB == 1 (4*n*ld bytes per query); QB == 4 reuses each row load.
template <int QB>
__global__ void __launch_bounds__(kScanThreads)
angular_distances_kernel(const float *__restrict__ vectors, const double *__restrict__ pp, int64_t n,
                         int64_t ld, const double *__restrict__ queries, int64_t nq, int64_t q_ld,
                         int32_t dim, double *__restrict__ dist, int64_t dist_ld) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *qs = reinterpret_cast<double *>(smem_raw);          // [QB][ld]
    __shared__ double qq_s[QB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t q0 = (int64_t)blockIdx.y * QB;
    const int chunks = (int)(ld >> 2);

    for (int64_t i = threadIdx.x; i < (int64_t)QB * ld; i += kScanThreads) {
        int qi = (int)(i / ld), c = (int)(i % ld);
        double v = 0.0;
        if (q0 + qi < nq && c < dim) v = queries[(q0 + qi) * q_ld + c];
        qs[i] = v;
    }
    __syncthreads();
    if (warp < QB) {   // qq with the canonical tree
        const double *q = qs + (int64_t)warp * ld;
        double acc = 0.0;
        for (int c = lane; c < chunks; c += 32) {
            double2 a = *reinterpret_cast<const double2 *>(q + 4 * c);
            double2 b = *reinterpret_cast<const double2 *>(q + 4 * c + 2);
            acc = fma(a.x, a.x, acc); acc = fma(a.y, a.y, acc);
            acc = fma(b.x, b.x, acc); acc = fma(b.y, b.y, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) qq_s[warp] = acc;
    }
    __syncthreads();

    const int64_t warps_total = (int64_t)gridDim.x * kScanWarps;
    for (int64_t row = (int64_t)blockIdx.x * kScanWarps + warp; row < n; row += warps_total) {
        const float4 *src = reinterpret_cast<const float4 *>(vectors + row * ld);
        double acc[QB];
#pragma unroll
        for (int t = 0; t < QB; ++t) acc[t] = 0.0;
        int c = lane;
        // 4 independent 16-byte loads in flight per lane
        for (; c + 96 < chunks; c += 128) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = ldg_stream_f4(src + c + 32 * u);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                double a0 = v[u].x, a1 = v[u].y, a2 = v[u].z, a3 = v[u].w;
#pragma unroll
                for (int t = 0; t < QB; ++t) {
                    const double *q = qs + (int64_t)t * ld + 4 * (c + 32 * u);
                    double2 qa = *reinterpret_cast<const double2 *>(q);
                    double2 qb = *reinterpret_cast<const double2 *>(q + 2);
                    acc[t] = fma(a0, qa.x, acc[t]); acc[t] = fma(a1, qa.y, acc[t]);
                    acc[t] = fma(a2, qb.x, acc[t]); acc[t] = fma(a3, qb.y, acc[t]);
                }
            }
        }
        for (; c < chunks; c += 32) {
            float4 v = ldg_stream_f4(src + c);
            double a0 = v.x, a1 = v.y, a2 = v.z, a3 = v.w;
#pragma unroll
            for (int t = 0; t < QB; ++t) {
                const double *q = qs + (int64_t)t * ld + 4 * c;
                double2 qa = *reinterpret_cast<const double2 *>(q);
                double2 qb = *reinterpret_cast<const double2 *>(q + 2);
                acc[t] = fma(a0, qa.x, acc[t]); acc[t] = fma(a1, qa.y, acc[t]);
                acc[t] = fma(a2, qb.x, acc[t]); acc[t] = fma(a3, qb.y, acc[t]);
            }
        }
        const double ppr = pp[row];
#pragma unroll
        for (int t = 0; t < QB; ++t) {
            double pq = warp_sum(acc[t]);
            if (lane == 0 && q0 + t < nq)
                dist[(q0 + t) * dist_ld + row] = angular_from_sums(ppr, qq_s[t], pq);
        }
    }
}

// ------------------------------------------------------------------ exact top-k select
constexpr int kSelThreads = 1024;
constexpr int kSelItems = 8;
constexpr int kSelChunk = kSelThreads * kSelItems;   // 8192 keys per CTA
constexpr int kSelCap = 1024;                         // survivors the fast path sorts
constexpr int kSelMaxK = 2048;

// bitonic sort of P (power of two) (key,id) pairs in shared memory under `before`
template <bool kWithIds>
__device__ void bitonic_sort_smem(double *sd, int *si, int P) {
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < (P >> 1); i += blockDim.x) {
                int lo = 2 * i - (i & (stride - 1));
                int hi = lo + stride;
                bool asc = (lo & size) == 0;
                double dl = sd[lo], dh = sd[hi];
                int il = kWithIds ? si[lo] : 0, ih = kWithIds ? si[hi] : 0;
                bool hi_first = kWithIds ? before(dh, ih, dl, il) : (dh < dl);
                bool lo_first = kWithIds ? before(dl, il, dh, ih) : (dl < dh);
                bool swap = asc ? hi_first : lo_first;
                if (swap) {
                    sd[lo] = dh; sd[hi] = dl;
                    if (kWithIds) { si[lo] = ih; si[hi] = il; }
                }
            }
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kSelThreads)
select_topk_kernel(const double *__restrict__ keys, const int32_t *__restrict__ ids, int64_t n,
                   int64_t key_ld, int32_t id_base, int32_t k, int32_t *__restrict__ out_ids,
                   double *__restrict__ out_dist, int64_t out_q_stride) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sd = reinterpret_cast<double *>(smem_raw);            // [kSelChunk]
    int *si = reinterpret_cast<int *>(sd + kSelChunk);            // [kSelChunk]
    __shared__ int s_count;
    __shared__ double s_pivot;

    const int tid = threadIdx.x;
    const int64_t q = blockIdx.y;
    const int64_t base = (int64_t)blockIdx.x * kSelChunk;
    const int m = (int)min((int64_t)kSelChunk, n - base);
    const int kk = min(k, m);
    const double *kq = keys + q * key_ld + base;
    const int32_t *iq = ids ? ids + q * key_ld + base : nullptr;
    int32_t *oi = out_ids + q * out_q_stride + (int64_t)blockIdx.x * k;
    double *od = out_dist + q * out_q_stride + (int64_t)blockIdx.x * k;
    const double inf = INFINITY;

    double d[kSelItems];
    int id[kSelItems];
#pragma unroll
    for (int j = 0; j < kSelItems; ++j) {
        int idx = j * kSelThreads + tid;
        bool ok = idx < m;
        d[j] = ok ? kq[idx] : inf;
        id[j] = ok ? (iq ? iq[idx] : id_base + (int32_t)(base + idx)) : -1;
        if (ok && id[j] < 0) d[j] = inf;      // padding entries from a previous level
    }

    int P;            // sorted prefix lives in sd/si[0..P)
    bool done = false;
    if (m <= kSelCap) {
        sd[tid] = d[0]; si[tid] = id[0];
        P = kSelCap;
        done = true;
    } else {
        // pivot from a strided sample of 1024 keys
        double sv = kq[(int)(((int64_t)tid * m) / kSelThreads)];
        sd[tid] = sv;
        if (tid == 0) s_count = 0;
        bitonic_sort_smem<false>(sd, si, kSelThreads);
        if (tid == 0) {
            double f = (double)kSelThreads / (double)m;
            double want = kk * f;
            int r = (int)(want + 4.0 * sqrt(want) + 4.0);
            s_pivot = sd[min(r, kSelThreads - 1)];
        }
        __syncthreads();
        const double pivot = s_pivot;
        int mine = 0;
#pragma unroll
        for (int j = 0; j < kSelItems; ++j) mine += (d[j] <= pivot) ? 1 : 0;
        int wsum = mine;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(kFull, wsum, o);
        if ((tid & 31) == 0 && wsum) atomicAdd(&s_count, wsum);
        __syncthreads();
        const int total = s_count;
        __syncthreads();
        if (total >= kk && total <= kSelCap) {
            if (tid == 0) s_count = 0;
            sd[tid] = inf; si[tid] = -1;
            __syncthreads();
#pragma unroll
            for (int j = 0; j < kSelItems; ++j) {
                if (d[j] <= pivot) {
                    int at = atomicAdd(&s_count, 1);
                    sd[at] = d[j]; si[at] = id[j];
                }
            }
            P = kSelCap;
            done = true;
        }
    }
    if (!done) {   // heavy ties or an unlucky pivot: sort the whole chunk
#pragma unroll
        for (int j = 0; j < kSelItems; ++j) {
            sd[j * kSelThreads + tid] = d[j];
            si[j * kSelThreads + tid] = id[j];
        }
        P = kSelChunk;
    }
    bitonic_sort_smem<true>(sd, si, P);
    for (int i = tid; i < k; i += kSelThreads) {
        bool ok = i < kk && si[i] >= 0;
        oi[i] = ok ? si[i] : -1;
        od[i] = ok ? sd[i] : inf;
    }
}

static int sm_count_cached() { return sm_count_current(); }

// grid (row blocks, query): +inf for every row of the query's group (nothing for a query labelled < 0)
__global__ void __launch_bounds__(256)
mask_excluded_kernel(double *__restrict__ dist, int64_t n, int64_t dist_ld, const int32_t *__restrict__ row_group,
                     const int32_t *__restrict__ query_group) {
    const int64_t q = blockIdx.y;
    const int32_t g = query_group[q];
    if (g < 0) return;
    double *dq = dist + q * dist_ld;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
        if (row_group[i] == g) dq[i] = INFINITY;
}

__global__ void pad_masked_kernel(int32_t *__restrict__ ids, const double *__restrict__ dist, int64_t total) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < total && isinf(dist[i])) ids[i] = -1;
}

int launch_mask_excluded(double *dist, int64_t n, int64_t dist_ld, int64_t nq, const int32_t *row_group,
                         const int32_t *query_group, cudaStream_t s) {
    if (n <= 0 || nq <= 0) return MORNA_OK;
    for (int64_t q0 = 0; q0 < nq; q0 += 65535) {
        const int64_t cnt = std::min<int64_t>(nq - q0, 65535);
        int64_t bx = (n + 255) / 256, cap = ((int64_t)sm_count_cached() * 16 + cnt - 1) / cnt;
        if (bx > cap) bx = cap;
        mask_excluded_kernel<<<dim3((unsigned)bx, (unsigned)cnt), 256, 0, s>>>(dist + q0 * dist_ld, n, dist_ld, row_group,
                                                                              query_group + q0);
        MORNA_LAUNCH_CHECK();
    }
    return MORNA_OK;
}

int launch_pad_masked(int32_t *ids, const double *dist, int64_t total, cudaStream_t s) {
    if (total <= 0) return MORNA_OK;
    pad_masked_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(ids, dist, total);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

static size_t select_level_entries(int64_t n, int32_t k) {
    int64_t chunks = (n + kSelChunk - 1) / kSelChunk;
    return chunks > 1 ? (size_t)chunks * k : 0;
}

}  // namespace morna

using namespace morna;

extern "C" int morna_row_norms(const float *vectors, int64_t n, int32_t dim, int64_t ld, double *pp,
                               void *stream) {
    if (!vectors || !pp || n < 0 || dim <= 0 || ld < dim || (ld & 3)) return MORNA_ERR_INVALID_ARGUMENT;
    if (n == 0) return MORNA_OK;
    int64_t blocks = (n + kScanWarps - 1) / kScanWarps;
    int64_t cap = (int64_t)sm_count_cached() * 8;
    if (blocks > cap) blocks = cap;
    row_norms_kernel<<<(unsigned)blocks, kScanThreads, 0, (cudaStream_t)stream>>>(vectors, n, ld, pp);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

// Wide --features (a staged query of ld doubles no longer fits shared memory, ld * 8 > 200 KB, i.e. D > 25,600): the
// same scan with the query read from global memory (L1/L2-resident: every warp of the grid reads the same vector).
// Same lane/chunk partition, same sums, same bits.
__global__ void __launch_bounds__(kScanThreads)
angular_distances_wide_kernel(const float *__restrict__ vectors, const double *__restrict__ pp, int64_t n, int64_t ld,
                              const double *__restrict__ queries, int64_t nq, int64_t q_ld, int32_t dim,
                              double *__restrict__ dist, int64_t dist_ld) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t q = blockIdx.y;
    const double *qsrc = queries + q * q_ld;
    const int chunks = (int)(ld >> 2);
    double qq = 0.0;
    for (int c = lane; c < chunks; c += 32) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const double a = 4 * c + t < dim ? __ldg(qsrc + 4 * c + t) : 0.0;
            qq = fma(a, a, qq);
        }
    }
    qq = warp_sum(qq);
    const int64_t warps_total = (int64_t)gridDim.x * kScanWarps;
    for (int64_t row = (int64_t)blockIdx.x * kScanWarps + warp; row < n; row += warps_total) {
        const float4 *src = reinterpret_cast<const float4 *>(vectors + row * ld);
        double acc = 0.0;
        int c = lane;
        for (; c + 96 < chunks; c += 128) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = ldg_stream_f4(src + c + 32 * u);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = 4 * (c + 32 * u);
                const double q0 = e < dim ? __ldg(qsrc + e) : 0.0, q1 = e + 1 < dim ? __ldg(qsrc + e + 1) : 0.0;
                const double q2 = e + 2 < dim ? __ldg(qsrc + e + 2) : 0.0, q3 = e + 3 < dim ? __ldg(qsrc + e + 3) : 0.0;
                acc = fma((double)v[u].x, q0, acc); acc = fma((double)v[u].y, q1, acc);
                acc = fma((double)v[u].z, q2, acc); acc = fma((double)v[u].w, q3, acc);
            }
        }
        for (; c < chunks; c += 32) {
            const float4 v = ldg_stream_f4(src + c);
            const int e = 4 * c;
            const double q0 = e < dim ? __ldg(qsrc + e) : 0.0, q1 = e + 1 < dim ? __ldg(qsrc + e + 1) : 0.0;
            const double q2 = e + 2 < dim ? __ldg(qsrc + e + 2) : 0.0, q3 = e + 3 < dim ? __ldg(qsrc + e + 3) : 0.0;
            acc = fma((double)v.x, q0, acc); acc = fma((double)v.y, q1, acc);
            acc = fma((double)v.z, q2, acc); acc = fma((double)v.w, q3, acc);
        }
        const double pq = warp_sum(acc);
        if (lane == 0) dist[q * dist_ld + row] = angular_from_sums(pp[row], qq, pq);
    }
}

static int launch_distances_wide(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                 const double *queries, int64_t nq, int64_t q_ld, double *dist, int64_t dist_ld,
                                 cudaStream_t stream) {
    if (nq > 65535) return MORNA_ERR_INVALID_ARGUMENT;
    int64_t blocks = (n + kScanWarps - 1) / kScanWarps;
    int64_t cap = ((int64_t)sm_count_cached() * 8 + nq - 1) / nq;
    if (cap < 1) cap = 1;
    if (blocks > cap) blocks = cap;
    dim3 grid((unsigned)blocks, (unsigned)nq);
    angular_distances_wide_kernel<<<grid, kScanThreads, 0, stream>>>(vectors, pp, n, ld, queries, nq, q_ld, dim, dist, dist_ld);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

template <int QB>
static int launch_distances(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                            const double *queries, int64_t nq, int64_t q_ld, double *dist,
                            int64_t dist_ld, cudaStream_t stream) {
    size_t smem = (size_t)QB * ld * sizeof(double);
    if (smem > 200 * 1024) return MORNA_ERR_INVALID_ARGUMENT;
    auto kern = angular_distances_kernel<QB>;
    if (smem > 48 * 1024) {
        int rca = ensure_dynamic_smem((const void *)kern, smem);
        if (rca != MORNA_OK) return rca;
    }
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    int64_t qgroups = (nq + QB - 1) / QB;
    int64_t blocks = (n + kScanWarps - 1) / kScanWarps;
    int64_t cap = ((int64_t)sm_count_cached() * per_sm + qgroups - 1) / qgroups;
    if (cap < 1) cap = 1;
    if (blocks > cap) blocks = cap;
    if (qgroups > 65535) return MORNA_ERR_INVALID_ARGUMENT;
    dim3 grid((unsigned)blocks, (unsigned)qgroups);
    kern<<<grid, kScanThreads, smem, stream>>>(vectors, pp, n, ld, queries, nq, q_ld, dim, dist, dist_ld);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" int morna_angular_distances(const float *vectors, const double *pp, int64_t n, int32_t dim,
                                       int64_t ld, const double *queries, int64_t nq, int64_t q_ld,
                                       double *dist, int64_t dist_ld, void *stream) {
    if (!vectors || !pp || !queries || !dist || n < 0 || nq < 0 || dim <= 0 || ld < dim || (ld & 3) ||
        q_ld < dim || dist_ld < n)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (n == 0 || nq == 0) return MORNA_OK;
    cudaStream_t s = (cudaStream_t)stream;
    int64_t done = 0;
    // groups of 4 queries share each row load; the remainder goes one by one
    while (done < nq) {
        int64_t left = nq - done;
        int64_t take = left >= 4 ? std::min<int64_t>(left / 4 * 4, 65535 * 4) : left;
        int rc;
        if (left >= 4 && (size_t)4 * ld * sizeof(double) <= 200 * 1024)
            rc = launch_distances<4>(vectors, pp, n, dim, ld, queries + done * q_ld, take, q_ld,
                                     dist + done * dist_ld, dist_ld, s);
        else {
            take = std::min<int64_t>(left, 65535);
            if ((size_t)ld * sizeof(double) <= 200 * 1024)
                rc = launch_distances<1>(vectors, pp, n, dim, ld, queries + done * q_ld, take, q_ld,
                                         dist + done * dist_ld, dist_ld, s);
            else
                rc = launch_distances_wide(vectors, pp, n, dim, ld, queries + done * q_ld, take, q_ld,
                                           dist + done * dist_ld, dist_ld, s);
        }
        if (rc != MORNA_OK) return rc;
        done += take;
    }
    return MORNA_OK;
}

extern "C" size_t morna_select_topk_workspace_bytes(int64_t n, int64_t nq, int32_t k) {
    // two ping-pong partial-result buffers sized for the first reduction level
    size_t entries = select_level_entries(n, k) * (size_t)(nq > 0 ? nq : 1);
    return 2 * (align_up(entries * sizeof(double), 256) + align_up(entries * sizeof(int32_t), 256)) + 256;
}

namespace morna {

// K7 merge of per-shard results: G lists per query, each already sorted under the reference rule
// (distance ascending, equal distances id descending; padding = id -1 / +inf at the tail).  One CTA
// per query; every entry finds its global rank as its position in its own list plus, for every other
// list, the number of entries that come before it (binary search), and entries of rank < k_out are
// written straight to their place.  Input layout [G][nq][k_in], as an all-gather of [nq][k_in]
// tensors leaves it.
constexpr int kMergeThreads = 128;

__global__ void __launch_bounds__(kMergeThreads)
merge_sorted_topk_kernel(const double *__restrict__ dists, const int32_t *__restrict__ ids, int32_t n_lists, int64_t nq,
                         int32_t k_in, int32_t k_out, int64_t dist_list_stride, int64_t id_list_stride,
                         int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sd = reinterpret_cast<double *>(smem_raw);                 // [n_lists * k_in]
    int32_t *si = reinterpret_cast<int32_t *>(sd + (size_t)n_lists * k_in);
    const int64_t q = blockIdx.x;
    const int total = n_lists * k_in;
    for (int e = threadIdx.x; e < total; e += kMergeThreads) {
        const int g = e / k_in, j = e - g * k_in;
        const int64_t src = q * k_in + j;                              // lists may sit anywhere: a stride per list
        sd[e] = dists[(int64_t)g * dist_list_stride + src]; si[e] = ids[(int64_t)g * id_list_stride + src];
    }
    for (int i = threadIdx.x; i < k_out; i += kMergeThreads) { out_ids[q * k_out + i] = -1; out_dist[q * k_out + i] = INFINITY; }
    __syncthreads();
    for (int e = threadIdx.x; e < total; e += kMergeThreads) {
        const int id = si[e];
        if (id < 0) continue;                                          // padding never outranks a real entry
        const double d = sd[e];
        const int g = e / k_in;
        int rank = e - g * k_in;                                       // entries before it in its own list
        for (int h = 0; h < n_lists; ++h) {
            if (h == g) continue;
            const double *ld = sd + h * k_in;
            const int32_t *li = si + h * k_in;
            int lo = 0, hi = k_in;                                     // first entry of list h that does NOT come before (d, id)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (li[mid] >= 0 && before(ld[mid], li[mid], d, id)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < k_out) { out_ids[q * k_out + rank] = id; out_dist[q * k_out + rank] = d; }
    }
}

}  // namespace morna

extern "C" int morna_merge_sorted_topk(const double *dists, const int32_t *ids, int32_t n_lists, int64_t nq, int32_t k_in,
                                       int32_t k_out, int32_t *out_ids, double *out_dist, void *stream) {
    if (!dists || !ids || !out_ids || !out_dist || n_lists <= 0 || nq < 0 || k_in <= 0 || k_out <= 0)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    const size_t smem = (size_t)n_lists * k_in * (sizeof(double) + sizeof(int32_t));
    if (smem > 200 * 1024 || nq > 0x7fffffff) return MORNA_ERR_INVALID_ARGUMENT;
    { int rca = ensure_dynamic_smem((const void *)morna::merge_sorted_topk_kernel, smem); if (rca != MORNA_OK) return rca; }
    morna::merge_sorted_topk_kernel<<<(unsigned)nq, morna::kMergeThreads, smem, (cudaStream_t)stream>>>(
        dists, ids, n_lists, nq, k_in, k_out, nq * k_in, nq * k_in, out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

// The same merge straight out of an all-gather of PACKED per-rank buffers: rank g's buffer is nq*k_in doubles
// (distances) followed by nq*k_in int32 (ids), and the gathered tensor is these buffers back to back.
extern "C" int morna_merge_packed_topk(const void *packed, int32_t n_lists, int64_t nq, int32_t k_in, int32_t k_out,
                                       int32_t *out_ids, double *out_dist, void *stream) {
    if (!packed || !out_ids || !out_dist || n_lists <= 0 || nq < 0 || k_in <= 0 || k_out <= 0) return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    const size_t smem = (size_t)n_lists * k_in * (sizeof(double) + sizeof(int32_t));
    if (smem > 200 * 1024 || nq > 0x7fffffff) return MORNA_ERR_INVALID_ARGUMENT;
    { int rca = ensure_dynamic_smem((const void *)morna::merge_sorted_topk_kernel, smem); if (rca != MORNA_OK) return rca; }
    const int64_t per_rank_bytes = nq * k_in * 12;                     // 8-byte aligned: nq*k_in*12 is a multiple of 4; require of 8
    if (per_rank_bytes % 8) return MORNA_ERR_INVALID_ARGUMENT;
    const double *dists = (const double *)packed;
    const int32_t *ids = (const int32_t *)((const unsigned char *)packed + nq * k_in * 8);
    morna::merge_sorted_topk_kernel<<<(unsigned)nq, morna::kMergeThreads, smem, (cudaStream_t)stream>>>(
        dists, ids, n_lists, nq, k_in, k_out, per_rank_bytes / 8, per_rank_bytes / 4, out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" int morna_select_topk(const double *keys, const int32_t *ids, int64_t n, int64_t key_ld,
                                 int32_t id_base, int64_t nq, int32_t k, int32_t *out_ids,
                                 double *out_dist, void *workspace, size_t workspace_bytes, void *stream) {
    if (!keys || !out_ids || !out_dist || n < 0 || nq < 0 || k <= 0 || k > kSelMaxK || key_ld < n)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    if (nq > 65535) return MORNA_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < morna_select_topk_workspace_bytes(n, nq, k)) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t smem = (size_t)kSelChunk * (sizeof(double) + sizeof(int));
    { int rca = ensure_dynamic_smem((const void *)select_topk_kernel, smem); if (rca != MORNA_OK) return rca; }
    size_t entries = select_level_entries(n, k) * (size_t)nq;
    unsigned char *ws = (unsigned char *)workspace;
    double *bufd[2];
    int32_t *bufi[2];
    size_t off = 0;
    for (int b = 0; b < 2; ++b) {
        bufd[b] = (double *)(ws + off); off += align_up(entries * sizeof(double), 256);
        bufi[b] = (int32_t *)(ws + off); off += align_up(entries * sizeof(int32_t), 256);
    }
    const double *cur_k = keys;
    const int32_t *cur_i = ids;
    int64_t cur_n = n, cur_ld = key_ld;
    int flip = 0;
    if (n == 0) cur_n = 0;
    for (;;) {
        int64_t chunks = cur_n > 0 ? (cur_n + kSelChunk - 1) / kSelChunk : 1;
        dim3 grid((unsigned)chunks, (unsigned)nq);
        if (chunks == 1) {
            select_topk_kernel<<<grid, kSelThreads, smem, s>>>(cur_k, cur_i, cur_n, cur_ld, id_base, k,
                                                              out_ids, out_dist, (int64_t)k);
            MORNA_LAUNCH_CHECK();
            break;
        }
        int64_t next_n = chunks * k;
        select_topk_kernel<<<grid, kSelThreads, smem, s>>>(cur_k, cur_i, cur_n, cur_ld, id_base, k,
                                                          bufi[flip], bufd[flip], next_n);
        MORNA_LAUNCH_CHECK();
        cur_k = bufd[flip]; cur_i = bufi[flip]; cur_n = next_n; cur_ld = next_n;
        flip ^= 1;
    }
    return MORNA_OK;
}

static int64_t knn_query_tile(int64_t n, int64_t nq) {
    const int64_t budget = (int64_t)256 << 20;   // bytes of distance scratch per tile
    int64_t t = budget / (8 * (n > 0 ? n : 1));
    if (t < 4) t = 4;
    t = t / 4 * 4;
    if (t > 16384) t = 16384;
    if (t > nq) t = nq;
    return t > 0 ? t : 1;
}

extern "C" size_t morna_knn_exact_workspace_bytes(int64_t n, int64_t nq, int32_t k) {
    int64_t tile = knn_query_tile(n, nq);
    return align_up((size_t)tile * (size_t)(n > 0 ? n : 1) * sizeof(double), 256) +
           morna_select_topk_workspace_bytes(n, tile, k) + 256;
}

extern "C" int morna_knn_exact(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                               int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                               int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                               void *stream) {
    return morna_knn_exact_excl(vectors, pp, n, dim, ld, id_base, queries, nq, q_ld, k, out_ids, out_dist, workspace,
                                workspace_bytes, nullptr, nullptr, stream);
}

extern "C" int morna_knn_exact_excl(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                    int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                                    int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                                    const int32_t *row_group, const int32_t *query_group, void *stream) {
    if (!workspace || workspace_bytes < morna_knn_exact_workspace_bytes(n, nq, k))
        return MORNA_ERR_WORKSPACE_TOO_SMALL;
    if (n <= 0 || nq < 0 || k <= 0 || k > kSelMaxK || !row_group != !query_group) return MORNA_ERR_INVALID_ARGUMENT;
    int64_t tile = knn_query_tile(n, nq);
    double *dist = (double *)workspace;
    size_t dist_bytes = align_up((size_t)tile * (size_t)n * sizeof(double), 256);
    void *sel_ws = (unsigned char *)workspace + dist_bytes;
    size_t sel_bytes = workspace_bytes - dist_bytes;
    for (int64_t q0 = 0; q0 < nq; q0 += tile) {
        int64_t cnt = std::min<int64_t>(tile, nq - q0);
        int rc = morna_angular_distances(vectors, pp, n, dim, ld, queries + q0 * q_ld, cnt, q_ld, dist, n, stream);
        if (rc != MORNA_OK) return rc;
        if (row_group && (rc = launch_mask_excluded(dist, n, n, cnt, row_group, query_group + q0, (cudaStream_t)stream)) != MORNA_OK)
            return rc;
        rc = morna_select_topk(dist, nullptr, n, n, id_base, cnt, k, out_ids + q0 * k, out_dist + q0 * k,
                               sel_ws, sel_bytes, stream);
        if (rc != MORNA_OK) return rc;
        if (row_group && (rc = launch_pad_masked(out_ids + q0 * k, out_dist + q0 * k, cnt * k, (cudaStream_t)stream)) != MORNA_OK)
            return rc;
    }
    return MORNA_OK;
}
