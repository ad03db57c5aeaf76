// Group-capped search: the nearest rows, but at most max_per_group rows of any one group (e.g. one study).
//
// Two pieces live here:
//  - cap_select_kernel: the selection passes of the tensor-core route (pilot thresholds, refinement between row blocks,
//    final candidate lists) when every row carries a cap label.  They take the place of kth_warp_kernel modes 1 / 2 / 0;
//    the GEMM, the workspace, the list swaps and the FP64 re-rank are those of the uncapped route (search_batched.cu).
//  - the walk (morna_cap_sorted_lists): lists already in the reference order, each entry kept iff fewer than
//    max_per_group entries of its group were kept before it, up to a per-list limit.
// DESIGN.md §4 argues why the capped thresholds and the pruning below never drop a row of the answer.
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include "common.cuh"

namespace morna {

namespace {

constexpr int kCapThreads = 512, kCapWarps = kCapThreads / 32;
constexpr int kCapMaxEntries = 8192;                   // the pilot block's dumped scores (kKthMax in search_batched.cu)
constexpr int kCapPer = kCapMaxEntries / kCapThreads;  // sorted entries per thread
constexpr uint64_t kNoEntry = ~0ull;                   // sorts after every real entry

__device__ __forceinline__ uint32_t score_key(float v) {       // monotone float -> uint (float_key of search_batched.cu)
    const uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_score(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// block-wide sum of one int per thread, returned to every thread (red: one int per warp)
template <int kWarps>
__device__ __forceinline__ int block_sum(int v, int *red) {
    v = __reduce_add_sync(kFull, v);
    __syncthreads();                                   // every thread has read red from the previous call
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) t += red[w];
    return t;
}

// exclusive prefix sum of one int per thread in thread order; `total` gets the block's sum
template <int kWarps>
__device__ __forceinline__ int block_excl_scan(int v, int *red, int &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += y;
    }
    __syncthreads();
    if (lane == 31) red[warp] = incl;
    __syncthreads();
    int before = 0;
    total = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        const int x = red[w];
        before += w < warp ? x : 0;
        total += x;
    }
    return before + incl - v;
}

// ascending bitonic sort of P (a power of two) keys in shared memory, an optional 16-bit payload moving with them
template <int kThreads>
__device__ __forceinline__ void bitonic_sort(uint64_t *key, uint16_t *pay, int P) {
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < (P >> 1); i += kThreads) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const uint64_t a = key[lo], b = key[hi];
                if ((a > b) == asc && a != b) {
                    key[lo] = b; key[hi] = a;
                    if (pay) { const uint16_t t = pay[lo]; pay[lo] = pay[hi]; pay[hi] = t; }
                }
            }
        }
    }
    __syncthreads();
}

// first position in key[0, s] whose group (high 32 bits) is that of key[s]: the sorted keys are group-major
__device__ __forceinline__ int group_start(const uint64_t *key, int s) {
    const uint64_t head = key[s] & 0xFFFFFFFF00000000ull;
    int lo = 0, hi = s;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (key[mid] < head) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// One CTA per query.  The query's entries (pilot: the dumped scores of rows n_begin ..; refine / final: its candidate
// list), minus excluded ones, are sorted by (cap label, score descending); an ungrouped row gets a label of its own.
// In that order an entry's within-group rank is its distance from the first entry of its group, and:
//  - the capped k-th score a = the k-th largest score among entries of rank < N (every group's best N), -inf when there
//    are fewer than k of them;
//  - an entry of rank >= N is pruned when its group's N-th best score, less 2 eps rounded outward, is still above it:
//    N rows of its group are strictly nearer in FP64, so the walk can never keep it;
//  - everything else scoring >= a - 2 eps is emitted (pilot / refine: the next candidate list and thr = a - 2 eps; final:
//    the list the FP64 re-rank scores).
// kMode as kth_warp_kernel: 1 pilot, 2 refine, 0 final.  Deterministic: the output order follows the sort.
template <int kMode>
__global__ void __launch_bounds__(kCapThreads)
cap_select_kernel(KthParams p, const int32_t *__restrict__ cap_group, int32_t max_per_group) {
    constexpr bool kPilot = kMode == 1, kRefine = kMode == 2;
    extern __shared__ __align__(16) unsigned char cs_smem[];
    __shared__ int red[kCapWarps];
    const int tid = threadIdx.x, q = blockIdx.x;
    int count;
    if (kPilot) count = p.n0;
    else {
        count = p.cand_cnt[q];
        if (count > p.cap) {                           // survivors were dropped: the FP64 route answers this query
            if (tid == 0) {
                if (!p.overflow[q]) atomicAdd(p.stats + 0, 1);
                p.overflow[q] = 1;
                if (kRefine) { p.cand_cnt[q] = 0; p.thr[q] = INFINITY; }
                else p.fin_cnt[q] = 0;
            }
            return;
        }
    }
    int P = 32;
    while (P < count) P <<= 1;
    uint64_t *skey = reinterpret_cast<uint64_t *>(cs_smem);                  // [P]
    uint16_t *sidx = reinterpret_cast<uint16_t *>(skey + P);                 // [P]: entry index < 8192
    const float *src = kPilot ? p.pilot + (int64_t)q * p.pilot_ld : p.cand_score + (int64_t)q * p.cap;
    const int32_t *ids_in = kPilot ? nullptr : p.cand_id + (int64_t)q * p.cap;
    const int32_t qgroup = p.row_group ? p.query_group[q] : -1;
    for (int i = tid; i < P; i += kCapThreads) {
        uint64_t key = kNoEntry;
        if (i < count) {
            const int64_t row = kPilot ? (int64_t)p.n_begin + i : (int64_t)ids_in[i] - p.id_base;
            if (qgroup < 0 || p.row_group[row] != qgroup) {                   // an excluded entry is absent
                const int32_t g = cap_group[row];
                const uint32_t label = g >= 0 ? (uint32_t)g : 0x80000000u | (uint32_t)i;
                key = ((uint64_t)label << 32) | (uint32_t)~score_key(src[i]);
            }
        }
        skey[i] = key;
        sidx[i] = (uint16_t)i;
    }
    bitonic_sort<kCapThreads>(skey, sidx, P);

    const int N = max_per_group;
    const float two_eps = __fmul_ru(2.0f, p.eps[q]);
    uint32_t eligible = 0, keepable = 0;               // bit j: sorted entry tid + j * kCapThreads
    int n_eligible = 0;
#pragma unroll
    for (int j = 0; j < kCapPer; ++j) {
        const int s = tid + j * kCapThreads;
        if (s >= P) break;
        const uint64_t key = skey[s];
        if (key == kNoEntry) continue;
        const int first = group_start(skey, s);
        if (s - first < N) {
            eligible |= 1u << j;
            keepable |= 1u << j;
            ++n_eligible;
        } else {
            const float nth = key_score(~(uint32_t)skey[first + N - 1]);
            if (!(__fsub_rd(nth, two_eps) > key_score(~(uint32_t)key))) keepable |= 1u << j;
        }
    }
    float cut = -INFINITY;                             // fewer than k eligible entries: nothing can be cut yet
    if (block_sum<kCapWarps>(n_eligible, red) >= p.k) {
        uint32_t best = 0;
        for (int bit = 31; bit >= 0; --bit) {
            const uint32_t trial = best | (1u << bit);
            int c = 0;
#pragma unroll
            for (int j = 0; j < kCapPer; ++j)
                c += ((eligible >> j) & 1u) && ~(uint32_t)skey[tid + j * kCapThreads] >= trial;
            if (block_sum<kCapWarps>(c, red) >= p.k) best = trial;
        }
        cut = __fsub_rd(key_score(best), two_eps);
    }
    const uint32_t cut_key = cut == -INFINITY ? 0u : score_key(cut);
    const int out_cap = (kPilot || kRefine) ? p.cap : p.fcap;
    int out = 0;
    for (int j = 0; j * kCapThreads < P; ++j) {
        const int s = tid + j * kCapThreads;
        uint32_t key = 0;
        bool keep = false;
        if ((keepable >> j) & 1u) {
            key = ~(uint32_t)skey[s];
            keep = key >= cut_key;
        }
        int total;
        const int at = out + block_excl_scan<kCapWarps>(keep ? 1 : 0, red, total);
        if (keep && at < out_cap) {
            const int idx = sidx[s];
            if (kPilot) {
                p.cand_score[(int64_t)q * p.cap + at] = key_score(key);
                p.cand_id[(int64_t)q * p.cap + at] = p.id_base + p.n_begin + idx;
            } else if (kRefine) {
                p.cand2_score[(int64_t)q * p.cap + at] = key_score(key);
                p.cand2_id[(int64_t)q * p.cap + at] = ids_in[idx];
            } else {
                p.fin_id[(int64_t)q * p.fcap + at] = ids_in[idx];
            }
        }
        out += total;
    }
    if (tid == 0) {
        if (kPilot || kRefine) {
            p.thr[q] = cut;
            p.cand_cnt[q] = out;                       // the filter pass appends after these
            if (kRefine) atomicAdd(p.stats + 1, count - out);
        } else {
            int kept = out;
            if (kept > p.fcap) { if (!p.overflow[q]) atomicAdd(p.stats + 0, 1); p.overflow[q] = 1; kept = 0; }
            p.fin_cnt[q] = kept;
            atomicAdd(p.stats + 1, count);
            atomicAdd(p.stats + 2, kept);
            atomicMax(p.stats + 3, kept);
        }
    }
}

// ------------------------------------------------------------------ the walk
constexpr int kWalkThreads = kCapWalkChunk / 2, kWalkWarps = kWalkThreads / 32;

struct CapWalkParams {
    const int64_t *offsets; int64_t in_ld;             // list j: [offsets[j], offsets[j+1]), or [j * in_ld, (j+1) * in_ld)
    const int32_t *ids; const double *dists;
    const int32_t *cap_group; int32_t id_base; int64_t n_rows;
    int32_t max_per_group; int64_t limit;              // limit < 0: none
    int32_t *tab_key; int32_t *tab_cnt;                // per-list hash tables (2 slots per entry); nullptr: one chunk per list
    int32_t *out_ids; double *out_dists; int64_t out_ld;   // out_ld > 0: list j at j * out_ld, padded; 0: at its input start
    int64_t *out_counts;
};

__device__ __forceinline__ int64_t slot_of(int32_t g, int64_t size) { return (int64_t)((uint32_t)g * 2654435761u) % size; }

__device__ __forceinline__ int table_count(const int32_t *tk, const int32_t *tc, int64_t size, int32_t g) {
    for (int64_t h = slot_of(g, size);; h = h + 1 == size ? 0 : h + 1) {
        const int32_t k = __ldcg(tk + h);
        if (k == g) return __ldcg(tc + h);
        if (k == -1) return 0;
    }
}

__device__ __forceinline__ void table_add(int32_t *tk, int32_t *tc, int64_t size, int32_t g, int add) {
    for (int64_t h = slot_of(g, size);; h = h + 1 == size ? 0 : h + 1) {
        const int32_t prev = atomicCAS(tk + h, -1, g);
        if (prev == -1) { __stcg(tc + h, add); return; }
        if (prev == g) { __stcg(tc + h, min(__ldcg(tc + h) + add, 1 << 30)); return; }
    }
}

// One CTA per list, kCapWalkChunk entries at a time.  A chunk's grouped entries are sorted by (group, position): an
// entry's rank within its group is its distance from the group's first entry plus what earlier chunks counted for the
// group (a hash table per list in global memory, 2 slots per entry of the list, so it never fills).  An entry is kept
// iff its rank is below N -- the walk keeps a group's first N entries, so that is "fewer than N kept before it" -- and
// fewer than `limit` entries were kept before it.  Ungrouped entries are always kept; id < 0 is padding and skipped.
__global__ void __launch_bounds__(kWalkThreads)
cap_walk_kernel(CapWalkParams p) {
    __shared__ uint64_t skey[kCapWalkChunk];
    __shared__ int rank_at[kCapWalkChunk];
    __shared__ int red[kWalkWarps];
    const int tid = threadIdx.x;
    const int64_t j = blockIdx.x;
    const int64_t start = p.offsets ? p.offsets[j] : j * p.in_ld;
    const int64_t len = p.offsets ? p.offsets[j + 1] - start : p.in_ld;
    const int64_t size = 2 * len;
    int32_t *tk = p.tab_key ? p.tab_key + 2 * start : nullptr;
    int32_t *tc = p.tab_cnt ? p.tab_cnt + 2 * start : nullptr;
    const int64_t limit = p.limit < 0 ? INT64_MAX : p.limit;
    const int64_t ob = p.out_ld > 0 ? j * p.out_ld : start;
    int64_t kept = 0;
    for (int64_t c0 = 0; c0 < len && kept < limit; c0 += kCapWalkChunk) {
        const int m = (int)min((int64_t)kCapWalkChunk, len - c0);
        int P = 32;
        while (P < m) P <<= 1;
        for (int i = tid; i < P; i += kWalkThreads) {
            uint64_t key = kNoEntry;
            int r = INT_MAX;
            if (i < m) {
                const int32_t id = p.ids[start + c0 + i];
                if (id >= 0) {
                    const int64_t row = (int64_t)id - p.id_base;
                    const int32_t g = row >= 0 && row < p.n_rows ? p.cap_group[row] : -1;
                    r = 0;
                    if (g >= 0) key = ((uint64_t)(uint32_t)g << 32) | (uint32_t)i;
                }
            }
            skey[i] = key;
            rank_at[i] = r;
        }
        bitonic_sort<kWalkThreads>(skey, nullptr, P);
        for (int s = tid; s < P; s += kWalkThreads) {
            const uint64_t key = skey[s];
            if (key == kNoEntry) continue;
            const int32_t g = (int32_t)(key >> 32);
            const int base = (tk && c0 > 0) ? table_count(tk, tc, size, g) : 0;
            rank_at[(uint32_t)key] = base + (s - group_start(skey, s));
        }
        __syncthreads();
        if (tk && c0 + m < len) {                      // later chunks follow: the last entry of each group adds its run
            for (int s = tid; s < P; s += kWalkThreads) {
                const uint64_t key = skey[s];
                if (key == kNoEntry || (s + 1 < P && (skey[s + 1] >> 32) == (key >> 32))) continue;
                table_add(tk, tc, size, (int32_t)(key >> 32), s - group_start(skey, s) + 1);
            }
        }
        const int i0 = 2 * tid;
        const bool k0 = i0 < m && rank_at[i0] < p.max_per_group;
        const bool k1 = i0 + 1 < m && rank_at[i0 + 1] < p.max_per_group;
        int total;
        int64_t at = kept + block_excl_scan<kWalkWarps>((int)k0 + (int)k1, red, total);
        if (k0) {
            if (at < limit) { p.out_ids[ob + at] = p.ids[start + c0 + i0]; p.out_dists[ob + at] = p.dists[start + c0 + i0]; }
            ++at;
        }
        if (k1 && at < limit) { p.out_ids[ob + at] = p.ids[start + c0 + i0 + 1]; p.out_dists[ob + at] = p.dists[start + c0 + i0 + 1]; }
        kept = min(limit, kept + total);
        __syncthreads();                               // skey and rank_at are refilled by the next chunk
    }
    if (p.out_ld > 0)
        for (int64_t i = kept + tid; i < p.out_ld; i += kWalkThreads) { p.out_ids[ob + i] = -1; p.out_dists[ob + i] = INFINITY; }
    if (p.out_counts && tid == 0) p.out_counts[j] = kept;
}

// offsets[0] = 0, offsets[j + 1] = counts[0] + ... + counts[j] (one CTA)
__global__ void __launch_bounds__(1024)
cap_offsets_kernel(const int64_t *__restrict__ counts, int64_t n, int64_t *__restrict__ offsets) {
    __shared__ long long red[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long carry = 0;
    if (tid == 0) offsets[0] = 0;
    for (int64_t b = 0; b < n; b += 1024) {
        const long long v = b + tid < n ? counts[b + tid] : 0;
        long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += y;
        }
        __syncthreads();
        if (lane == 31) red[warp] = incl;
        __syncthreads();
        long long before = 0, total = 0;
        for (int w = 0; w < 32; ++w) { before += w < warp ? red[w] : 0; total += red[w]; }
        if (b + tid < n) offsets[b + tid + 1] = carry + before + incl;
        carry += total;
    }
}

// list j's kept entries, left at its input start by the walk, moved to out_offsets[j]
__global__ void __launch_bounds__(256)
cap_compact_kernel(const int64_t *__restrict__ in_off, const int64_t *__restrict__ out_off, const int32_t *__restrict__ ids,
                   const double *__restrict__ dists, int32_t *__restrict__ out_ids, double *__restrict__ out_dists) {
    const int64_t j = blockIdx.x, from = in_off[j], to = out_off[j], cnt = out_off[j + 1] - to;
    for (int64_t i = threadIdx.x; i < cnt; i += 256) { out_ids[to + i] = ids[from + i]; out_dists[to + i] = dists[from + i]; }
}

struct CapListsWs { size_t tab_key, tab_cnt, ids, dists, counts, total; };
CapListsWs cap_lists_ws_layout(int64_t n_lists, int64_t total) {
    CapListsWs w{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off += align_up(bytes > 0 ? bytes : 1, 256); return at; };
    w.tab_key = take((size_t)2 * total * sizeof(int32_t));
    w.tab_cnt = take((size_t)2 * total * sizeof(int32_t));
    w.ids = take((size_t)total * sizeof(int32_t));
    w.dists = take((size_t)total * sizeof(double));
    w.counts = take((size_t)n_lists * sizeof(int64_t));
    w.total = off;
    return w;
}

int launch_walk(const CapWalkParams &wp, int64_t n_lists, cudaStream_t s) {
    if (n_lists == 0) return MORNA_OK;
    if (n_lists > INT_MAX) return MORNA_ERR_INVALID_ARGUMENT;
    cap_walk_kernel<<<(unsigned)n_lists, kWalkThreads, 0, s>>>(wp);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

}  // namespace

int launch_cap_select(int mode, const KthParams &p, const int32_t *cap_group, int32_t max_per_group, int64_t nq,
                      cudaStream_t s) {
    const int entries = mode == 1 ? p.n0 : p.cap;
    if (entries > kCapMaxEntries || nq > INT_MAX || !cap_group || max_per_group < 1) return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    int P = 32;
    while (P < entries) P <<= 1;
    const size_t smem = (size_t)P * (sizeof(uint64_t) + sizeof(uint16_t));
    const void *kern = mode == 1 ? (const void *)cap_select_kernel<1> : mode == 2 ? (const void *)cap_select_kernel<2>
                                                                                  : (const void *)cap_select_kernel<0>;
    int rc = ensure_dynamic_smem(kern, smem);
    if (rc != MORNA_OK) return rc;
    if (mode == 1) cap_select_kernel<1><<<(unsigned)nq, kCapThreads, smem, s>>>(p, cap_group, max_per_group);
    else if (mode == 2) cap_select_kernel<2><<<(unsigned)nq, kCapThreads, smem, s>>>(p, cap_group, max_per_group);
    else cap_select_kernel<0><<<(unsigned)nq, kCapThreads, smem, s>>>(p, cap_group, max_per_group);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

int launch_cap_walk_strided(const int32_t *ids, const double *dists, int64_t n_lists, int64_t in_ld, const int32_t *cap_group,
                            int32_t id_base, int64_t n_rows, int32_t max_per_group, int64_t limit, int32_t *out_ids,
                            double *out_dists, int64_t out_ld, cudaStream_t s) {
    if (in_ld > kCapWalkChunk || out_ld <= 0 || limit < 0 || limit > out_ld) return MORNA_ERR_INVALID_ARGUMENT;
    CapWalkParams wp{};
    wp.in_ld = in_ld; wp.ids = ids; wp.dists = dists; wp.cap_group = cap_group; wp.id_base = id_base; wp.n_rows = n_rows;
    wp.max_per_group = max_per_group; wp.limit = limit; wp.out_ids = out_ids; wp.out_dists = out_dists; wp.out_ld = out_ld;
    return launch_walk(wp, n_lists, s);
}

}  // namespace morna

using namespace morna;

extern "C" size_t morna_cap_sorted_lists_workspace_bytes(int64_t n_lists, int64_t total) {
    if (n_lists < 0 || total < 0) return 0;
    return cap_lists_ws_layout(n_lists, total).total;
}

extern "C" int morna_cap_sorted_lists(const int64_t *offsets, int64_t n_lists, const int32_t *ids, const double *dists,
                                      int64_t total, const int32_t *cap_group, int32_t id_base, int64_t n_rows,
                                      int32_t max_per_group, int64_t limit, int64_t *out_offsets, int32_t *out_ids,
                                      double *out_dists, int64_t out_ld, void *workspace, size_t workspace_bytes,
                                      void *stream) {
    if (n_lists < 0 || total < 0 || n_rows < 0 || max_per_group < 1 || out_ld < 0 || !offsets || !cap_group ||
        (total > 0 && (!ids || !dists)) || (out_ld > 0 && (limit < 0 || limit > out_ld)) || (out_ld == 0 && !out_offsets) ||
        ((out_ld > 0 ? n_lists : total) > 0 && (!out_ids || !out_dists)) || n_lists > INT_MAX)
        return MORNA_ERR_INVALID_ARGUMENT;
    const CapListsWs w = cap_lists_ws_layout(n_lists, total);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace;
    if (total > 0) MORNA_CUDA_TRY(cudaMemsetAsync(ws + w.tab_key, 0xff, (size_t)2 * total * sizeof(int32_t), s));
    CapWalkParams wp{};
    wp.offsets = offsets; wp.ids = ids; wp.dists = dists; wp.cap_group = cap_group; wp.id_base = id_base; wp.n_rows = n_rows;
    wp.max_per_group = max_per_group; wp.limit = limit;
    wp.tab_key = (int32_t *)(ws + w.tab_key); wp.tab_cnt = (int32_t *)(ws + w.tab_cnt);
    if (out_ld > 0) {                                  // padded [n_lists x out_ld]
        wp.out_ids = out_ids; wp.out_dists = out_dists; wp.out_ld = out_ld;
        return launch_walk(wp, n_lists, s);
    }
    // CSR: the walk leaves each list's kept entries at its input start in the workspace, then they move to their places
    wp.out_ids = (int32_t *)(ws + w.ids); wp.out_dists = (double *)(ws + w.dists); wp.out_ld = 0;
    wp.out_counts = (int64_t *)(ws + w.counts);
    int rc = launch_walk(wp, n_lists, s);
    if (rc != MORNA_OK) return rc;
    cap_offsets_kernel<<<1, 1024, 0, s>>>(wp.out_counts, n_lists, out_offsets);
    MORNA_LAUNCH_CHECK();
    if (n_lists > 0) {
        cap_compact_kernel<<<(unsigned)n_lists, 256, 0, s>>>(offsets, out_offsets, wp.out_ids, wp.out_dists, out_ids, out_dists);
        MORNA_LAUNCH_CHECK();
    }
    return MORNA_OK;
}
