// Batched exact angular kNN on the tensor cores.
//
//   1. rows and queries are normalised and rounded to fp16 (prep kernels); the rounding
//      residual norms give a rigorous per-query bound eps on |fp16 score - true cosine|
//   2. a TMA-fed tcgen05 GEMM (fp16 x fp16 -> fp32 in TMEM) scores queries x samples;
//      its epilogue either dumps a pilot block of scores or keeps only the scores above a
//      per-query threshold  thr = (k-th largest pilot score) - 2*eps
//   3. per query, the exact k-th largest fp16 score a_k over the survivors is found and
//      every sample with score >= a_k - 2*eps goes to the final candidate list -- a
//      superset of the true top-k (ties included)
//   4. candidates are re-ranked with the same FP64 sums the exact scan uses, and sorted
//      under the reference order, so ids and distances equal morna_knn_exact bit for bit.
// Replaces the N x D Python loop of exact_search_nn (morna.py:697-712) for query batches.
#include <cuda_fp16.h>
#include <limits.h>
#include <math.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace morna {

// ------------------------------------------------------------------ operand preparation
constexpr int kPrepThreads = 256;

// warp per stored row: h = fp16(v / |v|), residual norm -> global max
__global__ void __launch_bounds__(kPrepThreads)
prep_samples_kernel(const float *__restrict__ vectors, const double *__restrict__ pp, int64_t n, int64_t ld,
                    __half *__restrict__ hs, int64_t ld_h, float *__restrict__ rho_max) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (kPrepThreads / 32);
    const int chunks = (int)(ld >> 2), chunks_h = (int)(ld_h >> 2);
    for (int64_t row = (int64_t)blockIdx.x * (kPrepThreads / 32) + (threadIdx.x >> 5); row < n; row += warps_total) {
        const float4 *src = reinterpret_cast<const float4 *>(vectors + row * ld);
        uint2 *dst = reinterpret_cast<uint2 *>(hs + row * ld_h);
        const double norm = sqrt(pp[row]);
        const double inv = norm > 0.0 ? 1.0 / norm : 0.0;
        double res = 0.0;
        for (int c = lane; c < chunks_h; c += 32) {
            float4 v = c < chunks ? ldg_stream_f4(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            double x[4] = {v.x * inv, v.y * inv, v.z * inv, v.w * inv};
            __half h[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                h[t] = __float2half_rn((float)x[t]);
                double r = x[t] - (double)__half2float(h[t]);
                res = fma(r, r, res);
            }
            uint2 packed;
            packed.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
            packed.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
            dst[c] = packed;
        }
        res = warp_sum(res);
        if (lane == 0) {
            float rho = __double2float_ru(sqrt(res));
            atomicMax(reinterpret_cast<int *>(rho_max), __float_as_int(rho));   // rho >= 0: int order == float order
        }
    }
}

// warp per query: qq with the canonical tree, fp16 normalised row, eps of the query
__global__ void __launch_bounds__(kPrepThreads)
prep_queries_kernel(const double *__restrict__ queries, int64_t nq, int64_t nq_pad, int32_t dim, int64_t q_ld,
                    __half *__restrict__ hq, int64_t ld_h, double *__restrict__ qq_out, float *__restrict__ eps_out,
                    const float *__restrict__ rho_max, float eps_acc, uint8_t *__restrict__ overflow,
                    int32_t *__restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (kPrepThreads / 32);
    const int chunks_h = (int)(ld_h >> 2);
    for (int64_t row = (int64_t)blockIdx.x * (kPrepThreads / 32) + (threadIdx.x >> 5); row < nq_pad; row += warps_total) {
        uint2 *dst = reinterpret_cast<uint2 *>(hq + row * ld_h);
        if (row >= nq) {
            for (int c = lane; c < chunks_h; c += 32) dst[c] = make_uint2(0u, 0u);
            continue;
        }
        const double *q = queries + row * q_ld;
        const bool vec_ok = ((q_ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(queries) & 15) == 0);
        // chunk c of the row as four doubles (zeros past the end); kPrepInFlight chunks are loaded before any is used:
        // one warp per query leaves the loop latency-bound otherwise
        auto load_chunk = [&](int c, double (&a)[4]) {
            if (vec_ok && 4 * c + 3 < dim) {
                const double2 lo = *reinterpret_cast<const double2 *>(q + 4 * c), hi = *reinterpret_cast<const double2 *>(q + 4 * c + 2);
                a[0] = lo.x; a[1] = lo.y; a[2] = hi.x; a[3] = hi.y;
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) a[t] = (4 * c + t < dim) ? q[4 * c + t] : 0.0;
            }
        };
        constexpr int kPrepInFlight = 4;
        double acc = 0.0;
        bool huge = false;                               // the re-rank stages q * 2^896 (f32_scaled_f64)
        for (int c0 = lane; 4 * c0 < dim; c0 += 32 * kPrepInFlight) {       // same lane/chunk partition and order as the scan
            double a[kPrepInFlight][4];
#pragma unroll
            for (int u = 0; u < kPrepInFlight; ++u) load_chunk(c0 + 32 * u, a[u]);      // chunks past the row are zeros: fma(0, 0, acc) == acc
#pragma unroll
            for (int u = 0; u < kPrepInFlight; ++u) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    huge |= !(fabs(a[u][t]) < kScaledQueryMax);
                    acc = fma(a[u][t], a[u][t], acc);
                }
            }
        }
        acc = warp_sum(acc);
        if (__any_sync(kFull, huge) && overflow && lane == 0) {      // left to the exact scan
            overflow[row] = 1;
            atomicAdd(stats + 0, 1);
        }
        const double norm = sqrt(acc);
        const double inv = norm > 0.0 ? 1.0 / norm : 0.0;
        double res = 0.0;
        for (int c0 = lane; c0 < chunks_h; c0 += 32 * kPrepInFlight) {
            double a[kPrepInFlight][4];
#pragma unroll
            for (int u = 0; u < kPrepInFlight; ++u) load_chunk(c0 + 32 * u, a[u]);
#pragma unroll
            for (int u = 0; u < kPrepInFlight; ++u) {
                const int c = c0 + 32 * u;
                if (c >= chunks_h) break;
                __half h[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    double x = a[u][t] * inv;
                    h[t] = __float2half_rn((float)x);
                    double r = x - (double)__half2float(h[t]);
                    res = fma(r, r, res);
                }
                uint2 packed;
                packed.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
                packed.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
                dst[c] = packed;
            }
        }
        res = warp_sum(res);
        if (lane == 0) {
            qq_out[row] = acc;
            const float rs = *rho_max, rq = __double2float_ru(sqrt(res));
            // |fp16 score - cos| <= rho_s + |h_s| rho_q + accumulation error, |h_s| <= 1 + rho_s
            eps_out[row] = __fadd_ru(__fadd_ru(rs, __fmul_ru(__fadd_ru(1.0f, rs), rq)), eps_acc);
        }
    }
}

// ------------------------------------------------------------------ exact re-rank + final order
constexpr int kRrThreads = 128;                // 4 warps per CTA, several CTAs per SM
constexpr int kOrderThreads = 128;

__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ double2 ldg_f64x2_hint(const double *p, uint64_t pol) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;"
                 : "=d"(r.x), "=d"(r.y) : "l"(p), "l"(pol));
    return r;
}

struct RerankParams {
    const float *vectors; const double *pp; int64_t ld; int32_t dim, id_base, n;
    const double *queries; int64_t q_ld; const double *qq;
    const int32_t *fin_id; const int32_t *fin_cnt; const uint8_t *overflow;
    int32_t fcap, nq, phases, phase_rows;
    int32_t sort_rows;              // key 34: candidates of a query walked in ascending row order (L2 reuse across queries)
    int32_t rows_evict_first;       // key 32: L2 policy of the candidate-row loads (0 evict_normal = default, 1 evict_first, 2 evict_last, 3 mixed, 4 no hint)
    double *fin_dist;
    unsigned long long *queue;      // warp kernel: next item; zero when the batch's lists are complete
    int32_t subs;                   // warp kernel: a query's candidate list is dealt out in 32-entry windows to `subs` items
};

// Exact FP64 distances of every (query, candidate row) pair.  A work item is (query, row phase):
// the CTA stages the query once in shared memory (pre-multiplied by 2^896, see f32_scaled_f64),
// compacts the candidates whose rows fall in the phase's row range, and each warp then takes kRows
// candidate rows at a time so that one shared-memory read of a query chunk feeds kRows FMAs -- the
// load/store unit, not HBM, limited the one-row-per-warp version.  Per row the sum is the canonical
// one (lane l owns float4 chunks l, l+32, ...; one accumulator; fixed butterfly), so the distances
// equal the exact scan's bit for bit.  Items are walked phase-major: with few rows and many queries
// (rows re-ranked several times per batch) the row range of a phase stays L2-resident while all
// queries pass over it; phases == 1 is the plain query-major gather.
constexpr int kRrFatSubs = 5;                  // groups of 4 warps in one SM-filling CTA (rerank_fat_kernel)

template <int kRows, bool kPipe, int kSubs>
__device__ __forceinline__ void rerank_dist_body(const RerankParams &p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // kSubs > 1: the CTA is kSubs independent groups of kRrThreads threads, each with its own staging area, its own
    // named barrier and its own items (drawn from the batch's counter)
    const int sub = kSubs > 1 ? (int)threadIdx.x / kRrThreads : 0;
    const size_t sub_bytes = ((size_t)p.ld * sizeof(double) + (size_t)p.fcap * sizeof(int) + 15) & ~(size_t)15;
    double *qs = reinterpret_cast<double *>(smem_raw + (size_t)sub * sub_bytes);      // [ld]  query * 2^896
    int *list = reinterpret_cast<int *>(qs + p.ld);                      // [fcap] positions in the candidate list
    __shared__ int s_count_all[kSubs];
    __shared__ long long s_item[kSubs];
    int &s_count = s_count_all[sub];
    auto group_sync = [&]() {
        if (kSubs == 1) __syncthreads();
        else asm volatile("bar.sync %0, %1;" :: "r"(sub + 1), "n"(kRrThreads) : "memory");
    };
    const int tid = kSubs > 1 ? (int)threadIdx.x % kRrThreads : (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int chunks = (int)(p.ld >> 2);
    const uint64_t pol = l2_policy_evict_first();
    uint64_t row_pol;
    const int rp_mode = p.rows_evict_first;          // 0 evict_normal, 1 evict_first, 2 evict_last, 3 half evict_last / half evict_first, 4 no hint
    if (rp_mode == 1) row_pol = pol;
    else if (rp_mode == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(row_pol));
    else if (rp_mode == 3) asm volatile("createpolicy.fractional.L2::evict_last.L2::evict_first.b64 %0, 0.5;" : "=l"(row_pol));
    else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(row_pol));
    auto row_ld = [&](const float4 *ptr) {
        if (rp_mode == 4) return ldg_stream_f4(ptr);
        float4 r;
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(ptr), "l"(row_pol));
        return r;
    };
    const int64_t total = (int64_t)p.nq * p.phases;
    for (int64_t t = blockIdx.x; ; t += gridDim.x) {
        if (kSubs > 1) {
            group_sync();                                                // previous item is done with s_item
            if (tid == 0) s_item[sub] = (long long)atomicAdd(p.queue, 1ULL);
            group_sync();
            t = s_item[sub];
        }
        if (t >= total) break;
        const int ph = (int)(t / p.nq), q = (int)(t - (int64_t)ph * p.nq);
        if (p.overflow[q]) continue;                                     // answered by the exact scan afterwards
        const int count = min(p.fin_cnt[q], p.fcap);
        const int32_t *ids = p.fin_id + (int64_t)q * p.fcap;
        const int lo = p.id_base + ph * p.phase_rows;
        const int hi = ph == p.phases - 1 ? INT_MAX : lo + p.phase_rows;
        group_sync();                                                 // previous item is done with qs/list
        if (warp == 0) {
            int m = 0;
            for (int i0 = 0; i0 < count; i0 += 32) {
                const int i = i0 + lane;
                const int id = i < count ? ids[i] : -1;
                const bool keep = i < count && id >= lo && id < hi;
                const unsigned mask = __ballot_sync(kFull, keep);
                if (keep) list[m + __popc(mask & ((1u << lane) - 1u))] = i;
                m += __popc(mask);
            }
            if (lane == 0) s_count = m;
        }
        group_sync();
        const int m = s_count;
        if (m == 0) continue;
        if (p.sort_rows && m <= 256 && (size_t)p.ld * sizeof(double) >= 3 * 256 * sizeof(int)) {
            // Walk the candidates in ascending row order (key 34): the CTAs that run side by side then sweep the matrix
            // roughly together and more of the rows listed by several queries are still in L2 when the next one asks
            // (ncu at the headline shape: L2 hit rate 30.7 -> 37.4 %, DRAM reads 3.91 -> 3.38 GB, 723 -> 696 us; the sweep
            // is loose -- the i-th smallest of ~118 random row ids varies by +-2300 rows between queries -- so most rows
            // still come from HBM).  Rank by counting in the still unused query staging area; results do not depend on
            // the order of the walk.
            int *key = reinterpret_cast<int *>(qs), *sorted = key + 256;
            if (tid < m) key[tid] = ids[list[tid]];
            if (tid + kRrThreads < m) key[tid + kRrThreads] = ids[list[tid + kRrThreads]];
            group_sync();
            for (int i = tid; i < m; i += kRrThreads) {
                const int mine = key[i];
                int rank = 0;
                for (int j = 0; j < m; ++j) { const int o = key[j]; rank += (o < mine) | ((o == mine) & (j < i)); }
                sorted[rank] = list[i];
            }
            group_sync();
            for (int i = tid; i < m; i += kRrThreads) list[i] = sorted[i];
            group_sync();
        }
        {
            const double *qsrc = p.queries + (int64_t)q * p.q_ld;
            if ((p.q_ld & 1) == 0 && (p.dim & 1) == 0) {
                for (int c = 2 * tid; c < (int)p.ld; c += 2 * kRrThreads) {
                    double2 v = make_double2(0.0, 0.0);
                    if (c < p.dim) v = ldg_f64x2_hint(qsrc + c, pol);
                    qs[c] = v.x * kTwo896; qs[c + 1] = v.y * kTwo896;
                }
            } else {
                for (int c = tid; c < (int)p.ld; c += kRrThreads) qs[c] = c < p.dim ? qsrc[c] * kTwo896 : 0.0;
            }
        }
        group_sync();
        const double qqv = p.qq[q];
        for (int g = warp * kRows; g < m; g += (kRrThreads / 32) * kRows) {
            const float4 *src[kRows];
            int pos[kRows];
            int64_t row[kRows];
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                pos[u] = list[min(g + u, m - 1)];                        // the tail repeats the last row
                row[u] = (int64_t)ids[pos[u]] - p.id_base;
                src[u] = reinterpret_cast<const float4 *>(p.vectors + row[u] * p.ld);
            }
            double acc[kRows];
#pragma unroll
            for (int u = 0; u < kRows; ++u) acc[u] = 0.0;
            int c = lane;
            if (kPipe) {
                // (Asking L2 for each row's lines 1-12 KB ahead of the loads with prefetch.global.L2, across pass boundaries,
                // was measured: 0.78-0.93 ms against 0.79 -- the gather is bound by DRAM/L2 throughput, not by latency.)
                // software pipeline: the loads of chunk step i+1 are in flight while step i is accumulated (the plain loop
                // below waits for all its loads, then computes with nothing in flight: ncu shows 9 of 10 issue slots lost
                // to long-scoreboard stalls)
                float4 va[kRows], vb[kRows];
                if (c < chunks) {
#pragma unroll
                    for (int u = 0; u < kRows; ++u) va[u] = row_ld(src[u] + c);
                }
                for (; c < chunks; c += 64) {
                    const int c2 = c + 32, c3 = c + 64;
                    if (c2 < chunks) {
#pragma unroll
                        for (int u = 0; u < kRows; ++u) vb[u] = row_ld(src[u] + c2);
                    }
                    {
                        const double2 qa = *reinterpret_cast<const double2 *>(qs + 4 * c);
                        const double2 qb = *reinterpret_cast<const double2 *>(qs + 4 * c + 2);
#pragma unroll
                        for (int u = 0; u < kRows; ++u) {
                            acc[u] = fma(f32_scaled_f64(va[u].x), qa.x, acc[u]);
                            acc[u] = fma(f32_scaled_f64(va[u].y), qa.y, acc[u]);
                            acc[u] = fma(f32_scaled_f64(va[u].z), qb.x, acc[u]);
                            acc[u] = fma(f32_scaled_f64(va[u].w), qb.y, acc[u]);
                        }
                    }
                    if (c3 < chunks) {
#pragma unroll
                        for (int u = 0; u < kRows; ++u) va[u] = row_ld(src[u] + c3);
                    }
                    if (c2 < chunks) {
                        const double2 qa = *reinterpret_cast<const double2 *>(qs + 4 * c2);
                        const double2 qb = *reinterpret_cast<const double2 *>(qs + 4 * c2 + 2);
#pragma unroll
                        for (int u = 0; u < kRows; ++u) {
                            acc[u] = fma(f32_scaled_f64(vb[u].x), qa.x, acc[u]);
                            acc[u] = fma(f32_scaled_f64(vb[u].y), qa.y, acc[u]);
                            acc[u] = fma(f32_scaled_f64(vb[u].z), qb.x, acc[u]);
                            acc[u] = fma(f32_scaled_f64(vb[u].w), qb.y, acc[u]);
                        }
                    }
                }
                c = chunks;
            }
            for (; c + 32 < chunks; c += 64) {
                float4 v[2][kRows];
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int u = 0; u < kRows; ++u) v[h][u] = row_ld(src[u] + c + 32 * h);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const double2 qa = *reinterpret_cast<const double2 *>(qs + 4 * (c + 32 * h));
                    const double2 qb = *reinterpret_cast<const double2 *>(qs + 4 * (c + 32 * h) + 2);
#pragma unroll
                    for (int u = 0; u < kRows; ++u) {
                        acc[u] = fma(f32_scaled_f64(v[h][u].x), qa.x, acc[u]);
                        acc[u] = fma(f32_scaled_f64(v[h][u].y), qa.y, acc[u]);
                        acc[u] = fma(f32_scaled_f64(v[h][u].z), qb.x, acc[u]);
                        acc[u] = fma(f32_scaled_f64(v[h][u].w), qb.y, acc[u]);
                    }
                }
            }
            for (; c < chunks; c += 32) {
                const double2 qa = *reinterpret_cast<const double2 *>(qs + 4 * c);
                const double2 qb = *reinterpret_cast<const double2 *>(qs + 4 * c + 2);
#pragma unroll
                for (int u = 0; u < kRows; ++u) {
                    const float4 v = row_ld(src[u] + c);
                    acc[u] = fma(f32_scaled_f64(v.x), qa.x, acc[u]);
                    acc[u] = fma(f32_scaled_f64(v.y), qa.y, acc[u]);
                    acc[u] = fma(f32_scaled_f64(v.z), qb.x, acc[u]);
                    acc[u] = fma(f32_scaled_f64(v.w), qb.y, acc[u]);
                }
            }
            double mine = 0.0;
            int my_pos = 0;
            int64_t my_row = 0;
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                const double s = warp_sum(acc[u]);
                if (lane == u) { mine = s; my_pos = pos[u]; my_row = row[u]; }
            }
            if (lane < kRows && g + lane < m)
                p.fin_dist[(int64_t)q * p.fcap + my_pos] = angular_from_sums(p.pp[my_row], qqv, mine);
        }
    }
}

template <int kRows, bool kPipe = false>
__global__ void __launch_bounds__(kRrThreads)
rerank_dist_kernel(const RerankParams p) {
    rerank_dist_body<kRows, kPipe, 1>(p);
}

// The same work in CTAs that fill an SM each (kRrFatSubs groups of four warps, 140 KB of shared memory at D = 3000) and
// come in clusters of two like the GEMM's CTA pairs: a launch of X such CTAs holds exactly X SMs and the scoring kernels of
// the NEXT batch, launched with the remaining SMs as their grid, run beside it (SM partition, DESIGN.md section 5.2).
template <int kRows, bool kPipe>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kRrThreads * kRrFatSubs, 1)
rerank_fat_kernel(const RerankParams p) {
    rerank_dist_body<kRows, kPipe, kRrFatSubs>(p);
}

// ---- warp-granular re-rank: no shared-memory query, no block barriers -------------------------------------
// A work item is (row phase, query), taken from a global counter in phase-major order, and belongs to ONE
// warp: it compacts the query's candidates whose rows lie in the phase's row range (lane-ballot, a 4 KB list
// per warp), then walks them kRows rows at a time; the query chunk a lane needs is read straight from global
// memory (L1/L2: the same 24 KB per pass) and pre-multiplied by 2^896, the rows stream past L1.  Because all
// warps of the GPU draw consecutive items, they work on one phase together: the phase's rows (sized to sit in
// L2) are fetched from HBM once and then hit in L2 for the other ~Q*k/N queries that list them -- the CTA-per-
// query kernel above read 3.9 GB from HBM per headline batch for 0.6 GB of distinct rows.  Per row the sum is
// the canonical one (lane l owns float4 chunks l, l+32, ...; one accumulator; fixed butterfly): bit-equal to
// the exact scan.  The same device function runs as helper warps inside the GEMM kernel (see knn_gemm2_kernel).
constexpr int kRwWarps = 8;

__device__ __forceinline__ double2 ldg_f64x2(const double *p) {
    double2 r;
    asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}

// the four query values of chunk c, times 2^896; zero beyond dim
__device__ __forceinline__ void load_query_chunk(const double *__restrict__ qsrc, int c, int dim, bool vec_ok, double (&qv)[4]) {
    if (vec_ok && 4 * c + 3 < dim) {
        const double2 a = ldg_f64x2(qsrc + 4 * c), b = ldg_f64x2(qsrc + 4 * c + 2);
        qv[0] = a.x * kTwo896; qv[1] = a.y * kTwo896; qv[2] = b.x * kTwo896; qv[3] = b.y * kTwo896;
    } else {
#pragma unroll
        for (int t = 0; t < 4; ++t) qv[t] = 4 * c + t < dim ? __ldg(qsrc + 4 * c + t) * kTwo896 : 0.0;
    }
}

// kRows candidate rows (the first cnt of them live) against one query; kSteps chunk steps of loads in flight
template <int kRows, int kSteps, bool kAll>
__device__ __forceinline__ void rerank_rows(const float4 *const (&src)[kRows], int cnt, const double *__restrict__ qsrc,
                                            int dim, int chunks, bool vec_ok, int lane, double (&acc)[kRows]) {
#pragma unroll
    for (int u = 0; u < kRows; ++u) acc[u] = 0.0;
    int c = lane;
    for (; c + 32 * (kSteps - 1) < chunks; c += 32 * kSteps) {
        float4 v[kSteps][kRows];
#pragma unroll
        for (int h = 0; h < kSteps; ++h)
#pragma unroll
            for (int u = 0; u < kRows; ++u)
                if (kAll || u < cnt) v[h][u] = ldg_stream_f4(src[u] + c + 32 * h);
#pragma unroll
        for (int h = 0; h < kSteps; ++h) {
            double qv[4];
            load_query_chunk(qsrc, c + 32 * h, dim, vec_ok, qv);
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                if (kAll || u < cnt) {
                    acc[u] = fma(f32_scaled_f64(v[h][u].x), qv[0], acc[u]);
                    acc[u] = fma(f32_scaled_f64(v[h][u].y), qv[1], acc[u]);
                    acc[u] = fma(f32_scaled_f64(v[h][u].z), qv[2], acc[u]);
                    acc[u] = fma(f32_scaled_f64(v[h][u].w), qv[3], acc[u]);
                }
            }
        }
    }
    if (kSteps > 1) {
        for (; c < chunks; c += 32) {
            double qv[4];
            load_query_chunk(qsrc, c, dim, vec_ok, qv);
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                if (kAll || u < cnt) {
                    const float4 v = ldg_stream_f4(src[u] + c);
                    acc[u] = fma(f32_scaled_f64(v.x), qv[0], acc[u]);
                    acc[u] = fma(f32_scaled_f64(v.y), qv[1], acc[u]);
                    acc[u] = fma(f32_scaled_f64(v.z), qv[2], acc[u]);
                    acc[u] = fma(f32_scaled_f64(v.w), qv[3], acc[u]);
                }
            }
        }
    }
}

template <int kRows, int kSteps>
__device__ __forceinline__ void rerank_warp_item(const RerankParams &p, long long t, int *list, int lane) {
    const int sub = (int)(t % p.subs);
    t /= p.subs;
    const int ph = (int)(t / p.nq), q = (int)(t - (long long)ph * p.nq);
    if (p.overflow[q]) return;                                           // answered by the exact scan afterwards
    const int count = min(p.fin_cnt[q], p.fcap);
    const int32_t *ids = p.fin_id + (int64_t)q * p.fcap;
    const int lo = p.id_base + ph * p.phase_rows;
    const int hi = ph == p.phases - 1 ? INT_MAX : lo + p.phase_rows;
    int m = 0;
    for (int i0 = 32 * sub; i0 < count; i0 += 32 * p.subs) {
        const int i = i0 + lane;
        const int id = i < count ? ids[i] : -1;
        const bool keep = i < count && id >= lo && id < hi;
        const unsigned mask = __ballot_sync(kFull, keep);
        if (keep) list[m + __popc(mask & ((1u << lane) - 1u))] = i;
        m += __popc(mask);
    }
    if (m == 0) return;
    __syncwarp();
    const double *qsrc = p.queries + (int64_t)q * p.q_ld;
    const bool vec_ok = ((p.q_ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(p.queries) & 15) == 0);
    const int chunks = (int)(p.ld >> 2);
    const double qqv = p.qq[q];
    for (int g = 0; g < m; g += kRows) {
        const int cnt = min(kRows, m - g);
        const float4 *src[kRows];
        int my_pos = 0;
        int64_t my_row = 0;
#pragma unroll
        for (int u = 0; u < kRows; ++u) {
            const int pos = list[min(g + u, m - 1)];
            const int64_t row = (int64_t)ids[pos] - p.id_base;
            src[u] = reinterpret_cast<const float4 *>(p.vectors + row * p.ld);
            if (lane == u) { my_pos = pos; my_row = row; }
        }
        double acc[kRows];
        rerank_rows<kRows, kSteps, false>(src, cnt, qsrc, p.dim, chunks, vec_ok, lane, acc);
        double mine = 0.0;
#pragma unroll
        for (int u = 0; u < kRows; ++u) {
            if (u < cnt) {                                               // cnt is warp-uniform
                const double s = warp_sum(acc[u]);
                if (lane == u) mine = s;
            }
        }
        if (lane < cnt) p.fin_dist[(int64_t)q * p.fcap + my_pos] = angular_from_sums(p.pp[my_row], qqv, mine);
    }
    __syncwarp();
}

// draws items until the counter passes the end (or *stop turns non-zero, for helper warps that must leave with their CTA)
template <int kRows, int kSteps>
__device__ __forceinline__ void rerank_warp_loop(const RerankParams &p, int *list, int lane, const volatile int *stop) {
    const long long total = (long long)p.nq * p.phases * p.subs;
    for (;;) {
        if (stop && *stop) break;
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(p.queue, 1ull);
        t = __shfl_sync(kFull, t, 0);
        if ((long long)t >= total) break;
        rerank_warp_item<kRows, kSteps>(p, (long long)t, list, lane);
    }
}

template <int kRows, int kSteps>
__global__ void __launch_bounds__(kRwWarps * 32, 2)
rerank_warp_kernel(const RerankParams p) {
    extern __shared__ __align__(16) int rw_lists[];                      // [kRwWarps][fcap]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    rerank_warp_loop<kRows, kSteps>(p, rw_lists + warp * p.fcap, lane, nullptr);
}

// One CTA per query: candidates sorted under the reference order (bitonic network in shared
// memory), first k written out; short lists are padded with id -1 / +inf.
__global__ void __launch_bounds__(kOrderThreads)
rerank_order_kernel(const int32_t *__restrict__ fin_id, const int32_t *__restrict__ fin_cnt,
                    const double *__restrict__ fin_dist, const uint8_t *__restrict__ overflow, int32_t fcap,
                    int32_t k, int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sd = reinterpret_cast<double *>(smem_raw);                 // [P]
    int *si = reinterpret_cast<int *>(sd + fcap);                      // [P]
    const int tid = threadIdx.x, q = blockIdx.x;
    int32_t *oi = out_ids + (int64_t)q * k;
    double *od = out_dist + (int64_t)q * k;
    if (overflow[q]) {
        for (int i = tid; i < k; i += kOrderThreads) { oi[i] = -1; od[i] = INFINITY; }
        return;
    }
    const int count = min(fin_cnt[q], fcap);
    int P = 32;
    while (P < count) P <<= 1;
    for (int i = tid; i < P; i += kOrderThreads) {
        const bool have = i < count;
        sd[i] = have ? fin_dist[(int64_t)q * fcap + i] : INFINITY;
        si[i] = have ? fin_id[(int64_t)q * fcap + i] : -1;
    }
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = tid; i < (P >> 1); i += kOrderThreads) {
                int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                bool asc = (lo & size) == 0;
                double dl = sd[lo], dh = sd[hi];
                int il = si[lo], ih = si[hi];
                bool swap = asc ? before(dh, ih, dl, il) : before(dl, il, dh, ih);
                if (swap) { sd[lo] = dh; sd[hi] = dl; si[lo] = ih; si[hi] = il; }
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < k; i += kOrderThreads) {
        bool ok = i < count && si[i] >= 0;
        oi[i] = ok ? si[i] : -1;
        od[i] = ok ? sd[i] : INFINITY;
    }
}

// ------------------------------------------------------------------ GEMM + filter epilogue
namespace gemm {
constexpr int BM = 128, BN = 256, BK = 64, STAGES = 4, UMMA_K = 16;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int THREADS = 192;                    // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int ACC_STAGES = 2, TMEM_COLS = ACC_STAGES * BN;   // 512 columns = all of TMEM
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
}  // namespace gemm

struct GemmParams {
    int32_t relaxed_ns;    // > 0: epilogue warps sleep this long between polls of the accumulator barrier (key 22)
    int32_t l2_keep;       // key 33, experiment: operand tiles loaded with an evict_last L2 policy
    int32_t dry_epilogue;  // key 23, timing experiments only: the filter epilogue finds the survivors but does not append them
    long long *debug;      // optional [gridDim.x][4] cycle counters of the MMA thread (full-barrier wait, accumulator wait, total) and the epilogue
    int32_t nq, n_begin, n_end, kblocks, m_blocks, n_tiles, mode, cap, id_base;
    float *pilot; int64_t pilot_ld;
    const float *thr; float *cand_score; int32_t *cand_id; int32_t *cand_cnt;
};

__global__ void __launch_bounds__(gemm::THREADS, 1)
knn_gemm_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_s, GemmParams p) {
    using namespace gemm;
    using namespace tc;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;        // SWIZZLE_128B wants 1024-byte tiles
    const uint32_t bars = base + STAGES * STAGE_BYTES;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
    auto tfull_bar = [&](int a) { return bars + 8u * (2 * STAGES + a); };
    auto tempty_bar = [&](int a) { return bars + 8u * (2 * STAGES + ACC_STAGES + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * STAGES + 2 * ACC_STAGES);
    volatile uint32_t *tmem_slot_ptr =
        reinterpret_cast<volatile uint32_t *>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmap_q);
        prefetch_tmap(&tmap_s);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 128); }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc<1>(tmem_slot, TMEM_COLS);
        tmem_relinquish<1>();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    const int total_tiles = p.m_blocks * p.n_tiles;
    if (warp == 0) {
        if (lane == 0) {     // ===== TMA producer
            int stage = 0; uint32_t phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                const int m_blk = t % p.m_blocks, n_tile = t / p.m_blocks;
                const int row_q = m_blk * BM, row_s = p.n_begin + n_tile * BN;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    const uint32_t a_dst = base + stage * STAGE_BYTES, b_dst = a_dst + A_BYTES;
                    mbar_expect_tx(full_bar(stage), STAGE_BYTES);
                    tma_load_2d(a_dst, &tmap_q, full_bar(stage), kb * BK, row_q);
                    tma_load_2d(b_dst, &tmap_s, full_bar(stage), kb * BK, row_s);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {     // ===== MMA issuer (one thread)
            constexpr uint32_t idesc = instr_desc_f16(BM, BN, /*fp16*/ 0);
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
                mbar_wait(tempty_bar(acc), acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t a_src = base + stage * STAGE_BYTES, b_src = a_src + A_BYTES;
                    const uint64_t da = smem_desc_sw128(a_src), db = smem_desc_sw128(b_src);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k)      // +32 bytes along K = +2 in the address field
                        umma_f16<1>(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    umma_commit(empty_bar(stage));             // frees the smem stage when the MMAs retire
                    if (kb == p.kblocks - 1) umma_commit(tfull_bar(acc));
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {                 // ===== epilogue: thread = TMEM lane = query row
        const int quarter = warp & 3;                          // TMEM lanes a warp may read: 32*(warp%4)..+31
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
            const int m_blk = t % p.m_blocks, n_tile = t / p.m_blocks;
            const int row = m_blk * BM + quarter * 32 + lane;
            const bool row_ok = row < p.nq;
            const int col_tile = p.n_begin + n_tile * BN;
            float thr = INFINITY;
            if (p.mode == 1 && row_ok) thr = p.thr[row];
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN;
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t r[32];
                tmem_ld_32x32(taddr + c * 32, r);
                tmem_ld_wait();
                const int col0 = col_tile + c * 32;
                const int valid = min(32, p.n_end - col0);
                if (p.mode == 0) {
                    if (row_ok && valid > 0) {
                        float *dst = p.pilot + (int64_t)row * p.pilot_ld + (col0 - p.n_begin);
                        if (valid == 32) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4 *>(dst + j) =
                                    make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < valid) dst[j] = __uint_as_float(r[j]);
                        }
                    }
                } else {
                    uint32_t mask = 0;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        mask |= (uint32_t)(__uint_as_float(r[j]) >= thr && j < valid) << j;
                    if (mask) {
                        int at = atomicAdd(p.cand_cnt + row, __popc(mask));
                        float *cs = p.cand_score + (int64_t)row * p.cap;
                        int32_t *ci = p.cand_id + (int64_t)row * p.cap;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            if ((mask >> j) & 1u) {
                                if (at < p.cap) { cs[at] = __uint_as_float(r[j]); ci[at] = p.id_base + col0 + j; }
                                ++at;
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(tempty_bar(acc));
            if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc<1>(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------ 2-CTA variant (cta_group::2)
// A CTA pair owns a 256-query x 256-sample tile: CTA r holds query rows r*128.. and loads half of
// the sample tile (rows r*128..), the leader issues M=256 UMMAs that read both CTAs' shared memory
// and write both CTAs' TMEM.  Per-CTA shared-memory traffic drops from 48 KB to 32 KB per k-block.
namespace gemm2 {
constexpr int BM = 128, BN = 256, BN_HALF = 128, BK = 64, UMMA_K = 16;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN_HALF * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;   // 32 KB
constexpr int THREADS = 192;                   // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int HELPER_WARPS = 8;                // warps 6-13: re-rank items of the PREVIOUS batch (LSU/FP64/HBM are idle under the MMAs)
constexpr int THREADS_ALL = THREADS + 32 * HELPER_WARPS;
constexpr int ACC_STAGES = 2, TMEM_COLS = ACC_STAGES * BN;
constexpr int HELPER_BYTES = HELPER_WARPS * 1024 * 4 + 16;          // a candidate list per helper warp + the stop flag
constexpr int smem_bytes(int stages) { return stages * STAGE_BYTES + 1024 + 256 + HELPER_BYTES; }
}  // namespace gemm2

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}

// Warps 6-13 take no part in the GEMM: while the tensor cores work through this batch's tiles they draw re-rank
// items of the previous batch (rr.queue != nullptr) from its queue -- the re-rank is a gather of candidate rows
// through LSU + FP64 units the GEMM leaves idle.  They stop taking items when this CTA's epilogue has finished
// its last tile; whatever is left in the queue is drained by rerank_warp_kernel afterwards.
// kCluster = 2: the cluster is one CTA pair.  kCluster = 4 (experiment, key 0 = 2): two pairs that work on the same sample
// tile for two different 256-query blocks; every CTA fetches a QUARTER of the sample tile and multicasts it to its
// counterpart in the other pair, so the sample operand leaves L2 once per two pair-tiles (25 % fewer L2->SM bytes per flop);
// a stage is free when BOTH pairs' MMAs have retired (two arrivals on every CTA's empty barrier).
template <int kStages, bool kHelpers, int kCluster>
__device__ __forceinline__ void
knn_gemm2_body(const CUtensorMap &tmap_q, const CUtensorMap &tmap_s, const GemmParams &p, const RerankParams &rr) {
    using namespace gemm2;
    constexpr bool kQuad = kCluster == 4;
    using namespace tc;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = base + kStages * STAGE_BYTES;
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (kStages + s); };
    auto tfull_bar = [&](int a) { return bars + 8u * (2 * kStages + a); };
    auto tempty_bar = [&](int a) { return bars + 8u * (2 * kStages + ACC_STAGES + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * kStages + 2 * ACC_STAGES);
    volatile uint32_t *tmem_slot_ptr =
        reinterpret_cast<volatile uint32_t *>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
    int *helper_lists = reinterpret_cast<int *>(smem_raw + (bars + 256u - smem_u32(smem_raw)));     // [HELPER_WARPS][1024]
    volatile int *helper_stop = helper_lists + (kHelpers ? HELPER_WARPS * 1024 : 0);                 // (no lists without helpers)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_ctarank();               // rank in the cluster; the pair is (crank & ~1, crank | 1)
    const uint32_t rank = crank & 1u;                       // rank within the pair
    const uint32_t leader_rank = crank & ~1u;
    const int pair_in_cluster = (int)(crank >> 1);
    const bool leader = rank == 0;
    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmap_q);
        prefetch_tmap(&tmap_s);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), kQuad ? 2 : 1); }
        for (int a = 0; a < ACC_STAGES; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 256); }
        fence_barrier_init();
        *helper_stop = 0;
    }
    if (warp == 2) {
        tmem_alloc<2>(tmem_slot, TMEM_COLS);
        tmem_relinquish<2>();
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    // work units: a pair (kCluster 2) or a cluster of two pairs (kCluster 4) owns one (query group, sample tile) at a time
    const int pair = blockIdx.x / kCluster, pairs = gridDim.x / kCluster;
    const int m_pairs = (p.m_blocks + 1) >> 1;              // 256-row query blocks
    const int m_groups = kQuad ? (m_pairs + 1) >> 1 : m_pairs;
    const int total_tiles = m_groups * p.n_tiles;
    auto m_pair_of = [&](int t) { return kQuad ? 2 * (t % m_groups) + pair_in_cluster : t % m_groups; };
    if (warp == 0) {
        if (lane == 0) {     // ===== TMA producer (every CTA); bytes are counted on its pair leader's barrier
            int stage = 0; uint32_t phase = 0;
            uint64_t keep = 0;                               // experiment (key 33): operand tiles marked evict_last in L2
            if (p.l2_keep) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(keep));
            for (int t = pair; t < total_tiles; t += pairs) {
                const int m_pair = m_pair_of(t), n_tile = t / m_groups;
                const int row_q = m_pair * 2 * BM + (int)rank * BM;
                const int row_s = p.n_begin + n_tile * BN + (int)rank * BN_HALF + (kQuad ? pair_in_cluster * (BN_HALF / 2) : 0);
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    if (p.relaxed_ns > 1) mbar_wait_relaxed(empty_bar(stage), phase ^ 1, 20u);
                    else mbar_wait(empty_bar(stage), phase ^ 1);
                    const uint32_t a_dst = base + stage * STAGE_BYTES, b_dst = a_dst + A_BYTES;
                    const uint32_t bar0 = mapa_rank(full_bar(stage), leader_rank);
                    if (leader) mbar_expect_tx(full_bar(stage), 2 * STAGE_BYTES);
                    if (p.l2_keep) tma_load_2d_pair_hint(a_dst, &tmap_q, bar0, kb * BK, row_q, keep);
                    else tma_load_2d_pair(a_dst, &tmap_q, bar0, kb * BK, row_q);
                    if (kQuad)       // my quarter of the sample tile, to me and to my counterpart in the other pair
                        tma_load_2d_pair_multicast(b_dst + pair_in_cluster * (B_BYTES / 2), &tmap_s, bar0, kb * BK, row_s,
                                                   (uint16_t)((1u << crank) | (1u << (crank ^ 2u))));
                    else if (p.l2_keep)
                        tma_load_2d_pair_hint(b_dst, &tmap_s, bar0, kb * BK, row_s, keep);
                    else
                        tma_load_2d_pair(b_dst, &tmap_s, bar0, kb * BK, row_s);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && leader) {     // ===== MMA issuer: one thread of the leader CTA
            constexpr uint32_t idesc = instr_desc_f16(2 * BM, BN, /*fp16*/ 0);
            int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
            long long w_full = 0, w_acc = 0;
            const long long t_begin = clock64();
            for (int t = pair; t < total_tiles; t += pairs) {
                long long c0 = p.debug ? clock64() : 0;
                mbar_wait(tempty_bar(acc), acc_phase ^ 1);
                if (p.debug) w_acc += clock64() - c0;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    c0 = p.debug ? clock64() : 0;
                    mbar_wait(full_bar(stage), phase);
                    if (p.debug) w_full += clock64() - c0;
                    tc_fence_after();
                    const uint32_t a_src = base + stage * STAGE_BYTES, b_src = a_src + A_BYTES;
                    const uint64_t da = smem_desc_sw128(a_src), db = smem_desc_sw128(b_src);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k)
                        umma_f16<2>(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                    umma_commit_pair(empty_bar(stage), kQuad ? 0xF : 0x3);     // frees the stage in every CTA that TMA writes for it
                    if (kb == p.kblocks - 1) umma_commit_pair(tfull_bar(acc), (uint16_t)(0x3u << leader_rank));
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
            }
            if (p.debug) { p.debug[blockIdx.x * 4 + 0] = w_full; p.debug[blockIdx.x * 4 + 1] = w_acc; p.debug[blockIdx.x * 4 + 2] = clock64() - t_begin; }
        }
    } else if (kHelpers && warp >= THREADS / 32) {     // ===== helper warps: re-rank items of the previous batch
        if (rr.queue) rerank_warp_loop<8, 2>(rr, helper_lists + (warp - THREADS / 32) * 1024, lane, helper_stop);
    } else {                 // ===== epilogue: thread = TMEM lane = query row of this CTA's half
        const int quarter = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        long long e_busy = 0;
        for (int t = pair; t < total_tiles; t += pairs) {
            const int m_pair = m_pair_of(t), n_tile = t / m_groups;
            const int row = m_pair * 2 * BM + (int)rank * BM + quarter * 32 + lane;
            const bool row_ok = row < p.nq;
            const int col_tile = p.n_begin + n_tile * BN;
            float thr = INFINITY;
            if (p.mode == 1 && row_ok) thr = p.thr[row];
            if (p.relaxed_ns) mbar_wait_relaxed(tfull_bar(acc), acc_phase, (unsigned)p.relaxed_ns);
            else mbar_wait(tfull_bar(acc), acc_phase);
            const long long e0 = p.debug ? clock64() : 0;
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN;
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t r[32];
                tmem_ld_32x32(taddr + c * 32, r);
                tmem_ld_wait();
                const int col0 = col_tile + c * 32;
                const int valid = min(32, p.n_end - col0);
                if (p.mode == 0) {
                    if (row_ok && valid > 0) {
                        float *dst = p.pilot + (int64_t)row * p.pilot_ld + (col0 - p.n_begin);
                        if (valid == 32) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4 *>(dst + j) =
                                    make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < valid) dst[j] = __uint_as_float(r[j]);
                        }
                    }
                } else {
                    // one returning atomic per 32-column chunk and row with a survivor.  (Reserving a row's slots once per
                    // tile -- two passes over the TMEM chunks -- was measured slower: 0.789 vs 0.767 ms per filter pass.)
                    uint32_t mask = 0;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        mask |= (uint32_t)(__uint_as_float(r[j]) >= thr && j < valid) << j;
                    if (mask && !p.dry_epilogue) {                 // (dry: timing experiment without the appends; results invalid)
                        int at = atomicAdd(p.cand_cnt + row, __popc(mask));
                        float *cs = p.cand_score + (int64_t)row * p.cap;
                        int32_t *ci = p.cand_id + (int64_t)row * p.cap;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            if ((mask >> j) & 1u) {
                                if (at < p.cap) { cs[at] = __uint_as_float(r[j]); ci[at] = p.id_base + col0 + j; }
                                ++at;
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive_cluster(tempty_bar(acc), leader_rank);       // the pair leader's MMA thread waits for both CTAs
            if (p.debug) e_busy += clock64() - e0;
            if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
        if (p.debug && warp == 2 && lane == 0) p.debug[blockIdx.x * 4 + 3] = e_busy;
        if (warp == 2 && lane == 0) *helper_stop = 1;      // this CTA's tiles are done: helpers finish their item and leave
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc<2>(tmem_base, TMEM_COLS);
}

template <int kStages, bool kHelpers>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kHelpers ? gemm2::THREADS_ALL : gemm2::THREADS, 1)
knn_gemm2_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_s, GemmParams p,
                 const RerankParams rr) {
    knn_gemm2_body<kStages, kHelpers, 2>(tmap_q, tmap_s, p, rr);
}

template <int kStages>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(gemm2::THREADS, 1)
knn_gemm4_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_s, GemmParams p,
                 const RerankParams rr) {
    knn_gemm2_body<kStages, false, 4>(tmap_q, tmap_s, p, rr);
}

// ------------------------------------------------------------------ k-th largest + filter
constexpr int kKthThreads = 256, kKthItems = 32, kKthMax = kKthThreads * kKthItems;   // 8192 entries

__device__ __forceinline__ uint32_t float_key(float v) {      // monotone float -> uint
    uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct KthParams {
    int32_t k, n0, n_begin, id_base, cap, fcap;
    const float *pilot; int64_t pilot_ld;
    const float *eps;
    float *thr;
    float *cand_score; int32_t *cand_id; int32_t *cand_cnt;
    float *cand2_score; int32_t *cand2_id;        // refine mode: the compacted list goes here
    int32_t *fin_id; int32_t *fin_cnt;
    uint8_t *overflow; int32_t *stats;
    float *kth_bound;                             // modes 3 / 4: per-query lower bound of the k-th best true cosine
    // modes 0-2, per-query exclusion (nullptr = off): the row behind entry idx (pilot: row n_begin + idx; lists:
    // cand_id[idx] - id_base) is absent for query q iff query_group[q] >= 0 && row_group[row] == query_group[q]
    const int32_t *row_group; const int32_t *query_group;
};

// key of the kk-th largest of the keys one warp holds in registers (kItems per lane; 0 = padding)
template <int kItems>
__device__ __forceinline__ uint32_t warp_kth_largest(const uint32_t (&key)[kItems], int kk) {
    // every real key lies between the smallest non-zero and the largest key the warp holds, so the answer shares their
    // common leading bits: the bisection starts below them (scores of one query differ in ~23 of their 32 key bits)
    uint32_t hi = 0u, lo = ~0u;
#pragma unroll
    for (int j = 0; j < kItems; ++j) { hi = max(hi, key[j]); lo = min(lo, key[j] ? key[j] : ~0u); }
    hi = __reduce_max_sync(kFull, hi);
    lo = __reduce_min_sync(kFull, lo);
    if (hi == 0u || kk <= 0) return 0u;                       // nothing but padding
    const int first = 31 - __clz((int)(hi ^ lo) | 1);         // highest bit in which two real keys can differ (bit 0 at least)
    uint32_t best = first < 31 ? hi & ~((2u << first) - 1u) : 0u;
    for (int bit = first; bit >= 0; --bit) {
        const uint32_t trial = best | (1u << bit);
        int c = 0;
#pragma unroll
        for (int j = 0; j < kItems; ++j) c += key[j] >= trial;
        c = __reduce_add_sync(kFull, c);
        if (c >= kk) best = trial;
    }
    return best;
}

constexpr int kCandCapConst = 4096;                   // = kCandCap below
constexpr int kKwWarps = 8, kKwSlots = 32;            // one warp per query; 32 survivors per lane
constexpr int kKwSmem = kKwWarps * 32 * kKwSlots * (int)(sizeof(uint32_t) + sizeof(uint16_t));   // 48 KB: four CTAs per SM, 4096 queries resident at once

// One WARP per query (8 queries per CTA, no block barriers).
//   kMode 1 (pilot) : input = dumped pilot scores -> thr[q] and the pilot's survivors start the candidate list
//   kMode 0 (final) : input = candidate list      -> final candidate list
//   kMode 2 (refine): input = candidate list      -> thr[q] tightened to (k-th largest so far) - 2 eps and the
//                     list compacted into the second buffer; run between row blocks so that the list stays
//                     short however many rows one call scores
// A pivot taken from a 512-entry sample cuts the stream to a few hundred survivors that stay in
// lane-private shared-memory lists; the exact k-th largest a_k of the survivors (= of all entries) is
// found with warp-wide counts, and everything >= a_k - 2 eps is written out.  If the pivot misses
// (too few survivors, a lane list overflows, or a_k - 2 eps falls below the pivot) the warp falls
// back to a streaming bisection over all entries, which is exact for any input.
//   kMode 3 (bound) : input = candidate list      -> kth_bound[q] = (k-th largest score) - eps, nothing emitted.  Rows-sharded
//                     search: the maximum of this bound over the ranks is a lower bound of the GLOBAL k-th best cosine
//   kMode 4 (emit)  : input = candidate list      -> final candidate list = everything >= kth_bound[q] - eps
// With an exclusion (modes 0-2) an excluded entry is absent everywhere: it never enters the lane lists, the bisection
// does not count it and nothing emits it; kk is the number of ALLOWED entries when fewer than k are allowed, and then
// the threshold stays -inf and every allowed entry is emitted.  Labels are looked up only for entries that pass the
// pivot (or, without a usable pivot, in the fallback passes).
template <int kMode>
__global__ void __launch_bounds__(kKwWarps * 32)
kth_warp_kernel(KthParams p, int nq) {
    constexpr bool kPilot = kMode == 1, kRefine = kMode == 2, kBound = kMode == 3, kEmit = kMode == 4;
    extern __shared__ __align__(16) uint32_t kw_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x * kKwWarps + warp;
    if (q >= nq) return;
    uint32_t *lkey = kw_smem + warp * 32 * kKwSlots;              // [slot][lane]
    uint16_t *lidx = reinterpret_cast<uint16_t *>(kw_smem + kKwWarps * 32 * kKwSlots) + warp * 32 * kKwSlots;   // entry index < 8192
    static_assert(kKthMax <= 65536 && kCandCapConst <= 65536, "entry indices are kept in 16 bits");
    int count;
    if (kPilot) count = p.n0;
    else {
        count = p.cand_cnt[q];
        if (count > p.cap) {            // survivors were dropped: the exact scan must answer this query
            if (lane == 0) {
                if (!p.overflow[q]) atomicAdd(p.stats + 0, 1);
                p.overflow[q] = 1;
                if (kRefine) { p.cand_cnt[q] = 0; p.thr[q] = INFINITY; }      // collect nothing more for it
                else if (kBound) { for (int i = 0; i < p.k; ++i) p.kth_bound[(int64_t)q * p.k + i] = -INFINITY; }   // this rank's exact scan answers; no bound from here
                else p.fin_cnt[q] = 0;
            }
            return;
        }
    }
    const float *src = kPilot ? p.pilot + (int64_t)q * p.pilot_ld : p.cand_score + (int64_t)q * p.cap;
    int kk = min(p.k, count);
    const int out_cap = (kPilot || kRefine) ? p.cap : p.fcap;
    const float eps = p.eps[q];
    const int32_t qgroup = (!kBound && !kEmit && p.row_group) ? p.query_group[q] : -1;
    const bool excl = qgroup >= 0;                              // warp-uniform
    auto allowed = [&](int idx) -> bool {
        const int64_t row = kPilot ? (int64_t)p.n_begin + idx : (int64_t)p.cand_id[(int64_t)q * p.cap + idx] - p.id_base;
        return p.row_group[row] != qgroup;
    };

    uint32_t best = 0;          // key of the kk-th largest entry
    bool lists_ok = false;      // lane lists hold every entry >= pivot
    uint32_t pivot = 0;
    int mine = 0;               // survivors in this lane's list
    if (kk > 0 && !kEmit) {
        if (count > 32 * kKwSlots) {                 // pivot from 512 strided samples
            uint32_t sk[16];
            const int stride = count >> 9;
#pragma unroll
            for (int j = 0; j < 16; ++j) sk[j] = float_key(src[(j * 32 + lane) * stride]);
            const float want = (float)kk * 512.0f / (float)count;
            const int r = (int)(want + 4.0f * sqrtf(want) + 4.0f);
            pivot = r <= 512 ? warp_kth_largest<16>(sk, r) : 0u;
        }
        // stream: lane owns float4 groups lane, lane+32, ...; survivors go to its private list
        const int groups = (count + 3) >> 2;
        bool overflowed = false;
        const float pivot_f = pivot ? key_float(pivot) : -INFINITY;
        constexpr int kInFlight = 8;                                         // 16-byte loads in flight per lane (the stream is latency bound)
        for (int g0 = lane; g0 < groups; g0 += 32 * kInFlight) {
            float4 v[kInFlight];
#pragma unroll
            for (int u = 0; u < kInFlight; ++u) {
                const int g = g0 + 32 * u;
                v[u] = g < groups ? __ldcs(reinterpret_cast<const float4 *>(src + 4 * g))   // rows are 16-byte aligned and padded; read once
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if (pivot != 0u) {
                // With a pivot only a few per cent of the entries pass, but for almost every one of a lane's 32 entries SOME
                // lane of the warp has a survivor, so a branch per entry makes the whole warp walk the insertion code 32
                // times per step (ncu: two thirds of the pilot pass's instructions).  Instead: a bit per entry from a float
                // compare (key order refines float order -- only -0 < +0 differs -- so v >= pivot_f holds for every entry
                // whose key reaches the pivot), then a loop over the set bits, as long as the busiest lane's count (~5).
                uint32_t bits = 0u;
#pragma unroll
                for (int u = 0; u < kInFlight; ++u) {
                    bits |= (v[u].x >= pivot_f ? 1u : 0u) << (4 * u);
                    bits |= (v[u].y >= pivot_f ? 1u : 0u) << (4 * u + 1);
                    bits |= (v[u].z >= pivot_f ? 1u : 0u) << (4 * u + 2);
                    bits |= (v[u].w >= pivot_f ? 1u : 0u) << (4 * u + 3);
                }
                while (bits) {
                    const int e = __ffs((int)bits) - 1;
                    bits &= bits - 1u;
                    const int idx = 4 * (g0 + 32 * (e >> 2)) + (e & 3);
                    if (idx < count) {
                        // entry e of the 32 this lane holds: a select tree over the registers (31 selects; reading the
                        // value again by index instead cost a DRAM / L2 round trip per survivor)
                        float s16[16], s8[8], s4[4], s2[2];
#pragma unroll
                        for (int u = 0; u < kInFlight; ++u) {
                            s16[2 * u] = (e & 1) ? v[u].y : v[u].x;
                            s16[2 * u + 1] = (e & 1) ? v[u].w : v[u].z;
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) s8[i] = (e & 2) ? s16[2 * i + 1] : s16[2 * i];
#pragma unroll
                        for (int i = 0; i < 4; ++i) s4[i] = (e & 4) ? s8[2 * i + 1] : s8[2 * i];
#pragma unroll
                        for (int i = 0; i < 2; ++i) s2[i] = (e & 8) ? s4[2 * i + 1] : s4[2 * i];
                        const uint32_t key = float_key((e & 16) ? s2[1] : s2[0]);
                        if (key >= pivot && (!excl || allowed(idx))) {
                            if (mine < kKwSlots) { lkey[mine * 32 + lane] = key; lidx[mine * 32 + lane] = (uint16_t)idx; }
                            else overflowed = true;
                            ++mine;
                        }
                    }
                }
                continue;
            }
#pragma unroll
            for (int u = 0; u < kInFlight; ++u) {
                const int g = g0 + 32 * u;
                const float vv[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    // (no pivot: every entry is a survivor)
                    if (vv[t] >= pivot_f) {
                        const int idx = 4 * g + t;
                        const uint32_t key = float_key(vv[t]);
                        if (idx < count && key >= pivot && (!excl || allowed(idx))) {
                            if (mine < kKwSlots) { lkey[mine * 32 + lane] = key; lidx[mine * 32 + lane] = (uint16_t)idx; }
                            else overflowed = true;
                            ++mine;
                        }
                    }
                }
            }
        }
        const int m = __reduce_add_sync(kFull, mine);
        const bool any_over = __any_sync(kFull, overflowed);
        if (excl && pivot == 0u && !any_over) kk = min(kk, m);      // the lists hold every allowed entry
        lists_ok = !any_over && m >= kk;
        if (lists_ok) {
            uint32_t sk[kKwSlots];
#pragma unroll
            for (int j = 0; j < kKwSlots; ++j) sk[j] = j < mine ? lkey[j * 32 + lane] : 0u;
            best = warp_kth_largest<kKwSlots>(sk, kk);
        } else {                                     // streaming bisection over every (allowed) entry
            if (excl) {
                int ca = 0;
                for (int i = lane; i < count; i += 32) ca += allowed(i);
                kk = min(kk, __reduce_add_sync(kFull, ca));
            }
            for (int bit = 31; bit >= 0 && kk > 0; --bit) {
                const uint32_t trial = best | (1u << bit);
                int c = 0;
                for (int i = lane; i < count; i += 32) c += float_key(src[i]) >= trial && (!excl || allowed(i));
                c = __reduce_add_sync(kFull, c);
                if (c >= kk) best = trial;
            }
        }
    }
    if (kBound) {
        // This rank's contribution to the global bound: lower bounds (score - eps) of the true cosines of its k best
        // rows (any k distinct rows do; -inf pads a shorter list).  The lists are built by a later kEmit launch.
        float *dst = p.kth_bound + (int64_t)q * p.k;
        for (int i = lane; i < p.k; i += 32) dst[i] = -INFINITY;
        __syncwarp();
        int outb = 0;
        auto put = [&](bool keep, float score) {
            const unsigned mask = __ballot_sync(kFull, keep);
            const int at = outb + __popc(mask & ((1u << lane) - 1u));
            if (keep && at < p.k) dst[at] = __fsub_rd(score, eps);
            outb += __popc(mask);
        };
        if (kk > 0) {
            if (lists_ok) {
                const int most = __reduce_max_sync(kFull, mine);
                for (int j = 0; j < most && outb < p.k; ++j) {
                    const bool have = j < mine;
                    const uint32_t key = have ? lkey[j * 32 + lane] : 0u;
                    put(have && key >= best, key_float(key));
                }
            } else {
                for (int i0 = 0; i0 < count && outb < p.k; i0 += 32) {
                    const int i = i0 + lane;
                    const float v = i < count ? src[i] : 0.f;
                    put(i < count && float_key(v) >= best, v);
                }
            }
        }
        return;
    }
    // cannot prune while fewer than k scores have been seen
    float cut = -INFINITY;
    if (kEmit) { const float b = p.kth_bound[q]; if (b > -INFINITY) cut = __fsub_rd(b, eps); }
    else if (kk >= p.k) cut = __fsub_rd(key_float(best), __fmul_ru(2.0f, eps));
    const uint32_t cut_key = cut == -INFINITY ? 0u : float_key(cut);
    int out = 0;
    auto emit = [&](bool keep, float score, int idx) {
        const unsigned mask = __ballot_sync(kFull, keep);
        const int at = out + __popc(mask & ((1u << lane) - 1u));
        if (keep && at < out_cap) {
            if (kPilot) {
                p.cand_score[(int64_t)q * p.cap + at] = score;
                p.cand_id[(int64_t)q * p.cap + at] = p.id_base + p.n_begin + idx;
            } else if (kRefine) {
                p.cand2_score[(int64_t)q * p.cap + at] = score;
                p.cand2_id[(int64_t)q * p.cap + at] = p.cand_id[(int64_t)q * p.cap + idx];
            } else {
                p.fin_id[(int64_t)q * p.fcap + at] = p.cand_id[(int64_t)q * p.cap + idx];
            }
        }
        out += __popc(mask);
    };
    if (lists_ok && cut_key >= pivot) {              // every entry >= cut sits in the lane lists
        const int most = __reduce_max_sync(kFull, mine);
        if (kPilot) {
            for (int j = 0; j < most; ++j) {
                const bool have = j < mine;
                const uint32_t key = have ? lkey[j * 32 + lane] : 0u;
                emit(have && key >= cut_key, key_float(key), have ? (int)lidx[j * 32 + lane] : 0);
            }
        } else {
            // the emitted entry's row id is read from the candidate list: four steps' loads are issued before their stores
            // (one step at a time, every store waited for its own load: half of the final pass's stall samples in ncu)
            const int32_t *ids_in = p.cand_id + (int64_t)q * p.cap;
            for (int j0 = 0; j0 < most; j0 += 4) {
                bool keep[4];
                uint32_t key[4];
                int32_t id[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 + u;
                    const bool have = j < mine;
                    key[u] = have ? lkey[j * 32 + lane] : 0u;
                    keep[u] = have && key[u] >= cut_key;
                    id[u] = keep[u] ? ids_in[lidx[j * 32 + lane]] : 0;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const unsigned mask = __ballot_sync(kFull, keep[u]);
                    const int at = out + __popc(mask & ((1u << lane) - 1u));
                    if (keep[u] && at < out_cap) {
                        if (kRefine) {
                            p.cand2_score[(int64_t)q * p.cap + at] = key_float(key[u]);
                            p.cand2_id[(int64_t)q * p.cap + at] = id[u];
                        } else {
                            p.fin_id[(int64_t)q * p.fcap + at] = id[u];
                        }
                    }
                    out += __popc(mask);
                }
            }
        }
    } else {
        for (int i0 = 0; i0 < count; i0 += 32) {
            const int i = i0 + lane;
            const float v = i < count ? src[i] : 0.f;
            bool keep = i < count && v >= cut;
            if (excl && keep) keep = allowed(i);
            emit(keep, v, i);
        }
    }
    if (lane == 0) {
        if (kPilot || kRefine) {
            p.thr[q] = cut;
            p.cand_cnt[q] = out;                     // the filter pass appends after these
            if (kRefine) atomicAdd(p.stats + 1, count - out);        // survivors dropped here still count as first-pass survivors
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

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int g_tmap_promotion = 3;   // key 24: L2 promotion of the operand tensor maps (0 none, 1 64 B, 2 128 B, 3 256 B)

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// fp16 row-major [rows x ld_h] -> tiles of box_rows x 64 halves, 128-byte swizzle, zero fill out of range
static int make_tmap(CUtensorMap *map, const void *ptr, uint64_t rows, uint64_t ld_h, uint32_t box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return MORNA_ERR_CUDA;
    cuuint64_t dims[2] = {ld_h, rows};
    cuuint64_t strides[1] = {ld_h * sizeof(__half)};
    cuuint32_t box[2] = {(cuuint32_t)gemm::BK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapL2promotion promo = g_tmap_promotion == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE
                                        : g_tmap_promotion == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                        : g_tmap_promotion == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { g_last_cuda_error = (int)r; return MORNA_ERR_CUDA; }
    return MORNA_OK;
}

static int sm_count_b() { return sm_count_current(); }

constexpr int kCandCap = kCandCapConst, kFinCap = 1024, kPilotMax = kKthMax;
constexpr int64_t kBatchedMaxRows = (int64_t)1 << 24;      // rows one call may score (ids are int32; TMA row coordinate)

// tuning knobs for experiments (morna_debug_set_tuning): GEMM variant and pipeline depth
static int g_gemm_pair = 1;       // 1: CTA pairs (cta_group::2), 0: single CTAs
static int g_gemm_stages = 4;
static int g_block_rows = 131072;  // rows scored between two refinements of the candidate lists (key 9)
static int g_pilot_rows = kKthMax; // rows of the pilot block whose scores are dumped for the first thresholds (key 10)
static int g_block_growth = 1;     // key 36: factor by which the blocks after the first grow (1 = equal blocks, the default: doubling saves
                                   // four refinements at 1 M rows but measured within the run-to-run noise, profiles/r02_block_rows_sweep.log)
static int g_first_block = 0;      // rows up to the first refinement (key 11); 0 = g_block_rows
static int g_rerank_ctas_per_sm = 0; // key 13: cap on resident re-rank CTAs per SM (0 = whatever fits)
static int g_rerank_rows = 4;     // candidate rows per warp pass of the re-rank (2, 4, 8; 16 for the warp kernel)
static int g_rerank_phase_mb = -1; // row range kept L2-resident per re-rank phase; 0 = never split; -1 = 64 MB for the warp kernel, unsplit otherwise
static int g_rerank_kernel = 1;    // key 14: 0 = warp-granular items from a global queue, 1 = one CTA per query (shared-memory query)
static int g_rerank_ctas = 0;      // key 15: CTAs per SM of the warp kernel (0 = what fits)
static int g_rerank_subs = 0;      // key 16: items per query of the unsplit warp re-rank (0 = 4)
static int g_side_job = 0;         // key 17: 1 = side jobs on: helper warps in the GEMM kernel re-rank the previous batch (measured slower:
                                   // the GEMM's TMA stream and the helpers' gathers queue behind each other, DESIGN.md section 5)
static int g_rerank_sort_rows = 1;     // key 34: candidates walked in ascending row order (ncu: 3.91 -> 3.38 GB DRAM, 723 -> 696 us)
static int g_rerank_evict_first = 0;   // key 32 (measured, scripts/rerank_policy_sweep.py: an explicit evict_normal hint is 1-4 % faster than none)
static int g_gemm_l2_keep = 0;         // key 33
static int g_rerank_fat_sms = 0;   // key 30: > 0 = the re-rank runs as this many SM-filling CTAs ...
static int g_gemm_pairs_cap = 0;   // key 31: ... and the GEMM kernels use at most this many CTA pairs (0 = all SMs)
static int g_rerank_pipe = 1;      // key 18: CTA-per-query re-rank with software-pipelined row loads
static long long *g_gemm_debug = nullptr;   // morna_debug_gemm_counters: device buffer for the MMA thread's wait counters
static int g_gemm_relaxed_ns = 0;  // key 22
static int g_gemm_dry = 0;         // key 23
static int g_carveout_hint = 0;    // key 19: ask for the maximum shared-memory carve-out on the batched path's kernels (co-residency across streams)
static int g_rerank_oneshot = 1;   // key 20: CTA-per-query re-rank launched as one CTA per item (default; 0 = persistent grid): its CTAs retire one by
                                   // one, so the next batch's first kernels start under its tail (1.875 -> 1.834 ms per headline batch)


static int launch_knn_gemm(const CUtensorMap &tmap_q, const CUtensorMap &tmap_s, const GemmParams &gp, cudaStream_t s,
                           const RerankParams *side = nullptr) {
    if (!g_gemm_pair) {
        int rca = ensure_dynamic_smem((const void *)knn_gemm_kernel, gemm::SMEM_BYTES);
        if (rca != MORNA_OK) return rca;
        int tiles = gp.m_blocks * gp.n_tiles;
        int grid = tiles < sm_count_b() ? tiles : sm_count_b();
        knn_gemm_kernel<<<grid, gemm::THREADS, gemm::SMEM_BYTES, s>>>(tmap_q, tmap_s, gp);
        MORNA_LAUNCH_CHECK();
        return MORNA_OK;
    }
    if (g_gemm_pair == 2 && !side && (gp.m_blocks % 4) == 0) {          // experiment: clusters of two pairs, multicast sample tile
        auto kern4 = knn_gemm4_kernel<4>;
        const int smem4 = gemm2::smem_bytes(4) - gemm2::HELPER_BYTES + 16;
        int rca = ensure_dynamic_smem((const void *)kern4, smem4);
        if (rca != MORNA_OK) return rca;
        int tiles4 = (gp.m_blocks / 4) * gp.n_tiles;
        int clusters = 0;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(4 * (sm_count_b() / 4)); cfg.blockDim = dim3(gemm2::THREADS); cfg.dynamicSmemBytes = smem4; cfg.stream = s;
        if (cudaOccupancyMaxActiveClusters(&clusters, kern4, &cfg) != cudaSuccess || clusters < 1) { cudaGetLastError(); clusters = sm_count_b() / 4; }
        if (clusters > sm_count_b() / 4) clusters = sm_count_b() / 4;
        if (tiles4 < clusters) clusters = tiles4;
        RerankParams none{};
        kern4<<<4 * clusters, gemm2::THREADS, smem4, s>>>(tmap_q, tmap_s, gp, none);
        MORNA_LAUNCH_CHECK();
        return MORNA_OK;
    }
    const int stages = g_gemm_stages == 4 ? 4 : 6;
    // two builds of the kernel: with the helper warps (side job given) and without them -- the plain one is not held to the
    // register budget of 448 threads
    auto kern = side ? (stages == 4 ? knn_gemm2_kernel<4, true> : knn_gemm2_kernel<6, true>)
                     : (stages == 4 ? knn_gemm2_kernel<4, false> : knn_gemm2_kernel<6, false>);
    const int smem = gemm2::smem_bytes(stages);
    int rca = ensure_dynamic_smem((const void *)kern, smem);
    if (rca != MORNA_OK) return rca;
    int tiles = ((gp.m_blocks + 1) / 2) * gp.n_tiles;
    int pairs = sm_count_b() / 2;
    if (g_gemm_pairs_cap > 0 && pairs > g_gemm_pairs_cap) pairs = g_gemm_pairs_cap;     // SM partition: the rest belongs to the re-rank
    if (tiles < pairs) pairs = tiles;
    RerankParams rr{};
    if (side) rr = *side;
    if (g_carveout_hint) cudaFuncSetAttribute((const void *)kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    // without a side job the helper warps are not launched at all (192 threads, no candidate-list shared memory)
    const int threads = side ? gemm2::THREADS_ALL : gemm2::THREADS;
    const int smem_launch = side ? smem : smem - gemm2::HELPER_BYTES + 16;
    kern<<<2 * pairs, threads, smem_launch, s>>>(tmap_q, tmap_s, gp, rr);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

struct BatchWs {
    size_t hq, qq, eps, pilot, thr, cand_score, cand_id, cand2_score, cand2_id, cand_cnt, fin_id, fin_cnt, fin_dist, queue, total;
    int64_t nq_pad, n0, pilot_ld;
};
static BatchWs batch_ws_layout(int64_t n, int64_t nq, int64_t ld_h) {
    BatchWs w{};
    w.nq_pad = (nq + 2 * gemm::BM - 1) / (2 * gemm::BM) * (2 * gemm::BM);      // CTA pairs own 256 query rows
    w.n0 = n < g_pilot_rows ? n : g_pilot_rows;
    if (w.n0 > g_block_rows) w.n0 = g_block_rows;
    w.pilot_ld = (w.n0 + 3) / 4 * 4;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off += align_up(bytes, 256); return at; };
    w.hq = take((size_t)w.nq_pad * ld_h * sizeof(__half));
    w.qq = take((size_t)nq * sizeof(double));
    w.eps = take((size_t)nq * sizeof(float));
    w.pilot = take((size_t)nq * w.pilot_ld * sizeof(float));
    w.thr = take((size_t)nq * sizeof(float));
    w.cand_score = take((size_t)nq * kCandCap * sizeof(float));
    w.cand_id = take((size_t)nq * kCandCap * sizeof(int32_t));
    if (n > g_block_rows || (g_first_block > 0 && n > g_first_block)) {   // several row blocks: lists refined between them (ping-pong)
        w.cand2_score = take((size_t)nq * kCandCap * sizeof(float));
        w.cand2_id = take((size_t)nq * kCandCap * sizeof(int32_t));
    }
    w.cand_cnt = take((size_t)nq * sizeof(int32_t));
    w.fin_id = take((size_t)nq * kFinCap * sizeof(int32_t));
    w.fin_cnt = take((size_t)nq * sizeof(int32_t));
    w.fin_dist = take((size_t)nq * kFinCap * sizeof(double));
    w.queue = take(sizeof(unsigned long long));
    w.total = off + 1024;
    return w;
}

static int make_rerank_params(RerankParams &rp, bool &warp_kernel, const float *vectors, const double *pp, int64_t n,
                              int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq, int64_t q_ld,
                              int32_t k, const uint8_t *overflow, void *workspace, size_t workspace_bytes);
static bool side_jobs_enabled() { return g_gemm_pair && g_side_job; }

}  // namespace morna

using namespace morna;

extern "C" int64_t morna_tensor_operand_ld(int32_t dim) { return ((int64_t)dim + gemm::BK - 1) / gemm::BK * gemm::BK; }

extern "C" int morna_prepare_tensor_operand(const float *vectors, const double *pp, int64_t n, int32_t dim,
                                            int64_t ld, void *hs, int64_t ld_h, float *rho_max, void *stream) {
    if (!vectors || !pp || !hs || !rho_max || n < 0 || dim <= 0 || ld < dim || (ld & 3) ||
        ld_h != morna_tensor_operand_ld(dim))
        return MORNA_ERR_INVALID_ARGUMENT;
    cudaStream_t s = (cudaStream_t)stream;
    MORNA_CUDA_TRY(cudaMemsetAsync(rho_max, 0, sizeof(float), s));
    if (n == 0) return MORNA_OK;
    int64_t blocks = (n + 7) / 8;
    if (blocks > (int64_t)sm_count_b() * 8) blocks = (int64_t)sm_count_b() * 8;
    prep_samples_kernel<<<(unsigned)blocks, kPrepThreads, 0, s>>>(vectors, pp, n, ld, (__half *)hs, ld_h, rho_max);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" size_t morna_knn_batched_workspace_bytes(int64_t n, int64_t nq, int32_t dim, int32_t k) {
    (void)k;
    if (n <= 0 || nq <= 0 || dim <= 0) return 1024;
    return batch_ws_layout(n, nq, morna_tensor_operand_ld(dim)).total;
}

// Scoring half of morna_knn_batched: fp16 tensor-core scores, thresholds and the final candidate
// lists of every query, left in the workspace (tensor-core bound; touches HBM lightly).
// final_mode: 0 = final candidate lists, 1 = this rank's score bounds only (kth_bound), 2 = leave the first-pass lists
static int score_impl(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                      int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                      uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes,
                      void *const *phase_events, const morna_rerank_job *side_job, float *kth_bound, int final_mode,
                      const int32_t *row_group, const int32_t *query_group, void *stream) {
    if (!hs || !rho_max || !queries || !overflow || !stats || n <= 0 || n > kBatchedMaxRows || nq <= 0 || dim <= 0 ||
        q_ld < dim || k <= 0 || k > kFinCap / 2 || ld_h != morna_tensor_operand_ld(dim) || !row_group != !query_group ||
        (row_group && final_mode == 1))
        return MORNA_ERR_INVALID_ARGUMENT;
    BatchWs w = batch_ws_layout(n, nq, ld_h);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    RerankParams side{};
    const RerankParams *side_ptr = nullptr;
    if (side_job) {                 // the previous batch's re-rank rides in this batch's GEMM launches
        if (side_job->workspace == workspace) return MORNA_ERR_INVALID_ARGUMENT;
        bool warp_kernel = true;
        int rcj = make_rerank_params(side, warp_kernel, side_job->vectors, side_job->pp, side_job->n, side_job->dim,
                                     side_job->ld, side_job->id_base, side_job->queries, side_job->nq, side_job->q_ld,
                                     side_job->k, side_job->overflow, side_job->workspace, side_job->workspace_bytes);
        if (rcj != MORNA_OK) return rcj;
        if (warp_kernel && side_jobs_enabled()) side_ptr = &side;            // otherwise everything is left to the resume call
    }
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace;
    __half *hq = (__half *)(ws + w.hq);
    double *qq = (double *)(ws + w.qq);
    float *eps = (float *)(ws + w.eps);
    float *pilot = (float *)(ws + w.pilot);
    float *thr = (float *)(ws + w.thr);
    float *cand_score = (float *)(ws + w.cand_score);
    int32_t *cand_id = (int32_t *)(ws + w.cand_id);
    int32_t *cand_cnt = (int32_t *)(ws + w.cand_cnt);
    int32_t *fin_id = (int32_t *)(ws + w.fin_id);
    int32_t *fin_cnt = (int32_t *)(ws + w.fin_cnt);

    int phase = 0;
    auto mark = [&]() { if (phase_events) cudaEventRecord((cudaEvent_t)phase_events[phase], s); ++phase; };
    mark();                                                      // 0: start
    MORNA_CUDA_TRY(cudaMemsetAsync(overflow, 0, (size_t)nq, s));
    MORNA_CUDA_TRY(cudaMemsetAsync(stats, 0, 4 * sizeof(int32_t), s));
    MORNA_CUDA_TRY(cudaMemsetAsync(cand_cnt, 0, (size_t)nq * sizeof(int32_t), s));
    MORNA_CUDA_TRY(cudaMemsetAsync(ws + w.queue, 0, sizeof(unsigned long long), s));     // this batch's re-rank queue

    // fp32 accumulation of dim products, each add off by at most one truncation ulp of a
    // partial sum bounded by |h_s||h_q| <= ~1; chain length dim/16 MMAs plus the in-MMA tree
    const float eps_acc = (float)((double)(dim / 16 + 8) * 2.384185791015625e-07 * 1.01);
    {
        int64_t blocks = (w.nq_pad + 7) / 8;
        if (blocks > (int64_t)sm_count_b() * 8) blocks = (int64_t)sm_count_b() * 8;
        prep_queries_kernel<<<(unsigned)blocks, kPrepThreads, 0, s>>>(queries, nq, w.nq_pad, dim, q_ld, hq, ld_h, qq,
                                                                    eps, rho_max, eps_acc, overflow, stats);
        MORNA_LAUNCH_CHECK();
    }
    mark();                                                      // 1: queries prepared
    CUtensorMap tmap_q, tmap_s;
    int rc = make_tmap(&tmap_q, hq, (uint64_t)w.nq_pad, (uint64_t)ld_h, gemm::BM);
    if (rc != MORNA_OK) return rc;
    rc = make_tmap(&tmap_s, hs, (uint64_t)n, (uint64_t)ld_h,
                   g_gemm_pair == 2 && !side_ptr && (w.nq_pad / gemm::BM) % 4 == 0 ? gemm2::BN_HALF / 2 : g_gemm_pair ? gemm2::BN_HALF : gemm::BN);
    if (rc != MORNA_OK) return rc;
    GemmParams gp{};
    gp.debug = g_gemm_debug; gp.relaxed_ns = g_gemm_relaxed_ns; gp.dry_epilogue = g_gemm_dry; gp.l2_keep = g_gemm_l2_keep;
    gp.nq = (int32_t)nq; gp.kblocks = (int32_t)(ld_h / gemm::BK); gp.m_blocks = (int32_t)(w.nq_pad / gemm::BM);
    gp.cap = kCandCap; gp.id_base = id_base; gp.pilot = pilot; gp.pilot_ld = w.pilot_ld; gp.thr = thr;
    gp.cand_score = cand_score; gp.cand_id = cand_id; gp.cand_cnt = cand_cnt;
    auto launch_gemm = [&](int32_t n_begin, int32_t n_end, int32_t mode) -> int {
        gp.n_begin = n_begin; gp.n_end = n_end; gp.mode = mode;
        gp.n_tiles = (n_end - n_begin + gemm::BN - 1) / gemm::BN;
        return launch_knn_gemm(tmap_q, tmap_s, gp, s, side_ptr);
    };
    KthParams kp{};
    kp.k = k; kp.n0 = (int32_t)w.n0; kp.n_begin = 0; kp.id_base = id_base; kp.cap = kCandCap; kp.fcap = kFinCap;
    kp.pilot = pilot; kp.pilot_ld = w.pilot_ld; kp.eps = eps; kp.thr = thr; kp.cand_score = cand_score;
    kp.cand_id = cand_id; kp.cand_cnt = cand_cnt; kp.fin_id = fin_id; kp.fin_cnt = fin_cnt; kp.overflow = overflow;
    kp.stats = stats; kp.row_group = row_group; kp.query_group = query_group;
    if ((rc = ensure_dynamic_smem((const void *)kth_warp_kernel<1>, kKwSmem)) != MORNA_OK) return rc;
    if ((rc = ensure_dynamic_smem((const void *)kth_warp_kernel<0>, kKwSmem)) != MORNA_OK) return rc;
    if ((rc = ensure_dynamic_smem((const void *)kth_warp_kernel<2>, kKwSmem)) != MORNA_OK) return rc;
    const unsigned kth_grid = (unsigned)((nq + kKwWarps - 1) / kKwWarps);

    rc = launch_gemm(0, (int32_t)w.n0, 0);                       // pilot block: dump scores
    if (rc != MORNA_OK) return rc;
    mark();                                                      // 2: pilot GEMM
    kth_warp_kernel<1><<<kth_grid, kKwWarps * 32, kKwSmem, s>>>(kp, (int)nq);
    MORNA_LAUNCH_CHECK();
    mark();                                                      // 3: thresholds
    // the rest in blocks of g_block_rows rows: keep scores above thr; between blocks thr is tightened to the
    // k-th best seen so far and the lists are compacted, so a later block adds ~k entries per query, not ~N/n0 * k
    // (key 36 lets the blocks grow geometrically: after the first refinement a query's threshold passes ~k/rows_seen of the
    // rows, so a block as large as everything seen so far adds about k entries to its list; off by default)
    int64_t step = g_block_rows;
    for (int64_t b0 = w.n0; b0 < n;) {
        int64_t b1 = b0 == w.n0 ? (int64_t)(g_first_block > 0 ? g_first_block : g_block_rows) : b0 + step;
        if (b0 != w.n0 && g_block_growth > 1) step *= g_block_growth;
        if (b1 <= b0) b1 = b0 + step;      // key 11 (or key 9) at or below the pilot rows: the first block is `step` rows, not the rest
        if (b1 > n) b1 = n;
        rc = launch_gemm((int32_t)b0, (int32_t)b1, 1);
        if (rc != MORNA_OK) return rc;
        b0 = b1;
        if (b0 < n) {
            kp.cand2_score = (float *)(ws + w.cand2_score);
            kp.cand2_id = (int32_t *)(ws + w.cand2_id);
            kth_warp_kernel<2><<<kth_grid, kKwWarps * 32, kKwSmem, s>>>(kp, (int)nq);
            MORNA_LAUNCH_CHECK();
            // the compacted lists are now the current ones
            float *ts = kp.cand_score; kp.cand_score = kp.cand2_score; kp.cand2_score = ts;
            int32_t *ti = kp.cand_id; kp.cand_id = kp.cand2_id; kp.cand2_id = ti;
            const size_t to = w.cand_score; w.cand_score = w.cand2_score; w.cand2_score = to;
            const size_t tj = w.cand_id; w.cand_id = w.cand2_id; w.cand2_id = tj;
            gp.cand_score = kp.cand_score; gp.cand_id = kp.cand_id;
        }
    }
    mark();                                                      // 4: filter GEMM(s)
    if (final_mode == 2) return MORNA_OK;
    if (final_mode == 1) {       // rows-sharded search: only this rank's bounds; morna_knn_batched_finalize builds the lists
        kp.kth_bound = kth_bound;
        if ((rc = ensure_dynamic_smem((const void *)kth_warp_kernel<3>, kKwSmem)) != MORNA_OK) return rc;
        kth_warp_kernel<3><<<kth_grid, kKwWarps * 32, kKwSmem, s>>>(kp, (int)nq);
    } else {
        kth_warp_kernel<0><<<kth_grid, kKwWarps * 32, kKwSmem, s>>>(kp, (int)nq);
    }
    MORNA_LAUNCH_CHECK();
    mark();                                                      // 5: final candidate lists
    return MORNA_OK;
}

extern "C" int morna_knn_batched_score(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                                       int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                                       uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes,
                                       void *const *phase_events, const morna_rerank_job *side_job, float *kth_bound,
                                       void *stream) {
    return score_impl(hs, ld_h, rho_max, n, dim, id_base, queries, nq, q_ld, k, overflow, stats, workspace, workspace_bytes,
                      phase_events, side_job, kth_bound, kth_bound ? 1 : 0, nullptr, nullptr, stream);
}

extern "C" int morna_knn_batched_score_excl(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                                            int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                                            uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes,
                                            void *const *phase_events, const morna_rerank_job *side_job, float *kth_bound,
                                            const int32_t *row_group, const int32_t *query_group, void *stream) {
    return score_impl(hs, ld_h, rho_max, n, dim, id_base, queries, nq, q_ld, k, overflow, stats, workspace, workspace_bytes,
                      phase_events, side_job, kth_bound, kth_bound ? 1 : 0, row_group, query_group, stream);
}

namespace morna {
// which of the two first-pass list buffers is current after a scoring call: one swap per refinement between row blocks
static int list_swaps(int64_t n, const BatchWs &w) {
    int swaps = 0;                                               // (the same walk as score_impl's block loop)
    int64_t step = g_block_rows;
    for (int64_t b0 = w.n0; b0 < n;) {
        int64_t b1 = b0 == w.n0 ? (int64_t)(g_first_block > 0 ? g_first_block : g_block_rows) : b0 + step;
        if (b0 != w.n0 && g_block_growth > 1) step *= g_block_growth;
        if (b1 <= b0) b1 = b0 + step;
        if (b1 > n) b1 = n;
        b0 = b1;
        if (b0 < n) ++swaps;
    }
    return swaps;
}

// Approximate mode: the k best rows by fp16 tensor-core score, no FP64 re-rank.  One CTA per query sorts the
// first-pass list (score descending, then id descending) in shared memory; distance = sqrt(2 - 2 score).
constexpr int kApproxThreads = 512;
__global__ void __launch_bounds__(kApproxThreads)
approx_topk_kernel(const float *__restrict__ cand_score, const int32_t *__restrict__ cand_id, const int32_t *__restrict__ cand_cnt,
                   int32_t cap, int32_t k, uint8_t *__restrict__ overflow, int32_t *__restrict__ stats,
                   int32_t *__restrict__ out_ids, double *__restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *ss = reinterpret_cast<float *>(smem_raw);          // [P]
    int *si = reinterpret_cast<int *>(ss + cap);              // [P]
    const int q = blockIdx.x, tid = threadIdx.x;
    int32_t *oi = out_ids + (int64_t)q * k;
    double *od = out_dist + (int64_t)q * k;
    const int count = cand_cnt[q];
    if (count > cap || overflow[q]) {                        // survivors were dropped (massive ties): the exact scan answers
        if (tid == 0) { if (!overflow[q]) atomicAdd(stats + 0, 1); overflow[q] = 1; }
        for (int i = tid; i < k; i += kApproxThreads) { oi[i] = -1; od[i] = INFINITY; }
        return;
    }
    int P = 32;
    while (P < count) P <<= 1;
    for (int i = tid; i < P; i += kApproxThreads) {
        const bool have = i < count;
        ss[i] = have ? cand_score[(int64_t)q * cap + i] : -INFINITY;
        si[i] = have ? cand_id[(int64_t)q * cap + i] : -1;
    }
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = tid; i < (P >> 1); i += kApproxThreads) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const float sl = ss[lo], sh = ss[hi];
                const int il = si[lo], ih = si[hi];
                const bool hi_first = sh > sl || (sh == sl && ih > il);      // larger score first, then larger id
                const bool lo_first = sl > sh || (sl == sh && il > ih);
                if (asc ? hi_first : lo_first) { ss[lo] = sh; ss[hi] = sl; si[lo] = ih; si[hi] = il; }
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < k; i += kApproxThreads) {
        const bool ok = i < count && si[i] >= 0;
        oi[i] = ok ? si[i] : -1;
        double d = 2.0 - 2.0 * (double)ss[i < P ? i : 0];
        if (d < 0.0) d = 0.0;
        od[i] = ok ? sqrt(d) : INFINITY;
    }
    if (tid == 0) atomicAdd(stats + 1, count);
}
}  // namespace morna

extern "C" int morna_knn_batched_approx(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                                        int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                                        int32_t *out_ids, double *out_dist, uint8_t *overflow, int32_t *stats,
                                        void *workspace, size_t workspace_bytes, void *stream) {
    if (!out_ids || !out_dist) return MORNA_ERR_INVALID_ARGUMENT;
    int rc = score_impl(hs, ld_h, rho_max, n, dim, id_base, queries, nq, q_ld, k, overflow, stats, workspace, workspace_bytes,
                        nullptr, nullptr, nullptr, 2, nullptr, nullptr, stream);
    if (rc != MORNA_OK) return rc;
    BatchWs w = batch_ws_layout(n, nq, ld_h);
    unsigned char *ws = (unsigned char *)workspace;
    const int swaps = list_swaps(n, w);
    const float *cs = (const float *)(ws + ((swaps & 1) ? w.cand2_score : w.cand_score));
    const int32_t *ci = (const int32_t *)(ws + ((swaps & 1) ? w.cand2_id : w.cand_id));
    const size_t smem = (size_t)kCandCap * (sizeof(float) + sizeof(int));
    morna::approx_topk_kernel<<<(unsigned)nq, morna::kApproxThreads, smem, (cudaStream_t)stream>>>(
        cs, ci, (const int32_t *)(ws + w.cand_cnt), kCandCap, k, overflow, stats, out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

namespace morna {
// k-th largest of the n_lists * k lower bounds the ranks gathered for a query (one warp per query, bisection on the
// monotone keys): at least k distinct rows over all shards have a true cosine >= the result.
template <int kPerLane>
__global__ void __launch_bounds__(256)
union_kth_kernel(const float *__restrict__ vals, int32_t n_lists, int64_t nq, int32_t k, float *__restrict__ bound) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (q >= nq) return;
    const int total = n_lists * k;
    uint32_t best = 0;
    if (kPerLane > 0) {                       // the values fit in registers: one load each, 32 counting steps on registers
        uint32_t key[kPerLane > 0 ? kPerLane : 1];
#pragma unroll
        for (int j = 0; j < kPerLane; ++j) {
            const int e = j * 32 + lane;
            key[j] = 0u;                      // below every real key
            if (e < total) { const int g = e / k, i = e - g * k; key[j] = float_key(vals[((int64_t)g * nq + q) * k + i]); }
        }
        for (int bit = 31; bit >= 0; --bit) {
            const uint32_t trial = best | (1u << bit);
            int c = 0;
#pragma unroll
            for (int j = 0; j < kPerLane; ++j) c += key[j] >= trial;
            c = __reduce_add_sync(kFull, c);
            if (c >= k) best = trial;
        }
    } else {
        for (int bit = 31; bit >= 0; --bit) {
            const uint32_t trial = best | (1u << bit);
            int c = 0;
            for (int e = lane; e < total; e += 32) {
                const int g = e / k, j = e - g * k;
                c += float_key(vals[((int64_t)g * nq + q) * k + j]) >= trial;
            }
            c = __reduce_add_sync(kFull, c);
            if (c >= k) best = trial;
        }
    }
    if (lane == 0) bound[q] = best ? key_float(best) : -INFINITY;     // fewer than k values in all: no bound
}
}  // namespace morna

extern "C" int morna_union_kth_bound(const float *vals, int32_t n_lists, int64_t nq, int32_t k, float *bound, void *stream) {
    if (!vals || !bound || n_lists <= 0 || nq < 0 || k <= 0) return MORNA_ERR_INVALID_ARGUMENT;
    if (nq == 0) return MORNA_OK;
    const unsigned grid = (unsigned)((nq + 7) / 8);
    const int64_t total = (int64_t)n_lists * k;
    if (total <= 32 * 8) morna::union_kth_kernel<8><<<grid, 256, 0, (cudaStream_t)stream>>>(vals, n_lists, nq, k, bound);
    else if (total <= 32 * 32) morna::union_kth_kernel<32><<<grid, 256, 0, (cudaStream_t)stream>>>(vals, n_lists, nq, k, bound);
    else morna::union_kth_kernel<0><<<grid, 256, 0, (cudaStream_t)stream>>>(vals, n_lists, nq, k, bound);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

// Rows-sharded search, second half of the scoring: every query's final candidate list from a bound on the k-th best
// cosine that holds over ALL shards -- the caller all-reduces (MAX) the kth_bound arrays the ranks' scoring calls wrote.
// A row of the global top-k has true cosine >= that bound, hence a score >= bound - eps of this rank.
extern "C" int morna_knn_batched_finalize(int64_t n, int64_t nq, int32_t dim, int32_t k, const float *kth_bound,
                                          uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes,
                                          void *stream) {
    if (!kth_bound || !overflow || !stats || n <= 0 || n > kBatchedMaxRows || nq <= 0 || dim <= 0 || k <= 0 || k > kFinCap / 2)
        return MORNA_ERR_INVALID_ARGUMENT;
    BatchWs w = batch_ws_layout(n, nq, morna_tensor_operand_ld(dim));
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    unsigned char *ws = (unsigned char *)workspace;
    // which of the two list buffers is current: one swap per refinement between row blocks (same walk as the scoring call)
    const int swaps = list_swaps(n, w);
    KthParams kp{};
    kp.k = k; kp.n0 = (int32_t)w.n0; kp.cap = kCandCap; kp.fcap = kFinCap; kp.eps = (const float *)(ws + w.eps);
    kp.cand_score = (float *)(ws + ((swaps & 1) ? w.cand2_score : w.cand_score));
    kp.cand_id = (int32_t *)(ws + ((swaps & 1) ? w.cand2_id : w.cand_id));
    kp.cand_cnt = (int32_t *)(ws + w.cand_cnt); kp.fin_id = (int32_t *)(ws + w.fin_id); kp.fin_cnt = (int32_t *)(ws + w.fin_cnt);
    kp.overflow = overflow; kp.stats = stats; kp.kth_bound = const_cast<float *>(kth_bound);
    { int rca = ensure_dynamic_smem((const void *)kth_warp_kernel<4>, kKwSmem); if (rca != MORNA_OK) return rca; }
    kth_warp_kernel<4><<<(unsigned)((nq + kKwWarps - 1) / kKwWarps), kKwWarps * 32, kKwSmem, (cudaStream_t)stream>>>(kp, (int)nq);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

namespace morna {

// parameters of a batch's re-rank from the workspace its scoring half filled
static int make_rerank_params(RerankParams &rp, bool &warp_kernel, const float *vectors, const double *pp, int64_t n,
                              int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq, int64_t q_ld,
                              int32_t k, const uint8_t *overflow, void *workspace, size_t workspace_bytes) {
    if (!vectors || !pp || !queries || !overflow || n <= 0 || n > kBatchedMaxRows || nq <= 0 || dim <= 0 || ld < dim ||
        (ld & 3) || q_ld < dim || k <= 0 || k > kFinCap / 2)
        return MORNA_ERR_INVALID_ARGUMENT;
    BatchWs w = batch_ws_layout(n, nq, morna_tensor_operand_ld(dim));
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    unsigned char *ws = (unsigned char *)workspace;
    rp = RerankParams{};
    rp.vectors = vectors; rp.pp = pp; rp.ld = ld; rp.dim = dim; rp.id_base = id_base; rp.n = (int32_t)n;
    rp.queries = queries; rp.q_ld = q_ld; rp.qq = (const double *)(ws + w.qq);
    rp.fin_id = (const int32_t *)(ws + w.fin_id); rp.fin_cnt = (const int32_t *)(ws + w.fin_cnt); rp.overflow = overflow;
    rp.fcap = kFinCap; rp.nq = (int32_t)nq; rp.fin_dist = (double *)(ws + w.fin_dist);
    rp.queue = (unsigned long long *)(ws + w.queue);
    rp.rows_evict_first = g_rerank_evict_first;
    rp.sort_rows = g_rerank_sort_rows;
    // phases: only when a row is re-ranked several times per batch (otherwise every row is read at
    // most about once and splitting would only re-read the queries)
    rp.phases = 1; rp.phase_rows = (int32_t)n; rp.subs = 1;
    const double reuse = (double)nq * (1.2 * k) / (double)n;
    const size_t rr_smem = (size_t)ld * sizeof(double) + (size_t)kFinCap * sizeof(int);
    warp_kernel = g_rerank_kernel == 0 || rr_smem > 200 * 1024;
    const int phase_mb = g_rerank_phase_mb >= 0 ? g_rerank_phase_mb : (warp_kernel ? 64 : 0);
    if (phase_mb > 0 && reuse >= 3.0) {
        int64_t rows = ((int64_t)phase_mb << 20) / ((int64_t)ld * 4);
        if (rows < 1024) rows = 1024;
        if (rows < n) {
            rp.phases = (int32_t)((n + rows - 1) / rows);
            rp.phase_rows = (int32_t)((n + rp.phases - 1) / rp.phases);
        }
    }
    if (warp_kernel && rp.phases == 1) rp.subs = g_rerank_subs > 0 ? g_rerank_subs : 4;     // short items: helper warps leave promptly
    return MORNA_OK;
}

}  // namespace morna

// Re-rank half: exact FP64 distances of the candidate lists a previous morna_knn_batched_score left
// in the same workspace, ordered under the reference rule (HBM/L2-gather bound; no tensor cores).
// resume != 0: a later morna_knn_batched_score call carried this batch as its side job -- only what its
// helper warps left in the queue is re-ranked here.
extern "C" int morna_knn_batched_rerank(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                        int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                                        int32_t *out_ids, double *out_dist, const uint8_t *overflow, void *workspace,
                                        size_t workspace_bytes, int32_t resume, void *stream) {
    if (!out_ids || !out_dist) return MORNA_ERR_INVALID_ARGUMENT;
    RerankParams rp;
    bool warp_kernel = true;
    int rc = make_rerank_params(rp, warp_kernel, vectors, pp, n, dim, ld, id_base, queries, nq, q_ld, k, overflow, workspace,
                                workspace_bytes);
    if (rc != MORNA_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (resume && !(warp_kernel && side_jobs_enabled())) resume = 0;        // no helper warps ran: the whole batch is still to do
    if (warp_kernel) {
        // warp-granular items (any dim: the query is read from global memory)
        if (!resume) MORNA_CUDA_TRY(cudaMemsetAsync(rp.queue, 0, sizeof(unsigned long long), s));
        auto kern = g_rerank_rows == 16 ? rerank_warp_kernel<16, 1> : g_rerank_rows == 2 ? rerank_warp_kernel<4, 4>
                                                                                       : rerank_warp_kernel<8, 2>;
        const size_t smem = (size_t)kRwWarps * kFinCap * sizeof(int);
        // shared-memory carve-out at its maximum, so that CTAs of this kernel and the GEMM (130 KB) can share an SM
        MORNA_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int per_sm = 0;
        MORNA_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRwWarps * 32, smem));
        if (per_sm < 1) per_sm = 1;
        if (g_rerank_ctas > 0 && per_sm > g_rerank_ctas) per_sm = g_rerank_ctas;
        const int64_t items = (int64_t)nq * rp.phases * rp.subs;
        int64_t grid = (int64_t)per_sm * sm_count_b();
        if (grid * kRwWarps > items) grid = (items + kRwWarps - 1) / kRwWarps;
        kern<<<(unsigned)grid, kRwWarps * 32, smem, s>>>(rp);
        MORNA_LAUNCH_CHECK();
    } else {
        const size_t rr_smem = (size_t)ld * sizeof(double) + (size_t)kFinCap * sizeof(int);
        auto kern = g_rerank_rows == 2 ? rerank_dist_kernel<2> : g_rerank_rows == 4 ? rerank_dist_kernel<4> : rerank_dist_kernel<8>;
        if (g_rerank_pipe) kern = g_rerank_rows == 4 ? rerank_dist_kernel<4, true> : g_rerank_rows == 16 ? rerank_dist_kernel<16, true>
                                                                                                        : rerank_dist_kernel<8, true>;
        if ((rc = ensure_dynamic_smem((const void *)kern, rr_smem)) != MORNA_OK) return rc;
        int per_sm = 0;
        MORNA_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRrThreads, rr_smem));
        if (per_sm < 1) per_sm = 1;
        if (g_rerank_ctas_per_sm > 0 && per_sm > g_rerank_ctas_per_sm) per_sm = g_rerank_ctas_per_sm;
        const int64_t items = (int64_t)nq * rp.phases;
        int64_t rr_grid = (int64_t)per_sm * sm_count_b();
        if (rr_grid > items || g_rerank_oneshot) rr_grid = items;
        if (g_carveout_hint) cudaFuncSetAttribute((const void *)kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        const size_t fat_smem = (((size_t)ld * sizeof(double) + (size_t)kFinCap * sizeof(int) + 15) & ~(size_t)15) * kRrFatSubs;
        if (g_rerank_fat_sms > 0 && rp.phases == 1 && fat_smem <= 200 * 1024) {
            // SM partition: X SM-filling CTAs (in pairs); the scoring kernels' grids leave those SMs alone (key 30)
            auto fat = rerank_fat_kernel<4, true>;
            if ((rc = ensure_dynamic_smem((const void *)fat, fat_smem)) != MORNA_OK) return rc;
            MORNA_CUDA_TRY(cudaMemsetAsync(rp.queue, 0, sizeof(unsigned long long), s));
            int ctas = g_rerank_fat_sms / 2 * 2;
            if (ctas > sm_count_b()) ctas = sm_count_b() / 2 * 2;
            if (ctas < 2) ctas = 2;
            fat<<<(unsigned)ctas, kRrThreads * kRrFatSubs, fat_smem, s>>>(rp);
        } else {
            kern<<<(unsigned)rr_grid, kRrThreads, rr_smem, s>>>(rp);
        }
        MORNA_LAUNCH_CHECK();
    }
    const size_t or_smem = (size_t)kFinCap * (sizeof(double) + sizeof(int));
    rerank_order_kernel<<<(unsigned)nq, kOrderThreads, or_smem, s>>>(rp.fin_id, rp.fin_cnt, rp.fin_dist, overflow, kFinCap, k,
                                                                    out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" int morna_knn_batched(const float *vectors, const double *pp, const void *hs, int64_t ld_h,
                                 const float *rho_max, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                                 const double *queries, int64_t nq, int64_t q_ld, int32_t k, int32_t *out_ids,
                                 double *out_dist, uint8_t *overflow, int32_t *stats, void *workspace,
                                 size_t workspace_bytes, void *const *phase_events, void *stream) {
    if (!vectors || !pp || !out_ids || !out_dist || ld < dim || (ld & 3)) return MORNA_ERR_INVALID_ARGUMENT;
    int rc = morna_knn_batched_score(hs, ld_h, rho_max, n, dim, id_base, queries, nq, q_ld, k, overflow, stats,
                                     workspace, workspace_bytes, phase_events, nullptr, nullptr, stream);
    if (rc != MORNA_OK) return rc;
    rc = morna_knn_batched_rerank(vectors, pp, n, dim, ld, id_base, queries, nq, q_ld, k, out_ids, out_dist, overflow,
                                  workspace, workspace_bytes, 0, stream);
    if (rc == MORNA_OK && phase_events) cudaEventRecord((cudaEvent_t)phase_events[6], (cudaStream_t)stream);
    return rc;
}

// Raw fp16 tensor-core scores of a query block against the first n0 samples, plus the
// per-query error bound -- used by tests to validate eps against exact cosines.
extern "C" int morna_debug_tensor_scores(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                                         const double *queries, int64_t nq, int64_t q_ld, float *scores,
                                         int64_t scores_ld, float *eps_out, void *workspace, size_t workspace_bytes,
                                         void *stream) {
    if (!hs || !rho_max || !queries || !scores || !eps_out || n <= 0 || nq <= 0 || scores_ld < n || (scores_ld & 3) ||
        ld_h != morna_tensor_operand_ld(dim))
        return MORNA_ERR_INVALID_ARGUMENT;
    BatchWs w = batch_ws_layout(n, nq, ld_h);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace;
    __half *hq = (__half *)(ws + w.hq);
    double *qq = (double *)(ws + w.qq);
    const float eps_acc = (float)((double)(dim / 16 + 8) * 2.384185791015625e-07 * 1.01);
    int64_t blocks = (w.nq_pad + 7) / 8;
    prep_queries_kernel<<<(unsigned)blocks, kPrepThreads, 0, s>>>(queries, nq, w.nq_pad, dim, q_ld, hq, ld_h, qq,
                                                                eps_out, rho_max, eps_acc, nullptr, nullptr);
    MORNA_LAUNCH_CHECK();
    CUtensorMap tmap_q, tmap_s;
    int rc = make_tmap(&tmap_q, hq, (uint64_t)w.nq_pad, (uint64_t)ld_h, gemm::BM);
    if (rc != MORNA_OK) return rc;
    rc = make_tmap(&tmap_s, hs, (uint64_t)n, (uint64_t)ld_h,
                   g_gemm_pair == 2 && (w.nq_pad / gemm::BM) % 4 == 0 ? gemm2::BN_HALF / 2 : g_gemm_pair ? gemm2::BN_HALF : gemm::BN);
    if (rc != MORNA_OK) return rc;
    GemmParams gp{};
    gp.nq = (int32_t)nq; gp.kblocks = (int32_t)(ld_h / gemm::BK); gp.m_blocks = (int32_t)(w.nq_pad / gemm::BM);
    gp.n_begin = 0; gp.n_end = (int32_t)n; gp.mode = 0; gp.pilot = scores; gp.pilot_ld = scores_ld;
    gp.n_tiles = (gp.n_end + gemm::BN - 1) / gemm::BN;
    return launch_knn_gemm(tmap_q, tmap_s, gp, s);
}

// ------------------------------------------------------------------ range search, tensor-core route
// With the radius known up front there is no pilot, no k-th selection and no refinement between row blocks: the query
// prep, one filter GEMM over all rows with thresholds fixed before it starts, and an FP64 check of every survivor.
//
// Threshold.  Let c be the exact cosine of (q, i) and d_fp the FP64 distance the scan returns.  d_fp <= R implies
// c >= 1 - R^2/2 - delta_fp, where delta_fp covers the canonical sums' rounding (at most ~dim * 2^-53 relative to
// |p||q|, 3.3e-12 at dim = 30,000) and that of the division, sqrt and the final subtraction (a few ulps of 2).  The
// fp16 score s has |s - c| <= eps[q] (prep_queries_kernel).  So every row in range scores
// s >= (1 - R^2/2) - eps[q] - delta_fp >= (1 - R^2/2) - eps[q] - 2^-30, and thr[q] is that double rounded down to a
// float: the filter drops no row in range.  A zero query or zero row scores 0 and sits at sqrt(2); it passes whenever
// R >= sqrt(2), where the bound is <= -eps - 2^-30 < 0.
namespace morna {

constexpr int kRangeMaxQueries = 4096;
constexpr int kRangeWarps = 8;
constexpr int kRangeEmitThreads = 512;

struct RangeWs {
    size_t hq, qq, eps, thr, cand_score, cand_id, cand_cnt, match_id, match_dist, match_cnt, prep_stats, total;
    int64_t nq_pad;
};
static RangeWs range_ws_layout(int64_t nq, int64_t ld_h) {
    RangeWs w{};
    w.nq_pad = (nq + 2 * gemm::BM - 1) / (2 * gemm::BM) * (2 * gemm::BM);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off += align_up(bytes, 256); return at; };
    w.hq = take((size_t)w.nq_pad * ld_h * sizeof(__half));
    w.qq = take((size_t)nq * sizeof(double));
    w.eps = take((size_t)nq * sizeof(float));
    w.thr = take((size_t)nq * sizeof(float));
    w.cand_score = take((size_t)nq * kCandCap * sizeof(float));
    w.cand_id = take((size_t)nq * kCandCap * sizeof(int32_t));
    w.cand_cnt = take((size_t)nq * sizeof(int32_t));
    w.match_id = take((size_t)nq * kCandCap * sizeof(int32_t));
    w.match_dist = take((size_t)nq * kCandCap * sizeof(double));
    w.match_cnt = take((size_t)nq * sizeof(int32_t));
    w.prep_stats = take(4 * sizeof(int32_t));
    w.total = off + 1024;
    return w;
}

__global__ void range_thr_kernel(const float *__restrict__ eps, const uint8_t *__restrict__ overflow, int32_t nq, double R,
                                 float *__restrict__ thr) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const double t = (1.0 - 0.5 * R * R) - (double)eps[q] - 0x1p-30;
    thr[q] = overflow[q] ? INFINITY : __double2float_rd(t);      // a flagged query collects nothing: the FP64 route answers it
}

struct RangeCheckParams {
    const float *vectors; const double *pp; int64_t ld; int32_t dim, id_base, nq;
    const double *queries; int64_t q_ld; const double *qq;
    const int32_t *cand_id; const int32_t *cand_cnt; const uint8_t *overflow;
    double R;
    int32_t *match_id; double *match_dist; int32_t *match_cnt;
    const int32_t *row_group; const int32_t *query_group;      // per-query exclusion (nullptr = off), as in KthParams
};

// A work item is (32-candidate window, query) of a first-pass list, one warp each: the window's rows go through
// rerank_rows (canonical sums, query read from global memory, so any dim) 4 at a time, and the rows within R are
// appended to the query's match list.  Windows past a list's end, and queries that overflowed, are skipped.
__global__ void __launch_bounds__(kRangeWarps * 32)
range_check_kernel(const RangeCheckParams p) {
    constexpr int kRows = 4, kWindows = kCandCap / 32;
    const int lane = threadIdx.x & 31;
    const long long total = (long long)p.nq * kWindows;
    const long long warps = (long long)gridDim.x * kRangeWarps;
    const bool vec_ok = ((p.q_ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(p.queries) & 15) == 0);
    const int chunks = (int)(p.ld >> 2);
    for (long long t = (long long)blockIdx.x * kRangeWarps + (threadIdx.x >> 5); t < total; t += warps) {
        // window-major: the live items (the first windows of every query) are spread evenly over the warps
        const int win = (int)(t / p.nq), q = (int)(t - (long long)win * p.nq), i0 = win * 32;
        const int count = p.cand_cnt[q];
        if (count > kCandCap || p.overflow[q] || i0 >= count) continue;
        const int m = min(32, count - i0);
        const int32_t *ids = p.cand_id + (int64_t)q * kCandCap + i0;
        const double *qsrc = p.queries + (int64_t)q * p.q_ld;
        const double qqv = p.qq[q];
        const int32_t qgroup = p.row_group ? p.query_group[q] : -1;
        for (int g = 0; g < m; g += kRows) {
            const int cnt = min(kRows, m - g);
            const float4 *src[kRows];
            int my_id = 0;
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                const int id = ids[min(g + u, m - 1)];
                src[u] = reinterpret_cast<const float4 *>(p.vectors + (int64_t)(id - p.id_base) * p.ld);
                if (lane == u) my_id = id;
            }
            double acc[kRows];
            rerank_rows<kRows, 4, false>(src, cnt, qsrc, p.dim, chunks, vec_ok, lane, acc);
            double mine = 0.0;
#pragma unroll
            for (int u = 0; u < kRows; ++u) {
                if (u < cnt) {                                           // cnt is warp-uniform
                    const double s = warp_sum(acc[u]);
                    if (lane == u) mine = s;
                }
            }
            double d = 0.0;
            if (lane < cnt) d = angular_from_sums(p.pp[my_id - p.id_base], qqv, mine);
            const bool keep = lane < cnt && !(qgroup >= 0 && p.row_group[my_id - p.id_base] == qgroup) && d <= p.R;
            const unsigned mask = __ballot_sync(kFull, keep);
            if (mask) {
                int at = 0;
                if (lane == 0) at = atomicAdd(p.match_cnt + q, __popc(mask));
                at = __shfl_sync(kFull, at, 0) + __popc(mask & ((1u << lane) - 1u));
                if (keep) {                                              // at < kCandCap: matches are a subset of the list
                    p.match_id[(int64_t)q * kCandCap + at] = my_id;
                    p.match_dist[(int64_t)q * kCandCap + at] = d;
                }
            }
        }
    }
}

__global__ void range_finish_kernel(const int32_t *__restrict__ cand_cnt, const int32_t *__restrict__ match_cnt, int32_t nq,
                                    uint8_t *__restrict__ overflow, int32_t *__restrict__ counts,
                                    unsigned long long *__restrict__ stats) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int c = cand_cnt[q];
    const bool over = overflow[q] || c > kCandCap;
    const int m = over ? 0 : match_cnt[q];
    overflow[q] = over ? 1 : 0;
    counts[q] = m;
    if (over) atomicAdd(stats + 0, 1ull);
    if (c) atomicAdd(stats + 1, (unsigned long long)c);
    if (m) { atomicAdd(stats + 2, (unsigned long long)m); atomicMax(stats + 3, (unsigned long long)m); }
}

// One CTA per query: its matches sorted under the reference order (bitonic network in shared memory), written to
// out[offsets[q], offsets[q+1]).
__global__ void __launch_bounds__(kRangeEmitThreads)
range_emit_kernel(const int32_t *__restrict__ match_id, const double *__restrict__ match_dist, const int32_t *__restrict__ match_cnt,
                  const uint8_t *__restrict__ overflow, const int64_t *__restrict__ offsets, int32_t *__restrict__ out_ids,
                  double *__restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *sd = reinterpret_cast<double *>(smem_raw);                 // [kCandCap]
    int *si = reinterpret_cast<int *>(sd + kCandCap);                  // [kCandCap]
    const int tid = threadIdx.x, q = blockIdx.x;
    const int64_t o = offsets[q];
    const int64_t room = offsets[q + 1] - o;
    if (overflow[q] || room <= 0) return;
    const int count = min(match_cnt[q], kCandCap);
    int P = 32;
    while (P < count) P <<= 1;
    for (int i = tid; i < P; i += kRangeEmitThreads) {
        const bool have = i < count;
        sd[i] = have ? match_dist[(int64_t)q * kCandCap + i] : INFINITY;
        si[i] = have ? match_id[(int64_t)q * kCandCap + i] : -1;
    }
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = tid; i < (P >> 1); i += kRangeEmitThreads) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool asc = (lo & size) == 0;
                const double dl = sd[lo], dh = sd[hi];
                const int il = si[lo], ih = si[hi];
                if (asc ? before(dh, ih, dl, il) : before(dl, il, dh, ih)) { sd[lo] = dh; sd[hi] = dl; si[lo] = ih; si[hi] = il; }
            }
        }
    }
    __syncthreads();
    const int n_out = (int)min((int64_t)count, room);
    for (int i = tid; i < n_out; i += kRangeEmitThreads) { out_ids[o + i] = si[i]; out_dist[o + i] = sd[i]; }
}

}  // namespace morna

extern "C" size_t morna_range_batched_workspace_bytes(int64_t n, int64_t nq, int32_t dim) {
    if (n <= 0 || nq <= 0 || dim <= 0) return 1024;
    return range_ws_layout(nq, morna_tensor_operand_ld(dim)).total;
}

extern "C" int morna_range_batched(const float *vectors, const double *pp, const void *hs, int64_t ld_h, const float *rho_max,
                                   int64_t n, int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq,
                                   int64_t q_ld, double max_distance, int32_t *counts, uint8_t *overflow, int64_t *stats,
                                   void *workspace, size_t workspace_bytes, void *stream) {
    return morna_range_batched_excl(vectors, pp, hs, ld_h, rho_max, n, dim, ld, id_base, queries, nq, q_ld, max_distance, counts,
                                    overflow, stats, workspace, workspace_bytes, nullptr, nullptr, stream);
}

extern "C" int morna_range_batched_excl(const float *vectors, const double *pp, const void *hs, int64_t ld_h, const float *rho_max,
                                        int64_t n, int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq,
                                        int64_t q_ld, double max_distance, int32_t *counts, uint8_t *overflow, int64_t *stats,
                                        void *workspace, size_t workspace_bytes, const int32_t *row_group,
                                        const int32_t *query_group, void *stream) {
    if (!row_group != !query_group) return MORNA_ERR_INVALID_ARGUMENT;
    if (!vectors || !pp || !hs || !rho_max || !queries || !counts || !overflow || !stats || n <= 0 || n > kBatchedMaxRows ||
        nq <= 0 || nq > kRangeMaxQueries || dim <= 0 || ld < dim || (ld & 3) || q_ld < dim ||
        ld_h != morna_tensor_operand_ld(dim) || !(max_distance >= 0.0) || isinf(max_distance))
        return MORNA_ERR_INVALID_ARGUMENT;
    const RangeWs w = range_ws_layout(nq, ld_h);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace;
    __half *hq = (__half *)(ws + w.hq);
    double *qq = (double *)(ws + w.qq);
    float *eps = (float *)(ws + w.eps);
    float *thr = (float *)(ws + w.thr);
    int32_t *cand_cnt = (int32_t *)(ws + w.cand_cnt);
    int32_t *match_cnt = (int32_t *)(ws + w.match_cnt);
    MORNA_CUDA_TRY(cudaMemsetAsync(overflow, 0, (size_t)nq, s));
    MORNA_CUDA_TRY(cudaMemsetAsync(stats, 0, 4 * sizeof(int64_t), s));
    MORNA_CUDA_TRY(cudaMemsetAsync(cand_cnt, 0, (size_t)nq * sizeof(int32_t), s));
    MORNA_CUDA_TRY(cudaMemsetAsync(match_cnt, 0, (size_t)nq * sizeof(int32_t), s));
    MORNA_CUDA_TRY(cudaMemsetAsync(ws + w.prep_stats, 0, 4 * sizeof(int32_t), s));

    const float eps_acc = (float)((double)(dim / 16 + 8) * 2.384185791015625e-07 * 1.01);     // as in score_impl
    {
        int64_t blocks = (w.nq_pad + 7) / 8;
        if (blocks > (int64_t)sm_count_b() * 8) blocks = (int64_t)sm_count_b() * 8;
        prep_queries_kernel<<<(unsigned)blocks, kPrepThreads, 0, s>>>(queries, nq, w.nq_pad, dim, q_ld, hq, ld_h, qq, eps, rho_max,
                                                                    eps_acc, overflow, (int32_t *)(ws + w.prep_stats));
        MORNA_LAUNCH_CHECK();
    }
    range_thr_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(eps, overflow, (int32_t)nq, max_distance, thr);
    MORNA_LAUNCH_CHECK();

    CUtensorMap tmap_q, tmap_s;
    int rc = make_tmap(&tmap_q, hq, (uint64_t)w.nq_pad, (uint64_t)ld_h, gemm::BM);
    if (rc != MORNA_OK) return rc;
    rc = make_tmap(&tmap_s, hs, (uint64_t)n, (uint64_t)ld_h,
                   g_gemm_pair == 2 && (w.nq_pad / gemm::BM) % 4 == 0 ? gemm2::BN_HALF / 2 : g_gemm_pair ? gemm2::BN_HALF : gemm::BN);
    if (rc != MORNA_OK) return rc;
    GemmParams gp{};
    gp.debug = g_gemm_debug; gp.relaxed_ns = g_gemm_relaxed_ns; gp.l2_keep = g_gemm_l2_keep;
    gp.nq = (int32_t)nq; gp.kblocks = (int32_t)(ld_h / gemm::BK); gp.m_blocks = (int32_t)(w.nq_pad / gemm::BM);
    gp.cap = kCandCap; gp.id_base = id_base; gp.thr = thr;
    gp.cand_score = (float *)(ws + w.cand_score); gp.cand_id = (int32_t *)(ws + w.cand_id); gp.cand_cnt = cand_cnt;
    gp.n_begin = 0; gp.n_end = (int32_t)n; gp.mode = 1;
    gp.n_tiles = (int32_t)((n + gemm::BN - 1) / gemm::BN);
    if ((rc = launch_knn_gemm(tmap_q, tmap_s, gp, s)) != MORNA_OK) return rc;

    RangeCheckParams cp{};
    cp.vectors = vectors; cp.pp = pp; cp.ld = ld; cp.dim = dim; cp.id_base = id_base; cp.nq = (int32_t)nq;
    cp.queries = queries; cp.q_ld = q_ld; cp.qq = qq; cp.cand_id = gp.cand_id; cp.cand_cnt = cand_cnt; cp.overflow = overflow;
    cp.R = max_distance; cp.match_id = (int32_t *)(ws + w.match_id); cp.match_dist = (double *)(ws + w.match_dist);
    cp.match_cnt = match_cnt; cp.row_group = row_group; cp.query_group = query_group;
    int per_sm = 0;
    MORNA_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, range_check_kernel, kRangeWarps * 32, 0));
    if (per_sm < 1) per_sm = 1;
    const int64_t items = nq * (kCandCap / 32);
    int64_t grid = (int64_t)per_sm * sm_count_b();
    if (grid * kRangeWarps > items) grid = (items + kRangeWarps - 1) / kRangeWarps;
    range_check_kernel<<<(unsigned)grid, kRangeWarps * 32, 0, s>>>(cp);
    MORNA_LAUNCH_CHECK();
    range_finish_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(cand_cnt, match_cnt, (int32_t)nq, overflow, counts,
                                                                    (unsigned long long *)stats);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" int morna_range_batched_emit(int64_t n, int64_t nq, int32_t dim, const int64_t *offsets, const uint8_t *overflow,
                                        int32_t *out_ids, double *out_dist, const void *workspace, size_t workspace_bytes,
                                        void *stream) {
    if (!offsets || !overflow || !out_ids || !out_dist || n <= 0 || n > kBatchedMaxRows || nq <= 0 || nq > kRangeMaxQueries ||
        dim <= 0)
        return MORNA_ERR_INVALID_ARGUMENT;
    const RangeWs w = range_ws_layout(nq, morna_tensor_operand_ld(dim));
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    const unsigned char *ws = (const unsigned char *)workspace;
    const size_t smem = (size_t)kCandCap * (sizeof(double) + sizeof(int));
    { int rca = ensure_dynamic_smem((const void *)range_emit_kernel, smem); if (rca != MORNA_OK) return rca; }
    range_emit_kernel<<<(unsigned)nq, kRangeEmitThreads, smem, (cudaStream_t)stream>>>(
        (const int32_t *)(ws + w.match_id), (const double *)(ws + w.match_dist), (const int32_t *)(ws + w.match_cnt), overflow,
        offsets, out_ids, out_dist);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

/* Experiment knobs, process-wide: key 0 = GEMM variant (1 CTA pairs / 0 single CTA),
 * key 1 = shared-memory pipeline stages of the pair variant (4 or 6). */
namespace morna { void set_single_tma(int v); void set_acc_pipelined(int v); void set_acc_split(int v); void set_acc_variant(int v); void set_acc_shift(int v); void set_ids_early_exit(int v); void set_single_prefetch(int v); void set_single_prefetch_rows(int v); void set_single_chain(int v); void set_sparse_tile_mb(int v); }

/* Experiment hook: device buffer of gridDim.x * 4 int64 that the pair GEMM's MMA thread fills with its wait cycles (NULL = off). */
extern "C" int morna_debug_gemm_counters(void *buffer) { g_gemm_debug = (long long *)buffer; return MORNA_OK; }

extern "C" int morna_debug_set_tuning(int32_t key, int32_t value) {
    if (key == 0) g_gemm_pair = value == 2 ? 2 : (value ? 1 : 0);
    else if (key == 3) morna::set_single_tma(value);
    else if (key == 4) morna::set_acc_pipelined(value);
    else if (key == 1) g_gemm_stages = value;
    else if (key == 5) g_rerank_rows = value;
    else if (key == 13) g_rerank_ctas_per_sm = value;
    else if (key == 9) g_block_rows = value >= 256 ? value : 131072;
    else if (key == 10) g_pilot_rows = value >= 256 && value <= kPilotMax ? value : kPilotMax;
    else if (key == 11) g_first_block = value > 0 ? value : 0;
    else if (key == 7) morna::set_acc_split(value);
    else if (key == 8) morna::set_acc_variant(value);
    else if (key == 12) morna::set_acc_shift(value);
    else if (key == 25) morna::set_ids_early_exit(value);
    else if (key == 27) morna::set_single_prefetch(value);
    else if (key == 28) morna::set_single_prefetch_rows(value);
    else if (key == 29) morna::set_single_chain(value);
    else if (key == 35) morna::set_sparse_tile_mb(value);
    else if (key == 36) g_block_growth = value >= 1 && value <= 8 ? value : 1;
    else if (key == 6) g_rerank_phase_mb = value;
    else if (key == 14) g_rerank_kernel = value;
    else if (key == 15) g_rerank_ctas = value;
    else if (key == 16) g_rerank_subs = value;
    else if (key == 17) g_side_job = value;
    else if (key == 18) g_rerank_pipe = value;
    else if (key == 32) g_rerank_evict_first = value >= 0 && value <= 4 ? value : 0;
    else if (key == 33) g_gemm_l2_keep = value ? 1 : 0;
    else if (key == 34) g_rerank_sort_rows = value ? 1 : 0;
    else if (key == 30) g_rerank_fat_sms = value > 0 ? value : 0;
    else if (key == 31) g_gemm_pairs_cap = value > 0 ? value : 0;
    else if (key == 19) g_carveout_hint = value;
    else if (key == 20) g_rerank_oneshot = value;
    else if (key == 22) g_gemm_relaxed_ns = value;
    else if (key == 23) g_gemm_dry = value;
    else if (key == 24) g_tmap_promotion = value;

    else return MORNA_ERR_INVALID_ARGUMENT;
    return MORNA_OK;
}
