// Shared device/host helpers for the morna_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/morna_b200.h"

namespace morna {

extern thread_local int g_last_cuda_error;
void count_launch(int n = 1);
// SM count of the current device and the dynamic-shared-memory opt-in of a kernel, both cached per device ordinal
// behind a mutex (function attributes are per device; several host threads / GPUs may call in)
int sm_count_current();
int ensure_dynamic_smem(const void *kernel, size_t bytes);

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return MORNA_ERR_CUDA;
}

#define MORNA_CUDA_TRY(expr)                                   \
    do {                                                       \
        cudaError_t _e = (expr);                               \
        if (_e != cudaSuccess) return ::morna::cuda_fail(_e);  \
    } while (0)

// after a kernel launch: pick up launch-configuration errors without synchronising
#define MORNA_LAUNCH_CHECK()                                   \
    do {                                                       \
        ::morna::count_launch();                               \
        cudaError_t _e = cudaGetLastError();                   \
        if (_e != cudaSuccess) return ::morna::cuda_fail(_e);  \
    } while (0)

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

__device__ __forceinline__ float4 ldg_stream_f4(const float4 *p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ double warp_sum(double v) {
    // fixed butterfly: every lane ends with the same value, order independent of data
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// The one summation tree used for pp, qq and pq everywhere (row norms, distance
// scan, re-rank): lane l owns float4 chunks l, l+32, ... in increasing order, one
// double accumulator per lane, FMA per element, then the butterfly above.  Equal
// inputs therefore give bit-equal sums, which makes a stored row sit at distance
// exactly 0 from itself (morna.py:101-114 has the same property sequentially).
struct Dot3 { double pp, pq; };

// float -> double without the conversion unit (F2F.F64.F32 issues at a quarter of the DFMA rate and
// was the re-rank's busiest pipe): the float's sign/exponent/mantissa bits dropped into a double
// *without re-biasing the exponent*, i.e. exactly v * 2^-896 -- zeros and denormals included, three
// integer instructions.  The other FMA operand carries the 2^896 (kTwo896), so
//   fma(f32_scaled_f64(v), q * 2^896, acc) == fma((double)v, q, acc)   bit for bit
// whenever q * 2^896 is finite (|q| < 2^128).  Inf/NaN inputs are not supported on this path.
constexpr double kTwo896 = 0x1p896;
constexpr double kScaledQueryMax = 0x1p127;
__device__ __forceinline__ double f32_scaled_f64(float v) {
    const int b = __float_as_int(v);
    return __hiloint2double((b >> 3) & (int)0x8fffffff, b << 29);
}

// angular distance from the three sums; morna.py:109-114 plus a clamp at 0
__device__ __forceinline__ double angular_from_sums(double pp, double qq, double pq) {
    double ppqq = pp * qq;
    double d = 2.0;
    if (ppqq > 0.0) d = 2.0 - 2.0 * pq / sqrt(ppqq);
    if (d < 0.0) d = 0.0;
    return sqrt(d);
}

// order of the reference's result list (morna.py:705-712): smaller distance first,
// equal distances -> larger id first
__device__ __forceinline__ bool before(double da, int ia, double db, int ib) {
    return da < db || (da == db && ia > ib);
}

// bitonic sort of P (power of two) (key,id) pairs in shared memory under `before`
template <bool kWithIds>
__device__ inline void bitonic_sort_smem(double *sd, int *si, int P) {
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

// Per-query exclusion on the FP64 routes (search_exact.cu).  Row i is excluded for query q iff
// query_group[q] >= 0 && row_group[i] == query_group[q]; the mask writes +inf into the distance scratch
// [nq x dist_ld] of every excluded pair, so a selection after it never prefers an excluded row to a real
// distance (<= 2).  The padding pass turns the selected +inf entries into id -1 (the padding of short lists).
int launch_mask_excluded(double *dist, int64_t n, int64_t dist_ld, int64_t nq, const int32_t *row_group,
                         const int32_t *query_group, cudaStream_t s);
int launch_pad_masked(int32_t *ids, const double *dist, int64_t total, cudaStream_t s);

// Parameters of the selection passes between the GEMM launches of the batched path (kth_warp_kernel, search_batched.cu,
// and its group-capped counterpart cap_select_kernel, search_capped.cu)
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

// Group-capped search (search_capped.cu): the passes that take the place of kth_warp_kernel modes 1 (pilot), 2 (refine)
// and 0 (final) when every row of the call carries a cap label (cap_group; < 0: ungrouped) and at most max_per_group rows
// of a label may be returned
int launch_cap_select(int mode, const KthParams &p, const int32_t *cap_group, int32_t max_per_group, int64_t nq,
                      cudaStream_t s);

// The walk of morna_cap_sorted_lists on fixed-stride lists (list j = entries [j * in_ld, (j + 1) * in_ld), at most
// kCapWalkChunk long), written padded to [n_lists x out_ld]: the last step of the capped tensor-core route.
constexpr int kCapWalkChunk = 1024;
int launch_cap_walk_strided(const int32_t *ids, const double *dists, int64_t n_lists, int64_t in_ld, const int32_t *cap_group,
                            int32_t id_base, int64_t n_rows, int32_t max_per_group, int64_t limit, int32_t *out_ids,
                            double *out_dists, int64_t out_ld, cudaStream_t s);

}  // namespace morna
