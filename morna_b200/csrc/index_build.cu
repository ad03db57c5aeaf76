// Index build: feature hashing, first-seen internal ids, order-faithful scatter-add,
// float32 round/store.  Replaces morna.py:369-388 and the add_item cast (:405-407).
#include <math.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace morna {

// ------------------------------------------------------------------ K1 hashing
__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }

// MurmurHash3_x86_32, seed 0 (what mmh3.hash computes at morna.py:369)
__device__ __forceinline__ uint32_t murmur3_32(const uint8_t *__restrict__ key, int len) {
    const uint32_t c1 = 0xcc9e2d51u, c2 = 0x1b873593u;
    uint32_t h = 0;
    const int nblocks = len >> 2;
    for (int i = 0; i < nblocks; ++i) {
        const uint8_t *p = key + 4 * i;          // keys are byte-packed: no alignment assumed
        uint32_t k = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
        k *= c1; k = rotl32(k, 15); k *= c2;
        h ^= k; h = rotl32(h, 13); h = h * 5u + 0xe6546b64u;
    }
    const uint8_t *tail = key + 4 * nblocks;
    uint32_t k = 0;
    const int rem = len & 3;
    if (rem == 3) k ^= (uint32_t)tail[2] << 16;
    if (rem >= 2) k ^= (uint32_t)tail[1] << 8;
    if (rem >= 1) {
        k ^= tail[0];
        k *= c1; k = rotl32(k, 15); k *= c2; h ^= k;
    }
    h ^= (uint32_t)len;
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}

__global__ void __launch_bounds__(256)
hash_junctions_kernel(const uint8_t *__restrict__ keys, const int32_t *__restrict__ key_off, int64_t n_rows,
                      int32_t dim, int32_t *__restrict__ raw, int32_t *__restrict__ bucket,
                      int8_t *__restrict__ sign) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows;
         j += (int64_t)gridDim.x * blockDim.x) {
        int32_t b = key_off[j], e = key_off[j + 1];
        int32_t h = (int32_t)murmur3_32(keys + b, e - b);
        int32_t m = h % dim;                 // C remainder has the dividend's sign ...
        if (m < 0) m += dim;                 // ... Python's floor-mod does not (morna.py:371)
        raw[j] = h; bucket[j] = m; sign[j] = h < 0 ? (int8_t)-1 : (int8_t)1;
    }
}

// ------------------------------------------------------------------ K2 internal ids
__global__ void __launch_bounds__(256)
ids_init_kernel(unsigned long long *first_pos, int32_t *vals, int64_t m, unsigned long long sentinel) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
        first_pos[i] = sentinel;
        vals[i] = (int32_t)i;
    }
}

// one warp per row: earliest pair position of every sample among passing rows
__global__ void __launch_bounds__(256)
first_position_kernel(const int64_t *__restrict__ row_off, const uint8_t *__restrict__ pass, int64_t row_begin, int64_t n_rows,
                      const int32_t *__restrict__ sample, int32_t max_sample_id,
                      unsigned long long *__restrict__ first_pos, const int32_t *__restrict__ seen, int32_t need) {
    if (seen && *seen >= need) return;           // every sample already has its first position among earlier rows
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t j = row_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < n_rows; j += warps_total) {
        if (!pass[j]) continue;
        const int64_t b = row_off[j], e = row_off[j + 1];
        for (int64_t p = b + lane; p < e; p += 32) {
            int32_t s = sample[p];
            // positions only ever decrease: a plain (possibly stale) read filters nearly every atomic
            if ((uint32_t)s <= (uint32_t)max_sample_id && (unsigned long long)p < __ldcg(&first_pos[s]))
                atomicMin(&first_pos[s], (unsigned long long)p);
        }
    }
}

// Same result with a CTA-local table in shared memory (sample ids <= kFirstPosSmemIds, nnz < 2^32):
// a pair only reaches the global atomic when it lowers this CTA's own minimum for the sample.
constexpr int kFirstPosSmemIds = 49152;      // 192 KB of uint32

__global__ void __launch_bounds__(512)
first_position_smem_kernel(const int64_t *__restrict__ row_off, const uint8_t *__restrict__ pass, int64_t row_begin, int64_t n_rows,
                           const int32_t *__restrict__ sample, int32_t max_sample_id,
                           unsigned long long *__restrict__ first_pos, const int32_t *__restrict__ seen, int32_t need) {
    extern __shared__ uint32_t s_first[];            // [max_sample_id + 1]
    if (seen && *seen >= need) return;               // every sample already has its first position among earlier rows
    for (int i = threadIdx.x; i <= max_sample_id; i += blockDim.x) s_first[i] = 0xffffffffu;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
    int64_t j = row_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    // the next row's bounds are fetched while the current row streams: one exposed latency per row, not two
    int64_t b = 0, e = 0;
    bool ok = false;
    if (j < n_rows) { ok = pass[j] != 0; b = row_off[j]; e = row_off[j + 1]; }
    while (j < n_rows) {
        const int64_t jn = j + warps_total;
        int64_t bn = 0, en = 0;
        bool okn = false;
        if (jn < n_rows) { okn = pass[jn] != 0; bn = row_off[jn]; en = row_off[jn + 1]; }
        for (int64_t p0 = b; ok && p0 < e; p0 += 512) {     // sixteen independent loads in flight per lane
            int32_t sv[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int64_t p = p0 + u * 32 + lane;
                sv[u] = p < e ? __ldg(sample + p) : -1;
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int64_t p = p0 + u * 32 + lane;
                // a warp meets its rows in increasing position order, so after a sample's first sighting in
                // this CTA a plain read almost always ends the matter; the atomic is the rare case
                if ((uint32_t)sv[u] <= (uint32_t)max_sample_id && (uint32_t)p < s_first[sv[u]]) {
                    const uint32_t old = atomicMin(&s_first[sv[u]], (uint32_t)p);
                    if ((uint32_t)p < old) atomicMin(&first_pos[sv[u]], (unsigned long long)p);
                }
            }
        }
        j = jn; b = bn; e = en; ok = okn;
    }
}

// seen[0] += sample ids that have a first position.  The first-seen order depends only on first occurrences: once as many
// ids have been met as there are distinct samples in passing rows (the caller's count, or the whole id space), later rows
// cannot change anything.
__global__ void __launch_bounds__(256)
ids_seen_count_kernel(const unsigned long long *__restrict__ first_pos, int64_t m, unsigned long long sentinel,
                      int32_t *__restrict__ seen) {
    int mine = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
        mine += first_pos[i] < sentinel;
    mine = __reduce_add_sync(0xffffffffu, mine);
    if (mine && (threadIdx.x & 31) == 0) atomicAdd(seen, mine);
}

__global__ void __launch_bounds__(256)
ids_assign_kernel(const unsigned long long *__restrict__ sorted_pos, const int32_t *__restrict__ sorted_sample,
                  int64_t m, unsigned long long sentinel, int32_t *__restrict__ id_of_sample,
                  int32_t *__restrict__ n_kept) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
        bool seen = sorted_pos[i] < sentinel;
        id_of_sample[sorted_sample[i]] = seen ? (int32_t)i : -1;
        bool next_seen = (i + 1 < m) && sorted_pos[i + 1] < sentinel;
        if (seen && !next_seen) *n_kept = (int32_t)(i + 1);
        if (i == 0 && !seen) *n_kept = 0;
    }
}

// ------------------------------------------------------------------ K3 scatter-add
__global__ void __launch_bounds__(256)
bucket_keys_kernel(const uint8_t *__restrict__ pass, const int32_t *__restrict__ bucket, int64_t n_rows,
                   int32_t dim, int32_t *__restrict__ keys, int32_t *__restrict__ vals) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += (int64_t)gridDim.x * blockDim.x) {
        keys[j] = pass[j] ? bucket[j] : dim;   // rows under the threshold sort past the last bucket
        vals[j] = (int32_t)j;
    }
}

// begin[b] = first position in the bucket-sorted row list whose key >= b, b in [0, dim+1]
__global__ void __launch_bounds__(256)
bucket_begin_kernel(const int32_t *__restrict__ sorted_keys, int64_t n_rows, int32_t dim,
                    int32_t *__restrict__ begin) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n_rows; i += (int64_t)gridDim.x * blockDim.x) {
        int32_t prev = i > 0 ? sorted_keys[i - 1] : -1;
        int32_t cur = i < n_rows ? sorted_keys[i] : dim + 1;
        for (int32_t b = prev + 1; b <= cur; ++b) begin[b] = (int32_t)i;
    }
}

constexpr int kAccThreads = 512;
constexpr int kAccTile = 24576;   // doubles of one bucket column held in shared memory (192 KB)

// CTA (b, t) owns bucket b for internal ids [lo, hi).  Rows of the bucket are applied
// in file order with a barrier between rows, so each cell sees its addends in the
// reference's order (morna.py:376-388) and the double sums are bit-identical.
__global__ void __launch_bounds__(kAccThreads)
index_accumulate_kernel(const int32_t *__restrict__ use_flag, const int64_t *__restrict__ row_off, const int8_t *__restrict__ sign,
                        const double *__restrict__ idf, const int32_t *__restrict__ sample,
                        const int32_t *__restrict__ cov, const int32_t *__restrict__ id_of_sample,
                        const int32_t *__restrict__ rows_by_bucket, const int32_t *__restrict__ bucket_begin,
                        int32_t id_lo, int32_t id_hi, int32_t tile, double *__restrict__ acc, int64_t acc_ld) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *col = reinterpret_cast<double *>(smem_raw);
    const int b = blockIdx.x;
    const int32_t lo = id_lo + (int32_t)blockIdx.y * tile;
    const int32_t hi = min(id_hi, lo + tile);
    const int32_t width = hi - lo;
    const int32_t r_begin = bucket_begin[b], r_end = bucket_begin[b + 1];
    double *out = acc + (int64_t)b * acc_ld + (lo - id_lo);
    if (use_flag && !*use_flag) return;      // the sample-range variant answers
    if (r_begin == r_end) {                  // an empty bucket: its column is zero (the caller does not pre-fill acc)
        for (int i = threadIdx.x; i < width; i += kAccThreads) out[i] = 0.0;
        return;
    }
    for (int i = threadIdx.x; i < width; i += kAccThreads) col[i] = 0.0;
    __syncthreads();
    for (int32_t r = r_begin; r < r_end; ++r) {
        const int32_t j = rows_by_bucket[r];
        const double w = idf[j];
        const double mult = (double)sign[j];
        const int64_t pb = row_off[j], pe = row_off[j + 1];
        for (int64_t p = pb + threadIdx.x; p < pe; p += kAccThreads) {
            int32_t id = id_of_sample[sample[p]];
            if (id >= lo && id < hi) {
                double tfidf = (double)cov[p] * w;
                atomicAdd(&col[id - lo], mult * tfidf);
            }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < width; i += kAccThreads) out[i] = col[i];
}

// ---- pipelined variant -------------------------------------------------------------------------
// Same order-faithful accumulation, but the bucket's pairs are treated as one virtual stream
// (rows of the bucket concatenated in file order) cut into batches of kAcc2Threads*kAcc2U pairs.
// Three batches are in flight per CTA: sample/coverage loads for batch i+2, the id_of_sample gather
// for batch i+1, and the ordered shared-memory adds of batch i (a barrier between rows), so the two
// dependent global-memory latencies are hidden instead of being paid once per row.
constexpr int kAcc2Threads = 512, kAcc2U = 4, kAcc2Batch = kAcc2Threads * kAcc2U;
constexpr int kAcc2Window = 512;          // rows of the bucket whose metadata sits in shared memory
constexpr int kAcc2Tile = 22528;          // doubles of the bucket column per CTA (176 KB)
constexpr size_t kAcc2MetaBytes = (size_t)kAcc2Window * (8 + 8) + (size_t)(kAcc2Window + 1) * 4 + 16;

__global__ void __launch_bounds__(256)
sorted_row_len_kernel(const int32_t *__restrict__ use_flag, const int64_t *__restrict__ row_off,
                      const int32_t *__restrict__ rows_by_bucket, int64_t n_rows, int64_t *__restrict__ len) {
    if (use_flag && !*use_flag) return;      // the sample-range variant answers
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t j = rows_by_bucket[i];
        len[i] = row_off[j + 1] - row_off[j];
    }
}

// Streaming form of the "every row ascends" question, position-parallel instead of warp-per-row: a bit per
// pair position marks the row starts, then every pair is compared with its predecessor unless it starts a row.
// (All rows are checked, also those under the threshold: a stray descending row there only costs the fast path.)
__global__ void __launch_bounds__(256)
row_start_bits_kernel(const int64_t *__restrict__ row_off, int64_t n_rows, int64_t nnz, uint32_t *__restrict__ bits) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = row_off[j];
        if (p < nnz && row_off[j + 1] > p) atomicOr(bits + (p >> 5), 1u << (p & 31));
    }
}

__global__ void __launch_bounds__(256)
pairs_ascending_kernel(const int32_t *__restrict__ sample, int64_t nnz, const uint32_t *__restrict__ bits,
                       int32_t *__restrict__ not_ascending) {
    // thread = 4 consecutive positions (one 16-byte load) plus the element before them; four such groups in flight
    const int64_t groups = nnz >> 2;                           // whole groups; the tail is checked by thread 0
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    bool bad = false;
    for (int64_t g0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g0 < groups; g0 += 4 * stride) {
        int4 v[4];
        int32_t prev[4];
        uint32_t word[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t g = g0 + u * stride;
            const bool have = g < groups;
            v[u] = have ? __ldg(reinterpret_cast<const int4 *>(sample) + g) : make_int4(0, 1, 2, 3);
            prev[u] = have && g > 0 ? __ldg(sample + 4 * g - 1) : -1;
            word[u] = have ? __ldg(bits + (g >> 3)) : 0xffffffffu;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t g = g0 + u * stride;
            const uint32_t start = (word[u] >> ((4 * g) & 31)) & 0xfu;     // row-start flags of the four positions
            bad |= !(start & 1u) && v[u].x <= prev[u];
            bad |= !(start & 2u) && v[u].y <= v[u].x;
            bad |= !(start & 4u) && v[u].z <= v[u].y;
            bad |= !(start & 8u) && v[u].w <= v[u].z;
            bad |= (v[u].x | v[u].y | v[u].z | v[u].w) < 0;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t p = 4 * groups; p < nnz; ++p) {
            const bool start = (bits[p >> 5] >> (p & 31)) & 1u;
            bad |= sample[p] < 0 || (!start && p > 0 && sample[p] <= sample[p - 1]);
        }
    if (bad) *not_ascending = 1;
}

// rows whose sample ids are strictly increasing or strictly decreasing cannot list a sample twice;
// flags[0] = some passing row is neither, flags[1] = some passing row is not strictly increasing
__global__ void __launch_bounds__(256)
rows_monotonic_kernel(const int32_t *__restrict__ use_flag, const int64_t *__restrict__ row_off,
                      const uint8_t *__restrict__ pass, int64_t n_rows, const int32_t *__restrict__ sample,
                      int32_t *__restrict__ flags) {
    if (use_flag && !*use_flag) return;      // every row ascends: nothing to classify
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t j = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < n_rows; j += warps_total) {
        if (!pass[j]) continue;
        const int64_t b = row_off[j], e = row_off[j + 1];
        bool up = true, down = true;
        int32_t carry = 0;
        for (int64_t p0 = b; p0 < e; p0 += 128) {          // four independent chunks in flight
            int32_t c[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t p = p0 + 32 * u + lane;
                c[u] = p < e ? __ldg(sample + p) : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t p = p0 + 32 * u + lane;
                int32_t a = __shfl_up_sync(kFull, c[u], 1);
                if (lane == 0) a = carry;
                carry = __shfl_sync(kFull, c[u], 31);
                const bool have = p < e && p > b;          // the row's first pair has no predecessor
                up &= !have || c[u] > a; down &= !have || c[u] < a;
            }
        }
        if (lane == 0 && e > b) up &= sample[b] >= 0;       // (negative ids would index before the slices)
        up = __all_sync(kFull, up); down = __all_sync(kFull, down);
        if (lane == 0 && !up && !down) flags[0] = 1;
        if (lane == 0 && !up) flags[1] = 1;
    }
}

template <bool kAtomic>
__global__ void __launch_bounds__(kAcc2Threads)
index_accumulate2_kernel(const int32_t *__restrict__ use_flag, const int32_t *__restrict__ run_flag,
                         const int64_t *__restrict__ row_off, const int8_t *__restrict__ sign,
                         const double *__restrict__ idf, const int32_t *__restrict__ sample,
                         const int32_t *__restrict__ cov, const int32_t *__restrict__ id_of_sample,
                         const int32_t *__restrict__ rows_by_bucket, const int32_t *__restrict__ bucket_begin,
                         const int64_t *__restrict__ voff, int32_t id_lo, int32_t id_hi, int32_t tile,
                         double *__restrict__ acc, int64_t acc_ld) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *col = reinterpret_cast<double *>(smem_raw);                       // [tile]
    double *s_w = col + tile;                                                 // [window] sign * idf
    int64_t *s_delta = reinterpret_cast<int64_t *>(s_w + kAcc2Window);        // [window] real offset - virtual offset
    int32_t *s_voff = reinterpret_cast<int32_t *>(s_delta + kAcc2Window);     // [window + 1] virtual offsets - V0
    __shared__ int s_rows[8];                                                 // first/last row of the 4 batches in flight
    const int tid = threadIdx.x;
    const int b = blockIdx.x;
    const int32_t lo = id_lo + (int32_t)blockIdx.y * tile;
    const int32_t hi = min(id_hi, lo + tile);
    const int32_t width = hi - lo;
    const int32_t r_begin = bucket_begin[b], r_end = bucket_begin[b + 1];
    double *out = acc + (int64_t)b * acc_ld + (lo - id_lo);
    // the atomic and the plain variant are both launched; the monotonicity flag picks the one that runs
    if (use_flag && !*use_flag) return;
    if ((*run_flag != 0) != kAtomic) return;
    if (r_begin == r_end) {                  // an empty bucket: its column is zero (the caller does not pre-fill acc)
        for (int i = tid; i < width; i += kAcc2Threads) out[i] = 0.0;
        return;
    }
    for (int i = tid; i < width; i += kAcc2Threads) col[i] = 0.0;

    for (int32_t w0 = r_begin; w0 < r_end; w0 += kAcc2Window) {
        const int nrows = min(kAcc2Window, r_end - w0);
        const int64_t V0 = voff[w0], V1 = voff[w0 + nrows];
        __syncthreads();                     // previous window fully applied; metadata may be replaced
        for (int i = tid; i <= nrows; i += kAcc2Threads) s_voff[i] = (int32_t)(voff[w0 + i] - V0);
        for (int i = tid; i < nrows; i += kAcc2Threads) {
            const int32_t j = rows_by_bucket[w0 + i];
            s_w[i] = (double)sign[j] * idf[j];            // +-idf: (+-idf)*cov == +-(idf*cov) bit for bit
            s_delta[i] = row_off[j] - voff[w0 + i];
        }
        __syncthreads();
        const int64_t total = V1 - V0;
        const int n_batches = (int)((total + kAcc2Batch - 1) / kAcc2Batch);

        // register stages: L = loaded (sample, cov, row), G = gathered (id, value, row)
        int32_t l_s[kAcc2U], l_c[kAcc2U], l_r[kAcc2U];
        int32_t g_id[kAcc2U], g_r[kAcc2U];
        double g_v[kAcc2U];
        auto load_batch = [&](int bi) {
            // one binary search for the thread's first pair, then a forward walk: its next pairs are
            // kAcc2Threads further along the stream, usually in the same or the next row
            int a = 0;
            const int64_t v_first = (int64_t)bi * kAcc2Batch + tid;
            if (bi < n_batches && v_first < total) {
                int z = nrows;
                while (z - a > 1) { const int m = (a + z) >> 1; if (s_voff[m] <= (int32_t)v_first) a = m; else z = m; }
            }
            const int64_t v_last = min(total, (int64_t)(bi + 1) * kAcc2Batch) - 1;      // last pair of the batch
#pragma unroll
            for (int u = 0; u < kAcc2U; ++u) {
                const int64_t v = v_first + u * kAcc2Threads;                            // relative to V0
                l_r[u] = -1;
                if (bi < n_batches && v < total) {
                    while (a + 1 < nrows && s_voff[a + 1] <= (int32_t)v) ++a;
                    const int64_t p = V0 + v + s_delta[a];
                    l_s[u] = __ldg(sample + p); l_c[u] = __ldg(cov + p); l_r[u] = a;
                    if (v == (int64_t)bi * kAcc2Batch) s_rows[(bi & 3) * 2] = a;         // first row of the batch
                    if (v == v_last) s_rows[(bi & 3) * 2 + 1] = a;                       // last row of the batch
                }
            }
        };
        auto gather_batch = [&]() {
#pragma unroll
            for (int u = 0; u < kAcc2U; ++u) {
                g_r[u] = l_r[u];
                if (l_r[u] >= 0) {
                    g_id[u] = __ldg(id_of_sample + l_s[u]);
                    g_v[u] = (double)l_c[u] * s_w[l_r[u]];
                }
            }
        };
        load_batch(0);
        gather_batch();                      // batch 0 gathered
        load_batch(1);
        __syncthreads();                     // s_rows of batches 0 and 1 visible
        for (int bi = 0; bi < n_batches; ++bi) {
            // keep a copy of the batch to apply, then advance the two younger stages
            int32_t a_id[kAcc2U], a_r[kAcc2U];
            double a_v[kAcc2U];
#pragma unroll
            for (int u = 0; u < kAcc2U; ++u) { a_id[u] = g_id[u]; a_r[u] = g_r[u]; a_v[u] = g_v[u]; }
            gather_batch();                  // batch bi+1: its id gather flies during the adds below
            load_batch(bi + 2);
            // rows covered by batch bi (recorded when it was loaded, at least one barrier ago), in file order
            const int ra = s_rows[(bi & 3) * 2], rb = s_rows[(bi & 3) * 2 + 1];
            for (int r = ra; r <= rb; ++r) {
#pragma unroll
                for (int u = 0; u < kAcc2U; ++u)
                    if (a_r[u] == r && a_id[u] >= lo && a_id[u] < hi) {
                        if (kAtomic) atomicAdd(&col[a_id[u] - lo], a_v[u]);     // a row may repeat a sample
                        else col[a_id[u] - lo] += a_v[u];                        // distinct ids within the row
                    }
                __syncthreads();
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < width; i += kAcc2Threads) out[i] = col[i];
}

// ---- sample-range variant ----------------------------------------------------------------------
// intropolis lists each row's samples in strictly ascending order (rows that do not are detected and
// take the variants above).  The sample-id space is cut into P ranges of 2^shift ids, and ONE WARP owns
// (bucket, range): it walks the bucket's rows in file order and applies, for each row, the contiguous
// segment of the row that falls in its range -- distinct samples, so lanes never collide within a row,
// and a __syncwarp() between rows orders the rows.  Every cell therefore still sees its addends in the
// reference's order (morna.py:376-388: bit-identical doubles), but there is no block barrier, no
// id_of_sample gather in the loop, and several small CTAs share an SM.
//   pre-pass  row_segments_kernel: one warp per bucket-sorted row -> the row's P+1 segment offsets,
//             its start position and +-idf, stored in sorted order (coalesced for the consumer)
//   main      index_accumulate3_kernel: warp = (bucket, range), slice of 2^shift doubles in shared memory
constexpr int kAcc3Warps = 4, kAcc3Threads = kAcc3Warps * 32;
constexpr int kAcc3Group = 8;        // rows whose first 32 pairs are loaded together
constexpr int kAcc3Unroll = 4;       // 32-pair chunks in flight inside a long segment

struct RowMeta { int64_t pos; double w; };      // first pair of the row, sign * idf

// Pre-pass, one thread per (bucket-sorted row, range boundary): the first position of the row whose
// sample id reaches the boundary, by binary search -- valid if the row is ascending, which the main
// kernel verifies on every pair it loads.  Also the row's start position and +-idf, in sorted order.
__global__ void __launch_bounds__(256)
row_segments_kernel(const int64_t *__restrict__ row_off, const int8_t *__restrict__ sign,
                    const double *__restrict__ idf, const int32_t *__restrict__ sample,
                    const int32_t *__restrict__ rows_by_bucket, const int32_t *__restrict__ bucket_begin, int32_t dim,
                    int32_t shift, int32_t n_ranges, int32_t *__restrict__ seg, RowMeta *__restrict__ meta) {
    const int32_t n_pass = bucket_begin[dim];                  // rows under the threshold sort past the last bucket
    const int64_t total = (int64_t)n_pass * (n_ranges + 1);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        // (32-bit division when the index fits: a 64-bit divide is a hundred instructions on this path)
        const int64_t r = total <= 0xffffffffll ? (int64_t)((uint32_t)i / (uint32_t)(n_ranges + 1)) : i / (n_ranges + 1);
        const int32_t q = (int32_t)(i - r * (n_ranges + 1));
        const int32_t j = rows_by_bucket[r];
        const int64_t b = row_off[j];
        const int32_t n = (int32_t)(row_off[j + 1] - b);
        if (q == 0) { meta[r].pos = b; meta[r].w = (double)sign[j] * idf[j]; }
        int32_t lo = 0, hi = n;                                // first p in [0, n] with sample[b + p] >= q << shift
        if (q == n_ranges) lo = n;
        else if (q > 0 && n > 0) {
            const int32_t bound = q << shift;
            // The ids of a row are spread over [first, last] roughly evenly: start next to the interpolated position and
            // gallop outwards (a few probes in one or two cache lines instead of log2(n) scattered ones), then bisect the
            // bracket.  Any ascending row gives the same answer as a plain binary search.
            const int32_t first = __ldg(sample + b), last = __ldg(sample + b + n - 1);
            if (bound <= first) hi = 0;
            else if (bound > last) lo = n;
            else {
                int32_t g = (int32_t)((float)(bound - first) * (float)(n - 1) / (float)max(last - first, 1));   // (a guess: float is enough)
                g = min(max(g, 0), n - 1);
                if (__ldg(sample + b + g) < bound) {           // answer is to the right of g
                    lo = g + 1;
                    int32_t stepw = 4;
                    while (lo + stepw < n && __ldg(sample + b + lo + stepw - 1) < bound) { lo += stepw; stepw <<= 1; }
                    hi = min(n, lo + stepw);
                } else {                                       // sample[g] >= bound: answer is at or left of g
                    hi = g;
                    int32_t stepw = 4;
                    while (hi - stepw > 0 && __ldg(sample + b + hi - stepw) >= bound) { hi -= stepw; stepw <<= 1; }
                    lo = max(0, hi - stepw);
                }
            }
            while (lo < hi) {
                const int32_t mid = (lo + hi) >> 1;
                if (__ldg(sample + b + mid) < bound) lo = mid + 1; else hi = mid;
            }
        }
        seg[i] = lo;
    }
}

// A chunk: up to 32 consecutive pairs of one row that fall in one sample-id range.
struct __align__(16) ChunkDesc { int32_t pos; int32_t cnt_end; double w; };   // first pair, pairs | last-of-row << 8, +-idf

// chunks per (range, sorted row), range-major so that one exclusive scan gives every (bucket, range) list
// its place:  cnt[p * n_pass + r] = ceil(n / 32), n = pairs of row r in range p
__global__ void __launch_bounds__(256)
chunk_count_kernel(const int32_t *__restrict__ not_ascending, const int32_t *__restrict__ seg,
                   const int32_t *__restrict__ bucket_begin, int32_t dim, int32_t n_ranges, int64_t n_rows_cap,
                   int32_t *__restrict__ cnt) {
    const int64_t n_pass = bucket_begin[dim];
    const int64_t total = *not_ascending ? 0 : n_pass * n_ranges;    // unusable offsets: empty lists
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n_rows_cap * n_ranges; i += (int64_t)gridDim.x * blockDim.x) {
        int32_t c = 0;
        if (i < total) {
            const int64_t p = total <= 0xffffffffll ? (int64_t)((uint32_t)i / (uint32_t)n_pass) : i / n_pass, r = i - p * n_pass;
            const int32_t *sg = seg + r * (n_ranges + 1) + p;
            c = (max(sg[1] - sg[0], 0) + 31) >> 5;
        }
        cnt[i] = c;                                            // zeros past the passing rows: the scan covers the whole array
    }
}

__global__ void __launch_bounds__(256)
chunk_fill_kernel(const int32_t *__restrict__ not_ascending, const int32_t *__restrict__ seg, const RowMeta *__restrict__ meta,
                  const int32_t *__restrict__ bucket_begin, int32_t dim, int32_t n_ranges, const int32_t *__restrict__ chunk_off,
                  ChunkDesc *__restrict__ desc) {
    if (*not_ascending) return;
    const int64_t n_pass = bucket_begin[dim];
    const int64_t total = n_pass * n_ranges;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = total <= 0xffffffffll ? (int64_t)((uint32_t)i / (uint32_t)n_pass) : i / n_pass, r = i - p * n_pass;
        const int32_t *sg = seg + r * (n_ranges + 1) + p;
        const int32_t lo = sg[0], n = max(sg[1] - lo, 0);
        if (n == 0) continue;
        const RowMeta mt = meta[r];
        const int32_t pos0 = (int32_t)mt.pos + lo;             // nnz < 2^31 (checked by the host entry)
        ChunkDesc *out = desc + chunk_off[i];
        for (int32_t c = 0; c < n; c += 32) {
            ChunkDesc d;
            d.pos = pos0 + c; d.cnt_end = min(32, n - c) | ((c + 32 >= n) << 8); d.w = mt.w;
            *out++ = d;
        }
    }
}

// One warp = (bucket, sample-id range).  Its work arrives as a ready-made list of chunks in file order
// (chunk_fill_kernel): the warp streams the list -- descriptors 32 at a time through a two-slot ring in
// shared memory, the pairs of the next eight chunks in flight while the current eight are added -- and a
// __syncwarp() follows the last chunk of each row, so rows are applied in file order; the chunks of one
// row hold distinct samples.  Every cell sees its addends in the reference's order (morna.py:376-388).
// Runs only if rows_monotonic_kernel found every passing row strictly ascending.
__global__ void __launch_bounds__(kAcc3Threads)
index_accumulate3_kernel(const int32_t *__restrict__ not_ascending, const int32_t *__restrict__ sample,
                         const int32_t *__restrict__ cov, const int32_t *__restrict__ id_of_sample,
                         const int32_t *__restrict__ bucket_begin, int32_t dim, const int32_t *__restrict__ chunk_off,
                         const ChunkDesc *__restrict__ desc, int32_t shift, int32_t n_ranges, int32_t max_sample_id,
                         int32_t id_lo, int32_t id_hi, double *__restrict__ acc, int64_t acc_ld) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (*not_ascending) return;                                // the order-by-barrier variants run instead
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x;
    const int range = blockIdx.y * kAcc3Warps + warp;
    if (range >= n_ranges) return;                             // no block-wide barrier below
    const int32_t width = 1 << shift, range_lo = range << shift;
    double *slice = reinterpret_cast<double *>(smem_raw) + (size_t)warp * width;
    ChunkDesc *ring = reinterpret_cast<ChunkDesc *>(smem_raw + (size_t)kAcc3Warps * width * sizeof(double)) + 64 * warp;
    const int64_t n_pass = bucket_begin[dim];
    const int32_t d_begin = chunk_off[(int64_t)range * n_pass + bucket_begin[b]];
    const int32_t d_end = chunk_off[(int64_t)range * n_pass + bucket_begin[b + 1]];
    const int n_chunks = d_end - d_begin;
    if (bucket_begin[b] == bucket_begin[b + 1]) {              // an empty bucket: its column is zero (acc is not pre-filled)
        double *zero = acc + (int64_t)b * acc_ld;
        for (int i = range * 32 + lane; i < id_hi - id_lo; i += n_ranges * 32) zero[i] = 0.0;
        return;
    }
    for (int i = lane; i < width; i += 32) slice[i] = 0.0;
    const int n_groups = (n_chunks + kAcc3Group - 1) / kAcc3Group;
    const ChunkDesc *list = desc + d_begin;

    // descriptors: this lane's entry of a batch of 32 -> registers, published to the ring when the batch is reached
    int4 pending = make_int4(0, 0, 0, 0);
    auto fetch_batch = [&](int batch) {
        const int i = 32 * batch + lane;
        pending = i < n_chunks ? __ldg(reinterpret_cast<const int4 *>(list + i)) : make_int4(0, 0, 0, 0);
    };
    auto publish_batch = [&](int batch) {
        __syncwarp();                                          // nobody still reads the slot being replaced
        reinterpret_cast<int4 *>(ring + 32 * (batch & 1))[lane] = pending;
        __syncwarp();
    };
    auto issue = [&](int g, int32_t (&ps)[kAcc3Group], int32_t (&pc)[kAcc3Group]) {
        if ((g & 3) == 0) { publish_batch(g >> 2); fetch_batch((g >> 2) + 1); }
        const ChunkDesc *slot = ring + 32 * ((g >> 2) & 1) + (g & 3) * kAcc3Group;
#pragma unroll
        for (int u = 0; u < kAcc3Group; ++u) {
            const int2 pc2 = *reinterpret_cast<const int2 *>(slot + u);        // pos, cnt_end (broadcast read)
            const bool have = lane < (pc2.y & 0xff);
            ps[u] = have ? __ldg(sample + pc2.x + lane) : -1;
            pc[u] = have ? __ldg(cov + pc2.x + lane) : 0;
        }
    };
    auto apply = [&](int g, const int32_t (&ps)[kAcc3Group], const int32_t (&pc)[kAcc3Group]) {
        const ChunkDesc *slot = ring + 32 * ((g >> 2) & 1) + (g & 3) * kAcc3Group;
#pragma unroll
        for (int u = 0; u < kAcc3Group; ++u) {
            const ChunkDesc d = slot[u];
            if (ps[u] >= 0) {
                double *cell = slice + (ps[u] - range_lo);
                *cell = __dadd_rn(*cell, __dmul_rn((double)pc[u], d.w));        // product rounded, then added: as the reference
            }
            if (d.cnt_end >> 8) __syncwarp();                  // the row is complete: rows are applied in file order
        }
    };

    fetch_batch(0);
    int32_t sa[kAcc3Group], ca[kAcc3Group], sb[kAcc3Group], cb[kAcc3Group];
    if (n_groups > 0) issue(0, sa, ca);
    for (int g = 0; g < n_groups; g += 2) {
        if (g + 1 < n_groups) issue(g + 1, sb, cb);            // next group's loads fly during this group's adds
        apply(g, sa, ca);
        if (g + 1 >= n_groups) break;
        if (g + 2 < n_groups) issue(g + 2, sa, ca);
        apply(g + 1, sb, cb);
    }
    __syncwarp();
    // the slice is in sample-id order; the accumulator is indexed by internal id
    double *out = acc + (int64_t)b * acc_ld;
    for (int i = lane; i < width; i += 32) {
        const int32_t s = range_lo + i;
        if (s > max_sample_id) break;
        const int32_t id = id_of_sample[s];
        if (id >= id_lo && id < id_hi) out[id - id_lo] = slice[i];
    }
}

// ------------------------------------------------------------------ round + transpose
__global__ void __launch_bounds__(256)
round_store_kernel(const double *__restrict__ acc, int64_t acc_ld, int32_t n_ids, int32_t dim,
                   float *__restrict__ vectors, int64_t ld) {
    __shared__ double tile[32][33];
    const int id0 = blockIdx.x * 32, b0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {        // r: bucket within tile, x: id within tile
        int b = b0 + r, id = id0 + threadIdx.x;
        tile[r][threadIdx.x] = (b < dim && id < n_ids) ? acc[(int64_t)b * acc_ld + id] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {        // r: id within tile, x: bucket within tile
        int id = id0 + r, b = b0 + threadIdx.x;
        if (id < n_ids && b < ld) vectors[(int64_t)id * ld + b] = (float)tile[threadIdx.x][r];
    }
}

static int bits_for(uint64_t v) {
    int b = 1;
    while (b < 64 && (v >> b)) ++b;
    return b;
}

struct IdsWs { size_t first_pos, sorted_pos, vals_in, vals_out, cub, cub_bytes, flags, total; };
static IdsWs ids_ws_layout(int64_t m) {
    IdsWs w{};
    size_t off = 0;
    w.first_pos = off; off += align_up((size_t)m * 8, 256);
    w.sorted_pos = off; off += align_up((size_t)m * 8, 256);
    w.vals_in = off; off += align_up((size_t)m * 4, 256);
    w.vals_out = off; off += align_up((size_t)m * 4, 256);
    size_t cub_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const unsigned long long *)nullptr,
                                    (unsigned long long *)nullptr, (const int32_t *)nullptr,
                                    (int32_t *)nullptr, (int)m, 0, 64);
    w.cub = off; w.cub_bytes = cub_bytes; off += align_up(cub_bytes, 256);
    w.flags = off; off += 256;
    w.total = off + 256;
    return w;
}

constexpr int kAcc3MaxRanges = 32;
struct AccWs { size_t keys_in, keys_out, vals_in, vals_out, begin, cub, cub_bytes, len, voff, scan, scan_bytes, flag, seg, meta,
               ccnt, coff, cscan, cscan_bytes, desc, bits, total; };
static AccWs acc_ws_layout(int64_t n_rows, int64_t nnz, int32_t dim) {
    AccWs w{};
    size_t off = 0;
    w.keys_in = off; off += align_up((size_t)n_rows * 4, 256);
    w.keys_out = off; off += align_up((size_t)n_rows * 4, 256);
    w.vals_in = off; off += align_up((size_t)n_rows * 4, 256);
    w.vals_out = off; off += align_up((size_t)n_rows * 4, 256);
    w.begin = off; off += align_up((size_t)(dim + 2) * 4, 256);
    size_t cub_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const int32_t *)nullptr, (int32_t *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, (int)n_rows, 0, 32);
    w.cub = off; w.cub_bytes = cub_bytes; off += align_up(cub_bytes, 256);
    w.len = off; off += align_up((size_t)(n_rows + 1) * 8, 256);
    w.voff = off; off += align_up((size_t)(n_rows + 1) * 8, 256);
    size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int64_t *)nullptr, (int64_t *)nullptr, (int)(n_rows + 1));
    w.scan = off; w.scan_bytes = scan_bytes; off += align_up(scan_bytes, 256);
    w.flag = off; off += 256;
    w.seg = off; off += align_up((size_t)n_rows * (kAcc3MaxRanges + 1) * 4, 256);
    w.meta = off; off += align_up((size_t)n_rows * sizeof(RowMeta), 256);
    // chunk lists of the warp-per-range variant: counts and offsets per (range, row), descriptors
    const size_t cells = (size_t)n_rows * kAcc3MaxRanges + 1;
    w.ccnt = off; off += align_up(cells * 4, 256);
    w.coff = off; off += align_up(cells * 4, 256);
    size_t cscan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, cscan_bytes, (const int32_t *)nullptr, (int32_t *)nullptr, (int)cells);
    w.cscan = off; w.cscan_bytes = cscan_bytes; off += align_up(cscan_bytes, 256);
    w.desc = off; off += align_up(((size_t)(nnz > 0 ? nnz : 0) / 32 + cells) * sizeof(ChunkDesc), 256);
    w.bits = off; off += align_up(((size_t)(nnz > 0 ? nnz : 0) / 32 + 2) * 4, 256);
    w.total = off + 256;
    return w;
}

static int g_acc_pipelined = 1;      // morna_debug_set_tuning key 4
static int g_acc_split = 1;          // morna_debug_set_tuning key 7: id tiles per bucket column (more CTAs per SM)
static int g_acc_shift = 10;         // morna_debug_set_tuning key 12: log2 of the sample-id range width (>= 10)
static int g_acc_variant = 3;        // morna_debug_set_tuning key 8: 3 = sample-range warps first, else barrier-per-row only
static int g_ids_early_exit = 1;     // morna_debug_set_tuning key 25: the id pass stops once every sample id has been met
void set_ids_early_exit(int v) { g_ids_early_exit = v ? 1 : 0; }
void set_acc_pipelined(int v) { g_acc_pipelined = v ? 1 : 0; }
void set_acc_split(int v) { g_acc_split = v > 0 ? v : 1; }
void set_acc_variant(int v) { g_acc_variant = v; }
void set_acc_shift(int v) { g_acc_shift = v >= 10 && v <= 12 ? v : 10; }

static unsigned grid_for(int64_t work, int threads) {
    int64_t g = (work + threads - 1) / threads;
    if (g < 1) g = 1;
    if (g > 148 * 32) g = 148 * 32;
    return (unsigned)g;
}

}  // namespace morna

using namespace morna;

extern "C" int morna_hash_junctions(const uint8_t *keys, const int32_t *key_off, int64_t n_rows, int32_t dim,
                                    int32_t *raw, int32_t *bucket, int8_t *sign, void *stream) {
    if (n_rows < 0 || dim <= 0 || !key_off || !raw || !bucket || !sign) return MORNA_ERR_INVALID_ARGUMENT;
    if (n_rows == 0) return MORNA_OK;
    if (!keys) return MORNA_ERR_INVALID_ARGUMENT;
    hash_junctions_kernel<<<grid_for(n_rows, 256), 256, 0, (cudaStream_t)stream>>>(keys, key_off, n_rows, dim,
                                                                                  raw, bucket, sign);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" int morna_idf_host(const int64_t *running_freq, const uint8_t *pass, int64_t n_rows,
                              int64_t sample_count, double *idf) {
    if (n_rows < 0 || (n_rows > 0 && (!running_freq || !pass || !idf))) return MORNA_ERR_INVALID_ARGUMENT;
    for (int64_t j = 0; j < n_rows; ++j) {
        if (pass[j] && running_freq[j] > 0)
            idf[j] = log((double)sample_count / (double)running_freq[j]);   // morna.py:372-374
        else
            idf[j] = 0.0;
    }
    return MORNA_OK;
}

extern "C" size_t morna_assign_internal_ids_workspace_bytes(int64_t n_rows, int64_t nnz, int32_t max_sample_id) {
    (void)n_rows; (void)nnz;
    if (max_sample_id < 0) return 256;
    return ids_ws_layout((int64_t)max_sample_id + 1).total;
}

extern "C" int morna_assign_internal_ids(const int64_t *row_off, const uint8_t *pass, int64_t n_rows,
                                         const int32_t *sample, int64_t nnz, int32_t max_sample_id,
                                         int64_t distinct_samples, int32_t *id_of_sample, int32_t *n_kept, void *workspace,
                                         size_t workspace_bytes, void *stream) {
    if (!row_off || !pass || !id_of_sample || !n_kept || n_rows < 0 || nnz < 0 || max_sample_id < 0)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nnz > 0 && !sample) return MORNA_ERR_INVALID_ARGUMENT;
    const int64_t m = (int64_t)max_sample_id + 1;
    IdsWs w = ids_ws_layout(m);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char *ws = (unsigned char *)workspace;
    auto *first_pos = (unsigned long long *)(ws + w.first_pos);
    auto *sorted_pos = (unsigned long long *)(ws + w.sorted_pos);
    auto *vals_in = (int32_t *)(ws + w.vals_in);
    auto *vals_out = (int32_t *)(ws + w.vals_out);
    const unsigned long long sentinel = (unsigned long long)nnz;   // one past the last pair position
    ids_init_kernel<<<grid_for(m, 256), 256, 0, s>>>(first_pos, vals_in, m, sentinel);
    MORNA_LAUNCH_CHECK();
    if (n_rows > 0 && nnz > 0) {
        // Rows in three growing stretches (1/64, 1/8, all) with a count in between: real inputs meet every sample within
        // the first few thousand rows, and the later launches then return at once instead of streaming the sample ids of
        // the whole file.  `need` = the caller's number of distinct samples (an upper bound is safe: the count is then
        // never reached and the whole stream is read, as it is for an id space with holes and no count).
        auto *seen = (int32_t *)(ws + w.flags);
        MORNA_CUDA_TRY(cudaMemsetAsync(seen, 0, 2 * sizeof(int32_t), s));
        const int32_t need = distinct_samples > 0 && distinct_samples < m ? (int32_t)distinct_samples : (int32_t)m;
        const int64_t cuts[4] = {0, g_ids_early_exit ? n_rows / 64 : 0, g_ids_early_exit ? n_rows / 8 : 0, n_rows};
        int checks = 0;
        for (int ph = 0; ph < 3; ++ph) {
            const int64_t r0 = cuts[ph], r1 = cuts[ph + 1], rows = r1 - r0;
            if (rows <= 0) continue;
            const int32_t *gate = checks ? seen + (checks - 1) : nullptr;
            if (m <= kFirstPosSmemIds && nnz < 0xffffffffLL) {
                const size_t smem = (size_t)m * sizeof(uint32_t);
                if (smem > 48 * 1024)
                    MORNA_CUDA_TRY(cudaFuncSetAttribute(first_position_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                        (int)(kFirstPosSmemIds * sizeof(uint32_t))));
                int per_sm = (int)((220 * 1024) / (smem + 1024));
                if (per_sm > 4) per_sm = 4;
                if (per_sm < 1) per_sm = 1;
                int64_t blocks = (rows + 15) / 16;
                if (blocks > (int64_t)sm_count_current() * per_sm) blocks = (int64_t)sm_count_current() * per_sm;
                first_position_smem_kernel<<<(unsigned)blocks, 512, smem, s>>>(row_off, pass, r0, r1, sample, max_sample_id,
                                                                             first_pos, gate, need);
            } else {
                first_position_kernel<<<grid_for(rows * 32, 256), 256, 0, s>>>(row_off, pass, r0, r1, sample,
                                                                              max_sample_id, first_pos, gate, need);
            }
            MORNA_LAUNCH_CHECK();
            if (r1 < n_rows && checks < 2) {
                ids_seen_count_kernel<<<grid_for(m, 256), 256, 0, s>>>(first_pos, m, sentinel, seen + checks);
                MORNA_LAUNCH_CHECK();
                ++checks;
            }
        }
    }
    size_t cub_bytes = w.cub_bytes;
    MORNA_CUDA_TRY(cub::DeviceRadixSort::SortPairs(ws + w.cub, cub_bytes, first_pos, sorted_pos, vals_in, vals_out,
                                                   (int)m, 0, bits_for(sentinel), s));
    count_launch(3);
    ids_assign_kernel<<<grid_for(m, 256), 256, 0, s>>>(sorted_pos, vals_out, m, sentinel, id_of_sample, n_kept);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" size_t morna_index_accumulate_workspace_bytes(int64_t n_rows, int64_t nnz, int32_t dim) {
    if (n_rows < 0 || dim <= 0) return 256;
    return acc_ws_layout(n_rows, nnz, dim).total;
}

extern "C" int morna_index_accumulate(const int64_t *row_off, const uint8_t *pass, const int32_t *bucket,
                                      const int8_t *sign, const double *idf, int64_t n_rows,
                                      const int32_t *sample, const int32_t *cov, int64_t nnz,
                                      const int32_t *id_of_sample, int32_t max_sample_id, int32_t id_lo, int32_t id_hi,
                                      int32_t dim, double *acc, int64_t acc_ld, void *workspace,
                                      size_t workspace_bytes, void *stream) {
    if (!row_off || !pass || !bucket || !sign || !idf || !id_of_sample || !acc || n_rows < 0 || nnz < 0 ||
        max_sample_id < 0 || dim <= 0 || id_lo < 0 || id_hi < id_lo || acc_ld < (int64_t)(id_hi - id_lo) || n_rows > 0x7fffffff)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (nnz > 0 && (!sample || !cov)) return MORNA_ERR_INVALID_ARGUMENT;
    AccWs w = acc_ws_layout(n_rows, nnz, dim);
    if (!workspace || workspace_bytes < w.total) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    if (n_rows == 0 || id_hi == id_lo) {     // nothing to add: cells [0, id_hi - id_lo) are zero, the rest stays untouched
        if (id_hi > id_lo)
            MORNA_CUDA_TRY(cudaMemset2DAsync(acc, (size_t)acc_ld * sizeof(double), 0, (size_t)(id_hi - id_lo) * sizeof(double),
                                             (size_t)dim, s));
        return MORNA_OK;
    }
    // (no zero-fill of acc: the kernels below write every cell [0, id_hi - id_lo) of every bucket column -- the sums of a
    // bucket with rows, zeros for an empty bucket; 8*N*D bytes less traffic, 0.8 ms at --features 30000)
    unsigned char *ws = (unsigned char *)workspace;
    auto *keys_in = (int32_t *)(ws + w.keys_in);
    auto *keys_out = (int32_t *)(ws + w.keys_out);
    auto *vals_in = (int32_t *)(ws + w.vals_in);
    auto *vals_out = (int32_t *)(ws + w.vals_out);
    auto *begin = (int32_t *)(ws + w.begin);
    bucket_keys_kernel<<<grid_for(n_rows, 256), 256, 0, s>>>(pass, bucket, n_rows, dim, keys_in, vals_in);
    MORNA_LAUNCH_CHECK();
    size_t cub_bytes = w.cub_bytes;
    // LSD radix sort is stable: rows of one bucket stay in file order
    MORNA_CUDA_TRY(cub::DeviceRadixSort::SortPairs(ws + w.cub, cub_bytes, keys_in, keys_out, vals_in, vals_out,
                                                   (int)n_rows, 0, bits_for((uint64_t)dim), s));
    count_launch(3);
    bucket_begin_kernel<<<grid_for(n_rows + 1, 256), 256, 0, s>>>(keys_out, n_rows, dim, begin);
    MORNA_LAUNCH_CHECK();
    const int32_t range = id_hi - id_lo;
    auto *flag = (int32_t *)(ws + w.flag);                 // [0] a row repeats a sample, [1] a row is not ascending
    MORNA_CUDA_TRY(cudaMemsetAsync(flag, 0, 2 * sizeof(int32_t), s));
    const int32_t *use_old = nullptr;                      // nullptr: the barrier-per-row variants run unconditionally
    // few rows per bucket (very wide --features): the per-(bucket, range) set-up of the warp variant is not
    // amortised and the barrier-per-row variants are faster (measured: 30,000 features over 1.1 M rows)
    const bool enough_rows = g_acc_variant == 4 || n_rows / dim >= 64 || n_rows < 4096;
    if ((g_acc_variant == 3 || g_acc_variant == 4) && enough_rows && nnz < 0x7fffffff) {
        // sample-id ranges of 2^shift ids, at most kAcc3MaxRanges of them, at least 1024 ids wide
        int32_t shift = g_acc_shift;
        while (((int64_t)max_sample_id >> shift) + 1 > kAcc3MaxRanges) ++shift;
        const int32_t n_ranges = (int32_t)(((int64_t)max_sample_id >> shift) + 1);
        auto *seg = (int32_t *)(ws + w.seg);
        auto *meta = (RowMeta *)(ws + w.meta);
        auto *bits = (uint32_t *)(ws + w.bits);
        MORNA_CUDA_TRY(cudaMemsetAsync(bits, 0, ((size_t)nnz / 32 + 2) * 4, s));
        row_start_bits_kernel<<<grid_for(n_rows, 256), 256, 0, s>>>(row_off, n_rows, nnz, bits);
        MORNA_LAUNCH_CHECK();
        if (((uintptr_t)sample & 15) == 0) {
            pairs_ascending_kernel<<<grid_for(nnz / 16 + 1, 256), 256, 0, s>>>(sample, nnz, bits, flag + 1);
        } else {                                               // (16-byte loads need an aligned array)
            rows_monotonic_kernel<<<grid_for(n_rows * 32, 256), 256, 0, s>>>(nullptr, row_off, pass, n_rows, sample, flag);
        }
        MORNA_LAUNCH_CHECK();
        // (One warp per row streaming its sample ids -- ascending check and range offsets in one pass instead of the check
        // plus a binary search per row and boundary -- was built and measured slower: 1.1-1.45 ms against 0.37 + 0.34 ms;
        // rows are short (median 150 pairs) and the per-row set-up dominates.)
        row_segments_kernel<<<grid_for(n_rows * (n_ranges + 1), 256), 256, 0, s>>>(row_off, sign, idf, sample, vals_out, begin,
                                                                                 dim, shift, n_ranges, seg, meta);
        MORNA_LAUNCH_CHECK();
        const size_t smem3 = (size_t)kAcc3Warps * (((size_t)1 << shift) * sizeof(double) + 64 * sizeof(ChunkDesc));
        if (smem3 <= 200 * 1024 && (int64_t)n_rows * n_ranges < 0x7fffffff) {
            auto *ccnt = (int32_t *)(ws + w.ccnt);
            auto *coff = (int32_t *)(ws + w.coff);
            auto *desc = (ChunkDesc *)(ws + w.desc);
            const int64_t cells = (int64_t)n_rows * n_ranges + 1;
            chunk_count_kernel<<<grid_for(cells, 256), 256, 0, s>>>(flag + 1, seg, begin, dim, n_ranges, n_rows, ccnt);
            MORNA_LAUNCH_CHECK();
            size_t cscan_bytes = w.cscan_bytes;
            MORNA_CUDA_TRY(cub::DeviceScan::ExclusiveSum(ws + w.cscan, cscan_bytes, ccnt, coff, (int)cells, s));
            count_launch(2);
            chunk_fill_kernel<<<grid_for(cells, 256), 256, 0, s>>>(flag + 1, seg, meta, begin, dim, n_ranges, coff, desc);
            MORNA_LAUNCH_CHECK();
            MORNA_CUDA_TRY(cudaFuncSetAttribute(index_accumulate3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
            dim3 grid3((unsigned)dim, (unsigned)((n_ranges + kAcc3Warps - 1) / kAcc3Warps));
            index_accumulate3_kernel<<<grid3, kAcc3Threads, smem3, s>>>(flag + 1, sample, cov, id_of_sample, begin, dim, coff, desc,
                                                                      shift, n_ranges, max_sample_id, id_lo, id_hi, acc, acc_ld);
            MORNA_LAUNCH_CHECK();
            use_old = flag + 1;                            // the variants below run only if a row was not ascending
        }
    }
    if (g_acc_pipelined) {
        auto *len = (int64_t *)(ws + w.len);
        auto *voff = (int64_t *)(ws + w.voff);
        MORNA_CUDA_TRY(cudaMemsetAsync(len + n_rows, 0, sizeof(int64_t), s));
        sorted_row_len_kernel<<<grid_for(n_rows, 256), 256, 0, s>>>(use_old, row_off, vals_out, n_rows, len);
        MORNA_LAUNCH_CHECK();
        size_t scan_bytes = w.scan_bytes;
        MORNA_CUDA_TRY(cub::DeviceScan::ExclusiveSum(ws + w.scan, scan_bytes, len, voff, (int)(n_rows + 1), s));
        count_launch(2);
        int32_t tile2 = range < kAcc2Tile ? range : kAcc2Tile;
        if (g_acc_split > 1) { const int32_t t = (range + g_acc_split - 1) / g_acc_split; if (t < tile2) tile2 = t; }
        const int32_t tiles2 = (range + tile2 - 1) / tile2;
        const size_t smem2 = (size_t)tile2 * sizeof(double) + kAcc2MetaBytes;
        if (smem2 > 48 * 1024) {
            MORNA_CUDA_TRY(cudaFuncSetAttribute(index_accumulate2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)(kAcc2Tile * sizeof(double) + kAcc2MetaBytes)));
            MORNA_CUDA_TRY(cudaFuncSetAttribute(index_accumulate2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)(kAcc2Tile * sizeof(double) + kAcc2MetaBytes)));
        }
        rows_monotonic_kernel<<<grid_for(n_rows * 32, 256), 256, 0, s>>>(use_old, row_off, pass, n_rows, sample, flag);
        MORNA_LAUNCH_CHECK();
        dim3 grid2((unsigned)dim, (unsigned)tiles2);
        index_accumulate2_kernel<false><<<grid2, kAcc2Threads, smem2, s>>>(use_old, flag, row_off, sign, idf, sample, cov, id_of_sample,
                                                                         vals_out, begin, voff, id_lo, id_hi, tile2, acc, acc_ld);
        MORNA_LAUNCH_CHECK();
        index_accumulate2_kernel<true><<<grid2, kAcc2Threads, smem2, s>>>(use_old, flag, row_off, sign, idf, sample, cov, id_of_sample,
                                                                        vals_out, begin, voff, id_lo, id_hi, tile2, acc, acc_ld);
        MORNA_LAUNCH_CHECK();
        return MORNA_OK;
    }
    const int32_t tile = range < kAccTile ? range : kAccTile;
    const int32_t tiles = (range + tile - 1) / tile;
    const size_t smem = (size_t)tile * sizeof(double);
    if (smem > 48 * 1024)
        MORNA_CUDA_TRY(cudaFuncSetAttribute(index_accumulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)(kAccTile * sizeof(double))));
    dim3 grid((unsigned)dim, (unsigned)tiles);
    index_accumulate_kernel<<<grid, kAccThreads, smem, s>>>(use_old, row_off, sign, idf, sample, cov, id_of_sample, vals_out,
                                                          begin, id_lo, id_hi, tile, acc, acc_ld);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}

extern "C" int morna_round_store(const double *acc, int64_t acc_ld, int32_t n_ids, int32_t dim, float *vectors,
                                 int64_t ld, void *stream) {
    if (!acc || !vectors || n_ids < 0 || dim <= 0 || ld < dim || (ld & 3) || acc_ld < n_ids)
        return MORNA_ERR_INVALID_ARGUMENT;
    if (n_ids == 0) return MORNA_OK;
    dim3 grid((unsigned)((n_ids + 31) / 32), (unsigned)((ld + 31) / 32));
    if (grid.y > 65535) return MORNA_ERR_INVALID_ARGUMENT;
    round_store_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(acc, acc_ld, n_ids, dim, vectors, ld);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}
