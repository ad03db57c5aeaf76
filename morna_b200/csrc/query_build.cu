// Query vectors from an intropolis file: the join of every query row's junction key against the index's
// junction keys (the keys of basename.freq.mor), on the device.  The reference tests `key in sample_frequencies`
// once per query junction in Python (morna.py:1456-1473); at intropolis sizes that is millions of dict lookups.
// The hash, the internal ids and the order-faithful scatter-add of the query rows are index_build.cu's kernels.
#include "common.cuh"

namespace morna {

// slots: a power of two, at least twice the key count (load factor <= 1/2 keeps probe chains short)
static int64_t table_slots(int64_t n_keys) {
    int64_t s = 2;
    while (s < 2 * n_keys) s <<= 1;
    return s;
}

__global__ void __launch_bounds__(256)
table_fill_kernel(int32_t *__restrict__ slots, int64_t n_slots) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_slots; i += (int64_t)gridDim.x * blockDim.x)
        slots[i] = -1;
}

// Keys are distinct (they are dict keys), so insertion needs no equality test: a key takes the first free slot from
// its home slot on.  Which key lands in which slot depends on the order of the CAS calls; the set of keys on every
// probe chain does not, so lookups are deterministic.
__global__ void __launch_bounds__(256)
table_build_kernel(const int32_t *__restrict__ raw, int64_t n_keys, int32_t *__restrict__ slots, uint32_t mask) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_keys; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t s = (uint32_t)raw[i] & mask;
        while (atomicCAS(&slots[s], -1, (int32_t)i) != -1) s = (s + 1) & mask;
    }
}

__device__ __forceinline__ bool same_bytes(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b, int32_t len) {
    for (int32_t i = 0; i < len; ++i)
        if (a[i] != b[i]) return false;
    return true;
}

// One thread per query row: probe from the home slot until the equal key (same hash, same length, same bytes) or a
// free slot.  count[key] counts the rows that found each key (a key met on two rows needs the host merge).
__global__ void __launch_bounds__(256)
lookup_kernel(const int32_t *__restrict__ slots, uint32_t mask, const uint8_t *__restrict__ tkeys,
              const int32_t *__restrict__ tkey_off, const int32_t *__restrict__ traw, const uint8_t *__restrict__ keys,
              const int32_t *__restrict__ key_off, const int32_t *__restrict__ raw, int64_t n_rows,
              const double *__restrict__ key_idf, int32_t *__restrict__ match, uint8_t *__restrict__ pass,
              double *__restrict__ idf, int32_t *__restrict__ count) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += (int64_t)gridDim.x * blockDim.x) {
        const int32_t h = raw[j], b = key_off[j], len = key_off[j + 1] - b;
        uint32_t s = (uint32_t)h & mask;
        int32_t m = -1;
        for (;;) {
            const int32_t v = slots[s];
            if (v < 0) break;
            const int32_t tb = tkey_off[v];
            if (traw[v] == h && tkey_off[v + 1] - tb == len && same_bytes(tkeys + tb, keys + b, len)) {
                m = v;
                break;
            }
            s = (s + 1) & mask;
        }
        match[j] = m;
        pass[j] = m >= 0 ? 1 : 0;
        idf[j] = m >= 0 ? key_idf[m] : 0.0;
        if (m >= 0) atomicAdd(&count[m], 1);
    }
}

// One warp per row: flags of the matched rows whose pairs the scatter-add would not combine as the reference does
// (bit 0: the key was found on another row too; bit 1: the sample ids are not strictly ascending, so one may repeat).
__global__ void __launch_bounds__(256)
row_flags_kernel(const int32_t *__restrict__ match, const int32_t *__restrict__ count, const int64_t *__restrict__ row_off,
                 const int32_t *__restrict__ sample, int64_t n_rows, uint8_t *__restrict__ flags,
                 int32_t *__restrict__ n_flagged) {
    const int lane = threadIdx.x & (kWarp - 1);
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x / kWarp);
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kWarp; r < n_rows; r += warps) {
        const int32_t m = match[r];                       // uniform across the warp
        int f = 0;
        if (m >= 0) {
            if (count[m] > 1) f = 1;
            const int64_t b = row_off[r], e = row_off[r + 1];
            bool bad = false;
            for (int64_t i = b + 1 + lane; i < e; i += kWarp) bad |= sample[i] <= sample[i - 1];
            if (__any_sync(kFull, bad)) f |= 2;
        }
        if (lane == 0) {
            flags[r] = (uint8_t)f;
            if (f) atomicAdd(n_flagged, 1);
        }
    }
}

static unsigned grid_of(int64_t work, int threads) {
    int64_t g = (work + threads - 1) / threads;
    if (g < 1) g = 1;
    if (g > 148 * 32) g = 148 * 32;
    return (unsigned)g;
}

}  // namespace morna

using namespace morna;

extern "C" size_t morna_junction_table_bytes(int64_t n_keys) {
    if (n_keys < 0) return 0;
    return (size_t)table_slots(n_keys) * sizeof(int32_t);
}

extern "C" int morna_junction_table_build(const uint8_t *keys, const int32_t *key_off, const int32_t *raw, int64_t n_keys,
                                          void *table, size_t table_bytes, void *stream) {
    if (n_keys < 0 || n_keys > (1LL << 30) || !table || (n_keys > 0 && (!keys || !key_off || !raw)))
        return MORNA_ERR_INVALID_ARGUMENT;
    const int64_t n_slots = table_slots(n_keys);
    if (table_bytes < (size_t)n_slots * sizeof(int32_t)) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    auto *slots = (int32_t *)table;
    table_fill_kernel<<<grid_of(n_slots, 256), 256, 0, s>>>(slots, n_slots);
    MORNA_LAUNCH_CHECK();
    if (n_keys > 0) {
        table_build_kernel<<<grid_of(n_keys, 256), 256, 0, s>>>(raw, n_keys, slots, (uint32_t)(n_slots - 1));
        MORNA_LAUNCH_CHECK();
    }
    return MORNA_OK;
}

extern "C" size_t morna_junction_lookup_workspace_bytes(int64_t n_keys) {
    if (n_keys < 0) return 256;
    return align_up((size_t)n_keys * sizeof(int32_t), 256) + 256;
}

extern "C" int morna_junction_lookup(const void *table, size_t table_bytes, const uint8_t *table_keys,
                                     const int32_t *table_key_off, const int32_t *table_raw, const double *key_idf,
                                     int64_t n_keys, const uint8_t *keys, const int32_t *key_off, const int32_t *raw,
                                     const int64_t *row_off, const int32_t *sample, int64_t n_rows, int32_t *match,
                                     uint8_t *pass, double *idf, uint8_t *flags, int32_t *n_flagged, void *workspace,
                                     size_t workspace_bytes, void *stream) {
    if (n_keys < 0 || n_keys > (1LL << 30) || n_rows < 0 || !table || !n_flagged ||
        (n_keys > 0 && (!table_keys || !table_key_off || !table_raw || !key_idf)) ||
        (n_rows > 0 && (!keys || !key_off || !raw || !row_off || !sample || !match || !pass || !idf || !flags)))
        return MORNA_ERR_INVALID_ARGUMENT;
    const int64_t n_slots = table_slots(n_keys);
    if (table_bytes < (size_t)n_slots * sizeof(int32_t)) return MORNA_ERR_INVALID_ARGUMENT;
    const size_t count_bytes = align_up((size_t)n_keys * sizeof(int32_t), 256);
    if (!workspace || workspace_bytes < count_bytes + 256) return MORNA_ERR_WORKSPACE_TOO_SMALL;
    cudaStream_t s = (cudaStream_t)stream;
    auto *count = (int32_t *)workspace;
    MORNA_CUDA_TRY(cudaMemsetAsync(n_flagged, 0, sizeof(int32_t), s));
    if (n_rows == 0) return MORNA_OK;
    if (n_keys > 0) MORNA_CUDA_TRY(cudaMemsetAsync(count, 0, (size_t)n_keys * sizeof(int32_t), s));
    lookup_kernel<<<grid_of(n_rows, 256), 256, 0, s>>>((const int32_t *)table, (uint32_t)(n_slots - 1), table_keys,
                                                       table_key_off, table_raw, keys, key_off, raw, n_rows, key_idf,
                                                       match, pass, idf, count);
    MORNA_LAUNCH_CHECK();
    row_flags_kernel<<<grid_of(n_rows * kWarp, 256), 256, 0, s>>>(match, count, row_off, sample, n_rows, flags, n_flagged);
    MORNA_LAUNCH_CHECK();
    return MORNA_OK;
}
