/* morna_b200 -- C ABI of the B200-native replacement for morna's hot path.
 *
 * The reference (commanderson/morna, Python 2) has no FFI of its own: its only
 * native boundaries on this path are the third-party wheels `mmh3` and `annoy`
 * and the pure-Python loops around them.  Each entry point below names the
 * reference lines (morna.py) whose work it takes over.  A maintainer binds this
 * header from Python with ctypes (see INTEGRATION.md); the in-repo binding is
 * morna_b200/_lib.py.
 *
 * Conventions
 *   - extern "C"; every function returns an int status: 0 = MORNA_OK, < 0 = error
 *     (morna_status_string() names it).  Nothing throws, exits or prints.
 *   - Pointers marked [dev] are device pointers owned by the caller (for example a
 *     torch tensor's data_ptr()); [host] are host pointers.  The library never
 *     allocates device memory: scratch space is a caller-provided workspace whose
 *     size the matching *_workspace_bytes() function reports.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     the call returns without synchronising unless stated otherwise.
 *   - Calls on different streams / host threads / devices are independent.  The only process-wide state is (a) a
 *     mutex-protected cache, per device ordinal, of the SM count and of each kernel's shared-memory opt-in, and
 *     (b) the experiment knobs of morna_debug_set_tuning (tests and tuning scripts only; set them before searching).
 *   - Row-major matrices carry an explicit leading dimension `ld` in elements.
 *     Sample vectors: float32, ld % 4 == 0, pad columns [dim, ld) must be zero.
 */
#ifndef MORNA_B200_H
#define MORNA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MORNA_ABI_VERSION 4

enum {
    MORNA_OK = 0,
    MORNA_ERR_INVALID_ARGUMENT = -1,
    MORNA_ERR_WORKSPACE_TOO_SMALL = -2,
    MORNA_ERR_CUDA = -3,          /* a CUDA runtime/driver call failed; see morna_last_cuda_error() */
    MORNA_ERR_UNSUPPORTED_DEVICE = -4, /* not an sm_100 device */
    MORNA_ERR_NO_SAMPLES = -5,    /* morna.py:399-403: no internal ids were assigned */
    MORNA_ERR_CAPACITY = -6       /* an output list overflowed its caller-provided capacity */
};

int morna_abi_version(void);
const char *morna_status_string(int status);
/* last CUDA error code seen by the calling thread inside this library (0 = none) */
int morna_last_cuda_error(void);
/* number of kernels this library has launched from the calling process (monotone counter) */
int64_t morna_kernel_launch_count(void);
/* A caller that captured calls of this library into a CUDA graph reports every replay here (kernels = the launches the
 * capture counted), so the counter keeps meaning "kernels of this library that ran". */
int morna_note_graph_replay(int64_t kernels);
/* sm count / compute capability of the current device */
int morna_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor);

/* ------------------------------------------------------------------ index build */

/* Feature-hash J junction keys.  Replaces mmh3.hash + sign + floor-mod at
 * morna.py:369-371 (and :625-627 for queries).
 *   keys    [dev] packed key bytes ("chr start end", ASCII, no terminators)
 *   key_off [dev] int32[J+1] byte offsets into keys
 *   raw     [dev] int32[J]  MurmurHash3_x86_32(key, seed 0) as signed int32
 *   bucket  [dev] int32[J]  raw mod dim, Python floor-mod (always in [0, dim))
 *   sign    [dev] int8[J]   -1 if raw < 0 else +1
 */
int morna_hash_junctions(const uint8_t *keys, const int32_t *key_off, int64_t n_rows,
                         int32_t dim, int32_t *raw, int32_t *bucket, int8_t *sign,
                         void *stream);

/* Per-row idf on the HOST with the C library's log(), i.e. the very function
 * CPython's math.log calls: idf[j] = log((double)sample_count / running_freq[j]),
 * 0 where pass[j] == 0.  Replaces morna.py:372-374.  All pointers [host]. */
int morna_idf_host(const int64_t *running_freq, const uint8_t *pass, int64_t n_rows,
                   int64_t sample_count, double *idf);

/* First-seen internal ids.  Replaces the try/except at morna.py:377-382: scanning
 * passing rows in file order and each row's sample list left to right, the i-th
 * distinct sample id met gets internal id i.
 *   row_off      [dev] int64[J+1] CSR offsets into sample[]
 *   pass         [dev] uint8[J]   1 if len(samples) >= sample_threshold (morna.py:361)
 *   sample       [dev] int32[nnz] sample ids, each in [0, max_sample_id]
 *   distinct_samples   number of distinct sample ids in the input if the caller counted them (count_samples,
 *                morna.py:789-822; an over-estimate is safe, an under-estimate is not), else 0.  Once that many ids have
 *                been met the remaining rows are not read: first-seen ids depend on first occurrences only.
 *   id_of_sample [dev] int32[max_sample_id+1] out: internal id or -1
 *   n_kept       [dev] int32[1]   out: number of ids assigned (.stats.mor line 2)
 */
size_t morna_assign_internal_ids_workspace_bytes(int64_t n_rows, int64_t nnz, int32_t max_sample_id);
int morna_assign_internal_ids(const int64_t *row_off, const uint8_t *pass, int64_t n_rows,
                              const int32_t *sample, int64_t nnz, int32_t max_sample_id, int64_t distinct_samples,
                              int32_t *id_of_sample, int32_t *n_kept,
                              void *workspace, size_t workspace_bytes, void *stream);

/* Host tokenizer (no GPU): intropolis text rows -> the binary CSR the kernels stream.  Replaces the
 * per-row Python of go_index's loop (morna.py:848-853): key = first three tab-separated fields joined
 * by single spaces, samples / coverages = comma lists of the last two fields, zip() -> min length.
 * `text` holds whole '\n'-separated lines.  Rows that are not plainly canonical (leading/trailing
 * whitespace, fewer than five fields, lists of unequal length, anything but unsigned decimal integers
 * without leading zeros)
 * get needs_python[row] = 1 and an empty entry: the caller re-tokenises them with the reference's
 * str.strip/str.split/int() semantics, so results never differ from the reference's.
 *   morna_tokenize_count: sizes for the caller's allocations (rows, key bytes, pairs)
 *   morna_tokenize_fill:  keys [key_bytes], key_off int32[rows+1], row_off int64[rows+1], sample/cov
 *                         int32[pairs], line_off int64[rows+1] (byte offset of each line in text),
 *                         needs_python uint8[rows].  All host memory. */
int morna_tokenize_count(const char *text, size_t nbytes, int32_t n_threads, int64_t *n_rows,
                         int64_t *key_bytes, int64_t *n_pairs);
int morna_tokenize_fill(const char *text, size_t nbytes, int32_t n_threads, uint8_t *keys, int32_t *key_off,
                        int64_t *row_off, int32_t *sample, int32_t *cov, int64_t *line_off,
                        uint8_t *needs_python);

/* Scatter-add of sign * (coverage * idf) into per-sample vectors.  Replaces the
 * per-pair loop at morna.py:376-388.  Sums are double and every (sample, bucket)
 * cell is accumulated in file row order, so cells equal the reference's Python
 * floats bit for bit (when a row does not list the same sample twice).  Rows whose
 * sample ids are strictly ascending (as intropolis writes them) take the fast path:
 * one warp per (bucket, sample-id range), no block barriers; any other input takes the
 * barrier-per-row path with the same results.
 * The accumulator is bucket-major: acc[b * acc_ld + (internal_id - id_lo)], and
 * only internal ids in [id_lo, id_hi) are accumulated (multi-GPU shards by id
 * range, each rank streaming the same rows).  The call writes every cell [0, id_hi - id_lo) of every
 * column (zeros where nothing was added; id_of_sample must map onto every id of the range, as
 * morna_assign_internal_ids' output does); cells at or beyond id_hi - id_lo are not touched.
 *   bucket/sign/idf  [dev] per-row, from morna_hash_junctions / morna_idf_host
 *   cov              [dev] int32[nnz] coverages
 *   id_of_sample     [dev] int32[max_sample_id + 1] from morna_assign_internal_ids
 *   acc              [dev] double[dim * acc_ld], acc_ld >= id_hi - id_lo
 */
size_t morna_index_accumulate_workspace_bytes(int64_t n_rows, int64_t nnz, int32_t dim);
int morna_index_accumulate(const int64_t *row_off, const uint8_t *pass, const int32_t *bucket,
                           const int8_t *sign, const double *idf, int64_t n_rows,
                           const int32_t *sample, const int32_t *cov, int64_t nnz,
                           const int32_t *id_of_sample, int32_t max_sample_id, int32_t id_lo, int32_t id_hi,
                           int32_t dim, double *acc, int64_t acc_ld,
                           void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ query vectors from a junction file */

/* Device hash table of an index's junction keys (the keys of basename.freq.mor), so that the rows of a query file are
 * joined against them on the device instead of one `key in sample_frequencies` test per row (morna.py:1456-1473).
 * Open addressing over a power of two of int32 slots (at least twice the key count), linear probing; a slot holds a
 * key index or -1.  Slot placement may differ between builds; lookups do not.
 *   keys/key_off [dev] the n_keys keys, packed as for morna_hash_junctions; keys must be distinct
 *   raw          [dev] int32[n_keys] their morna_hash_junctions raw hashes (any dim)
 *   table        [dev] out, morna_junction_table_bytes(n_keys) bytes */
size_t morna_junction_table_bytes(int64_t n_keys);
int morna_junction_table_build(const uint8_t *keys, const int32_t *key_off, const int32_t *raw, int64_t n_keys,
                               void *table, size_t table_bytes, void *stream);

/* Join of n_rows query rows against the table.  Replaces the per-junction `key in sample_frequencies` test and the
 * idf of finalize_query (morna.py:609-629) for every row of a query file.
 *   table_keys/table_key_off/table_raw [dev] what the table was built from;  key_idf [dev] double[n_keys], the idf
 *                of each key (morna_idf_host: the device computes no log)
 *   keys/key_off/raw [dev] the query rows' keys and raw hashes;  row_off [dev] int64[n_rows+1], sample [dev] int32[nnz]
 *   match  [dev] int32[n_rows] out: index of the key equal to row j's key (same length and bytes), or -1
 *   pass   [dev] uint8[n_rows] out: match >= 0
 *   idf    [dev] double[n_rows] out: key_idf[match], 0 without a match
 *   flags  [dev] uint8[n_rows] out, 0 for unmatched rows: bit 0 = another row matched the same key, bit 1 = the row's
 *               sample ids are not strictly ascending (a sample may repeat).  morna_index_accumulate adds such
 *               rows' pairs one by one, where the reference sums the coverages of a repeated (key, sample) first.
 *   n_flagged [dev] int32[1] out: number of rows with flags != 0 (the only value a caller need read in the common case)
 * Workspace: morna_junction_lookup_workspace_bytes(n_keys). */
size_t morna_junction_lookup_workspace_bytes(int64_t n_keys);
int morna_junction_lookup(const void *table, size_t table_bytes, const uint8_t *table_keys, const int32_t *table_key_off,
                          const int32_t *table_raw, const double *key_idf, int64_t n_keys, const uint8_t *keys,
                          const int32_t *key_off, const int32_t *raw, const int64_t *row_off, const int32_t *sample,
                          int64_t n_rows, int32_t *match, uint8_t *pass, double *idf, uint8_t *flags, int32_t *n_flagged,
                          void *workspace, size_t workspace_bytes, void *stream);

/* Round the double accumulator to the float32 sample matrix, row = internal id.
 * Replaces Annoy add_item's float cast at morna.py:405-407 / 422-424.
 *   vectors [dev] float32[n_ids * ld], pad columns zero-filled by this call */
int morna_round_store(const double *acc, int64_t acc_ld, int32_t n_ids, int32_t dim,
                      float *vectors, int64_t ld, void *stream);

/* ------------------------------------------------------------------ exact search */

/* Per-row squared norms pp[i] = sum_j v[i][j]^2 in double, with the same
 * summation tree the distance kernels use for pq and qq (so a stored row queried
 * against itself is at distance exactly 0, as in the reference).  Part of
 * cosine_distance, morna.py:101-108, hoisted out of the per-query loop.
 *   pp [dev] double[n] */
int morna_row_norms(const float *vectors, int64_t n, int32_t dim, int64_t ld, double *pp,
                    void *stream);

/* Exact angular distances of nq queries to n stored rows:
 *   d = sqrt(max(0, 2 - 2*pq/sqrt(pp*qq))) if pp*qq > 0 else sqrt(2)
 * with pp, qq, pq accumulated in double over float32-valued rows -- morna.py:101-114
 * (the reference leaves a rounding-negative radicand unclamped and would raise).
 *   queries [dev] double[nq * q_ld]  (q_ld >= dim)
 *   dist    [dev] double[nq * dist_ld]
 */
int morna_angular_distances(const float *vectors, const double *pp, int64_t n, int32_t dim,
                            int64_t ld, const double *queries, int64_t nq, int64_t q_ld,
                            double *dist, int64_t dist_ld, void *stream);

/* Exact top-k of each of nq key lists under the reference's order
 * (morna.py:705-712): distance ascending, equal distances by id DESCENDING.
 *   keys   [dev] double[nq * key_ld]      (n valid entries per list)
 *   ids    [dev] int32[nq * key_ld] or NULL; NULL means id = id_base + position
 *   out_ids/out_dist [dev] [nq * k]; lists shorter than k are padded with id -1, +inf
 */
size_t morna_select_topk_workspace_bytes(int64_t n, int64_t nq, int32_t k);
int morna_select_topk(const double *keys, const int32_t *ids, int64_t n, int64_t key_ld,
                      int32_t id_base, int64_t nq, int32_t k,
                      int32_t *out_ids, double *out_dist,
                      void *workspace, size_t workspace_bytes, void *stream);

/* Merge of per-shard exact top-k lists (the one exchange step of the row-sharded search): n_lists lists
 * per query, each sorted under the reference order and padded with id -1 / +inf, laid out
 * [n_lists][nq][k_in] as an all-gather of [nq][k_in] tensors leaves them.  Equal to morna_select_topk
 * over the concatenation (ids are distinct across shards), by rank counting instead of a selection. */
int morna_merge_sorted_topk(const double *dists, const int32_t *ids, int32_t n_lists, int64_t nq,
                            int32_t k_in, int32_t k_out, int32_t *out_ids, double *out_dist, void *stream);
/* The same merge straight out of an all-gather of packed per-rank buffers: rank g contributes nq*k_in doubles
 * (distances) followed by nq*k_in int32 (ids); `packed` [dev] is these n_lists buffers back to back (nq*k_in even). */
int morna_merge_packed_topk(const void *packed, int32_t n_lists, int64_t nq, int32_t k_in, int32_t k_out,
                            int32_t *out_ids, double *out_dist, void *stream);

/* exact_search_nn for nq queries in one call (morna.py:681-712): distances + top-k.
 * Internally tiles the queries so the distance scratch stays bounded. */
size_t morna_knn_exact_workspace_bytes(int64_t n, int64_t nq, int32_t k);
int morna_knn_exact(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                    int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                    int32_t *out_ids, double *out_dist,
                    void *workspace, size_t workspace_bytes, void *stream);
/* Per-query exclusion ("which OTHER samples resemble this one"): every *_excl entry point below takes the arguments of
 * its plain form plus
 *   row_group   [dev] int32[n]   label of each row of the call (row i = id id_base + i)
 *   query_group [dev] int32[nq]  label of each query
 * and treats row i as absent for query q iff query_group[q] >= 0 && row_group[i] == query_group[q].  Both NULL (the
 * plain form) or both set.  Results equal the plain call's over the rows that are not excluded, bit for bit; a query
 * left with fewer than k rows gets a shorter list padded with id -1 / +inf.  Here the FP64 distances of excluded pairs
 * are set to +inf before the selection, and the selected +inf entries are turned into padding. */
int morna_knn_exact_excl(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                         int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                         int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                         const int32_t *row_group, const int32_t *query_group, void *stream);

/* exact_search_nn for ONE query, HBM-bound, one kernel: every warp streams its share of the rows once
 * (4*n*ld bytes) and computes each row's exact distance with the FP64 sums of morna_knn_exact; the
 * last CTA to finish selects the k nearest under the reference order from a float key per row and
 * the stored doubles, so ids and distances are identical to morna_knn_exact.
 *   query    [dev] double[dim]
 *   fallback [dev] int32[1]  out: 1 if ties overflowed the candidate list or a query value is
 *                            >= 2^127 in magnitude (outputs then hold nothing valid and
 *                            morna_knn_exact must answer), else 0
 * The first 256 bytes of the workspace are a control block that must be zero before the first call
 * (morna_knn_single_workspace_init); every call leaves it zero again, so a workspace is
 * initialised once and reused.  One call at a time per workspace. */
size_t morna_knn_single_workspace_bytes(int64_t n);
int morna_knn_single_workspace_init(void *workspace, size_t workspace_bytes, void *stream);
int morna_knn_single(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                     int32_t id_base, const double *query, int32_t k, int32_t *out_ids, double *out_dist,
                     int32_t *fallback, void *workspace, size_t workspace_bytes, void *stream);
/* A stream of single queries (the per-query loop of exact_search_nn, morna.py:697-712, called once per query of a
 * query file): n_queries kernels of morna_knn_single back to back on `stream`, query j = queries + j*query_stride,
 * answers in out_ids/out_dist[j*k ..], fallback[j] per query.  The kernels after the first are launched with
 * programmatic stream serialisation: query j+1's scan begins when every CTA of query j has finished its share of the
 * scan -- or, by default, of its first pass over its rows -- so one CTA's selection tail and the launch gap run under the next scan.  Every query is still one full pass
 * over the matrix.  The workspace is TWO morna_knn_single workspaces back to back (2 * morna_knn_single_workspace_bytes(n)),
 * each initialised with morna_knn_single_workspace_init; the queries must be ready before the call is enqueued. */
int morna_knn_single_stream(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                            int32_t id_base, const double *queries, int64_t query_stride, int32_t n_queries,
                            int32_t k, int32_t *out_ids, double *out_dist, int32_t *fallback, void *workspace,
                            size_t workspace_bytes, void *stream);

/* exact_search_nn over a SPARSE index (rows with at most morna_sparse_max_nnz() non-zero buckets, e.g. an index built
 * from a handful of junctions such as the reference's tests/tiny_intropolis.tsv, where thousands of rows are parallel
 * and tie): the rows are given in CSR form and a (query, row) distance costs nnz(row) multiply-adds.  The non-zero
 * terms are added in the dense kernels' order, so ids and distances are bit-identical to morna_knn_exact.
 *   row_off [dev] int64[n+1]   cols [dev] int32[nnz] ascending within a row   vals [dev] float32[nnz] (non-zero)
 *   plan    [dev] int32[n]     summation plan of every row: bit 30 set = no plan (any row may say so); otherwise, for a
 *                              row of nnz <= 3 entries, bits 8..12 = nnz and bits 2e..2e+1 = the accumulator (0, 1, 2) entry e
 *                              adds into, the result being (a0 + a1) + a2.  Entries whose summation lane (col/4)%32 is
 *                              equal share an accumulator; of three distinct lanes the two with the largest
 *                              lowbit(lane_i xor lane_j) take accumulators 0 and 1.  (MornaSearch._build_csr makes it.)
 *   pp      [dev] double[n] squared row norms (morna_row_norms of the dense rows) */
int32_t morna_sparse_max_nnz(void);
size_t morna_knn_exact_sparse_workspace_bytes(int64_t n, int64_t nq, int32_t k);
int morna_knn_exact_sparse(const int64_t *row_off, const int32_t *cols, const float *vals, const int32_t *plan,
                           const double *pp, int64_t n, int32_t dim, int32_t id_base, const double *queries, int64_t nq,
                           int64_t q_ld, int32_t k, int32_t *out_ids, double *out_dist, void *workspace,
                           size_t workspace_bytes, void *stream);
/* The same with a per-query exclusion (see morna_knn_exact_excl): excluded pairs are masked between the distance
 * kernel and the selection. */
int morna_knn_exact_sparse_excl(const int64_t *row_off, const int32_t *cols, const float *vals, const int32_t *plan,
                                const double *pp, int64_t n, int32_t dim, int32_t id_base, const double *queries, int64_t nq,
                                int64_t q_ld, int32_t k, int32_t *out_ids, double *out_dist, void *workspace,
                                size_t workspace_bytes, const int32_t *row_group, const int32_t *query_group, void *stream);

/* ------------------------------------------------------------------ batched search (tensor cores) */

/* Leading dimension (in halves) of the fp16 tensor-core operand for `dim` features:
 * dim rounded up to the 64-element K tile. */
int64_t morna_tensor_operand_ld(int32_t dim);

/* Build the tensor-core operand of an index block: hs[i] = fp16(v[i] / |v[i]|), zero padded
 * to ld_h, and rho_max = max_i |v[i]/|v[i]| - hs[i]|_2, the rounding residual that bounds the
 * fp16 score error.  Index-side, once per loaded block.
 *   hs      [dev] fp16[n * ld_h]      rho_max [dev] float[1] */
int morna_prepare_tensor_operand(const float *vectors, const double *pp, int64_t n, int32_t dim,
                                 int64_t ld, void *hs, int64_t ld_h, float *rho_max, void *stream);

/* exact_search_nn for a batch of queries (morna.py:681-712) with the N x D contraction on the
 * tcgen05 tensor cores: fp16 scores with a rigorous error bound select a candidate superset
 * of the true top-k, which is re-ranked with the same FP64 sums as morna_knn_exact, so ids
 * and distances are identical to morna_knn_exact.  n <= 2^24 rows per call; rows are scored in blocks of
 * 131072 and between blocks every query's threshold is tightened to the k-th best score so far, so the
 * candidate lists stay short however many rows the call covers.
 *   overflow [dev] uint8[nq]  1 where a candidate list overflowed (massive ties): those
 *                             queries hold id -1 / +inf and must be answered by morna_knn_exact
 *   stats    [dev] int32[4]   {overflowed queries, sum of first-pass survivors,
 *                              sum of re-ranked candidates, max re-ranked candidates}
 *   phase_events [host] NULL, or 7 cudaEvent_t recorded on `stream` at the phase boundaries
 *                (start, queries prepared, pilot GEMM, thresholds, filter GEMM, final lists,
 *                re-rank) so a caller can time each kernel of the step */
size_t morna_knn_batched_workspace_bytes(int64_t n, int64_t nq, int32_t dim, int32_t k);
int morna_knn_batched(const float *vectors, const double *pp, const void *hs, int64_t ld_h,
                      const float *rho_max, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                      const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                      int32_t *out_ids, double *out_dist, uint8_t *overflow, int32_t *stats,
                      void *workspace, size_t workspace_bytes, void *const *phase_events, void *stream);

/* The two halves of morna_knn_batched, for callers that pipeline consecutive batches.  The scoring half is
 * tensor-core bound and leaves LSU, FP64 units and HBM idle; the re-rank half is an HBM/L2 gather.  So the scoring
 * call of batch i+1 can carry the re-rank of batch i as a SIDE JOB: extra warps inside its GEMM kernels draw the
 * previous batch's (query, candidate rows) items from a queue in that batch's workspace while the tensor cores run.
 *
 *   morna_knn_batched_score(batch i+1, side_job = batch i)    -- same stream
 *   morna_knn_batched_rerank(batch i, resume = 1)             -- finishes what the helper warps left, orders, writes out
 *
 * morna_knn_batched_score leaves each query's candidate list in `workspace`; morna_knn_batched_rerank must be given
 * the same workspace, queries, n, nq, k and overflow array and be ordered after it (same stream, or an event).
 * A side job names another batch's arguments exactly as its own morna_knn_batched_rerank call will (its workspace
 * must differ from the scoring call's).  resume = 0 re-ranks the whole batch (no side job was given). */
typedef struct morna_rerank_job {
    const float *vectors; const double *pp; int64_t n; int32_t dim; int64_t ld; int32_t id_base;
    const double *queries; int64_t nq; int64_t q_ld; int32_t k;
    const uint8_t *overflow; void *workspace; size_t workspace_bytes;
} morna_rerank_job;

int morna_knn_batched_score(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                            int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                            uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes,
                            void *const *phase_events, const morna_rerank_job *side_job, float *kth_bound,
                            void *stream);
/* The scoring half with a per-query exclusion (see morna_knn_exact_excl; row_group covers this call's n rows): an
 * excluded entry is absent from every selection pass (pilot threshold, refinement between row blocks, final lists), so
 * the final lists hold only allowed rows and morna_knn_batched_rerank then orders them as usual.  Excluded rows can
 * still take first-pass list slots (the filter GEMM does not look at labels); a query whose list overflows is flagged
 * as usual and must be answered by morna_knn_exact_excl.  kth_bound must be NULL (rows-sharded search has no
 * exclusion). */
int morna_knn_batched_score_excl(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                                 int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                                 uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes,
                                 void *const *phase_events, const morna_rerank_job *side_job, float *kth_bound,
                                 const int32_t *row_group, const int32_t *query_group, void *stream);
/* Rows-sharded search (one process per GPU, each holding a block of rows): give the scoring call a
 * kth_bound [dev] float[nq * k]; instead of the final candidate lists it then writes, per query, lower bounds of the
 * true cosines of its k best rows (score minus this rank's error bound; -inf pads a shorter list or an overflowed
 * query).  The ranks all-gather these (4*nq*k bytes each, NCCL) and morna_union_kth_bound takes, per query, the k-th
 * largest of the n_lists * k values: at least k rows over all shards have a true cosine at or above it.
 * morna_knn_batched_finalize then builds each rank's candidate lists from that GLOBAL bound (rows scoring
 * >= bound - eps of the rank): the ranks together re-rank about k rows per query, not k rows each.  Then
 * morna_knn_batched_rerank as usual; the per-rank lists are merged with morna_merge_sorted_topk.
 *   vals  [dev] float[n_lists * nq * k], layout [list][query][k] (what an all-gather leaves)
 *   bound [dev] float[nq] out (-inf where fewer than k finite values exist) */
int morna_union_kth_bound(const float *vals, int32_t n_lists, int64_t nq, int32_t k, float *bound, void *stream);
int morna_knn_batched_finalize(int64_t n, int64_t nq, int32_t dim, int32_t k, const float *kth_bound,
                               uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes, void *stream);
int morna_knn_batched_rerank(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                             int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                             int32_t *out_ids, double *out_dist, const uint8_t *overflow, void *workspace,
                             size_t workspace_bytes, int32_t resume, void *stream);

/* Approximate mode (the reference's default search asks Annoy for approximate neighbours, morna.py:632-678; there is
 * no forest here): the k best rows by fp16 tensor-core score, WITHOUT the exact re-rank -- the scoring half of
 * morna_knn_batched followed by a per-query sort of the first-pass list.  Ids can differ from the exact answer where
 * two cosines are closer than the fp16 error (recall@k is measured against morna_knn_batched by bench.py and the
 * tests); distances are sqrt(2 - 2 score), off by up to ~1e-4.  Same workspace, overflow and stats as morna_knn_batched. */
int morna_knn_batched_approx(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                             int32_t id_base, const double *queries, int64_t nq, int64_t q_ld, int32_t k,
                             int32_t *out_ids, double *out_dist, uint8_t *overflow, int32_t *stats,
                             void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ range search
 * Every row within an angular distance R of a query: the rows i with d(q, i) <= R, d the exact FP64 distance of
 * morna_knn_exact (bit for bit), ids global (id_base + row), each list ordered under the reference order (distance
 * ascending, equal distances id descending).  R is a finite double >= 0.  Results are CSR: the caller reads the counts,
 * builds offsets[nq + 1] (int64, offsets[0] = 0) and gives them to the second call, which writes query j's list to
 * out_ids / out_dist [offsets[j], offsets[j + 1]).  No call synchronises.
 *
 * Tensor-core route (nq <= 4096, n <= 2^24): the queries are prepared as for morna_knn_batched, one filter GEMM over
 * all n rows keeps every row whose fp16 score reaches thr[q] = rd_float((1 - R^2/2) - eps[q] - 2^-30) (a superset of
 * the rows in range, see DESIGN.md section 4), and each survivor's exact distance is checked against R.
 *   counts   [dev] int32[nq]  out: rows in range per query; 0 for an overflowed query
 *   overflow [dev] uint8[nq]  out: 1 where more than 4096 rows passed the filter or a query value is >= 2^127 in
 *                             magnitude; those queries must be answered by the FP64 route
 *   stats    [dev] int64[4]   out: {overflowed queries, first-pass survivors (all queries, uncapped),
 *                              rows in range of the other queries, max rows in range of one query}
 * morna_range_batched_emit writes the sorted lists of the queries that did not overflow (at most 4096 each; a query's
 * list is cut to its offsets' length) from the state the first call left in the same workspace. */
size_t morna_range_batched_workspace_bytes(int64_t n, int64_t nq, int32_t dim);
int morna_range_batched(const float *vectors, const double *pp, const void *hs, int64_t ld_h, const float *rho_max,
                        int64_t n, int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq,
                        int64_t q_ld, double max_distance, int32_t *counts, uint8_t *overflow, int64_t *stats,
                        void *workspace, size_t workspace_bytes, void *stream);
/* The tensor-core route with a per-query exclusion (see morna_knn_exact_excl): excluded survivors of the filter are
 * dropped before the d <= R check, so counts, lists and stats cover allowed rows only. */
int morna_range_batched_excl(const float *vectors, const double *pp, const void *hs, int64_t ld_h, const float *rho_max,
                             int64_t n, int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq,
                             int64_t q_ld, double max_distance, int32_t *counts, uint8_t *overflow, int64_t *stats,
                             void *workspace, size_t workspace_bytes, const int32_t *row_group, const int32_t *query_group,
                             void *stream);
int morna_range_batched_emit(int64_t n, int64_t nq, int32_t dim, const int64_t *offsets, const uint8_t *overflow,
                             int32_t *out_ids, double *out_dist, const void *workspace, size_t workspace_bytes,
                             void *stream);

/* FP64 route (any n, nq, query values): the distance scan of morna_knn_exact in query tiles of bounded scratch.  The
 * count call writes counts [dev] int32[nq]; the fill call scans again, compacts each query's matches in descending
 * row order and sorts every list by distance with a stable segmented radix sort (so equal distances stay id
 * descending).  total = offsets[nq] (< 2^31 per call); workspace_bytes(n, nq, 0) suffices for the count call. */
size_t morna_range_exact_workspace_bytes(int64_t n, int64_t nq, int64_t total);
int morna_range_exact_count(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                            const double *queries, int64_t nq, int64_t q_ld, double max_distance, int32_t *counts,
                            void *workspace, size_t workspace_bytes, void *stream);
int morna_range_exact_fill(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                           const double *queries, int64_t nq, int64_t q_ld, double max_distance, const int64_t *offsets,
                           int64_t total, int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                           void *stream);
/* The FP64 route with a per-query exclusion (see morna_knn_exact_excl): each tile's distances are masked before both the
 * count and the fill pass, so an excluded pair sits at +inf > R in both and counts and lists agree. */
int morna_range_exact_count_excl(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                 const double *queries, int64_t nq, int64_t q_ld, double max_distance, int32_t *counts,
                                 void *workspace, size_t workspace_bytes, const int32_t *row_group,
                                 const int32_t *query_group, void *stream);
int morna_range_exact_fill_excl(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                                const double *queries, int64_t nq, int64_t q_ld, double max_distance, const int64_t *offsets,
                                int64_t total, int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes,
                                const int32_t *row_group, const int32_t *query_group, void *stream);

/* Merge of per-rank range lists (the rows-sharded range search, after one all-gather of packed per-rank buffers).
 *   gathered     [dev] n_lists buffers back to back, 8-byte aligned; buffer g is cap doubles (distances) followed by cap
 *                int32 (ids), cap even (so every buffer stays 8-byte aligned), the same cap for every rank
 *   rank_offsets [dev] int64[n_lists * (nq + 1)]: rank g's CSR offsets (rank_offsets[g * (nq + 1)] = 0); query j's list
 *                of rank g is entries [off[j], off[j + 1]) of buffer g, off[nq] <= cap, slots past off[nq] are padding
 *   out_offsets  [dev] int64[nq + 1]: out_offsets[j] = sum over ranks of query j's earlier lists (out_offsets[0] = 0);
 *                total = out_offsets[nq]
 *   out_ids / out_dist [dev] [total]: query j's merged list at [out_offsets[j], out_offsets[j + 1])
 * Preconditions: each rank's list for a query is ordered under the reference order (distance ascending, equal distances
 * id descending), and no id occurs on two ranks.  The merge is a permutation (ids and distance bits copied unchanged),
 * by rank counting: an entry's place is its index in its own list plus, per other rank, the entries of that rank's list
 * for the same query that come before it.  Any list length; nq == 0 or total == 0 does nothing. */
int morna_merge_sorted_csr(const void *gathered, int32_t n_lists, int64_t nq, int64_t cap, const int64_t *rank_offsets,
                           const int64_t *out_offsets, int64_t total, int32_t *out_ids, double *out_dist, void *stream);

/* Group-capped search: per query, the nearest rows with at most max_per_group (N >= 1) rows of any one group.  Every row
 * carries a cap label (int32; < 0: ungrouped, a group of its own).  The answer is the walk over the brute-force list of
 * the allowed rows in the reference order (distance ascending, equal distances id descending): a row is kept iff fewer
 * than N rows of its group were kept before it, and the walk stops after k kept rows.
 *
 * The walk as a primitive, on lists already in the reference order:
 *   offsets   [dev] int64[n_lists + 1]: list j is entries [offsets[j], offsets[j + 1]) of ids / dists (total entries)
 *   cap_group [dev] int32[n_rows]: the label of id i is cap_group[i - id_base]; an id outside the rows is ungrouped;
 *             an id < 0 is padding and skipped
 *   limit     at most this many entries kept per list (< 0: no limit)
 *   out_ld > 0: list j written to out_ids / out_dists [n_lists x out_ld], padded with id -1 / +inf (0 <= limit <= out_ld;
 *             out_offsets unused)
 *   out_ld == 0: a CSR -- out_offsets [dev] int64[n_lists + 1] from 0, list j's kept entries at [out_offsets[j],
 *             out_offsets[j + 1]) of out_ids / out_dists (room for `total` entries)
 * Ids and distance bits are copied unchanged; no host synchronisation; any list length. */
size_t morna_cap_sorted_lists_workspace_bytes(int64_t n_lists, int64_t total);
int morna_cap_sorted_lists(const int64_t *offsets, int64_t n_lists, const int32_t *ids, const double *dists, int64_t total,
                           const int32_t *cap_group, int32_t id_base, int64_t n_rows, int32_t max_per_group, int64_t limit,
                           int64_t *out_offsets, int32_t *out_ids, double *out_dists, int64_t out_ld, void *workspace,
                           size_t workspace_bytes, void *stream);
/* The capped top-k on the tensor cores (arguments as morna_knn_batched; cap_group covers this call's n rows; row_group /
 * query_group: an optional exclusion as in morna_knn_batched_score_excl, both NULL or both set).  The selection passes
 * use capped k-th scores (the k-th best score among every group's best N) for their thresholds and drop an entry once N
 * rows of its group score more than 2 eps above it; the final lists are re-ranked in FP64 as usual, sorted whole and
 * walked.  out_ids / out_dist [nq x k] are the exact capped answer, bit for bit, padded with id -1 / +inf, for every
 * query not flagged in overflow (its lists overflowed: answer it with the walk over its full FP64 list).  1 <= k <= 512,
 * n <= 2^24.  stats as morna_knn_batched.
 *   block_ends [host] n_block_ends ascending row counts: after the pilot, blocks of rows end at these (ends at or below
 *              the pilot's rows are skipped), then the usual blocks follow, with a capped refinement between blocks.
 *              While the rows scored so far hold few capped entries the thresholds are weak (absent below k) and the
 *              filter appends most rows of a block, so a block must be small for the lists to stay below 4096 entries.
 *              Any schedule gives the same results (a list that overflows goes to the FP64 route); MornaSearch sizes the
 *              blocks from the labels alone. */
size_t morna_knn_batched_capped_workspace_bytes(int64_t n, int64_t nq, int32_t dim, int32_t k);
int morna_knn_batched_capped(const float *vectors, const double *pp, const void *hs, int64_t ld_h, const float *rho_max,
                             int64_t n, int32_t dim, int64_t ld, int32_t id_base, const double *queries, int64_t nq,
                             int64_t q_ld, int32_t k, const int32_t *cap_group, int32_t max_per_group,
                             const int64_t *block_ends, int32_t n_block_ends, const int32_t *row_group,
                             const int32_t *query_group, int32_t *out_ids, double *out_dist,
                             uint8_t *overflow, int32_t *stats, void *workspace, size_t workspace_bytes, void *stream);

/* Within-group search, grouped FP64 route: each query against the rows of its own group only (at most 8192 rows),
 * many groups in one call.  The caller lists the rows grouped and the queries sorted by group:
 *   group_rows  [dev] int32 local row ids (0 .. n-1); the rows of one group are contiguous and ascending
 *   queries     [dev] float64 [nq x q_ld], every query's group a run of consecutive queries
 *   row_begin   [dev] int32[nq]: where query j's group starts in group_rows
 *   seg_off     [dev] int64[nq + 1] from 0: query j's segment of the distance scratch (the workspace) is
 *               [seg_off[j], seg_off[j + 1]), one entry per row of its group, at most max_segment (<= 8192) entries;
 *               total = seg_off[nq]
 *   items       [dev] int32[n_items x 4], 16-byte aligned: {first query, query count 1..8, first row (index into
 *               group_rows), row count}; the queries of an item share one group, the rows are part of it, and together
 *               the items cover every (query, row of its group) pair once.  An item's queries are staged once and every
 *               row it names is read once for all of them; items of one group should be adjacent (their rows stay in L2)
 *   exclude_rows [dev] int32[nq] or NULL: a local row left out of query j's list (-1: none)
 *   out_slot    [dev] int32[nq]: the output row of query j
 * Distances are the canonical sums of morna_angular_distances, bit for bit.  No host synchronisation.
 * Top-k: out_ids / out_dist [.. x k], row out_slot[j] = the first k of query j's segment under the reference order (ids
 * id_base + row), padded with id -1 / +inf (an excluded row is padding too). */
size_t morna_within_group_workspace_bytes(int64_t total);
int morna_within_group_topk(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld, int32_t id_base,
                            const int32_t *group_rows, const double *queries, int64_t nq, int64_t q_ld, const int32_t *items,
                            int64_t n_items, const int64_t *seg_off, int64_t total, const int32_t *row_begin,
                            int32_t max_segment, const int32_t *exclude_rows, const int32_t *out_slot, int32_t k,
                            int32_t *out_ids, double *out_dist, void *workspace, size_t workspace_bytes, void *stream);
/* Range, in two calls: the count writes counts [dev] int64[out_slot[j]] = the entries of query j's segment with
 * d <= max_distance (finite, >= 0) and leaves the distances in the workspace; the fill, given the unchanged workspace and
 * out_offsets [dev] int64 (query j's list at [out_offsets[out_slot[j]], out_offsets[out_slot[j] + 1]), its length the
 * count), writes each list in the reference order. */
int morna_within_group_range_count(const float *vectors, const double *pp, int64_t n, int32_t dim, int64_t ld,
                                   const int32_t *group_rows, const double *queries, int64_t nq, int64_t q_ld,
                                   const int32_t *items, int64_t n_items, const int64_t *seg_off, int64_t total,
                                   const int32_t *row_begin, int32_t max_segment, const int32_t *exclude_rows,
                                   const int32_t *out_slot, double max_distance, int64_t *counts, void *workspace,
                                   size_t workspace_bytes, void *stream);
int morna_within_group_range_fill(int64_t nq, const int32_t *group_rows, int32_t id_base, const int64_t *seg_off,
                                  int64_t total, const int32_t *row_begin, int32_t max_segment, const int32_t *out_slot,
                                  const int64_t *out_offsets, int32_t *out_ids, double *out_dist, const void *workspace,
                                  size_t workspace_bytes, void *stream);

/* Test hook: raw fp16 tensor-core scores [nq x n] (n <= 8192) and the per-query bound eps. */
int morna_debug_tensor_scores(const void *hs, int64_t ld_h, const float *rho_max, int64_t n, int32_t dim,
                              const double *queries, int64_t nq, int64_t q_ld, float *scores,
                              int64_t scores_ld, float *eps_out, void *workspace, size_t workspace_bytes,
                              void *stream);

/* Experiment knobs (process-wide; not part of the drop-in surface; every setting returns the same results):
 *   0  GEMM variant (1 = CTA pairs with cta_group::2, 0 = single CTAs)      1  GEMM pipeline stages (4 or 6)
 *   3  single query: rows per warp pass (1..5, 0 = automatic)               4  index: pipelined barrier-per-row kernel (1) or the simple one (0)
 *   5  re-rank: candidate rows per warp pass (2, 4, 8, 16)                   6  re-rank: MB of rows per L2 phase (0 = no phases, -1 = automatic)
 *   7  index: id tiles per bucket column of the barrier-per-row kernel      8  index: 3 = warp-per-range kernel when it pays, 4 = always, 0 = never
 *   9  batched: rows scored between threshold refinements (default 131072)  10 batched: pilot rows (256..8192)
 *   11 batched: rows before the first refinement (0 = key 9's value)        12 index: log2 width of the sample-id ranges (10..12)
 *   13 re-rank (CTA-per-query kernel): cap on resident CTAs per SM          14 re-rank kernel: 0 = warp-granular queue items, 1 = CTA per query
 *   15 re-rank (warp kernel): CTAs per SM (0 = what fits)                   16 re-rank: items per query when not split into phases (0 = 4)
 *   17 side jobs: 0 = helper warps off (resume calls then re-rank everything)
 *   29 single-query stream: 0 = plain launches, 1 = next query starts after the scan, 2 = after the first row pass (default),
 *      3 = at once (each kernel waits for its predecessor before its first workspace write; measured equal to 2)
 *   34 re-rank: 1 = each query's candidates walked in ascending row order (default), 0 = emission order
 *   35 sparse exact path: MB of distance scratch per query tile (default 1700)
 *   36 batched: growth factor of the row blocks after the first (default 1 = equal blocks of key 9's size) */
int morna_debug_set_tuning(int32_t key, int32_t value);
/* Experiment hook: [dev] int64[grid * 4] that the pair GEMM's MMA-issuing thread fills with the cycles it spent waiting for
 * operand tiles (TMA) and for a free accumulator (epilogue), and its total; NULL switches it off (default). */
int morna_debug_gemm_counters(void *buffer);

#ifdef __cplusplus
}
#endif
#endif /* MORNA_B200_H */
