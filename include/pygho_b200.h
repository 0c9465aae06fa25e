/*
 * pygho_b200 -- C ABI of the B200 (sm_100a) kernels behind PygHO's pygho.backend layer.
 *
 * The reference (GraphPKU/PygHO) is pure Python on torch and has no FFI seam; the
 * natural boundary is the pygho.backend function API (SURVEY.md section 8b).  Every
 * entry point below replaces one ATen call chain of the reference; the citation after
 * each declaration is the reference code it stands in for (paths relative to
 * /root/reference/pygho).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless said
 *     otherwise; `stream` is a cudaStream_t passed as void*.
 *   - functions never allocate and never synchronise; outputs and workspaces are
 *     provided by the caller (size queries: *_ws_bytes).  Data-dependent sizes are
 *     written to device counters that the caller reads back once per batch.
 *   - return value: 0 on success, >0 a cudaError_t, <0 an argument error;
 *     pgh_last_error() returns a static, thread-local description.
 *   - value tensors are row-major (rows, dense) float32; plan indices are int32;
 *     API-level indices (LongTensor in the reference) are int64.
 *   - aggr: 0 sum, 1 mean, 2 max, 3 min.  Rows that receive nothing are 0 for every
 *     aggr (backend/utils.py:50-55: zero init + include_self=False).
 */
#ifndef PYGHO_B200_H
#define PYGHO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGH_SUM 0
#define PGH_MEAN 1
#define PGH_MAX 2
#define PGH_MIN 3

const char* pgh_last_error(void);
int pgh_abi_version(void);
/* fills {device ordinal, SM count, L2 bytes, cc major, cc minor}; host pointer */
int pgh_device_info(int32_t* out5);
/* run-time tuning knobs; host call.  Keys 2, 3 and 5 = fused BatchNorm kernels (CTAs per SM, rows
 * in flight, forward elements in flight; 0 = default): only the work split changes,
 * reductions stay deterministic for a given setting.  Key 7 = bit mask of mamamm profiling
 * ablations (0 = off, the default; others switch parts of the kernel off).  Key 8 = programmatic dependent
 * launch (1 = on, the default; 0 = every kernel fully serialised).  Any other key is an
 * argument error. */
int pgh_set_tuning(int key, int value);
/* profiling hook: device buffer of n_words uint64 that the pipelined mamamm kernel fills
 * with %globaltimer stamps of its three warp roles (CTA 0 only); NULL switches it off */
int pgh_debug_trace(void* device_buf, int64_t n_words);

/* ------------------------------------------------------------------ value kernels */

/* Fused gather - multiply - segmented reduce.
 *   out[r,:] = aggr_{t in seg(r)} A(t) * B(t),  seg(r) = [rowptr[r], rowptr[r+1])  or {r} if rowptr==NULL
 *   A(t) = a_val[ia(t),:] * (a_scale ? a_scale[ia(t)] : 1),  ia(t) = c ? c[t] : t
 *   B(t) = b_val ? b_val[ib(t),:] : 1,                       ib(t) = d ? d[t] : t
 * n_entries = rowptr[n_rows] when the caller knows it (0 = unknown); it only tunes the
 * work split (rows per warp), never the result.
 * Deterministic (sequential in t), no atomics, one coalesced store per output row.
 * Replaces gather+gather+mul+scatter_reduce_ of backend/Spspmm.py:314-315, Spmm.py:40-43,
 * the scatter of SpTensor.py:388-394 (sparse pooling), the gather of SpTensor.py:476
 * (unpooling) and every autograd replay of those (index_add_ / gather).            */
int pgh_seg_gmr_f32(const float* a_val, const int32_t* c, const float* a_scale,
                    const float* b_val, const int32_t* d, const int32_t* rowptr,
                    int64_t n_rows, int64_t n_entries, int64_t dense, int aggr, float* out,
                    void* stream);

/* Same with explicit row strides (in floats) so operands / the output may be column slices
 * of wider row-major tensors (e.g. one third of a concatenated feature buffer);
 * accumulate != 0 (sum / mean only) adds the result to what `out` already holds, which is
 * how several gradient contributions to one operand are summed without extra passes. */
int pgh_seg_gmr_ld_f32(const float* a_val, int64_t lda, const int32_t* c, const float* a_scale,
                       const float* b_val, int64_t ldb, const int32_t* d, const int32_t* rowptr,
                       int64_t n_rows, int64_t n_entries, int64_t dense, int aggr, int accumulate,
                       float* out, int64_t ldo, void* stream);

/* pgh_seg_gmr_ld_f32 with a fused row epilogue (dense % 128 == 0, 16-byte aligned rows, sum or
 * mean):  out[r,:] = add_src[r,:] + reduction(r) (+ add_src2[r,:])   and, if copy_src != NULL,
 * copy_dst[r,:] = copy_src[r,:]; add_src / add_src2 may be NULL (add_src2 needs add_src).  One
 * SSWL layer uses it twice: the forward writes X next to X (x) A in the concatenated buffer
 * (reference Conv.py:97-103 `catvalue`) without a separate copy; the backward adds the gradient
 * slice of the concatenation AND the gradient of the residual connection (example/zinc.py:286,
 * X + conv(X)) to dX inside the reduction instead of two more passes over the tuples.       */
int pgh_seg_gmr_fused_f32(const float* a_val, int64_t lda, const int32_t* c, const float* a_scale,
                          const float* b_val, int64_t ldb, const int32_t* d, const int32_t* rowptr,
                          int64_t n_rows, int64_t n_entries, int64_t dense, int aggr,
                          const float* add_src, int64_t ld_add, const float* add_src2,
                          int64_t ld_add2, const float* copy_src, int64_t ld_copy_src,
                          float* copy_dst, int64_t ld_copy_dst, float* out, int64_t ldo,
                          void* stream);

/* max/min backward, step 1: gscaled[r,:] = grad[r,:] / (#{t in seg(r): A(t)*B(t) == out[r,:]}
 *                                                       + [out[r,:] == 0])
 * (torch's scatter_reduce amax/amin backward splits the gradient evenly among ties and
 * counts the zero-initialised output itself as one of them). */
int pgh_seg_tie_scale_f32(const float* a_val, const int32_t* c, const float* b_val,
                          const int32_t* d, const int32_t* rowptr, int64_t n_rows,
                          int64_t dense, const float* out, const float* grad,
                          float* gscaled, void* stream);

/* max/min backward, step 2 (transposed plan, rows p of the operand being differentiated):
 *   g_self[p,:] = sum_{t in seg(p)} [self[p,:]*O(t) == out[row(t),:]] * gscaled[row(t),:] * O(t)
 *   O(t) = other_val ? other_val[io(t),:] : 1,  row(t) = row_idx ? row_idx[t] : t          */
int pgh_seg_select_bwd_f32(const float* self_val, const float* other_val,
                           const int32_t* other_idx, const int32_t* row_idx,
                           const int32_t* rowptr, int64_t n_rows, int64_t dense,
                           const float* out, const float* gscaled, float* g_self,
                           void* stream);

/* inv[r] = 1 / max(rowptr[r+1]-rowptr[r], 1)  (mean backward scale) */
int pgh_inv_count_f32(const int32_t* rowptr, int64_t n_rows, float* inv, void* stream);

/* Integer segmented reduce for coalescing integer tuple features
 * (SpTupleSampler.py:126 coalesces distances with "min"); mean floors like torch. */
int pgh_seg_reduce_i64(const int64_t* val, const int32_t* perm, const int32_t* rowptr,
                       int64_t n_rows, int64_t dense, int aggr, int64_t* out, void* stream);

/* ------------------------------------------------------------------- plan kernels */

/* key[i] = pack of the listed rows of ind (row-major (sd, ld) int64), `bits` per field,
 * first listed row most significant (backend/SpTensor.py:10-42 indicehash).
 * info[0] += #negative entries, info[1] += #entries >= 2^bits.                          */
int pgh_pack_keys(const int64_t* ind, int64_t ld, const int32_t* rows_host, int n_rows_sel,
                  int bits, int64_t nnz, int64_t* key, int32_t* info, void* stream);
/* out (sd, ld) int64 <- key  (backend/SpTensor.py:45-87 decodehash) */
int pgh_unpack_keys(const int64_t* key, int64_t n, int sd, int bits, int64_t* out,
                    int64_t ld, void* stream);
/* mixed-radix flatten / unflatten (backend/SpTensor.py:90-164); dims on host */
int pgh_pack_tight(const int64_t* ind, int64_t ld, const int32_t* rows_host,
                   const int64_t* dims_host, int n_rows_sel, int64_t nnz, int64_t* key,
                   int32_t* info, void* stream);
int pgh_unpack_tight(const int64_t* key, int64_t n, const int64_t* dims_host, int sd,
                     int64_t* out, int64_t ld, void* stream);

/* stable LSD radix sort of (key, iota) pairs on bits [0, end_bit) (torch.argsort /
 * the sort inside torch.unique, backend/Spspmm.py:102,135-142, SpTensor.py:190) */
size_t pgh_sort_ws_bytes(int64_t n);
int pgh_sort_keys_perm(const int64_t* key_in, int64_t n, int end_bit, int64_t* key_out,
                       int32_t* perm_out, void* ws, size_t ws_bytes, void* stream);
/* the same for int32 keys (row ids: what the CSR builders sort); workspace pgh_sort_ws_bytes(n) */
int pgh_sort_i32_perm(const int32_t* key_in, int64_t n, int end_bit, int32_t* key_out,
                      int32_t* perm_out, void* ws, size_t ws_bytes, void* stream);

/* run-length unique of sorted keys: ukey[0..count), seg[i] = index of key[i]'s run,
 * count written to *count_dev (torch.unique(sorted, return_inverse), Spspmm.py:135) */
size_t pgh_unique_ws_bytes(int64_t n);
int pgh_unique_sorted(const int64_t* key_sorted, int64_t n, int64_t* ukey, int32_t* seg,
                      int32_t* count_dev, void* ws, size_t ws_bytes, void* stream);

/* rowptr (n_rows+1) of a non-decreasing int32 key array with values in [0, n_rows) */
int pgh_rowptr_from_sorted(const int32_t* key_sorted, int64_t n, int64_t n_rows,
                           int32_t* rowptr, void* stream);

/* For each query q: lo[q] = lower_bound(sorted, q), off = exclusive scan of match counts,
 * off[m] = total (2x torch.searchsorted + cumsum, backend/Spspmm.py:114-126)            */
size_t pgh_match_ws_bytes(int64_t m);
int pgh_match_ranges(const int64_t* sorted_keys, int64_t n, const int64_t* queries, int64_t m,
                     int32_t* lo, int64_t* off, void* ws, size_t ws_bytes, void* stream);
/* expand the ranges: for t in [0,total): c[t] = q with off[q] <= t < off[q+1],
 * d[t] = perm2[lo[c] + t - off[c]]   (repeat_interleave/arange, Spspmm.py:128-131)      */
int pgh_expand_pairs(const int64_t* off, const int32_t* lo, const int32_t* perm2, int64_t m,
                     int64_t total, int32_t* c, int32_t* d, void* stream);
/* key[t] = pack(rest dims of ind1[:,c[t]], rest dims of ind2[:,d[t]])  (Spspmm.py:133-137) */
int pgh_pair_keys(const int64_t* ind1, int64_t ld1, int sd1, int dim1, const int64_t* ind2,
                  int64_t ld2, int sd2, int dim2, const int32_t* c, const int32_t* d,
                  int64_t total, int bits, int64_t* key, int32_t* info, void* stream);

/* pos[i] = index of keys[i] in sorted unique tkeys, -1 if absent
 * (spsphadamard_ind, backend/Spspmm.py:174-183; SpTensor.unpooling :454-468)            */
int pgh_lookup_sorted(const int64_t* tkeys, int64_t nt, const int64_t* keys, int64_t n,
                      int32_t* pos, void* stream);

/* order-preserving compaction of triples with a[t] >= 0; optional remap a = map[a] first
 * (filterind, backend/Spspmm.py:218-222).  count -> *count_dev                            */
size_t pgh_compact_ws_bytes(int64_t n);
int pgh_compact_triples(const int32_t* a, const int32_t* map, const int32_t* c,
                        const int32_t* d, int64_t n, int32_t* oa, int32_t* oc, int32_t* od,
                        int32_t* count_dev, void* ws, size_t ws_bytes, void* stream);

/* small conversions / gathers used while assembling plans */
int pgh_i64_to_i32(const int64_t* src, int64_t n, int32_t* dst, int32_t* info, void* stream);
int pgh_i32_to_i64(const int32_t* src, int64_t n, int64_t* dst, void* stream);
int pgh_gather_i32(const int32_t* src, const int32_t* idx, int64_t n, int32_t* dst, void* stream);
int pgh_gather_i64_as_i32(const int64_t* src, const int32_t* idx, int64_t n, int32_t* dst,
                          void* stream);
/* Whole CSR regrouping of a reference-format plan acd (3, T) int64 (the `acd` / `bcd` tensors
 * of backend/Spspmm.py:57-222) in one call: idx32 (3, T) = a, c, d as int32 and, for every
 * grouping in `which` (bit 1 = by a over n_out rows, 2 = by c over n_a rows, 4 = by d over n_b
 * rows): rowptr (rows + 1) and the two other index arrays gathered into that grouping's stable
 * order (first/second: by a -> (c, d), by c -> (a, d), by d -> (a, c)).  A key equal to the
 * row count sorts behind rowptr[rows] (filler entries of capacity-padded plans). */
size_t pgh_acd_regroup_ws_bytes(int64_t T);
int pgh_acd_regroup(const int64_t* acd, int64_t T, int64_t n_out, int64_t n_a, int64_t n_b,
                    int which, int32_t* idx32, int32_t* rowptr_a, int32_t* first_a,
                    int32_t* second_a, int32_t* rowptr_c, int32_t* first_c, int32_t* second_c,
                    int32_t* rowptr_d, int32_t* first_d, int32_t* second_d, void* ws,
                    size_t ws_bytes, void* stream);
/* Index structures of one embedding lookup (the encoders of the reference models,
 * example/zinc.py:233-239) in one call: idx32 (n), perm (n) = stable sort of the positions by index
 * value, levels = the row pointers of the deterministic reduction tree of the weight gradient,
 * concatenated: while size > max(2 V, 4 chunk): an array of V + ceil(size / chunk) + 1 entries
 * (size = its row count afterwards), then one of V + 1.  bounds_ws: 2 (V + 1) ints of scratch. */
size_t pgh_embedding_plan_ws_bytes(int64_t n);
int pgh_embedding_plan(const void* idx, int idx_is_i64, int64_t n, int64_t V, int64_t chunk,
                       int32_t* idx32, int32_t* perm, int32_t* levels, int64_t levels_len,
                       int32_t* bounds_ws, void* ws, size_t ws_bytes, void* stream);
/* Row-wise concatenation of two CSR groupings over the same n_rows rows (rowptr (n_rows + 1),
 * first / second (T)): row r of the result = the entries of grouping 1's row r followed by those of
 * grouping 2's row r, first indices remapped to stride * first + off.  Entries behind
 * rowptr[n_rows] (fillers of capacity-padded plans) become zeros behind the result's last row. */
int pgh_merge_groups_i32(const int32_t* rowptr1, const int32_t* first1, const int32_t* second1,
                         int64_t T1, const int32_t* rowptr2, const int32_t* first2,
                         const int32_t* second2, int64_t T2, int64_t n_rows, int stride, int off1,
                         int off2, int32_t* rowptr_out, int32_t* first_out, int32_t* second_out,
                         void* stream);
/* info[0] += number of descents key[i] > key[i+1] (0 <=> non-decreasing);
 * with strict != 0 equal neighbours count as well (sorted AND duplicate free) */
int pgh_check_sorted_i64(const int64_t* key, int64_t n, int strict, int32_t* info,
                         void* stream);

/* --------------------------------------------------------------------- masked path */

/* 2-FWL contraction of (b, n, n, dense) fp32 tensors (backend/Mamamm.py:7-64):
 *   out[b,i,k,:] = mask[b,i,k] ? sum_j A'[b,i,j,:] * B'[b,j,k,:] : 0
 *   A' = A if !trans_a else A with dims 1,2 swapped (dim1==1); same for B (dim2==2).
 * Operand pads must already be zero (MaskedTensor keeps pads at padvalue 0).
 * ext (optional, (b,3) int32) = per-graph valid extents (n_i, n_j, n_k): everything outside
 * is known to be zero in the operands / masked in the output, so it is neither read nor
 * multiplied (exact: the skipped terms are zeros).
 * algo 0 = CUDA-core tiled kernel (exact fp32), 1 = tcgen05 TF32 tensor-core kernel with one
 * CTA per (graph, 8-channel slab), 2 = the same tiles and MMAs in a persistent
 * warp-specialised pipeline (same bits as 1; falls back to 1 when two tile stages do not fit
 * in shared memory), 4 = exact fp32 FMAs from a TMA-fed shared-memory ring (same bits as 0;
 * shapes its ring cannot hold run on 0).
 * order (optional, (b) int32, a permutation of 0..b-1) = the order in which algo 4's work queue
 * hands out the graphs; largest first keeps the tail of the launch short.  Never changes the
 * result.                                                                                 */
int pgh_mamamm_f32(const float* A, int trans_a, const float* B, int trans_b,
                   const uint8_t* mask, const int32_t* ext, const int32_t* order, int64_t b,
                   int64_t n_i, int64_t n_j, int64_t n_k, int64_t dense, int algo, float* out,
                   void* stream);
/* ext2[g] = (1 + last valid row, 1 + last valid column) of a (b, n1, n2) mask */
int pgh_mask_extents(const uint8_t* mask, int64_t b, int64_t n1, int64_t n2, int32_t* ext2,
                     void* stream);

/* masked pooling of (b, n1, n2, dense) over dim 1, dim 2 or both (backend/MaTensor.py:175-206)
 *   red_dims: 1 -> over n1 (out (b,n2,dense)), 2 -> over n2 (out (b,n1,dense)), 3 -> both (out (b,dense))
 * out_mask (uint8) = any(mask) over the reduced dims.  max/min of no valid entry -> 0.   */
int pgh_masked_pool_f32(const float* data, const uint8_t* mask, int64_t b, int64_t n1,
                        int64_t n2, int64_t dense, int red_dims, int aggr, float* out,
                        uint8_t* out_mask, void* stream);
/* its backward: g_data = mask ? w * g_out[broadcast] : 0 with w = 1 (sum), 1/count (mean),
 * [data == out]/ties (max/min)                                                          */
int pgh_masked_pool_bwd_f32(const float* data, const uint8_t* mask, const float* out,
                            const float* g_out, int64_t b, int64_t n1, int64_t n2,
                            int64_t dense, int red_dims, int aggr, float* g_data,
                            void* stream);
/* out = mask ? data : value  (MaskedTensor.fill_masked, backend/MaTensor.py:113-128) */
int pgh_masked_fill_f32(const float* data, const uint8_t* mask, int64_t rows, int64_t dense,
                        float value, float* out, void* stream);

/* ------------------------------------------------------- tuplewise MLP (SURVEY 8f rank 2) */

/* BatchNorm1d (training mode, statistics over ALL tuples of the batch) fused with the
 * activation that follows it in the reference MLP block Linear -> BatchNorm -> act
 * (honn/utils.py:46-61, 85-142).  act: 0 identity, 1 SiLU, 2 ReLU.  C % 4 == 0, C <= 1024.
 *   stats      : mean[c], rstd[c] = 1/sqrt(biased var + eps); optional running-stat update
 *   fwd        : z = act(gamma * (y - mean) * rstd + beta) (+ residual)
 *   bwd_reduce : sums = (S1, S2) = (sum dyh, sum dyh * xh) over the rows, dbeta = S1, dgamma = S2
 *   bwd_apply  : dy = gamma * rstd * (dyh - S1/n - xh * S2/n); dbias = column sums of dy
 * Every reduction finishes inside its own launch (two-level "last CTA done" ticket, fixed
 * summation order: deterministic).
 *   ws       : pgh_bn_ws_bytes(rows, C) bytes of scratch
 *   tickets  : 64 int32 words, zero before the first use; the kernels leave them zero
 *   num_batches_tracked : NULL or the BatchNorm1d counter (int64), incremented by stats
 *   rows_dev : NULL, or a device int32 holding the number of VALID rows (<= rows): the tensors
 *              are padded to a fixed capacity `rows` (CUDA-graph replay of steps whose batches
 *              differ in size); pad rows are excluded from all sums, get z = 0 and dy = 0
 *   accumulate : dgamma / dbeta / dbias += result (gradient buffers of a flat bucket) instead of =
 * Cross-rank statistics (SyncBN, the single-process semantics of the reference under graph
 * sharding): stats with local_out != NULL writes the rank-local (mean, M2, count) rows (3, C)
 * and stops; pgh_bn_sync_finalize_f32 merges the all-gathered (world, 3, C) triples in rank
 * order (Chan), writes mean / rstd / running stats and inv_n[0] = 1 / total rows.  bwd_reduce's
 * `sums` are all-reduced (sum) by the caller before bwd_apply, which then takes inv_n. */
size_t pgh_bn_ws_bytes(int64_t rows, int64_t C);
int pgh_bn_stats_f32(const float* y, int64_t rows, int64_t C, const int32_t* rows_dev, float eps,
                     float momentum, float* mean, float* rstd, float* running_mean,
                     float* running_var, float* local_out, int64_t* num_batches_tracked,
                     void* ws, size_t ws_bytes, int32_t* tickets, void* stream);
int pgh_bn_sync_finalize_f32(const float* gathered, int64_t world, int64_t C, float eps,
                             float momentum, float* mean, float* rstd, float* running_mean,
                             float* running_var, float* inv_n, void* stream);
/* Linear layer with the BatchNorm statistics in its epilogue (honn/utils.py:85-142: nn.Linear
 * followed by BatchNorm1d over all tuples): y = x @ w^T + bias for row-major x (M, K), w (N, K),
 * and mean / rstd / running statistics of y over the valid rows exactly as pgh_bn_stats_f32
 * would compute them from y (same argument meaning incl. rows_dev, local_out,
 * num_batches_tracked, tickets) -- without a second pass over y.  TMA-fed tcgen05 TF32 GEMM
 * (csrc/linear_stats.cu).  Supported shapes: pgh_linear_stats_supported() (N == 128, K % 32 == 0);
 * ws: pgh_linear_stats_ws_bytes(M). */
int pgh_linear_stats_supported(int64_t M, int64_t K, int64_t N);
size_t pgh_linear_stats_ws_bytes(int64_t M);
int pgh_linear_stats_f32(const float* x, int64_t M, int64_t K, const float* w, int64_t N,
                         const float* bias, const int32_t* rows_dev, float* y, float eps,
                         float momentum, float* mean, float* rstd, float* running_mean,
                         float* running_var, float* local_out, int64_t* num_batches_tracked,
                         void* ws, size_t ws_bytes, int32_t* tickets, void* stream);
/* Eval-mode Linear -> BatchNorm1d (running statistics) -> activation in ONE pass (the same
 * TMA / tcgen05 TF32 GEMM, csrc/linear_stats.cu):
 *   z = act((x @ w^T + bias - running_mean) * rsqrt(running_var + eps) * gamma + beta) (+ residual)
 * act: 0 none, 1 SiLU, 2 ReLU.  bias, gamma (1), beta (0), residual ((M, N), 16-byte aligned) and
 * rows_dev may be NULL; rows >= *rows_dev get z = 0.  Reads the running statistics, writes only z
 * (32-byte aligned).  Shapes as pgh_linear_stats_supported(); no workspace, no tickets. */
int pgh_linear_bn_eval_f32(const float* x, int64_t M, int64_t K, const float* w, int64_t N,
                           const float* bias, const float* gamma, const float* beta,
                           const float* running_mean, const float* running_var, float eps, int act,
                           const float* residual, const int32_t* rows_dev, float* z, void* stream);
/* AdamW (torch.optim.AdamW semantics: decoupled decay, bias correction) over ONE flat buffer of
 * all parameters / gradients / moments of the model (the optimisation step of example/zinc.py:
 * 368-383 as a single launch instead of one multi-tensor launch per dtype/device group).
 * step: device float = updates done so far (the caller increments it afterwards: graph
 * capturable); grad_scale folds the 1 / world_size of the data-parallel gradient average in. */
int pgh_adamw_flat_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                       int64_t n, const float* step, float lr, float beta1, float beta2, float eps,
                       float weight_decay, float grad_scale, void* stream);
/* out[e] (+)= sum_k part[k * n + e], k < slabs, n % 4 == 0: reduction over the row slabs of a
 * split-K weight-gradient GEMM (dW = dy^T x over all tuples, honn/utils.py:85-142 backward),
 * optionally accumulating into the parameter's gradient buffer; fixed order */
int pgh_sum_slabs_f32(const float* part, int64_t slabs, int64_t n, float* out, int accumulate,
                      void* stream);
/* residual may be NULL; z = act(...) + residual is the `X + conv(X)` of example/zinc.py:286
 * folded into the last block of the layer's MLP */
int pgh_bn_act_res_fwd_f32(const float* y, const float* mean, const float* rstd,
                           const float* gamma, const float* beta, int64_t rows, int64_t C,
                           const int32_t* rows_dev, int act, const float* residual, float* z,
                           void* stream);
int pgh_bn_act_bwd_reduce_f32(const float* dz, const float* y, const float* mean, const float* rstd,
                              const float* gamma, const float* beta, int64_t rows, int64_t C,
                              const int32_t* rows_dev, int act, float* sums, float* dgamma,
                              float* dbeta, int accumulate, void* ws, size_t ws_bytes,
                              int32_t* tickets, void* stream);
int pgh_bn_act_bwd_apply_f32(const float* dz, const float* y, const float* mean, const float* rstd,
                             const float* gamma, const float* beta, const float* sums,
                             const float* inv_n, int64_t rows, int64_t C, const int32_t* rows_dev,
                             int act, float* dy, float* dbias, int accumulate, void* ws,
                             size_t ws_bytes, int32_t* tickets, void* stream);

/* ------------------------------------- batch preparation on the device (SURVEY 8f rank 1 + 3) */

/* All-pairs hop distances of every graph of a block-diagonal batch, one CTA per graph:
 * the adjacency lives in shared memory as bit rows, a warp runs the breadth-first search of
 * one root node with one 32-bit word of the visited / frontier sets per lane.
 *   edge_src/edge_dst : (E) int64 GLOBAL node ids, edges of graph g are [edge_ptr[g], edge_ptr[g+1])
 *   node_ptr, edge_ptr, sq_ptr : (B+1) int64; sq_ptr[g] = sum_{h<g} n_h^2
 *   D[sq_ptr[g] + i*n_g + j] = dist(i -> j) if <= cutoff else 255   (uint8, cutoff <= 254)
 *   cnt[node_ptr[g] + i] = #{j : dist <= cutoff}   (int32, may be NULL)
 * The search follows edges from target to source like the reference's k_hop_subgraph
 * (hodata/SpTupleSampler.py:12-88, flow='source_to_target'); graphs of up to 1024 nodes.
 * Replaces the per-node Python loop of KhopSampler (SpTupleSampler.py:91-126) and scipy's
 * shortest_path in spdsampler (MaTupleSampler.py:11-31).                                     */
int pgh_graph_dist_u8(const int64_t* edge_src, const int64_t* edge_dst, const int64_t* node_ptr,
                      const int64_t* edge_ptr, const int64_t* sq_ptr, int64_t n_graphs,
                      int64_t max_nodes, int cutoff, uint8_t* D, int32_t* cnt, void* stream);
/* Tuples {(i, j) : dist(i, j) <= cutoff} of the whole batch, sorted by (i, j), with the
 * distance as feature -- what KhopSampler + the collate offsets of SpHoData.__inc__
 * (hodata/SpData.py:60-77) produce.  node_graph: (N) int64 graph id of every node;
 * rowptr: (N+1) int64 exclusive scan of cnt; tupleid: (2, T) int64 row-major; feat: (T) int64. */
int pgh_khop_emit(const uint8_t* D, const int64_t* node_ptr, const int64_t* sq_ptr,
                  const int64_t* node_graph, const int64_t* rowptr, int64_t n_nodes,
                  int64_t n_tuples, int64_t* tupleid, int64_t* feat, void* stream);
/* I2Sampler (hodata/SpTupleSampler.py:129-174) for a whole batch: for every directed edge
 * e = (i, j) the nodes k within `hop` of i or of j; tupleid (3, T) = (i, j, k) in edge order then
 * k order, feat (T, 2) = (min(dist(i,k), hop+1), min(dist(j,k), hop+1)).  D from
 * pgh_graph_dist_u8 with cutoff >= hop + 1.  count -> scan (caller) -> emit.                  */
int pgh_i2_count(const uint8_t* D, const int64_t* edge_src, const int64_t* edge_dst,
                 const int64_t* node_ptr, const int64_t* sq_ptr, const int64_t* node_graph,
                 int64_t n_edges, int hop, int32_t* cnt, void* stream);
int pgh_i2_emit(const uint8_t* D, const int64_t* edge_src, const int64_t* edge_dst,
                const int64_t* node_ptr, const int64_t* sq_ptr, const int64_t* node_graph,
                const int64_t* rowptr, int64_t n_edges, int64_t n_tuples, int hop,
                int64_t* tupleid, int64_t* feat, void* stream);
/* Dense shortest-path-distance features padded to (B, nmax, nmax): out = min(dist, clamp)
 * (unreachable -> clamp), mask = (i < n_g) & (j < n_g), pads hold `fill`.  spdsampler
 * (MaTupleSampler.py:11-31) + to_dense_tuplefeat (MaData.py:152-212) in one pass.
 * D must come from pgh_graph_dist_u8 with cutoff >= clamp - 1.                               */
int pgh_spd_dense_i64(const uint8_t* D, const int64_t* node_ptr, const int64_t* sq_ptr,
                      int64_t n_graphs, int64_t nmax, int clamp, int64_t fill, int64_t* out,
                      uint8_t* mask, void* stream);
/* Resistance distances of every graph of a block-diagonal batch, one CTA per graph:
 *   R[sq_ptr[g] + i*n_g + j] = L+[i,i] + L+[j,j] - 2 L+[i,j]   (float32, the layout of D above)
 * with L+ the Moore-Penrose pseudo-inverse of the combinatorial Laplacian of the SIMPLE
 * undirected graph (both edge directions count once, duplicates once, self-loops dropped:
 * spdsampler's directed=False).  Pairs in different components get L+[i,i] + L+[j,j]; an
 * isolated node has L+[i,i] = 0.  fp64 inversion in shared memory (n_g(n_g+1) doubles plus the
 * bit-set adjacency), so graphs of 1..128 nodes; R is bit-symmetric with an exact 0 diagonal.
 * Replaces the per-graph pinv of rdsampler (MaTupleSampler.py:34-57).                         */
int pgh_resistance_f32(const int64_t* edge_src, const int64_t* edge_dst, const int64_t* node_ptr,
                       const int64_t* edge_ptr, const int64_t* sq_ptr, int64_t n_graphs,
                       int64_t max_nodes, float* R, void* stream);
/* rdsampler's padding (MaTupleSampler.py:34-57 + to_dense_tuplefeat, MaData.py:152-212):
 * out (B, nmax, nmax) = R of pgh_resistance_f32 where mask = (i < n_g) & (j < n_g), `fill`
 * elsewhere.                                                                                  */
int pgh_rd_dense_f32(const float* R, const int64_t* node_ptr, const int64_t* sq_ptr,
                     int64_t n_graphs, int64_t nmax, float fill, float* out, uint8_t* mask,
                     void* stream);
/* to_dense_x (MaData.py:109-149): out[g, i, :] = src[ptr[g] + i, :] for i < n_g, `fill`
 * elsewhere; mask[g, i] = i < n_g.  Elements are copied as raw 4- or 8-byte words
 * (elem_bytes), fill is the raw bit pattern.                                                  */
int pgh_pad_rows(const void* src, const int64_t* ptr, int64_t n_graphs, int64_t nmax,
                 int64_t width, int elem_bytes, uint64_t fill, void* out, uint8_t* mask,
                 void* stream);
/* to_dense_adj (MaData.py:26-72): out[g, r, c, :] = edge_attr[e, :] for every edge e=(r, c)
 * of graph g = edge_graph[e], `fill` elsewhere; mask marks the edges.  node_ptr != NULL means
 * the indices are global and node_ptr[g] is subtracted.  The call fills the pads itself
 * (one fill pass + one scatter pass, stream-ordered).                                         */
int pgh_dense_adj(const int64_t* edge_src, const int64_t* edge_dst, const int64_t* edge_graph,
                  const int64_t* node_ptr, const void* edge_attr, int64_t n_edges,
                  int64_t n_graphs, int64_t nmax, int64_t width, int elem_bytes, uint64_t fill,
                  void* out, uint8_t* mask, void* stream);

/* n independent device-to-device copies in one launch (host arrays of device pointers and byte
 * counts; sizes and addresses multiples of 4): a freshly prepared batch -> the static buffers of a
 * captured training step (the role of `.to(device)` + batch transform of hodata/Wrapper.py:90-98
 * for graph-replayed steps). */
int pgh_multi_copy(const void* const* src, void* const* dst, const int64_t* bytes, int n,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PYGHO_B200_H */
