/*
 * pcompanion_b200 - C ABI of the B200-native P-Companion hot path.
 *
 * The reference (emreatilgan/P-Companion) has no FFI: its boundary is a set of PyTorch
 * nn.Modules and a Python graph class (SURVEY.md 8b).  This header is the boundary the
 * Python host (the pcompanion_b200 package, which mirrors those classes) binds with ctypes.  Every
 * entry point cites the reference code it replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; sizes are element counts;
 *   - `stream` is a cudaStream_t passed as void*; entry points enqueue work and return, they
 *     never allocate, synchronise or keep state (workspace is supplied by the caller);
 *   - return value: PC_OK or an error code; pc_last_error() gives the message (thread local);
 *   - kernels are compiled for sm_100a only; there is no CPU fallback.
 */
#ifndef PCOMPANION_B200_H
#define PCOMPANION_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pc_stream_t;

#define PC_OK 0
#define PC_ERR_INVALID 1     /* bad argument (null pointer, unsupported size) */
#define PC_ERR_CUDA 2        /* a CUDA runtime call failed */
#define PC_ERR_WORKSPACE 3   /* workspace too small */
#define PC_ERR_UNSUPPORTED 4 /* shape outside what the kernels are instantiated for */

#define PC_ABI_VERSION 1

int pc_abi_version(void);
const char* pc_last_error(void);
/* sm count / compute capability of the current device (host out-params). */
int pc_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host);

/* ------------------------------------------------------------------ (1) BPG -> CSR
 * Replaces the Python dict/set graph of src/data/bpg.py:7-38 and the inline set algebra of
 * src/data/synthetic_data.py:89-90,110-128.  An edge (src, dst) is the key src<<32 | dst, so
 * ascending key order == (src, dst) order == CSR order. */

/* keys[i] = src[i] << 32 | dst[i]        (bpg.py:19-22 add_edge, integer ids) */
int pc_edge_keys_pack(const int32_t* src, const int32_t* dst, int64_t n, uint64_t* keys, pc_stream_t stream);
/* inverse of pack */
int pc_edge_keys_unpack(const uint64_t* keys, int64_t n, int32_t* src, int32_t* dst, pc_stream_t stream);

/* LSD radix sort (8-bit digits) of 64-bit keys, ascending, result in `keys`.
 * digit_mask bit d set => byte d of the key takes part (callers that know the id range skip
 * the all-zero bytes).  Workspace: pc_sort_keys_workspace_bytes(n). */
size_t pc_sort_keys_workspace_bytes(int64_t n);
int pc_sort_keys(uint64_t* keys, int64_t n, uint32_t digit_mask, void* workspace, size_t workspace_bytes,
                 pc_stream_t stream);

/* Set semantics of edges[type].add(...) (bpg.py:21): drop adjacent duplicates of a sorted
 * array.  *n_out (device int64) receives the count.  Workspace: pc_compact_workspace_bytes(n). */
size_t pc_compact_workspace_bytes(int64_t n);
int pc_unique_sorted_keys(const uint64_t* keys, int64_t n, uint64_t* out, int64_t* n_out, void* workspace,
                          size_t workspace_bytes, pc_stream_t stream);

/* Sorted-unique set algebra: out = { x in a : (x in b) == keep_if_present }.
 * keep_if_present=1 -> a n b   (bpg.py:58-63, synthetic_data.py:89 "Bcv n Bpv")
 * keep_if_present=0 -> a - b   (bpg.py:51-56, synthetic_data.py:89-90 "- Bcp", "- (Bpv u Bcv)") */
int pc_set_filter_sorted(const uint64_t* a, int64_t na, const uint64_t* b, int64_t nb, int keep_if_present,
                         uint64_t* out, int64_t* n_out, void* workspace, size_t workspace_bytes,
                         pc_stream_t stream);

/* Sorted-unique keys -> CSR: rowptr[r] = #keys with src < r, col[e] = dst of key e.
 * Row i then lists get_neighbors(i, edge_type) in ascending order (bpg.py:24-31). */
int pc_csr_from_sorted_keys(const uint64_t* keys, int64_t n_edges, int64_t n_rows, int64_t* rowptr, int32_t* col,
                            pc_stream_t stream);

/* keys_t[e] = col[e] << 32 | row(e): the transposed edge list (sort it and call
 * pc_csr_from_sorted_keys to obtain the CSC used by the deterministic backward). */
int pc_csr_transpose_keys(const int64_t* rowptr, const int32_t* col, int64_t n_rows, int64_t n_edges,
                          uint64_t* keys_t, pc_stream_t stream);

/* ------------------------------------------------------------------ (2) Product2Vec GAT
 * Replaces the attention core of nn.MultiheadAttention as product2vec.py:24-29,60 calls it
 * (need_weights branch: q*sqrt(1/dh), bmm, softmax, dropout, bmm) and its autograd
 * (BmmBackward / SoftmaxBackward), over a CSR instead of zero-padded dense neighbours.
 *
 *   q      [n_dst, 128]  projected queries (NOT pre-scaled)
 *   kv     [n_src, 256]  projected keys (cols 0..127) | values (cols 128..255)
 *   rowptr [n_dst+1], col [E]: row i attends to kv[col[rowptr[i] .. rowptr[i+1])]
 *   o      [n_dst, 128]  sum_j softmax_j(s_ij) v_j per head (before out_proj); 0 for empty rows
 *   stats  [n_dst, 2, heads] fp32: [:,0,:] = log2-sum-exp of the scaled logits (written by fwd),
 *                                  [:,1,:] = delta = dO.O per head (written by bwd_dst)
 *   dropout_p in [0,1): attention-weight dropout (product2vec.py:27); the keep mask is a
 *   counter-based hash of (seed, dst, src, head), regenerated in the backward kernels.
 * embed dim is 128 (config.py:8); heads in {1,2,4,8}.  All three kernels are deterministic
 * (fixed summation order per row, no float atomics). */
/* q, d_o, dq and dkv carry a row stride in floats (ld_*), so Q and dO can be the two halves of one
 * [n, 256] buffer (one 1 KiB gather per edge in the src-major backward) and dQ | dK|dV the
 * column blocks of one [n, 384] buffer (a single K=384 dgrad GEMM for the packed in-projection).
 * dst_ids (int32 [n_dst], may be NULL): node id of row r for the dropout mask when the rows are virtual (see hub nodes). */
int pc_gat_fwd(const float* q, int64_t ld_q, const float* kv, const int64_t* rowptr, const int32_t* col, int64_t n_dst,
               int heads, float dropout_p, uint64_t seed, const int32_t* dst_ids, float* o, float* stats, pc_stream_t stream);
/* dst-major backward: dq [n_dst,128]; fills stats[:,1,:]. */
int pc_gat_bwd_dst(const float* q, int64_t ld_q, const float* kv, const int64_t* rowptr, const int32_t* col,
                   int64_t n_dst, int heads, float dropout_p, uint64_t seed, const int32_t* dst_ids, const float* o,
                   const float* d_o, int64_t ld_do, float* stats, float* dq, int64_t ld_dq, pc_stream_t stream);
/* stats[:,1,:] = dO . O per head on its own (pc_gat_bwd_dst also writes it); lets the src-major pass run
 * first so the multi-GPU path can start returning halo gradients while the dst-major pass computes. */
int pc_gat_delta(const float* o, const float* d_o, int64_t ld_do, int64_t n, int heads, float* stats, pc_stream_t stream);
/* src-major backward over the CSC (colptr [n_src+1], row [E] = dst ids per src, ascending):
 * dkv [n_src, 256].  A RANGE of source columns [c0, c0 + n) is processed by passing colptr + c0, kv + c0 * 256,
 * dkv + c0 * ld_dkv, n and src_base = c0 (colptr holds absolute offsets into `row`; src_base keeps the dropout
 * mask keyed on the true column id): the multi-GPU backward runs one range per halo owner so that each owner's
 * partials start travelling while the next range is computed. */
int pc_gat_bwd_src(const float* q, int64_t ld_q, const float* kv, const int64_t* colptr, const int32_t* row,
                   int64_t n_src, int heads, float dropout_p, uint64_t seed, const float* d_o, int64_t ld_do,
                   const float* stats, float* dkv, int64_t ld_dkv, int64_t src_base, const int32_t* src_ids,
                   pc_stream_t stream);
/* Hub nodes (SURVEY H8).  One warp walks one CSR row, so a row with 10^5 neighbours would take tens of milliseconds on
 * its own.  The host splits such rows into "virtual rows" - consecutive slices of the row's neighbour list, listed in
 * a small second CSR - and runs the same kernels on them (dst_ids / src_ids give the real node id of a virtual row
 * for the dropout mask; NULL = the row index itself).  pc_gat_merge_segments folds the per-slice softmax states back
 * into the row: O = sum_v O_v 2^(lse_v - lse), lse = log2 sum_v 2^(lse_v), slices in ascending order (deterministic);
 * virtual rows [seg_ptr[h], seg_ptr[h+1]) belong to row hub_rows[h].  The backward partial gradients of the slices
 * are summed with pc_rows_segment_sum. */
int pc_gat_merge_segments(const float* o_seg, const float* stats_seg, const int64_t* seg_ptr, const int64_t* hub_rows,
                          int64_t n_hubs, int heads, float* o, float* stats, pc_stream_t stream);

/* Dense row projection on the tensor cores (tcgen05, 3xTF32 split => fp32-faithful, see gemm.cu):
 *   Y[m, n] = epilogue( A[m, k] . W[n, k]^T + bias[n] )
 * Replaces the addmm behind nn.Linear (product2vec.py:14-21), the packed in-/out-projection of
 * nn.MultiheadAttention (:24-29, :60) and, on the transposed weight, their dgrad GEMMs.
 * A row-major with leading dimension lda; W row-major [n, k] (nn.Linear layout); k % 32 == 0,
 * n % 32 == 0, n <= 768.  Columns [0, split) go to out0 (ld0), [split, n) to out1 (ld1) - the
 * Q | K|V outputs of the packed in-projection.  epilogue: 0 bias, 1 tanh(. + bias),
 * 2 (. + bias) * (1 - aux^2) (gradient through tanh, aux = tanh output),
 * 3 row r keeps (. + bias) if rowptr[r+1] > rowptr[r] else takes aux[r, :] (product2vec.py:76),
 * 4 (. + bias) + aux,
 * 5 row r keeps (. + bias) if rowptr[r+1] > rowptr[r] else 0 (backward of that select: no masked copy of the gradient),
 * 6 (. + bias), plus aux[r, :] on the rows WITHOUT neighbours (their gradient bypasses the attention).
 * col_sums (float64 [2, n], may be NULL; epilogue 0 and n <= 256 only): column sums of Y and of Y^2 over the m rows, taken
 * from the output tiles while they are still in shared memory (the BatchNorm statistics of product2vec.py:16 without
 * a pass over Y); per-CTA float64 partials summed in CTA order, bit-reproducible. */
size_t pc_linear_workspace_bytes(int n, int k);   /* holds the weight pre-split into tf32 hi | lo */
int pc_linear_tf32x3(const float* a, int64_t m, int k, int64_t lda, const float* w, int n, const float* bias,
                     int epilogue, const float* aux, int64_t ld_aux, const int64_t* rowptr, float* out0, int64_t ld0,
                     int split, float* out1, int64_t ld1, double* col_sums, void* workspace, size_t workspace_bytes,
                     pc_stream_t stream);

/* Weight / bias gradient of such a projection (autograd's AddmmBackward for the weight):
 *   dW[n, k] = sum_m dY[m, n] X[m, k],  db[n] = sum_m dY[m, n]  (db may be NULL)
 * n % 128 == 0, k % 32 == 0, k <= 256; fixed reduction order (bit-reproducible). */
size_t pc_wgrad_workspace_bytes(int n, int k);
int pc_wgrad_tf32x3(const float* dy, int64_t m, int n, int64_t ld_dy, const float* x, int k, int64_t ld_x, float* dw,
                    float* db, void* workspace, size_t workspace_bytes, pc_stream_t stream);

/* BatchNorm1d + tanh of the FFN (product2vec.py:16-17) and the backward of the row select (:76).
 * pc_col_stats: sums[0,c] = sum_r x[r,c], sums[1,c] = sum_r x[r,c]^2 (float64, fixed order) - the batch
 *   statistics (and what SyncBN all-reduces).  pc_bn_bwd_reduce: sums[0,c] = sum_r dy, sums[1,c] =
 *   sum_r dy * (x - mean) * rstd.  pc_scale_shift_tanh: y = [tanh](x * scale[c] + shift[c]).
 * pc_affine2: out = ca[c] * a + cb[c] * b + cc[c] (BatchNorm input gradient with folded coefficients).
 * pc_mask_split: rows with neighbours -> kept = g, rest = 0; rows without -> kept = 0, rest = g. */
size_t pc_col_reduce_workspace_bytes(int n);
int pc_col_stats(const float* x, int64_t m, int n, int64_t ldx, double* sums, void* workspace, size_t workspace_bytes,
                 pc_stream_t stream);
/* sums[0, c] = sum of x[r, c] over the rows r WITHOUT neighbours (rowptr[r+1] == rowptr[r]), sums[1, :] = 0.  Under the
 * "rows without neighbours keep ffn(x)" select of product2vec.py:76 the out-projection's bias gradient is the column
 * sum of d_emb over all rows (a by-product of pc_wgrad_tf32x3) minus this; rows with neighbours are skipped before their
 * data is read.  Same fixed-order float64 reduction and workspace as pc_col_stats. */
int pc_col_sum_unselected(const float* x, int64_t m, int n, int64_t ldx, const int64_t* rowptr, double* sums, void* workspace,
                        size_t workspace_bytes, pc_stream_t stream);
int pc_bn_bwd_reduce(const float* dy, int64_t ld_dy, const float* x, int64_t ldx, int64_t m, int n, const float* mean,
                     const float* rstd, double* sums, void* workspace, size_t workspace_bytes, pc_stream_t stream);
int pc_scale_shift_tanh(const float* x, int64_t ldx, int64_t m, int n, const float* scale, const float* shift,
                        int apply_tanh, float* y, int64_t ldy, pc_stream_t stream);
int pc_affine2(const float* a, int64_t lda, const float* b, int64_t ldb, int64_t m, int n, const float* ca,
               const float* cb, const float* cc, float* out, int64_t ldo, pc_stream_t stream);
int pc_mask_split(const float* g, int64_t m, int n, const int64_t* rowptr, float* kept, float* rest, pc_stream_t stream);

/* ------------------------------------------------------------------ (3) hinge losses
 * Row hinge:  per[r] = max(0, margin - ||a_r - p_g + eps|| + mean_k ||a_r - n_{g,k} + eps||),
 * g = r / a_per_group, loss = mean_r per[r].
 *   triplet (product2vec.py:137-154): a_per_group = 1, kneg = 5, eps = 1e-6 (F.pairwise_distance)
 *   item    (p_companion.py:105-119):  a = proj[B*K,128], a_per_group = K, kneg = 1, eps = 0
 * d_p / d_n may be NULL (required NULL when a_per_group > 1: positives are data there). */
int pc_hinge_rows_fwd(const float* a, const float* p, const float* n, int64_t rows, int a_per_group, int kneg,
                      int dim, float margin, float eps, float* per_row, float* loss, pc_stream_t stream);
int pc_hinge_rows_bwd(const float* a, const float* p, const float* n, int64_t rows, int a_per_group, int kneg,
                      int dim, float margin, float eps, const float* grad_loss, float* d_a, float* d_p, float* d_n,
                      pc_stream_t stream);
/* Type hinge (p_companion.py:95-103): per[i] = max(0, margin - S[i,pos_i] + S[i,neg_i]).
 * bwd writes the two non-zeros of each row into a caller-zeroed d_sims. */
int pc_hinge_type_fwd(const float* sims, const int64_t* pos, const int64_t* neg, int64_t rows, int64_t n_types,
                      float margin, float* per_row, float* loss, pc_stream_t stream);
int pc_hinge_type_bwd(const float* sims, const int64_t* pos, const int64_t* neg, int64_t rows, int64_t n_types,
                      float margin, const float* grad_loss, float* d_sims, pc_stream_t stream);

/* Negative sampling for the triplet batches (data_loader.py:27-40 _get_negative_samples): for every anchor,
 * k products drawn uniformly that are != anchor, not in the anchor's similar set (row `anchor` of the
 * similarity-pair CSR, columns ascending) and pairwise distinct; -1 pads when fewer than k exist.
 * Reproducible from (seed, batch slot). */
int pc_sample_negatives(const int32_t* anchor, const int64_t* sim_rowptr, const int32_t* sim_col, int64_t batch,
                        int32_t n_nodes, int k, uint64_t seed, int32_t* out, pc_stream_t stream);
/* Feature rows of one triplet batch in one launch (data_loader.py:27-88,171-206 and the three forward calls of
 * product2vec.py:132-134, without collate_fn's zero padding).  table [N, dim] with row stride ld (floats), anchor and
 * positive int64 [batch], negatives int64 [batch, kneg], the co-view CSR (rowptr int64 [N + 1], col int32) and
 * nbr_ptr int64 [batch + 1], the exclusive prefix sum of the anchors' co-view degrees (nbr_ptr[0] = 0,
 * nbr_ptr[batch] = n_nbr; the caller computes it).  Writes
 *   rows float [batch + n_nbr + batch + batch * kneg, dim] = anchors | neighbour rows | positives | negatives,
 *     anchor b's neighbours at rows batch + nbr_ptr[b] .. in ascending CSR order (collate_fn's order);
 *   edge_row int32 [n_nbr]: the batch slot of every neighbour row, i.e. the CSC row list of the batch graph
 *     (row b attends to neighbour rows nbr_ptr[b] .. nbr_ptr[b + 1]).
 * One warp per anchor, 16-byte copies.  dim % 4 == 0, dim <= 1024, ld % 4 == 0, table and rows 16-byte aligned,
 * batch and n_nbr < 2^31, kneg >= 1; col / edge_row may be NULL when n_nbr == 0.  Indices are not checked: an anchor,
 * positive or negative outside [0, N), or an nbr_ptr that is not the prefix sum of the anchors' degrees, is undefined
 * behaviour (as for pc_sample_negatives and pc_rows_gather). */
int pc_triplet_batch_rows(const float* table, int64_t ld, int dim, const int64_t* anchor, const int64_t* positive,
                          const int64_t* negatives, int64_t batch, int kneg, const int64_t* rowptr, const int32_t* col,
                          const int64_t* nbr_ptr, int64_t n_nbr, float* rows, int32_t* edge_row, pc_stream_t stream);

/* ------------------------------------------------------------------ (4) retrieval
 * Replaces torch.matmul + torch.topk of p_companion.py:60-64, metrics.py:21,89 and the
 * per-type filter -> matmul -> topk loop of inference.py:93-113.
 * score[r,p] = sum_d double(q[r,d]) * double(c[p,d]) accumulated sequentially over d in float64 (the
 * products of float32 values are exact in float64, so the value is fully defined; oracle/retrieval.py
 * mirrors it); ranking = (score desc, index asc); padding = (-inf, -1).
 *
 * pc_topk_groups, pc_topk_by_type, pc_topk_rows and pc_topk_merge accept 1 <= k <= PC_TOPK_MAX_K.  k <= 32
 * runs a warp-distributed sorted list (one entry per lane); a larger k runs a selection whose candidates are
 * appended to shared-memory buffers with atomics and compacted by sorting.  The append order therefore varies
 * from run to run, but (score, index) is a strict total order and the scores are exactly defined, so any exact
 * selection returns the same entries in the same order: results are bit-for-bit reproducible for every k.
 *
 * pc_topk_groups: score rows are processed in groups of at most 8 that rank the same contiguous run
 * members[seg_begin[g] .. seg_end[g]) of catalog row ids (the members of one complementary type in a
 * type-sorted permutation from pc_sort_keys; members == NULL means the identity, i.e. a slice of the
 * catalog).  Group g holds the rows row_ids[grp_begin[g] .. grp_begin[g+1]).  A catalog row is read
 * once per group (for k > 32, once per sub-batch of the group's rows whose candidate buffers fit in shared
 * memory: 8 rows up to k = 256 at dim 128).  dim % 16 == 0, dim <= 1024.  Results land at the original row positions. */
#define PC_TOPK_MAX_K 1024
size_t pc_topk_groups_workspace_bytes(int64_t rows, int k, int splits);
int pc_topk_groups(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                   const int32_t* row_ids, const int32_t* grp_begin, const int64_t* seg_begin, const int64_t* seg_end,
                   int64_t n_groups, int k, int splits, int64_t index_base, double* out_scores, int64_t* out_idx,
                   void* workspace, size_t workspace_bytes, pc_stream_t stream);
/* Same ranking with the grouping done on the device (no host read-back between the query upload and the result):
 * row r ranks members[type_offsets[t] .. type_offsets[t+1]) for t = row_type[r] (row_type NULL: every row ranks
 * type 0, i.e. pass n_types = 1 and type_offsets = {0, P} for an unrestricted ranking); a row_type outside
 * [0, n_types) gives an all-padding row, as `if not type_products: continue` of inference.py:97-98.  Internally:
 * keys type << 32 | row, stable radix sort on the type bytes (pc_sort_keys), one pass that marks every eighth
 * row of a type's run as the start of a group (for k > 32: every row count the large-k kernel ranks in one
 * pass), then a ranking kernel with one CTA row per position that ranks each group as pc_topk_groups does. */
size_t pc_topk_by_type_workspace_bytes(int64_t rows, int k, int splits);
int pc_topk_by_type(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                    const int64_t* type_offsets, int n_types, const int32_t* row_type, int k, int splits,
                    int64_t index_base, double* out_scores, int64_t* out_idx, void* workspace, size_t workspace_bytes,
                    pc_stream_t stream);
/* Rank of a target (the full-catalog form of hit_at_k, src/utils/metrics.py:7-26, over the per-type filter of
 * inference.py:93-113): out_rank[r] = number of products of row r's run members[type_offsets[t] .. type_offsets[t+1])
 * (t = row_type[r]; row_type NULL: type 0, pass n_types = 1 and type_offsets = {0, P}) whose (score, global index)
 * ranks strictly before (score(q[r], target_rows[r]), target_idx[r]) under the ranking rule above; -1 when t is outside
 * [0, n_types).  target_rows [rows, dim] is the target's catalog row and target_idx [rows] its global index (ties).
 * Membership of the target in the run is not checked: the caller gives -1 to rows whose target is not a member.  For
 * a member, 0 <= out_rank[r] < k  <=>  the target is in row r's pc_topk_by_type list for k, at position out_rank[r].
 * The target's score is computed with the streaming pass's arithmetic, so it is the same bits.  Grouping as
 * pc_topk_by_type (k <= 32); the counts of every split are added into out_rank (integers: deterministic), so splits
 * need no workspace and no merge.  members, type_offsets, index_base, dim and rows < 2^31 as pc_topk_by_type. */
size_t pc_rank_by_type_workspace_bytes(int64_t rows);
int pc_rank_by_type(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                    const int64_t* type_offsets, int n_types, const int32_t* row_type, const float* target_rows,
                    const int64_t* target_idx, int splits, int64_t index_base, int64_t* out_rank, void* workspace,
                    size_t workspace_bytes, pc_stream_t stream);
/* Exclusion lists: row r ignores the products of a list E_r.  Lists hold GLOBAL product indices (int64) in CSR form,
 * excl_offsets [n_lists + 1] and excl_idx [excl_offsets[n_lists]], ascending within each list, duplicates allowed.
 * row_list [rows] (int32) maps score row r to its list; a value outside [0, n_lists) means no exclusions; row_list NULL:
 * row r uses list r.  Entries outside this catalog (shard) or of another type have no effect, so one set of lists
 * serves every shard unchanged.  n_lists == 0: no row has exclusions (the list pointers may be NULL).
 *
 * pc_topk_by_type_excluding: the exact top-k of row r's run with the products of E_r removed.  Arguments,
 * workspace (pc_topk_by_type_workspace_bytes), ranking rule, score bits, (-inf, -1) padding and reproducibility are
 * those of pc_topk_by_type; with every list empty the output equals pc_topk_by_type bit for bit.  A product is
 * looked up in E_r (binary search) only after it ranks before the current k-th entry of its row. */
int pc_topk_by_type_excluding(const float* q, int64_t rows, int dim, const float* catalog, const int32_t* members,
                              const int64_t* type_offsets, int n_types, const int32_t* row_type, int k, int splits,
                              int64_t index_base, const int64_t* excl_offsets, const int64_t* excl_idx, int64_t n_lists,
                              const int32_t* row_list, double* out_scores, int64_t* out_idx, void* workspace,
                              size_t workspace_bytes, pc_stream_t stream);
/* Filtered rank: run after pc_rank_by_type on the same stream with the same q, catalog, target_rows, target_idx,
 * row_type and index_base.  For every row with inout_rank[r] >= 0 it subtracts the number of DISTINCT entries e of E_r
 * that are local (index_base <= e < index_base + n_products), of row r's type (type_id [n_products] int32 is the
 * catalog's local type of each row; any local product when row_type is NULL, i.e. the run is the whole catalog) and
 * whose (score(q[r], e), e) ranks strictly before (score(q[r], target_rows[r]), target_idx[r]).  Both scores use the
 * streaming pass's arithmetic in its order, so they are the bits pc_rank_by_type compared: the result is the number of
 * products of the run that are not in E_r and rank before the target, and a target listed in E_r never removes
 * itself.  For every k, 0 <= rank < k exactly when pc_topk_by_type_excluding with E_r - {target} lists the target, at
 * position rank.  One warp per row; rows -1 stay -1. */
int pc_rank_remove_excluded(const float* q, int64_t rows, int dim, const float* catalog, int64_t n_products,
                            const int32_t* type_id, const int32_t* row_type, const float* target_rows,
                            const int64_t* target_idx, int64_t index_base, const int64_t* excl_offsets,
                            const int64_t* excl_idx, int64_t n_lists, const int32_t* row_list, int64_t* inout_rank,
                            pc_stream_t stream);
/* Dense whole-catalog variant on the tensor cores (north_star part 4): scores = Q . C^T as a TF32 tcgen05
 * GEMM (never materialised; approximate scores only select candidates), per-type mask (type_id[p] == row_type[r]; row_type NULL or < 0 = no mask) and a
 * per-row candidate list fused into the epilogue, then exact float64 re-scoring + ranking of the candidates.
 * `units` = product ranges per 128-row block (parallelism).  flags[r] = 1 when the guard band cannot prove
 * that no dropped product belongs to the top-k (the caller re-runs such rows on pc_topk_by_type); results of
 * unflagged rows are identical to pc_topk_groups.  k <= 16, dim % 32 == 0, dim <= 128. */
size_t pc_score_topk_workspace_bytes(int64_t rows, int units);
int pc_score_topk_dense(const float* q, int64_t rows, int dim, const float* catalog, int64_t products,
                        const int32_t* type_id, const int32_t* row_type, int k, int units, int64_t index_base,
                        float max_norm, double* out_scores, int64_t* out_idx, int32_t* flags, void* workspace,
                        size_t workspace_bytes, pc_stream_t stream);
/* Row-wise top-k of a materialised fp32 matrix [rows, cols] (torch.topk of p_companion.py:64 and
 * metrics.py:21), same ranking rule; scores are returned as exact doubles of the inputs. */
size_t pc_topk_rows_workspace_bytes(int64_t rows, int k, int splits);
int pc_topk_rows(const float* values, int64_t rows, int64_t cols, int k, int splits, double* out_scores,
                 int64_t* out_idx, void* workspace, size_t workspace_bytes, pc_stream_t stream);
/* Merge `lists` candidate lists per row ([rows, lists*k] (score, idx), idx < 0 = padding) into the
 * global top-k with ties -> lowest index (per-shard merge of SURVEY 8e; also the split merge). */
int pc_topk_merge(const double* scores, const int64_t* idx, int64_t rows, int lists, int k, double* out_scores,
                  int64_t* out_idx, pc_stream_t stream);

/* ------------------------------------------------------------------ P-Companion joint model (small dense layers)
 * Type scoring with the row top-k fused into the GEMM epilogue (p_companion.py:60-64: comp_base @ W^T, topk(3)):
 * scores[m, n] = A[m, k] . W[n, k]^T on the tensor cores (same fp32-faithful 3 x TF32 kernel as pc_linear_tf32x3, any n
 * with n % 4 == 0, no bias), the best `topk` (<= 4) columns of every row tracked in the epilogue (ties -> lowest
 * column) and merged per row.  `out` (the [m, n] matrix, row stride ld_out) may be NULL: the scores are then never
 * written.  out_scores double [m, topk], out_idx int64 [m, topk]. */
size_t pc_type_scores_topk_workspace_bytes(int64_t m, int n, int k, int topk);
int pc_type_scores_topk(const float* a, int64_t m, int k, int64_t lda, const float* w, int n, float* out, int64_t ld_out,
                        int topk, double* out_scores, int64_t* out_idx, void* workspace, size_t workspace_bytes,
                        pc_stream_t stream);
/* Two-layer MLP of type_transition.py:15-20 on gathered rows: x = table[idx[r]] (idx NULL: table[r]),
 * hidden = dropout(relu(W1 x + b1)), out = W2 hidden + b2.  W1 [hid, d_in], W2 [d_out, hid] row-major (nn.Linear
 * layout).  dropout_p in [0,1): counter-based mask from (seed, row, unit), survivors scaled by 1/(1-p) (torch's
 * Philox stream cannot be matched; pass 0 in eval mode).  seed_dev (device uint64, may be NULL) is added to `seed` at
 * run time: a step captured in a CUDA graph gets a fresh mask per replay by incrementing that counter inside the graph.
 * `hidden` [rows, hid] is kept for the backward. */
int pc_mlp2_fwd(const float* table, const int64_t* idx, int64_t rows, int d_in, int hid, int d_out, const float* w1,
                const float* b1, const float* w2, const float* b2, float dropout_p, uint64_t seed, const uint64_t* seed_dev,
                float* hidden, float* out, pc_stream_t stream);
/* Backward: d_x [rows, d_in] (may be NULL), d_w1, d_b1, d_w2, d_b2 (each may be NULL); the weight gradients are summed
 * per CTA in row order and then over the CTAs in CTA order (deterministic).  dropout_p as in the forward. */
size_t pc_mlp2_bwd_workspace_bytes(int d_in, int hid, int d_out);
int pc_mlp2_bwd(const float* d_out_rows, const float* table, const int64_t* idx, const float* hidden, int64_t rows, int d_in,
                int hid, int d_out, const float* w1, const float* w2, float dropout_p, float* d_x, float* d_w1, float* d_b1,
                float* d_w2, float* d_b2, void* workspace, size_t workspace_bytes, pc_stream_t stream);
/* item_prediction.py:33-38: out[b, t, :] = pi[b, :] * tp[b * kt + t, :]  (pi = item_projection(q), tp =
 * type_projection(T), both from pc_linear_tf32x3) and its backward d_pi = sum_t d_out * tp, d_tp = d_out * pi. */
int pc_item_combine_fwd(const float* pi, const float* tp, int64_t rows, int kt, int dim, float* out, pc_stream_t stream);
int pc_item_combine_bwd(const float* d_out, const float* pi, const float* tp, int64_t rows, int kt, int dim, float* d_pi,
                        float* d_tp, pc_stream_t stream);
/* Gradient of the type hinge (p_companion.py:95-103) with respect to the FACTORS of S = base . W^T: only S[i, pos_i] and
 * S[i, neg_i] carry gradient, so d_base[i] = c_i (W[neg_i] - W[pos_i]) and W gets -c_i base[i] on row pos_i, +c_i base[i] on
 * row neg_i, c_i = grad / rows where the hinge of row i is active (per_row[i] > 0) and pos_i != neg_i.  vals [2 rows, width]:
 * slot i -> pos_i, slot rows + i -> neg_i (summed per type by pc_rows_segment_sum). */
int pc_hinge_type_factored_bwd(const float* per_row, const int64_t* pos, const int64_t* neg, const float* grad,
                               const float* base, const float* weight, int64_t rows, int width, float* d_base, float* vals,
                               pc_stream_t stream);

/* ------------------------------------------------------------------ multi-GPU halo helpers
 * Row gather (pack boundary K|V rows before the all-to-all) and deterministic scatter-add
 * (owner-side reduction of returned dK|dV partials in fixed peer order). width in floats, %4==0. */
int pc_rows_gather(const float* table, const int64_t* index, int64_t n, int width, float* out, pc_stream_t stream);
int pc_rows_scatter_add(const float* rows, const int64_t* index, int64_t n, int width, float* table,
                        pc_stream_t stream);
/* Owner-side reduction of the returned halo partials in one pass: table[r, :] += sum over p = 0..world-1, in that
 * order, of rows[slot[p * n + r], :] for slot >= 0 (slot int32 [world, n], -1 = peer p holds no partial of row r). */
int pc_rows_reduce_peers(const float* rows, const int32_t* slot, int world, int64_t n, int width, float* table,
                         pc_stream_t stream);
/* Fused halo pack + exchange over NVLink / NVSwitch peer memory, ONE launch for all peers (new: the reference has
 * no multi-GPU path).  Rows j in [row_off[p], row_off[p+1]) of the send list go to peer p:
 *   src = table + (index ? index[j] : src_row0[p] + (j - row_off[p])) * ld
 *   dst = peer_base[p] + (dst_row0[p] + (j - row_off[p])) * width
 * peer_base[p] is the peer's halo table as mapped into THIS process (CUDA IPC / symmetric memory).  row_off
 * [world+1], peer_base, src_row0, dst_row0 [world] are HOST arrays (world <= PC_MAX_PEERS).  The send list is
 * walked cyclically from row `first_row` (rank r passes row_off[(r+1) % world], so that the ranks do not all store
 * into the same GPU at the same time).  Visibility on the peers is the caller's job: a stream-ordered cross-rank
 * barrier after the launch. */
#define PC_MAX_PEERS 16
int pc_halo_push(const float* table, int64_t ld, const int64_t* index, int world, const int64_t* row_off,
                 float* const* peer_base, const int64_t* src_row0, const int64_t* dst_row0, int64_t first_row,
                 int width, pc_stream_t stream);
/* out[r, :] = sum_{e in [rowptr[r], rowptr[r+1])} rows[col[e], :] in ascending e, zeros for empty rows: the
 * deterministic gradient of a row gather table[index] (the index list is turned into a CSR with the BPG sort
 * kernels), used for the embedding rows a triplet batch touches (product2vec.py:132-134 on a shared table). */
int pc_rows_segment_sum(const float* rows, const int64_t* rowptr, const int32_t* col, int64_t n, int width, float* out,
                        pc_stream_t stream);

/* The same as ONE call from an index list: out[n_rows, width] = dense gradient of table[index] given the gradient rows
 * [slots, width] (slot s belongs to table row index[s]); keys index << 32 | slot, stable radix sort on the row bytes,
 * CSR, pc_rows_segment_sum; every output row is multiplied by scale[0] (device scalar, may be NULL).  Replaces the atomicAdd-based backward of nn.Embedding / advanced indexing
 * (p_companion.py:54,66; product2vec.py:132-134 on a shared table) with a deterministic one. */
size_t pc_rows_index_grad_workspace_bytes(int64_t slots, int64_t n_rows);
int pc_rows_index_grad(const float* rows, const int64_t* index, int64_t slots, int64_t n_rows, int width, const float* scale,
                       float* out, void* workspace, size_t workspace_bytes, pc_stream_t stream);
/* Triplet hinge (product2vec.py:137-154) on rows of ONE table picked by index: slot_rows int64 [(2 + kneg) batch] =
 * anchors | positives | negatives (negative k of triplet b at 2 batch + b kneg + k).  Reads the rows straight from the
 * table (no gathered copy); per_row [batch], loss = mean; slot_grads [(2 + kneg) batch, dim] (may be NULL) receives the
 * gradient row of every slot for an upstream gradient of ONE - pc_rows_index_grad with scale = the upstream gradient
 * then gives d_table.  dim % 4 == 0, dim <= 512. */
int pc_triplet_indexed(const float* table, const int64_t* slot_rows, int64_t batch, int kneg, int dim, float margin, float eps,
                       float* per_row, float* loss, float* slot_grads, pc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PCOMPANION_B200_H */
