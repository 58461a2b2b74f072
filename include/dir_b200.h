/*
 * dir_b200.h -- C ABI of libdir_b200.so: the B200 (sm_100a) embedding + FM / cross hot path.
 *
 * The reference (yinyajun/Details-In-Recommendation) is pure Python over TensorFlow 1.x and
 * has no FFI for this path; its boundary is four Python calls made while the graph is built
 * (SURVEY.md section 8b).  Each entry point below names the reference lines it stands in for.
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Every pointer is a DEVICE pointer unless its name ends
 *    in _host.  The caller owns all memory, including workspaces (query the size first).
 *  - Nothing here allocates, frees or caches device memory, creates streams or synchronises
 *    the device: all work is enqueued on `stream` (a cudaStream_t; NULL = legacy default stream).
 *  - Return value: 0 on success, a negative errno-style code otherwise
 *      DIR_EINVAL  bad shape / alignment / unsupported size
 *      DIR_ENOMEM  workspace too small
 *      DIR_EIO     CUDA launch error (text in dir_last_error())
 *  - fp32 data, int64 feature ids (the reference's dtypes: DeepCrossNetwork.py:330-332,
 *    models/DeepFM/test01.py:11-13).  Row-major.  `table`, `accum`, `emb`, `S`, `u` need
 *    16-byte alignment of every row: row strides are multiples of 4 floats.
 *  - Re-entrant: no global mutable state except a thread-local error string and an atomic
 *    launch counter.
 */
#ifndef DIR_B200_H
#define DIR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIR_EINVAL (-22)
#define DIR_ENOMEM (-12)
#define DIR_EIO (-5)

#define DIR_OPT_SGD 0     /* T[r] -= lr*g                         (models/LFM/Biased LFM/train.py:44) */
#define DIR_OPT_ADAGRAD 1 /* acc[r] += g*g; T[r] -= lr*g/sqrt(acc[r])  (deepFM.py:61 'Adagrad')    */

#define DIR_OPT_FTRL 2    /* linear weights only: [TF] SparseApplyFtrl (deepFM.py:58 'Ftrl')         */
#define DIR_OPT_PROXIMAL_ADAGRAD 3 /* [TF] SparseApplyProximalAdagrad (models/ESMM/train.py:137-139):
                                      a += g*g; eta = lr/sqrt(a); p = T - g*eta;
                                      T = sign(p) * max(|p| - eta*l1, 0) / (1 + l2*eta); single-GPU layer only */

typedef void* dir_stream_t; /* cudaStream_t */

/* Optimizer of the linear scope (first-order weights), which the reference trains separately from
 * the embedding / DNN scope: linear_optimizer='Ftrl' vs dnn_optimizer='Adagrad'
 * (models/DeepFM/deepFM.py:58-61, 230-241).  A HOST struct; NULL where it is accepted means "the
 * tables' optimizer and learning rate".  Ftrl is tf.train.FtrlOptimizer with its defaults
 * learning_rate_power = -0.5, l2_shrinkage = 0, applied to the de-duplicated gradient g of a weight w:
 *     n' = n + g^2;  sigma = (sqrt(n') - sqrt(n)) / lr;  z += g - sigma * w
 *     w  = |z| > l1 ? (sign(z) * l1 - z) / (sqrt(n') / lr + 2 * l2) : 0
 * n is `lin_accum` (initial_accumulator_value 0.1), z the 'linear' slot (zeros). */
/* l1 / l2 of a ProximalAdagrad TABLE optimizer (HOST struct; NULL = 0, 0) */
typedef struct dir_table_opt {
  float l1, l2;
} dir_table_opt;

typedef struct dir_linear_opt {
  int optimizer; /* DIR_OPT_SGD | DIR_OPT_ADAGRAD | DIR_OPT_FTRL | DIR_OPT_PROXIMAL_ADAGRAD */
  float lr;
  float l1, l2;  /* Ftrl / ProximalAdagrad l1 / l2_regularization_strength */
  float* z;      /* DEVICE: Ftrl 'linear' slot, lin_stride floats apart like lin (NULL otherwise) */
} dir_linear_opt;

int dir_version(void);
const char* dir_last_error(void);
/* kernels this library has launched since it was loaded (process-wide) */
uint64_t dir_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Forward: multi-field lookup + first order + FM second order, one pass over the ids.
 * Replaces, for one-id-per-field inputs,
 *   myself_input_layer                     models/DeepFM/deepFM.py:363-400  -> emb
 *   linear_logit_fn (linear_model, 'sum')  models/DeepFM/deepFM.py:255-275  -> first
 *   fm_logit_fn                            models/DeepFM/deepFM.py:321-335  -> fm
 *   tf.feature_column.input_layer          models/DeepCrossNetwork/DeepCrossNetwork.py:126 -> emb (= x0)
 *
 *   table[n_rows] rows of K floats, `row_stride` floats apart (row_stride >= K, multiple of 4)
 *   lin[n_rows]   first-order weight of each row, `lin_stride` floats apart (may be NULL: no first order)
 *   bias          1 float (may be NULL)
 *   feature_index [B,F] int64 ids local to their field; feature_value [B,F] or NULL (= all 1.0)
 *   field_offset  [F] int64: global row = field_offset[f] + id
 *   field_rows    [F] int64 rows of each field, or NULL (then only row < n_rows is checked: the
 *                 classic one-shared-table / global-id layout passes field_offset = 0, NULL)
 *   n_rows        rows in `table`
 * Lookups with id < 0 or feature_value <= 0 are pruned ([TF] _safe_embedding_lookup_sparse):
 * zero vector, no gradient.  Ids beyond their field are pruned too and, when `oob_flag` is not
 * NULL, *oob_flag is set to 1 (TF's CPU Gather raises InvalidArgumentError there).
 *   emb  [B,F,K] or NULL   e[b,f,:] = value * table[row]
 *   S    [B,K]   or NULL   sum over fields of e (the backward needs it)
 *   first[B], fm[B]  (first may be NULL when lin is NULL)
 *   sort_keys [B*F] uint32 or NULL: global row of each lookup, n_rows for pruned ones
 *                 (input of dir_embed_bwd_sort; requires n_rows < 2^32-1)
 * K in {4, 8, 16, 32, 64}.
 */
int dir_embed_fm_fwd(const float* table, int64_t row_stride, const float* lin, int64_t lin_stride,
                     const float* bias, const int64_t* feature_index, const float* feature_value,
                     const int64_t* field_offset, const int64_t* field_rows, int64_t n_rows,
                     int64_t B, int F, int K, float* emb, float* S, float* first, float* fm,
                     uint32_t* sort_keys, int* oob_flag, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Backward + sparse row-wise update.  Replaces TF autodiff of the ops above plus
 * optimizer.minimize (models/DeepFM/deepFM.py:230-241; Unique + UnsortedSegmentSum +
 * _deduplicate_indexed_slices + SparseApplyAdagrad / ScatterSub inside TF).
 *
 * Step 1, dir_embed_bwd_sort: stable LSD radix sort of (global row, lookup position).
 *   workspace layout is private; sorted keys / positions are found again by step 2 in the
 *   same workspace.
 * Step 2, dir_embed_bwd_reduce_update: for each run of equal rows, in lookup order,
 *     G_r  = sum value * (g_fm[b] * (S[b] - value*T_r) + u[b,f])     (K floats)
 *     g1_r = sum value * g_first[b]
 *   then T_r / lin_r are updated in place with `optimizer`.  Deterministic: fixed chunking of
 *   the sorted list, sequential sums inside a chunk, fixed-order combine across chunks; no
 *   floating-point atomics.  Pruned lookups do not touch their row.
 *   field_sel / n_sel: the fields whose lookups were sorted (dir_shard_keys with the same list:
 *   sorted entries index the compact [B, n_sel] list); NULL = all F fields.
 *   onerow_fields / n_onerow (<= 64): fields whose table has ONE row (a numeric feature scaled by
 *   feature_value).  Every sample hits the same row, so these are left out of the sort and reduced
 *   as a column sum over the batch (fixed order); they need feature_index / field_offset.
 *   accum / lin_accum: accumulators with the same strides as table / lin (NULL for SGD).
 *   optimizer: DIR_OPT_SGD | DIR_OPT_ADAGRAD | DIR_OPT_PROXIMAL_ADAGRAD (table_opt: its l1 / l2, NULL = 0).
 *   linear_opt (host, may be NULL): the linear scope's own optimizer, see dir_linear_opt.
 *   lin == NULL skips the first-order update.  u == NULL means no upstream embedding gradient.
 *   n_unique_out (device int64, may be NULL) receives the number of distinct rows updated.
 */
size_t dir_embed_bwd_workspace_bytes(int64_t n_lookups, int K);
int dir_embed_bwd_sort(const uint32_t* sort_keys, int64_t n_lookups, int64_t n_rows,
                       void* workspace, size_t workspace_bytes, dir_stream_t stream);
int dir_embed_bwd_reduce_update(float* table, float* accum, int64_t row_stride, float* lin,
                                float* lin_accum, int64_t lin_stride, const int64_t* feature_index,
                                const float* feature_value, const int64_t* field_offset,
                                const float* g_first, const float* g_fm, const float* S,
                                const float* u, int64_t B, int F, int K, int64_t n_rows,
                                const int32_t* field_sel, int n_sel, const int32_t* onerow_fields,
                                int n_onerow, int optimizer, float lr, const dir_table_opt* table_opt,
                                const dir_linear_opt* linear_opt, void* workspace,
                                size_t workspace_bytes, int64_t* n_unique_out, dir_stream_t stream);

/* The one-row fields of dir_embed_bwd_reduce_update on their own.  They touch rows no sorted lookup touches, so
 * a caller may run them on a second stream next to the sorted part (call that one with n_onerow = 0).  Fixed-order,
 * fp64-carried column sums over the batch; workspace of dir_shard_dense_workspace_bytes(K); n_unique_out receives
 * the number of one-row fields whose row was updated. */
int dir_embed_bwd_onerow_update(float* table, float* accum, int64_t row_stride, float* lin, float* lin_accum,
                                int64_t lin_stride, const int64_t* feature_index, const float* feature_value,
                                const int64_t* field_offset, const float* g_first, const float* g_fm,
                                const float* S, const float* u, int64_t B, int F, int K,
                                const int32_t* onerow_fields, int n_onerow, int optimizer, float lr,
                                const dir_table_opt* table_opt, const dir_linear_opt* linear_opt,
                                float clip_norm, void* workspace,
                                size_t workspace_bytes, int64_t* n_unique_out, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * tf.clip_by_norm on the tables' gradient (models/DeepCrossNetwork/DeepCrossNetwork.py:282-289: every gradient
 * is clipped to norm 100 before apply_gradients).  The reference holds one variable per column and [TF]
 * embedding_lookup_sparse de-duplicates ids before the gather, so a column's gradient is an IndexedSlices of its
 * per-distinct-row sums and the factor clip / max(||values||, clip) is ONE PER COLUMN, known only once all of the
 * column's sums are: the clipped backward is two passes (used only when a clip norm is set):
 *   dir_shard_unique (G = 1)          numbers the distinct rows of the sorted list: uidx, unique rows, their count
 *   dir_embed_bwd_reduce_emit_local   per-distinct-row sums -> gu[u] = (G[K], g1)
 *   dir_field_sqnorms                 per column: sum of squares of G and of g1 (fixed order, fp64)
 *   dir_rows_apply_clipped            scale by the column's factor, fused Adagrad / SGD (and linear) update
 * clip_norm of dir_embed_bwd_onerow_update (0 = none) does the same for one-row fields, whose variable is one row.
 *   unique_rows [n_capacity] uint32 global rows (ascending), n_unique_dev device int64 their count,
 *   partials    dir_field_sqnorms_bytes(F) bytes of scratch written by dir_field_sqnorms
 */
int dir_embed_bwd_reduce_emit_local(const float* table, int64_t row_stride, const float* feature_value,
                                    const float* g_first, const float* g_fm, const float* S, const float* u,
                                    const uint32_t* uidx, int64_t B, int F, int K, int64_t n_rows,
                                    const int32_t* field_sel, int n_sel, float* gu, int64_t gu_stride,
                                    void* workspace, size_t workspace_bytes, dir_stream_t stream);
size_t dir_field_sqnorms_bytes(int F);
int dir_field_sqnorms(const float* gu, int64_t gu_stride, const uint32_t* unique_rows,
                      const int64_t* n_unique_dev, const int64_t* field_offset, int F, int K, int64_t n_rows,
                      double* partials, dir_stream_t stream);
int dir_rows_apply_clipped(float* table, float* accum, int64_t row_stride, float* lin, float* lin_accum,
                           int64_t lin_stride, const float* gu, int64_t gu_stride, const uint32_t* unique_rows,
                           const int64_t* n_unique_dev, int64_t n_capacity, const int64_t* field_offset, int F,
                           int K, const double* partials, float clip_norm, int optimizer, float lr,
                           const dir_linear_opt* linear_opt, int64_t* n_unique_out, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * [TF] tf.train.AdamOptimizer on a table (the reference's DCN optimizer, models/DeepCrossNetwork/train.py:104-124).
 * On an IndexedSlices gradient TF decays the moments of EVERY row of the variable, not only the batch's:
 *   lr_t = lr * sqrt(1 - beta2_power) / (1 - beta1_power)        (fp32, the powers before this step)
 *   m = m * beta1;  m[r] += g_r * (1 - beta1);  v = v * beta2;  v[r] += (g_r * g_r) * (1 - beta2)
 *   T = T - (lr_t * m) / (sqrt(v) + epsilon)                      every row
 *   then beta1_power *= beta1, beta2_power *= beta2                (they start at beta1, beta2)
 * dir_rows_apply_adam is that step as one sweep over all n_rows rows, laid out [T(K) | m(K) | v(K)] with
 * row_stride >= 3K, after dir_shard_unique + dir_embed_bwd_reduce_emit_local (gu, unique_rows, n_unique_dev as for
 * dir_rows_apply_clipped; n_capacity = 0: no gradient, gu / unique_rows / n_unique_dev may be NULL).
 *   partials (NULL = no clip): dir_field_sqnorms' output, every column's gradient scaled by clip_by_norm(clip_norm)
 *   lin (may be NULL): first-order weights of the rows with a gradient, stepped by linear_opt (required with lin:
 *   Adam on the first-order weights is not supported); lin_accum as for dir_embed_bwd_reduce_update
 *   adam->beta_power: DEVICE float[2] = (beta1_power, beta2_power), read by the sweep and advanced after it on the
 *   same stream, so a captured CUDA graph applies the right bias correction at every replay.
 * Deterministic (no atomics).  Rows whose m and v are zero and that have no gradient are left unwritten (they do
 * not change).
 */
typedef struct dir_adam_opt {
  float lr, beta1, beta2, epsilon;  /* lr > 0, 0 <= beta < 1, epsilon > 0 */
  float* beta_power;                /* DEVICE float[2] */
} dir_adam_opt;
int dir_rows_apply_adam(float* table, int64_t row_stride, int64_t n_rows, int K, float* lin, float* lin_accum,
                        int64_t lin_stride, const dir_linear_opt* linear_opt, const float* gu, int64_t gu_stride,
                        const uint32_t* unique_rows, const int64_t* n_unique_dev, int64_t n_capacity,
                        const int64_t* field_offset, int F, const double* partials, float clip_norm,
                        const dir_adam_opt* adam, int64_t* n_unique_out, dir_stream_t stream);

/* Where step 1 left the sorted (row, position) pairs inside its workspace (read-only views). */
int dir_embed_bwd_sorted(const void* workspace, int64_t n_lookups, const uint32_t** sorted_keys,
                         const uint32_t** sorted_pos);

/* ---------------------------------------------------------------------------------------------
 * Row-sharded tables over G ranks of one NVSwitch box: owner = global row mod G, local row =
 * global row div G, every rank keeps ceil(n_rows / G) rows; the batch stays data-parallel.
 * The reference has no counterpart beyond the partitioner hook around its embedding variables
 * (models/DeepFM/deepFM.py:163-175: under a TF parameter-server cluster the variables are
 * sharded by row and ids / IndexedSlices travel over gRPC).  Here only DISTINCT rows travel,
 * once per step in each direction.
 *
 * Id-only part:
 * dir_shard_keys: keys[b*n_sel + j] = owner * cap + local row of field field_sel[j], cap = ceil(n_rows / G);
 *   pruned lookups (id < 0, value <= 0, id beyond its field) get G * cap, the `n_rows` to pass to
 *   dir_embed_bwd_sort.  With G = 1 the key is the global row: this is also how the single-GPU layer forms
 *   its sort keys.  field_sel == NULL: all F fields.
 * dir_shard_unique, on the sorted list:
 *   uidx[i]               index of sorted entry i's key among the distinct keys
 *   unique_local_rows[u]  local row (at its owner) of distinct key u; grouped by owner, ascending
 *   inv[b*F + f]          int64 index of that lookup's row in the exchanged buffer, -1 if pruned: the
 *                         feature_index to hand to dir_embed_fm_fwd (f = field_sel[j] of the sorted entry);
 *                         may be NULL
 *   owner_off[g], g = 0..G   distinct keys owned by ranks < g (owner_off[G] = their total)
 * dir_shard_dense_inv: one-row (numeric) fields are replicated parameters, not exchanged: inv[b, f] =
 *   tail_row + j where the lookup survives (id == 0, value > 0), else -1.
 */
int dir_shard_keys(const int64_t* feature_index, const float* feature_value,
                   const int64_t* field_offset, const int64_t* field_rows, int64_t n_rows, int64_t B,
                   int F, int G, const int32_t* field_sel, int n_sel, uint32_t* keys, int* oob_flag,
                   dir_stream_t stream);
/* Bags (CSR, as dir_embed_bag_fm_fwd takes them): keys[j] for entry j of bag_index, pruned entries (id < 0,
 * weight <= 0, id beyond its field) get the key G * cap.  The sorted list then indexes ENTRIES: dir_shard_unique
 * with field_sel = NULL leaves inv[j] = row of entry j in the exchanged buffer. */
int dir_shard_bag_keys(const int64_t* bag_offsets, const int64_t* bag_index, const float* bag_weight, int64_t nnz,
                       const int64_t* field_offset, const int64_t* field_rows, int64_t n_rows, int64_t B, int F,
                       int G, uint32_t* keys, int* oob_flag, dir_stream_t stream);
/* dir_shard_keys followed by dir_embed_bwd_sort on the same stream, as one call: the key kernel counts the sort's
 * first digit while the keys are in registers (one pass over the keys and one launch less).  `keys` is still
 * written (the sort's first pass reads it); workspace as for dir_embed_bwd_sort with n_lookups = B * n_sel. */
int dir_shard_keys_sort(const int64_t* feature_index, const float* feature_value, const int64_t* field_offset,
                        const int64_t* field_rows, int64_t n_rows, int64_t B, int F, int G,
                        const int32_t* field_sel, int n_sel, uint32_t* keys, int* oob_flag, void* workspace,
                        size_t workspace_bytes, dir_stream_t stream);
size_t dir_shard_unique_workspace_bytes(int64_t n_lookups);
int dir_shard_unique(const uint32_t* sorted_keys, const uint32_t* sorted_pos, int64_t n_lookups,
                     int64_t n_rows, int G, const int32_t* field_sel, int n_sel, int F, uint32_t* uidx,
                     int32_t* unique_local_rows, int64_t* inv, int64_t* owner_off, void* workspace,
                     size_t workspace_bytes, dir_stream_t stream);
int dir_shard_dense_inv(const int64_t* feature_index, const float* feature_value,
                        const int32_t* onerow_fields, int n_onerow, int64_t B, int F, int64_t tail_row,
                        int64_t* inv, int* oob_flag, dir_stream_t stream);

/* Exchange over NVLink peer memory, driven from the device (csrc/shard_peer.cu).  No NCCL and
 * no host read on the step: data-dependent counts travel as headers and are read by the kernels, every
 * launch is sized by capacities, so the whole step -- id phase included -- replays from a CUDA graph.
 * Every rank allocates one exchange buffer per parity (consecutive steps alternate) with the layout below
 * and maps its peers' buffers (symmetric memory); the host layer runs a device-side cross-rank barrier
 * where marked.  One-row fields are replicated parameters: their gradient partial sums meet in every rank's
 * buffer and are applied by every rank in rank order.
 *
 *   requester q                                         owner o
 *   dir_shard_ids_push     hdr[q] = (count, base_u), ids[q][0..count)  -->  o's buffer
 *   ---- barrier ----
 *                                                       dir_shard_slots         slot[row * G + q] = epoch | i + 1
 *                                                       dir_shard_gather_send   T[row] -> q's rows[base_u + i],
 *                                                                               w[row] -> q's w[base_u + i]
 *   ---- barrier ----
 *   dir_embed_fm_fwd(rows, w, inv)
 *   dir_embed_bwd_reduce_emit_to   per-distinct-row sums -->  o's g[q][i]
 *   dir_shard_g1_push              first-order sums      -->  o's g1[q][i]
 *   dir_shard_dense_emit           one-row fields        -->  every rank's dense[q][j]
 *   ---- barrier ----
 *                                                       dir_shard_owner_update  ranks' sums added in rank
 *                                                         order (slot tells who else asked), fused update
 *   dir_shard_dense_apply  (every rank)
 *
 * slot: uint32 [n_local_rows * G] per exchange buffer, zero before the first step (the owner never sorts: a
 * requester sends a row at most once, so a cell is written by one thread).  err_flag (device int, zero-initialised): 1 = a
 * requester had more distinct rows than seg_cap / u_cap, 2 = a received local row is out of range; nothing is
 * written out of bounds in either case, the host layer raises.
 */
typedef struct dir_peer_layout {
  int G, rank, K, n_dense;   /* ranks, this rank, embedding size, replicated one-row fields (<= 64)     */
  int64_t seg_cap;           /* rows one requester may ask of one owner in a step                         */
  int64_t u_cap;             /* distinct rows one requester may ask for in total                          */
  /* byte offsets inside every rank's exchange buffer (filled by dir_peer_layout_init)                    */
  int64_t off_hdr;           /* int64 [G][4]              owner <- requester q: (count, base_u, -, -)      */
  int64_t off_ids;           /* int32 [G][seg_cap]        owner <- requesters: local rows asked for        */
  int64_t off_rows;          /* float [u_cap + n_dense][K]  requester <- owners; replicated rows behind   */
  int64_t off_w;             /* float [u_cap + n_dense]     requester <- owners: first-order weights      */
  int64_t off_g;             /* float [G][seg_cap][K]     owner <- requesters: per-row gradient sums       */
  int64_t off_g1;            /* float [G][seg_cap]        owner <- requesters: first-order gradient sums   */
  int64_t off_dense;         /* float [G][n_dense][K+4]   every rank <- every rank: (G[K], g1, touched, 0, 0) */
  int64_t total_bytes;       /* size of the buffer                                                        */
  const int64_t* peer_base;  /* DEVICE int64 [G]: peer-mapped address of each rank's buffer               */
  char* local;               /* DEVICE: this rank's own buffer (256-byte aligned)                         */
} dir_peer_layout;
int dir_peer_layout_init(int G, int rank, int K, int n_dense, int64_t seg_cap, int64_t u_cap,
                         dir_peer_layout* out);
/* slot_epoch: device uint32[2] per exchange buffer, {0, 0} before the first step.  A slot cell is
 * (epoch << 24) | (i + 1) and counts only while its epoch is the current one, so the map is never cleared after a
 * step; dir_shard_ids_push advances the epoch (1..255), dir_shard_slots zeroes the whole map when it wraps. */
int dir_shard_ids_push(const dir_peer_layout* layout, const int32_t* unique_local_rows,
                       const int64_t* owner_off, int64_t n_capacity, int* err_flag, uint32_t* slot_epoch,
                       dir_stream_t stream);
/* zero_counter (device int64, may be NULL) is set to 0: the counter dir_shard_owner_update / dir_shard_dense_apply
 * of the same step then add the rows they update to (no memset node between the step's kernels) */
int dir_shard_slots(const dir_peer_layout* layout, uint32_t* slot, int64_t n_local_rows,
                    const uint32_t* slot_epoch, int* err_flag, int64_t* zero_counter, dir_stream_t stream);
/* dense_table / dense_lin: the replicated one-row fields' rows [n_dense] (copied behind this rank's own
 * exchanged rows so that dir_embed_fm_fwd finds them at u_cap + j); NULL when n_dense == 0.
 * ctas_per_sm (1..8, else 8): the kernel is NVLink-bound; a small grid leaves the SMs to a kernel running next to it */
int dir_shard_gather_send(const dir_peer_layout* layout, const float* table, int64_t row_stride,
                          const float* lin, int64_t lin_stride, const float* dense_table,
                          int64_t dense_row_stride, const float* dense_lin, int ctas_per_sm,
                          dir_stream_t stream);
/* The requester's per-distinct-row gradient sums (the chunking of dir_embed_bwd_reduce_update, rows read from
 * the exchanged rows at uidx[i]): each distinct row's G[K] is stored straight into its owner's buffer over NVLink
 * as soon as its run is summed (no round trip through HBM, the NVLink stores overlap
 * the kernel's gathers); g1 goes to g1_local[u] and is shipped by dir_shard_g1_push.  The sorted list covers
 * the fields field_sel[n_sel] (NULL: all); owner_off[G+1] as written by dir_shard_unique. */
int dir_embed_bwd_reduce_emit_to(const dir_peer_layout* layout, const float* feature_value,
                                 const float* g_first, const float* g_fm, const float* S, const float* u,
                                 const uint32_t* uidx, const int64_t* owner_off, int64_t B, int F,
                                 int64_t n_keys, const int32_t* field_sel, int n_sel, float* g1_local,
                                 void* workspace, size_t workspace_bytes, dir_stream_t stream);
/* The same for bags (models/DeepFM/deepFM.py:53, 77 through a sharded table): the sorted list indexes the nnz
 * ENTRIES (dir_shard_bag_keys); entry_slot / entry_x / emb are what dir_embed_bag_fm_fwd left (run on the exchanged
 * row buffer with bag_index = inv), gradients as in dir_embed_bag_bwd_reduce_update. */
int dir_embed_bag_bwd_reduce_emit_to(const dir_peer_layout* layout, const float* bag_weight,
                                     const uint32_t* entry_slot, const float* entry_x, int64_t nnz, const float* emb,
                                     const float* g_first, const float* g_fm, const float* S, const float* u,
                                     const uint32_t* uidx, const int64_t* owner_off, int64_t B, int F,
                                     int64_t n_keys, float* g1_local, void* workspace, size_t workspace_bytes,
                                     dir_stream_t stream);
int dir_shard_g1_push(const dir_peer_layout* layout, const float* g1_local, const int64_t* owner_off,
                      int64_t n_capacity, dir_stream_t stream);
/* one-row fields: each field's gradient over THIS rank's samples (fixed-order fp64-carried column sums) ->
 * dense[rank][j] of every rank's buffer.  dense_field_offset[F] maps a field to its row of dense_table. */
size_t dir_shard_dense_workspace_bytes(int K);
int dir_shard_dense_emit(const dir_peer_layout* layout, const float* dense_table, int64_t row_stride,
                         const int64_t* feature_index, const float* feature_value,
                         const int64_t* dense_field_offset, const float* g_first, const float* g_fm,
                         const float* S, const float* u, const int32_t* onerow_fields, int64_t B, int F,
                         void* workspace, size_t workspace_bytes, dir_stream_t stream);
/* n_unique_inout += local rows updated.  layout_b / slot_b / slot_epoch_b (NULL, or all three): the batch was
 * exchanged as TWO micro-batches, each through an exchange buffer and slot map of its own (so that the row exchange of
 * the second overlaps the forward of the first); half s of rank q counts as virtual requester s * G + q and the merge
 * runs over both buffers in that order -- still one update per row and batch. */
int dir_shard_owner_update(const dir_peer_layout* layout, const uint32_t* slot, float* table, float* accum,
                           int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride,
                           int64_t n_local_rows, const uint32_t* slot_epoch, int optimizer, float lr,
                           const dir_table_opt* table_opt, const dir_linear_opt* linear_opt,
                           const dir_peer_layout* layout_b,
                           const uint32_t* slot_b, const uint32_t* slot_epoch_b, int64_t* n_unique_inout,
                           dir_stream_t stream);
/* shard_row[j] >= 0 names the row of the sharded table that mirrors replica j (on the rank that owns it), so
 * the sharded table stays a faithful view; n_unique_inout += fields touched (pass it on one rank only) */
int dir_shard_dense_apply(const dir_peer_layout* layout, float* dense_table, float* dense_accum,
                          int64_t row_stride, float* dense_lin, float* dense_lin_accum, int optimizer,
                          float lr, const dir_table_opt* table_opt, const dir_linear_opt* linear_opt,
                          float* shard_table, float* shard_accum,
                          int64_t shard_row_stride, float* shard_lin, float* shard_lin_accum,
                          float* shard_lin_z, int64_t shard_lin_stride, const int64_t* shard_row,
                          const dir_peer_layout* layout_b, int64_t* n_unique_inout, dir_stream_t stream);
/* tf.clip_by_norm of every column's gradient on the row-sharded tables (models/DeepCrossNetwork/DeepCrossNetwork.py:
 * 282-289), one factor per column over its MERGED per-row sums (every rank's requests of a row added as the owner
 * update adds them).  One buffer (one exchange buffer; no second micro-batch), after the grads barrier:
 *   dir_shard_owner_sqnorms         per leading arrival (sum g^2, g1^2) in fp64 -> sq_scratch[G * seg_cap][2], then
 *                                   per column and slice -> norm[rank][F][kClipSlices][2] of EVERY rank; norm_peers
 *                                   is a device array of the G ranks' norm buffers ([G][F][16][2] doubles each)
 *   ---- barrier ----
 *   dir_shard_owner_update_clipped  partials[F][16][2] = sum over q of norm[q] in rank order (the same on every rank),
 *                                   then the owner update with each merged sum scaled by clip / max(||G_f||, clip)
 *                                   (the first-order sums by their own column factor)
 *   dir_shard_dense_apply_clipped   the replicated one-row fields: each a column of one row, clipped by its own sum
 * local_field_offset[F+1]: the first local row of each column on this rank (ascending), then n_local_rows.
 * with_g1: the g1 sums are live (first-order weights trained).  SGD or Adagrad only (tables and replicas). */
int dir_shard_owner_sqnorms(const dir_peer_layout* layout, const uint32_t* slot, const uint32_t* slot_epoch,
                            int64_t n_local_rows, const int64_t* local_field_offset, int F, int with_g1,
                            double* sq_scratch, const uint64_t* norm_peers, dir_stream_t stream);
int dir_shard_owner_update_clipped(const dir_peer_layout* layout, const uint32_t* slot, float* table, float* accum,
                                   int64_t row_stride, float* lin, float* lin_accum, int64_t lin_stride,
                                   int64_t n_local_rows, const uint32_t* slot_epoch, int optimizer, float lr,
                                   const dir_linear_opt* linear_opt, const int64_t* local_field_offset, int F,
                                   const double* norm, double* partials, float clip_norm, int64_t* n_unique_inout,
                                   dir_stream_t stream);
int dir_shard_dense_apply_clipped(const dir_peer_layout* layout, float* dense_table, float* dense_accum,
                                  int64_t row_stride, float* dense_lin, float* dense_lin_accum, int optimizer,
                                  float lr, const dir_linear_opt* linear_opt, float* shard_table, float* shard_accum,
                                  int64_t shard_row_stride, float* shard_lin, float* shard_lin_accum,
                                  float* shard_lin_z, int64_t shard_lin_stride, const int64_t* shard_row,
                                  float clip_norm, int64_t* n_unique_inout, dir_stream_t stream);
/* [TF] tf.train.AdamOptimizer on the row-sharded tables (models/DeepCrossNetwork/train.py:104-124, after
 * clip_by_norm(., 100) of DeepCrossNetwork.py:282-289): Adam._apply_sparse_shared on this rank's shard, then
 * Adam._finish -- dir_rows_apply_adam's step and arithmetic, with the merged sums of every requester as the gradient.
 * After the grads barrier (and, with a clip, dir_shard_owner_sqnorms + its barrier), one sweep of all n_local_rows
 * rows [T(K) | m(K) | v(K)] (row_stride >= 3K): every row decays, a row that some requester asked for adds the
 * requesters' sums merged in rank order (the leader rule and order of dir_shard_owner_update, so the sum is the one
 * the norm pass squared), rows with zero m and v and no gradient are left unwritten.  Run it every step, also when no
 * lookup of this rank's batch survived: TF's Adam steps every row.
 *   norm (NULL = no clip): this step's norm buffer; partials[F][16][2] receives the rank-order combine (as in
 *   dir_shard_owner_update_clipped) and every merged sum is scaled by its column's clip_by_norm factor, looked up
 *   from local_field_offset[F+1]
 *   lin (may be NULL): first-order weights of the rows with a gradient, stepped by linear_opt (required with lin:
 *   Adam does not train first-order weights) with the merged, clipped g1
 *   adam->beta_power: DEVICE float[2], read by the sweep and advanced after it on the same stream
 *   n_unique_inout (may be NULL) += local rows that had a gradient
 * layout->n_dense must be 0 (under Adam every field goes through the exchange); seg_cap < 2^24.  Deterministic: no
 * floating-point atomics, independent of the grid; one buffer (no second micro-batch). */
int dir_shard_owner_apply_adam(const dir_peer_layout* layout, const uint32_t* slot, const uint32_t* slot_epoch,
                               float* table, int64_t row_stride, int64_t n_local_rows, float* lin, float* lin_accum,
                               int64_t lin_stride, const dir_linear_opt* linear_opt,
                               const int64_t* local_field_offset, int F, const double* norm, double* partials,
                               float clip_norm, const dir_adam_opt* adam, int64_t* n_unique_inout,
                               dir_stream_t stream);
/* cfg4-sized tables are filled on the device: value(global row, k) from a counter hash of (seed, row, k) --
 * a sum of four 16-bit uniforms, centred and scaled to standard deviation `sd` (|value| < 3.47 sd) -- so any row
 * can be reproduced on the host without the table (oracle/deepctr_oracle.counter_rows).  Fills
 * table[i, 0:K] for local row i = global row (i * G + rank); rows past n_rows are zero. */
int dir_table_init_counter(float* table, int64_t row_stride, int64_t n_local_rows, int K, int G, int rank,
                           int64_t n_rows, uint64_t seed, float sd, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Multi-hot / weighted bags: every (sample, field) holds a variable-length list of (id, weight) --
 * the capability `myself_input_layer` exists for (models/DeepFM/deepFM.py:53, 77, 363-400; the
 * weighted column of dataset/SequenceTensorFlowDataset/test4.py:50-55, 113-116).  CSR layout:
 *   bag_offsets [B*F + 1] int64, slot s = b*F + f owns entries bag_offsets[s] .. bag_offsets[s+1]
 *   bag_index   [nnz] int64 ids local to the slot's field;  bag_weight [nnz] fp32 or NULL (= 1.0)
 * [TF] _safe_embedding_lookup_sparse: entries with id < 0 or weight <= 0 are pruned, then
 *   DIR_COMBINER_SUM    e = sum w T[id]
 *   DIR_COMBINER_MEAN   e = sum w T[id] / sum w        (embedding_column's default)
 *   DIR_COMBINER_SQRTN  e = sum w T[id] / sqrt(sum w^2)
 * an empty bag is the zero vector; the first-order term always combines with 'sum'
 * (linear_model(sparse_combiner='sum'), deepFM.py:255-263).  emb [B,F,K] is required (the backward
 * reads it); S, first, fm as in dir_embed_fm_fwd.  Per-entry outputs for the backward (all or none):
 *   sort_keys [nnz]  global row, n_rows when pruned  -> dir_embed_bwd_sort(sort_keys, nnz, n_rows, ...)
 *   entry_slot [nnz] slot of the entry;  entry_x [nnz] its effective scale w / norm (0 when pruned)
 * dir_embed_bag_bwd_reduce_update: on the sorted (row, entry) list, per distinct row
 *     G_r = sum_j x_j (g_fm[b] (S[b] - e_s) + u[s]),   g1_r = sum_j w_j g_first[b]
 * then the fused update, exactly as dir_embed_bwd_reduce_update (same determinism, same optimizers).
 */
#define DIR_COMBINER_SUM 0
#define DIR_COMBINER_MEAN 1
#define DIR_COMBINER_SQRTN 2
int dir_embed_bag_fm_fwd(const float* table, int64_t row_stride, const float* lin, int64_t lin_stride,
                         const float* bias, const int64_t* bag_offsets, const int64_t* bag_index,
                         const float* bag_weight, int64_t nnz, const int64_t* field_offset,
                         const int64_t* field_rows, int64_t n_rows, int64_t B, int F, int K,
                         int combiner, float* emb, float* S, float* first, float* fm,
                         uint32_t* sort_keys, uint32_t* entry_slot, float* entry_x, int* oob_flag,
                         dir_stream_t stream);
int dir_embed_bag_bwd_reduce_update(float* table, float* accum, int64_t row_stride, float* lin,
                                    float* lin_accum, int64_t lin_stride, const float* bag_weight,
                                    const uint32_t* entry_slot, const float* entry_x, int64_t nnz,
                                    const float* emb, const float* g_first, const float* g_fm,
                                    const float* S, const float* u, int64_t B, int F, int K,
                                    int64_t n_rows, int optimizer, float lr,
                                    const dir_linear_opt* linear_opt, void* workspace,
                                    size_t workspace_bytes, int64_t* n_unique_out,
                                    dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Column feed -> [B,F] inputs.  The reference's input_fn hands the graph one tensor per column --
 * ids for categorical columns, floats for numeric ones (models/DeepCrossNetwork/train.py:127-156,
 * columns built at :57-100; DeepFM consumes the same dict, models/DeepFM/deepFM.py:159-177).  The
 * host ships those columns only; this widens them, on the device, into the resolved pair the
 * kernels above read:
 *   sparse_index [B, n_sparse] int32 (index_bytes = 4) or int64 (index_bytes = 8)
 *   dense_value  [B, n_dense]  fp32
 *   field_src    [F] int32: j >= 0 -> field f is categorical column j: (id, 1.0)
 *                           j <  0 -> field f is numeric column -j-1, a one-row table: (0, x)
 *   feature_index [B,F] int64, feature_value [B,F] fp32 (outputs)
 */
int dir_expand_features(const void* sparse_index, int index_bytes, const float* dense_value,
                        const int32_t* field_src, int64_t B, int F, int n_sparse, int n_dense,
                        int64_t* feature_index, float* feature_value, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Front end: raw feature -> index, the step in front of the lookup.  The reference declares its categorical columns
 * with tf.feature_column.categorical_column_with_hash_bucket / _with_vocabulary_list
 * (models/DeepCrossNetwork/train.py:57-100, models/ESMM/train.py:65-90) and accepts bucketized_column
 * (models/DeepCrossNetwork/DeepCrossNetwork.py:58); TensorFlow resolves them per batch on the host.  Here a decoded
 * batch's strings travel as ONE byte buffer + offsets[n+1] (string i = bytes[offsets[i] .. offsets[i+1])) and are
 * resolved on the device, one thread per value, straight into a column of feature_index (out_stride = F):
 *   dir_hash_bucket         [TF] string_to_hash_bucket_fast: Fingerprint64(s) mod hash_bucket_size, Fingerprint64 =
 *                           FarmHash farmhashna::Hash64 (published algorithm); integer features are hashed through
 *                           their decimal string, as TF does
 *   dir_vocabulary_lookup   index of s in the vocabulary list, default_value (-1: pruned by the lookup) when absent;
 *                           the table is (sorted fingerprints, list index of each) built on the host with
 *                           dir_fingerprint64_host
 *   dir_bucketize           [TF] Bucketize: number of boundaries <= value (boundaries ascending)
 *   dir_fingerprint64       the raw 64-bit fingerprints (as int64 bits)
 */
uint64_t dir_fingerprint64_host(const uint8_t* bytes_host, int64_t len);
int dir_fingerprint64(const uint8_t* bytes, const int64_t* offsets, int64_t n, int64_t* out, dir_stream_t stream);
int dir_hash_bucket(const uint8_t* bytes, const int64_t* offsets, int64_t n, int64_t num_buckets, int64_t* out,
                    int64_t out_stride, dir_stream_t stream);
int dir_vocabulary_lookup(const uint8_t* bytes, const int64_t* offsets, int64_t n,
                          const uint64_t* vocab_fingerprints, const int64_t* vocab_index, int64_t n_vocab,
                          int64_t default_value, int64_t* out, int64_t out_stride, dir_stream_t stream);
int dir_bucketize(const float* values, int64_t n, int64_t value_stride, const float* boundaries, int n_boundaries,
                  int64_t* out, int64_t out_stride, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * tf.feature_column.input_layer in the reference's own DCN convention
 * (models/DeepCrossNetwork/DeepCrossNetwork.py:126 over the columns of train.py:88-100): all dense
 * columns side by side, sorted by column name -- numeric columns 1-wide, indicator columns one-hot,
 * embedding columns K-wide (the rows dir_embed_fm_fwd gathered).  The host lays the d output columns
 * out in three int32[d] maps:
 *   col_kind 0 numeric    col_src = column of numeric[B, n_numeric]
 *            1 indicator  col_src = column of indicator_ids[B, n_indicator] (int64), col_arg = class:
 *                         1.0 where the id equals the class, else 0.0 (ids < 0 / out of vocabulary: zeros)
 *            2 embedding  col_src = component of emb[B, emb_width]
 * dir_input_layer_bwd returns the embedding columns' slice of dL/dx0 as u[B, emb_width], the upstream
 * gradient of dir_embed_bwd_reduce_update; emb_col[emb_width] = the x0 column of each component (-1: unused).
 */
int dir_input_layer_fwd(const float* numeric, int n_numeric, const int64_t* indicator_ids,
                        int n_indicator, const float* emb, int emb_width, const int32_t* col_kind,
                        const int32_t* col_src, const int32_t* col_arg, int64_t B, int d, float* x0,
                        dir_stream_t stream);
int dir_input_layer_bwd(const float* dx0, const int32_t* emb_col, int64_t B, int d, int emb_width,
                        float* u, dir_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * DCN cross network, all L layers in one pass.  Replaces _cross_architecture / _cross_op
 * (models/DeepCrossNetwork/DeepCrossNetwork.py:336-367): x_{l+1} = (x0 * (x_l . w_l) + b_l) + x_l.
 *   x0 [B,d], cross_w / cross_b [L,d] (names as DeepCrossNetwork.py:329-332), xL [B,d],
 *   s [B,L] or NULL: per-sample scalars saved for the backward (s[b,l] = x0[b] . w_l; the
 *   kernels use x_l = x0 * c_l + sum_{j<l} b_j, so x_l . w_l follows from these).   d <= 1024.
 * Evaluated as x_L = x0 * c_L + sum_l b_l with c_L from a scalar recurrence: equal to the
 * reference's layer-by-layer ((x0*s)+b)+x up to rounding (a few ulp of the largest term).
 */
int dir_cross_fwd(const float* x0, const float* cross_w, const float* cross_b, int64_t B, int d,
                  int L, float* xL, float* s, dir_stream_t stream);

/* Backward of the cross stack (TF autodiff behind compute_gradients, DeepCrossNetwork.py:283).
 *   dy [B,d] -> dx0 [B,d], dw [L,d], db [L,d]; s [B,L] as written by dir_cross_fwd, or NULL
 *   (recomputed; always recomputed when L > 8).
 * dw / db are reduced in a fixed order (per-CTA partials in `workspace`, then one combine).
 */
size_t dir_cross_bwd_workspace_bytes(int64_t B, int d, int L);
int dir_cross_bwd(const float* x0, const float* cross_w, const float* cross_b, const float* dy,
                  const float* s, int64_t B, int d, int L, float* dx0, float* dw, float* db,
                  void* workspace, size_t workspace_bytes, dir_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DIR_B200_H */
