/* agcf.h -- C-ABI of libagcf.so: the B200 (sm_100a) graph-CF hot path.
 *
 * The reference (CoderWZW/ARLib) has NO FFI: its hot path is Python calling
 * PyTorch.  These entry points are what a binding for that path would bind; the
 * Python surface in arlib_b200/ (drop-in recommender.* / util.*) sits strictly on
 * top of them via ctypes.  Each function cites the reference code it replaces
 * (file:line relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into memory owned by the caller (PyTorch
 *     in this repo) unless the name ends in _host; the library allocates nothing
 *     and keeps no global state; workspace sizes come from *_ws_bytes queries;
 *   - every call takes an explicit stream (a cudaStream_t passed as void*), only
 *     enqueues work on it and is capturable in a CUDA graph;
 *   - return value: 0 = ok, <0 = AGCF_E* below; nothing throws;
 *   - fp32 everywhere, int32 indices; tables are row-major [rows, d], 16-byte
 *     aligned, d in {8, 16, 32, 64, 128, 256};
 *   - a "node" id is a row of the stacked table [users; items] (N = U + I); item
 *     ids handed to the loss / sampler / eval calls are item-local (0..I-1).
 */
#ifndef AGCF_H_
#define AGCF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGCF_OK            0
#define AGCF_EINVAL       (-1)  /* bad argument (null pointer, size, alignment)      */
#define AGCF_EUNSUPPORTED (-2)  /* shape outside the compiled set (d, K, B limits)   */
#define AGCF_ECUDA        (-3)  /* a CUDA runtime call failed; see agcf_last_cuda_error */
#define AGCF_EWORKSPACE   (-4)  /* workspace too small                               */

typedef void* agcf_stream_t;    /* cudaStream_t */
#define AGCF_MAX_PEERS 8        /* GPUs of one NVSwitch box */
#define AGCF_MAX_ACC_TERMS 8    /* tables of agcf_spmm_args.acc_terms */

int         agcf_abi_version(void);
const char* agcf_strerror(int code);
int         agcf_last_cuda_error(void);   /* cudaError_t of the last AGCF_ECUDA on this thread */
const char* agcf_last_cuda_error_where(void);  /* its message and the library source line that saw it */
int         agcf_device_sm_count(void);

/* ------------------------------------------------------------------ adjacency
 * val[p] = fl(fl(d_row[i] * w[p]) * d_col[col[p]])  for p in row i, no FMA
 * contraction -- the association of (D.A).D in scipy.
 * Replaces: util/DataLoader.py:73-87 (normalize_graph_mat) and
 * recommender/LightGCN.py:212-215 (_init_uiAdj); d_row/d_col are computed on the
 * host with the reference's own numpy expression (bit-exactness, DESIGN.md). */
int agcf_norm_adj_csr(const int32_t* rowptr, const int32_t* col, const float* w,
                      const float* d_row, const float* d_col, float* val,
                      int32_t n_rows, int64_t nnz, agcf_stream_t stream);

/* row -> COO expansion helper: row_of[p] = i for p in [rowptr[i], rowptr[i+1]) */
int agcf_csr_expand_rows(const int32_t* rowptr, int32_t* row_of, int32_t n_rows, int64_t nnz,
                         agcf_stream_t stream);

/* ---------------------------------------------------------------- propagation
 * One normalized-adjacency propagation Y = A X with a fused epilogue, CSR fp32.
 *   t[i,:]       = sum_p val[p] * X[col[p],:]  (+ addend[i,:] if addend)
 *   if noise:      t[i,:] += sign(t[i,:]) * noise[i,:]/max(||noise[i,:]||,1e-12) * eps
 *   if Y:          Y[i,:] = t[i,:]
 *   if acc_out:    acc_out[i,:] = ((acc_in ? acc_in[i,:] : 0) + t[i,:]) / acc_div
 * Work plan (built once per graph by the caller; arlib_b200/graph.py is the reference builder): row i
 * with deg non-zeros is cut into nseg = max(1, ceil(deg / S)) segments, S <= 64 recommended.  Work item
 * v is four int32 {start, len, row, k | nseg << 16}: entries col/val[start .. start+len) of row `row`,
 * segment k of nseg; items sorted by len descending; n_vrows items (a row without non-zeros is one
 * item of len 0).  Rows with nseg > 1 own nseg consecutive slots of `partial` ([slots][d] floats) starting
 * at vpart[v] (same value for all items of the row); `tickets` ([slots] int32) must be zero on entry
 * and is zero again on exit.  Partials are added in segment order by the segment that arrives last:
 * results are deterministic.  Launches that share partial/tickets must be stream-ordered.
 * Rows absent from the plan are not touched (multi-GPU: a rank's plan holds its own rows only).
 * row_mask / col_mask (nullable bitmaps, bit k of word k/32): only rows whose bit is set are computed
 * and written; rows of X whose bit is clear are known to be all-zero and are not gathered (the last
 * forward layer only needs the batch's rows, the first backward layer only sees the batch's gradient
 * rows).
 * Multi-GPU (row-partitioned tables): peer_Y_host / peer_acc_host are HOST arrays of n_peers device
 * pointers to the other ranks' copies of Y / acc_out (peer-mapped over NVLink): the epilogue stores
 * every computed row there too -- the per-layer all-gather is fused into the SpMM and overlaps it
 * row by row.  Visibility on the peers needs a barrier after.
 * mc_Y / mc_acc (nullable): NVSwitch MULTICAST addresses of Y / acc_out (a multicast object bound
 * to every rank's copy): the epilogue then issues ONE multimem.st per 16 bytes and the switch
 * replicates it to all GPUs -- a rank's NVLink egress per layer is its rows once, not once per peer;
 * the peer arrays are ignored when these are given.
 * Forward AND backward of the encoder: A is symmetric so A^T = A.
 * Replaces: torch.sparse.mm + stack + mean in recommender/LightGCN.py:230-240,
 * the noise lines of recommender/SimGCL.py:202-206 / XSimGCL.py:211-215, and the
 * autograd of those (transposed SpMM + mean backward). */
int agcf_spmm_csr_f32(const int32_t* vrows, const int32_t* vpart, int32_t n_vrows,
                      const int32_t* col, const float* val, float* partial, int32_t* tickets,
                      const float* X, float* Y,
                      const float* addend,
                      const float* acc_in, float* acc_out, float acc_div,
                      const float* noise, float eps,
                      const uint32_t* row_mask, const uint32_t* col_mask,
                      void* const* peer_Y_host, void* const* peer_acc_host, int32_t n_peers,
                      void* mc_Y, void* mc_acc,
                      int32_t d, agcf_stream_t stream);

/* The same launch with every argument in one plain-C struct (zero-initialise, then fill), plus what the fused
 * training step adds:
 *   n_vrows_dev   nullable device int32: the item count of a per-batch work list (agcf_spmm_batch_worklists);
 *                 the grid is sized for n_vrows (the list's capacity) and items >= *n_vrows_dev are skipped, so the
 *                 launch is capturable in a CUDA graph although the count changes from batch to batch;
 *   adam_*        fused optimizer: the row's o = (acc_in + t) / acc_div is the gradient of torch.optim.Adam's update
 *                 of adam_p / adam_m / adam_v ([rows, d] tables like Y), coefficients from agcf_adam_coefs;
 *                 acc_out may then be null (the gradient table is never written).  Same bits as agcf_adam_step_f32;
 *   zero_acc_in   != 0: rows of acc_in that were non-zero are set to zero after they were read (acc_in is the batch
 *                 gradient G, non-zero on <= 3B rows: replaces agcf_zero_rows); acc_in must not be X;
 *   noise_main    != 0: perturb the main outputs with the Philox stream below (instead of a `noise` table);
 *   aux_Y[q]      q < 2, nullable: extra outputs aux_Y[q][i,:] = t[i,:] perturbed with their OWN noise (table aux_noise[q]
 *                 if given, else Philox stream aux_stream[q]) while Y / acc_out stay clean (or take the main noise):
 *                 SimGCL's clean pass and its two perturbed passes share A E0, one launch writes all three tables;
 *   noise_seed    != 0: the U[0,1) noise of the SimGCL / XSimGCL perturbation is drawn IN the
 *                 epilogue -- Philox4x32-10, key = noise_seed, counter = (float4 slot of the element,
 *                 *noise_step << 32 | noise_stream) -- instead of read from an [rows, d] table; noise_stream / aux_stream tell
 *                 layers / passes apart, noise_step (nullable device int32) is the training-step counter, so a
 *                 replayed CUDA graph perturbs every step differently;
 *   sched         nullable device int32[2], zero on entry and zero again on exit: the launch then runs PERSISTENT CTAs
 *                 (148 x resident CTAs per SM) that take blocks of work items from this counter in plan order instead
 *                 of one CTA per block -- no CTA turnover gaps and no tail of idle SMs; launches sharing it must be
 *                 stream-ordered;
 *   flags         reserved, must be 0;
 *   mask_bits     number of bits of row_mask / col_mask (= rows of X), or 0 if unknown: the narrow-row (d <= 16) variant
 *                 of the column-masked launch copies the bitmap into shared memory when it is given and fits;
 *   acc_terms     n_acc_terms (0 .. AGCF_MAX_ACC_TERMS) [rows, d] tables that take the place of acc_in (which must then be
 *                 null): acc_out = (((acc_terms[0] + acc_terms[1]) + ...) + t) / acc_div, plain fp32 adds in that order.
 *                 The last propagation layer forms the layer sum this way at the rows it computes, so the earlier
 *                 layers need only write their Y.  Not with noise, col_mask or adam.
 *   addend_mask   nullable bitmap over rows (like row_mask): rows of addend / acc_in whose bit is clear are known to be
 *                 exactly zero and are not loaded; +0.0f is added in their place.  With zero_acc_in, every row whose bit
 *                 is set is set to +0.0f (instead of the rows that read non-zero).  The backward layers of the training
 *                 step pass the batch's node bitmap: the gradient G is non-zero only at the batch's rows.  Not with
 *                 acc_terms or noise.
 * A launch with col_mask (and no noise) runs the sparse variant (ballot over the live entries of a chunk, only
 * those are gathered): identical results. */
typedef struct agcf_spmm_args {
  const int32_t* vrows; const int32_t* vpart; int32_t n_vrows; const int32_t* n_vrows_dev;
  const int32_t* col; const float* val; float* partial; int32_t* tickets;
  const float* X; float* Y; const float* addend;
  const float* acc_in; float* acc_out; float acc_div;
  const float* noise; float eps;
  uint64_t noise_seed; uint32_t noise_stream; const int32_t* noise_step; int32_t noise_main;
  float* aux_Y[2]; const float* aux_noise[2]; uint32_t aux_stream[2];
  const uint32_t* row_mask; const uint32_t* col_mask;
  void* const* peer_Y_host; void* const* peer_acc_host; int32_t n_peers;
  void* mc_Y; void* mc_acc;
  float* adam_p; float* adam_m; float* adam_v; const float* adam_coefs;
  float adam_beta1; float adam_beta2; float adam_eps;
  int32_t zero_acc_in;
  int32_t* sched;
  int32_t d;
  int32_t flags;
  int32_t mask_bits;
  const float* acc_terms[8];
  int32_t n_acc_terms;
  const uint32_t* addend_mask;
} agcf_spmm_args;
int agcf_spmm_csr_f32_ex(const agcf_spmm_args* args, agcf_stream_t stream);

/* Per-batch work lists for the LAST forward layer (the loss reads F only at the batch's <= 3B nodes): for every
 * batch b < n_batches, from its sorted distinct nodes seg_node[b*seg_stride ..][0 .. n_seg[b]) (agcf_bpr_group_batches),
 * write the batch's own SpMM plan: wl_vrows[b][w] = {start, len, row, k | nseg << 16} (rows with more than split_above
 * non-zeros cut into segments of `segment`), wl_vpart[b][w] = the row's first partial slot (numbered per batch),
 * wl_count[b] = number of items (<= cap, the per-batch capacity of both arrays).  Nodes outside [row0, row1) are
 * skipped (multi-GPU: another rank's rows).  Pass wl_vrows + b*cap*4 / wl_vpart + b*cap / wl_count + b to
 * agcf_spmm_csr_f32_ex with n_vrows = cap; partial / tickets need cap slots. */
int agcf_spmm_batch_worklists(const int32_t* seg_node, const int32_t* n_seg, int32_t n_batches, int32_t seg_stride,
                              const int32_t* rowptr, int32_t row0, int32_t row1, int32_t split_above, int32_t segment,
                              int32_t* wl_vrows, int32_t* wl_vpart, int32_t* wl_count, int32_t cap,
                              agcf_stream_t stream);

/* gval[p] (+)= <H[i,:], E[col[p],:]> for p in row i (accumulate != 0 adds).
 * Replaces: autograd of torch.sparse.mm w.r.t. the sparse operand, restricted to
 * the stored pattern -- attack/White/PGA.py:97-117, recommender/LightGCN.py:40-43,58-59. */
int agcf_sddmm_csr_f32(const int32_t* rowptr, const int32_t* col,
                       const float* H, const float* E, float* gval, int32_t accumulate,
                       const int32_t* row_order, int32_t n_rows, int32_t d, agcf_stream_t stream);

/* pack [user_emb; item_emb] into one [N,d] table (torch.cat of LightGCN.py:231)
 * and the inverse split-add used by its backward. */
int agcf_concat_rows_f32(const float* a, int64_t n_a, const float* b, int64_t n_b,
                         float* out, int32_t d, agcf_stream_t stream);

/* -------------------------------------------------------------------- sampler
 * One epoch of BPR triples on device (Philox4x32-10, counter-based):
 *   position t of the epoch takes edge perm(t) of (e_user, e_item) where perm is a
 *   keyed bijection of [0,E) (every edge exactly once per epoch), and a negative
 *   item drawn uniformly from [0,I) and re-drawn while it is in the user's
 *   rejection set rej_items[rej_rowptr[u] .. rej_rowptr[u+1]) (sorted ascending).
 * Replaces: util/sampler.py:4-30 (next_batch_pairwise): shuffle + per-row
 * rejection sampling; batches are consecutive slices [b*B, min((b+1)*B, E)). */
int agcf_bpr_sample_epoch(const int32_t* e_user, const int32_t* e_item, int32_t n_edges,
                          const int32_t* rej_rowptr, const int32_t* rej_items, int32_t n_items,
                          uint64_t seed, uint64_t epoch,
                          int32_t* out_u, int32_t* out_i, int32_t* out_j, agcf_stream_t stream);

/* ----------------------------------------------------------------------- loss
 * Group the 3*B node occurrences of each batch by node (atomic-free scatter
 * plan).  For batch b (triples [b*B, min((b+1)*B,T)) ), nb = its triple count:
 *   occ   [b*3B + k]   k < 3*nb : occurrence ids role*nb + t, sorted by (node, id);
 *                                 role 0 = user, 1 = positive, 2 = negative
 *   seg_off[b*(3B+1)+s] s <= n_seg: start of segment s in occ (one segment = one node)
 *   seg_node[b*3B + s] : the node (users 0..U-1, items U..U+I-1)
 *   n_seg[b]
 *   node_mask[b*ceil(n_nodes/32) + w] (nullable): bitmap of the batch's nodes -- the
 *                                 row / column mask of the batch-sparse SpMM layers
 * 3*B must be <= 16384. One CTA per batch; all batches of an epoch in one call. */
int agcf_bpr_group_batches(const int32_t* u, const int32_t* i, const int32_t* j,
                           int32_t n_triples, int32_t batch, int32_t n_users,
                           int32_t* occ, int32_t* seg_off, int32_t* seg_node, int32_t* n_seg,
                           int32_t n_nodes, uint32_t* node_mask, agcf_stream_t stream);

/* Fused gather - score - BPR - L2 forward for one batch of nb triples on the
 * propagated table F [N,d]:
 *   x_t = <F[u],F[U+i]> - <F[u],F[U+j]>
 *   out[0] = loss = mean_t -log(1e-7 + sigmoid(x_t)) + reg*(||F[u_.]||_F + ||F[U+i_.]||_F)
 *   out[1] = bpr term, out[2] = ||F[u_.]||_F, out[3] = ||F[U+i_.]||_F
 *   coef[t] = d loss / d x_t
 * ws: agcf_bpr_ws_bytes(nb) bytes.  Deterministic (fixed-order reductions).
 * Replaces: util/loss.py:5-9 (bpr_loss), :25-29 (l2_reg_loss) and the three
 * index gathers of recommender/LightGCN.py:51-54. */
int64_t agcf_bpr_ws_bytes(int32_t nb);
int agcf_bpr_forward(const float* F, const int32_t* u, const int32_t* i, const int32_t* j,
                     int32_t nb, int32_t n_users, int32_t d, float reg,
                     float* out4, float* coef, void* ws, agcf_stream_t stream);

/* The same forward when the tables are COLUMN-sharded over `world` GPUs (d here is the local slice
 * width): agcf_bpr_partial computes each triple's share {<u,i>, <u,j>, |u|^2, |i|^2} on this rank's
 * slice and stores it into slot `rank` of the exchange buffer of EVERY rank (xchg_all_host: HOST array
 * of `world` device pointers, own buffer included, peer-mapped over NVLink; agcf_bpr_xchg_bytes(cap)
 * bytes each, cap >= nb, ZERO before the first use).  agcf_bpr_finish sums the shares in rank order --
 * the same bits on every rank -- and produces out4 / coef exactly like agcf_bpr_forward.
 * No barrier between the two calls: every value travels as one 64-bit word {*xchg_ctr + 1 : 32 | float : 32}
 * (a single-copy-atomic store), and agcf_bpr_finish spins until the words it needs carry the current
 * stamp (it gives up with a NaN loss after 4 s if a rank never shows up).  xchg_ctr is a device int32
 * EXCHANGE COUNTER private to the buffer: both calls read it, the buffer is double-buffered on its
 * parity, and agcf_bpr_finish advances it by one when its last block retires -- so no stamp is ever
 * used twice, whatever the caller does to its optimizer step (warm-up launches before a CUDA-graph
 * capture, restores).  Every rank must issue the same sequence of partial / finish pairs.  NULL = a
 * single use of a zeroed buffer.  This is the ONLY exchange of a d-sharded training step: 32*nb
 * bytes per peer. */
int64_t agcf_bpr_xchg_bytes(int32_t cap);
int agcf_bpr_partial(const float* F, const int32_t* u, const int32_t* i, const int32_t* j,
                     int32_t nb, int32_t n_users, int32_t d, int32_t rank, int32_t cap,
                     const int32_t* xchg_ctr, void* const* xchg_all_host, int32_t world,
                     agcf_stream_t stream);
int agcf_bpr_finish(const void* xchg, int32_t world, int32_t cap, int32_t nb, float reg,
                    int32_t* xchg_ctr, float* out4, float* coef, void* ws, agcf_stream_t stream);

/* Backward of the above into the dense gradient of F, atomic-free: one
 * half-warp per node segment sums that node's contributions in occurrence order
 *   user : coef*(F[i]-F[j]) + reg*F[u]/||F[u_.]||     positive: coef*F[u] + reg*F[i]/||F[i_.]||
 *   negative: -coef*F[u]
 * and writes G[node,:] = scale * sum (scale folds the 1/(L+1) of the layer mean
 * and any upstream grad).  Rows of G not named by a segment are NOT touched (the
 * caller zeroes G, or passes touched rows to agcf_zero_rows afterwards).
 * Replaces: autograd of util/loss.py:5-9,25-29 + index_put_(accumulate) backward. */
int agcf_bpr_backward(const float* F, const int32_t* u, const int32_t* i, const int32_t* j,
                      int32_t nb, int32_t n_users, int32_t d, float reg, float scale,
                      const float* out4, const float* coef,
                      const int32_t* occ, const int32_t* seg_off, const int32_t* seg_node,
                      const int32_t* n_seg, float* G, agcf_stream_t stream);

/* The id lists of the contrastive loss of SimGCL / XSimGCL -- torch.unique of the batch's users and of its
 * POSITIVE items (recommender/SimGCL.py:213-214, XSimGCL.py:40-41) -- for every batch, from the grouping above:
 * cl_users[b*batch ..] / cl_items[b*batch ..] = sorted TABLE rows (items: n_users + item), n_cl[2b], n_cl[2b+1] =
 * their counts.  (The reference passes the ids through float32; exact below 2^24.) */
int agcf_bpr_cl_ids(const int32_t* occ, const int32_t* seg_off, const int32_t* seg_node, const int32_t* n_seg,
                    int32_t n_triples, int32_t batch, int32_t n_users,
                    int32_t* cl_users, int32_t* cl_items, int32_t* n_cl, agcf_stream_t stream);

/* G[seg_node[s],:] = 0 for s < *n_seg (undo of agcf_bpr_backward's writes) */
int agcf_zero_rows(const int32_t* seg_node, const int32_t* n_seg, int32_t max_seg,
                   float* G, int32_t d, agcf_stream_t stream);

/* ---------------------------------------------------------------- contrastive loss
 * InfoNCE between two views of the same n rows (util/loss.py:42-49; callers recommender/SimGCL.py:212-219,
 * XSimGCL.py:39-44 with the batch's unique users / positive items, n <= batch size):
 *   h = v / max(||v||, 1e-12) per row;  S = h1 h2^T / temperature;
 *   loss[0] = mean_r -log( exp(S_rr) / sum_c exp(S_rc) )        (no max-subtraction, like the reference)
 * view1 / view2 are [n, d] matrices, or -- with `rows` (n device int32 ids) -- TABLES whose rows rows[r] form the
 * views (the gather of `emb[idx]` fused into the normalisation).  n_dev (nullable device int32): the actual row
 * count, <= n; grids and the workspace are sized for n, so a launch sequence captured in a CUDA graph serves
 * batches whose number of unique ids differs.
 * The n x n logits never reach memory (tiles in registers / shared memory, fp32 CUDA cores: a TF32 product would
 * put ~1e-2 relative error on exp(S)).  `ws` (agcf_infonce_ws_bytes(n, d) bytes) receives the normalized views, the
 * row sums and scratch; agcf_infonce_backward takes the SAME workspace, untouched since the forward call (same n,
 * n_dev), and produces scale * grad_loss[0] * d loss / d view (grad_loss nullable = 1): grad_viewK is [n, d], or
 * -- with rowsK -- a table whose rows rowsK[r] receive the rows of the gradient (ids must be unique);
 * accumulateK != 0 adds to what is there.  Either gradient may be null.
 * Deterministic (partials combined in a fixed order).  d in {8, 16, 32, 64, 128, 256}. */
int64_t agcf_infonce_ws_bytes(int32_t n, int32_t d);
int agcf_infonce_forward(const float* view1, const float* view2, const int32_t* rows, int32_t n, const int32_t* n_dev,
                         int32_t d, float temperature, float* loss, void* ws, int64_t ws_bytes, agcf_stream_t stream);
int agcf_infonce_backward(int32_t n, const int32_t* n_dev, int32_t d, float temperature, const float* grad_loss,
                          float scale, void* ws, int64_t ws_bytes,
                          float* grad_view1, const int32_t* rows1, int32_t accumulate1,
                          float* grad_view2, const int32_t* rows2, int32_t accumulate2, agcf_stream_t stream);

/* ------------------------------------------------------------------ NGCF layer
 * The dense half of an NGCF layer around the propagation P = A E (agcf_spmm_csr_f32):
 *   forward   Enext = leaky_relu([P + E | P * E] W, 0.01), W = [W1 ; W2] ([2d, d] row-major, out = in @ W);
 *             if acc_out: acc_out = ((acc_in ? acc_in : 0) + Enext) / acc_div   (running layer mean)
 *   backward  dZ = dOut * (Enext > 0 ? 1 : 0.01);  [dA | dB] = dZ W^T  (WT = W transposed, [d, 2d]);
 *             dP = dA + dB * E;  dEdir = dA + dB * P;  dW_partial[b] = this CTA's share of [P + E | P * E]^T dZ
 *             ([n_partials][2d*d]; d <= 64: the launch runs n_partials persistent CTAs, d = 128 and 256: the
 *             weight gradient is split into n_partials row slices, dW_partial[b] the share of slice b);
 *             the gradient of E is then A dP + dEdir (next agcf_spmm_csr_f32, addend = dEdir);
 *   reduce    dW = sum_b dW_partial[b] in b order (deterministic).
 * Uses A (E W1) = (A E) W1: one propagation per layer where the reference runs two.  d in {8, 16, 32, 64, 128, 256}.
 * Replaces: the loop body of NGCF_Encoder.forward (recommender/NGCF.py:197-212: torch.mm x 2,
 * torch.sparse.mm x 2, leaky_relu, the element-wise product / sums) and its autograd. */
int agcf_ngcf_dense_forward(const float* P, const float* E, const float* W, float* Enext,
                            const float* acc_in, float* acc_out, float acc_div,
                            int32_t n_rows, int32_t d, agcf_stream_t stream);
int agcf_ngcf_dense_backward(const float* dOut, const float* Enext, const float* P, const float* E,
                             const float* WT, float* dP, float* dEdir, float* dW_partial,
                             int32_t n_partials, int32_t n_rows, int32_t d, agcf_stream_t stream);
int agcf_ngcf_reduce_wgrad(const float* dW_partial, int32_t n_partials, float* dW, int32_t d,
                           agcf_stream_t stream);
/* Row-partitioned variants (multi-GPU, one rank's rows [r0, r1) of the row-partitioned layout): the same
 * computation, and every stored row also goes to the other ranks' copies, so that the next propagation can gather
 * it there.  Every row pointer (P, E, Enext, acc_*, dOut, dP, dEdir) points at row r0 of its table and n_rows =
 * r1 - r0; the peer pointers are offset the same way, so a row sits at the same index everywhere.
 *   peer_*_host  HOST arrays of n_peers device pointers to the other ranks' copies (peer-mapped over NVLink), each
 *                nullable: forward -- of Enext and of acc_out (the finished layer mean); backward -- of dP;
 *                reduce -- of dW (this rank's slot of every rank's symmetric [P, 2d*d] slot buffer);
 *   mc_*         nullable NVSwitch multicast addresses of the same ranges: one multimem.st reaches every copy and
 *                the peer arrays are ignored for that output.
 * The local outputs are bit-equal to the plain entry points'.  Visibility on the peers needs a barrier after.
 * Summing the P slots in rank order (agcf_ngcf_reduce_wgrad with n_partials = P) gives every rank the same dW. */
int agcf_ngcf_dense_forward_peers(const float* P, const float* E, const float* W, float* Enext,
                                  const float* acc_in, float* acc_out, float acc_div,
                                  int32_t n_rows, int32_t d,
                                  void* const* peer_Enext_host, void* const* peer_acc_host, int32_t n_peers,
                                  void* mc_Enext, void* mc_acc, agcf_stream_t stream);
int agcf_ngcf_dense_backward_peers(const float* dOut, const float* Enext, const float* P, const float* E,
                                   const float* WT, float* dP, float* dEdir, float* dW_partial,
                                   int32_t n_partials, int32_t n_rows, int32_t d,
                                   void* const* peer_dP_host, int32_t n_peers, void* mc_dP, agcf_stream_t stream);
int agcf_ngcf_reduce_wgrad_peers(const float* dW_partial, int32_t n_partials, float* dW, int32_t d,
                                 void* const* peer_dW_host, int32_t n_peers, void* mc_dW, agcf_stream_t stream);

/* ------------------------------------------------------------------ optimizer
 * torch.optim.Adam step (defaults: amsgrad=False, weight_decay=0, maximize=False)
 * over n contiguous fp32 elements:
 *   m += (g-m)*(1-b1); v = v*b2 + (1-b2)*g*g;
 *   p -= (lr/(1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * t = *step_dev + 1 if step_dev (device int32, NOT modified) else step (>=1).
 * peer_p_host (nullable): the updated parameters are also stored at the same offsets
 * of n_peers peer-mapped copies (multi-GPU: owner updates its rows everywhere), or -- when mc_p, the
 * multicast address of the same range, is given -- with one multimem.st that reaches every copy.
 * Replaces: optimizer.step() of recommender/LightGCN.py:32-35,64 when the caller
 * did not hand in its own optimizer. */
int agcf_adam_step_f32(float* p, const float* g, float* m, float* v, int64_t n,
                       float lr, float beta1, float beta2, float eps,
                       int32_t step, const int32_t* step_dev,
                       void* const* peer_p_host, int32_t n_peers, void* mc_p, agcf_stream_t stream);
int agcf_increment_i32(int32_t* counter, agcf_stream_t stream);

/* Hand-off inside a group of ranks that store into each other's tables (the column group of the grid layout: the
 * ranks that share a column slice), in place of an all-rank barrier launch.  flags: this rank's AGCF_MAX_PEERS int32
 * flag words (peer-mapped, ZERO before the first use, slot s written only by group member s); peer_flags_host: HOST
 * array of the n_peers partners' flag words (n_peers = group size - 1); my_slot: this rank's position in the group.
 * stamp = *stamp_dev + 1 is stored with a system-scope release into slot my_slot of every partner, then the kernel
 * waits (acquire) until every partner's slot of `flags` carries it, and sets *stamp_dev = stamp.  stamp_dev is a
 * device int32 private to the group and never restored, so no stamp is used twice; every member must issue the same
 * sequence of hand-offs.  Stores a kernel made before the hand-off (peer_Y / peer_acc / peer_p) are visible to every
 * partner's kernels after it.  A partner missing for 4 s sets *err = 1 (never cleared here) and the wait gives up. */
int agcf_group_handoff(int32_t* flags, void* const* peer_flags_host, int32_t n_peers, int32_t my_slot,
                       int32_t* stamp_dev, int32_t* err, agcf_stream_t stream);
/* if (increment) *step_dev += 1;  t = *step_dev + 1;  coefs = {lr / (1 - b1^t), sqrt(1 - b2^t)} -- the two
 * step-dependent scalars of the Adam update, for the optimizer fused into the last backward SpMM. */
int agcf_adam_coefs(int32_t* step_dev, int32_t increment, float lr, float beta1, float beta2, float* coefs,
                    agcf_stream_t stream);

/* ----------------------------------------------------------------- evaluation
 * Full-rank scoring + masked top-K for n_u users (rows user_rows[0..n_u) of Uemb,
 * or rows 0..n_u-1 if user_rows is null) against items [0,n_items) of Iemb:
 *   s[u,i] = <Uemb[u,:], Iemb[i,:]>  (fp32, k ascending, fused multiply-add);
 *   s[u, mask_items[mask_rowptr[u]..]] = -1e9;  top-K by the reference's rule
 *   (util/algorithm.py:155-167 incl. its tie rule, SURVEY.md 8a-11), output
 *   sorted by (score desc, item asc).  item_offset is added to output ids (item
 *   shards).  Stage 1 is a TF32 tcgen05 GEMM (impl=1) or an fp32 CUDA-core GEMM
 *   (impl=0) that only emits per-32-item group maxima; stage 2 selects candidate
 *   groups with a rigorous error margin; stage 3 re-scores candidates in exact
 *   fp32 -- so the result does not depend on impl.
 *   impl | AGCF_TOPK_KEEP_MASK_BITS: the caller guarantees that the workspace still holds the train-item mask bits of
 *   the PREVIOUS call on it with the same user_rows / n_u / n_items / d / item_offset / mask arrays (test() masks the
 *   same training items in every evaluation): stage 0 -- a memset of n_u * ceil(n_items / 32) words and the bit scatter,
 *   ~6 % of an evaluation at the Gowalla shape -- is skipped.  Nothing else in the workspace survives a call.
 * Replaces: recommender/LightGCN.py:86-90 (predict) + :148-156 (test loop) +
 * util/algorithm.py:155-167 (find_k_largest). */
#define AGCF_TOPK_KEEP_MASK_BITS 0x100
int64_t agcf_score_topk_ws_bytes(int32_t n_u, int32_t n_items, int32_t d, int32_t K);
int agcf_score_topk(const float* Uemb, const int32_t* user_rows, int32_t n_u,
                    const float* Iemb, int32_t n_items, int32_t d,
                    const int32_t* mask_rowptr, const int32_t* mask_items,
                    int32_t K, int32_t item_offset, int32_t impl,
                    float* out_val, int32_t* out_idx, int32_t* out_flags,
                    void* ws, int64_t ws_bytes, agcf_stream_t stream);

/* Stages 0 + 1 of agcf_score_topk alone: gmax_out[u][g] (nullable; [n_u][ceil(n_items/32)] floats) = the maximum
 * of the MASKED scores of user u over the 32 items of group g -- impl 1: the tcgen05 TF32 GEMM (approximate, within
 * 1.01 * 2^-9 * |u| * max|v|), impl 0: exact fp32.  Same workspace as agcf_score_topk (agcf_score_topk_ws_bytes).
 * The measurable unit of the one dense contraction of the path (bench.py times it on its own; tests check the TF32
 * error bound the exactness proof of the top-K relies on). */
int agcf_score_group_max(const float* Uemb, const int32_t* user_rows, int32_t n_u,
                         const float* Iemb, int32_t n_items, int32_t d,
                         const int32_t* mask_rowptr, const int32_t* mask_items, int32_t item_offset, int32_t impl,
                         float* gmax_out, void* ws, int64_t ws_bytes, agcf_stream_t stream);

/* merge P per-shard top-K lists (vals/idx: [P, n_u, K]) into one, same ordering */
int agcf_topk_merge(const float* vals, const int32_t* idx, int32_t P, int32_t n_u, int32_t K,
                    float* out_val, int32_t* out_idx, agcf_stream_t stream);

/* plain scores for a few users (predict): out[r,:] = Uemb[user_rows[r],:] . Iemb^T */
int agcf_score_rows(const float* Uemb, const int32_t* user_rows, int32_t n_u,
                    const float* Iemb, int32_t n_items, int32_t d, float* out, agcf_stream_t stream);

/* per-user hits / DCG / IDCG for nc cutoffs from top-K ids and the (sorted) test
 * CSR: out is [n_u, nc, 3] doubles (hits, dcg, idcg); inv_log[r] = 1/ln(r+2) is
 * supplied by the host so that sums are bit-identical to math.log's.
 * test_total[u] counts ALL test items of u incl. those unseen in train.
 * Replaces: util/metrics.py:9-15 (hits), :72-85 (NDCG) per-user loops. */
int agcf_rank_metrics(const int32_t* topk_idx, int32_t K, const int32_t* t_rowptr, const int32_t* t_items,
                      const int32_t* test_total, int32_t n_u, const int32_t* cutoffs, int32_t nc,
                      const double* inv_log, double* out, agcf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AGCF_H_ */
