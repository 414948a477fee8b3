/*
 * regnn_b200.h -- C ABI of libregnn_b200.so: hand-written sm_100a CUDA kernels for RE-GNN's
 * relation-embedded message passing (REGraphConv / REGATConv / REGATv2Conv / REMixHopConv).
 *
 * This is the drop-in boundary.  The reference has no FFI of its own: its layers call DGL 0.7.1
 * (`update_all`, `apply_edges`, `edge_softmax`) which dispatches to DGL's C++/CUDA `gspmm` /
 * `gsddmm` kernels.  Every entry point below cites the reference call site(s) it replaces, as
 * file:line under /root/reference.
 *
 * Conventions
 *   - all pointers are DEVICE pointers owned by the caller (the PyTorch allocator in our host
 *     code); nothing is allocated inside the library; scratch space is passed in explicitly and
 *     sized by the matching *_workspace_bytes() query;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it, except
 *     regnn_csr_build / regnn_etype_permute which synchronise `stream` once to report invalid
 *     node ids / edge types (one-time graph construction);
 *   - return value: 0 = REGNN_OK, negative = error; regnn_last_error_string() is thread-local;
 *   - fp32 values, int32 graph indices, uint8 0-based edge types inside the library; the int64 /
 *     1-based conventions of the reference (run_regnn.py:94-99, `e_feat - 1`) stop at
 *     regnn_csr_build / regnn_etype_permute;
 *   - every reduction has a fixed summation order (no floating-point atomics): results are
 *     bit-identical run to run.
 *
 * Graph layout (built once per graph by regnn_csr_build, kept resident in HBM)
 *   indptr[N+1], indices[E], eid[E], row[E]   destination-sorted CSR: slot s of row v holds the
 *                                             in-edge (indices[s] -> v) with edge id eid[s];
 *                                             slots of a row are ordered by edge id (stable sort)
 *   indptr_t[N+1], indices_t[E], slot_t[E]    source-sorted view: entry j of row u is the out-edge
 *                                             (u -> indices_t[j]) stored at CSR slot slot_t[j];
 *                                             entries of a row are ordered by CSR slot
 *   etype_csr[E], etype_t[E]                  uint8 0-based edge type per CSR slot / per entry
 */
#ifndef REGNN_B200_H_
#define REGNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REGNN_OK 0
#define REGNN_ERR_INVALID_ARG (-1)
#define REGNN_ERR_UNSUPPORTED_SHAPE (-2)
#define REGNN_ERR_CUDA (-3)
#define REGNN_ERR_WORKSPACE_TOO_SMALL (-4)

#define REGNN_MAX_RELATIONS 200 /* uint8 edge types; the backward kernels keep 8 x R x 32 lane-local bins in shared memory */
#define REGNN_MAX_HEADS 32
#define REGNN_MAX_NODE_TYPES 16 /* regnn_grouped_linear_*: node types per launch */

/* Long-row decomposition of one CSR view (built once per graph by the host, see re_gnn_b200/graph.py):
 * rows with more than `threshold` slots are cut into fragments of `threshold` consecutive slots so that
 * no single warp has to walk a hub row (ogbn-mag-scale graphs have rows with 1e4-1e5 in-edges).
 * Fragment partial results are combined in fragment order => still deterministic.
 * All pointers are device pointers; pass NULL instead of the struct for "no splitting". */
typedef struct regnn_rowsplit {
  const int32_t* long_rows;  /* [num_long]    ids of the rows longer than threshold, ascending */
  const int32_t* frag_ptr;   /* [num_long+1]  first fragment of each long row                  */
  const int32_t* frag_row;   /* [num_frags]   row id of each fragment                          */
  const int32_t* frag_begin; /* [num_frags]   first CSR slot of each fragment                  */
  int32_t num_long, num_frags, threshold;
} regnn_rowsplit_t;

/* Counter-based attention dropout of the fused REGAT / REGATv2 kernels (the alternative to an explicit [E,H] `keep`
 * tensor): the keep factor of edge id e and head h of the call is a pure function of (key, e, global head), computed in
 * registers from the edge id the kernel already loads, so every kernel, rank and partition of the graph sees the same
 * mask without storing or exchanging it:
 *   c      = e * num_heads_total + head_offset + h                          (64-bit counter)
 *   x      = mix32( lo32(c) ^ lo32(key) )
 *   x      = mix32( x + hi32(c) * 0x9E3779B1 + hi32(key) )                  (uint32 arithmetic, wrapping)
 *   keep   = x >= threshold ? scale : 0
 *   mix32(z): z ^= z >> 16; z *= 0x7feb352d; z ^= z >> 15; z *= 0x846ca68b; z ^= z >> 16
 * With drop probability p: threshold = floor(p * 2^32), scale = (float)(1 / (1 - p)); p = 0 is threshold 0, scale 1
 * (every factor is exactly 1).  head_offset / num_heads_total let a call over a slice of the heads reproduce that
 * slice of the full-H mask (num_heads_total >= head_offset + num_heads of the call).  Restated in
 * oracle/attn_dropout_oracle.py. */
typedef struct regnn_attn_dropout {
  uint64_t key;
  uint32_t threshold;
  float scale;
  int32_t head_offset;
  int32_t num_heads_total;
} regnn_attn_dropout_t;

int regnn_version(void);
const char* regnn_status_string(int status);
const char* regnn_last_error_string(void);
/* Upper bound on the number of thread blocks any regnn_* reduction kernel emits partial sums for: size every
 * `partials` scratch argument as regnn_max_partial_blocks() * <per-block entries> doubles. */
int regnn_max_partial_blocks(void);

/* ------------------------------------------------------------------------------------------------
 * Graph construction.  Replaces DGL's lazy in-CSR / out-CSR build behind
 * `dgl.DGLGraph(adjM)` ... `g.to(device)` (run_regnn.py:84-87) and the first `update_all`
 * (layer/REGraphConv.py:69).  src/dst: int64 [E] in edge-id order (what `g.edges()` returns,
 * run_regnn.py:95).  Hand-written stable LSD radix sort (8-bit digits) + prefix scans.
 * Returns REGNN_ERR_INVALID_ARG if any node id is outside [0, N).
 */
size_t regnn_csr_build_workspace_bytes(int64_t num_nodes, int64_t num_edges);
int regnn_csr_build(const int64_t* src, const int64_t* dst, int64_t num_nodes, int64_t num_edges,
                    int32_t* indptr, int32_t* indices, int32_t* eid, int32_t* row,
                    int32_t* indptr_t, int32_t* indices_t, int32_t* slot_t,
                    void* workspace, size_t workspace_bytes, void* stream);

/* `edge_weight[e_feat - 1]` indexing (layer/REGraphConv.py:61, REGATConv.py:75, REGATv2Conv.py:143,
 * REMixHopConv.py:53): converts the reference's 1-based int64 edge types (edge-id order) to uint8
 * 0-based types in CSR-slot order and in transposed-entry order.
 * Returns REGNN_ERR_INVALID_ARG if any type is outside [1, num_relations]. */
int regnn_etype_permute(const int64_t* etype_1based, const int32_t* eid, const int32_t* slot_t,
                        int64_t num_edges, int num_relations, uint8_t* etype_csr, uint8_t* etype_t,
                        int32_t* status_scratch /* device int32[1] */, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Relation-weighted in-degree normalisation:
 *   w = LeakyReLU_0.01(alpha * theta);  deg[v] = sum_{e in In(v)} w[etype e];
 *   norm[v] = max(deg[v], clamp_min) ^ exponent        (clamp_min = 1 in every HGB layer;
 *             clamp_min <= 0: no clamp, deg ^ exponent, and 0 for rows without in-edges -- the
 *             `deg.pow(-1)` of the MAG-stack layers, mag/regnn_saint.py:254-258)
 * Replaces `update_all(u_mul_e('nones','ew'), sum)` + clamp + pow
 * (layer/REGraphConv.py:58-75, layer/REMixHopConv.py:50-64; exponent -1: RESAGEConv.py:75-78).
 * theta: [R] (the [R,1] `edge_weight` parameter).  Row range [row_begin, row_end) lets a rank of a
 * destination-row partition compute only the rows it owns; deg/norm are indexed by global row id.
 */
/* counts[v*R + r] = number of in-edges of v with (0-based) relation r: a parameter-independent [N,R] int32
 * table built once per (graph, e_feat).  When passed to the two entry points below, the degree norm and its
 * gradient become dense streaming passes over it (no per-edge work per training step). */
int regnn_relation_counts(const int32_t* row, const uint8_t* etype_csr, int64_t num_edges, int64_t num_nodes,
                          int num_relations, int32_t* counts, void* stream);

int regnn_wdeg_norm_fwd(const int32_t* indptr, const uint8_t* etype_csr,
                        const int32_t* counts /* optional: then indptr/etype_csr may be NULL */, const float* theta,
                        float alpha, int num_relations, float exponent, float clamp_min, int64_t row_begin,
                        int64_t row_end, float* deg, float* norm, void* stream);
/* Backward of the above: d_theta[r] += alpha * LeakyReLU'(alpha*theta[r]) *
 *   sum_{e: etype e = r} d_deg[dst e],   d_deg[v] = [deg[v] >= 1] * q * max(deg,1)^(q-1) * d_norm[v].
 * partials: double [regnn_max_partial_blocks() * R] scratch.  d_theta is OVERWRITTEN. */
int regnn_wdeg_norm_bwd(const int32_t* indptr, const uint8_t* etype_csr, const int32_t* counts, const float* theta,
                        float alpha, int num_relations, float exponent, float clamp_min, int64_t row_begin,
                        int64_t row_end, const float* deg, const float* d_norm, double* partials,
                        float* d_theta, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Relation-weighted, degree-normalised SpMM (the REGCN / REMixHop aggregation):
 *   Y[v,:] = norm_dst[v] * sum_{s in row v} w[etype[s]] * norm_src[indices[s]] * X[indices[s],:]
 * Replaces `feat * norm` -> `update_all(u_mul_e('h','ew'), sum)` -> `rst * norm`
 * (layer/REGraphConv.py:76,84-98) and, with etype == NULL (w == 1), the un-weighted
 * `update_all(copy_u, sum)` of layer/REMixHopConv.py:78-82.  norm_src / norm_dst may be NULL (== 1).
 * The same entry point run on the transposed view (indptr_t, indices_t, etype_t) is the
 * backward pass w.r.t. X (DGL: gspmm on the reverse graph).
 * X: [*, F] with leading dimension ldx (floats); Y: rows [row_begin,row_end) written at Y[v*ldy].
 * row_order (optional, NULL = none): the rows of [0, row_end) NOT listed in split->long_rows, by descending
 * slot count (ties by ascending row id) -- [row_end - num_long] ids, built once per graph.  With it, a full
 * range (row_begin == 0) and F <= 128 (F % 4 == 0, 16-byte aligned rows) the lane-group kernel runs: 32/G
 * rows per warp (G = 4/8/16/32 lanes per row), each summed by one lane group in slot order (results identical to the whole-warp kernel).
 */
int regnn_spmm_fwd(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                   const float* theta, float alpha, int num_relations, const float* norm_src,
                   const float* norm_dst, const float* X, int64_t ldx, float* Y, int64_t ldy,
                   int64_t row_begin, int64_t row_end, int feat, const regnn_rowsplit_t* split,
                   float* split_workspace /* [split->num_frags * feat] floats, or NULL */,
                   const int32_t* row_order, void* stream);

/* Backward of regnn_spmm_fwd w.r.t. the relation weights and the norm vector (norm_src == norm_dst
 * == norm, the reference's case).  Given G = dL/dY, X, Y and dX (= the transposed regnn_spmm_fwd of G):
 *   d_norm[v]  = ( <Y[v],G[v]> + <X[v],dX[v]> ) / norm[v]
 *   d_theta[r] = alpha*LeakyReLU'(alpha*theta[r]) * sum_{e: etype=r} norm[src]norm[dst] <X[src],G[dst]>
 * (DGL: gsddmm(dot) for the edge-weight gradient + atomic index_put_ of `w[e_feat-1]`; here a
 * deterministic two-level reduction).  etype == NULL: only d_norm is produced (REMixHop).
 * norm_sides: bit 0 = the forward scaled the source side by norm, bit 1 = the destination side
 * (3 for REGraphConv / REMixHopConv; 1 for RESAGEConv, layer/RESAGEConv.py:82; 2 for REGINConv,
 * layer/REGINConv.py:61); the unscaled side drops out of both formulas.
 * partials: double [regnn_max_partial_blocks() * R].  d_theta is OVERWRITTEN; d_norm rows written. */
int regnn_spmm_bwd_w(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                     const float* theta, float alpha, int num_relations, const float* norm,
                     int norm_sides, const float* X, int64_t ldx, const float* Y, int64_t ldy, const float* G,
                     int64_t ldg, const float* dX, int64_t lddx, int64_t row_begin, int64_t row_end,
                     int feat, double* partials, float* d_theta, float* d_norm,
                     const regnn_rowsplit_t* split, void* stream);

/* Fused backward of regnn_spmm_fwd: ONE gather pass over the transposed view produces both
 *   dX[u]      = ns(u) * sum_{e in Out(u)} w[etype e] * nd(dst e) * G[dst e]       (DGL: gspmm on the reverse graph)
 *   d_theta[r] = alpha*LeakyReLU'(alpha*theta[r]) * sum_{e: etype=r} ns(src)*nd(dst)*<X[src], G[dst]>
 * (ns/nd = norm on the sides selected by norm_sides, else 1): the per-edge dot <X[u], G[dst]> reuses the
 * G[dst] row that the dX gather already holds in registers; X rows of the block are staged in shared
 * memory by TMA bulk copies.
 * d_norm (optional, lane-group kernel only: row_order_t, full range, F <= 128): the gradient w.r.t. the norm vector
 *   d_norm[u] = ( [sides&2] <Y[u],G[u]> + [sides&1] <X[u],dX[u]> ) / norm[u]
 * is produced in the same pass (Y = the forward result; the lane group that owns row u reads Y[u] and G[u] behind its
 * gathers), replacing the separate regnn_rowdot_norm_bwd pass of round 1.  NULL: not produced (use xdx +
 * regnn_rowdot_norm_bwd, the path of the whole-warp kernel and of the row-partitioned multi-GPU scheme).
 * partials: double [regnn_max_partial_blocks() * R]; d_theta is OVERWRITTEN;
 * split_workspace: split_t->num_frags * feat floats.  With row_order_t (F <= 128, full range) the lane-group
 * kernel runs instead and keeps X[u] in registers (no shared-memory tile). */
int regnn_spmm_bwd_fused(const int32_t* indptr_t, const int32_t* indices_t, const uint8_t* etype_t,
                         const float* theta, float alpha, int num_relations, const float* norm,
                         int norm_sides, const float* X, int64_t ldx, const float* G, int64_t ldg,
                         float* dX, int64_t lddx, int64_t row_begin, int64_t row_end, int feat,
                         double* partials, float* d_theta, float* xdx /* optional [N]: <X[u],dX[u]> per row */,
                         const float* Y /* forward result, needed for d_norm when sides & 2 */, int64_t ldy,
                         float* d_norm /* optional [N] */,
                         const regnn_rowsplit_t* split_t, float* split_workspace,
                         const int32_t* row_order_t /* as regnn_spmm_fwd's row_order, for the transposed view */,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Feature-sliced multi-GPU aggregation (no reference counterpart: the reference is single-device).
 * Every rank propagates ALL rows for F/P of the columns (a "column slab" [P*rows_per_rank, F/P]); the dense
 * layers around the aggregation are row-parallel (rank q owns rows [q*rows_per_rank, (q+1)*rows_per_rank)).
 * The two re-partitions run over peer-mapped memory (NVLink), not through a collective library:
 *   rows -> slabs: regnn_rows_to_slabs pushes this rank's row block, column slice q to rank q's slab;
 *   slabs -> rows: the *_scatter variants of the two SpMM entry points store each finished row straight into
 *                  its owner's row block (regnn_peer_rows_t) from the kernel epilogue -- compute and exchange
 *                  are one kernel; regnn_slabs_to_rows is the stand-alone push for the attention kernels.
 * The caller provides the peer-mapped buffers (e.g. CUDA VMM / IPC; the Python binding uses torch symmetric memory)
 * and a cross-rank barrier after each call before the written buffers are read. */
typedef struct regnn_peer_rows {
  float* const* base;    /* device array [num_ranks]: row block [rows_per_rank, ld] of every rank (peer-mapped) */
  int32_t num_ranks;
  int64_t rows_per_rank; /* row v belongs to rank v / rows_per_rank                                             */
  int64_t ld;            /* leading dimension of the row blocks (floats)                                        */
  int64_t col_offset;    /* first column this rank's slab covers                                                */
} regnn_peer_rows_t;

/* X: [num_rows, feat] row block (ld ldx).  Slice q (columns [q*feat/P, (q+1)*feat/P)) is written to
 * peer_slabs[q] + (row_offset + i) * (feat/P): per peer one contiguous range.  feat % (4*num_ranks) == 0. */
int regnn_rows_to_slabs(const float* X, int64_t ldx, int64_t num_rows, int feat, int num_ranks, int64_t row_offset,
                        float* const* peer_slabs /* device array [num_ranks] */, void* stream);

/* Halo exchange of destination-row blocks (partition.halo_propagate; it replaces the all-gather of the whole [N, F]
 * matrix that partition.partitioned_propagate does per direction): for every peer q, the rows
 * X[send_rows[send_ptr[q] .. send_ptr[q+1])] of this rank's row block are stored to
 * peer_bufs[q] + (recv_offset[q] + i) * ldb, i = 0, 1, ...  send_ptr [num_ranks+1] and recv_offset [num_ranks] are HOST
 * arrays (set up once per partition); send_rows (int32, local row ids) and peer_bufs [num_ranks] are device arrays; lists
 * may be empty.  The pointers need not be peer-mapped: P local buffers work the same.  feat % 4 == 0, 16-byte aligned
 * rows, num_ranks <= REGNN_HALO_MAX_RANKS. */
#define REGNN_HALO_MAX_RANKS 64
int regnn_halo_push(const float* X, int64_t ldx, int feat, const int32_t* send_rows, const int64_t* send_ptr,
                    const int64_t* recv_offset, float* const* peer_bufs, int64_t ldb, int num_ranks, int rank, void* stream);

/* The reverse exchange of the REGAT halo backward (partition.halo_gat: the logit gradient of an edge whose destination
 * is remote goes to the destination's owner, into its CSR slot): for every peer q, the rows X[k], k in
 * send_ptr[q] .. send_ptr[q+1], of this rank's [rows, width] buffer are stored to peer_bufs[q] + dst_rows[k] * ldb.
 * Any width >= 1 (stores are 4-byte words); send_ptr [num_ranks+1] is a HOST array, dst_rows (int32) and peer_bufs
 * [num_ranks] are device arrays; lists may be empty.  Local buffers work the same as peer-mapped ones.
 * num_ranks <= REGNN_HALO_MAX_RANKS. */
int regnn_halo_scatter(const float* X, int64_t ldx, int width, const int64_t* send_ptr, const int32_t* dst_rows,
                       float* const* peer_bufs, int64_t ldb, int num_ranks, int rank, void* stream);

/* The per-slot forward exchange of the REGATv2 halo backward (partition.halo_gatv2: regnn_gatv2_bwd_edges runs on the
 * owner of an edge's source, but regnn_gatv2_fwd stored the edge's logit and sign mask in its destination's slot): for
 * every peer q and k in send_ptr[q] .. send_ptr[q+1], slot s = send_slots[k] is stored to row
 * r = recv_offset[q] + (k - send_ptr[q]) of peer q's buffers: logit[s*H .. +H) to peer_logit[q] + r*H and
 * qmask[s*4C .. +4C) to peer_mask[q] + r*4C (C = num_chunks 128-bit words, the layout of regnn_gatv2_fwd's qmask).  Both
 * arrays move in one launch.  send_ptr [num_ranks+1] and recv_offset [num_ranks] are HOST arrays; send_slots (int32) and
 * peer_logit / peer_mask [num_ranks] are device arrays; lists may be empty.  Local buffers work the same as peer-mapped
 * ones.  qmask 16-byte aligned, num_ranks <= REGNN_HALO_MAX_RANKS. */
int regnn_halo_push_slots(const float* logit, int num_heads, const uint32_t* qmask, int num_chunks,
                          const int32_t* send_slots, const int64_t* send_ptr, const int64_t* recv_offset,
                          float* const* peer_logit, float* const* peer_mask, int num_ranks, int rank, void* stream);

/* The reverse re-partition for kernels without a scatter epilogue (the fused attention kernels, one head slice per
 * rank): S [num_rows, feat] is this rank's column slab (ld lds); row v is stored to
 * peers->base[v / rows_per_rank][(v % rows_per_rank) * ld + col_offset .. + feat). */
int regnn_slabs_to_rows(const float* S, int64_t lds, int64_t num_rows, int feat, const regnn_peer_rows_t* peers,
                        void* stream);

/* regnn_spmm_fwd over the full row range [0, num_rows) of a column slab (feat <= 128, feat % 4 == 0, row_order required) whose
 * result rows are stored to their owner ranks: peers->base[v / rows_per_rank][(v % rows_per_rank) * ld + col_offset].
 * y_local (optional, leading dimension ldl): the result slab is ALSO kept locally -- the backward pass then folds the
 * norm gradient of this rank's columns into its own kernel (regnn_spmm_bwd_fused_scatter's d_norm). */
int regnn_spmm_fwd_scatter(const int32_t* indptr, const int32_t* indices, const uint8_t* etype,
                           const float* theta, float alpha, int num_relations, const float* norm_src,
                           const float* norm_dst, const float* X, int64_t ldx, int64_t num_rows, int feat,
                           const regnn_rowsplit_t* split, float* split_workspace, const int32_t* row_order,
                           const regnn_peer_rows_t* peers, float* y_local, int64_t ldl, void* stream);

/* regnn_spmm_bwd_fused with the dX rows stored to their owner ranks; d_theta / xdx / d_norm stay local and cover this
 * rank's columns only.  d_norm (optional, with Y = the local result slab of regnn_spmm_fwd_scatter): every row's norm
 * gradient restricted to this rank's columns.  The norm's own backward is linear in d_norm, so each rank pushes its
 * column share through regnn_wdeg_norm_bwd and the caller sums R floats across ranks -- no N-float exchange and no
 * separate row-dot pass. */
int regnn_spmm_bwd_fused_scatter(const int32_t* indptr_t, const int32_t* indices_t, const uint8_t* etype_t,
                                 const float* theta, float alpha, int num_relations, const float* norm,
                                 int norm_sides, const float* X, int64_t ldx, const float* G, int64_t ldg,
                                 int64_t num_rows, int feat, double* partials, float* d_theta, float* xdx,
                                 const float* Y, int64_t ldy, float* d_norm,
                                 const regnn_rowsplit_t* split_t, float* split_workspace,
                                 const int32_t* row_order_t, const regnn_peer_rows_t* peers, void* stream);

/* d_norm[v] = ( [sides&2] <Y[v],G[v]> + [sides&1] <X[v],dX[v]> ) / norm[v] for rows [row_begin,row_end):
 * the gradient of regnn_spmm_fwd w.r.t. the norm vector (row-local, pure streaming).  If xdx (from
 * regnn_spmm_bwd_fused) is given, X and dX are not read. */
int regnn_rowdot_norm_bwd(const float* norm, int norm_sides, const float* X, int64_t ldx, const float* Y,
                          int64_t ldy, const float* G, int64_t ldg, const float* dX, int64_t lddx,
                          const float* xdx, int64_t row_begin, int64_t row_end, int feat, float* d_norm,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused REGAT layer core (layer/REGATConv.py:71-92): per destination v and head h
 *   l[e,h] = LeakyReLU_slope( el[src,h] + er[v,h] + w[etype,h] ),  w = LeakyReLU_0.01(alpha*theta)
 *   a      = softmax over In(v) of l  (per-destination max subtracted, no epsilon)
 *   out[v,h,:] = sum_e a[e,h] * keep[eid e, h] * feat[src,h,:]
 * Replaces apply_edges(u_add_v) + index/add/LeakyReLU + edge_softmax (4 kernels) +
 * update_all(u_mul_e, sum).  etype == NULL drops the relation term (`edge_feats=None`).
 * keep: optional [E,H] attention-dropout scale (0 or 1/(1-p)) in EDGE-ID order, NULL = none.
 * dropout: optional counter-based dropout (regnn_attn_dropout_t), keep_e computed from eid[slot]; NULL = none.  At
 *   most one of keep and dropout; either needs eid.  The factor multiplies a at the same place in both modes, so a
 *   keep tensor holding the hashed factors gives the same bits.
 * attn_out: optional [E,H] output of a*keep in EDGE-ID order (`get_attention`), NULL = skip.
 * Saves rowmax/rowsum [N,H] for the backward pass.  theta: [R,H].
 * Shapes of every REGAT / REGATv2 entry point below: 1 <= num_heads <= REGNN_MAX_HEADS, head_dim a power of two in
 * [4, 512], num_heads * head_dim <= 1024; anything else is REGNN_ERR_UNSUPPORTED_SHAPE.
 */
int regnn_gat_fwd(const int32_t* indptr, const int32_t* indices, const int32_t* eid,
                  const uint8_t* etype_csr, const float* theta, float alpha, int num_relations,
                  const float* feat, const float* el, const float* er, float negative_slope,
                  const float* keep, const regnn_attn_dropout_t* dropout, int num_heads, int head_dim,
                  int64_t row_begin, int64_t row_end,
                  float* out, float* rowmax, float* rowsum, float* attn_out, const regnn_rowsplit_t* split,
    float* split_workspace /* num_frags * (H*D + 2*H) floats, or NULL */,
    const int32_t* row_order /* as regnn_spmm_fwd's: degree-sorted rows that are not long, or NULL (natural order) */,
    void* stream);

/* Backward of regnn_gat_fwd as ONE gather pass (G = dL/d out).  The softmax backward of edge e = (u -> v) needs
 * da_e = <feat[u,h,:], G[v,h,:]>, a_e (recomputed from the saved row max / sum) and S_v = <out[v,h,:], G[v,h,:]>; the
 * source-major pass that produces d_feat[u] = sum_e a_e*keep_e*G[v] gathers G[v] anyway, so with the per-destination
 * statistics packed per (node, head) everything per edge is computed there -- DGL's autograd runs gsddmm(dot) over
 * feat[src] and a reverse-graph gspmm as two gather passes with [E,H] tensors in between.
 *
 * regnn_gat_bwd_stats: stats[v,h] = (er[v,h], rowmax[v,h], 1/rowsum[v,h], <out[v,h,:], G[v,h,:]>), float4 per (node, head).
 * er == NULL (REGATv2, no destination score): stats.x = 0. */
int regnn_gat_bwd_stats(const float* out, const float* G, const float* er, const float* rowmax, const float* rowsum,
                        int64_t num_nodes, int num_heads, int head_dim, float* stats /* [N,H,4] */, void* stream);

/* regnn_gat_bwd_edges: source-major pass over the transposed view:
 *   dpre_e  = (a_e*keep_e*da_e - a_e*S_v) * LeakyReLU'(pre_e)      -> dpre_csr[slot_t[j], h]  ([E,H], CSR slot order)
 *   d_feat[u,h,:] = sum_{e in Out(u)} a_e*keep_e * G[v,h,:]  (+ d_el[u,h]*attn_l[h,:] when attn_l != NULL: the gradient
 *                   through el = <feat, attn_l>, layer/REGATConv.py:68)
 *   d_el[u,h]     = sum_{e in Out(u)} dpre_e
 * etype_t: edge types per transposed entry; eid: slot -> edge id, read through slot_t (only with keep or dropout);
 * keep / dropout: as in regnn_gat_fwd (at most one). */
int regnn_gat_bwd_edges(const int32_t* indptr_t, const int32_t* indices_t, const int32_t* slot_t,
                        const uint8_t* etype_t, const int32_t* eid, const float* theta, float alpha, int num_relations,
                        const float* feat, const float* el, const float* stats, float negative_slope,
                        const float* keep, const regnn_attn_dropout_t* dropout, const float* G, int num_heads,
                        int head_dim, int64_t row_begin,
                        int64_t row_end, float* d_feat, float* d_el, float* dpre_csr, const float* attn_l,
                        const regnn_rowsplit_t* split_t /* of the transposed view */,
                        float* split_workspace /* num_frags * (H*D + 2*H) floats, or NULL */,
                        const int32_t* row_order_t, void* stream);

/* regnn_gat_bwd_reduce: the destination-side reductions of dpre_csr, pure streaming over [E,H] (one fused pass when the
 * row range is large, two specialised kernels on L2-resident graphs):
 *   d_er[v,h] = sum_{slots of row v} dpre_csr[slot,h]        d_theta[r,h] = alpha*LeakyReLU'(alpha*theta[r,h]) * sum_{etype=r} dpre
 * (deterministic: slot order per row; lane-local bins -> per-block double partials -> fixed-order finalize).
 * partials: double [regnn_max_partial_blocks() * R * H]; split_workspace: split->num_frags * H floats. */
int regnn_gat_bwd_reduce(const int32_t* indptr, const uint8_t* etype_csr, const float* theta, float alpha,
                         int num_relations, const float* dpre_csr, int num_heads, int64_t row_begin, int64_t row_end,
                         float* d_er, double* partials, float* d_theta, const regnn_rowsplit_t* split,
                         float* split_workspace, void* stream);

/* Projection scores of REGAT (layer/REGATConv.py:68-69: `el = (feat * attn_l).sum(-1)`, `er = (feat * attn_r).sum(-1)`,
 * two eager mul + sum pairs in the reference) in one streaming pass over feat [N,H,D]: el, er [N,H]. */
int regnn_attn_scores_fwd(const float* feat, const float* attn_l, const float* attn_r, int64_t num_nodes, int num_heads,
                          int head_dim, float* el, float* er, void* stream);

/* Parameter gradients of the projection scores: d_attn_l[h,d] = sum_n d_el[n,h]*feat[n,h,d], d_attn_r likewise
 * (deterministic: lane-local sums, per-block double partials, fixed-order finalize).  d_feat != NULL: the same pass adds
 * the destination-side score gradient to the feature gradient in place, d_feat[n,h,:] += d_er[n,h]*attn_r[h,:].
 * partials: double [regnn_max_partial_blocks() * 2*H*D]. */
int regnn_attn_scores_bwd(const float* feat, const float* d_el, const float* d_er, int64_t num_nodes, int num_heads,
                          int head_dim, double* partials, float* d_attn_l, float* d_attn_r, float* d_feat,
                          const float* attn_r, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused REGATv2 layer core (layer/REGATv2Conv.py:133-152):
 *   l[e,h] = sum_d attn[h,d] * LeakyReLU_slope( fs[src,h,d] + fd[v,h,d] ) + w[etype,h]
 *   a = edge_softmax(l);  out[v,h,:] = sum_e a*keep * fs[src,h,:]
 * The [E,H,D] intermediates of the reference are never materialised.  keep / dropout / attn_out as in regnn_gat_fwd.
 */
int regnn_gatv2_fwd(const int32_t* indptr, const int32_t* indices, const int32_t* eid,
                    const uint8_t* etype_csr, const float* theta, float alpha, int num_relations,
                    const float* fs, const float* fd, const float* attn, float negative_slope,
                    const float* keep, const regnn_attn_dropout_t* dropout, int num_heads, int head_dim,
                    int64_t row_begin,
                    int64_t row_end, float* out, float* rowmax, float* rowsum, float* attn_out,
                    float* logit_csr /* [E,H] CSR-slot order, or NULL (inference) */,
                    uint32_t* qmask /* [E, ceil(H*D/128), 4], or NULL; see below */,
                    const regnn_rowsplit_t* split,
    float* split_workspace /* num_frags * (H*D + 2*H) floats, or NULL */,
    const int32_t* row_order /* as regnn_gat_fwd */, void* stream);

/* Backward of regnn_gatv2_fwd: ONE gather pass (source-major) + one streaming pass (destination-major).  The forward
 * saved, per CSR slot, the raw logit l[e,h] (logit_csr) and the sign of every component of q = fs[src]+fd[dst] as a
 * 128-bit mask per 128-float slice of the H*D row (qmask: uint32 [E, ceil(H*D/128), 4]; bit l of word c = component c of
 * the l-th 128-bit chunk of the slice is > 0) -- LeakyReLU'(q) is one bit per feature.  With the per-destination
 * statistics stats[v,h] = (0, rowmax, 1/rowsum, <out[v,h,:], G[v,h,:]>) of regnn_gat_bwd_stats (er == NULL) every
 * per-edge quantity
 *   a = exp(l - rowmax)/rowsum,  dl = a*keep*<fs[u],G[v]> - a*<out[v],G[v]>
 * is local to the pass that gathers G[v] for d_fs[u]:
 *   regnn_gatv2_bwd_edges  d_fs[u,h,:] = sum_{Out(u)} ( a*keep*G[v,h,:] + dl*attn[h,:]*LeakyReLU'(q) ),  dl_csr[slot,h],
 *                          d_attn_src[h,:] = sum_u fs[u,h,:] (.) sum_{Out(u)} dl*LeakyReLU'(q)
 *   regnn_gatv2_bwd_dst    d_fd[v,h,:] = attn[h,:] (.) T[v],  T[v] = sum_{In(v)} dl*LeakyReLU'(q)   (no gather: dl_csr and
 *                          qmask are read in slot order),  d_attn_dst = sum_v fd[v] (.) T[v],  d_theta [R,H]
 * and d_attn = d_attn_src + d_attn_dst (the caller adds the two [H*D] vectors).
 * Both calls must cover rows whose slots the forward call covered; E * max(H, ceil(H*D/128)) < 2^32 (32-bit slot
 * offsets in the forward).  Deterministic: lane-local sums, per-block partials, fixed-order finalize.
 * block_partials: float [regnn_gatv2_bwd_edges_blocks(...) * H*D];  partials (edges): double [592 * H*D];
 * partials (dst): double [max(regnn_max_partial_blocks() * H*D, 592 * R*H)]. */
int64_t regnn_gatv2_bwd_edges_blocks(int64_t num_rows, int num_frags /* of split_t */, int num_long /* of split_t */,
                                     int num_heads, int head_dim, int ordered /* row_order_t given and row_begin == 0 */);
int regnn_gatv2_bwd_edges(const int32_t* indptr_t, const int32_t* indices_t, const int32_t* slot_t,
                          const int32_t* eid /* slot -> edge id through slot_t; only read with keep or dropout */,
                          const float* fs, const float* stats, const float* logit_csr, const uint32_t* qmask,
                          const float* attn, float negative_slope, const float* keep,
                          const regnn_attn_dropout_t* dropout /* as regnn_gat_fwd; at most one of keep and dropout */,
                          const float* G, int num_heads, int head_dim,
                          int64_t row_begin, int64_t row_end, float* d_fs, float* dl_csr, float* d_attn_src,
                          float* block_partials, double* partials, const regnn_rowsplit_t* split_t /* transposed view */,
    float* split_workspace /* num_frags * (H*D + 2*H) floats, or NULL */, const int32_t* row_order_t, void* stream);
int regnn_gatv2_bwd_dst(const int32_t* indptr, const uint8_t* etype_csr, const float* theta, float alpha,
                        int num_relations, const float* fd, const float* dl_csr, const uint32_t* qmask,
                        const float* attn, float negative_slope, int num_heads, int head_dim, int64_t row_begin,
                        int64_t row_end, float* d_fd, float* d_attn_dst, double* partials, float* d_theta,
                        const regnn_rowsplit_t* split,
    float* split_workspace /* num_frags * (H*D + 2*H) floats, or NULL */, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Neighbour sampling for the sampled-minibatch path (replaces torch_sparse's CPU `sample_adj` behind
 * `NeighborSampler(edge_index, sizes=[25, 20], ...)`, mag/regnn_ns.py:206-214).  For target i the kernel
 * writes up to `fanout` distinct CSR slots of its in-edges to out_slot[i*fanout + j] (-1 = none): all
 * in-edges if the in-degree is <= fanout, else a keyed pseudo-random subset without replacement
 * (4-round Feistel permutation with cycle walking; oracle/sampler_oracle.py is the bit-exact spec).
 * Counter-based: `key` = f(seed, epoch, rank, batch, layer); no RNG state. */
int regnn_sample_neighbors(const int32_t* indptr, const int64_t* targets, int64_t num_targets, int fanout,
                           uint64_t key, int32_t* out_slot, void* stream);

/* One layer of the sampler with device-resident sizes: samples `fanout` in-edges of every target (the slots of
 * regnn_sample_neighbors), relabels the frontier and compacts the sampled edges, with no host synchronisation.
 *   targets     [max_targets] global ids; the first *num_targets are used (num_targets NULL: all of them) -- the
 *               info[REGNN_SAMPLE_INFO_SOURCES] word of the previous layer, so layers chain on the device
 *   new_n_id    [max_sources >= max_targets + min(num_nodes, max_targets * fanout)]: the targets in their order, then
 *               every sampled source that is not a target, once, in ascending global id (torch.unique's order)
 *   src_local / dst_local / edge_id  [max_targets * fanout]: sampled edge e (targets in order, each target's slots in
 *               sample order) is new_n_id[src_local[e]] -> target dst_local[e], global edge id edge_id[e]
 *   row_off     [max_targets + 1]: exclusive scan of the per-target edge counts (the in-CSR offsets of the block)
 *   src_hist    [max_sources]: sampled out-edges per local source
 *   info        [REGNN_SAMPLE_INFO_WORDS] int32, zeroed and filled here (layout below)
 *   pos_map     [num_nodes] int32, every entry 0x7fffffff on entry; flags [num_nodes] uint32, all 0 on entry; both are
 *               restored before the last kernel ends, so one pair serves every layer and batch of a sampler
 * split_threshold: the long-row threshold of regnn_rowsplit_t the split statistics in info are counted for.
 * workspace: regnn_sample_layer_workspace_bytes(num_nodes, max_targets, fanout) bytes. */
enum {
  REGNN_SAMPLE_INFO_SOURCES = 0,          /* number of sources of the block (= targets of the next layer)        */
  REGNN_SAMPLE_INFO_EDGES = 1,            /* number of sampled edges                                             */
  REGNN_SAMPLE_INFO_EMPTY_ROWS = 2,       /* targets without a sampled in-edge                                   */
  REGNN_SAMPLE_INFO_IN_SPLIT = 3,         /* (long rows, fragments) of the in-view                               */
  REGNN_SAMPLE_INFO_IN_SPLIT_LOOPS = 5,   /*   ... with one self loop per target appended                        */
  REGNN_SAMPLE_INFO_OUT_SPLIT = 7,        /* (long rows, fragments) of the transposed view                       */
  REGNN_SAMPLE_INFO_OUT_SPLIT_LOOPS = 9,  /*   ... with one self loop per target appended                        */
  REGNN_SAMPLE_INFO_WORDS = 16
};
size_t regnn_sample_layer_workspace_bytes(int64_t num_nodes, int64_t max_targets, int fanout);
int regnn_sample_layer(const int32_t* indptr, const int32_t* indices, const int32_t* eid, int64_t num_nodes,
                       const int64_t* targets, int64_t max_targets, const int32_t* num_targets, int fanout,
                       uint64_t key, int split_threshold, int32_t* pos_map, uint32_t* flags, int64_t* new_n_id,
                       int64_t max_sources, int64_t* src_local, int64_t* dst_local, int64_t* edge_id,
                       uint32_t* row_off, int32_t* src_hist, int32_t* info, void* workspace, size_t workspace_bytes,
                       void* stream);

/* Both CSR views of one sampled block, bit-identical to regnn_csr_build + regnn_etype_permute +
 * regnn_relation_counts on the block's edge list src_local -> dst_local (+ one self loop per target when
 * self_loops, edge id num_sampled + v, typed num_edge_types + node_type[targets[v]]), without a host
 * synchronisation.  Inputs are regnn_sample_layer's outputs (sizes read back by the caller) and the 0-based global
 * edge_type / node_type.  Outputs: src / dst / etype1 [num_edges] in edge-id order (etype1 1-based), the CSR arrays
 * of regnn_csr_build over num_src nodes, et_csr / et_t of regnn_etype_permute, and counts [num_src * num_relations]
 * (NULL: not built).  An edge whose type lies outside [0, num_relations) stores 1 to *status (device int32, left
 * untouched otherwise: the caller zeroes it and reads it at its next synchronisation) and is typed 0 in et_csr / et_t /
 * counts.  workspace: regnn_csr_build_workspace_bytes(num_src, num_edges). */
int regnn_block_csr_build(const int64_t* src_local, const int64_t* dst_local, const int64_t* edge_id,
                          const uint32_t* row_off, const int64_t* targets, int64_t num_src, int64_t num_dst,
                          int64_t num_sampled, const int64_t* edge_type, const int64_t* node_type, int num_edge_types,
                          int self_loops, int num_relations, int64_t* src, int64_t* dst, int64_t* etype1,
                          int32_t* indptr, int32_t* indices, int32_t* eid, int32_t* row, int32_t* indptr_t,
                          int32_t* indices_t, int32_t* slot_t, uint8_t* et_csr, uint8_t* et_t, int32_t* counts,
                          int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* GraphSAINT random-walk roots (replaces torch_sparse `random_walk` behind
 * `GraphSAINTRandomWalkSampler(data, batch_size=20000, walk_length=2, ...)`, mag/regnn_saint.py:185-190):
 * root i starts at node hash(key, i) % N and takes `walk_length` steps along out-edges of the transposed view;
 * walks[i*(walk_length+1) + s] is the node after s steps.  Counter-based, bit-exact with the oracle. */
int regnn_random_walk(const int32_t* indptr_t, const int32_t* indices_t, int64_t num_nodes, int64_t num_roots,
                      int walk_length, uint64_t key, int64_t* walks, void* stream);

/* GraphSAINT subgraph induced by the walk nodes (replaces the relabelling and edge selection of
 * `GraphSAINTRandomWalkSampler`, mag/regnn_saint.py:185-190), in two calls with one small host read between them: the
 * host learns the induced edge count from info to size the edge arrays.  No host synchronisation inside either call;
 * the result does not depend on the order in which threads run.
 *   indptr / indices / eid  the graph's destination-sorted CSR over num_nodes nodes and num_edges slots
 *   nodes       [num_listed] int64 node ids, repeats allowed (the flattened walks of regnn_random_walk); ids outside
 *               [0, num_nodes) are ignored.  max_rows = min(num_nodes, num_listed)
 *   flags       [num_nodes] uint32, all 0 on entry to count; count sets the listed nodes' flags and fill clears them
 *               again, so one map serves every batch of a sampler
 * regnn_induced_subgraph_count:
 *   n_id        [max_rows]: the distinct listed nodes in ascending global id (torch.unique's order); the first
 *               info[REGNN_SAMPLE_INFO_SOURCES] = n_sub entries are written
 *   row_off     [max_rows + 1] uint32: in-CSR offsets of the subgraph (entries past n_sub hold the edge count), the
 *               row_off regnn_block_csr_build reads
 *   src_hist    [max_rows] int32: induced out-edges per subgraph node
 *   info        [REGNN_SAMPLE_INFO_WORDS] int32, zeroed and filled here: SOURCES = n_sub, EDGES = induced edges E_sub,
 *               EMPTY_ROWS, IN_SPLIT from the row lengths, OUT_SPLIT from src_hist; the *_LOOPS words stay 0 (the
 *               subgraph has no self loops of its own)
 * regnn_induced_subgraph_fill (num_rows = n_sub and num_sub_edges = E_sub, read back from info):
 *   src_local / dst_local / edge_id  [num_sub_edges] int64: induced edge e is n_id[src_local[e]] -> n_id[dst_local[e]]
 *               with global edge id edge_id[e], in (destination row, CSR slot) order -- its slot in the subgraph's
 *               in-CSR is e
 * Both calls take the same graph, num_listed and workspace, and the workspace (the flag scan and the table of 256-slot
 * row fragments, max_rows + ceil(num_edges / 256) entries) must be left untouched between them:
 * regnn_induced_subgraph_workspace_bytes(num_nodes, num_edges, num_listed) bytes.  Node ids and num_edges (hence E_sub)
 * must stay below 2^31 - 1. */
size_t regnn_induced_subgraph_workspace_bytes(int64_t num_nodes, int64_t num_edges, int64_t num_listed);
int regnn_induced_subgraph_count(const int32_t* indptr, const int32_t* indices, int64_t num_nodes, int64_t num_edges,
                                 const int64_t* nodes, int64_t num_listed, int split_threshold, uint32_t* flags,
                                 int64_t* n_id, uint32_t* row_off, int32_t* src_hist, int32_t* info, void* workspace,
                                 size_t workspace_bytes, void* stream);
int regnn_induced_subgraph_fill(const int32_t* indptr, const int32_t* indices, const int32_t* eid, int64_t num_nodes,
                                int64_t num_edges, int64_t num_listed, uint32_t* flags, const int64_t* n_id,
                                int64_t num_rows, int64_t num_sub_edges, int64_t* src_local, int64_t* dst_local,
                                int64_t* edge_id, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Grouped per-node-type input projection (model/REGCN.py:36-39, model/REGAT.py:56-58, model/REMixHop.py:89-92:
 * `fc_list[t](features_list[t])` per type + torch.cat; mag/regnn_ns.py:300-326 `group_input`: per type a boolean mask,
 * an index_select of the type's feature table, a Linear and a masked scatter):
 *   out[i,:] = W[type(i)] * x_{type(i)}[row(i),:] + b[type(i)]          for all node types in ONE launch.
 * Rows are visited in type-sorted order: seg_ptr[t] .. seg_ptr[t+1] are the sorted positions of type t (device array,
 * [T+1] int32), perm maps a sorted position to its row of `out` (NULL: rows already type-contiguous), local_idx maps a row
 * of `out` to the row of its type's table (NULL: position inside the segment).  x / ldx / k / w / b are HOST arrays of
 * length num_types (device pointers, leading dimensions, input widths; b or b[t] may be NULL); W[t] is nn.Linear's
 * [n_out, k[t]] row-major.  fp32 in and out; the products run on the tensor pipe as 3 x TF32 (split operands, fp32
 * accumulate), which keeps fp32 GEMM accuracy. */
int regnn_grouped_linear_fwd(int num_types, const float* const* x, const int64_t* ldx, const int* k,
                             const float* const* w, const float* const* b, int n_out, int64_t num_rows,
                             const int32_t* seg_ptr, const int64_t* perm, const int64_t* local_idx, float* out,
                             int64_t ldo, void* stream);

/* Weight / bias gradients of the above: dw_partials[t] is [splits, n_out, k[t]], db_partials[t] (optional) is
 * [splits, n_out]; split s holds the sum over the s-th part of the type's rows (row order, deterministic) -- the caller
 * adds the `splits` partials in order.  dout: dL/d out [num_rows, n_out] (leading dimension ldo). */
int regnn_grouped_linear_bwd(int num_types, const float* const* x, const int64_t* ldx, const int* k, int n_out,
                             int64_t num_rows, const int32_t* seg_ptr, const int64_t* perm, const int64_t* local_idx,
                             const float* dout, int64_t ldo, int splits, float* const* dw_partials,
                             float* const* db_partials, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* REGNN_B200_H_ */
