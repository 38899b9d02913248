/*
 * mpntrack_b200.h -- C ABI of libmpntrack_b200.so (sm_100a CUDA kernels for the
 * MPNTrackSeg neural-message-passing hot path).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name starts with h_ (host);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - tensors are dense row-major; float = fp32, indices as stated (the reference uses
 *     int64 edge_index, the library converts to int32 internally);
 *   - every function returns 0 on success, a negative MPN_E* code otherwise;
 *     mpn_last_error() returns a human-readable message for the calling thread;
 *   - functions are re-entrant and only enqueue work on `stream`, except the ones
 *     documented as "syncs", which must read a device counter to size their output
 *     (the same place where the reference's torch.where / boolean indexing syncs).
 *
 * Each entry point cites the reference interface it replaces (paths relative to the
 * reference's src/mot_neural_solver/).
 */
#ifndef MPNTRACK_B200_H
#define MPNTRACK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPN_OK 0
#define MPN_EINVAL (-1)   /* bad argument (shape, null pointer, unsupported width) */
#define MPN_ECUDA (-2)    /* CUDA runtime error, see mpn_last_error() */
#define MPN_ENOSPC (-3)   /* caller-provided output capacity too small */

const char* mpn_last_error(void);
/* ABI version of the shared object; bumped on any signature change. */
int mpn_abi_version(void);
/* Compute capability major*10+minor of the current device (100 on B200), <0 on error. */
int mpn_device_arch(void);

/* Number of kernel launches this library has issued so far in this process (monotonic). */
long long mpn_launch_count(void);
/* Per-kernel device timing of the message-passing kernels: between _begin and _end every
 * mp_edge_kernel / mp_node_kernel launch is bracketed by CUDA events on its own stream.
 * _end synchronises the device and returns summed milliseconds and launch counts,
 * index 0 = edge kernel, 1 = node kernel. */
int mpn_profile_begin(void);
int mpn_profile_end(double* h_ms /*[2]*/, long long* h_launches /*[2]*/);

/* ------------------------------------------------------------------ graph construction */

/* utils/graph.py:6-37  get_time_valid_conn_ixs(frame_num, max_frame_dist, ..)
 * Pairs (i<j) with 0 < |frame_i - frame_j| <= max_frame_dist (max_frame_dist < 0 means
 * 'max': no upper bound), restricted to nodes of the same window: node_graph_ptr[G+1]
 * gives each window's node range (pass NULL, G=0 for a single window).  Output order:
 * ascending i then ascending j.  Two-phase: _count writes per-row counts and the
 * exclusive scan row_start[N+1] (row_start[N] = total); SYNCS to return *h_total.
 * _fill writes pairs at row_start offsets. */
int mpn_time_valid_pairs_count(const int64_t* frame_num, int64_t num_nodes,
                               const int64_t* node_graph_ptr, int64_t num_graphs,
                               int64_t max_frame_dist, int64_t* row_start /*[N+1]*/,
                               int64_t* h_total, void* stream);
int mpn_time_valid_pairs_fill(const int64_t* frame_num, int64_t num_nodes,
                              const int64_t* node_graph_ptr, int64_t num_graphs,
                              int64_t max_frame_dist, const int64_t* row_start,
                              int64_t* out_row, int64_t* out_col, void* stream);

/* data/mot_graph.py:211, :299-303  F.pairwise_distance(reid[row], reid[col])
 * out[e] = || reid[row[e]] - reid[col[e]] + 1e-6 ||_2, fp32, fixed summation order. */
int mpn_pair_reid_dist(const float* reid, int64_t num_nodes, int64_t dim,
                       const int64_t* row, const int64_t* col, int64_t num_pairs,
                       float* out, void* stream);

/* utils/graph.py:40-87  get_knn_mask(pwise_dist, edge_ixs, num_nodes, top_k_nns, ..,
 *                                    reciprocal_k_nns, symmetric_edges)
 * keep[e] = in_k(row,col) AND/OR in_k(col,row); in_k(i,j) <=> j is among the top_k
 * entries of the ascending, index-stable sort of dense row i (missing pairs = +inf).
 * workspace: num_nodes*num_nodes floats + 2*num_nodes*8 bytes (mpn_knn_mask_workspace). */
int64_t mpn_knn_mask_workspace(int64_t num_nodes);
int mpn_knn_mask(const float* pwise_dist, const int64_t* row, const int64_t* col,
                 int64_t num_edges, int64_t num_nodes, int64_t top_k, int reciprocal,
                 int symmetric_edges, void* workspace, uint8_t* keep, void* stream);

/* Order-preserving compaction of pairs by a keep mask (edge_ixs.T[mask].T,
 * data/mot_graph.py:219; tracker/mpn_tracker.py:111-112).  SYNCS to return *h_kept.
 * scan_ws: (num_edges+1) int64. in/out may not alias. */
int mpn_compact_pairs(const int64_t* row, const int64_t* col, const float* dist,
                      const uint8_t* keep, int64_t num_edges, int64_t* scan_ws,
                      int64_t* out_row, int64_t* out_col, float* out_dist,
                      int64_t* h_kept, void* stream);

/* data/mot_graph.py:223-262 MOTGraph.assign_edge_labels: labels[e] = 1 for directed edges between detections of the
 * same identity (node_ids, -1 = false positive, never linked); closest != 0 ('closest' mode, the shipped default):
 * only the edge to the closest same-identity partner (by node index) in the future and in the past of edge_row[e];
 * closest == 0: 'all'.  workspace: 2 * num_nodes int32.  num_nodes < 2^31 - 1. */
int mpn_assign_edge_labels(const int64_t* edge_row, const int64_t* edge_col, int64_t num_edges,
                           const int64_t* node_ids, int64_t num_nodes, int closest, void* workspace,
                           float* labels, void* stream);

/* utils/graph.py:90-124 compute_edge_feats_dict + data/mot_graph.py:292-312 assembly.
 * For each undirected pair p (row<col) writes the feature row
 *   [dt, dx/hbar, dy/hbar, log(h_col/h_row), log(w_col/w_row), reid_dist]
 * to edge_attr[p] and edge_attr[p + num_pairs] (both directions share the row), and
 * edge_index = [ (row,col) ... , (col,row) ... ]  ([2, 2*num_pairs] int64).
 * frame is given as fp32 seconds numerator: secs = frame_f32 / fps. reid_dist may be
 * NULL (then 5 columns are written, attr_dim must be 5). */
int mpn_edge_feats_assemble(const int64_t* row, const int64_t* col, int64_t num_pairs,
                            const float* frame_f32, const float* bb_height,
                            const float* bb_width, const float* feet_x, const float* feet_y,
                            float fps, const float* reid_dist, int64_t attr_dim,
                            float* edge_attr /*[2P, attr_dim]*/, int64_t* edge_index /*[2,2P]*/,
                            void* stream);

/* Fused, batched edge construction for G independent windows (training-mode semantics of
 * data/mot_graph.py:195-221 = get_time_valid_conn_ixs + F.pairwise_distance + get_knn_mask with
 * symmetric_edges=False + boolean indexing), one host synchronisation in total.
 *   node_graph_ptr [G+1] (device AND host copy): node range of each window; node ids are batch-global.
 *   top_k < 0 keeps every time-valid pair (inference-mode graphs, data/mot_graph.py:209-210).
 * Outputs: kept pairs (row<col) sorted by (row, col) with their ReID distance, and
 * graph_pair_ptr [G+1] (device + host): pair range of each window.  capacity = size of the out arrays
 * (sum over windows of N_g*min(k, N_g) is always enough); MPN_ENOSPC if exceeded.
 * use_tensor_cores != 0 (and dim a multiple of 64, top_k >= 0): the dense distances come from a tcgen05 Gram
 * contraction (fp16 hi/lo split) and only pre-rank; rows whose k-th / (k+1)-th neighbours lie within the error
 * band are recomputed with the exact fp32 formula and re-ranked, and the distances returned for the kept pairs
 * are always the exact ones -- the kept edge set equals the exact path's at every embedding scale (each window is
 * packed under a power-of-two pre-scale, so the band bounds the Gram error).  h_stats (host, may be NULL):
 * [0] = the build that ran: 0 exact fp32 (also after a whole-call exact rerun: values of magnitude >= 65,000 or
 * more flagged rows than scratch slots), 1 dense Gram blocks + row select, 2 thresholded candidate lists; nonzero =
 * tensor cores.
 * [1] = number of rows that needed the exact repair.
 * workspace: mpn_knn_graph_workspace(N, sum_g N_g^2, G) bytes (dense fp32 distance blocks + packed embeddings). */
int64_t mpn_knn_graph_workspace(int64_t num_nodes, int64_t sum_sq_nodes, int64_t num_graphs);
int mpn_knn_graph_pairs(const int64_t* frame_num, const int64_t* node_graph_ptr,
                        const int64_t* h_node_graph_ptr, int64_t num_graphs, const float* reid,
                        int64_t dim, int64_t top_k, int reciprocal, int64_t max_frame_dist,
                        int use_tensor_cores, void* workspace, int64_t capacity, int64_t* out_row,
                        int64_t* out_col, float* out_dist, int64_t* graph_pair_ptr,
                        int64_t* h_graph_pair_ptr, int64_t* h_stats /*[2] or NULL*/, void* stream);

/* ------------------------------------------------------------------ model: layout */

/* Internal edge layout for the fused message-passing kernels ("slots"): directed edges
 * with row<col (the flow_out set, models/mpn.py:85) first, then those with row>col (the
 * flow_in set, models/mpn.py:91), each group sorted by row, original order kept inside a
 * row (stable), so that per-node aggregation is a contiguous, deterministic segment.
 *   slot_row/slot_col [E] int32, slot_edge [E] int32 (slot -> original edge id),
 *   out_ptr/in_ptr [N+1] int32 slot ranges per node; *h_num_out = #edges with row<col.
 * workspace bytes: mpn_edge_layout_workspace(E, N).  SYNCS (one 8-byte read). */
int64_t mpn_edge_layout_workspace(int64_t num_edges, int64_t num_nodes);
int mpn_edge_layout_build(const int64_t* edge_index /*[2,E]*/, int64_t num_edges,
                          int64_t num_nodes, void* workspace, int32_t* slot_row,
                          int32_t* slot_col, int32_t* slot_edge, int32_t* out_ptr,
                          int32_t* in_ptr, int64_t* h_num_out, void* stream);

/* ------------------------------------------------------------------ model: encoders */

/* models/mpn.py:351-352  AdaptiveAvgPool2d((1,1)) + view: x[N,C,HW] -> out[N,C], for `windows` windows at once:
 * window i reads x[i] [n[i],C,HW] and writes the next n[i] rows of out (out [sum n, C]).  x and n are host arrays.
 * The windows whose maps are 16-byte aligned (HW/4 a power of two up to 32) are pooled by one launch per 64
 * windows; the others by one scalar launch each. */
int mpn_avgpool(const float* const* x, const int64_t* n, int64_t windows, int64_t c, int64_t hw, float* out,
                void* stream);

/* models/mlp.py:12-23  one Linear(+ReLU) layer: out[M,O] = act(in[M,K] @ W[O,K]^T + b). */
int mpn_linear(const float* in, int64_t m, int64_t k, const float* w, const float* b,
               int64_t o, int relu, float* out, void* stream);

/* models/mpn.py:355 encoder.node_model for the shipped widths K -> 128 -> 32 (K a multiple of 64) on the
 * tcgen05 tensor cores: x [N,K] (already pooled, 16-byte aligned) -> out [N,32] = ReLU(W1 ReLU(W0 x + b0) + b1),
 * fp16 hi/lo split operands, each row of x, W0, W1 and the hidden layer at its own power-of-two scale, fp32
 * accumulation.  *status != 0: a non-finite value in x or the weights (or an x row beyond 2^73), rerun with
 * mpn_linear.  workspace: mpn_node_encoder_tc_workspace(K) bytes (packed weight image). */
int64_t mpn_node_encoder_tc_workspace(int64_t k0);
int mpn_node_encoder_tc(const float* x, int64_t n, int64_t k0, const float* w0, const float* b0,
                        int64_t hidden, const float* w1, const float* b1, int64_t out_dim,
                        void* workspace, float* out, int32_t* status, void* stream);

/* out[r] = in[idx[r]] for rows of `width` floats (edge_attr[slot_edge] for non-default
 * encoder widths, where the fused edge encoder below does not apply). */
int mpn_gather_rows(const float* in, const int32_t* idx, int64_t rows, int64_t width, float* out,
                    void* stream);

/* models/mpn.py:355 encoder.edge_model on edge_attr rows taken in slot order:
 * e_init[s] = MLP(edge_attr[slot_edge[s]]), widths dims[0..n_layers] (ReLU after every
 * layer whose width != 1).  weights[l] is W_l [dims[l+1], dims[l]], biases[l] [dims[l+1]]
 * (host arrays of device pointers).  Supported: dims[l] <= 32. */
int mpn_edge_encoder(const float* edge_attr, const int32_t* slot_edge, int64_t num_edges,
                     const int32_t* h_dims, int32_t n_layers, const float* const* h_weights,
                     const float* const* h_biases, float* e_init, void* stream);

/* ------------------------------------------------------------------ model: message passing */

/* Weights of the core network, plain nn.Linear layout W[out,in] (device pointers).
 * models/mpn.py:275-317, configs/tracking_cfg.yaml:134-168. */
typedef struct {
  int32_t dn;        /* node latent width (32)  */
  int32_t de;        /* edge latent width (16)  */
  int32_t edge_h;    /* edge MLP hidden (80)    */
  int32_t flow_h;    /* flow MLP hidden (56)    */
  int32_t cls_h;     /* classifier hidden (8)   */
  const float* edge_w0;  const float* edge_b0;   /* [edge_h, 4*dn+2*de]           */
  const float* edge_w1;  const float* edge_b1;   /* [de, edge_h]                  */
  const float* fin_w0;   const float* fin_b0;    /* flow_in  [flow_h, 2*dn+de]    */
  const float* fin_w1;   const float* fin_b1;    /* flow_in  [dn, flow_h]         */
  const float* fout_w0;  const float* fout_b0;   /* flow_out [flow_h, 2*dn+de]    */
  const float* fout_w1;  const float* fout_b1;   /* flow_out [dn, flow_h]         */
  const float* node_w;   const float* node_b;    /* [dn, 2*dn]                    */
  const float* cls_w0;   const float* cls_b0;    /* [cls_h, de]                   */
  const float* cls_w1;   const float* cls_b1;    /* [1, cls_h]                    */
  int32_t node_agg;      /* models/mpn.py:263-273 node_agg_fn: 0 = 'sum' (scatter_add), 1 = 'mean' (scatter_mean: sum /
                            max(count, 1)), 2 = 'max' (scatter_max; messages are post-ReLU, empty segments give 0) */
} mpn_core_weights;

typedef struct {
  int64_t num_nodes, num_edges, num_out;        /* num_out = #slots of the flow_out group */
  const int32_t* slot_row; const int32_t* slot_col; const int32_t* slot_edge;
  const int32_t* out_ptr;  const int32_t* in_ptr;
} mpn_edge_layout;

/* Bytes of scratch mpn_mp_forward needs (node state ping-pong, edge state ping-pong,
 * flow sums, tile partials). */
int64_t mpn_mp_workspace(int64_t num_nodes, int64_t num_edges);

/* models/mpn.py:364-381  the step loop: num_steps x { reattach, MetaLayer.forward
 * (EdgeModel :67-69, TimeAwareNodeModel :83-99), classifier :114 }.
 *   x_init [N,dn], e_init [E,de] (slot order)   -- encoder outputs (models/mpn.py:355-360)
 *   logits [num_class_steps, E] in ORIGINAL edge order: step s (1-based) is written to
 *          row s - first_class_step when s >= first_class_step (models/mpn.py:364,379-381);
 *          num_steps == 0 writes classifier(e_init) to row 0 (models/mpn.py:387-389).
 *   x_out [N,dn], e_out [E,de] (slot order) final latent states (may be NULL). */
int mpn_mp_forward(const mpn_core_weights* h_w, const mpn_edge_layout* h_g,
                   const float* x_init, const float* e_init, int32_t num_steps,
                   int32_t first_class_step, void* workspace, float* logits,
                   float* x_out, float* e_out, void* stream);

/* models/mpn.py:117-137  TimeAwareAttentionModel aggregation: per node, softmax of the edge logits over its
 * future (row<col) resp. past (row>col) neighbours (scatter_softmax, eps 1e-12) and the weighted sum of
 * the neighbours' feature maps z[col] ([N, feat], feat = C*H*W).  logits: [E] in the caller's edge
 * order (one classified step).  flow_in / flow_out: [N, feat]; nodes without neighbours get zeros. */
int mpn_attn_aggregate(const float* z, int64_t num_nodes, int64_t feat, const mpn_edge_layout* h_g,
                       const float* logits, float* flow_in, float* flow_out, void* stream);

/* Backward of mpn_attn_aggregate (training of the mask branch, pl_module/pl_module.py:107-118 back-propagates the
 * segmentation loss through models/mpn.py:117-137): g_in / g_out [N, feat] = d loss / d flow_in, flow_out;
 * perm_c [E] = the slots sorted by column (stable), ptr_c [N+1] its row pointer; w_slot [E] scratch.
 * Outputs: d_z [N, feat] and d_logits [E] (caller's edge order).  Fixed-order reductions. */
int mpn_attn_aggregate_backward(const float* z, int64_t num_nodes, int64_t feat, const mpn_edge_layout* h_g,
                                const float* logits, const float* g_in, const float* g_out, const int32_t* perm_c,
                                const int32_t* ptr_c, float* w_slot, float* d_z, float* d_logits, void* stream);

/* pl_module/pl_module.py:88-105  _compute_loss, tracking term: pos_weight = (#edges - #pos) / #pos (0 if no
 * positive), loss = weight * sum over the classified steps of mean BCEWithLogits(logits[s], labels, pos_weight).
 * logits [steps, E], labels [E] (0/1 floats).  Outputs: loss[1], pos_weight[1] (may be NULL) and, if grad is
 * not NULL, grad[steps, E] = d loss / d logits.  Fixed-order reductions.  ws: mpn_weighted_bce_workspace() bytes. */
int64_t mpn_weighted_bce_workspace(void);
int mpn_weighted_bce(const float* logits, const float* labels, int64_t steps, int64_t num_edges, float weight,
                     void* workspace, float* loss, float* pos_weight, float* grad, void* stream);

/* ------------------------------------------------------------------ training building blocks
 * pl_module/pl_module.py:122-135 (loss.backward(), Adam) for the core network, as deterministic fp32
 * kernels (fixed-order reductions, no float atomics).  The Python layer (mpntrackseg_b200/training.py)
 * composes them into the forward-with-activations and the backward of models/mpn.py:349-381. */

/* C[m,n] = act(op(A) op(B) + bias) (+ C if accumulate).  op(A)(i,k) = trans_a ? a[k*lda+i] : a[i*lda+k],
 * op(B)(k,j) = trans_b ? b[j*ldb+k] : b[k*ldb+j].  mask_a (may be NULL, same indexing as a with ldm): A is
 * multiplied by (mask_a > 0), i.e. the ReLU backward of the tensor that produced the gradient in A. */
int mpn_gemm(const float* a, int64_t lda, int trans_a, const float* mask_a, int64_t ldm, const float* b,
             int64_t ldb, int trans_b, const float* bias, int relu, int accumulate, float* c, int64_t ldc,
             int64_t m, int64_t n, int64_t k, void* stream);
/* out[j] (+)= sum_i a[i*lda+j] * (mask == NULL || mask[i*ldm+j] > 0)   (bias gradients) */
int mpn_colsum(const float* a, int64_t lda, const float* mask, int64_t ldm, int64_t m, int64_t n,
               int accumulate, float* out, void* stream);
/* out[r, col_off : col_off+width] = src[idx ? idx[r] : r, 0:width]   (torch.cat of gathered rows, models/mpn.py:69,86) */
int mpn_gather_cols(const float* src, int64_t lds, int64_t width, const int32_t* idx, int64_t rows, float* out,
                    int64_t ldo, int64_t col_off, void* stream);
/* out[node, col_off+f] (+)= sum over q in [ptr[node], ptr[node+1]) of in[(perm ? perm[q] : q)*ld + in_off + f]
 * in ascending q (scatter_add of models/mpn.py:89,96 and its transposes in the backward pass). */
int mpn_segment_sum(const float* in, int64_t ld, int64_t in_off, int64_t width, const int32_t* ptr,
                    const int32_t* perm, int64_t nodes, int accumulate, float* out, int64_t ldo,
                    int64_t col_off, void* stream);
/* mpn_segment_sum with a choice of reduction (the node_agg_fn of models/mpn.py:263-273): mode 0: sum; 1: mean (0 for an
 * empty segment); 2: max, the first strictly larger value in ascending q (torch_scatter's scatter_max), 0 for an empty
 * segment.  argmax (mode 2, may be NULL): int32 [nodes, width], the input row of each maximum, -1 for an empty
 * segment. */
int mpn_segment_reduce(const float* in, int64_t ld, int64_t in_off, int64_t width, const int32_t* ptr,
                       const int32_t* perm, int64_t nodes, int accumulate, float* out, int64_t ldo,
                       int64_t col_off, int mode, int32_t* argmax, void* stream);
/* Backward of a mean (mode 1) / max (mode 2) mpn_segment_sum without perm, for the slots q in [q0, q1):
 * out[q*ldo + f] = g[row[q]*ldg + f] / (ptr[row[q]+1] - ptr[row[q]])  (mean), or
 * out[q*ldo + f] = argmax[row[q]*width + f] == q ? g[row[q]*ldg + f] : 0  (max: the whole gradient to one argmax). */
int mpn_segment_grad(const float* g, int64_t ldg, const int32_t* row, const int32_t* ptr, const int32_t* argmax,
                     int64_t q0, int64_t q1, int64_t width, int mode, float* out, int64_t ldo, void* stream);
/* Linear -> BatchNorm1d (training mode) -> ReLU [-> Dropout] after the Linear: z [m, n] (row stride ldz) is the Linear
 * output.  Per column the mean and the biased variance over the m rows (two passes, fixed order) go to stats[0:n] and
 * (as 1/sqrt(var + eps)) stats[n:2n] (stats holds 4n floats; the backward uses the rest); running_mean / running_var
 * move by momentum towards the mean and the unbiased variance and *num_batches_tracked grows by 1, as
 * torch.nn.BatchNorm1d does.  y = ReLU(gamma (z - mean) / sqrt(var + eps) + beta), times keep / (1 - p) when p > 0
 * (see mpn_dropout_forward for the mask; mask may be NULL).  m == 1 is an error (MPN_EINVAL); m == 0 only increments
 * *num_batches_tracked. */
int mpn_batchnorm_forward(const float* z, int64_t ldz, int64_t m, int64_t n, const float* gamma, const float* beta,
                          float eps, float momentum, float* running_mean, float* running_var,
                          int64_t* num_batches_tracked, float* stats, float p, uint64_t seed, const int64_t* counter,
                          int call, float* y, int64_t ldy, uint8_t* mask, void* stream);
/* Its backward from dL/dy (g) and the stored y: g' = (y > 0) g gscale (gscale = 1 / (1 - p)),
 * ggamma += sum g' xhat, gbeta += sum g', gz = gamma / sqrt(var + eps) (g' - mean(g') - xhat mean(g' xhat)). */
int mpn_batchnorm_backward(const float* z, int64_t ldz, const float* g, int64_t ldg, const float* y, int64_t ldy,
                           int64_t m, int64_t n, const float* gamma, float* stats, float gscale, float* ggamma,
                           float* gbeta, float* gz, int64_t ldgz, void* stream);
/* In place on a ReLU output y [m, n]: y = y * keep / (1 - p), 0 < p < 1.  keep of element t = r*n + c is a Philox4x32-10
 * draw keyed by seed, with counter (*counter, the number of the training forward) and call (the dropout call within
 * it): independent of the launch configuration.  mask (may be NULL): uint8 [m, n] receives keep. */
int mpn_dropout_forward(float* y, int64_t ldy, int64_t m, int64_t n, float p, uint64_t seed, const int64_t* counter,
                        int call, uint8_t* mask, void* stream);
/* out = y > 0 ? g * scale : 0  (ReLU + dropout backward from the stored output; scale = 1 / (1 - p)) */
int mpn_dropout_backward(const float* g, int64_t ldg, const float* y, int64_t ldy, int64_t m, int64_t n, float scale,
                         float* out, int64_t ldo, void* stream);
/* g[i] = y[i] > 0 ? g[i] : 0 */
int mpn_relu_mask(float* g, const float* y, int64_t n, void* stream);
/* torch.optim.Adam step (configs/tracking_cfg.yaml:6-10: lr 1e-3, weight_decay 1e-4 as L2 term) on flat
 * buffers; grads are multiplied by grad_scale first (1/world_size after a summed all-reduce). */
int mpn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                  void* stream);

/* The same Adam step with the step number kept on the device: *d_step (int64) is incremented first, then used for the
 * bias corrections, so that a captured CUDA graph of a whole training step can be replayed. */
int mpn_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                      float beta1, float beta2, float eps, float weight_decay, int64_t* d_step, float grad_scale,
                      void* stream);

/* Same contract as mpn_mp_forward (1 <= num_steps <= 1000), evaluated on the tcgen05 tensor cores:
 * per 128-edge tile the four dense layers run as kind::f16 MMAs with fp16 hi/lo split operands
 * (hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM; ~22 significant bits per operand).
 * Range: step t runs on operands scaled by 2^-s_t, s_t chosen on the device from the previous step's largest
 * activation and the growth of the node state (exact power-of-two scaling of a piecewise-linear network;
 * s_t = 0 while values stay below 64), so node states far beyond the fp16 range stay on this path.
 * *status (device int32) is set non-zero only if a value still left the fp16 range (bit 1: one-step growth beyond the
 * 1024x headroom) or a step ran at s_t > 17, where the absolute resolution 2^(s_t-34) no longer resolves rows of
 * order 1, e.g. a quiet window batched with a loud one (bit 2); the outputs are then invalid and the caller must
 * rerun with mpn_mp_forward (fp32 kernels).
 * workspace bytes: mpn_mp_tc_workspace(N, E). */
int64_t mpn_mp_tc_workspace(int64_t num_nodes, int64_t num_edges);
int mpn_mp_forward_tc(const mpn_core_weights* h_w, const mpn_edge_layout* h_g, const float* x_init,
                      const float* e_init, int32_t num_steps, int32_t first_class_step,
                      void* workspace, float* logits, float* x_out, float* e_out, int32_t* status,
                      void* stream);

/* ------------------------------------------------------------------ rounding and identity assignment (after the path)
 * The sequence graph at this point is the undirected, pruned graph of utils/graph.py:165-207: one entry per pair,
 * row = earlier node.  Integer / comparison work only; results are deterministic and equal the reference's. */

/* utils/evaluation.py:370-414 compute_constr_satisfaction_rate: flow_out[v] = sum of edges_out over edges leaving v
 * (row == v), flow_in[v] over edges entering v (col == v), divided by 2 when undirected_edges != 0 (every pair stored
 * in both directions; pairs are then ordered here).  edges_out must be BINARISED (exactly 0 or 1; MPN_EINVAL otherwise).
 * flow_in / flow_out [N] may be NULL.  h_counts (host) = {#nodes with flow_in > 1, #nodes with flow_out > 1,
 * #constraints = #distinct rows + #distinct cols}; the rate is 1 - (h[0] + h[1]) / h[2].  SYNCS.
 * workspace: mpn_rounding_workspace(N) bytes. */
int64_t mpn_rounding_workspace(int64_t num_nodes);
int mpn_constr_satisfaction(const int64_t* row, const int64_t* col, const float* edges_out, int64_t num_edges,
                            int64_t num_nodes, int undirected_edges, void* workspace, float* flow_in, float* flow_out,
                            int64_t* h_counts /*[3]*/, void* stream);

/* tracker/projectors.py:11-67 GreedyProjector.project: round_preds = edge_preds > 0.5, then every violated outgoing
 * constraint (flow_out > 1), and after those every still-violated incoming one, keeps its active edge with the largest
 * prediction (the first one on ties) and switches the others off.  h_counts as above, for the INITIAL rounding
 * (projectors.py:22-25).  On return no node has more than one active edge per direction.  SYNCS. */
int mpn_greedy_project(const int64_t* row, const int64_t* col, const float* edge_preds, int64_t num_edges,
                       int64_t num_nodes, void* workspace, float* round_preds, int64_t* h_counts /*[3]*/, void* stream);

/* tracker/mpn_tracker.py:231-248 _assign_ped_ids: labels[v] = index of v's connected component in the graph of the
 * edges with edge_vals == 1, components numbered by their smallest node (scipy.sparse.csgraph.connected_components,
 * directed=False).  *h_num_components: number of components.  SYNCS.
 * workspace: mpn_connected_components_workspace(N) bytes. */
int64_t mpn_connected_components_workspace(int64_t num_nodes);
int mpn_connected_components(const int64_t* row, const int64_t* col, const float* edge_vals, int64_t num_edges,
                             int64_t num_nodes, void* workspace, int64_t* labels, int64_t* h_num_components, void* stream);

/* ------------------------------------------------------------------ MOTS output (after identity assignment)
 * tracker/mpn_tracker.py:267-298 + :398-417: each node's mask pasted into its frame (torchvision's
 * paste_masks_in_image), one owner per pixel within a frame, pycocotools RLE of every mask.  masks [N, M, M] fp32
 * probabilities; boxes [N, 4] int64 (x0, y0, x1, y1) = torchvision's expand_boxes(box, (M + 2 padding) / M) truncated
 * to integers (the caller computes them in its own dtype); the image is height x width with height * width <= 2^31 - 1.
 * p_i(y, x) = the zero-padded (M + 2 padding)^2 mask resized to h = max(y1 - y0 + 1, 1) by w = max(x1 - x0 + 1, 1)
 * with ATen's bilinear interpolation (align_corners = False), read at (y - y0, x - x0) inside the box clamped to the
 * image, 0 elsewhere; evaluated in double. */

/* out [N, H, W] fp32 = p_i(y, x): the dense paste, torchvision's paste_masks_in_image. */
int mpn_paste_masks(const float* masks, int64_t num_nodes, int64_t mask_size, int32_t padding, const int64_t* boxes,
                    int64_t height, int64_t width, float* out, void* stream);

/* Run-length encoding of the masks.  Within a frame (frame [N] int64, non-decreasing) pixel (y, x) belongs to the
 * node with the largest p_i(y, x), ties to the lower node index, NaN counting as -inf; node i's mask is the set of
 * pixels it owns where p_i > threshold.  Its RLE is pycocotools' rleEncode of the column-major H x W image (counts
 * start with the zeros, possibly 0) and its string rleToString's.  A node with an empty mask has no counts and no
 * characters.  Two phases, like mpn_time_valid_pairs_count / _fill:
 * _count writes area [N] (pixels of the mask) and the exclusive scans cnt_ptr / char_ptr [N+1] of each node's number of
 * counts and of characters; h_totals (host) = {total counts, total characters}.  MPN_EINVAL if frame decreases.  SYNCS.
 * _fill writes the int32 counts at cnt_ptr offsets and the characters (no terminator) at char_ptr offsets.
 * workspace: mpn_mots_rle_workspace(N) bytes. */
int64_t mpn_mots_rle_workspace(int64_t num_nodes);
int mpn_mots_rle_count(const float* masks, int64_t num_nodes, int64_t mask_size, int32_t padding, const int64_t* boxes,
                       const int64_t* frame, int64_t height, int64_t width, double threshold, void* workspace,
                       int64_t* area, int64_t* cnt_ptr /*[N+1]*/, int64_t* char_ptr /*[N+1]*/, int64_t* h_totals /*[2]*/,
                       void* stream);
int mpn_mots_rle_fill(const float* masks, int64_t num_nodes, int64_t mask_size, int32_t padding, const int64_t* boxes,
                      const int64_t* frame, int64_t height, int64_t width, double threshold, const int64_t* cnt_ptr,
                      const int64_t* char_ptr, int32_t* counts, uint8_t* chars, void* stream);

/* Diagnostics of the last mpn_mp_forward_tc run on `workspace` (same n, e): the scale exponents s_t and the maxima
 * they were derived from, entries [0, num_steps + 2) indexed by step (1-based).  h_* are HOST arrays and may be
 * NULL.  SYNCS. */
int mpn_mp_tc_read_schedule(const void* workspace, int64_t num_nodes, int64_t num_edges, int32_t num_steps,
                            int32_t* h_sched, float* h_amax, float* h_xmax, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPNTRACK_B200_H */
