/* dfw_b200.h - C ABI of the B200-native GraphSAGE hot path (libdfw_b200.so).
 *
 * Drop-in boundary for Deep-FEM-UAV-Wing's GNN surrogate.  The reference has no FFI of its
 * own: its boundary is the Python nn.Module contract
 *     GraphSAGEModel.forward(x, edge_index, batch=None)   src/deep_fem_uav_wing/gnn/model.py:74-99
 *     SAGEConv(H, H)(h, edge_index)                        model.py:63,90  (torch_geometric, un-vendored)
 *     MaskedMSELoss.forward(pred, target, mask)            model.py:126-153
 * and everything below sits UNDER a re-created gnn/model.py with the same names.  Each
 * entry point cites the reference expression it replaces.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no torch types.  All pointers are DEVICE pointers
 *    on the current device, contiguous row-major, 16-byte aligned.
 *  - The caller allocates everything (outputs and workspaces, sizes via *_ws_bytes); the
 *    library never allocates or frees device memory and keeps no pointer after return.
 *  - Every call takes the CUDA stream to launch on and is asynchronous with respect to the
 *    host.  Re-entrant, no global mutable state, safe to call from torch's autograd threads.
 *  - Return value: 0 = ok, non-zero = error; dfw_last_error() gives the thread-local message.
 *  - dtype: activations/weights are DFW_F32 or DFW_BF16; bias, LayerNorm affine, statistics,
 *    inv_deg and all accumulation are fp32.
 *  - CUDA-only: there is no CPU path behind these symbols.
 */
#ifndef DFW_B200_H
#define DFW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* dfw_stream_t;

enum { DFW_F32 = 0, DFW_BF16 = 1 };

/* epilogue / behaviour flags */
enum {
    DFW_EP_RELU = 1,      /* ReLU after (optional) LayerNorm                    model.py:92, :54,:56,:69 */
    DFW_EP_LAYERNORM = 2, /* row LayerNorm(eps, gamma, beta) before ReLU        model.py:64,91          */
    DFW_EP_RESIDUAL = 4,  /* out = residual + epilogue(...)                     model.py:95             */
    DFW_EP_DROPOUT = 8,   /* inverted dropout (train only)                      model.py:93, :70        */
    DFW_EP_SEED_IS_PTR = 16, /* `seed` is a DEVICE pointer to one uint64 (read by the kernel): lets a captured CUDA graph
                             draw a fresh dropout mask on every replay */
    DFW_EP_TRANSPOSE_W = 32, /* dfw_linear_fwd only: w1/w2 are given as [k, Hout] row-major (the FORWARD layer's weights,
                             used by its input gradient g W instead of x W^T); the transposition rides in the weight
                             preparation launch.  Needs a tensor-core eligible shape: ask dfw_linear_tc_eligible */
    DFW_EP_OUT_BF16 = 64  /* dfw_linear_fwd with dtype = DFW_F32, single operand, k1 <= 16, no LayerNorm / dropout / residual
                             (the encoder's first linear, model.py:53): `out` is written as bf16 - the fp32 result rounded to
                             nearest even at the store, i.e. what dfw_cast would make of it, without the fp32 round trip */
};

const char* dfw_last_error(void);
int dfw_abi_version(void);

/* ------------------------------------------------------------------------------------------
 * (a) edge_index -> CSR.   Replaces PyG's per-call gather/scatter bookkeeping behind
 *     SAGEConv.forward (call site model.py:90; edge_index int64 [2,E] from gnn/dataset.py:63).
 *     by_src = 0: rows = destination (edge_index[1]), col = source, sorted by (dst, src, edge id)
 *                 == numpy.lexsort((src, dst)); used by the forward mean.
 *     by_src = 1: rows = source, col = destination (transposed CSR) for the backward gather.
 *     rowptr int32 [N+1], col int32 [E], perm int32 [E] (may be NULL), inv_deg fp32 [N] (may be
 *     NULL) = 1/max(deg,1).  status int32 [2] (device): [0] = number of out-of-range endpoints
 *     (the CSR is invalid if non-zero), [1] = max degree.  Requires E, N < 2^31.
 * ---------------------------------------------------------------------------------------- */
size_t dfw_csr_ws_bytes(int64_t E, int64_t N);
int dfw_csr_build(const int64_t* edge_index, int64_t E, int64_t N, int by_src,
                  int32_t* rowptr, int32_t* col, int32_t* perm, float* inv_deg,
                  int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream);
/*     Transposed CSR (rows = source) for the backward gather, given the CSR by destination that dfw_csr_build made of
 *     the same edge_index.  Mesh graphs hold both directions of every edge (dataset.py:55-58); the call verifies that
 *     on the device (duplicate-free rows and a mirror for every edge) and then COPIES the CSR instead of building one;
 *     otherwise it runs the general build (by_src = 1).  No host synchronisation either way (capturable).
 *     status int32 [3]: [0], [1] as above for the general build, [2] = 1 when the graph was NOT symmetric.
 *     ws: dfw_csr_ws_bytes(E, N). */
int dfw_csr_transpose(const int64_t* edge_index, int64_t E, int64_t N, const int32_t* rowptr, const int32_t* col,
                      int32_t* rowptr_t, int32_t* col_t, int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (f1) graph construction from triangle faces (SURVEY 8f-1): _faces_to_edge_index (dataset.py:26-63) on the device.
 *     faces int64 [F,3] of node IDS.  sorted_ids (nullable) = the node ids in ascending order, id_perm (nullable) =
 *     index of sorted_ids[k] in the caller's node order (NULL = identity): the device form of node_id_to_idx
 *     (dataset.py:106).  sorted_ids == NULL: faces already hold 0-based indices.  Faces holding an unknown id are
 *     skipped (dataset.py:43-46); undirected edges are de-duplicated and emitted in both directions
 *     (dataset.py:49-58; a self pair (i,i) appears twice, as there).
 *     Outputs: CSR by destination rowptr int32 [N+1], col int32 [capacity 6F], inv_deg fp32 [N] (nullable),
 *     edge_index int64 [2, 6F] (nullable; row 0 = source, row 1 = destination, canonical (dst,src) order, the first
 *     *num_edges columns of each row are valid), num_edges int64 (device), status int32 [3] (device):
 *     [0] = placeholder pairs dropped (6 per skipped face), [1] = max degree, [2] = skipped faces.
 *     The graph is symmetric, so the same CSR serves the backward gather.
 * ---------------------------------------------------------------------------------------- */
size_t dfw_faces_ws_bytes(int64_t F, int64_t N);
int dfw_faces_to_csr(const int64_t* faces, int64_t F, const int64_t* sorted_ids, const int64_t* id_perm, int64_t N,
                     int32_t* rowptr, int32_t* col, float* inv_deg, int64_t* edge_index, int64_t* num_edges,
                     int32_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream);

/* Node features of build_graph_data (dataset.py:129-151) on the device:
 *   x [N,10] fp32 = [(pos - min)/range | normal/|normal| | global_params4], y [N,1] fp32 = log1p(stress) (nullable).
 *   pos, normal fp32 [N,3], stress fp32 [N] on the device; global_params4 = 4 HOST floats (dataset.py:122-127).
 *   x is bit-identical to the reference's numpy float32 arithmetic; y may differ in the last ulp (log1pf). */
size_t dfw_node_features_ws_bytes(int64_t N);
int dfw_node_features(const float* pos, const float* normal, const float* stress, const float* global_params4,
                      int normalize_pos, int log_scale, float* x, float* y, int64_t N, void* ws, size_t ws_bytes,
                      dfw_stream_t stream);
/*     Batched form for the design-screening loop (inference_gnn.py:380-398 handles one case at a time): B cases concatenated,
 *     rows case_ptr[b] .. case_ptr[b+1] (device int64 [B+1]), global_params device fp32 [B,4] (already scaled, dataset.py:122-127),
 *     per-case min-max normalisation.  Bit-identical to B calls of dfw_node_features.  max_case_rows sizes the grid. */
size_t dfw_node_features_batched_ws_bytes(int64_t B);
int dfw_node_features_batched(const float* pos, const float* normal, const float* stress, const float* global_params,
                              const int64_t* case_ptr, int64_t B, int64_t max_case_rows, int normalize_pos, int log_scale,
                              float* x, float* y, void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (b) deterministic segmented neighbour aggregation (no atomics):
 *        out[i,:] = (addend ? addend[i,:] : 0) + (row_scale ? row_scale[i] : 1) * sum_{k in row i} x[col[k],:]
 *     row_scale = inv_deg  -> PyG mean aggregation (SAGEConv aggr='mean', model.py:63);
 *     row_scale = NULL with the transposed CSR -> backward of that mean.
 *     x, addend, out: [N,H] dtype; fp32 accumulation in CSR order.  H*sizeof(dtype) % 16 == 0.
 * ---------------------------------------------------------------------------------------- */
int dfw_sage_aggregate(const int32_t* rowptr, const int32_t* col, const float* row_scale,
                       const void* x, const void* addend, void* out,
                       int64_t N, int64_t E, int64_t H, int dtype, dfw_stream_t stream);

/* Same gather with the scale on the SOURCE side:  out[i,:] = sum_{k in row i} src_scale[col[k]] * x[col[k],:]
 * With the transposed CSR and src_scale = inv_deg this is A^T D^-1 g, the adjoint of the mean aggregation applied to
 * the gradient BEFORE the weight contraction:  dL/dh = (A^T D^-1 g_y) lin_l.weight + g_y lin_r.weight  - one
 * aggregation of g_y followed by one fused two-operand linear, instead of two contractions and an aggregation
 * (autograd of SAGEConv, reference call site model.py:90 / loss.backward() train_gnn.py:57). */
int dfw_sage_aggregate_scaled(const int32_t* rowptr, const int32_t* col, const float* src_scale,
                              const void* x, void* out,
                              int64_t N, int64_t E, int64_t H, int dtype, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (b') the same mean / sum aggregation for bf16 rows on the tensor cores (block-sparse product; refined meshes, BASELINE.json
 *     config 4).  Replaces the same PyG expression as dfw_sage_aggregate (index_select + scatter_add_ + divide behind
 *     SAGEConv(aggr='mean'), call site model.py:90).  Rows are cut into blocks of 128 consecutive rows; a one-time PLAN of the
 *     CSR lists per block its source rows (plan_src: the block's own 128 rows first - the kernel fetches those as plain TMA
 *     tiles - then the distinct other sources ascending, padded to multiples of 64) and one 16-bit entry per distinct
 *     (source, row) pair - (multiplicity-1) << 13 | row << 6 | slot % 64, ordered by 64-source chunk (plan_slot) - with the
 *     chunk pointers in the block record (plan_rec: S, #entries, cptr[...]); per block  OUT[128,H] = ADJ[128,S] . X[S,H]
 *     runs as tcgen05.mma with fp32 accumulation (ADJ = edge multiplicities: exact products), row_scale in the epilogue.
 *     Result = the CSR-order fp32 sum up to the association order of the fp32 additions (<= 1 bf16 ulp after rounding).
 *
 *     dfw_agg_plan_sizes: array lengths for a graph of N rows / E edges: blk_meta int32 [4*nblocks], plan_src int32 [src_cap],
 *       plan_rec uint16 [136*nblocks], plan_slot uint16 [slot_cap]; ws of dfw_agg_plan_build: 8 bytes per block.
 *     dfw_agg_plan_build: status uint64 [2] (device): [0] = largest number of edges in a block - the plan is USABLE only if
 *       it is <= dfw_agg_plan_max_block_edges() (an edge repeated more than 8 times also pushes it above); [1] = total number of staged rows (sum of S over the blocks: the locality
 *       measure, staged rows per output row = [1] / N).  No host synchronisation.
 *     dfw_sage_aggregate_tc: x, out bf16 [N,H], H in {64,128,256}; row_scale fp32 [N] (inv_deg: mean) or NULL (sum).
 *       Rectangular use (partitioned meshes): `col` may name sources >= N - x then has more than N rows (the N destination rows first,
 *       halo rows behind them); every source outside a block's own 128 rows is staged as a halo row, wherever it lives.
 * ---------------------------------------------------------------------------------------- */
int dfw_agg_plan_sizes(int64_t N, int64_t E, int64_t* nblocks, int64_t* src_cap, int64_t* slot_cap);
int dfw_agg_plan_max_block_edges(void);
int dfw_agg_plan_build(const int32_t* rowptr, const int32_t* col, int64_t N, int64_t E,
                       int32_t* blk_meta, int32_t* plan_src, uint16_t* plan_rec, uint16_t* plan_slot,
                       uint64_t* status, void* ws, size_t ws_bytes, dfw_stream_t stream);
int dfw_sage_aggregate_tc(const int32_t* blk_meta, const int32_t* plan_src, const uint16_t* plan_rec, const uint16_t* plan_slot,
                          const float* row_scale, const void* x, void* out,
                          int64_t N, int64_t H, int dtype, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (c) fused node-wise linear:
 *        y   = a1 . w1^T (+ a2 . w2^T) (+ bias)                       [N,Hout]
 *        out = (residual +) dropout(relu(layernorm(y)))               per `flags`
 *     SAGEConv: a1 = mean-aggregate, w1 = lin_l.weight, bias = lin_l.bias, a2 = h,
 *     w2 = lin_r.weight (model.py:90), epilogue = model.py:91-95.  Encoder/decoder linears
 *     (model.py:52-57,67-72): a2 = NULL.  a1 [N,k1], w1 [Hout,k1], a2 [N,k2], w2 [Hout,k2].
 *     pre_out (nullable) receives y (saved for backward); ln_stats (nullable) receives
 *     (mean, rstd) per row [N,2].  rowdot_w (nullable, fp32 [Hout]) with rowdot_out fp32 [N]:
 *     rowdot_out[i] = sum_c out[i,c]*rowdot_w[c] + *rowdot_b  (decoder's Linear(64,1), model.py:71;
 *     rowdot_b is a device pointer to one fp32, nullable = 0)
 *     and `out` may then be NULL.  Dropout keep-mask is a pure function of
 *     (seed, row*Hout+col): the backward regenerates it.
 * ---------------------------------------------------------------------------------------- */
/*     Tensor-core path (tcgen05/TMEM/TMA; bf16 kind::f16, fp32 as error-compensated 3xTF32) is taken when
 *     16 <= Hout <= 256, Hout % 16 == 0, k*sizeof(dtype) % 16 == 0 and `ws` holds dfw_linear_ws_bytes();
 *     other shapes (e.g. the encoder's K = 10) run the exact-fp32 SIMT kernel.  ws may be NULL (SIMT). */
size_t dfw_linear_ws_bytes(int64_t Hout, int64_t k1, int64_t k2, int dtype);
/*     1 when (N, Hout, k1, k2, dtype) takes the tensor-core path given 16-byte aligned operands and a workspace
 *     (needed before asking for DFW_EP_TRANSPOSE_W); no CUDA call. */
int dfw_linear_tc_eligible(int64_t N, int64_t Hout, int64_t k1, int64_t k2, int dtype);
int dfw_linear_fwd(const void* a1, const void* w1, int64_t k1,
                   const void* a2, const void* w2, int64_t k2,
                   const float* bias, const float* ln_gamma, const float* ln_beta, float ln_eps,
                   const void* residual, float dropout_p, uint64_t seed,
                   void* out, void* pre_out, float* ln_stats,
                   const float* rowdot_w, const float* rowdot_b, float* rowdot_out,
                   int64_t N, int64_t Hout, int flags, int dtype,
                   void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (d1) backward of the epilogue of (c): given g_out = dL/d out, produce g_y = dL/d y.
 *      Recomputes xhat/relu mask from pre_out + ln_stats and the dropout mask from seed.
 *      Without DFW_EP_LAYERNORM, `act` (the saved forward OUTPUT: post-ReLU and post-dropout) gives the ReLU mask and the row-dot operand.
 *      dgamma/dbeta fp32 [Hout] (LayerNorm only).  ws: dfw_epilogue_bwd_ws_bytes.
 *      rowdot variant: g_rowdot fp32 [N] (dL/d rowdot_out) replaces g_out, and
 *      d_rowdot_w [Hout], d_rowdot_b [1] are produced.  d_bias (nullable, fp32 [Hout]) receives the column sums
 *      of g_y, i.e. the bias gradient of the linear that produced y (saves a pass in (d3)).
 * ---------------------------------------------------------------------------------------- */
size_t dfw_epilogue_bwd_ws_bytes(int64_t N, int64_t Hout);
int dfw_epilogue_bwd(const void* g_out, const float* g_rowdot, const float* rowdot_w,
                     const void* pre_out, const float* ln_stats, const void* act,
                     const float* ln_gamma, const float* ln_beta,
                     float dropout_p, uint64_t seed,
                     void* g_y, float* dgamma, float* dbeta, float* d_rowdot_w, float* d_rowdot_b, float* d_bias,
                     int64_t N, int64_t Hout, int flags, int dtype,
                     void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (d2) input gradients of (c):   g_a = (row_scale ? row_scale[i] : 1) * (g_y . w) (+ addend)
 *      g_y [N,Hout], w [Hout,K] -> g_a [N,K].  For SAGEConv: w = lin_l.weight with
 *      row_scale = inv_deg (then (b) over the transposed CSR finishes the mean's backward), and
 *      w = lin_r.weight with addend = the residual-path gradient.
 * ---------------------------------------------------------------------------------------- */
int dfw_linear_bwd_input(const void* g_y, const void* w, const float* row_scale, const void* addend,
                         void* g_a, int64_t N, int64_t Hout, int64_t K, int dtype,
                         void* ws /* dfw_linear_ws_bytes(K, Hout, 0, dtype), nullable */, size_t ws_bytes,
                         dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (d3) weight gradients of (c):  dW1 = g_y^T . a1  [Hout,k1], dW2 = g_y^T . a2 [Hout,k2],
 *      dbias = column sums of g_y [Hout] (nullable).  fp32 outputs.  Deterministic split over
 *      nodes + fixed-order second pass (no float atomics).  `accumulate` != 0 adds into dW/dbias.
 * ---------------------------------------------------------------------------------------- */
size_t dfw_linear_bwd_weight_ws_bytes(int64_t N, int64_t Hout, int64_t k1, int64_t k2);
int dfw_linear_bwd_weight(const void* g_y, const void* a1, int64_t k1, const void* a2, int64_t k2,
                          float* dw1, float* dw2, float* dbias,
                          int64_t N, int64_t Hout, int dtype, int accumulate,
                          void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (b+c) / (d) One-call SAGE layer (SURVEY 8b) - the launch sequences of the entry points above behind one call each,
 *      for hosts that drive a whole layer of   h' = h + dropout(relu(LayerNorm(lin_l(mean_j h_j) + lin_r(h))))
 *      (model.py:90-95) without a Python autograd tape.  Bit-identical to calling the pieces.
 *   fwd: agg [N,Hin] (the mean aggregate, saved for the backward), pre_out / ln_stats (nullable, saved for the backward),
 *        out [N,Hout].  flags: DFW_EP_LAYERNORM | DFW_EP_RELU | DFW_EP_DROPOUT [| DFW_EP_SEED_IS_PTR] | DFW_EP_RESIDUAL
 *        (residual = x, needs Hin == Hout), or 0 for a bare SAGEConv.  w_l, w_r [Hout,Hin] in the compute dtype.
 *   bwd: given g_out = dL/d out, the tensors the forward saved and the transposed CSR (dfw_csr_transpose):
 *        dw_l, dw_r fp32 [Hout,Hin], db_l fp32 [Hout] (nullable), dgamma/dbeta fp32 [Hout] (LayerNorm tail),
 *        g_x [N,Hin] (nullable: first layer).  flags as in the forward.  The input gradient takes the tensor-core
 *        contraction on the forward's weights, so (Hin, Hout) must satisfy dfw_linear_tc_eligible(N, Hin, Hout, Hout).
 * ---------------------------------------------------------------------------------------- */
size_t dfw_sage_layer_fwd_ws_bytes(int64_t N, int64_t Hin, int64_t Hout, int dtype);
int dfw_sage_layer_fwd(const int32_t* rowptr, const int32_t* col, const float* inv_deg, const void* x,
                       const void* w_l, const float* b_l, const void* w_r,
                       const float* ln_gamma, const float* ln_beta, float ln_eps, float dropout_p, uint64_t seed, int flags,
                       void* agg, void* pre_out, float* ln_stats, void* out,
                       int64_t N, int64_t E, int64_t Hin, int64_t Hout, int dtype,
                       void* ws, size_t ws_bytes, dfw_stream_t stream);
size_t dfw_sage_layer_bwd_ws_bytes(int64_t N, int64_t Hin, int64_t Hout, int dtype, int want_input_grad);
int dfw_sage_layer_bwd(const int32_t* rowptr_t, const int32_t* col_t, const float* inv_deg, const void* x, const void* agg,
                       const void* pre_out, const float* ln_stats, const void* w_l, const void* w_r,
                       const float* ln_gamma, const float* ln_beta, const void* g_out, float dropout_p, uint64_t seed, int flags,
                       void* g_x, float* dw_l, float* db_l, float* dw_r, float* dgamma, float* dbeta,
                       int64_t N, int64_t E, int64_t Hin, int64_t Hout, int dtype,
                       void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * One-call encoder / decoder MLP (SURVEY 8b) - the launch sequences of (c), (d1)-(d3) behind one call each.
 *   DFW_MLP2_ENCODER (model.py:52-57): hidden = relu(x W1^T + b1) [N,Hmid], out = relu(hidden W2^T + b2) [N,Hout];
 *        w2 [Hout,Hmid] in the compute dtype, b2 fp32 [Hout].
 *   DFW_MLP2_DECODER (model.py:67-72, out_channels = 1): hidden = dropout(relu(x W1^T + b1)) [N,Hmid] (nullable at
 *        inference), out = hidden . w2 + b2 as fp32 [N]; w2 fp32 [Hmid], b2 fp32 [1] device pointer (nullable); Hout = 1.
 *   bwd: g_out = dL/d out ([N,Hout] compute dtype / fp32 [N]); `out` = the encoder's saved output (ReLU mask; NULL for the
 *        decoder); dw1 fp32 [Hmid,K], db1 fp32 [Hmid] (nullable), dw2 fp32 [Hout,Hmid] / [Hmid], db2 fp32 [Hout] / [1]
 *        (nullable), g_x [N,K] (nullable).  flags: DFW_EP_SEED_IS_PTR or 0.
 * ---------------------------------------------------------------------------------------- */
enum { DFW_MLP2_ENCODER = 0, DFW_MLP2_DECODER = 1 };
size_t dfw_mlp2_fwd_ws_bytes(int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype);
int dfw_mlp2_fwd(const void* x, const void* w1, const float* b1, const void* w2, const float* b2,
                 float dropout_p, uint64_t seed, int flags, int mode, void* hidden, void* out,
                 int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype,
                 void* ws, size_t ws_bytes, dfw_stream_t stream);
size_t dfw_mlp2_bwd_ws_bytes(int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype, int mode, int want_input_grad);
int dfw_mlp2_bwd(const void* x, const void* hidden, const void* out, const void* w1, const void* w2, const void* g_out,
                 float dropout_p, uint64_t seed, int flags, int mode,
                 void* g_x, float* dw1, float* db1, float* dw2, float* db2,
                 int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype,
                 void* ws, size_t ws_bytes, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Masked MSE (model.py:126-153) without boolean indexing / host sync.
 *   result fp32 [2]: [0] = loss (mean: sum/max(count,1); sum: sum), [1] = number of selected
 *   elements.  mask uint8 [N] (nullable = all rows).  pred/target fp32 or bf16 [N,C].
 *   bwd: g_pred = g_loss * 2 (pred-target) * mask / (mean ? max(count,1) : 1).
 * ---------------------------------------------------------------------------------------- */
size_t dfw_masked_mse_ws_bytes(int64_t N, int64_t C);
int dfw_masked_mse_fwd(const void* pred, const void* target, const uint8_t* mask, int64_t N, int64_t C,
                       int reduction_mean, int dtype, float* result, void* ws, size_t ws_bytes,
                       dfw_stream_t stream);
int dfw_masked_mse_bwd(const void* pred, const void* target, const uint8_t* mask, const float* result,
                       const float* g_loss, int64_t N, int64_t C, int reduction_mean, int dtype,
                       void* g_pred, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Evaluation metrics on the device (SURVEY 8f-2): compute_metrics (model.py:156-216) without the full
 * D2H copies of model.py:173-179.  result (device, 8 doubles) =
 *   [mae, rmse, max_error, count] over all N*C elements, then the same over rows with mask[row] != 0;
 * log_scale != 0 applies expm1 to pred and target first (model.py:184-185); an empty subset reports zeros
 * (model.py:194-195); mask == NULL makes both halves equal (model.py:207-210).  Deterministic.
 * ---------------------------------------------------------------------------------------- */
size_t dfw_stress_metrics_ws_bytes(int64_t N, int64_t C);
int dfw_stress_metrics(const void* pred, const void* target, const uint8_t* mask, int64_t N, int64_t C,
                       int log_scale, int dtype, double* result, void* ws, size_t ws_bytes,
                       dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Design screening (BASELINE.json config 5): what a design that has not been through FEM needs on the device.
 *
 * (s1) Area-weighted vertex normals of a triangulated surface: the normal block of the reference's fem.py:390-424
 *     (restated at synth.py:146-151)
 *         fn = cross(p1 - p0, p2 - p0);  normal[v] = sum over the incidences (f, k) with faces[f, k] == v of fn[f]
 *     pos fp32 [N,3], faces int64 [F,3] of 0-based rows (several cases concatenated: rows of the concatenation).
 *     Out: normal fp32 [N,3] (0 for a vertex without a face; dfw_node_features maps |n| < 1e-8 to a zero feature),
 *     status int32 [1] (device) = faces skipped because an index was outside [0, N).  A face naming a vertex twice
 *     contributes twice, as with numpy.bincount.
 *     Determinism: fp32 sums in ascending incidence order 3f + k (the vertex -> incidence lists come from the canonical
 *     CSR build of dfw_csr_build), no float atomics: bitwise identical run to run, and a vertex reads only its own faces,
 *     so how cases are batched into one call cannot change it.  No host synchronisation.  Requires 3F, N < 2^31.
 * ---------------------------------------------------------------------------------------- */
size_t dfw_vertex_normals_ws_bytes(int64_t F, int64_t N);
int dfw_vertex_normals(const float* pos, int64_t N, const int64_t* faces, int64_t F, float* normal, int32_t* status,
                       void* ws, size_t ws_bytes, dfw_stream_t stream);

/* (s2) Per-case stress summary: a segmented reduction of the model output over case_ptr (device int64 [B+1],
 *     non-decreasing from 0 to N), one record per case - what a screening run ranks designs by, without bringing the
 *     prediction back to the host (the reference's inference_gnn.py copies it whole, per case).
 *     pred [N] (or [N,1]) in `dtype` holds log1p(stress) when log_scale != 0 (stress = expm1f(pred) in fp32, as in
 *     dfw_stress_metrics), pos fp32 [N,3].  Screened rows: mask[row] != 0 when mask (uint8 [N]) is given, else
 *     pos_y > root_band * (max_y - min_y) of the row's own case (fp64 comparison) - the rule behind the dataset's loss_mask
 *     (fem.py:637-640, restated at synth.py:154-155).
 *     out float64 [B,8]: [0] rows, [1] screened rows, [2] max stress over the screened rows, [3] row of that maximum within
 *     the case (lowest row on ties; -1 when none), [4] mean stress over the screened rows, [5] max stress over all rows,
 *     [6] screened rows with stress > allowable_pa (allowable_pa <= 0: none counted), [7] rows whose stress is not finite.
 *     Non-finite stresses are counted in [7] only: they take no part in [2]-[6].  An empty set reports 0 in [2], [4], [5], [6].
 *     Determinism: a case is cut into 2048-row chunks from its own first row; per chunk fp64 partial sums in a fixed
 *     order, chunks combined in ascending order, no float atomics - a record depends on its own case only, bitwise.
 *     The grid covers the chunks of all cases, so a large case shares a launch with small ones without serialising.
 * ---------------------------------------------------------------------------------------- */
size_t dfw_case_stress_summary_ws_bytes(int64_t N, int64_t B);
int dfw_case_stress_summary(const void* pred, int dtype, const float* pos, const uint8_t* mask, const int64_t* case_ptr,
                            int64_t B, int64_t N, double root_band, double allowable_pa, int log_scale, double* out,
                            void* ws, size_t ws_bytes, dfw_stream_t stream);

/* dtype conversion helper (weights fp32 -> bf16 copies for the bf16 path) */
int dfw_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, dfw_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * One-call inference forward of the whole model (model.py:74-99 in eval mode; the per-case body of
 * inference_gnn.py:224-328): encoder MLP, num_layers x [mean aggregation + fused SAGE linear with LayerNorm, ReLU,
 * residual], decoder MLP whose Linear(dec_mid, 1) is the epilogue's row dot.  The launches of the entry points above
 * behind ONE call (a Python host spends 0.5-0.8 ms per forward issuing them one by one); bit-identical to the pieces.
 *   x [N,in_dim] in x_dtype: DFW_F32 features are read as they are by the first linear (its weight then fp32 too),
 *   even when the compute dtype is bf16.   out: fp32 [N].
 *   weights: HOST array of 8 + 5*num_layers DEVICE pointers, matrices [out,in] row-major in the compute dtype
 *   (weights[0] in x_dtype), vectors fp32:
 *     [0..3]  encoder: W0 [enc_mid,in_dim], b0 [enc_mid], W1 [hidden,enc_mid], b1 [hidden]
 *     [4+5l..] layer l: lin_l.weight [hidden,hidden], lin_l.bias [hidden], lin_r.weight, LayerNorm weight, LayerNorm bias
 *     [last 4] decoder: W0 [dec_mid,hidden], b0 [dec_mid], w1 fp32 [dec_mid], b1 fp32 [1]      (biases nullable)
 * ---------------------------------------------------------------------------------------- */
size_t dfw_graphsage_forward_ws_bytes(int64_t N, int64_t in_dim, int64_t enc_mid, int64_t hidden, int64_t dec_mid,
                                      int x_dtype, int dtype);
int dfw_graphsage_forward(const int32_t* rowptr, const int32_t* col, const float* inv_deg, const void* x, int x_dtype,
                          const void* const* weights, int num_layers, int64_t N, int64_t E,
                          int64_t in_dim, int64_t enc_mid, int64_t hidden, int64_t dec_mid, float ln_eps, int dtype,
                          float* out, void* ws, size_t ws_bytes, dfw_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DFW_B200_H */
