// One-call SAGE layer (SURVEY 8b: dfw_sage_layer_fwd / dfw_sage_layer_bwd): the launch sequences that
// gnn/ops.py:SageConvFn issues piece by piece, behind one C entry point each, for hosts that drive a whole layer of
//     h' = h + dropout(relu(LayerNorm(lin_l(mean_j h_j) + lin_r(h))))          (reference model.py:90-95)
// without a Python autograd tape.  Host code only: every kernel belongs to the entry points it calls, so the results
// are bit-identical to the piecewise path (tests/test_gpu_kernels.py).  Workspace carve-up (all 256-byte aligned):
//   fwd: [linear]                                   bwd: [g_y | g_t | epilogue | weight-gradient | linear]
#include <algorithm>

#include "dfw_common.cuh"

namespace dfw {
namespace {
struct BwdWs {
    size_t o_gy, o_gt, o_epi, o_dw, o_lin, epi_bytes, dw_bytes, lin_bytes, total;
};
BwdWs carve_bwd(int64_t N, int64_t Hin, int64_t Hout, int dtype, bool want_gx) {
    const size_t e = dtype == DFW_F32 ? 4 : 2;
    BwdWs w{};
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off = align_up(off + b, 256); return o; };
    w.o_gy = take((size_t)N * Hout * e);
    w.o_gt = take(want_gx ? (size_t)N * Hout * e : 0);
    w.epi_bytes = dfw_epilogue_bwd_ws_bytes(N, Hout);
    w.o_epi = take(w.epi_bytes);
    w.dw_bytes = dfw_linear_bwd_weight_ws_bytes(N, Hout, Hin, Hin);
    w.o_dw = take(w.dw_bytes);
    w.lin_bytes = want_gx ? dfw_linear_ws_bytes(Hin, Hout, Hout, dtype) : 0;
    w.o_lin = take(w.lin_bytes);
    w.total = off + 256;
    return w;
}
inline char* base256(void* ws) { return reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~uintptr_t(255)); }
}  // namespace
}  // namespace dfw

extern "C" size_t dfw_sage_layer_fwd_ws_bytes(int64_t N, int64_t Hin, int64_t Hout, int dtype) {
    if (N < 0 || Hin < 1 || Hout < 1) return 0;
    return dfw_linear_ws_bytes(Hout, Hin, Hin, dtype);
}

extern "C" int dfw_sage_layer_fwd(const int32_t* rowptr, const int32_t* col, const float* inv_deg, const void* x, const void* w_l,
                                  const float* b_l, const void* w_r, const float* ln_gamma, const float* ln_beta, float ln_eps,
                                  float dropout_p, uint64_t seed, int flags, void* agg, void* pre_out, float* ln_stats, void* out,
                                  int64_t N, int64_t E, int64_t Hin, int64_t Hout, int dtype, void* ws, size_t ws_bytes,
                                  dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(x && w_l && w_r && agg && out, "dfw_sage_layer_fwd: null pointer");
    DFW_REQUIRE(!(flags & DFW_EP_RESIDUAL) || Hin == Hout, "dfw_sage_layer_fwd: the residual h + h_new needs Hin == Hout (%lld, %lld)",
                (long long)Hin, (long long)Hout);
    DFW_REQUIRE(!(flags & DFW_EP_TRANSPOSE_W), "dfw_sage_layer_fwd: weights are [Hout, Hin]");
    // dfw_linear_fwd takes a short workspace as "no tensor cores": the one-call layer would silently change kernels (and bits)
    const size_t need = dfw_sage_layer_fwd_ws_bytes(N, Hin, Hout, dtype);
    DFW_REQUIRE(ws_bytes >= need && (ws || need == 0), "dfw_sage_layer_fwd: workspace too small (%zu < %zu)", ws_bytes, need);
    int rc = dfw_sage_aggregate(rowptr, col, inv_deg, x, nullptr, agg, N, E, Hin, dtype, stream);
    if (rc) return rc;
    return dfw_linear_fwd(agg, w_l, Hin, x, w_r, Hin, b_l, ln_gamma, ln_beta, ln_eps, (flags & DFW_EP_RESIDUAL) ? x : nullptr, dropout_p,
                          seed, out, pre_out, ln_stats, nullptr, nullptr, nullptr, N, Hout, flags, dtype, ws, ws_bytes, stream);
}

extern "C" size_t dfw_sage_layer_bwd_ws_bytes(int64_t N, int64_t Hin, int64_t Hout, int dtype, int want_input_grad) {
    if (N < 0 || Hin < 1 || Hout < 1) return 0;
    return dfw::carve_bwd(N, Hin, Hout, dtype, want_input_grad != 0).total;
}

extern "C" int dfw_sage_layer_bwd(const int32_t* rowptr_t, const int32_t* col_t, const float* inv_deg, const void* x, const void* agg,
                                  const void* pre_out, const float* ln_stats, const void* w_l, const void* w_r, const float* ln_gamma,
                                  const float* ln_beta, const void* g_out, float dropout_p, uint64_t seed, int flags, void* g_x,
                                  float* dw_l, float* db_l, float* dw_r, float* dgamma, float* dbeta, int64_t N, int64_t E, int64_t Hin,
                                  int64_t Hout, int dtype, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(x && agg && g_out && dw_l && dw_r, "dfw_sage_layer_bwd: null pointer");
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_sage_layer_bwd: unknown dtype %d", dtype);
    const bool tail = flags & DFW_EP_LAYERNORM;  // the fused LayerNorm -> ReLU -> dropout -> residual tail of model.py:91-95
    DFW_REQUIRE(!tail || (pre_out && ln_stats && ln_gamma && ln_beta && dgamma && dbeta),
                "dfw_sage_layer_bwd: the LayerNorm tail needs pre_out, ln_stats, gamma/beta and dgamma/dbeta");
    DFW_REQUIRE(tail || !(flags & (DFW_EP_RELU | DFW_EP_DROPOUT | DFW_EP_RESIDUAL)),
                "dfw_sage_layer_bwd: ReLU / dropout / residual without LayerNorm is not a layer of this model");
    DFW_REQUIRE(!g_x || (w_l && w_r && rowptr_t && (col_t || E == 0) && inv_deg), "dfw_sage_layer_bwd: the input gradient needs the weights and the transposed CSR");
    const BwdWs w = carve_bwd(N, Hin, Hout, dtype, g_x != nullptr);
    DFW_REQUIRE(ws && ws_bytes >= w.total, "dfw_sage_layer_bwd: workspace too small (%zu < %zu)", ws_bytes, w.total);
    if (N == 0) {  // nothing flows: the parameter gradients of an empty batch are zero
        cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
        DFW_CUDA(cudaMemsetAsync(dw_l, 0, sizeof(float) * (size_t)Hout * Hin, s));
        DFW_CUDA(cudaMemsetAsync(dw_r, 0, sizeof(float) * (size_t)Hout * Hin, s));
        if (db_l) DFW_CUDA(cudaMemsetAsync(db_l, 0, sizeof(float) * (size_t)Hout, s));
        if (dgamma) DFW_CUDA(cudaMemsetAsync(dgamma, 0, sizeof(float) * (size_t)Hout, s));
        if (dbeta) DFW_CUDA(cudaMemsetAsync(dbeta, 0, sizeof(float) * (size_t)Hout, s));
        return 0;
    }
    char* base = base256(ws);
    const void* g_y = g_out;
    int rc;
    if (tail) {
        // g_y = dL/d(lin_l + lin_r): LayerNorm / ReLU / dropout backward, plus the column sums of g_y = lin_l's bias gradient
        void* gy = base + w.o_gy;
        rc = dfw_epilogue_bwd(g_out, nullptr, nullptr, pre_out, ln_stats, nullptr, ln_gamma, ln_beta, dropout_p, seed, gy, dgamma, dbeta,
                              nullptr, nullptr, db_l, N, Hout, flags & (DFW_EP_RELU | DFW_EP_LAYERNORM | DFW_EP_DROPOUT | DFW_EP_SEED_IS_PTR),
                              dtype, base + w.o_epi, w.epi_bytes, stream);
        if (rc) return rc;
        g_y = gy;
    }
    // dW_l = g_y^T agg, dW_r = g_y^T x (and db_l when there is no tail to emit it)
    rc = dfw_linear_bwd_weight(g_y, agg, Hin, x, Hin, dw_l, dw_r, tail ? nullptr : db_l, N, Hout, dtype, 0, base + w.o_dw, w.dw_bytes, stream);
    if (rc) return rc;
    if (!g_x) return 0;
    // dL/dx = (A^T D^-1 g_y) W_l + g_y W_r (+ g_out through the residual): aggregate the gradient first, then ONE two-operand
    // contraction on the forward's weights (DFW_EP_TRANSPOSE_W)
    DFW_REQUIRE(dfw_linear_tc_eligible(N, Hin, Hout, Hout, dtype), "dfw_sage_layer_bwd: (Hin=%lld, Hout=%lld) is outside the tensor-core "
                "path; use dfw_linear_bwd_input + dfw_sage_aggregate for this shape", (long long)Hin, (long long)Hout);
    void* g_t = base + w.o_gt;
    rc = dfw_sage_aggregate_scaled(rowptr_t, col_t, inv_deg, g_y, g_t, N, E, Hout, dtype, stream);
    if (rc) return rc;
    const bool res = tail && (flags & DFW_EP_RESIDUAL);
    return dfw_linear_fwd(g_t, w_l, Hout, g_y, w_r, Hout, nullptr, nullptr, nullptr, 0.f, res ? g_out : nullptr, 0.f, 0, g_x, nullptr, nullptr,
                          nullptr, nullptr, nullptr, N, Hin, DFW_EP_TRANSPOSE_W | (res ? DFW_EP_RESIDUAL : 0), dtype, base + w.o_lin, w.lin_bytes,
                          stream);
}

// ---- one-call encoder / decoder MLP (SURVEY 8b: dfw_mlp2_fwd / dfw_mlp2_bwd) ---------------------------------------
//   mode DFW_MLP2_ENCODER (model.py:52-57):  hidden = relu(x W1^T + b1),           out = relu(hidden W2^T + b2)   [N, Hout]
//   mode DFW_MLP2_DECODER (model.py:67-72):  hidden = dropout(relu(x W1^T + b1)),  out = hidden . w2 + b2         fp32 [N]
//     (out_channels = 1: the 64 -> 1 projection is the row-dot epilogue of the first linear; w2 fp32 [Hmid], b2 fp32 [1])
// Same launches as gnn/ops.py:LinearFn x 2 / DecoderTailFn, so the results are bit-identical to the model's path.
namespace dfw {
namespace {
struct MlpWs {
    size_t o_g2, o_gh, o_g1, o_epi, o_dw, o_lin, epi_bytes, dw_bytes, lin_bytes, total;
};
MlpWs carve_mlp_bwd(int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype, int mode, bool want_gx) {
    const size_t e = dtype == DFW_F32 ? 4 : 2;
    MlpWs w{};
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off = align_up(off + b, 256); return o; };
    const bool enc = mode == DFW_MLP2_ENCODER;
    w.o_g2 = take(enc ? (size_t)N * Hout * e : 0);   // dL/d(second pre-activation)
    w.o_gh = take(enc ? (size_t)N * Hmid * e : 0);   // dL/d hidden
    w.o_g1 = take((size_t)N * Hmid * e);             // dL/d(first pre-activation)
    w.epi_bytes = std::max(dfw_epilogue_bwd_ws_bytes(N, Hmid), enc ? dfw_epilogue_bwd_ws_bytes(N, Hout) : (size_t)0);
    w.o_epi = take(w.epi_bytes);
    w.dw_bytes = std::max(dfw_linear_bwd_weight_ws_bytes(N, Hmid, K, 0), enc ? dfw_linear_bwd_weight_ws_bytes(N, Hout, Hmid, 0) : (size_t)0);
    w.o_dw = take(w.dw_bytes);
    w.lin_bytes = std::max(enc ? dfw_linear_ws_bytes(Hmid, Hout, 0, dtype) : (size_t)0, want_gx ? dfw_linear_ws_bytes(K, Hmid, 0, dtype) : (size_t)0);
    w.o_lin = take(w.lin_bytes);
    w.total = off + 256;
    return w;
}
}  // namespace
}  // namespace dfw

extern "C" size_t dfw_mlp2_fwd_ws_bytes(int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype) {
    if (N < 0 || K < 1 || Hmid < 1 || Hout < 1) return 0;
    return std::max(dfw_linear_ws_bytes(Hmid, K, 0, dtype), dfw_linear_ws_bytes(Hout, Hmid, 0, dtype));
}

extern "C" int dfw_mlp2_fwd(const void* x, const void* w1, const float* b1, const void* w2, const float* b2, float dropout_p, uint64_t seed,
                            int flags, int mode, void* hidden, void* out, int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype,
                            void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(mode == DFW_MLP2_ENCODER || mode == DFW_MLP2_DECODER, "dfw_mlp2_fwd: unknown mode %d", mode);
    DFW_REQUIRE(x && w1 && w2 && out, "dfw_mlp2_fwd: null pointer");
    const size_t need = dfw_mlp2_fwd_ws_bytes(N, K, Hmid, Hout, dtype);  // see dfw_sage_layer_fwd
    DFW_REQUIRE(ws_bytes >= need && (ws || need == 0), "dfw_mlp2_fwd: workspace too small (%zu < %zu)", ws_bytes, need);
    const int seed_flag = flags & DFW_EP_SEED_IS_PTR;
    if (mode == DFW_MLP2_ENCODER) {
        DFW_REQUIRE(hidden, "dfw_mlp2_fwd: the encoder needs the hidden buffer");
        int rc = dfw_linear_fwd(x, w1, K, nullptr, nullptr, 0, b1, nullptr, nullptr, 1e-5f, nullptr, 0.f, 0, hidden, nullptr, nullptr, nullptr,
                                nullptr, nullptr, N, Hmid, DFW_EP_RELU, dtype, ws, ws_bytes, stream);
        if (rc) return rc;
        return dfw_linear_fwd(hidden, w2, Hmid, nullptr, nullptr, 0, b2, nullptr, nullptr, 1e-5f, nullptr, 0.f, 0, out, nullptr, nullptr, nullptr,
                              nullptr, nullptr, N, Hout, DFW_EP_RELU, dtype, ws, ws_bytes, stream);
    }
    DFW_REQUIRE(Hout == 1, "dfw_mlp2_fwd: the decoder mode is the out_channels = 1 tail (Hout = %lld)", (long long)Hout);
    const int f = DFW_EP_RELU | (dropout_p > 0.f ? (DFW_EP_DROPOUT | seed_flag) : 0);
    // hidden may be NULL at inference (nothing to save): only the row dot leaves the kernel
    return dfw_linear_fwd(x, w1, K, nullptr, nullptr, 0, b1, nullptr, nullptr, 1e-5f, nullptr, dropout_p, seed, hidden, nullptr, nullptr,
                          reinterpret_cast<const float*>(w2), b2, reinterpret_cast<float*>(out), N, Hmid, f, dtype, ws, ws_bytes, stream);
}

extern "C" size_t dfw_mlp2_bwd_ws_bytes(int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype, int mode, int want_input_grad) {
    if (N < 0 || K < 1 || Hmid < 1 || Hout < 1) return 0;
    return dfw::carve_mlp_bwd(N, K, Hmid, Hout, dtype, mode, want_input_grad != 0).total;
}

extern "C" int dfw_mlp2_bwd(const void* x, const void* hidden, const void* out, const void* w1, const void* w2, const void* g_out,
                            float dropout_p, uint64_t seed, int flags, int mode, void* g_x, float* dw1, float* db1, float* dw2, float* db2,
                            int64_t N, int64_t K, int64_t Hmid, int64_t Hout, int dtype, void* ws, size_t ws_bytes, dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(mode == DFW_MLP2_ENCODER || mode == DFW_MLP2_DECODER, "dfw_mlp2_bwd: unknown mode %d", mode);
    DFW_REQUIRE(x && hidden && w1 && w2 && g_out && dw1 && dw2, "dfw_mlp2_bwd: null pointer");
    const bool enc = mode == DFW_MLP2_ENCODER;
    DFW_REQUIRE(!enc || out, "dfw_mlp2_bwd: the encoder needs its saved output (ReLU mask)");
    DFW_REQUIRE(enc || Hout == 1, "dfw_mlp2_bwd: the decoder mode is the out_channels = 1 tail");
    const MlpWs w = carve_mlp_bwd(N, K, Hmid, Hout, dtype, mode, g_x != nullptr);
    DFW_REQUIRE(ws && ws_bytes >= w.total, "dfw_mlp2_bwd: workspace too small (%zu < %zu)", ws_bytes, w.total);
    char* base = base256(ws);
    void* g1 = base + w.o_g1;
    int rc;
    if (enc) {
        void* g2 = base + w.o_g2;
        void* gh = base + w.o_gh;
        // second linear: ReLU mask from the saved output, db2 = column sums, dW2 = g2^T hidden, g_hidden = g2 W2
        rc = dfw_epilogue_bwd(g_out, nullptr, nullptr, nullptr, nullptr, out, nullptr, nullptr, 0.f, 0, g2, nullptr, nullptr, nullptr, nullptr, db2,
                              N, Hout, DFW_EP_RELU, dtype, base + w.o_epi, w.epi_bytes, stream);
        if (rc) return rc;
        rc = dfw_linear_bwd_weight(g2, hidden, Hmid, nullptr, 0, dw2, nullptr, nullptr, N, Hout, dtype, 0, base + w.o_dw, w.dw_bytes, stream);
        if (rc) return rc;
        rc = dfw_linear_bwd_input(g2, w2, nullptr, nullptr, gh, N, Hout, Hmid, dtype, base + w.o_lin, dfw_linear_ws_bytes(Hmid, Hout, 0, dtype), stream);
        if (rc) return rc;
        // first linear
        rc = dfw_epilogue_bwd(gh, nullptr, nullptr, nullptr, nullptr, hidden, nullptr, nullptr, 0.f, 0, g1, nullptr, nullptr, nullptr, nullptr, db1,
                              N, Hmid, DFW_EP_RELU, dtype, base + w.o_epi, w.epi_bytes, stream);
        if (rc) return rc;
    } else {
        // g_out is dL/d(row dot) fp32 [N]: ReLU / dropout backward of the hidden layer, d w2, d b2 and db1 in one pass
        const int f = DFW_EP_RELU | (dropout_p > 0.f ? (DFW_EP_DROPOUT | (flags & DFW_EP_SEED_IS_PTR)) : 0);
        rc = dfw_epilogue_bwd(nullptr, reinterpret_cast<const float*>(g_out), reinterpret_cast<const float*>(w2), nullptr, nullptr, hidden, nullptr,
                              nullptr, dropout_p, seed, g1, nullptr, nullptr, dw2, db2, db1, N, Hmid, f, dtype, base + w.o_epi, w.epi_bytes, stream);
        if (rc) return rc;
    }
    rc = dfw_linear_bwd_weight(g1, x, K, nullptr, 0, dw1, nullptr, nullptr, N, Hmid, dtype, 0, base + w.o_dw, w.dw_bytes, stream);
    if (rc) return rc;
    if (!g_x) return 0;
    return dfw_linear_bwd_input(g1, w1, nullptr, nullptr, g_x, N, Hmid, K, dtype, base + w.o_lin, dfw_linear_ws_bytes(K, Hmid, 0, dtype), stream);
}

// ------------------------------------------------------------------------------------------------------------------------------
// One-call inference forward of the whole model (reference model.py:74-99 in eval mode; the loop body of inference_gnn.py:224-328):
// encoder MLP, L x (mean aggregation + fused SAGE linear with LayerNorm / ReLU / residual), decoder MLP with the 64 -> 1 row dot -
// the same launches gnn/model.py issues one Python call at a time (13 calls, ~0.5-0.8 ms of host time per forward: the config-5
// screening loop was host bound), behind one C call.  Bit-identical to the piecewise path.
// Workspace: [first-layer fp32 result (mixed mode) | mid | h_a | h_b | agg | linear workspace], all 256-byte aligned.
// ------------------------------------------------------------------------------------------------------------------------------
namespace dfw {
namespace {
struct FwdWs {
    size_t o_mid32, o_mid, o_ha, o_hb, o_agg, o_lin, lin_bytes, total;
};
FwdWs carve_forward(int64_t N, int64_t in_dim, int64_t enc_mid, int64_t H, int64_t dec_mid, int x_dtype, int dtype) {
    const size_t e = dtype == DFW_F32 ? 4 : 2;
    FwdWs w{};
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off = align_up(off + b, 256); return o; };
    const bool mixed = x_dtype == DFW_F32 && dtype != DFW_F32;
    w.o_mid32 = take(mixed ? (size_t)N * enc_mid * 4 : 0);
    w.o_mid = take((size_t)N * enc_mid * e);
    w.o_ha = take((size_t)N * H * e);
    w.o_hb = take((size_t)N * H * e);
    w.o_agg = take((size_t)N * H * e);
    w.lin_bytes = std::max({dfw_linear_ws_bytes(enc_mid, in_dim, 0, mixed ? DFW_F32 : dtype), dfw_linear_ws_bytes(H, enc_mid, 0, dtype),
                            dfw_linear_ws_bytes(H, H, H, dtype), dfw_linear_ws_bytes(dec_mid, H, 0, dtype)});
    w.o_lin = take(w.lin_bytes);
    w.total = off + 256;
    return w;
}
}  // namespace
}  // namespace dfw

extern "C" size_t dfw_graphsage_forward_ws_bytes(int64_t N, int64_t in_dim, int64_t enc_mid, int64_t hidden, int64_t dec_mid, int x_dtype,
                                                 int dtype) {
    if (N < 0 || in_dim < 1 || enc_mid < 1 || hidden < 1 || dec_mid < 1) return 0;
    return dfw::carve_forward(N, in_dim, enc_mid, hidden, dec_mid, x_dtype, dtype).total;
}

extern "C" int dfw_graphsage_forward(const int32_t* rowptr, const int32_t* col, const float* inv_deg, const void* x, int x_dtype,
                                     const void* const* weights, int num_layers, int64_t N, int64_t E, int64_t in_dim, int64_t enc_mid,
                                     int64_t hidden, int64_t dec_mid, float ln_eps, int dtype, float* out, void* ws, size_t ws_bytes,
                                     dfw_stream_t stream) {
    using namespace dfw;
    DFW_REQUIRE(x && weights && out && rowptr && inv_deg, "dfw_graphsage_forward: null pointer");
    DFW_REQUIRE(num_layers >= 0 && N >= 0, "dfw_graphsage_forward: bad sizes");
    DFW_REQUIRE(dtype == DFW_F32 || dtype == DFW_BF16, "dfw_graphsage_forward: dtype must be DFW_F32 or DFW_BF16");
    DFW_REQUIRE(x_dtype == DFW_F32 || x_dtype == dtype, "dfw_graphsage_forward: features are fp32 or in the compute dtype");
    const FwdWs w = carve_forward(N, in_dim, enc_mid, hidden, dec_mid, x_dtype, dtype);
    DFW_REQUIRE(ws && ws_bytes >= w.total, "dfw_graphsage_forward: workspace too small (%zu < %zu)", ws_bytes, w.total);
    const int nw = 8 + 5 * num_layers;
    for (int i = 0; i < nw; ++i) {
        const bool optional = (i == 1 || i == 3 || i == nw - 3 || i == nw - 1) || (i >= 4 && i < nw - 4 && (i - 4) % 5 == 1);  // biases
        DFW_REQUIRE(weights[i] || optional, "dfw_graphsage_forward: weights[%d] is NULL", i);
    }
    if (N == 0) return 0;
    char* b = base256(ws);
    void* lin = b + w.o_lin;
    const bool mixed = x_dtype == DFW_F32 && dtype != DFW_F32;
    void* mid = b + w.o_mid;
    // encoder (model.py:52-57): the first linear reads the raw features in THEIR dtype (see gnn/model.py), its output enters the compute dtype
    int rc;
    if (mixed && in_dim <= 16 && enc_mid % 4 == 0 && dtype == DFW_BF16) {
        // fp32 features, fp32 weights, fp32 arithmetic, bf16 result in one launch (same bits as the fp32 launch + dfw_cast below)
        rc = dfw_linear_fwd(x, weights[0], in_dim, nullptr, nullptr, 0, (const float*)weights[1], nullptr, nullptr, 1e-5f, nullptr, 0.f, 0, mid, nullptr,
                            nullptr, nullptr, nullptr, nullptr, N, enc_mid, DFW_EP_RELU | DFW_EP_OUT_BF16, DFW_F32, lin, w.lin_bytes, stream);
    } else if (mixed) {
        void* mid32 = b + w.o_mid32;
        rc = dfw_linear_fwd(x, weights[0], in_dim, nullptr, nullptr, 0, (const float*)weights[1], nullptr, nullptr, 1e-5f, nullptr, 0.f, 0, mid32, nullptr,
                            nullptr, nullptr, nullptr, nullptr, N, enc_mid, DFW_EP_RELU, DFW_F32, lin, w.lin_bytes, stream);
        if (rc) return rc;
        rc = dfw_cast(mid32, DFW_F32, mid, dtype, N * enc_mid, stream);
    } else {
        rc = dfw_linear_fwd(x, weights[0], in_dim, nullptr, nullptr, 0, (const float*)weights[1], nullptr, nullptr, 1e-5f, nullptr, 0.f, 0, mid, nullptr,
                            nullptr, nullptr, nullptr, nullptr, N, enc_mid, DFW_EP_RELU, dtype, lin, w.lin_bytes, stream);
    }
    if (rc) return rc;
    void* h = b + w.o_ha;
    void* h2 = b + w.o_hb;
    void* agg = b + w.o_agg;
    rc = dfw_linear_fwd(mid, weights[2], enc_mid, nullptr, nullptr, 0, (const float*)weights[3], nullptr, nullptr, 1e-5f, nullptr, 0.f, 0, h, nullptr, nullptr,
                        nullptr, nullptr, nullptr, N, hidden, DFW_EP_RELU, dtype, lin, w.lin_bytes, stream);
    if (rc) return rc;
    // SAGE layers (model.py:89-95, eval: no dropout, nothing saved)
    for (int l = 0; l < num_layers; ++l) {
        const void* const* lw = weights + 4 + 5 * l;
        rc = dfw_sage_layer_fwd(rowptr, col, inv_deg, h, lw[0], (const float*)lw[1], lw[2], (const float*)lw[3], (const float*)lw[4], ln_eps, 0.f, 0,
                                DFW_EP_LAYERNORM | DFW_EP_RELU | DFW_EP_RESIDUAL, agg, nullptr, nullptr, h2, N, E, hidden, hidden, dtype, lin, w.lin_bytes,
                                stream);
        if (rc) return rc;
        std::swap(h, h2);
    }
    // decoder (model.py:67-72, out_channels = 1): Linear -> ReLU -> (dropout off) -> Linear(dec_mid, 1) as the epilogue's row dot
    const void* const* dw = weights + 4 + 5 * num_layers;
    return dfw_mlp2_fwd(h, dw[0], (const float*)dw[1], dw[2], (const float*)dw[3], 0.f, 0, 0, DFW_MLP2_DECODER, nullptr, out, N, hidden, dec_mid, 1, dtype, lin,
                        w.lin_bytes, stream);
}
