"""Kernel-level parity (GPU, through the C ABI): CSR build bit-exact, aggregation, linear pieces."""
import os

import numpy as np
import pytest
import torch

from helpers import TOL_BF16, TOL_FP32, load_golden, rel_l2, rel_max
from oracle import csr_aggregate_c, csr_oracle_c
from oracle.sage_oracle import csr_oracle

pytestmark = pytest.mark.gpu

# DFW_FORCE_SIMT=1 (tests/test_gpu_linear_variants.py) routes every linear to the SIMT kernel: the entry points that need the
# tensor-core path by contract (the one-call SAGE backward's transposed-weight input gradient, DFW_EP_OUT_BF16) refuse it.
_needs_tc = pytest.mark.skipif(os.environ.get("DFW_FORCE_SIMT", "0")[:1] not in ("", "0"),
                               reason="needs the tensor-core linear, which DFW_FORCE_SIMT turns off")


@pytest.fixture(scope="module")
def ops():
    from deep_fem_uav_wing.gnn import ops as _ops

    return _ops


def _check_csr(ops, ei_np, n, by_src):
    ei = torch.from_numpy(ei_np).cuda()
    rowptr, col, perm, inv, status = ops.csr_build_raw(ei, n, by_src=by_src)
    o = csr_oracle_c(ei_np, n, "src" if by_src else "dst")
    assert int(status[0]) == 0
    assert torch.equal(rowptr.cpu(), torch.from_numpy(o[0]))
    assert torch.equal(col.cpu(), torch.from_numpy(o[1]))
    assert torch.equal(perm.cpu(), torch.from_numpy(o[2]))
    assert torch.equal(inv.cpu(), torch.from_numpy(o[3]))  # 1/max(deg,1): correctly rounded on both sides
    deg = np.diff(o[0])
    assert int(status[1]) == (int(deg.max()) if n else 0)


@pytest.mark.parametrize("by_src", [False, True])
def test_csr_bit_exact_random_and_edge_cases(ops, by_src):
    rng = np.random.default_rng(0)
    for n, e in ((1, 0), (7, 0), (1, 5), (50, 400), (1000, 20000), (5000, 5001), (4097, 100000)):
        ei = rng.integers(0, n, size=(2, e)).astype(np.int64)  # duplicates and self loops included
        _check_csr(ops, ei, n, by_src)


def test_csr_bit_exact_high_degree_rows(ops):
    rng = np.random.default_rng(1)
    # star with 6000 leaves (row longer than the 4096-key shared-memory sort), a 3000-row and a 33-row
    src = np.concatenate([np.arange(1, 6001), rng.integers(0, 7000, 3000), rng.integers(0, 7000, 33), rng.integers(0, 7000, 20000)])
    dst = np.concatenate([np.zeros(6000, np.int64), np.full(3000, 5), np.full(33, 9), rng.integers(0, 7000, 20000)])
    order = rng.permutation(src.size)
    ei = np.stack([src[order], dst[order]]).astype(np.int64)
    _check_csr(ops, ei, 7000, False)
    _check_csr(ops, ei, 7000, True)


def test_csr_bit_exact_on_meshes_and_golden_model_graphs(ops):
    from deep_fem_uav_wing.gnn import synth
    from helpers import load_golden

    for m in (synth.surface_tri_wing(20000, seed=42), synth.tet_lattice_wing(20000, seed=42),
              synth.tet_lattice_wing(5000, seed=1, node_order="random")):
        _check_csr(ops, m["edge_index"], m["num_nodes"], False)
        _check_csr(ops, m["edge_index"], m["num_nodes"], True)
    g = load_golden("model_tet500_h128_l4")
    _check_csr(ops, g["edge_index"], g["x"].shape[0], False)


def test_csr_reports_out_of_range(ops):
    ei = torch.tensor([[0, 1, 9, -1], [1, 2, 0, 0]], dtype=torch.int64).cuda()
    g = ops.get_graph(ei, 3)
    with pytest.raises(IndexError):
        g.check()
    with pytest.raises(TypeError):
        ops.csr_build_raw(ei.int(), 3)
    with pytest.raises(ValueError):
        ops.csr_build_raw(ei[0], 3)


def test_csr_input_order_invariance(ops):
    rng = np.random.default_rng(3)
    n, e = 3000, 30000
    ei = np.unique(rng.integers(0, n, size=(2, e)), axis=1).astype(np.int64)
    a = ops.csr_build_raw(torch.from_numpy(ei).cuda(), n)
    b = ops.csr_build_raw(torch.from_numpy(ei[:, rng.permutation(ei.shape[1])]).cuda(), n)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])  # canonical whatever the edge order


def test_csr_transpose_copies_symmetric_graphs_and_builds_the_rest(ops):
    """``dfw_csr_transpose`` == the by-source CSR of the oracle, bit-exact, whether the device-side symmetry check takes
    the copy path (mesh graphs, self loops) or the general build (one-directional edges, duplicate edges)."""
    from deep_fem_uav_wing.gnn import synth

    rng = np.random.default_rng(5)
    mesh = synth.surface_tri_wing(3000, seed=3)
    tet = synth.tet_lattice_wing(2000, seed=4)
    sym_loops = np.array([[0, 1, 1, 2, 2, 0, 3], [1, 0, 2, 1, 0, 2, 3]], dtype=np.int64)  # triangle + a self loop
    one_way = np.array([[0, 1, 2], [1, 2, 0]], dtype=np.int64)
    dup_sym = np.array([[0, 1, 0, 1], [1, 0, 1, 0]], dtype=np.int64)  # symmetric as a multigraph: general path
    cases = [(mesh["edge_index"], mesh["num_nodes"], 0), (tet["edge_index"], tet["num_nodes"], 0), (sym_loops, 5, 0),
             (one_way, 3, 1), (dup_sym, 2, 1), (rng.integers(0, 500, size=(2, 6000)).astype(np.int64), 500, 1),
             (np.zeros((2, 0), dtype=np.int64), 7, 0)]
    for ei_np, n, asym in cases:
        ei = torch.from_numpy(np.ascontiguousarray(ei_np)).cuda()
        rowptr, col, _, _, _ = ops.csr_build_raw(ei, n, by_src=False, want_perm=False)
        rp_t, col_t, status = ops.csr_transpose_raw(ei, n, rowptr, col)
        o = csr_oracle_c(ei_np, n, "src")
        assert int(status[2]) == asym
        assert torch.equal(rp_t.cpu(), torch.from_numpy(o[0])) and torch.equal(col_t.cpu(), torch.from_numpy(o[1]))


@pytest.mark.parametrize("h", [4, 16, 64, 128, 256, 96])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_aggregate_matches_oracle(ops, h, dtype):
    rng = np.random.default_rng(h)
    n, e = 3001, 25000
    ei = rng.integers(0, n, size=(2, e)).astype(np.int64)
    ei[1, :200] = 7  # one long row
    if dtype == torch.bfloat16 and (h * 2) % 16:
        pytest.skip("row not 16-byte aligned")
    x = torch.from_numpy(rng.standard_normal((n, h)).astype(np.float32)).to(dtype)
    rowptr, col, _, inv = csr_oracle_c(ei, n)
    ref = torch.from_numpy(csr_aggregate_c(rowptr, col, inv, x.float().numpy()))
    g = ops.get_graph(torch.from_numpy(ei).cuda(), n)
    got = ops.aggregate(g.rowptr, g.col, g.inv_deg, x.cuda())
    tol = TOL_FP32 if dtype == torch.float32 else TOL_BF16
    assert rel_max(got.float().cpu(), ref) < tol
    again = ops.aggregate(g.rowptr, g.col, g.inv_deg, x.cuda())
    assert torch.equal(got, again)  # deterministic: no atomics
    # sum mode + addend over the transposed CSR
    rp_t, col_t = g.transpose()
    ot = csr_oracle_c(ei, n, "src")
    add = torch.from_numpy(rng.standard_normal((n, h)).astype(np.float32)).to(dtype)
    ref_t = torch.from_numpy(csr_aggregate_c(ot[0], ot[1], None, x.float().numpy())) + add.float()
    got_t = ops.aggregate(rp_t, col_t, None, x.cuda(), addend=add.cuda())
    assert rel_max(got_t.float().cpu(), ref_t) < tol
    # source-scaled gather (adjoint of the mean): sum_k inv_deg[col[k]] * x[col[k]] over the transposed CSR
    inv_t = torch.from_numpy(inv)
    ref_s = torch.from_numpy(csr_aggregate_c(ot[0], ot[1], None, (x.float() * inv_t[:, None]).numpy()))
    got_s = ops.aggregate_scaled(rp_t, col_t, g.inv_deg, x.cuda())
    assert rel_max(got_s.float().cpu(), ref_s) < tol
    assert torch.equal(got_s, ops.aggregate_scaled(rp_t, col_t, g.inv_deg, x.cuda()))


def test_aggregate_properties_at_scale(ops):
    """Size-independent properties on a config-2-sized batch (4 x 50k nodes, H=128): linearity and
    permutation equivariance of the mean aggregation, transposed-sum adjointness."""
    from deep_fem_uav_wing.gnn import synth

    m = synth.tet_lattice_wing(200000, seed=9)
    n = m["num_nodes"]
    ei = torch.from_numpy(m["edge_index"]).cuda()
    g = ops.get_graph(ei, n)
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, 128, device="cuda", generator=gen)
    y = torch.randn(n, 128, device="cuda", generator=gen)
    ax, ay = ops.aggregate(g.rowptr, g.col, g.inv_deg, x), ops.aggregate(g.rowptr, g.col, g.inv_deg, y)
    axy = ops.aggregate(g.rowptr, g.col, g.inv_deg, 2.0 * x + y)
    assert rel_max(axy, 2.0 * ax + ay) < TOL_FP32
    # adjointness: <A x, y> == <x, A^T y> with A^T = transposed sum of inv_deg-scaled rows
    rp_t, col_t = g.transpose()
    aty = ops.aggregate(rp_t, col_t, None, y * g.inv_deg[:, None])
    lhs, rhs = (ax.double() * y.double()).sum().item(), (x.double() * aty.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-6 * max(abs(lhs), 1.0)
    # the source-scaled gather is the same adjoint without the pre-scaled copy
    aty2 = ops.aggregate_scaled(rp_t, col_t, g.inv_deg, y)
    assert rel_max(aty2, aty) < TOL_FP32
    # permutation equivariance
    perm = torch.randperm(n, device="cuda", generator=gen)
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(n, device="cuda")
    g2 = ops.get_graph(inv[ei], n)  # relabel node i -> inv[i]
    ax2 = ops.aggregate(g2.rowptr, g2.col, g2.inv_deg, x[perm])
    assert rel_max(ax2, ax[perm]) < TOL_FP32


def _ref_linear(a1, w1, a2, w2, b, ln, relu, res):
    y = a1.double() @ w1.double().T
    if a2 is not None:
        y = y + a2.double() @ w2.double().T
    if b is not None:
        y = y + b.double()
    out = y
    if ln is not None:
        out = torch.nn.functional.layer_norm(out, (out.shape[1],), ln[0].double(), ln[1].double(), 1e-5)
    if relu:
        out = out.relu()
    if res is not None:
        out = out + res.double()
    return y, out


@pytest.mark.parametrize("hout,k1,k2", [(64, 10, 0), (128, 64, 0), (64, 64, 64), (128, 128, 128), (256, 256, 256), (16, 16, 16), (64, 128, 0),
                                        (192, 64, 192)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_linear_fwd_and_bwd_pieces(ops, hout, k1, k2, dtype):
    torch.manual_seed(hout + k1)
    n = 777
    dev = "cuda"
    a1 = torch.randn(n, k1, device=dev).to(dtype)
    w1 = (torch.randn(hout, k1, device=dev) / k1**0.5).to(dtype)
    a2 = torch.randn(n, k2, device=dev).to(dtype) if k2 else None
    w2 = (torch.randn(hout, k2, device=dev) / k2**0.5).to(dtype) if k2 else None
    b = torch.randn(hout, device=dev)
    gamma, beta = torch.rand(hout, device=dev) + 0.5, torch.randn(hout, device=dev)
    res = torch.randn(n, hout, device=dev).to(dtype) if k2 == hout else None
    tol = TOL_FP32 if dtype == torch.float32 else TOL_BF16
    use_ln = k2 > 0
    out, pre, stats, _ = ops.linear_fwd(a1, w1, a2, w2, bias=b, ln=(gamma, beta) if use_ln else None, relu=True, residual=res,
                                        save_pre=True)
    y_ref, out_ref = _ref_linear(a1, w1, a2, w2, b, (gamma, beta) if use_ln else None, True, res)
    assert rel_max(pre.double(), y_ref) < tol
    assert rel_max(out.double(), out_ref) < (tol if dtype == torch.float32 else 3 * tol)
    if use_ln:
        mean = y_ref.mean(1)
        rstd = 1.0 / torch.sqrt(y_ref.var(1, unbiased=False) + 1e-5)
        assert rel_max(stats[:, 0].double(), mean) < max(tol, 1e-5) and rel_max(stats[:, 1].double(), rstd) < max(tol, 1e-5)
    # dx and dW pieces
    g = torch.randn(n, hout, device=dev).to(dtype)
    scale = torch.rand(n, device=dev)
    add = torch.randn(n, k1, device=dev).to(dtype)
    dx = ops.linear_bwd_input(g, w1, row_scale=scale, addend=add)
    dx_ref = scale.double()[:, None] * (g.double() @ w1.double()) + add.double()
    assert rel_max(dx.double(), dx_ref) < tol
    dw1, dw2, db = ops.linear_bwd_weight(g, a1, a2)
    assert rel_l2(dw1.double(), g.double().T @ a1.double()) < tol
    if k2:
        assert rel_l2(dw2.double(), g.double().T @ a2.double()) < tol
    assert rel_l2(db.double(), g.double().sum(0)) < tol
    dw1b, _, _ = ops.linear_bwd_weight(g, a1, a2)
    assert torch.equal(dw1, dw1b)  # fixed-order split reduction: bit-reproducible


@pytest.mark.parametrize("kin,hout", [(128, 128), (64, 128), (256, 64), (24, 40)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_linear_transposed_weights_equal_pretransposed(ops, kin, hout, dtype):
    """DFW_EP_TRANSPOSE_W (the SAGE layer's input gradient ``g_t W_l + g_y W_r + g_out`` on the forward's weights) is
    bit-identical to handing over ``W.t().contiguous()``; (24, 40) is not tensor-core eligible and takes the wrapper's
    explicit transposition."""
    torch.manual_seed(kin * 3 + hout)
    n, dev = 1501, "cuda"
    g_t = torch.randn(n, hout, device=dev).to(dtype)
    g_y = torch.randn(n, hout, device=dev).to(dtype)
    wl = (torch.randn(hout, kin, device=dev) / hout**0.5).to(dtype)  # forward layout [Hout, K]
    wr = (torch.randn(hout, kin, device=dev) / hout**0.5).to(dtype)
    g_out = torch.randn(n, kin, device=dev).to(dtype)
    a, _, _, _ = ops.linear_fwd(g_t, wl, g_y, wr, residual=g_out, transpose_w=True)
    b, _, _, _ = ops.linear_fwd(g_t, wl.t().contiguous(), g_y, wr.t().contiguous(), residual=g_out)
    assert a.shape == (n, kin) and torch.equal(a, b)
    ref = g_t.double() @ wl.double() + g_y.double() @ wr.double() + g_out.double()
    assert rel_max(a.double(), ref) < (TOL_FP32 if dtype == torch.float32 else TOL_BF16)
    c, _, _, _ = ops.linear_fwd(g_t, wl, transpose_w=True)
    assert rel_max(c.double(), g_t.double() @ wl.double()) < (TOL_FP32 if dtype == torch.float32 else TOL_BF16)


@pytest.mark.parametrize("k,hout,n", [(10, 64, 200003), (3, 64, 777), (8, 128, 4099), (16, 256, 1000), (12, 4, 65), (10, 64, 1)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_tiny_k_linear_forward_and_weight_gradient(ops, k, hout, n, dtype):
    """The encoder's first layer (``Linear(10, 64)``, model.py:53): tiled tiny-K kernels, forward and dW."""
    torch.manual_seed(k * 1000 + hout)
    dev = "cuda"
    x = torch.randn(n, k, device=dev).to(dtype)
    w = (torch.randn(hout, k, device=dev) / k**0.5).to(dtype)
    b = torch.randn(hout, device=dev)
    tol = TOL_FP32 if dtype == torch.float32 else TOL_BF16
    for relu in (True, False):
        out, _, _, _ = ops.linear_fwd(x, w, bias=b, relu=relu)
        ref = x.double() @ w.double().T + b.double()
        ref = torch.relu(ref) if relu else ref
        assert out.shape == (n, hout) and rel_max(out.double(), ref) < tol
    g = torch.randn(n, hout, device=dev).to(dtype)
    dw, _, _ = ops.linear_bwd_weight(g, x, None, want_bias=False)
    assert dw.dtype == torch.float32 and rel_l2(dw.double(), g.double().T @ x.double()) < (TOL_FP32 if dtype == torch.float32 else 1e-4)
    dw2, _, _ = ops.linear_bwd_weight(g, x, None, want_bias=False)
    assert torch.equal(dw, dw2)  # fixed tile -> block assignment, fixed-order reductions


@_needs_tc
@pytest.mark.parametrize("dtype,h,p", [(torch.float32, 128, 0.1), (torch.float32, 64, 0.0), (torch.bfloat16, 128, 0.2)])
def test_one_call_sage_layer_equals_the_piecewise_path(ops, dtype, h, p):
    """``dfw_sage_layer_fwd`` / ``dfw_sage_layer_bwd`` (SURVEY 8b) launch the same kernels as the autograd Function that the
    model uses: outputs and every gradient are bit-identical - with the fused LayerNorm tail and as a bare SAGEConv."""
    from deep_fem_uav_wing.gnn import synth

    torch.manual_seed(h)
    m = synth.tet_lattice_wing(3000, seed=11)
    n, dev = m["num_nodes"], "cuda"
    ei = torch.from_numpy(m["edge_index"]).to(dev)
    graph = ops.get_graph(ei, n)
    x = torch.randn(n, h, device=dev).to(dtype).requires_grad_(True)
    w_l = (torch.randn(h, h, device=dev) / h**0.5).requires_grad_(True)
    w_r = (torch.randn(h, h, device=dev) / h**0.5).requires_grad_(True)
    b_l = torch.randn(h, device=dev).requires_grad_(True)
    gamma = (torch.rand(h, device=dev) + 0.5).requires_grad_(True)
    beta = torch.randn(h, device=dev).requires_grad_(True)
    g_out = torch.randn(n, h, device=dev).to(dtype)
    seed = 1234567
    wl_c, wr_c = w_l.detach().to(dtype), w_r.detach().to(dtype)
    for tail in (True, False):
        for t in (x, w_l, w_r, b_l, gamma, beta):
            t.grad = None
        # piecewise: the model's autograd Function (gnn/ops.py:SageConvFn)
        ref = ops.SageConvFn.apply(x, w_l, b_l, w_r, gamma if tail else None, beta if tail else None, graph, 1e-5, p if tail else 0.0, seed, tail)
        ref.backward(g_out)
        # one call each way
        ln = (gamma.detach(), beta.detach()) if tail else None
        out, agg, pre, stats = ops.sage_layer_fwd(graph, x.detach(), wl_c, b_l.detach(), wr_c, ln=ln, dropout_p=p if tail else 0.0, seed=seed)
        assert torch.equal(out, ref.detach())
        g_x, dw_l, db_l, dw_r, dgamma, dbeta = ops.sage_layer_bwd(graph, x.detach(), agg, pre, stats, wl_c, wr_c, ln, g_out,
                                                                 dropout_p=p if tail else 0.0, seed=seed)
        assert torch.equal(g_x, x.grad) and torch.equal(dw_l, w_l.grad) and torch.equal(dw_r, w_r.grad) and torch.equal(db_l, b_l.grad)
        if tail:
            assert torch.equal(dgamma, gamma.grad) and torch.equal(dbeta, beta.grad)
        # first layer of a network: no input gradient wanted
        _, dw_l2, _, dw_r2, _, _ = ops.sage_layer_bwd(graph, x.detach(), agg, pre, stats, wl_c, wr_c, ln, g_out, dropout_p=p if tail else 0.0,
                                                      seed=seed, want_input_grad=False)
        assert torch.equal(dw_l2, dw_l) and torch.equal(dw_r2, dw_r)
    with pytest.raises(RuntimeError, match="tensor-core"):  # (24, 24) is not a tensor-core shape: the composite says so
        xs = torch.randn(n, 24, device=dev)
        ws_ = torch.randn(24, 24, device=dev)
        o, a, _, _ = ops.sage_layer_fwd(graph, xs, ws_, None, ws_)
        ops.sage_layer_bwd(graph, xs, a, None, None, ws_, ws_, None, torch.randn(n, 24, device=dev), has_bias=False)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_one_call_encoder_and_decoder_equal_the_piecewise_path(ops, dtype):
    """``dfw_mlp2_fwd`` / ``dfw_mlp2_bwd`` (SURVEY 8b) vs the autograd Functions the model uses for its encoder
    (two ``LinearFn``) and its decoder tail (``DecoderTailFn``): bit-identical outputs and gradients."""
    torch.manual_seed(7)
    n, dev = 3001, "cuda"

    def leaf(*shape, scale=1.0):
        return (torch.randn(*shape, device=dev) * scale).requires_grad_(True)

    # encoder: Linear(10, 64) -> ReLU -> Linear(64, 128) -> ReLU (model.py:52-57)
    x = torch.randn(n, 10, device=dev).to(dtype).requires_grad_(True)
    w1, b1, w2, b2 = leaf(64, 10, scale=0.3), leaf(64), leaf(128, 64, scale=0.12), leaf(128)
    g = torch.randn(n, 128, device=dev).to(dtype)
    h1 = ops.LinearFn.apply(x, w1, b1, True, 0.0, 0)
    h2 = ops.LinearFn.apply(h1, w2, b2, True, 0.0, 0)
    h2.backward(g)
    w1c, w2c = ops.cast(w1.detach(), dtype), ops.cast(w2.detach(), dtype)
    out, hidden = ops.mlp2_fwd(x.detach(), w1c, b1.detach(), w2c, b2.detach(), ops.MLP2_ENCODER)
    assert torch.equal(out, h2.detach()) and torch.equal(hidden, h1.detach())
    g_x, dw1, db1, dw2, db2 = ops.mlp2_bwd(x.detach(), hidden, out, w1c, w2c, g, ops.MLP2_ENCODER)
    assert torch.equal(g_x, x.grad) and torch.equal(dw1, w1.grad) and torch.equal(db1, b1.grad)
    assert torch.equal(dw2, w2.grad) and torch.equal(db2, b2.grad)
    g_x0, dw1b, _, _, _ = ops.mlp2_bwd(x.detach(), hidden, out, w1c, w2c, g, ops.MLP2_ENCODER, want_input_grad=False)
    assert g_x0 is None and torch.equal(dw1b, dw1)  # the model's first layer: x needs no gradient

    # decoder tail: Linear(128, 64) -> ReLU -> Dropout -> Linear(64, 1) (model.py:67-72)
    h = torch.randn(n, 128, device=dev).to(dtype).requires_grad_(True)
    w3, b3, w4, b4 = leaf(64, 128, scale=0.09), leaf(64), leaf(1, 64, scale=0.12), leaf(1)
    p, seed = 0.1, 424242
    y = ops.DecoderTailFn.apply(h, w3, b3, w4, b4, p, seed)
    gy = torch.randn(n, 1, device=dev).to(dtype)
    y.backward(gy)
    w3c = ops.cast(w3.detach(), dtype)
    w4f = w4.detach().float().reshape(-1).contiguous()
    out, hidden = ops.mlp2_fwd(h.detach(), w3c, b3.detach(), w4f, b4.detach(), ops.MLP2_DECODER, dropout_p=p, seed=seed)
    assert out.dtype == torch.float32 and out.shape == (n,)
    assert torch.equal(out.unsqueeze(1) if dtype == torch.float32 else ops.cast(out.unsqueeze(1), dtype), y.detach())
    g_h, dw3, db3, dw4, db4 = ops.mlp2_bwd(h.detach(), hidden, None, w3c, w4f, gy.reshape(-1).float(), ops.MLP2_DECODER, dropout_p=p, seed=seed)
    assert torch.equal(g_h, h.grad) and torch.equal(dw3, w3.grad) and torch.equal(db3, b3.grad)
    assert torch.equal(dw4.reshape(1, -1), w4.grad) and torch.equal(db4, b4.grad)
    out_inf, hid_inf = ops.mlp2_fwd(h.detach(), w3c, b3.detach(), w4f, b4.detach(), ops.MLP2_DECODER, save_hidden=False)
    assert hid_inf is None and out_inf.shape == (n,)  # inference: nothing saved, no dropout


def test_masked_mse_matches_reference_fixture(ops):
    from helpers import load_golden

    from deep_fem_uav_wing.gnn.model import MaskedMSELoss

    g = load_golden("loss_metrics")
    targ = torch.from_numpy(g["target"]).cuda()
    mask = torch.from_numpy(g["mask"]).cuda()
    for red in ("mean", "sum"):
        for mname, mm in (("mask", mask), ("none", None), ("allfalse", torch.zeros(50, dtype=torch.bool, device="cuda"))):
            pred = torch.from_numpy(g["pred"]).cuda().requires_grad_(True)
            loss = MaskedMSELoss(red)(pred, targ, mm)
            ref = float(g[f"loss_{red}_{mname}"])
            assert abs(loss.item() - ref) <= TOL_FP32 * max(1.0, abs(ref))
            assert loss.requires_grad
            if mname != "allfalse":
                loss.backward()
                assert rel_max(pred.grad.cpu(), g[f"grad_{red}_{mname}"]) < TOL_FP32
            else:
                strict = MaskedMSELoss(red, strict_empty=True)(pred, targ, mm)
                assert strict.item() == 0.0 and strict.requires_grad and strict.grad_fn is None  # fresh leaf (model.py:147-149)


@pytest.mark.parametrize("n", [0, 1, 50, 200003])
@pytest.mark.parametrize("log_scale", [True, False])
def test_stress_metrics_match_the_reference_formulas(ops, n, log_scale):
    """dfw_stress_metrics vs the oracle's restatement of compute_metrics (reference model.py:156-216): all nodes,
    masked nodes, no mask, all-False mask, empty input; fp32 tolerance 1e-5 (device expm1f vs numpy expm1)."""
    from deep_fem_uav_wing.gnn.model import compute_metrics, metrics_from_device
    from oracle.sage_oracle import compute_metrics_ref

    rng = np.random.default_rng(n + int(log_scale))
    pred = torch.from_numpy((rng.standard_normal((n, 1)) * 2.0 + 8.0).astype(np.float32))
    targ = torch.from_numpy((rng.standard_normal((n, 1)) * 2.0 + 8.0).astype(np.float32))
    masks = {"mask": torch.from_numpy(rng.random(n) > 0.3), "none": None, "allfalse": torch.zeros(n, dtype=torch.bool)}
    for name, m in masks.items():
        ref = compute_metrics_ref(pred, targ, m, log_scale=log_scale)
        got = compute_metrics(pred.cuda(), targ.cuda(), m.cuda() if m is not None else None, log_scale=log_scale)
        assert got.keys() == ref.keys()
        for sub in ("all_nodes", "masked_nodes"):
            assert got[sub]["count"] == ref[sub]["count"], (name, sub)
            for k in ("mae", "rmse", "max_error"):
                assert abs(got[sub][k] - ref[sub][k]) <= 1e-5 * max(abs(ref[sub][k]), 1e-30) + 1e-12, (name, sub, k, got[sub][k], ref[sub][k])
    # deterministic, and the device result converts to the same dict
    if n:
        a = ops.stress_metrics(pred.cuda(), targ.cuda(), masks["mask"].cuda(), log_scale)
        b = ops.stress_metrics(pred.cuda(), targ.cuda(), masks["mask"].cuda(), log_scale)
        assert torch.equal(a, b)
        assert metrics_from_device(a) == compute_metrics(pred.cuda(), targ.cuda(), masks["mask"].cuda(), log_scale=log_scale)


def _faces_case(ops, faces_np, node_ids_np, n):
    """device faces -> graph vs the oracle restatement of _faces_to_edge_index (+ the CSR oracle), bit-exact."""
    from helpers import canon_edges
    from oracle.sage_oracle import faces_to_edge_index_ref

    ids = {int(v): i for i, v in enumerate(node_ids_np)} if node_ids_np is not None else {i: i for i in range(n)}
    ref = canon_edges(faces_to_edge_index_ref(faces_np.tolist(), ids))
    g, ei = ops.faces_to_graph(torch.from_numpy(faces_np.astype(np.int64)).reshape(-1, 3).cuda(), n,
                               None if node_ids_np is None else torch.from_numpy(node_ids_np.astype(np.int64)).cuda())
    assert ei.dtype == torch.int64 and tuple(ei.shape) == ref.shape
    assert np.array_equal(ei.cpu().numpy(), ref)  # canonical (dst, src) order, same edge multiset as the reference
    rowptr, col, _, inv = csr_oracle_c(ref, n)
    assert torch.equal(g.rowptr.cpu(), torch.from_numpy(rowptr)) and torch.equal(g.col.cpu(), torch.from_numpy(col))
    assert torch.equal(g.inv_deg.cpu(), torch.from_numpy(inv))
    assert g.num_edges == ref.shape[1]
    # the registered graph is what the model's lookup returns, and its transpose is itself (symmetric)
    assert ops.get_graph(ei, n) is g and g.transpose()[1] is g.col
    return g, ei


def test_faces_to_graph_matches_reference_fixture_and_edge_cases(ops):
    gold = load_golden("faces_to_edge_index")
    faces = gold["faces"]  # the 12-triangle box of geometry.py:82-102 with node ids 10..17
    ids = np.arange(10, 18)
    g, ei = _faces_case(ops, faces, ids, 8)
    assert ei.shape == (2, 36) and int(g.skipped_faces.item()) == 0
    # a face touching an unknown id is skipped (dataset.py:43-46)
    g2, ei2 = _faces_case(ops, np.concatenate([faces, [[10, 11, 999]]]), ids, 8)
    assert torch.equal(ei2, ei) and int(g2.skipped_faces.item()) == 1
    # node ids given in a scrambled order (mapping through the sort permutation)
    rng = np.random.default_rng(0)
    perm = rng.permutation(8)
    _faces_case(ops, faces, ids[perm], 8)
    # degenerate faces: repeated vertices give self pairs, which the reference emits twice
    _faces_case(ops, np.array([[0, 0, 1], [2, 2, 2], [1, 3, 1]]), None, 5)
    # empty
    g0, ei0 = ops.faces_to_graph(torch.zeros(0, 3, dtype=torch.int64, device="cuda"), 4)
    assert ei0.shape == (2, 0) and g0.rowptr.tolist() == [0, 0, 0, 0, 0]


def test_faces_to_graph_on_a_config_sized_surface_mesh(ops):
    """50k-node closed wing surface (config 2's mesh): same edge_index as the host construction, and the model's
    forward on it equals the forward on the host-built edge_index."""
    from helpers import canon_edges
    from deep_fem_uav_wing.gnn import synth

    m = synth.surface_tri_wing(50000, seed=42)
    n = m["num_nodes"]
    g, ei = _faces_case(ops, m["faces"], None, n)
    assert np.array_equal(ei.cpu().numpy(), canon_edges(m["edge_index"]))
    x = torch.randn(n, 64, device="cuda")
    a = ops.aggregate(g.rowptr, g.col, g.inv_deg, x)
    g_host = ops.get_graph(torch.from_numpy(m["edge_index"]).cuda(), n)
    assert torch.equal(a, ops.aggregate(g_host.rowptr, g_host.col, g_host.inv_deg, x))
    # sync=False: no host read - col keeps its capacity, num_edges is the closed-surface estimate, the exact count stays on the device
    g2, none = ops.faces_to_graph(torch.from_numpy(m["faces"].astype(np.int64)).cuda(), n, want_edge_index=False, sync=False)
    assert none is None and int(g2.edge_count.item()) == g.num_edges and g2.col.numel() >= g.num_edges
    assert torch.equal(g2.rowptr, g.rowptr) and torch.equal(g2.col[: g.num_edges], g.col) and torch.equal(g2.inv_deg, g.inv_deg)
    assert torch.equal(a, ops.aggregate(g2.rowptr, g2.col, g2.inv_deg, x))
    with pytest.raises(ValueError):
        ops.faces_to_graph(torch.from_numpy(m["faces"].astype(np.int64)).cuda(), n, sync=False)


def test_node_features_batched_equals_per_case_calls(ops):
    """dfw_node_features_batched (B concatenated cases, per-case min-max) is bit-identical to B calls of dfw_node_features."""
    from deep_fem_uav_wing.gnn import synth

    meshes = [synth.surface_tri_wing(900 + 130 * i, seed=20 + i) for i in range(5)]
    gps = [[0.1 * i, 0.2, 0.3 + 0.05 * i, 0.4] for i in range(5)]
    xs, ys = [], []
    for m, gp in zip(meshes, gps):
        x, y = ops.node_features(torch.from_numpy(m["pos"]).cuda(), torch.from_numpy(m["normal"]).cuda(), torch.from_numpy(m["stress_vm_raw"]).cuda(), gp)
        xs.append(x)
        ys.append(y)
    ptr = np.concatenate([[0], np.cumsum([m["num_nodes"] for m in meshes])])
    xb, yb = ops.node_features_batched(torch.cat([torch.from_numpy(m["pos"]) for m in meshes]).cuda(), torch.cat([torch.from_numpy(m["normal"]) for m in meshes]).cuda(),
                                       torch.cat([torch.from_numpy(m["stress_vm_raw"]) for m in meshes]).cuda(), torch.tensor(gps, dtype=torch.float32).cuda(),
                                       torch.from_numpy(ptr).cuda(), max(m["num_nodes"] for m in meshes))
    assert torch.equal(xb, torch.cat(xs)) and torch.equal(yb, torch.cat(ys))
    xn, yn = ops.node_features_batched(torch.cat([torch.from_numpy(m["pos"]) for m in meshes]).cuda(), torch.cat([torch.from_numpy(m["normal"]) for m in meshes]).cuda(), None,
                                       torch.tensor(gps, dtype=torch.float32).cuda(), torch.from_numpy(ptr).cuda(), 2000, normalize_pos=False)
    assert yn is None and torch.equal(xn[:, 3:], xb[:, 3:]) and torch.equal(xn[:, :3], torch.cat([torch.from_numpy(m["pos"]) for m in meshes]).cuda())


@pytest.mark.parametrize("dt,H,N", [(torch.float32, 128, 128 * 2 + 1), (torch.float32, 128, 128 * 5 + 127), (torch.bfloat16, 64, 128 * 3 + 77),
                                    (torch.bfloat16, 256, 128 * 2 + 9)])
def test_tensor_core_linear_writes_nothing_outside_its_rows(ops, dt, H, N):
    """Guard bands around every output of the fused SAGE linear (ragged last tile: the persistent kernel's epilogue takes its
    predicated path there): `out`, `pre` and the LayerNorm statistics are written for rows 0..N-1 only, and the guarded call gives
    the same bits as the plain wrapper.  (compute-sanitizer is not available on the GPU pool: this is the bounds check.)"""
    from deep_fem_uav_wing.gnn import _cabi

    lib = _cabi.lib
    G = 160  # guard rows on both sides
    torch.manual_seed(N)
    agg = torch.randn(N, H, device="cuda").to(dt)
    x = torch.randn(N, H, device="cuda").to(dt)
    wl = (torch.randn(H, H, device="cuda") / H ** 0.5).to(dt)
    wr = (torch.randn(H, H, device="cuda") / H ** 0.5).to(dt)
    b, g, be = torch.randn(H, device="cuda"), torch.rand(H, device="cuda") + 0.5, torch.randn(H, device="cuda")
    ref_out, ref_pre, ref_stats, _ = ops.linear_fwd(agg, wl, x, wr, bias=b, ln=(g, be), relu=True, residual=x, dropout_p=0.1, seed=7, save_pre=True)

    def guarded(cols, dtype, sentinel):
        buf = torch.full((N + 2 * G, cols), sentinel, dtype=dtype, device="cuda")
        return buf, buf[G:G + N]

    sent = 1024.0  # exact in bf16
    out_b, out = guarded(H, dt, sent)
    pre_b, pre = guarded(H, dt, sent)
    st_b, st = guarded(2, torch.float32, sent)
    flags = _cabi.EP_LAYERNORM | _cabi.EP_RELU | _cabi.EP_RESIDUAL | _cabi.EP_DROPOUT
    dtc = _cabi.DFW_F32 if dt == torch.float32 else _cabi.DFW_BF16
    ws_bytes = lib.dfw_linear_ws_bytes(H, H, H, dtc)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _cabi.check(lib.dfw_linear_fwd(agg.data_ptr(), wl.data_ptr(), H, x.data_ptr(), wr.data_ptr(), H, b.data_ptr(), g.data_ptr(), be.data_ptr(), 1e-5,
                                   x.data_ptr(), 0.1, 7, out.data_ptr(), pre.data_ptr(), st.data_ptr(), None, None, None, N, H, flags, dtc,
                                   ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(out, ref_out) and torch.equal(pre, ref_pre) and torch.equal(st, ref_stats)
    for buf in (out_b, pre_b, st_b):
        assert bool((buf[:G].float() == sent).all()) and bool((buf[G + N:].float() == sent).all()), "a row outside [0, N) was written"


@_needs_tc
def test_tiny_k_linear_with_bf16_output_equals_fp32_launch_plus_cast(ops):
    """DFW_EP_OUT_BF16: the encoder's first linear (fp32 features and weights) stored as bf16 in one launch gives the bits of the
    fp32 launch followed by dfw_cast; shapes the tiny-K kernel does not take are refused."""
    from deep_fem_uav_wing.gnn import _cabi

    torch.manual_seed(0)
    for n, k, h in ((5000, 10, 64), (777, 3, 128), (1, 16, 4)):
        x = torch.randn(n, k, device="cuda")
        w = torch.randn(h, k, device="cuda") / k ** 0.5
        b = torch.randn(h, device="cuda")
        ref, _, _, _ = ops.linear_fwd(x, w, bias=b, relu=True)
        got, _, _, _ = ops.linear_fwd(x, w, bias=b, relu=True, out_bf16=True)
        assert got.dtype == torch.bfloat16 and torch.equal(got, ops.cast(ref, torch.bfloat16))
    x = torch.randn(256, 64, device="cuda")
    w = torch.randn(128, 64, device="cuda")
    with pytest.raises(RuntimeError, match="DFW_EP_OUT_BF16"):
        ops.linear_fwd(x, w, relu=True, out_bf16=True)  # K = 64 is a tensor-core shape
