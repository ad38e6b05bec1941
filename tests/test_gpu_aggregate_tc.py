"""Tensor-core block-sparse aggregation (GPU, through the C ABI): the device-built block plan against the numpy design oracle
(``oracle/blocked_agg_oracle.py``) bit for bit, and ``dfw_sage_aggregate_tc`` against the plain-C CSR aggregation
(``oracle/csr_oracle.c``) - mean and sum, H in {64, 128, 256}, ragged last blocks, isolated rows, duplicate edges, long rows,
random graphs with poor locality (many chunks per block)."""
import numpy as np
import pytest
import torch

from helpers import TOL_BF16, assert_bound, assert_no_rounding_bias, bf16_ulp, launched_kernels, record, rel_max, rounding_bias
from oracle import csr_aggregate_c, csr_oracle_c
from oracle.blocked_agg_oracle import build_blocks


def tc_agg_bound(rowptr, col, row_scale, x, S):
    """fp64 reference and per-element error bound of ``dfw_sage_aggregate_tc`` on the bf16 rows ``x`` it read.

    Row i of block b = i // 128 is r_i = s_i sum_j m_ij x_j (m_ij the multiplicity of edge j -> i, s_i the row scale or 1),
    and A_i = |s_i| sum_j m_ij |x_j|.  The kernel multiplies the block's [128 x 64] adjacency chunks (entries m_ij <= 8, exact
    in bf16) by the staged rows on the tensor cores.  Products of a bf16 value with a small integer are exact, so all the
    error comes from the fp32 accumulator in TMEM: every chunk adds four K = 16 steps into EVERY row of the block, so row i
    sees K_i = 4 ceil(max(S_b, 128) / 64) accumulate steps, S_b the block's staged rows from the plan.  Every partial sum is
    at most A_i / |s_i| in magnitude, and a step that TRUNCATES its result (as the tensor-core dW accumulator was found to
    do; round-to-nearest is not assumed) is off by less than one fp32 ulp of it, 2^-23 of that.  The epilogue's multiply by
    s_i rounds once more (2^-24).  So the pre-store error is
        E_i <= (K_i 2^-23 + 2^-24) A_i     (the second-order term K_i 2^-47 A_i is covered by a factor 1 + 2^-20),
    and the bf16 store adds at most half an ulp of the computed value, 2^-8 (|r_i| + E_i):
        |got - r_i| <= E_i + 2^-8 (|r_i| + E_i).
    Returns (r, E, bound) as float64 [n_rows, H] on x's device; S is the per-block staged row count (blk_meta[:, 1])."""
    dev = x.device
    n = rowptr.numel() - 1
    rp, cl = rowptr.to(dev).long(), col.to(dev).long()
    seg = torch.repeat_interleave(torch.arange(n, device=dev), rp[1:] - rp[:-1])
    x64 = x.double()
    r = torch.zeros(n, x.shape[1], dtype=torch.float64, device=dev)
    A = torch.zeros_like(r)
    for e0 in range(0, cl.numel(), 1 << 20):  # in slices: a gathered edge set of the 288k lattice would take 8 GB at once
        sl = slice(e0, e0 + (1 << 20))
        xs = x64.index_select(0, cl[sl])
        r.index_add_(0, seg[sl], xs)
        A.index_add_(0, seg[sl], xs.abs())
    if row_scale is not None:
        s = row_scale.to(dev).double()[:, None]
        r, A = r * s, A * s.abs()
    K = 4 * ((S.to(dev).long().clamp_min(128) + 63) // 64)[torch.arange(n, device=dev) // 128]
    E = (K.double() * 2.0 ** -23 + 2.0 ** -24)[:, None] * A * (1 + 2.0 ** -20)
    return r, E, E + 2.0 ** -8 * (r.abs() + E)


def _staged(plan, n):
    return plan.blk_meta.view(-1, 4)[:(n + 127) // 128, 1]


def test_tc_agg_bound_rejects_a_dropped_neighbour_and_a_truncating_store():
    rng = np.random.default_rng(3)
    n, h = 2048, 64  # >= 1e5 elements: the rounding-bias check applies
    ei = rng.integers(0, n, size=(2, 14 * n)).astype(np.int64)
    rowptr, col, _, inv = csr_oracle_c(ei, n)
    rowptr, col, inv = torch.from_numpy(rowptr), torch.from_numpy(col), torch.from_numpy(inv)
    x = torch.from_numpy(rng.standard_normal((n, h)).astype(np.float32)).bfloat16()
    S = torch.full(((n + 127) // 128,), 1000)
    r, E, bound = tc_agg_bound(rowptr, col, inv, x, S)
    assert assert_bound("rne", r.bfloat16(), r, bound) <= 1  # the exact result rounded to nearest even passes
    assert assert_no_rounding_bias("rne", r.bfloat16(), r, E) is not None
    # one neighbour dropped: the last edge of every row
    last = rowptr[1:] - 1
    has = rowptr[1:] > rowptr[:-1]
    dropped = r.clone()
    dropped[has] -= inv.double()[has][:, None] * x.double()[col[last[has]].long()]
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_bound("drop", dropped.bfloat16(), r, bound)
    # a store that truncates toward zero instead of rounding
    trunc = (r.float().view(torch.int32) & ~0xFFFF).view(torch.float32).bfloat16()
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_bound("trunc", trunc, r, bound)
    with pytest.raises(AssertionError, match="store error"):
        assert_no_rounding_bias("trunc", trunc, r, E)


@pytest.fixture(scope="module")
def ops():
    from deep_fem_uav_wing.gnn import ops as _ops

    return _ops


def _graphs():
    from deep_fem_uav_wing.gnn import synth

    rng = np.random.default_rng(0)
    out = {}
    out["tet_5k"] = (synth.tet_lattice_wing(5000, seed=1)["edge_index"], None)
    m = synth.surface_tri_wing(3000, seed=2)
    out["tri_3k"] = (m["edge_index"], m["num_nodes"])
    n = 1000
    ei = rng.integers(0, n, size=(2, 9000)).astype(np.int64)  # random: duplicates, self loops, ~14 chunks per block
    ei[1, :300] = 5  # one long row
    ei = ei[:, ei[1] != 77]  # one isolated row
    out["random_1k"] = (ei, n)
    out["single_row"] = (np.array([[0, 0, 0], [0, 0, 0]], dtype=np.int64), 1)
    out["no_edges"] = (np.zeros((2, 0), dtype=np.int64), 300)
    out["ragged_129"] = (rng.integers(0, 129, size=(2, 700)).astype(np.int64), 129)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tet_5k", "tri_3k", "random_1k", "single_row", "no_edges", "ragged_129"])
def test_block_plan_matches_design_oracle(ops, name):
    ei, n = _graphs()[name]
    n = int(ei.max()) + 1 if n is None else n
    rowptr, col, _, _ = csr_oracle_c(ei, n)
    plan = ops.build_agg_plan(torch.from_numpy(rowptr).cuda(), torch.from_numpy(col).cuda(), n)
    assert plan.check()
    blk_ptr, blk_src, _ = build_blocks(rowptr, col, 128)
    meta = plan.blk_meta.cpu().numpy().reshape(-1, 4)
    src = plan.plan_src.cpu().numpy()
    rec = plan.plan_rec.cpu().numpy().view(np.uint16).reshape(-1, 136)
    slots = plan.plan_slot.cpu().numpy().view(np.uint16)
    nb = (n + 127) // 128
    assert meta.shape[0] >= nb
    total = 0
    for b in range(nb):
        s_off, S, t_off, nent = (int(v) for v in meta[b])
        r0, r1 = 128 * b, min(128 * b + 128, n)
        e0, e1 = int(rowptr[r0]), int(rowptr[r1])
        # slots: the block's own rows hold 0 .. 127 (slot = row - r0, used or not), the distinct halo sources follow ascending
        distinct = blk_src[blk_ptr[b]:blk_ptr[b + 1]].astype(np.int64)  # the design oracle's ascending distinct sources
        halo = distinct[(distinct < r0) | (distinct >= r1)]
        assert S == 128 + halo.size and s_off % 64 == 0 and t_off % 8 == 0
        assert np.array_equal(src[s_off:s_off + 128], np.minimum(r0 + np.arange(128), n - 1))
        assert np.array_equal(src[s_off + 128:s_off + S], halo)
        pad = (S + 63) // 64 * 64
        assert np.all(src[s_off + S:s_off + pad] == (halo[-1] if halo.size else min(r0 + 127, n - 1)))
        # adjacency entries: one per distinct (slot, row) pair with its multiplicity, ordered by (slot, row)
        cols_b = col[e0:e1].astype(np.int64)
        own = (cols_b >= r0) & (cols_b < r1)
        slot_b = np.where(own, cols_b - r0, 128 + np.searchsorted(halo, cols_b))
        rows_of_edges = np.repeat(np.arange(r1 - r0), np.diff(rowptr[r0:r1 + 1]))
        pairs, counts = np.unique(np.stack([slot_b, rows_of_edges]), axis=1, return_counts=True) if e1 > e0 else (np.zeros((2, 0), np.int64), np.zeros(0, np.int64))
        want = ((counts - 1) << 13 | pairs[1] << 6 | (pairs[0] & 63)).astype(np.uint16)
        assert nent == want.size and rec[b, 0] == S and rec[b, 1] == nent
        assert np.array_equal(slots[t_off:t_off + nent], want)
        nch = pad // 64
        cptr = np.searchsorted(pairs[0], 64 * np.arange(nch + 1))
        assert np.array_equal(rec[b, 2:3 + nch], cptr.astype(np.uint16))
        total += S
    assert abs(plan.staged_rows_per_row * n - total) < 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 128, 256])
@pytest.mark.parametrize("name", ["tet_5k", "tri_3k", "random_1k", "single_row", "no_edges", "ragged_129"])
def test_aggregate_tc_matches_c_oracle(ops, name, h):
    ei, n = _graphs()[name]
    n = int(ei.max()) + 1 if n is None else n
    rng = np.random.default_rng(h)
    x = torch.from_numpy(rng.standard_normal((n, h)).astype(np.float32)).bfloat16()
    rowptr, col, _, inv = csr_oracle_c(ei, n)
    g = ops.get_graph(torch.from_numpy(ei).cuda(), n)
    plan = ops.build_agg_plan(g.rowptr, g.col, n)
    assert plan.check()
    for scale, inv_np in ((g.inv_deg, inv), (None, None)):  # mean, then plain sum
        ref = torch.from_numpy(csr_aggregate_c(rowptr, col, inv_np, x.float().numpy()))
        got, names = launched_kernels(lambda: ops.aggregate_tc(plan, scale, x.cuda(), g.num_edges))
        assert any("k_aggregate_tc" in k for k in names), sorted(set(names))
        assert got.dtype == torch.bfloat16 and got.shape == (n, h)
        gf = got.float().cpu()
        assert torch.isfinite(gf).all()
        err = rel_max(gf, ref) if ref.abs().max() > 0 else float(gf.abs().max())
        mism = int((got.cpu() != ref.bfloat16()).sum())
        assert err < TOL_BF16
        r, E, bound = tc_agg_bound(g.rowptr, g.col, scale, x.cuda(), _staged(plan, n))
        margin = assert_bound(f"aggregate_tc {name} H={h}", got, r, bound)
        bias = assert_no_rounding_bias(f"aggregate_tc {name} H={h}", got, r, E)
        record("aggregate_tc_vs_c_oracle", graph=name, H=h, mean=scale is not None, rel_max=err, bf16_mismatches=mism, elements=n * h,
               err_over_bound=margin, rounding_bias=bias)
        assert torch.equal(got, ops.aggregate_tc(plan, scale, x.cuda(), g.num_edges))  # deterministic
        same = ops.aggregate(g.rowptr, g.col, scale, x.cuda())
        assert rel_max(gf, same.float().cpu()) < 2.0 ** -7 if ref.abs().max() > 0 else True


@pytest.mark.gpu
def test_aggregate_tc_rejects_what_it_cannot_take(ops):
    from deep_fem_uav_wing.gnn import _cabi

    ei = np.array([[0, 1], [1, 0]], dtype=np.int64)
    g = ops.get_graph(torch.from_numpy(ei).cuda(), 2)
    plan = ops.build_agg_plan(g.rowptr, g.col, 2)
    with pytest.raises(TypeError):
        ops.aggregate_tc(plan, None, torch.zeros(2, 64, device="cuda"))
    with pytest.raises(_cabi.DfwError, match="64, 128 or 256"):
        ops.aggregate_tc(plan, None, torch.zeros(2, 96, device="cuda", dtype=torch.bfloat16))
    # a block with more edges than the plan holds is reported, not mis-computed
    n = 200
    hub = np.stack([np.arange(5000) % n, np.zeros(5000, dtype=np.int64)]).astype(np.int64)
    gh = ops.get_graph(torch.from_numpy(hub).cuda(), n)
    ph = ops.build_agg_plan(gh.rowptr, gh.col, n)
    assert not ph.check()
    # so is an edge repeated more often than the 3-bit multiplicity field holds
    rep = np.stack([np.zeros(9, dtype=np.int64), np.ones(9, dtype=np.int64)])
    gr = ops.get_graph(torch.from_numpy(rep).cuda(), 2)
    assert not ops.build_agg_plan(gr.rowptr, gr.col, 2).check()
    rep8 = rep[:, :8].copy()
    g8 = ops.get_graph(torch.from_numpy(rep8).cuda(), 2)
    p8 = ops.build_agg_plan(g8.rowptr, g8.col, 2)
    assert p8.check()
    out8 = ops.aggregate_tc(p8, None, torch.ones(2, 64, device="cuda", dtype=torch.bfloat16))
    assert out8[1].float().eq(8).all() and out8[0].float().eq(0).all()


@pytest.mark.gpu
def test_large_mesh_inference_path_relabels_nodes_and_matches_the_plain_path(ops, monkeypatch):
    """GraphSAGEModel bf16 inference on a randomly numbered tet mesh: the block plan + k-d relabelling path (input rows
    permuted once, output restored) must give the plain path's predictions in the CALLER's node order."""
    from deep_fem_uav_wing.gnn import synth
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    mesh = synth.tet_lattice_wing(120000, seed=3, node_order="random")
    n = mesh["num_nodes"]
    x, ei = torch.from_numpy(mesh["x"]).cuda(), torch.from_numpy(mesh["edge_index"]).cuda()
    torch.manual_seed(5)
    model = GraphSAGEModel(10, 128, 1, 2, dropout=0.0).cuda().eval().set_compute_dtype(torch.bfloat16)
    model.mesh_plan = "always"  # ('auto' prepares a mesh from its second forward on: covered at the end of this test)
    monkeypatch.setattr(ops, "TC_AGG_MIN_NODES", 1000)
    monkeypatch.setattr(ops, "TC_AGG_MIN_REUSE", 0.0)  # (the policy would leave a 120k-node mesh with ~4.5 staged rows per row to the gather kernel)
    tc_calls = []
    real_tc = ops.aggregate_tc
    monkeypatch.setattr(ops, "aggregate_tc", lambda *a, **k: (tc_calls.append(1), real_tc(*a, **k))[1])
    with torch.no_grad():
        out_plan = model(x, ei)
    assert len(tc_calls) == 2, "every SAGE layer of the large-mesh path must run the tensor-core block aggregation"
    ig = ops.get_inference_graph(ei, n, pos=x[:, :3], reorder="auto")
    assert ig.order is not None and ig.graph.plan.usable
    assert ig.staged_rows_per_row_given > 8 and ig.staged_rows_per_row < 4.8  # random numbering -> compact blocks
    assert torch.equal(torch.sort(ig.new_id).values, torch.arange(n, device="cuda"))
    record("kd_relabel_random_tet_120k", staged_given=ig.staged_rows_per_row_given, staged_kd=ig.staged_rows_per_row)
    monkeypatch.setattr(ops, "TC_AGG_MIN_NODES", 10 ** 12)
    with torch.no_grad():
        out_plain = model(x, ei)
    assert len(tc_calls) == 2  # the plain path stays on the gather kernel
    assert out_plan.shape == out_plain.shape == (n, 1)
    err = rel_max(out_plan.float().cpu(), out_plain.float().cpu())
    record("large_mesh_inference_path_vs_plain", rel_max=err)
    assert err < TOL_BF16
    # 'never': plan in the given numbering, no permutation
    monkeypatch.setattr(ops, "TC_AGG_MIN_NODES", 1000)
    model.node_reorder = "never"
    with torch.no_grad():
        out_never = model(x, ei)
    assert rel_max(out_never.float().cpu(), out_plain.float().cpu()) < TOL_BF16
    # 'auto': a mesh is prepared from its SECOND forward on (a screening loop sees every graph once)
    model.mesh_plan, model.node_reorder = "auto", "auto"
    ei_new = ei.clone()
    n0 = len(tc_calls)
    with torch.no_grad():
        first = model(x, ei_new)
        assert len(tc_calls) == n0
        second = model(x, ei_new)
        assert len(tc_calls) == n0 + 2
    assert rel_max(first.float().cpu(), out_plain.float().cpu()) < TOL_BF16 and rel_max(second.float().cpu(), out_plain.float().cpu()) < TOL_BF16


@pytest.mark.gpu
@pytest.mark.parametrize("order,reorder", [("native", "never"), ("random", "never"), ("random", "always")])
@pytest.mark.parametrize("h", [128, 256])
def test_aggregate_tc_long_pipelines_match_the_gather_kernel(ops, order, reorder, h):
    """Many blocks per CTA and many chunks per block (a randomly numbered lattice stages ~14 rows per output row): every
    barrier of the pipeline wraps its phase many times.  (A phase race in the own-row path passed every small-graph test and
    only showed beyond ~30 chunks per CTA.)  Every element is held to the fp64 bound of tc_agg_bound, and the gather kernel on
    the same CSR is compared for the record."""
    import bench

    ei, pos, n = bench.cfg4_lattice_device((30, 60, 160), torch.device("cuda"), order)
    ops._INF_CACHE.clear()
    ig = ops.get_inference_graph(ei, n, pos=pos, reorder=reorder)
    g = ig.graph
    assert g.plan.usable and (ig.order is not None) == (reorder == "always")
    x = torch.randn(n, h, device="cuda", generator=torch.Generator(device="cuda").manual_seed(h)).bfloat16()
    xp = x if ig.order is None else x.index_select(0, ig.order)
    got, names = launched_kernels(lambda: ops.aggregate_tc(g.plan, g.inv_deg, xp, g.num_edges))
    assert any("k_aggregate_tc" in k for k in names), sorted(set(names))
    ref = ops.aggregate(g.rowptr, g.col, g.inv_deg, xp)
    err = (got.float() - ref.float()).abs().max().item()
    mism = int((got != ref).sum())
    r, E, bound = tc_agg_bound(g.rowptr, g.col, g.inv_deg, xp, _staged(g.plan, n))
    margin = assert_bound(f"aggregate_tc 288k {order} {reorder} H={h}", got, r, bound)
    bias = assert_no_rounding_bias(f"aggregate_tc 288k {order} {reorder} H={h}", got, r, E)
    record("aggregate_tc_vs_gather_288k", order=order, reorder=reorder, H=h, max_abs=err, bf16_mismatches=mism, elements=n * h,
           staged_rows_per_row=g.plan.staged_rows_per_row, err_over_bound=margin, rounding_bias=bias)
    assert mism < 1e-3 * n * h
    ops._INF_CACHE.clear()
    ops.clear_graph_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 256])
def test_aggregate_tc_rectangular_sources_beyond_the_destination_rows(ops, h):
    """The partitioned layout: n_own destination rows whose sources index [own | halo] (more rows than destinations).  The block
    kernel with a plan of that rectangular CSR must match the gather kernel on the same CSR."""
    from deep_fem_uav_wing.gnn import synth

    mesh = synth.tet_lattice_wing(60000, seed=2)
    n_ext = mesh["num_nodes"]
    n_own = (n_ext * 2 // 3) // 128 * 128 + 37  # ragged last block
    ei = torch.from_numpy(mesh["edge_index"]).cuda()
    g = ops.get_graph(ei, n_ext)
    rowptr = g.rowptr[: n_own + 1].contiguous()
    e_loc = int(rowptr[-1].item())
    col = g.col[:e_loc].contiguous()
    assert int(col.max()) >= n_own  # there ARE halo sources behind the destination rows
    inv_deg = g.inv_deg[:n_own].contiguous()
    x = torch.randn(n_ext, h, device="cuda").bfloat16()
    plan = ops.build_agg_plan(rowptr, col, n_own)
    assert plan.check()
    got = ops.aggregate_tc(plan, inv_deg, x, e_loc, n_rows=n_own)
    want = ops.aggregate_rows(rowptr, col, inv_deg, x, n_own)
    assert got.shape == want.shape == (n_own, h)
    err = (got.float() - want.float()).abs().max().item() / want.float().abs().max().item()
    assert err < 1e-2, err
    mism = (got != want).float().mean().item()
    assert mism < 0.05, mism  # same fp32 sums up to association order: almost all elements round to the same bf16
    with pytest.raises(ValueError):
        ops.aggregate_tc(plan, inv_deg, x[: n_own - 1], e_loc, n_rows=n_own)


def _cancel_graph(n=4096, pairs=6, seed=7):
    """Every row takes `pairs` neighbour pairs (2m, 2m + 1) whose rows are x and almost -x: sums of large terms that cancel."""
    rng = np.random.default_rng(seed)
    m = rng.integers(0, n // 2, size=(n, pairs))
    src = np.stack([2 * m, 2 * m + 1], axis=2).reshape(n, -1)
    dst = np.repeat(np.arange(n), 2 * pairs)
    x = rng.standard_normal((n, 128)).astype(np.float32) * 64
    x[1::2] = -x[0::2] + rng.standard_normal((n // 2, 128)).astype(np.float32) * 2.0 ** -4
    return np.stack([src.reshape(-1), dst]).astype(np.int64), torch.from_numpy(x).bfloat16()


@pytest.mark.gpu
def test_aggregate_tc_cancellation_within_bound(ops):
    """Large terms that cancel to a small mean: the block product and the CSR-order sum round differently, by far more than one
    bf16 ulp of the RESULT, yet both stay within the bound relative to the sum of |terms|."""
    ei, x = _cancel_graph()
    n = x.shape[0]
    g = ops.get_graph(torch.from_numpy(ei).cuda(), n)
    plan = ops.build_agg_plan(g.rowptr, g.col, n)
    assert plan.check()
    got = ops.aggregate_tc(plan, g.inv_deg, x.cuda(), g.num_edges)
    r, E, bound = tc_agg_bound(g.rowptr, g.col, g.inv_deg, x.cuda(), _staged(plan, n))
    assert float((E / r.abs().clamp_min(1e-300)).median()) > 2.0 ** -9  # the construction cancels: E is a sizeable part of |r|
    margin = assert_bound("aggregate_tc cancellation", got, r, bound)
    gather = ops.aggregate(g.rowptr, g.col, g.inv_deg, x.cuda())
    ulps = ((got.double() - r).abs() / bf16_ulp(r)).max().item()
    ulps_gather = ((gather.double() - r).abs() / bf16_ulp(r)).max().item()
    record("aggregate_tc_cancellation", err_over_bound=margin, max_err_ulps_of_result=ulps, gather_max_err_ulps_of_result=ulps_gather,
           bf16_mismatches_vs_gather=int((got != gather).sum()), elements=got.numel())


@pytest.mark.gpu
def test_aggregate_tc_nonfinite_inputs_poison_the_blocks_that_stage_them(ops):
    """One +Inf and one NaN source.  The gather kernel makes exactly the rows that read them non-finite.  The block product
    multiplies EVERY staged row by a mostly-zero adjacency column (0 * Inf = NaN), so each block that stages a non-finite row
    - as one of its own 128 rows, as a halo source or as plan padding - comes out non-finite in every row.  Finite rows stay
    within the bound."""
    from deep_fem_uav_wing.gnn import synth

    mesh = synth.tet_lattice_wing(5000, seed=1)
    ei = mesh["edge_index"]
    n = int(ei.max()) + 1
    rng = np.random.default_rng(11)
    x = torch.from_numpy(rng.standard_normal((n, 64)).astype(np.float32)).bfloat16()
    x[1000, 5] = float("inf")
    x[3333, 17] = float("nan")
    g = ops.get_graph(torch.from_numpy(ei).cuda(), n)
    plan = ops.build_agg_plan(g.rowptr, g.col, n)
    assert plan.check()
    got = ops.aggregate_tc(plan, g.inv_deg, x.cuda(), g.num_edges).cpu()
    gather = ops.aggregate(g.rowptr, g.col, g.inv_deg, x.cuda()).cpu()
    bad_tc = set(torch.nonzero(~torch.isfinite(got.float()).all(dim=1)).flatten().tolist())
    bad_gather = set(torch.nonzero(~torch.isfinite(gather.float()).all(dim=1)).flatten().tolist())
    # the rows that read a non-finite source, from the CSR
    rp, cl = g.rowptr.cpu().numpy(), g.col.cpu().numpy()
    readers = set(np.repeat(np.arange(n), np.diff(rp))[np.isin(cl, [1000, 3333])].tolist())
    assert bad_gather == readers
    # every row of every block whose staged rows (plan_src over the padded S) include a non-finite source
    meta = plan.blk_meta.view(-1, 4).cpu().numpy()
    src = plan.plan_src.cpu().numpy()
    poisoned = [b for b in range((n + 127) // 128)
                if np.isin(src[meta[b, 0]:meta[b, 0] + (max(int(meta[b, 1]), 128) + 63) // 64 * 64], [1000, 3333]).any()]
    expect = {i for b in poisoned for i in range(128 * b, min(128 * b + 128, n))}
    record("aggregate_tc_nonfinite", gather_rows=sorted(bad_gather), tc_rows=len(bad_tc), tc_blocks=sorted({i // 128 for i in bad_tc}),
           staging_blocks=poisoned)
    assert bad_gather <= bad_tc
    assert bad_tc == expect
    fin = torch.tensor(sorted(set(range(n)) - bad_tc), dtype=torch.long)
    r, E, bound = tc_agg_bound(g.rowptr, g.col, g.inv_deg, x.cuda(), _staged(plan, n))
    assert_bound("aggregate_tc finite rows next to Inf / NaN", got[fin], r.cpu()[fin], bound.cpu()[fin])
