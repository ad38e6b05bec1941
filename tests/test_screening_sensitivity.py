"""Design sensitivities of the screener (gnn/screening.py, sensitivities=True): the KS aggregate and its seed
(dfw_case_ks_seed), the per-case column sums (dfw_case_column_sums), the input-gradient backward without weight-gradient
work, and the screener's records - against an fp64 restatement on the oracle model.

The restatement lives here, in the test that uses it: fp64 torch autograd on ``oracle.sage_oracle.GraphSAGEModelRef``
with the screened-set rule of ``test_screening.summary_oracle``.
"""
import copy
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from helpers import Arena, record

REPO = Path(__file__).resolve().parent.parent
PKG = REPO / "deep-fem-uav-wing_b200"
EPS64 = 2.0 ** -53
PARAM_OFFSET = {"span_m": 1.0, "chord_m": 0.2, "sweep_deg": 0.0, "thickness_ratio": 0.05}
PARAM_SCALE = {"span_m": 1.0, "chord_m": 0.3, "sweep_deg": 30.0, "thickness_ratio": 0.10}  # x[:, 6:10], dataset.py:122-127


# ---- fp64 restatement ------------------------------------------------------------------------------------------------
def screened_sets(u, pos_y, case_ptr, mask=None, root_band=0.05):
    """Per case, the rows (within the case) of S_b: screened (mask, or pos_y > root_band * (max_y - min_y) of the case, in
    fp64) and with a finite fp32 stress expm1f(u) - the rows ``summary_oracle`` takes the max stress over."""
    u = np.asarray(u, dtype=np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        fin = np.isfinite(np.expm1(u))
    sets = []
    for b in range(len(case_ptr) - 1):
        r0, r1 = int(case_ptr[b]), int(case_ptr[b + 1])
        if mask is not None:
            scr = np.asarray(mask[r0:r1]).astype(bool)
        elif r1 > r0:
            y = pos_y[r0:r1]
            scr = y.astype(np.float64) > root_band * (float(y.max()) - float(y.min()))
        else:
            scr = np.zeros(0, bool)
        sets.append(np.nonzero(scr & fin[r0:r1])[0])
    return sets


def ks_oracle(u64, case_ptr, sets, rho):
    """KS_b = max u + ln(sum exp(rho (u - max u))) / rho over S_b as differentiable fp64 torch scalars (None: empty set)."""
    out = []
    for b, idx in enumerate(sets):
        if idx.size == 0:
            out.append(None)
            continue
        v = u64[int(case_ptr[b]) + torch.from_numpy(idx)]
        out.append(torch.logsumexp(rho * v, 0) / rho)
    return out


def ks_and_seed_oracle(u, case_ptr, sets, rho):
    """fp64 [B,2] records [KS_b, |S_b|] and the fp64 seed dKS_b/du from the values ``u`` (autograd of sum_b KS_b)."""
    u64 = torch.from_numpy(np.asarray(u, dtype=np.float64)).requires_grad_()
    ks = ks_oracle(torch.nan_to_num(u64, nan=0.0, posinf=0.0, neginf=0.0), case_ptr, sets, rho)
    live = [k for k in ks if k is not None]
    seed = torch.autograd.grad(sum(live), u64)[0].numpy() if live else np.zeros(len(u))
    rec = np.array([[float(k.detach()) if k is not None else 0.0, len(s)] for k, s in zip(ks, sets)], dtype=np.float64).reshape(-1, 2)
    return rec, seed


def oracle_param_sensitivities(ref, x, edge_index, pos_y, case_ptr, rho, mask=None, dtype=torch.float64, seed=None):
    """Per case [KS_b, |S_b|, dKS_b/dx_6 .. dKS_b/dx_9 summed over the case's rows] of the oracle model in ``dtype``.
    With ``seed`` (an [N] array) the vector-Jacobian product uses that seed instead of the model's own dKS/du."""
    m = copy.deepcopy(ref).to(dtype)
    xt = torch.as_tensor(x).to(dtype).requires_grad_()
    pred = m(xt, torch.as_tensor(edge_index)).reshape(-1)
    sets = screened_sets(pred.detach().float().numpy(), pos_y, case_ptr, mask)
    ks = ks_oracle(pred.double(), case_ptr, sets, rho)
    if seed is None:
        live = [k for k in ks if k is not None]
        g = torch.autograd.grad(sum(live), xt)[0] if live else torch.zeros_like(xt)
    else:
        g = torch.autograd.grad(pred, xt, torch.as_tensor(seed).to(dtype))[0]
    g = g.double().numpy()
    out = np.zeros((len(case_ptr) - 1, 6))
    for b, k in enumerate(ks):
        r0, r1 = int(case_ptr[b]), int(case_ptr[b + 1])
        out[b, 0] = float(k.detach()) if k is not None else 0.0
        out[b, 1] = len(sets[b])
        out[b, 2:] = g[r0:r1, 6:10].sum(axis=0)
    return out


def ks_stress_and_gradient(rec):
    """ks_stress_pa and d ks_stress_pa / d (span_m, chord_m, sweep_deg, thickness_ratio) from [KS, n, dKS/dx_6..9]."""
    f = np.exp(rec[0])
    return np.expm1(rec[0]), np.array([f * rec[2 + j] / s for j, s in enumerate(PARAM_SCALE.values())])


def _oracle_model(hidden=16, layers=2, seed=0):
    from oracle.sage_oracle import GraphSAGEModelRef

    torch.manual_seed(seed)
    return GraphSAGEModelRef(10, hidden, 1, layers, dropout=0.0).eval()


def _union(meshes):
    """Disjoint union of synth meshes: x, edge_index, pos, case_ptr (numpy)."""
    offs = np.cumsum([0] + [m["num_nodes"] for m in meshes])
    x = np.concatenate([m["x"] for m in meshes])
    ei = np.concatenate([m["edge_index"] + o for m, o in zip(meshes, offs[:-1])], axis=1)
    pos = np.concatenate([m["pos"] for m in meshes])
    return x, ei, pos, offs.astype(np.int64)


# ---- CPU: the restatement itself -------------------------------------------------------------------------------------
def test_ks_known_answers():
    rho = 100.0
    ptr = np.array([0, 5, 12, 12, 16])
    u = np.array([1, 2, 3, 4, 7.5, 9, 9, 9, 9, 9, 9, 9, 3, 3, 3, 3], dtype=np.float32)
    y = np.zeros(16, np.float32)
    mask = np.zeros(16, bool)
    mask[4] = True           # case 0: one screened row
    mask[5:12] = True        # case 1: seven equal rows
    rec, seed = ks_and_seed_oracle(u, ptr, screened_sets(u, y, ptr, mask), rho)  # case 2 empty, case 3 no screened row
    assert rec[0, 0] == 7.5 and rec[0, 1] == 1 and seed[4] == 1.0 and seed[:4].tolist() == [0, 0, 0, 0]
    assert abs(rec[1, 0] - (9.0 + np.log(7) / rho)) <= 1e-15 and rec[1, 1] == 7
    assert np.allclose(seed[5:12], 1 / 7, rtol=1e-12, atol=0)  # exp(rho u - logsumexp): rounding of ~rho u
    assert rec[2].tolist() == [0, 0] and rec[3].tolist() == [0, 0] and seed[12:].tolist() == [0, 0, 0, 0]


def test_screened_set_is_the_summary_rule():
    from test_screening import _ragged_case, summary_oracle

    pos, pred, ptr = _ragged_case()
    pred[ptr[2] + 11] = 95.0  # finite u whose fp32 stress overflows: outside S_b, as outside the summary's max
    pos[ptr[2] + 11, 1] = 1.4
    with np.errstate(over="ignore", invalid="ignore"):
        pa = np.expm1(pred.astype(np.float32))
    ref = summary_oracle(pa, pos[:, 1], ptr)
    sets = screened_sets(pred, pos[:, 1], ptr)
    rec, seed = ks_and_seed_oracle(pred, ptr, sets, 100.0)
    for b, idx in enumerate(sets):
        r0 = int(ptr[b])
        if idx.size == 0:
            assert ref[b, 3] == -1 and rec[b, 1] == 0
            continue
        v = pred[r0 + idx]
        k = int(np.argmax(v))
        assert np.expm1(np.float32(v[k])) == np.float32(ref[b, 2]) and idx[k] == ref[b, 3]  # same max, same row
        assert float(v[k]) <= rec[b, 0] + 1e-12 and rec[b, 0] <= float(v[k]) + np.log(idx.size) / 100.0 + 1e-12
        assert abs(seed[r0:int(ptr[b + 1])].sum() - 1.0) <= 1e-12
    assert seed[ptr[2] + 11] == 0.0


def test_parameter_gradient_matches_central_differences():
    """Pins the definition and the 1, 0.3, 30, 0.10 constants: d ks_stress_pa / dp of the fp64 oracle against a central
    finite difference in each physical parameter, two cases in one union (a case's gradient is its own)."""
    from deep_fem_uav_wing.gnn import synth

    rho = 100.0
    meshes = [synth.surface_tri_wing(300, seed=7), synth.surface_tri_wing(420, seed=8)]
    x, ei, pos, ptr = _union(meshes)
    x = x.astype(np.float64)
    for b, mesh in enumerate(meshes):  # the exact scaled parameters, so the differences are centred on them
        x[ptr[b]:ptr[b + 1], 6:10] = [(mesh["params"][k] - PARAM_OFFSET[k]) / s for k, s in PARAM_SCALE.items()]
    ref = _oracle_model(hidden=16, layers=2, seed=3).double()
    base = oracle_param_sensitivities(ref, x, ei, pos[:, 1], ptr, rho)
    worst = 0.0
    for b, mesh in enumerate(meshes):
        ks_pa, grad = ks_stress_and_gradient(base[b])
        assert base[b, 1] > 0 and np.isfinite(grad).all()
        fd = []
        for j, (k, s) in enumerate(PARAM_SCALE.items()):
            h = 1e-5 * s
            vals = []
            for sign in (1, -1):
                xp = x.copy()
                xp[ptr[b]:ptr[b + 1], 6 + j] = (mesh["params"][k] + sign * h - PARAM_OFFSET[k]) / s
                vals.append(ks_stress_and_gradient(oracle_param_sensitivities(ref, xp, ei, pos[:, 1], ptr, rho)[b])[0])
            fd.append((vals[0] - vals[1]) / (2 * h))
        err = np.abs(np.array(fd) - grad).max() / np.abs(grad).max()
        worst = max(worst, err)
        assert err <= 1e-6, (b, fd, grad)
    record("sensitivity_oracle_central_difference", max_rel_err=worst)


def test_sensitivity_record_on_the_host():
    from deep_fem_uav_wing.gnn.screening import PARAM_SCALE as SCALE
    from deep_fem_uav_wing.gnn.screening import sensitivity_record

    assert SCALE == PARAM_SCALE
    r = np.array([10.0, 5.0, 1.0, 2.0, 3.0, 4.0])
    d = sensitivity_record(r)
    assert d["ks_stress_pa"] == float(np.expm1(10.0))
    assert d["d_ks_stress_pa"] == {"span_m": np.exp(10.0) * 1.0 / 1.0, "chord_m": np.exp(10.0) * 2.0 / 0.3,
                                   "sweep_deg": np.exp(10.0) * 3.0 / 30.0, "thickness_ratio": np.exp(10.0) * 4.0 / 0.10}
    assert sensitivity_record(np.array([0.0, 0.0, 0, 0, 0, 0])) == {"ks_stress_pa": None, "d_ks_stress_pa": None}


def test_new_symbols_validate_before_any_cuda_call():
    from deep_fem_uav_wing.gnn import _cabi

    lib = _cabi.lib
    fake = 256  # never dereferenced: every call below must fail its argument checks first
    ws = lib.dfw_case_stress_summary_ws_bytes(10, 2)

    def ks(pred=fake, dtype=0, pos=fake, mask=None, cp=fake, B=2, N=10, rho=100.0, out=fake, seed=fake, w=fake, nbytes=ws):
        return lib.dfw_case_ks_seed(pred, dtype, pos, mask, cp, B, N, 0.05, rho, out, seed, w, nbytes, None)

    for kw, msg in (({"B": -1}, b"negative"), ({"N": -3}, b"negative"), ({"dtype": 5}, b"dtype"), ({"rho": 0.0}, b"rho"),
                    ({"rho": -1.0}, b"rho"), ({"rho": float("nan")}, b"rho"), ({"rho": float("inf")}, b"rho"),
                    ({"cp": None}, b"null case_ptr"), ({"out": None}, b"null case_ptr or output"), ({"pred": None}, b"null pred"),
                    ({"seed": None}, b"null pred, seed"), ({"pos": None}, b"null pred, seed or pos"),
                    ({"nbytes": ws - 1}, b"workspace too small"), ({"w": None}, b"workspace too small")):
        assert ks(**kw) != 0, kw
        assert msg in lib.dfw_last_error() and b"dfw_case_ks_seed" in lib.dfw_last_error(), (kw, lib.dfw_last_error())

    def cs(a=fake, N=10, C=10, c0=6, nc=4, cp=fake, B=2, out=fake, w=fake, nbytes=ws):
        return lib.dfw_case_column_sums(a, N, C, c0, nc, cp, B, out, w, nbytes, None)

    for kw, msg in (({"N": -1}, b"negative"), ({"C": -1}, b"negative"), ({"c0": -1}, b"negative"), ({"nc": -2}, b"negative"),
                    ({"B": -1}, b"negative"), ({"c0": 7}, b"outside"), ({"a": None}, b"null input"),
                    ({"cp": None}, b"null case_ptr"), ({"out": None}, b"null case_ptr or output"),
                    ({"nbytes": ws - 1}, b"workspace too small"), ({"w": None}, b"workspace too small")):
        assert cs(**kw) != 0, kw
        assert msg in lib.dfw_last_error() and b"dfw_case_column_sums" in lib.dfw_last_error(), (kw, lib.dfw_last_error())


def test_screener_refuses_a_bad_rho():
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    for rho in (0.0, -5.0, float("inf"), float("nan")):
        with pytest.raises(ValueError, match="ks_rho"):
            DesignScreener(GraphSAGEModel(10, 16, 1, 1), sensitivities=True, ks_rho=rho)


# ---- GPU: the two kernels --------------------------------------------------------------------------------------------
def _ks_batch(seed=21):
    """Case sizes 1, 7, 2500 (> kChunkRows), 0 (empty), 40 (every y equal: nothing screened), 30000; values near the peak
    spread over several chunks so that many seed entries matter; NaN, +Inf and a finite u whose stress overflows."""
    rng = np.random.default_rng(seed)
    sizes = [1, 7, 2500, 0, 40, 30000]
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    N = int(ptr[-1])
    pos = rng.uniform(0.0, 1.5, size=(N, 3)).astype(np.float32)
    pos[ptr[4]:ptr[5], 1] = 0.0  # max_y - min_y = 0 and no y above 0: nothing screened
    u = rng.uniform(10.0, 18.0, size=N).astype(np.float32)
    for b in (2, 5):
        r = ptr[b] + rng.choice(sizes[b], size=min(sizes[b] // 10, 600), replace=False)
        u[r] = 18.0 + rng.uniform(0.0, 0.05, size=r.size).astype(np.float32)  # a few hundred rows within 0.05 of the max
        pos[r, 1] = 1.4
    u[ptr[5] + 17] = np.nan
    u[ptr[5] + 4000] = np.inf
    u[ptr[2] + 100] = 95.0
    pos[ptr[2] + 100, 1] = 1.4
    return pos, u, ptr


def _raw_ks(pred_d, pos_d, cp_d, mask_d, rho):
    from deep_fem_uav_wing.gnn import _cabi, ops

    N, B = pred_d.shape[0], cp_d.numel() - 1
    ar = Arena()
    out = ar.out((B, 2), torch.float64)
    seed = ar.out((N,), torch.float32)
    ws, nbytes = ar.ws(_cabi.lib.dfw_case_stress_summary_ws_bytes(N, B))
    _cabi.check(_cabi.lib.dfw_case_ks_seed(pred_d.data_ptr(), ops._dt(pred_d), pos_d.data_ptr(), ops._ptr(mask_d), cp_d.data_ptr(), B, N,
                                           0.05, rho, out.data_ptr(), seed.data_ptr(), ws.data_ptr(), nbytes,
                                           torch.cuda.current_stream().cuda_stream))
    ar.check("dfw_case_ks_seed")  # nothing written before or after out, seed and the workspace
    return out.cpu().numpy(), seed.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("masked", [False, True])
def test_case_ks_seed_against_fp64_restatement(dtype, masked):
    """Bounds (eps = 2^-53; n = |S_b|), per side - kernel and restatement each:
      * a term exp(rho (u - m)) is within eps |rho (u - m)| (argument rounding) + 2 eps (exp, product) of its value, and
        t |ln t| <= 1/e, so the terms together are off by at most (n/e + 2n) eps relative to s >= 1;
      * summing n positive terms in any order adds at most (n - 1) eps relative: rel(s) <= 4 n eps;
      * KS = m + ln(s) / rho: |dKS| <= (rel(s) + eps ln s) / rho + 2 eps |KS|.
    The seed w = t / s is rounded to fp32 once: |dw| <= 2^-24 w + (eps (|rho (u - m)| + 3) + 2 rel(s)) w + 2^-150."""
    from deep_fem_uav_wing.gnn import ops  # noqa: F401  (loads the library)

    rho = 100.0
    pos, u, ptr = _ks_batch()
    mask = (np.random.default_rng(3).random(len(u)) < 0.4) if masked else None
    pred_d = torch.from_numpy(u).cuda().to(dtype)
    u_used = pred_d.float().cpu().numpy()  # the kernel's own input, bf16-rounded in bf16
    got, seed = _raw_ks(pred_d, torch.from_numpy(pos).cuda(), torch.from_numpy(ptr).cuda(),
                        torch.from_numpy(mask.astype(np.uint8)).cuda() if masked else None, rho)
    sets = screened_sets(u_used, pos[:, 1], ptr, mask)
    ref, seed_ref = ks_and_seed_oracle(u_used, ptr, sets, rho)
    n = ref[:, 1]
    assert np.array_equal(got[:, 1], n)
    assert n[3] == 0 and (masked or n[4] == 0) and n[2] > 0 and n[5] > 0
    rel_s = 4 * np.maximum(n, 1) * EPS64
    bound_ks = 2 * ((rel_s + EPS64 * np.log(np.maximum(n, 1))) / rho + 2 * EPS64 * np.abs(ref[:, 0]))
    err_ks = np.abs(got[:, 0] - ref[:, 0])
    assert (err_ks <= bound_ks).all(), (err_ks, bound_ks)
    assert got[n == 0, 0].tolist() == [0.0] * int((n == 0).sum())
    rows_case = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    m_row = np.zeros(len(u))
    for b, idx in enumerate(sets):
        if idx.size:
            m_row[ptr[b] + idx] = u_used[ptr[b] + idx].max()
    arg = np.abs(rho * (u_used.astype(np.float64) - m_row))
    arg[~np.isfinite(arg)] = 0.0
    w = np.abs(seed_ref)
    bound_w = 2.0 ** -24 * w + 2 * (EPS64 * (arg + 3) + 2 * rel_s[rows_case]) * w + 2.0 ** -150
    err_w = np.abs(seed.astype(np.float64) - seed_ref)
    assert (err_w <= bound_w).all(), float((err_w / bound_w).max())
    record("sensitivity_ks_seed", dtype=str(dtype), masked=masked, ks_max_err_over_bound=float((err_ks / bound_ks).max()),
           seed_max_err_over_bound=float((err_w / bound_w).max()), seed_rows_above_1e_3=int((seed_ref > 1e-3).sum()))
    # the kernel's record and seed of a case do not depend on the other cases of the launch
    for b in range(len(ptr) - 1):
        r0, r1 = int(ptr[b]), int(ptr[b + 1])
        g1, s1 = _raw_ks(pred_d[r0:r1], torch.from_numpy(pos[r0:r1]).cuda(), torch.tensor([0, r1 - r0], device="cuda"),
                         torch.from_numpy(mask[r0:r1].astype(np.uint8)).cuda() if masked else None, rho)
        assert g1.tobytes() == got[b:b + 1].tobytes() and s1.tobytes() == seed[r0:r1].tobytes(), b


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [(6, 4), (1, 7), (0, 10)])
def test_case_column_sums_against_fp64(cols):
    from deep_fem_uav_wing.gnn import _cabi

    c0, nc = cols
    _, _, ptr = _ks_batch()
    N, B, C = int(ptr[-1]), len(ptr) - 1, 10
    a = np.random.default_rng(5).standard_normal((N, C)).astype(np.float32) * np.float32(1e-3)
    ar = Arena()
    a_d = ar.out((N, C), torch.float32, fill=torch.from_numpy(a))
    cp = torch.from_numpy(ptr).cuda()
    out = ar.out((B, nc), torch.float64)
    ws, nbytes = ar.ws(_cabi.lib.dfw_case_stress_summary_ws_bytes(N, B))
    _cabi.check(_cabi.lib.dfw_case_column_sums(a_d.data_ptr(), N, C, c0, nc, cp.data_ptr(), B, out.data_ptr(), ws.data_ptr(), nbytes,
                                               torch.cuda.current_stream().cuda_stream))
    ar.check("dfw_case_column_sums")
    got = out.cpu().numpy()
    a64 = a.astype(np.float64)[:, c0:c0 + nc]
    for b in range(B):
        r0, r1 = int(ptr[b]), int(ptr[b + 1])
        ref = a64[r0:r1].sum(axis=0)
        bound = 2 * max(r1 - r0, 1) * EPS64 * np.abs(a64[r0:r1]).sum(axis=0)  # n eps sum|a| per side
        assert (np.abs(got[b] - ref) <= bound).all(), (b, got[b], ref)
    assert got[3].tolist() == [0.0] * nc  # the empty case
    from deep_fem_uav_wing.gnn import ops

    for b in range(B):  # a case alone gives the same bits
        r0, r1 = int(ptr[b]), int(ptr[b + 1])
        alone = ops.case_column_sums(a_d[r0:r1], torch.tensor([0, r1 - r0], device="cuda"), c0, nc).cpu().numpy()
        assert alone.tobytes() == got[b:b + 1].tobytes(), b


# ---- GPU: the vector-Jacobian product --------------------------------------------------------------------------------
def _device_model(ref, dtype):
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    m = GraphSAGEModel(10, ref.hidden_channels, 1, ref.num_layers, dropout=0.0)
    m.load_state_dict(ref.state_dict(), strict=True)
    return m.cuda().eval().set_compute_dtype(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_vjp_of_the_kernel_seed_against_fp64_oracle(dtype):
    """The product's dKS/dx_6..9 per case against the oracle's autograd with THE SAME seed (the kernel's), so forward
    error is excluded.  Small meshes: no activation within forward rounding of a ReLU kink (DESIGN section 2)."""
    from deep_fem_uav_wing.gnn import ops, synth

    rho = 100.0
    meshes = [synth.surface_tri_wing(n, seed=60 + i) for i, n in enumerate((400, 700, 1000))]
    x, ei, pos, ptr = _union(meshes)
    ref = _oracle_model(hidden=64, layers=3, seed=4)
    model = _device_model(ref, dtype)
    x_d = torch.from_numpy(x).cuda().requires_grad_()
    params = {k: v.detach() for k, v in model.named_parameters()}
    cp = torch.from_numpy(ptr).cuda()
    with torch.enable_grad():
        pred = torch.func.functional_call(model, params, (x_d, torch.from_numpy(ei).cuda()))
    ks, seed = ops.case_ks_seed(pred, torch.from_numpy(pos).cuda(), cp, rho=rho)
    g_x, = torch.autograd.grad(pred, x_d, seed.view_as(pred))
    got = ops.case_column_sums(g_x, cp, 6, 4).cpu().numpy()
    seed_np = seed.cpu().numpy()
    r64 = oracle_param_sensitivities(ref, x, ei, pos[:, 1], ptr, rho, dtype=torch.float64, seed=seed_np)[:, 2:]
    r32 = oracle_param_sensitivities(ref, x, ei, pos[:, 1], ptr, rho, dtype=torch.float32, seed=seed_np)[:, 2:]
    for b in range(len(meshes)):
        e = np.abs(got[b] - r64[b]).max() / np.abs(r64[b]).max()
        e32 = np.abs(r32[b] - r64[b]).max() / np.abs(r64[b]).max()
        record("sensitivity_vjp", dtype=str(dtype), case=b, rel_err=e, oracle32_rel_err=e32)
        if dtype == torch.float32:
            assert e < max(1e-5, 3 * e32), (b, e, e32)
        else:
            assert e <= 2e-2, (b, e)


# ---- GPU: the screener -----------------------------------------------------------------------------------------------
def _geometry_cases(sizes, seed0=100):
    from deep_fem_uav_wing.gnn import synth

    return [synth.geometry_case(synth.surface_tri_wing(n, seed=seed0 + i)) for i, n in enumerate(sizes)]


def _model(dtype, seed=0):
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    torch.manual_seed(seed)
    return GraphSAGEModel(10, 128, 1, 4).cuda().eval().set_compute_dtype(dtype)


NEW_FIELDS = ("ks_stress_pa", "d_ks_stress_pa")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_sensitivity_records_are_batch_independent_and_leave_the_summary_alone(dtype):
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    sizes = [600, 4000, 1200, 9000, 800, 2500, 700, 5200, 3000, 640, 7000, 1500, 900, 2000, 6000, 1000]
    cases = _geometry_cases(sizes)
    model = _model(dtype)
    plain = DesignScreener(model, max_nodes_per_launch=10**6, allowable_pa=5e6).screen(cases)
    together = DesignScreener(model, max_nodes_per_launch=10**6, allowable_pa=5e6, sensitivities=True).screen(cases)
    alone = DesignScreener(model, max_nodes_per_launch=1, allowable_pa=5e6, sensitivities=True).screen(cases)
    assert together == alone  # every float compared exactly
    ratios = []
    for p, s in zip(plain, together):
        assert s["status"] == "success" and {k: v for k, v in s.items() if k not in NEW_FIELDS} == p  # bitwise, field by field
        assert s["max_stress_pa"] <= s["ks_stress_pa"]
        assert s["ks_stress_pa"] <= np.expm1(np.log1p(s["max_stress_pa"]) + np.log(s["n_screened"]) / 100.0) * (1 + 1e-6)
        assert sorted(s["d_ks_stress_pa"]) == sorted(PARAM_SCALE) and all(np.isfinite(v) for v in s["d_ks_stress_pa"].values())
        ratios.append(s["ks_stress_pa"] / s["max_stress_pa"])
    record("sensitivity_screener_ks_over_max", dtype=str(dtype), min=min(ratios), max=max(ratios))


@pytest.mark.gpu
def test_sensitivity_screen_does_no_weight_gradient_work_and_leaves_the_model_alone(monkeypatch):
    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.model import MaskedMSELoss
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    calls = []
    real = ops.linear_bwd_weight
    monkeypatch.setattr(ops, "linear_bwd_weight", lambda *a, **k: calls.append(1) or real(*a, **k))
    model = _model(torch.float32)
    model.convs[1].lin_r.weight.requires_grad_(False)  # a frozen parameter stays frozen
    before = {k: p.requires_grad for k, p in model.named_parameters()}
    cases = _geometry_cases([1500 + 37 * i for i in range(40)], seed0=300)
    screener = DesignScreener(model, max_nodes_per_launch=12_000, result_ring=2, sensitivities=True)
    ref = screener.screen(cases)
    assert calls == []
    assert all(p.grad is None for p in model.parameters())
    assert {k: p.requires_grad for k, p in model.named_parameters()} == before
    # no host wait per launch: the sensitivity path enqueues without synchronising, like the plain screener
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = screener.screen(cases)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert got == ref and all(r["ks_stress_pa"] is not None for r in got)
    # a training step still computes every weight gradient: one dfw_linear_bwd_weight per linear layer group
    from deep_fem_uav_wing.gnn import synth

    mesh = synth.surface_tri_wing(2000, seed=5)
    model.train()
    out = model(torch.from_numpy(mesh["x"]).cuda(), torch.from_numpy(mesh["edge_index"]).cuda())
    MaskedMSELoss()(out, torch.from_numpy(mesh["y"]).cuda(), torch.from_numpy(mesh["loss_mask"]).cuda()).backward()
    assert len(calls) == 2 + model.num_layers + 1
    assert all((p.grad is not None) == p.requires_grad for p in model.parameters())


@pytest.mark.gpu
def test_screen_cli_sensitivities(tmp_path):
    from test_screening import _checkpoint

    _checkpoint(tmp_path)
    env = dict(os.environ, PYTHONPATH=str(PKG))
    cmd = [sys.executable, str(PKG / "scripts" / "screen_gnn.py"), "--root", str(tmp_path), "--checkpoint", "checkpoints/m.pt",
           "--synthetic", "32", "--seed", "700", "--synthetic-nodes", "3000", "--top-k", "3", "--sensitivities", "--out", "s.jsonl"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    recs = [json.loads(line) for line in (tmp_path / "s.jsonl").read_text().splitlines()]
    ok = [x for x in recs if x["status"] == "success"]
    assert len(recs) == 32 and len(ok) == 32 and "#1 " in r.stdout
    for x in ok:
        vals = [x["ks_stress_pa"]] + [x["d_ks_stress_pa"][k] for k in PARAM_SCALE]
        assert len(vals) == 5 and all(isinstance(v, float) and np.isfinite(v) for v in vals)
        assert x["ks_stress_pa"] >= x["max_stress_pa"]
