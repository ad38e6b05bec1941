"""Element-wise error bounds for the fused linear family against fp64, on every kernel the host code dispatches to.

The family is dfw_linear_fwd, dfw_linear_bwd_input, dfw_linear_bwd_weight and dfw_epilogue_bwd.  Every reference is computed
in fp64 from exactly the tensors the kernel read (bf16 operands cast up, the saved pre_out / ln_stats / act of a backward),
so the only legitimate errors are the fp32 accumulation and the final store, and both are bounded per element.  With
u = 2^-24, r the exact value and S the fp64 sum of the absolute values of its terms (bias included):

  short reductions stored fp32 (y, pre_out, bwd_input; K terms)   (K + 8) * 2u * S
  stored bf16                                                     + 2^-8 * |r|   (one bf16 ulp at most; RNE gives half)
  LayerNorm output                                                |g| rstd E (2 + |xhat|) + (H + 8) 2u (|g xhat| + |b|),
                                                                  E = the row's largest y bound; ReLU is 1-Lipschitz,
                                                                  dropout scales by 1/(1-p)
  long reductions over nodes (dW, dbias, dgamma, dbeta, ...)      2^-16 * S per element, and tensor-wide
                                                                  rel_l2(got, r) <= max(4 rel_l2(cpu_fp32, r), 2^-20)

The 2u covers a tensor-core accumulation that truncates and the dropped lo*lo term of 3xTF32.  Each row also asserts
WHICH kernel ran (torch.profiler kernel names), every raw-ABI output and workspace sits inside sentinel-filled guard bands,
and every bf16 output of >= 1e5 elements is checked for a rounding bias (truncation instead of round-to-nearest-even).

The kernel-selection switches (DFW_FORCE_SIMT, DFW_TC_PERSIST) are read once per process:
tests/test_gpu_linear_variants.py re-runs this file in a subprocess per switch, and the rows read os.environ to know
which kernel to expect."""
import json
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

from helpers import Arena, assert_bound, assert_no_rounding_bias, bf16_ulp, launched_kernels, record, rel_l2, rounding_bias

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "deep-fem-uav-wing_b200")

U = 2.0 ** -24
F32, BF16 = torch.float32, torch.bfloat16


def _atoi(s):
    m = re.match(r"\s*[+-]?\d+", s or "")
    return int(m.group()) if m else 0


# the same parsing as the library: force_simt() (dfw_linear.cu) and the atoi() switches of dfw_linear_tc.cu
_simt_env = os.environ.get("DFW_FORCE_SIMT", "")
SIMT = bool(_simt_env) and _simt_env[0] != "0"
PERSIST = _atoi(os.environ.get("DFW_TC_PERSIST", "1")) != 0


# ---- bound helpers (CPU, no device needed) ------------------------------------------------------------------------
def short_bound(S, K, r=None, bf16=False):
    """Per-element bound of a K-term fp32 reduction; `bf16` adds the store to bf16 (half an ulp of the computed value)."""
    b = (K + 8) * 2 * U * S.double()
    if bf16:
        b = b + 2.0 ** -8 * (r.double().abs() + b)
    return b


def long_check(name, got, r, S, cpu32, extra=None, chain_bound=None):
    """Reductions over nodes: 2^-16 S per element (+ `extra`) and rel_l2 no worse than 4x CPU fp32 (floor 2^-20).
    `chain_bound`: a per-element error bound derived from the kernel's own accumulation chain (see tc_dw_chain_bound); its
    relative 2-norm widens the tensor-wide limit where that chain is longer than a CPU summation's."""
    bound = 2.0 ** -16 * S.double() + (extra if extra is not None else 0.0)
    m = assert_bound(name, got, r, bound)
    if float(r.double().abs().max()) == 0.0:
        return m, None
    e, e_cpu = rel_l2(got, r), rel_l2(cpu32.to(r.device), r)
    lim = max(4 * e_cpu, 2.0 ** -20)
    if chain_bound is not None:
        lim = max(lim, float(chain_bound.double().norm() / r.double().norm()))
    assert e <= lim, f"{name}: rel_l2 {e:.3g} > {lim:.3g} (CPU fp32 on the same inputs: {e_cpu:.3g})"
    return m, e / lim


def ln_out_bound(g, rstd, E, xh, beta, H):
    """First-order propagation of the row's y error E (per row) through LayerNorm, plus its own fp32 rounding."""
    return (g.abs() * rstd[:, None] * E[:, None] * (2 + xh.abs()) + (H + 8) * 2 * U * ((g * xh).abs() + beta.abs()))


# ---- unit tests of the helpers: they must accept RNE of the exact result and reject the three planted faults ------
def _cpu_problem(sign, n=4096, k=64, h=96, seed=0):
    gen = torch.Generator().manual_seed(seed)
    if sign == "nonneg":
        a, w, b = torch.rand(n, k, generator=gen), torch.rand(h, k, generator=gen) / k, torch.rand(h, generator=gen)
    else:
        a, w, b = torch.randn(n, k, generator=gen), torch.randn(h, k, generator=gen) / k ** 0.5, torch.randn(h, generator=gen)
    a, w = a.to(BF16).double(), w.to(BF16).double()
    r = a @ w.T + b.double()
    S = a.abs() @ w.abs().T + b.double().abs()
    return a, w, r, S


@pytest.mark.parametrize("sign", ["mixed", "nonneg"])
def test_bound_helpers_accept_round_to_nearest_even(sign):
    a, w, r, S = _cpu_problem(sign)
    K = a.shape[1]
    assert assert_bound("fp32", r.float(), r, short_bound(S, K)) <= 1
    assert assert_bound("bf16", r.to(BF16), r, short_bound(S, K, r, bf16=True)) <= 1
    bias, n = rounding_bias(r.to(BF16), r, short_bound(S, K))
    assert n > 100_000 and abs(bias) < 0.05
    dw_r = a.T @ a
    long_check("dW", dw_r.float(), dw_r, a.abs().T @ a.abs(), (a.float().T @ a.float()))


def _truncate_bf16(r):
    bits = r.float().view(torch.int32) & ~0xFFFF
    return bits.view(torch.float32).to(BF16)  # exact: the low half is already zero


@pytest.mark.parametrize("sign", ["mixed", "nonneg"])
def test_bound_helpers_reject_truncation_dropped_term_and_two_ulp_error(sign):
    a, w, r, S = _cpu_problem(sign)
    K = a.shape[1]
    # (1) a store that truncates toward zero: the rounding-bias check
    bias, _ = rounding_bias(_truncate_bf16(r), r, short_bound(S, K))
    assert bias < -0.3
    with pytest.raises(AssertionError, match="store error"):
        assert_no_rounding_bias("trunc", _truncate_bf16(r), r, short_bound(S, K))
    # (2) one term of the reduction dropped (K chunk lost, bias column skipped ...)
    dropped = (r - a[:, 7:8] * w[:, 7][None, :]).float()
    with pytest.raises(AssertionError, match="outside the bound"):
        assert_bound("drop", dropped, r, short_bound(S, K))
    no_bias = (a @ w.T).float()
    if sign == "nonneg":  # a bias in [0, 1) against a per-element bound of ~1e-5 |r|
        with pytest.raises(AssertionError, match="outside the bound"):
            assert_bound("nobias", no_bias, r, short_bound(S, K))
    dw_r = a.T @ a
    dw_drop = (a[1:].T @ a[1:]).float()  # one node's contribution lost
    with pytest.raises(AssertionError):
        long_check("dW drop", dw_drop, dw_r, a.abs().T @ a.abs(), (a.float().T @ a.float()))
    # (3) a 2-ulp error on a single bf16 element
    got = r.to(BF16)
    i = int(r.abs().flatten().argmax())
    bits = got.flatten().view(torch.int16).clone()
    bits[i] += 2  # same sign, two ulps further from zero
    with pytest.raises(AssertionError, match="1 of"):
        assert_bound("2ulp", bits.view(BF16).view_as(got), r, short_bound(S, K, r, bf16=True))


# ---- workspace queries at N = 0 / 1 (CPU; a SIGFPE in the child fails the test instead of killing pytest) ---------
_WS_SWEEP = r"""
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from deep_fem_uav_wing.gnn import _cabi
lib = _cabi.lib
n = int(sys.argv[2])
calls = {
    "dfw_csr_ws_bytes": [(3 * n, n)],
    "dfw_faces_ws_bytes": [(n, n)],
    "dfw_node_features_ws_bytes": [(n,)],
    "dfw_node_features_batched_ws_bytes": [(n,)],
    "dfw_linear_ws_bytes": [(128, 128, 128, 0), (64, 10, 0, 1)],
    "dfw_epilogue_bwd_ws_bytes": [(n, 4), (n, 128), (n, 256)],
    "dfw_linear_bwd_weight_ws_bytes": [(n, 128, 128, 128), (n, 64, 10, 0), (n, 48, 40, 24), (n, 6, 10, 0), (n, 256, 256, 0)],
    "dfw_sage_layer_fwd_ws_bytes": [(n, 128, 128, d) for d in (0, 1)],
    "dfw_sage_layer_bwd_ws_bytes": [(n, 128, 128, d, g) for d in (0, 1) for g in (0, 1)],
    "dfw_mlp2_fwd_ws_bytes": [(n, 10, 64, 128, d) for d in (0, 1)] + [(n, 128, 64, 1, d) for d in (0, 1)],
    "dfw_mlp2_bwd_ws_bytes": [(n, 10, 64, 128, d, 0, g) for d in (0, 1) for g in (0, 1)]
                             + [(n, 128, 64, 1, d, 1, g) for d in (0, 1) for g in (0, 1)],
    "dfw_masked_mse_ws_bytes": [(n, 1), (n, 3)],
    "dfw_stress_metrics_ws_bytes": [(n, 1)],
    "dfw_vertex_normals_ws_bytes": [(n, n)],
    "dfw_case_stress_summary_ws_bytes": [(n, 1), (n, n)],
    "dfw_graphsage_forward_ws_bytes": [(n, 10, 64, 128, 64, x, d) for x in (0, 1) for d in (0, 1)],
}
out = {}
for name, arg_sets in calls.items():
    out[name] = [int(getattr(lib, name)(*a)) for a in arg_sets]
nb, sc, slc = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
out["dfw_agg_plan_sizes"] = [lib.dfw_agg_plan_sizes(n, 3 * n, ctypes.byref(nb), ctypes.byref(sc), ctypes.byref(slc)), nb.value, sc.value, slc.value]
print(json.dumps(out))
"""


def _header_ws_queries():
    text = open(os.path.join(REPO, "include", "dfw_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dfw_[a-z0-9_]+_ws_bytes)\s*\(", text)))


@pytest.mark.parametrize("n", [0, 1])
def test_every_workspace_query_returns_at_n0_and_n1(n):
    """dw_plan divided by zero at N = 0 (SIGFPE in dfw_linear_bwd_weight_ws_bytes and every query built on it)."""
    r = subprocess.run([sys.executable, "-c", _WS_SWEEP, PKG, str(n)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, f"workspace sweep at N={n} died with rc {r.returncode}: {r.stderr[-2000:]}"
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert sorted(k for k in got if k.endswith("_ws_bytes")) == _header_ws_queries()  # a new query joins the sweep
    assert got["dfw_agg_plan_sizes"][0] == 0
    assert all(v > 0 for v in got["dfw_linear_bwd_weight_ws_bytes"])  # the N = 0 branch still needs its second pass


# ======================================== GPU part =================================================================
def _ops():
    from deep_fem_uav_wing.gnn import _cabi

    return _cabi


def _dt(t):
    return 0 if t.dtype == F32 else 1


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _seed(name):
    return zlib.crc32(name.encode()) & 0x7FFFFFFF


def assert_kernels(row, names, expect, absent=()):
    if not names:
        print(f"[{row}] torch.profiler saw no CUDA kernels: the kernel-name assertion is skipped")
        return
    for pat in ([expect] if isinstance(expect, str) else expect):
        assert any(re.search(pat, n) for n in names), f"{row}: expected a kernel matching {pat!r}, launched {sorted(set(names))}"
    for pat in absent:
        assert not any(re.search(pat, n) for n in names), f"{row}: unexpected kernel matching {pat!r} in {sorted(set(names))}"


def _tc_kernel(dtype, N, H, k1, k2):
    """The tensor-core forward kernel dfw_linear_fwd picks (dfw_linear_tc.cu, linear_tc_eligible / linear_tc_launch), or None."""
    e = 4 if dtype == F32 else 2
    if SIMT or not (16 <= H <= 256 and H % 16 == 0 and (H * e) % 128 == 0 and (k1 * e) % 16 == 0 and (k2 * e) % 16 == 0):
        return None
    npad, regions, tiles = (H + 15) // 16 * 16, 2 if dtype == F32 else 1, (N + 127) // 128
    if PERSIST and 2 * regions * npad <= 512 and H % 32 == 0 and tiles >= 2:
        return r"k_linear_tcp<"
    return r"k_linear_tc<"


def _operand(shape, dt, sign, gen, scale=1.0):
    if sign == "nonneg":
        t = torch.rand(shape, generator=gen, device="cuda") * scale
    else:
        t = torch.randn(shape, generator=gen, device="cuda") * scale
    return t.to(dt)


def _keep(seed, N, H, p):
    from oracle.sage_oracle import dropout_keep_scale

    return torch.from_numpy(dropout_keep_scale(seed, N, H, p)).cuda().double()


# ---- forward ----------------------------------------------------------------------------------------------------------
# (id, dtype, N, Hout, k1, k2, tail).  tail: full = LayerNorm + ReLU + dropout + residual with pre_out and stats;
# ln = LayerNorm + ReLU with pre_out and stats; bare = y only (the persistent kernel's !y_in_tmem branch);
# rowdot = the decoder: ReLU + dropout + row dot with out = NULL.
NBIG = 56909  # 445 tiles of 128 rows: 3 per CTA on 148 SMs, ragged last tile
FWD_ROWS = [
    ("persist_f32_h128_full", F32, NBIG, 128, 128, 128, "full"),
    ("persist_f32_h128_bare", F32, NBIG, 128, 128, 0, "bare"),
    ("persist_bf16_h64_full", BF16, NBIG, 64, 64, 64, "full"),
    ("persist_bf16_h256_full", BF16, NBIG, 256, 256, 256, "full"),
    ("persist_bf16_h256_bare", BF16, NBIG, 256, 256, 0, "bare"),
    ("persist_f32_h64_rowdot", F32, NBIG, 64, 128, 0, "rowdot"),
    ("persist_bf16_h64_rowdot", BF16, NBIG, 64, 128, 0, "rowdot"),
    ("classic_f32_n1", F32, 1, 128, 128, 128, "full"),
    ("classic_bf16_n77", BF16, 77, 256, 256, 256, "full"),
    ("classic_f32_n128", F32, 128, 64, 64, 64, "full"),
    ("classic_bf16_n128_bare", BF16, 128, 128, 64, 0, "bare"),
    ("classic_f32_h192", F32, NBIG, 192, 64, 192, "full"),
    ("classic_f32_h256", F32, NBIG, 256, 256, 0, "ln"),
    ("simt_f32_h48", F32, 5003, 48, 64, 48, "full"),
    ("simt_bf16_h96", BF16, 5003, 96, 96, 96, "full"),
    ("simt_f32_h40", F32, 5003, 40, 40, 0, "bare"),
    ("simt_bf16_h40_rowdot", BF16, 5003, 40, 64, 0, "rowdot"),
    ("simt_f32_k10_ln", F32, 5003, 64, 10, 0, "ln"),
]


def _run_fwd(a1, w1, a2, w2, bias, gamma, beta, residual, p, seed, rdw, rdb, flags, N, H, want_out, want_pre, want_stats,
             out_dtype=None, use_ws=True):
    cabi = _ops()
    dt = a1.dtype
    k1, k2 = a1.shape[1], (a2.shape[1] if a2 is not None else 0)
    ar = Arena()
    out = ar.out((N, H), out_dtype or dt) if want_out else None
    pre = ar.out((N, H), dt) if want_pre else None
    stats = ar.out((N, 2), F32) if want_stats else None
    rd = ar.out((N,), F32) if rdw is not None else None
    ws, ws_bytes = ar.ws(cabi.lib.dfw_linear_ws_bytes(H, k1, k2, _dt(a1))) if use_ws else (None, 0)

    def call():
        cabi.check(cabi.lib.dfw_linear_fwd(_p(a1), _p(w1), k1, _p(a2), _p(w2), k2, _p(bias), _p(gamma), _p(beta), 1e-5, _p(residual),
                                           p, seed, _p(out), _p(pre), _p(stats), _p(rdw), _p(rdb), _p(rd), N, H, flags, _dt(a1),
                                           _p(ws), ws_bytes, _stream()))

    _, names = launched_kernels(call)
    return dict(out=out, pre=pre, stats=stats, rowdot=rd), names, ar


def fwd_reference(a1, w1, a2, w2, bias, ln, relu, keep, residual, rdw, rdb, bf16):
    """fp64 result and per-element bound of every output of dfw_linear_fwd."""
    ops_ = [(a1, w1)] + ([(a2, w2)] if a2 is not None else [])
    y = sum(a.double() @ w.double().T for a, w in ops_)
    S = sum(a.double().abs() @ w.double().abs().T for a, w in ops_)
    K = sum(a.shape[1] for a, _ in ops_)
    if bias is not None:
        y, S = y + bias.double(), S + bias.double().abs()
    H = y.shape[1]
    Ey = short_bound(S, K)
    res = {"pre": (y, short_bound(S, K, y, bf16), Ey)}
    v, Ev = y, Ey
    if ln is not None:
        g, b = ln[0].double(), ln[1].double()
        mean = y.mean(1)
        var = y.var(1, unbiased=False)
        rstd = 1.0 / torch.sqrt(var + 1e-5)
        xh = (y - mean[:, None]) * rstd[:, None]
        E = Ey.max(1).values
        v = xh * g + b
        Ev = ln_out_bound(g, rstd, E, xh, b, H)
        res["mean"] = (mean, E + (H + 8) * 2 * U * y.abs().mean(1))
        res["rstd"] = (rstd, rstd * (2 * rstd * E + (H + 8) * 2 * U + 8 * U))
    if relu:
        v = v.clamp_min(0)
    if keep is not None:
        v, Ev = v * keep, Ev * keep + 2 * U * (v * keep).abs()
    if rdw is not None:
        w64 = rdw.double()
        rb = rdb.double() if rdb is not None else torch.zeros(1, dtype=torch.float64, device=v.device)
        res["rowdot"] = (v @ w64 + rb, Ev @ w64.abs() + (H + 8) * 2 * U * ((v.abs() @ w64.abs()) + rb.abs()))
    if residual is not None:
        r64 = residual.double()
        v, Ev = v + r64, Ev + 2 * U * ((v + r64).abs() + r64.abs())
    res["out"] = (v, Ev + (2.0 ** -8 * (v.abs() + Ev) if bf16 else 0.0), Ev)
    return res


def _fwd_inputs(name, dt, N, H, k1, k2, sign):
    gen = torch.Generator(device="cuda").manual_seed(_seed(name + sign))
    a1 = _operand((N, k1), dt, sign, gen)
    w1 = _operand((H, k1), dt, sign, gen, 1.0 / k1 if sign == "nonneg" else k1 ** -0.5)
    a2 = _operand((N, k2), dt, sign, gen) if k2 else None
    w2 = _operand((H, k2), dt, sign, gen, 1.0 / k2 if sign == "nonneg" else k2 ** -0.5) if k2 else None
    bias = _operand((H,), F32, sign, gen)
    gamma = (torch.rand(H, generator=gen, device="cuda") + 0.5) * (1 if sign == "nonneg" else torch.sign(torch.randn(H, generator=gen, device="cuda")))
    beta = torch.randn(H, generator=gen, device="cuda") * 0.5
    return gen, a1, w1, a2, w2, bias, gamma, beta


def _check_outputs(row, got, ref, bf16):
    margins = {}
    for key in ("pre", "out"):
        if got.get(key) is not None:
            r, b, pre_store = ref[key]
            margins[key] = assert_bound(f"{row}/{key}", got[key], r, b)
            if bf16:
                bias = assert_no_rounding_bias(f"{row}/{key}", got[key], r, pre_store)
                if bias is not None:
                    margins[key + "_bias_ulp"] = bias
    if got.get("stats") is not None:
        margins["mean"] = assert_bound(f"{row}/mean", got["stats"][:, 0], *ref["mean"])
        margins["rstd"] = assert_bound(f"{row}/rstd", got["stats"][:, 1], *ref["rstd"])
    if got.get("rowdot") is not None:
        margins["rowdot"] = assert_bound(f"{row}/rowdot", got["rowdot"], *ref["rowdot"])
    return margins


@pytest.mark.gpu
@pytest.mark.parametrize("sign", ["mixed", "nonneg"])
@pytest.mark.parametrize("row", FWD_ROWS, ids=[r[0] for r in FWD_ROWS])
def test_linear_fwd_within_bounds(row, sign):
    name, dt, N, H, k1, k2, tail = row
    cabi = _ops()
    gen, a1, w1, a2, w2, bias, gamma, beta = _fwd_inputs(name, dt, N, H, k1, k2, sign)
    p, seed = (0.1, 1234 + N) if tail in ("full", "rowdot") else (0.0, 0)
    ln = tail in ("full", "ln")
    relu = tail != "bare"
    residual = _operand((N, H), dt, "mixed", gen) if tail == "full" else None
    rdw = torch.randn(H, generator=gen, device="cuda") / H ** 0.5 if tail == "rowdot" else None
    rdb = torch.randn(1, generator=gen, device="cuda") if tail == "rowdot" else None
    flags = ((cabi.EP_LAYERNORM if ln else 0) | (cabi.EP_RELU if relu else 0) | (cabi.EP_DROPOUT if p else 0)
             | (cabi.EP_RESIDUAL if residual is not None else 0))
    got, names, ar = _run_fwd(a1, w1, a2, w2, bias, gamma if ln else None, beta if ln else None, residual, p, seed, rdw, rdb, flags,
                              N, H, want_out=tail != "rowdot", want_pre=tail in ("full", "ln"), want_stats=ln)
    ar.check(name)
    assert_kernels(name, names, _tc_kernel(dt, N, H, k1, k2) or r"\bk_linear<")
    keep = _keep(seed, N, H, p) if p else None
    ref = fwd_reference(a1, w1, a2, w2, bias, (gamma, beta) if ln else None, relu, keep, residual, rdw, rdb, dt == BF16)
    margins = _check_outputs(name, got, ref, dt == BF16)
    record(f"linear_bounds/fwd/{name}/{sign}", kernel=sorted(set(names)), simt=SIMT, persist=PERSIST, **margins)


TINY_ROWS = [(k, h, dt) for k in (3, 10, 16) for h in (4, 64, 256) for dt in ("f32", "bf16", "f32_out_bf16")]


@pytest.mark.gpu
@pytest.mark.parametrize("k,h,kind", TINY_ROWS, ids=[f"k{k}_h{h}_{d}" for k, h, d in TINY_ROWS])
def test_linear_fwd_tiny_k_within_bounds(k, h, kind):
    """The encoder's first linear: tiled tiny-K kernel (no workspace, so k = 16 does not take the tensor cores)."""
    cabi = _ops()
    if kind == "f32_out_bf16" and SIMT:
        pytest.skip("DFW_EP_OUT_BF16 is the tiny-K kernel only; DFW_FORCE_SIMT refuses it")
    name = f"tiny_k{k}_h{h}_{kind}"
    dt = BF16 if kind == "bf16" else F32
    N = 20011
    for sign in ("mixed", "nonneg"):
        _, a1, w1, _, _, bias, _, _ = _fwd_inputs(name, dt, N, h, k, 0, sign)
        out_dtype = BF16 if kind == "f32_out_bf16" else None
        flags = cabi.EP_RELU | (cabi.EP_OUT_BF16 if out_dtype else 0)
        got, names, ar = _run_fwd(a1, w1, None, None, bias, None, None, None, 0.0, 0, None, None, flags, N, h, True, False, False,
                                  out_dtype=out_dtype, use_ws=False)
        ar.check(name)
        assert_kernels(name, names, r"\bk_linear<" if SIMT else r"k_smallk_fwd_tiled")
        ref = fwd_reference(a1, w1, None, None, bias, None, True, None, None, None, None, (out_dtype or dt) == BF16)
        margins = _check_outputs(name, got, ref, (out_dtype or dt) == BF16)
        record(f"linear_bounds/fwd_tiny/{name}/{sign}", kernel=sorted(set(names)), simt=SIMT, **margins)


@pytest.mark.gpu
def test_bf16_relu_mask_of_forward_and_backward_differ_only_at_zero():
    """In bf16 the forward decides ReLU on the fp32 y, the backward on the bf16-rounded pre_out (with the fp32 stats).
    This pins down where the two decisions may differ: within 2 bf16 ulps of y (propagated to z) of z = 0."""
    cabi = _ops()
    name, N, H = "mask_mismatch_bf16_h128", NBIG, 128
    _, a1, w1, a2, w2, bias, gamma, beta = _fwd_inputs(name, BF16, N, H, H, H, "mixed")
    got, _, ar = _run_fwd(a1, w1, a2, w2, bias, gamma, beta, None, 0.0, 0, None, None, cabi.EP_LAYERNORM | cabi.EP_RELU, N, H,
                          True, True, True)
    ar.check(name)
    ref = fwd_reference(a1, w1, a2, w2, bias, (gamma, beta), True, None, None, None, None, True)
    y = ref["pre"][0]
    g64, b64 = gamma.double(), beta.double()
    mean, rstd = y.mean(1, keepdim=True), 1.0 / torch.sqrt(y.var(1, unbiased=False, keepdim=True) + 1e-5)
    z_exact = (y - mean) * rstd * g64 + b64
    st = got["stats"].double()
    z_bwd = (got["pre"].double() - st[:, :1]) * st[:, 1:] * g64 + b64
    fwd_pos, bwd_pos = got["out"] > 0, z_bwd > 0
    diff = fwd_pos != bwd_pos
    # y error (fp32 accumulation) + 2 bf16 ulps of y, through z = g (y - mean) rstd
    slack = g64.abs() * rstd * (2 * bf16_ulp(y) + ref["pre"][2]) + 64 * U * (z_exact.abs() + b64.abs())
    outside = diff & (z_exact.abs() > slack)
    assert not bool(outside.any()), f"{int(outside.sum())} forward/backward ReLU decisions differ away from z = 0"
    record(f"linear_bounds/{name}", mismatches=int(diff.sum()), elements=N * H)


# ---- bwd_input --------------------------------------------------------------------------------------------------------
DX_ROWS = [  # (id, dtype, N, Hout (reduction), K (output columns))
    ("dx_tc_f32_k128", F32, NBIG, 128, 128),
    ("dx_tc_bf16_k64", BF16, NBIG, 256, 64),
    ("dx_tc_bf16_k256_n77", BF16, 77, 128, 256),
    ("dx_simt_f32_k40", F32, 5003, 64, 40),
    ("dx_simt_bf16_k48", BF16, 5003, 96, 48),
]


@pytest.mark.gpu
@pytest.mark.parametrize("sign", ["mixed", "nonneg"])
@pytest.mark.parametrize("row", DX_ROWS, ids=[r[0] for r in DX_ROWS])
def test_linear_bwd_input_within_bounds(row, sign):
    name, dt, N, Hout, K = row
    cabi = _ops()
    gen = torch.Generator(device="cuda").manual_seed(_seed(name + sign))
    g = _operand((N, Hout), dt, sign, gen)
    w = _operand((Hout, K), dt, sign, gen, 1.0 / Hout if sign == "nonneg" else Hout ** -0.5)
    rs = torch.rand(N, generator=gen, device="cuda") + 0.1
    add = _operand((N, K), dt, sign, gen)
    ar = Arena()
    ga = ar.out((N, K), dt)
    ws, ws_bytes = ar.ws(cabi.lib.dfw_linear_ws_bytes(K, Hout, 0, _dt(g)))
    _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_linear_bwd_input(g.data_ptr(), w.data_ptr(), rs.data_ptr(), add.data_ptr(), ga.data_ptr(),
                                                                          N, Hout, K, _dt(g), ws.data_ptr(), ws_bytes, _stream())))
    ar.check(name)
    assert_kernels(name, names, _tc_kernel(dt, N, K, Hout, 0) or r"\bk_linear<")
    prod = g.double() @ w.double()
    S = g.double().abs() @ w.double().abs()
    r = rs.double()[:, None] * prod + add.double()
    Ef = short_bound(rs.double()[:, None] * S + add.double().abs(), Hout)
    b = Ef + (2.0 ** -8 * (r.abs() + Ef) if dt == BF16 else 0.0)
    margins = {"g_a": assert_bound(f"{name}/g_a", ga, r, b)}
    if dt == BF16:
        bias = assert_no_rounding_bias(f"{name}/g_a", ga, r, Ef)
        if bias is not None:
            margins["g_a_bias_ulp"] = bias
    record(f"linear_bounds/bwd_input/{name}/{sign}", kernel=sorted(set(names)), simt=SIMT, **margins)


# ---- bwd_weight -------------------------------------------------------------------------------------------------------
DW_ROWS = [  # (id, dtype, Hout, k1, k2, dbias, misaligned g_y)
    ("tc_f32", F32, 128, 128, 64, True, False),
    ("tc_bf16", BF16, 128, 128, 64, True, False),
    ("tinyk_tiled_f32", F32, 64, 10, 0, False, False),
    ("tinyk_tiled_bf16", BF16, 256, 16, 0, False, False),
    ("tinyk_legacy_h6", F32, 6, 10, 0, False, False),
    ("tinyk_legacy_misaligned_bf16", BF16, 64, 3, 0, False, True),
    ("simt_splitk_f32", F32, 48, 40, 24, True, False),
    ("simt_splitk_bf16", BF16, 96, 40, 0, True, False),
]


_SPARE = []


def _pn(t):
    """Device pointer of an operand; an empty one (N = 0) still gets a valid address, since the ABI rejects NULL operands and
    torch reports 0 as the address of an empty tensor."""
    if t is None:
        return None
    if t.numel():
        return t.data_ptr()
    if not _SPARE:
        _SPARE.append(torch.empty(256, dtype=torch.uint8, device="cuda"))
    return _SPARE[0].data_ptr()


def tc_dw_chain_bound(g, a, Hout, k1, k2, tf32):
    """Per-element error bound of the tensor-core dW (dfw_linear_dw_tc.cu) from its accumulation chain.

    dw_plan_tc cuts the nodes into `splits` slices of `per` nodes (about two CTAs per SM).  A CTA accumulates its slice's
    [128 x 128] partial tile in TMEM, one MMA per k-step of 16 nodes (bf16) or 8 nodes (tf32), and the tensor core truncates
    the fp32 accumulator at every step: the error of step t is below one ulp, 2u |P_t|, of the running partial P_t.  fp32
    adds a second accumulator per step (the cross terms of 3xTF32), counted here with the same P_t.  k_dw_reduce then adds
    the `splits` partials in fp32: a warp keeps four sums over every 32nd partial, adds them in pairs, and the eight warps'
    sums are added in order, so no partial passes through more than ceil(splits / 32) + 10 roundings.
    So  |err| <= 2u (c sum_t |P_t| + (ceil(splits / 32) + 10) sum_s |P_s|),  c = 2 for fp32, 1 for bf16.
    The truncations share a sign, so their sum grows with the slice length instead of its square root, and on 2e5 nodes
    the tensor-wide rel_l2 of a correct kernel can exceed 4x a CPU fp32 summation (2^-20 floor)."""
    from math import ceil

    N = g.shape[0]
    tiles = max(1, ((Hout + 127) // 128) * ((k1 + 127) // 128 + (k2 + 127) // 128))
    splits = max(1, 2 * 148 // tiles)
    per = max(32, ceil(ceil(N / splits) / 32) * 32)
    splits = max(1, ceil(N / per))
    kstep, c = (8, 2) if tf32 else (16, 1)
    g64, a64 = g.double(), a.double()
    chain = torch.zeros(g.shape[1], a.shape[1], dtype=torch.float64, device=g.device)
    finals = torch.zeros_like(chain)
    for s0 in range(0, N, per):
        gs, as_ = g64[s0:s0 + per], a64[s0:s0 + per]
        nb = -(-gs.shape[0] // kstep)
        pad = nb * kstep - gs.shape[0]
        gs = torch.nn.functional.pad(gs, (0, 0, 0, pad)).view(nb, kstep, -1)
        as_ = torch.nn.functional.pad(as_, (0, 0, 0, pad)).view(nb, kstep, -1)
        prefix = torch.bmm(gs.transpose(1, 2), as_).cumsum(0)
        chain += prefix.abs().sum(0)
        finals += prefix[-1].abs()
    return 2 * U * (c * chain + (ceil(splits / 32) + 10) * finals)


def _dw_expect(row, N):
    name, dt, Hout, k1, k2, dbias, mis = row
    if N == 0:
        return [r"k_dw_reduce<"], [r"\bk_linear<", r"k_dw_tc", r"smallk"]
    if SIMT or name.startswith("simt"):
        return [r"\bk_linear<", r"k_dw_reduce<"], [r"k_dw_tc", r"smallk"]
    if name.startswith("tc"):
        return [r"k_dw_tc"] + ([r"k_colsum_partial"] if dbias else []), [r"\bk_linear<"]
    if "legacy" in name:
        return [r"k_linear_smallk_dw", r"k_smallk_dw_reduce"], [r"k_smallk_dw_tiled"]
    return [r"k_smallk_dw_tiled", r"k_smallk_dw_reduce"], [r"k_linear_smallk_dw"]


@pytest.mark.gpu
@pytest.mark.parametrize("N", [0, 1, 129, 200003])
@pytest.mark.parametrize("row", DW_ROWS, ids=[r[0] for r in DW_ROWS])
def test_linear_bwd_weight_within_bounds(row, N):
    """Every dW path, plain and with accumulate = 1 into a prefilled dW / dbias (an ABI-only option)."""
    name, dt, Hout, k1, k2, want_db, misaligned = row
    cabi = _ops()
    gen = torch.Generator(device="cuda").manual_seed(_seed(name) + N)
    for sign in ("mixed", "nonneg"):
        g = _operand((N, Hout), dt, sign, gen)
        if misaligned:  # one element past a 16-byte boundary: the tiled tiny-K kernel's vector loads are ruled out
            g = torch.empty(N * Hout + 1, dtype=dt, device="cuda")[1:].view(N, Hout).copy_(g)
        a1 = _operand((N, k1), dt, sign, gen)
        a2 = _operand((N, k2), dt, sign, gen) if k2 else None
        ws_bytes = cabi.lib.dfw_linear_bwd_weight_ws_bytes(N, Hout, k1, k2)
        r1 = g.double().T @ a1.double()
        S1 = g.double().abs().T @ a1.double().abs()
        r2 = g.double().T @ a2.double() if k2 else None
        S2 = g.double().abs().T @ a2.double().abs() if k2 else None
        rb, Sb = g.double().sum(0), g.double().abs().sum(0)
        gc, a1c = g.float().cpu(), a1.float().cpu()
        cpu = {"dw1": gc.T @ a1c, "dw2": gc.T @ a2.float().cpu() if k2 else None, "db": gc.sum(0)}
        for acc in (0, 1):
            ar = Arena()
            pre = {"dw1": torch.randn(Hout, k1, generator=gen, device="cuda"),
                   "dw2": torch.randn(Hout, k2, generator=gen, device="cuda") if k2 else None,
                   "db": torch.randn(Hout, generator=gen, device="cuda") if want_db else None}
            outs = {k: (ar.out(v.shape, F32, fill=v if acc else None) if v is not None else None) for k, v in pre.items()}
            ws, _ = ar.ws(ws_bytes)
            _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_linear_bwd_weight(
                _pn(g), _pn(a1), k1, _pn(a2), k2, outs["dw1"].data_ptr(), _p(outs["dw2"]), _p(outs["db"]), N, Hout, _dt(g), acc,
                ws.data_ptr(), ws_bytes, _stream())))
            row_id = f"{name}/N{N}/{sign}/acc{acc}"
            ar.check(row_id)
            present, absent = _dw_expect(row, N)
            assert_kernels(row_id, names, present, absent)
            margins = {}
            for key, r, S in (("dw1", r1, S1), ("dw2", r2, S2), ("db", rb, Sb)):
                if outs[key] is None:
                    continue
                if N == 0:  # nothing to reduce: zeros, or dW left exactly as it was
                    expect = pre[key] if acc else torch.zeros_like(pre[key])
                    assert torch.equal(outs[key], expect), f"{row_id}/{key}: N = 0 must write zeros / leave dW untouched"
                    continue
                if acc:
                    p64 = pre[key].double()
                    margins[key] = assert_bound(f"{row_id}/{key}", outs[key], p64 + r,
                                                2.0 ** -16 * S + 2 * U * (p64.abs() + r.abs()))
                else:
                    chain = None
                    if name.startswith("tc") and not SIMT and key != "db":  # dbias is the separate fp32 colsum kernel
                        chain = tc_dw_chain_bound(g, a1 if key == "dw1" else a2, Hout, k1, k2, dt == F32)
                    margins[key], margins[key + "_l2_use"] = long_check(f"{row_id}/{key}", outs[key], r, S, cpu[key], chain_bound=chain)
            record(f"linear_bounds/bwd_weight/{row_id}", kernel=sorted(set(names)), simt=SIMT, **margins)


# ---- epilogue_bwd -----------------------------------------------------------------------------------------------------
def _ln_saved(name, dt, N, H, gen):
    """pre_out, ln_stats, gamma, beta with no |z| within 2^-12 (|g xhat| + |b|) of 0: the recomputed ReLU mask is then
    the same in fp32 and fp64."""
    pre = torch.randn(N, H, generator=gen, device="cuda") * 2 + 0.3
    pre = pre.to(dt)
    p64 = pre.double()
    mean, var = p64.mean(1), p64.var(1, unbiased=False)
    stats = torch.stack([mean, 1.0 / torch.sqrt(var + 1e-5)], 1).float()
    gamma = (torch.rand(H, generator=gen, device="cuda") + 0.5) * torch.sign(torch.randn(H, generator=gen, device="cuda"))
    beta = torch.randn(H, generator=gen, device="cuda") * 0.5
    g64, b64 = gamma.double(), beta.double()
    st = stats.double()
    for _ in range(20):
        xh = (pre.double() - st[:, :1]) * st[:, 1:]
        near = (xh * g64 + b64).abs() < 2.0 ** -12 * ((g64 * xh).abs() + b64.abs())
        if not bool(near.any()):
            break
        fresh = (torch.randn(N, H, generator=gen, device="cuda") * 2 + 0.3).to(dt)
        pre = torch.where(near, fresh, pre)
    else:
        raise AssertionError("could not keep z away from 0")
    return pre, stats, gamma, beta


def _run_eb(g_out, g_rowdot, rdw, pre, stats, act, gamma, beta, p, seed, flags, N, H, dt, want):
    cabi = _ops()
    ar = Arena()
    gy = ar.out((N, H), dt)
    o = {k: (ar.out((n,), F32) if k in want else None) for k, n in (("dgamma", H), ("dbeta", H), ("d_rowdot_w", H), ("d_rowdot_b", 1), ("d_bias", H))}
    ws, ws_bytes = ar.ws(cabi.lib.dfw_epilogue_bwd_ws_bytes(N, H))
    _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_epilogue_bwd(
        _p(g_out), _p(g_rowdot), _p(rdw), _p(pre), _p(stats), _p(act), _p(gamma), _p(beta), p, seed, gy.data_ptr(), _p(o["dgamma"]),
        _p(o["dbeta"]), _p(o["d_rowdot_w"]), _p(o["d_rowdot_b"]), _p(o["d_bias"]), N, H, flags, int(dt == BF16),
        ws.data_ptr(), ws_bytes, _stream())))
    return gy, o, names, ar


EB_N = 200003
ACT_ROWS = [(h, dt, kind) for h in (4, 12, 64, 256) for dt in (F32, BF16) for kind in ("relu", "rowdot")]


@pytest.mark.gpu
@pytest.mark.parametrize("h,dt,kind", ACT_ROWS, ids=[f"h{h}_{'f32' if d == F32 else 'bf16'}_{k}" for h, d, k in ACT_ROWS])
def test_epilogue_bwd_packed_rows_within_bounds(h, dt, kind):
    """k_act_bwd: the encoder's ReLU (mask from the saved output `act`) and the decoder's row dot with dropout; at H = 12 the
    256 threads of a block do not divide into whole rows."""
    cabi = _ops()
    name = f"act_bwd_h{h}_{dt}_{kind}"
    N = EB_N
    gen = torch.Generator(device="cuda").manual_seed(_seed(name))
    p, seed = (0.2, 99) if kind == "rowdot" else (0.0, 0)
    keep = _keep(seed, N, h, p) if p else torch.ones(N, h, dtype=torch.float64, device="cuda")
    act = (torch.randn(N, h, generator=gen, device="cuda").clamp_min(0).double() * keep).to(dt)  # saved output: post-ReLU, post-dropout
    rdw = torch.randn(h, generator=gen, device="cuda") if kind == "rowdot" else None
    g_rowdot = torch.randn(N, generator=gen, device="cuda") if kind == "rowdot" else None
    g_out = torch.randn(N, h, generator=gen, device="cuda").to(dt) if kind == "relu" else None
    flags = cabi.EP_RELU | (cabi.EP_DROPOUT if p else 0)
    m = (act.double() > 0).double()
    if kind == "rowdot":
        g_in = g_rowdot.double()[:, None] * rdw.double()[None, :]
    else:
        g_in = g_out.double()
    r_gy = g_in * keep * m
    for want_bias in (False, True):
        want = {"d_bias"} if want_bias else set()
        if kind == "rowdot":
            want |= {"d_rowdot_w", "d_rowdot_b"}
        gy, o, names, ar = _run_eb(g_out, g_rowdot, rdw, None, None, act, None, None, p, seed, flags, N, h, dt, want)
        row_id = f"{name}/bias{int(want_bias)}"
        ar.check(row_id)
        assert_kernels(row_id, names, r"k_act_bwd<", [r"k_epilogue_bwd<"])
        Ef = short_bound(r_gy.abs(), 1)
        margins = {"g_y": assert_bound(f"{row_id}/g_y", gy, r_gy, Ef + (2.0 ** -8 * (r_gy.abs() + Ef) if dt == BF16 else 0.0))}
        if dt == BF16:
            margins["g_y_bias_ulp"] = assert_no_rounding_bias(f"{row_id}/g_y", gy, r_gy, Ef)
        if want_bias:
            cpu = (g_in.float().cpu() * keep.float().cpu() * m.float().cpu()).sum(0)
            margins["d_bias"], _ = long_check(f"{row_id}/d_bias", o["d_bias"], r_gy.sum(0), (r_gy.abs() + Ef).sum(0), cpu)
        if kind == "rowdot":
            a64 = act.double()
            cpu_w = (g_rowdot.cpu()[:, None] * act.float().cpu()).sum(0)
            margins["d_rowdot_w"], _ = long_check(f"{row_id}/d_rowdot_w", o["d_rowdot_w"], g_rowdot.double() @ a64,
                                                  g_rowdot.double().abs() @ a64.abs(), cpu_w)
            margins["d_rowdot_b"], _ = long_check(f"{row_id}/d_rowdot_b", o["d_rowdot_b"], g_rowdot.double().sum().reshape(1),
                                                  g_rowdot.double().abs().sum().reshape(1), g_rowdot.cpu().sum().reshape(1))
        record(f"linear_bounds/epilogue_bwd/{row_id}", kernel=sorted(set(names)), **margins)


LN_ROWS = [(spec, h, dt) for spec in (0, 1, 3) for h in (64, 128, 192, 256) for dt in (F32, BF16)]


@pytest.mark.gpu
@pytest.mark.parametrize("spec,h,dt", LN_ROWS, ids=[f"spec{s}_h{h}_{'f32' if d == F32 else 'bf16'}" for s, h, d in LN_ROWS])
def test_epilogue_bwd_layernorm_within_bounds(spec, h, dt):
    """k_epilogue_bwd: SPEC 0 = LayerNorm without ReLU (run-time flags, with dropout), 1 = the SAGE tail, 3 = the tail with
    dropout; one lane group per 16 bytes (H <= 128) or two (H in {192, 256})."""
    cabi = _ops()
    name = f"ln_bwd_spec{spec}_h{h}_{dt}"
    N = EB_N
    gen = torch.Generator(device="cuda").manual_seed(_seed(name))
    pre, stats, gamma, beta = _ln_saved(name, dt, N, h, gen)
    relu = spec != 0
    p, seed = (0.15, 4242) if spec in (0, 3) else (0.0, 0)
    flags = cabi.EP_LAYERNORM | (cabi.EP_RELU if relu else 0) | (cabi.EP_DROPOUT if p else 0)
    g_out = torch.randn(N, h, generator=gen, device="cuda").to(dt)
    keep = _keep(seed, N, h, p) if p else torch.ones(N, h, dtype=torch.float64, device="cuda")
    st = stats.double()
    mean, rstd = st[:, :1], st[:, 1:]
    g64, b64 = gamma.double(), beta.double()
    xh = (pre.double() - mean) * rstd
    m = ((xh * g64 + b64) > 0).double() if relu else torch.ones_like(xh)
    gg0 = g_out.double() * keep * m
    gh = gg0 * g64
    s1, s2 = gh.mean(1, keepdim=True), (gh * xh).mean(1, keepdim=True)
    r_gy = rstd * (gh - s1 - xh * s2)
    S_gy = rstd * (gh.abs() + gh.abs().mean(1, keepdim=True) + xh.abs() * (gh * xh).abs().mean(1, keepdim=True))
    Ef = short_bound(S_gy, h)
    # CPU fp32 on the same inputs: the yardstick of the column sums
    c_xh = (pre.float().cpu() - stats.cpu()[:, :1]) * stats.cpu()[:, 1:]
    c_gg0 = g_out.float().cpu() * keep.float().cpu() * m.float().cpu()
    c_gh = c_gg0 * gamma.cpu()
    c_gy = stats.cpu()[:, 1:] * (c_gh - c_gh.mean(1, keepdim=True) - c_xh * (c_gh * c_xh).mean(1, keepdim=True))
    for want_bias in (False, True):
        want = {"dgamma", "dbeta"} | ({"d_bias"} if want_bias else set())
        gy, o, names, ar = _run_eb(g_out, None, None, pre, stats, None, gamma, beta, p, seed, flags, N, h, dt, want)
        row_id = f"{name}/bias{int(want_bias)}"
        ar.check(row_id)
        assert_kernels(row_id, names, rf"k_epilogue_bwd<[^>]*,\s*{spec}>", [r"k_act_bwd<"])
        margins = {"g_y": assert_bound(f"{row_id}/g_y", gy, r_gy, Ef + (2.0 ** -8 * (r_gy.abs() + Ef) if dt == BF16 else 0.0))}
        if dt == BF16:
            margins["g_y_bias_ulp"] = assert_no_rounding_bias(f"{row_id}/g_y", gy, r_gy, Ef)
        margins["dgamma"], _ = long_check(f"{row_id}/dgamma", o["dgamma"], (gg0 * xh).sum(0), (gg0 * xh).abs().sum(0) * (1 + 4 * U),
                                          (c_gg0 * c_xh).sum(0))
        margins["dbeta"], _ = long_check(f"{row_id}/dbeta", o["dbeta"], gg0.sum(0), gg0.abs().sum(0), c_gg0.sum(0))
        if want_bias:
            margins["d_bias"], _ = long_check(f"{row_id}/d_bias", o["d_bias"], r_gy.sum(0), (S_gy + Ef).sum(0), c_gy.sum(0))
        record(f"linear_bounds/epilogue_bwd/{row_id}", kernel=sorted(set(names)), **margins)


# ---- small related checks ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cast_is_bit_identical_to_torch():
    """dfw_cast fp32 <-> bf16 against torch.Tensor.to: round-to-nearest-even ties, subnormals, overflow to +-Inf, +-0, +-Inf;
    NaNs compared with isnan.  Every bf16 bit pattern, plus 2^20 random fp32 bit patterns."""
    from deep_fem_uav_wing.gnn import _cabi

    specials = [0.0, -0.0, float("inf"), float("-inf"), float("nan"), 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8),
                2.0 ** -149, 2.0 ** -133 + 2.0 ** -141, 3 * 2.0 ** -141, 1e-40, -1e-40, 2.0 ** -126, 3.3961e38, 3.4028e38, -3.4028e38,
                float(np.finfo(np.float32).max), 65504.0, 2.0 ** 127 * (2 - 2.0 ** -8)]
    gen = torch.Generator().manual_seed(5)
    rnd = torch.randint(-2 ** 31, 2 ** 31 - 1, (1 << 20,), generator=gen, dtype=torch.int64).to(torch.int32).view(F32)
    ties = ((torch.arange(-4096, 4096, dtype=torch.int32) << 16) | 0x8000).view(F32)  # exactly half-way between two bf16
    src = torch.cat([torch.tensor(specials, dtype=F32), rnd, ties])
    d_src = src.cuda()
    d_dst = torch.empty(src.numel(), dtype=BF16, device="cuda")
    _cabi.check(_cabi.lib.dfw_cast(d_src.data_ptr(), 0, d_dst.data_ptr(), 1, src.numel(), _stream()))
    want, got = src.to(BF16), d_dst.cpu()
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan)
    assert torch.equal(got[~nan].view(torch.int16), want[~nan].view(torch.int16)), "fp32 -> bf16 differs from torch"
    allb = torch.arange(-2 ** 15, 2 ** 15, dtype=torch.int32).to(torch.int16).view(BF16)
    d32 = torch.empty(allb.numel(), dtype=F32, device="cuda")
    d16 = allb.cuda()
    _cabi.check(_cabi.lib.dfw_cast(d16.data_ptr(), 1, d32.data_ptr(), 0, allb.numel(), _stream()))
    want32, got32 = allb.to(F32), d32.cpu()
    nan = torch.isnan(want32)
    assert torch.equal(torch.isnan(got32), nan)
    assert torch.equal(got32[~nan].view(torch.int32), want32[~nan].view(torch.int32)), "bf16 -> fp32 differs from torch"


@pytest.mark.gpu
@pytest.mark.parametrize("mean", [True, False])
def test_masked_mse_bf16_within_bounds(mean):
    """dfw_masked_mse_fwd/bwd in bf16, C = 3, N = 200003, against fp64 (loss: a long reduction; gradient: one product)."""
    from deep_fem_uav_wing.gnn import _cabi

    N, C = 200003, 3
    gen = torch.Generator(device="cuda").manual_seed(11 + mean)
    pred = torch.randn(N, C, generator=gen, device="cuda").to(BF16)
    targ = torch.randn(N, C, generator=gen, device="cuda").to(BF16)
    mask = (torch.rand(N, generator=gen, device="cuda") < 0.7).to(torch.uint8)
    ar = Arena()
    res = ar.out((2,), F32)
    gp = ar.out((N, C), BF16)
    ws, ws_bytes = ar.ws(_cabi.lib.dfw_masked_mse_ws_bytes(N, C))
    g_loss = torch.tensor([0.75], device="cuda")
    _cabi.check(_cabi.lib.dfw_masked_mse_fwd(pred.data_ptr(), targ.data_ptr(), mask.data_ptr(), N, C, int(mean), 1, res.data_ptr(),
                                             ws.data_ptr(), ws_bytes, _stream()))
    _cabi.check(_cabi.lib.dfw_masked_mse_bwd(pred.data_ptr(), targ.data_ptr(), mask.data_ptr(), res.data_ptr(), g_loss.data_ptr(), N, C,
                                             int(mean), 1, gp.data_ptr(), _stream()))
    ar.check("masked_mse")
    d = pred.double() - targ.double()
    m = mask.double()[:, None]
    cnt = float(mask.sum()) * C
    div = max(cnt, 1.0) if mean else 1.0
    sq = (d * d * m).sum()
    r_loss = sq / div
    assert res[1].item() == cnt
    cpu = ((pred.float().cpu() - targ.float().cpu()) ** 2 * mask.cpu().float()[:, None]).sum() / div
    m_loss, _ = long_check("masked_mse/loss", res[:1], r_loss.reshape(1), r_loss.reshape(1), cpu.reshape(1))
    r_g = 2 * 0.75 * d * m / div
    Ef = short_bound(r_g.abs(), 1) + 4 * U * r_g.abs()  # the fp32 scale 2 g / count carries two roundings of its own
    m_g = assert_bound("masked_mse/g_pred", gp, r_g, Ef + 2.0 ** -8 * (r_g.abs() + Ef))
    bias = assert_no_rounding_bias("masked_mse/g_pred", gp, r_g, Ef)
    record(f"linear_bounds/masked_mse/mean{int(mean)}", loss=m_loss, g_pred=m_g, g_pred_bias_ulp=bias)
