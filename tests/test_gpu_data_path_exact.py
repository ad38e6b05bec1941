"""The data-path kernels element by element: node features, vertex normals, stress metrics and the fp32 masked MSE.

Every number a user sees passes through these four small kernels, so each is compared with a CPU restatement of the
same operation, at the sizes where their loops and grids change shape and at the values where the guards decide:

- ``dfw_node_features`` / ``dfw_node_features_batched`` (``k_pos_minmax``, ``k_node_features``, ``k_pos_minmax_cases``,
  ``k_node_features_cases``): x bit for bit against a numpy float32 restatement of ``dataset.py:108-121``, y within
  1 ulp of the fp64 ``log1p`` rounded to fp32 (CUDA's documented ``log1pf`` bound).  A zero is compared by value: numpy's
  min over ``+0`` and ``-0`` depends on their order.  A NaN coordinate makes its axis NaN in every row of its case.
- ``dfw_vertex_normals`` (``k_incidence_expand``, ``k_vertex_normals``): bit for bit against a numpy float32 oracle
  that forms each face normal with separate products in ``numpy.cross`` order and sums a vertex's faces in ascending
  incidence id 3f + k.
- ``dfw_stress_metrics`` (``k_stress_metrics<float|bf16>``): exact on inputs whose fp32 partials are exact; elsewhere
  ``max_error`` and ``count`` exact and mae / rmse inside bounds derived from the kernel's summation order.  A NaN
  error makes all three statistics of its subset NaN.
- ``dfw_masked_mse_fwd/bwd`` fp32 (``k_mse_fwd``, ``k_mse_bwd``): the loss exact on small-integer differences and
  bounded otherwise; every gradient element within three roundings of fp64.

Raw-ABI outputs and workspaces sit in guard bands (``helpers.Arena``), every call asserts from torch.profiler which
kernels ran, NaN is compared by position, and the achieved margins go to ``record()``."""
import ctypes
import math
import re
from fractions import Fraction

import numpy as np
import pytest
import torch

from helpers import Arena, launched_kernels, record

F32, BF16 = torch.float32, torch.bfloat16
U = 2.0 ** -24          # fp32 unit roundoff
UD = 2.0 ** -53         # fp64 unit roundoff
NUM_SMS = 148           # dfw_common.cuh kNumSMs
MAX_BLOCKS = NUM_SMS * 4  # kFeatMaxBlocks, kMetMaxBlocks, kMseMaxBlocks
G_LOSS = 0.75


def _cabi():
    from deep_fem_uav_wing.gnn import _cabi

    return _cabi


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _ptr(t):
    return t.data_ptr() if t is not None and t.numel() else None


def assert_kernels(row, names, expect, absent=()):
    for pat in expect:
        assert any(re.search(pat, n) for n in names), f"{row}: expected a kernel matching {pat!r}, launched {sorted(set(names))}"
    for pat in absent:
        assert not any(re.search(pat, n) for n in names), f"{row}: unexpected kernel matching {pat!r} in {sorted(set(names))}"


# ---- comparisons (CPU) ------------------------------------------------------------------------------------------------
def _ordered(a):
    """fp32 bits as integers in the order of the values (-0 and +0 both map to 0)."""
    i = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    return np.where(i < 0, -(i & 0x7FFFFFFF), i)


def mismatches(got, ref, zero_by_value):
    """Mask of elements that differ: NaN by position, everything else by bits (zeros by value if asked)."""
    got, ref = np.asarray(got, np.float32), np.asarray(ref, np.float32)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    gn, rn = np.isnan(got), np.isnan(ref)
    diff = (got.view(np.uint32) != ref.view(np.uint32)) & ~gn & ~rn
    if zero_by_value:
        diff &= ~((got == 0) & (ref == 0))
    return diff | (gn != rn)


def assert_same(name, got, ref, zero_by_value=False):
    bad = mismatches(got, ref, zero_by_value)
    n = int(bad.sum())
    if n:
        i = int(np.flatnonzero(bad)[0])
        raise AssertionError(f"{name}: {n} of {bad.size} elements differ (first at flat index {i}: got {np.asarray(got).flat[i]!r}, "
                             f"ref {np.asarray(ref).flat[i]!r})")


def ulp_distance(got, ref):
    """Largest distance in fp32 steps between got and ref; NaN must sit at the same positions (inf - inf counts 0)."""
    got, ref = np.asarray(got, np.float32), np.asarray(ref, np.float32)
    gn, rn = np.isnan(got), np.isnan(ref)
    assert np.array_equal(gn, rn), f"NaN at {np.flatnonzero(gn != rn)[:5]}"
    ok = ~gn
    return int(np.abs(_ordered(got[ok]) - _ordered(ref[ok])).max()) if ok.any() else 0


def gamma(n, u=U):
    """gamma_n = n u / (1 - n u): the relative error bound of n roundings in a chain."""
    return n * u / (1.0 - n * u)


# ---- node features: oracle -------------------------------------------------------------------------------------------
def features_oracle(pos, normal, stress, gp, case_ptr, normalize_pos, log_scale):
    """numpy float32 restatement of ``dataset.py:108-121`` for B concatenated cases: rows case_ptr[b]..case_ptr[b+1] use
    their own min / max and gp[b].  numpy's minimum / maximum propagate NaN.  The norm is written out as numpy's
    ``linalg.norm`` evaluates it in float32: sqrt((x*x + y*y) + z*z)."""
    pos, normal = np.asarray(pos, np.float32).reshape(-1, 3), np.asarray(normal, np.float32).reshape(-1, 3)
    case_ptr = np.asarray(case_ptr, np.int64)
    lens = np.diff(case_ptr)
    case = np.repeat(np.arange(len(lens)), lens)
    with np.errstate(all="ignore"):
        if normalize_pos:
            mn = np.zeros((len(lens), 3), np.float32)
            mx = np.zeros((len(lens), 3), np.float32)
            nz = np.flatnonzero(lens > 0)
            if nz.size:
                mn[nz] = np.minimum.reduceat(pos, case_ptr[:-1][nz], axis=0)
                mx[nz] = np.maximum.reduceat(pos, case_ptr[:-1][nz], axis=0)
            rg = mx - mn
            rg[rg < np.float32(1e-8)] = np.float32(1.0)
            xp = (pos - mn[case]) / rg[case]
        else:
            xp = pos.copy()
        nx, ny, nzc = normal[:, 0], normal[:, 1], normal[:, 2]
        ln = np.sqrt((nx * nx + ny * ny) + nzc * nzc)
        ln[ln < np.float32(1e-8)] = np.float32(1.0)
        xn = normal / ln[:, None]
        x = np.concatenate([xp, xn, np.asarray(gp, np.float32).reshape(-1, 4)[case]], axis=1).astype(np.float32)
        y = None
        if stress is not None:
            s = np.asarray(stress, np.float32).reshape(-1)
            y = (np.log1p(s.astype(np.float64)).astype(np.float32) if log_scale else s.copy()).reshape(-1, 1)
    return x, y


def check_features(name, x, y, xr, yr, log_scale):
    """x by bits (zeros by value), y by bits without log_scale and within 1 ulp with it.  Returns y's ulp distance."""
    assert_same(f"{name}/x", x, xr, zero_by_value=True)
    if yr is None:
        return 0
    if not log_scale:
        assert_same(f"{name}/y", y, yr)
        return 0
    d = ulp_distance(y, yr)
    assert d <= 1, f"{name}/y: log1pf is {d} ulp from the correctly rounded log1p (CUDA documents 1 ulp)"
    return d


# ---- node features: device runs --------------------------------------------------------------------------------------
def run_features(pos, normal, stress, gp4, normalize_pos, log_scale):
    """dfw_node_features on one case through the raw ABI; returns numpy (x, y)."""
    cabi = _cabi()
    N = len(pos)
    pos_d, nrm_d = _dev(np.asarray(pos, np.float32).reshape(-1, 3)), _dev(np.asarray(normal, np.float32).reshape(-1, 3))
    st_d = _dev(np.asarray(stress, np.float32)) if stress is not None else None
    ar = Arena()
    x = ar.out((N, 10), F32)
    y = ar.out((N, 1), F32) if stress is not None else None
    ws, wsb = ar.ws(cabi.lib.dfw_node_features_ws_bytes(N))
    gp = (ctypes.c_float * 4)(*[float(v) for v in np.asarray(gp4, np.float32)])
    _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_node_features(
        pos_d.data_ptr(), nrm_d.data_ptr(), _ptr(st_d), gp, int(normalize_pos), int(log_scale), x.data_ptr(), _ptr(y), N, ws.data_ptr(), wsb,
        _stream())))
    ar.check("node_features")
    if N:
        assert_kernels("node_features", names, [r"\bk_node_features\b"] + ([r"\bk_pos_minmax\b"] if normalize_pos else []),
                       [r"_cases\b"] + ([] if normalize_pos else [r"\bk_pos_minmax\b"]))
    return x.cpu().numpy(), (y.cpu().numpy() if y is not None else None)


def run_features_batched(pos, normal, stress, gp, case_ptr, max_case_rows, normalize_pos, log_scale):
    cabi = _cabi()
    N, B = len(pos), len(case_ptr) - 1
    pos_d, nrm_d = _dev(np.asarray(pos, np.float32).reshape(-1, 3)), _dev(np.asarray(normal, np.float32).reshape(-1, 3))
    st_d = _dev(np.asarray(stress, np.float32)) if stress is not None else None
    gp_d, cp_d = _dev(np.asarray(gp, np.float32).reshape(-1, 4)), _dev(np.asarray(case_ptr, np.int64))
    ar = Arena()
    x = ar.out((N, 10), F32)
    y = ar.out((N, 1), F32) if stress is not None else None
    ws, wsb = ar.ws(cabi.lib.dfw_node_features_batched_ws_bytes(B))
    _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_node_features_batched(
        _ptr(pos_d), _ptr(nrm_d), _ptr(st_d), gp_d.data_ptr(), cp_d.data_ptr(), B, int(max_case_rows), int(normalize_pos), int(log_scale),
        _ptr(x), _ptr(y), ws.data_ptr(), wsb, _stream())))
    ar.check("node_features_batched")
    assert_kernels("node_features_batched", names, [r"\bk_node_features_cases\b"] + ([r"\bk_pos_minmax_cases\b"] if normalize_pos else []),
                   [r"\bk_node_features\b", r"\bk_pos_minmax\b"] + ([] if normalize_pos else [r"\bk_pos_minmax_cases\b"]))
    return x.cpu().numpy(), (y.cpu().numpy() if y is not None else None)


def _random_case(rng, n, with_zero_normals=True):
    pos = (rng.standard_normal((n, 3)) * [2.0, 0.5, 0.1] + [-1.0, 3.0, -0.05]).astype(np.float32)
    normal = rng.standard_normal((n, 3)).astype(np.float32)
    if with_zero_normals and n > 10:
        normal[rng.random(n) < 0.01] = 0.0
    stress = (rng.gamma(2.0, 3e6, n)).astype(np.float32)
    gp = rng.uniform(-1, 1, 4).astype(np.float32)
    return pos, normal, stress, gp


# ---- vertex normals: oracle ------------------------------------------------------------------------------------------
def normals_f32_oracle(pos, faces):
    """Area-weighted vertex normals in float32, in the kernel's operation order: per face a = p1 - p0, b = p2 - p0 and
    cross(a, b) in ``numpy.cross`` order with every product rounded on its own; per vertex the face normals of its
    incidences 3f + k added in ascending id, starting from +0.  A face with an index outside [0, N) is skipped and
    counted.  The loop runs over the rank within each vertex's incidence list, so a fan of degree d costs d numpy passes."""
    pos = np.asarray(pos, np.float32).reshape(-1, 3)
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    N = len(pos)
    valid = ((f >= 0) & (f < N)).all(axis=1)
    out = np.zeros((N, 3), np.float32)
    g = f[valid]
    if len(g) == 0:
        return out, int((~valid).sum())
    with np.errstate(all="ignore"):
        p0, p1, p2 = pos[g[:, 0]], pos[g[:, 1]], pos[g[:, 2]]
        a, b = p1 - p0, p2 - p0
        fn = np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1],
                       a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                       a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)
        inc_v = g.reshape(-1)  # incidences of the valid faces in ascending id
        inc_f = np.repeat(np.arange(len(g)), 3)
        order = np.argsort(inc_v, kind="stable")
        vs = inc_v[order]
        rank = np.arange(len(order)) - np.searchsorted(vs, vs, side="left")
        by_rank = np.argsort(rank, kind="stable")
        edges = np.searchsorted(rank[by_rank], np.arange(int(rank.max()) + 2))
        for r in range(int(rank.max()) + 1):
            sel = order[by_rank[edges[r]:edges[r + 1]]]  # at most one incidence per vertex
            v = inc_v[sel]
            out[v] = out[v] + fn[inc_f[sel]]
    return out, int((~valid).sum())


def run_normals(pos, faces):
    cabi = _cabi()
    pos = np.asarray(pos, np.float32).reshape(-1, 3)
    faces = np.asarray(faces, np.int64).reshape(-1, 3)
    N, F = len(pos), len(faces)
    pos_d, f_d = _dev(pos), _dev(faces)
    ar = Arena()
    out = ar.out((N, 3), F32)
    st = ar.out((1,), torch.int32)
    ws, wsb = ar.ws(cabi.lib.dfw_vertex_normals_ws_bytes(F, N))
    _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_vertex_normals(_ptr(pos_d), N, _ptr(f_d), F, _ptr(out), st.data_ptr(),
                                                                                ws.data_ptr(), wsb, _stream())))
    ar.check("vertex_normals")
    assert_kernels("vertex_normals", names, ([r"\bk_incidence_expand\b"] if F else []) + ([r"\bk_vertex_normals\b"] if N else []),
                   ([] if F else [r"\bk_incidence_expand\b"]) + ([] if N else [r"\bk_vertex_normals\b"]))
    return out.cpu().numpy(), int(st.item())


def check_normals(name, pos, faces):
    n, st = run_normals(pos, faces)
    nr, st_r = normals_f32_oracle(pos, faces)
    assert st == st_r, f"{name}: status {st}, expected {st_r} skipped faces"
    assert_same(name, n, nr)
    record(f"data_path/vertex_normals/{name}", N=len(n), F=int(np.asarray(faces).size // 3), skipped=st, bit_mismatches=0,
           nonfinite=int((~np.isfinite(nr)).sum()))
    return n


# ---- stress metrics: reference and bounds ----------------------------------------------------------------------------
def met_grid(total):
    """dfw_stress_metrics' grid: (threads, terms per thread)."""
    blocks = max(1, min(-(-total // 1024), MAX_BLOCKS))
    return blocks * 256, max(1, -(-total // (blocks * 256)))


def metrics_ref(e, mask, C):
    """The 8 statistics in fp64 from the kernel's fp32 element errors e [N*C]; also (sum e, sum e^2) per subset."""
    out, sums = [], []
    for sel in (None, mask):
        ee = e if sel is None else e[np.repeat(np.asarray(sel, bool), C)]
        cnt = ee.size
        if cnt == 0:
            out += [0.0, 0.0, 0.0, 0.0]
            sums.append((0.0, 0.0))
            continue
        e64 = ee.astype(np.float64)
        s1, s2 = float(e64.sum()), float((e64 * e64).sum())
        out += [s1 / cnt, math.sqrt(s2 / cnt), float(ee.max()), float(cnt)]
        sums.append((s1, s2))
    return np.array(out), sums


def mae_bound(total, s1, cnt):
    """A per-thread fp32 chain of k terms (k - 1 roundings), then fp64 (tree over the threads, the reference's own
    pairwise sum, the division)."""
    T, k = met_grid(total)
    return (gamma(k - 1) * s1 + gamma(T + 64, UD) * s1) / cnt * (1 + 2 * UD) if cnt else 0.0


def rmse_bound(total, s2, cnt):
    """k fma roundings on sum e^2, then fp64; a relative error d of the sum is at most d/2 (1 + d) after the root."""
    if not cnt:
        return 0.0
    T, k = met_grid(total)
    d = gamma(k) + gamma(T + 64, UD)
    return math.sqrt(s2 / cnt) * (d / 2 * (1 + d) + 4 * UD)


def run_metrics(pred_d, targ_d, mask_d, N, C, log_scale):
    cabi = _cabi()
    dt = pred_d.dtype
    ar = Arena()
    res = ar.out((8,), torch.float64)
    ws, wsb = ar.ws(cabi.lib.dfw_stress_metrics_ws_bytes(N, C))
    _, names = launched_kernels(lambda: cabi.check(cabi.lib.dfw_stress_metrics(
        _ptr(pred_d), _ptr(targ_d), _ptr(mask_d), N, C, int(log_scale), cabi.DFW_F32 if dt == F32 else cabi.DFW_BF16, res.data_ptr(),
        ws.data_ptr(), wsb, _stream())))
    ar.check("stress_metrics")
    assert_kernels("stress_metrics", names, [re.escape("k_stress_metrics<float>" if dt == F32 else "k_stress_metrics<__nv_bfloat16>")])
    return res.cpu().numpy()


def device_errors(pred_d, targ_d, log_scale):
    """The kernel's fp32 element errors |p - t|, with torch.expm1 on the same device tensors when log_scale."""
    p, t = pred_d.float(), targ_d.float()
    if log_scale:
        p, t = torch.expm1(p), torch.expm1(t)
    return (p - t).abs().reshape(-1).cpu().numpy()


# ---- masked MSE: bounds ----------------------------------------------------------------------------------------------
def mse_grid(total):
    blocks = max(1, min(-(-total // 256), MAX_BLOCKS))
    return blocks, max(1, -(-total // (blocks * 256)))


def mse_loss_bound(total, s, cnt, mean):
    """k fma roundings per thread, 5 warp-shuffle and 7 block additions in fp32, an fp64 sum of the block partials and
    the division, then the fp32 store."""
    blocks, k = mse_grid(total)
    L = s / max(cnt, 1) if mean else s
    g = gamma(k + 12) + gamma(blocks + 64, UD)
    return L * (g + U * (1 + g))


# ---- CPU: the oracles and bounds themselves --------------------------------------------------------------------------
def _f32(v):
    return float(np.float32(v))


def test_features_oracle_is_numpy_and_correctly_rounded():
    """The restatement gives the bits of the reference's own numpy code and of one correctly rounded float32 operation per
    step (Python floats carry every fp32 +, -, *, /, sqrt exactly before the one rounding)."""
    rng = np.random.default_rng(0)
    pos, normal, stress, gp = _random_case(rng, 400)
    pos[:5, 2] = 7.0  # ties on the max
    x, y = features_oracle(pos, normal, stress, gp, [0, 400], True, True)
    mn, mx = pos.min(axis=0), pos.max(axis=0)
    rg = mx - mn
    rg[rg < 1e-8] = 1.0
    nl = np.linalg.norm(normal, axis=1, keepdims=True)
    nl[nl < 1e-8] = 1.0
    ref = np.concatenate([(pos - mn) / rg, normal / nl, np.tile(gp, (400, 1))], axis=1).astype(np.float32)
    assert_same("oracle/numpy", x, ref, zero_by_value=True)
    for i in range(0, 400, 7):
        for a in range(3):
            assert x[i, a] == _f32(_f32(float(pos[i, a]) - float(mn[a])) / _f32(float(mx[a]) - float(mn[a])))
        sq = _f32(_f32(_f32(float(normal[i, 0]) ** 2) + _f32(float(normal[i, 1]) ** 2)) + _f32(float(normal[i, 2]) ** 2))
        ln = _f32(math.sqrt(sq)) if sq else 0.0
        ln = ln if ln >= _f32(1e-8) else 1.0
        for a in range(3):
            assert x[i, 3 + a] == _f32(float(normal[i, a]) / ln)
        assert y[i, 0] == _f32(math.log1p(float(stress[i])))
    # the guards: a range below float32(1e-8) becomes 1; float32(1e-8) itself is kept (numpy 2 compares in float32)
    g = np.float32(1e-8)
    p = np.array([[0, 0, 0], [g, np.nextafter(g, np.float32(0)), np.nextafter(g, np.float32(1))]], np.float32)
    x, _ = features_oracle(p, np.ones((2, 3), np.float32), None, np.zeros(4), [0, 2], True, True)
    assert x[1, :3].tolist() == [1.0, _f32(np.nextafter(g, np.float32(0))), 1.0]
    # NaN poisons its axis of its case only; +-Inf give NaN on the infinite row and 0 elsewhere
    p = rng.standard_normal((6, 3)).astype(np.float32)
    p[1, 0], p[4, 1] = np.nan, np.inf
    x, _ = features_oracle(p, np.ones((6, 3), np.float32), None, np.zeros((2, 4)), [0, 3, 6], True, True)
    assert np.isnan(x[:3, 0]).all() and not np.isnan(x[3:, 0]).any() and np.isfinite(x[:3, 1:]).all()
    assert np.isnan(x[4, 1]) and (x[[3, 5], 1] == 0).all()


def test_normals_oracle_against_exact_rationals_and_a_scalar_loop():
    """Small-integer coordinates make every float32 step exact: the oracle equals the exact rational sum.  On random
    coordinates it equals a scalar loop that rounds each operation (Python float, then float32) in ascending incidence
    order, with repeated vertices, duplicated and invalid faces, and an isolated vertex."""
    rng = np.random.default_rng(1)
    pos = rng.integers(-50, 50, (12, 3)).astype(np.float32)
    faces = rng.integers(0, 11, (40, 3))  # vertex 11 is isolated
    n, st = normals_f32_oracle(pos, faces)
    exact = [[Fraction(0)] * 3 for _ in range(12)]
    for f in faces:
        p0, p1, p2 = (pos[i].astype(np.float64) for i in f)
        c = np.cross(p1 - p0, p2 - p0)
        for k in range(3):
            for a in range(3):
                exact[f[k]][a] += Fraction(c[a])
    assert st == 0 and n.tolist() == [[float(v) for v in r] for r in exact]
    assert n[11].view(np.uint32).tolist() == [0, 0, 0]

    pos = rng.standard_normal((30, 3)).astype(np.float32)
    faces = np.concatenate([rng.integers(0, 29, (200, 3)), [[0, 0, 5], [3, 3, 3], [1, 2, 30], [-1, 2, 3], [4, 5, 1 << 40]]])
    faces = np.concatenate([faces, faces[:20]])  # duplicated faces
    n, st = normals_f32_oracle(pos, faces)
    ref = np.zeros((30, 3), np.float32)
    for inc in range(3 * len(faces)):
        f = faces[inc // 3]
        if not ((f >= 0) & (f < 30)).all():
            continue
        o = [float(v) for v in pos[f[0]]]
        a = [_f32(float(pos[f[1]][c]) - o[c]) for c in range(3)]
        b = [_f32(float(pos[f[2]][c]) - o[c]) for c in range(3)]
        fn = [_f32(_f32(a[1] * b[2]) - _f32(a[2] * b[1])), _f32(_f32(a[2] * b[0]) - _f32(a[0] * b[2])),
              _f32(_f32(a[0] * b[1]) - _f32(a[1] * b[0]))]
        v = f[inc % 3]
        ref[v] = [_f32(float(ref[v][c]) + fn[c]) for c in range(3)]
    assert st == 3 and n.view(np.uint32).tolist() == ref.view(np.uint32).tolist()


def test_metrics_reference_and_bounds_reject_a_dropped_term():
    """Exact partials give the rational mean bit for bit; at 2M elements the mae, rmse and MSE-loss bounds each reject a
    sum that lost its largest term."""
    e = np.array([1, 2, 3, 0, 2], np.float32)
    r, _ = metrics_ref(e, np.array([1, 0, 1, 1, 0], bool), 1)
    assert r.tolist() == [1.6, math.sqrt(18 / 5), 3.0, 5.0, float(Fraction(4, 3)), math.sqrt(10 / 3), 3.0, 3.0]
    assert math.isnan(metrics_ref(np.float32([1, np.nan]), None, 1)[0][2])
    rng = np.random.default_rng(2)
    n = 2_000_003
    e = np.abs(rng.standard_normal(n)).astype(np.float64)
    s1, s2 = e.sum(), (e * e).sum()
    drop = e.max()
    assert abs(s1 / n - (s1 - drop) / n) > mae_bound(n, s1, n)
    assert abs(math.sqrt(s2 / n) - math.sqrt((s2 - drop * drop) / n)) > rmse_bound(n, s2, n)
    assert abs(s2 / n - (s2 - drop * drop) / n) > mse_loss_bound(n, s2, n, True)
    assert abs(s2 - (s2 - drop * drop)) > mse_loss_bound(n, s2, n, False)
    assert met_grid(606208) == (MAX_BLOCKS * 256, 4) and met_grid(606209) == (MAX_BLOCKS * 256, 5) and met_grid(1025) == (512, 3)
    assert ulp_distance(np.float32([1.0, np.inf, 0.0]), np.float32([np.nextafter(np.float32(1), np.float32(2)), np.inf, -0.0])) == 1


# ---- GPU: node features -----------------------------------------------------------------------------------------------
FEAT_N = [1, 2, 255, 256, 257, 151_551, 151_552, 151_553, 2_000_003]   # 151 552 = 148 * 4 blocks * 256 threads


@pytest.mark.gpu
@pytest.mark.parametrize("N", FEAT_N)
def test_node_features_bit_exact_at_size(N):
    rng = np.random.default_rng(N)
    pos, normal, stress, gp = _random_case(rng, N)
    worst = 0
    for normalize_pos in (True, False):
        for log_scale in (True, False):
            x, y = run_features(pos, normal, stress, gp, normalize_pos, log_scale)
            xr, yr = features_oracle(pos, normal, stress, gp, [0, N], normalize_pos, log_scale)
            worst = max(worst, check_features(f"features/N{N}/norm{int(normalize_pos)}/log{int(log_scale)}", x, y, xr, yr, log_scale))
        x0, y0 = run_features(pos, normal, None, gp, normalize_pos, True)
        assert y0 is None and x0.tobytes() == x.tobytes()  # stress = None: the same x
    record(f"data_path/node_features/N{N}", bit_mismatches=0, y_max_ulp=worst)


FEAT_CASES = [0, 1, 2, 16_383, 16_384, 16_385, 20_000, 300_001, 0, 7]   # 16 384 = 64 x-blocks * 256 threads


@pytest.mark.gpu
def test_node_features_batched_bit_exact_and_equal_to_per_case_calls():
    rng = np.random.default_rng(7)
    ptr = np.concatenate([[0], np.cumsum(FEAT_CASES)]).astype(np.int64)
    N, B = int(ptr[-1]), len(FEAT_CASES)
    pos, normal, stress, _ = _random_case(rng, N)
    gp = rng.uniform(-1, 1, (B, 4)).astype(np.float32)
    worst = 0
    for normalize_pos in (True, False):
        for log_scale in (True, False):
            xr, yr = features_oracle(pos, normal, stress, gp, ptr, normalize_pos, log_scale)
            runs = [run_features_batched(pos, normal, stress, gp, ptr, m, normalize_pos, log_scale) for m in (1, max(FEAT_CASES), 10 * max(FEAT_CASES))]
            for x, y in runs[1:]:  # max_case_rows only sizes the grid
                assert x.tobytes() == runs[0][0].tobytes() and y.tobytes() == runs[0][1].tobytes()
            x, y = runs[0]
            worst = max(worst, check_features(f"features_batched/norm{int(normalize_pos)}/log{int(log_scale)}", x, y, xr, yr, log_scale))
            for b in range(B):
                r0, r1 = ptr[b], ptr[b + 1]
                assert (x[r0:r1, 6:] == gp[b]).all(), f"case {b}: global parameters of another case"
                if r1 > r0:
                    xb, yb = run_features(pos[r0:r1], normal[r0:r1], stress[r0:r1], gp[b], normalize_pos, log_scale)
                    assert xb.tobytes() == x[r0:r1].tobytes() and yb.tobytes() == y[r0:r1].tobytes(), f"case {b} differs from its own call"
    record("data_path/node_features_batched/ragged", cases=B, rows=N, bit_mismatches=0, y_max_ulp=worst)


@pytest.mark.gpu
def test_node_features_batched_65535_one_row_cases():
    """The y-grid limit: every case one row, so its range is 0 (-> 1) and x[:3] = +0; its own global parameters."""
    rng = np.random.default_rng(8)
    B = 65_535
    ptr = np.arange(B + 1, dtype=np.int64)
    pos, normal, stress, _ = _random_case(rng, B)
    gp = rng.uniform(-1, 1, (B, 4)).astype(np.float32)
    x, y = run_features_batched(pos, normal, stress, gp, ptr, 1, True, True)
    xr, yr = features_oracle(pos, normal, stress, gp, ptr, True, True)
    d = check_features("features_batched/one_row", x, y, xr, yr, True)
    assert (x[:, :3] == 0).all() and (x[:, 6:] == gp).all()
    for b in list(range(0, B, 4099)) + [B - 1]:  # a sample of the per-case calls
        xb, yb = run_features(pos[b:b + 1], normal[b:b + 1], stress[b:b + 1], gp[b], True, True)
        assert xb.tobytes() == x[b:b + 1].tobytes() and yb.tobytes() == y[b:b + 1].tobytes()
    record("data_path/node_features_batched/65535_cases", bit_mismatches=0, y_max_ulp=d)


def _edge_cases():
    """(name, pos, normal, stress) cases, each its own min / max scope."""
    rng = np.random.default_rng(9)
    g = np.float32(1e-8)
    below, above = np.nextafter(g, np.float32(0)), np.nextafter(g, np.float32(1))
    cases = []

    def add(name, pos, normal=None, stress=None):
        n = len(pos)
        normal = rng.standard_normal((n, 3)).astype(np.float32) if normal is None else np.asarray(normal, np.float32)
        stress = rng.uniform(0, 1e7, n).astype(np.float32) if stress is None else np.asarray(stress, np.float32)
        cases.append((name, np.asarray(pos, np.float32), normal, stress))

    p = rng.standard_normal((300, 3)).astype(np.float32)
    p[:, 1] = 2.5
    add("constant_axis", p)
    p = np.zeros((5, 3), np.float32)
    p[1] = [g, below, above]
    p[2] = [g / 2, below / 3, above / 4]
    add("range_at_guard", p)
    p = np.zeros((4, 3), np.float32) + np.float32(-3.0)
    p[1] = [-3.0 + 2 ** -22, -3.0 + 2 ** -21, -3.0 + 2 ** -20]  # ranges of 1, 2 and 4 ulp of 3.0: far above 1e-8
    add("negative_tiny_range", p)
    add("negative", (rng.standard_normal((700, 3)) * 5 - 20).astype(np.float32))
    p = rng.uniform(0, 1, (9, 3)).astype(np.float32)
    p[:, 2] = [0.0, -0.0, 0.0, 0.5, -0.0, 0.0, 1.0, -0.0, 0.25]  # root plane at z = 0 with both signs
    add("signed_zero_root", p)
    s = np.float32(1e-8)
    nrm = np.array([[s, 0, 0], [below, 0, 0], [above, 0, 0], [0, -s, 0], [s / 2, s / 2, s / 2], [s, s, s], [0, 0, 0], [-0.0, 0, -0.0],
                    [1e-40, -1e-41, 3e-45], [1e-20, 1e-20, 0], [1e20, 1, 0], [-3e19, 3e19, 1e19], [1e19, 0, 0]], np.float32)
    add("normal_guard_and_overflow", rng.standard_normal((len(nrm), 3)).astype(np.float32), nrm)
    for what, v in (("nan", np.nan), ("pinf", np.inf), ("ninf", -np.inf)):
        p = rng.standard_normal((40, 3)).astype(np.float32)
        p[17, 0] = v
        p[3, 2] = v
        nrm = rng.standard_normal((40, 3)).astype(np.float32)
        nrm[5, 1] = v
        st = rng.uniform(0, 1e7, 40).astype(np.float32)
        st[9] = v
        add(f"{what}_in_pos_normal_stress", p, nrm, st)
    add("stress_minus_one", rng.standard_normal((6, 3)), stress=[-1.0, -1.5, -0.999999, -3e38, 0.0, -0.0])
    add("empty_between", np.zeros((0, 3)))
    add("single_nan_row", np.float32([[np.nan, 1.0, -0.0]]))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("log_scale", [True, False])
@pytest.mark.parametrize("normalize_pos", [True, False])
def test_node_features_edge_values(normalize_pos, log_scale):
    """Guards at and around 1e-8 (range and |n|), constant axes, signed zeros, subnormal and overflowing normals, NaN and
    +-Inf in pos / normal / stress, stress <= -1 - each case in both forms; the guards' pattern is pinned too."""
    cases = _edge_cases()
    pos = np.concatenate([c[1] for c in cases])
    normal = np.concatenate([c[2] for c in cases])
    stress = np.concatenate([c[3] for c in cases])
    ptr = np.concatenate([[0], np.cumsum([len(c[1]) for c in cases])]).astype(np.int64)
    gp = np.arange(4 * len(cases), dtype=np.float32).reshape(-1, 4) / 7
    xr, yr = features_oracle(pos, normal, stress, gp, ptr, normalize_pos, log_scale)
    x, y = run_features_batched(pos, normal, stress, gp, ptr, int(np.diff(ptr).max()), normalize_pos, log_scale)
    d = check_features("features_edge/batched", x, y, xr, yr, log_scale)
    for b, (name, p, n, s) in enumerate(cases):
        if not len(p):
            continue
        xb, yb = run_features(p, n, s, gp[b], normalize_pos, log_scale)
        xo, yo = features_oracle(p, n, s, gp[b], [0, len(p)], normalize_pos, log_scale)
        d = max(d, check_features(f"features_edge/{name}", xb, yb, xo, yo, log_scale))
        assert_same(f"features_edge/{name}/forms", xb, x[ptr[b]:ptr[b + 1]], zero_by_value=True)
    by = {c[0]: ptr[i] for i, c in enumerate(cases)}
    if normalize_pos:
        r = by["range_at_guard"] + 1  # range float32(1e-8) kept, one ulp below -> 1, one ulp above kept
        assert x[r, :3].tolist() == [1.0, float(np.nextafter(np.float32(1e-8), np.float32(0))), 1.0]
        r = by["nan_in_pos_normal_stress"]
        assert np.isnan(x[r:r + 40, 0]).all() and np.isnan(x[r:r + 40, 2]).all() and not np.isnan(x[r:r + 40, 1]).any()
        assert np.isnan(x[by["single_nan_row"], 0]) and x[by["single_nan_row"], 1] == 0
    r = by["normal_guard_and_overflow"]
    assert (x[r + 10, 3:6] == 0).all() and (x[r + 11, 3:6] == 0).all()  # squares overflow: |n| = inf
    assert x[r + 8, 3:6].tolist() == [float(np.float32(v)) for v in (1e-40, -1e-41, 3e-45)]  # subnormal: |n| = 0 -> 1
    if log_scale:
        r = by["stress_minus_one"]
        assert y[r, 0] == -np.inf and np.isnan(y[r + 1, 0]) and np.isnan(y[r + 3, 0])
    record(f"data_path/node_features/edges/norm{int(normalize_pos)}/log{int(log_scale)}", cases=len(cases), bit_mismatches=0, y_max_ulp=d)


# ---- GPU: vertex normals ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["native", "random"])
def test_vertex_normals_bit_exact_on_wings(order):
    from deep_fem_uav_wing.gnn import synth

    mesh = synth.surface_tri_wing(20000, seed=11, node_order=order)
    check_normals(f"wing_{order}", mesh["pos"], mesh["faces"])


@pytest.mark.gpu
def test_vertex_normals_fan_of_degree_70000():
    n = 70_001
    t = np.linspace(0, 2 * np.pi, n, endpoint=False)
    pos = np.concatenate([[[0.1, -0.2, 0.3]], np.stack([np.cos(t), np.sin(t), 0.01 * np.sin(7 * t)], 1)]).astype(np.float32)
    faces = np.stack([np.zeros(n - 1, np.int64), np.arange(1, n), np.arange(2, n + 1)], 1)
    normal = check_normals("fan_70000", pos, faces)
    assert np.isfinite(normal).all()


@pytest.mark.gpu
def test_vertex_normals_degenerate_duplicated_isolated_and_invalid_faces():
    from deep_fem_uav_wing.gnn import synth

    mesh = synth.surface_tri_wing(3000, seed=13, node_order="random")
    pos = np.concatenate([mesh["pos"], np.float32([[5, 5, 5], [6, 6, 6]])])  # two isolated vertices at the end
    N = len(pos)
    f = mesh["faces"].astype(np.int64)
    rep = np.array([[0, 0, 1], [2, 3, 3], [4, 5, 4], [6, 6, 6]], np.int64)
    f = np.concatenate([f[:500], rep, f[:50], f[500:], f[-30:]])  # repeated vertices, duplicated faces
    isolated = np.setdiff1d(np.arange(N), f)
    n = check_normals("degenerate_duplicated", pos, f)
    assert len(isolated) >= 2 and (n[isolated].view(np.uint32) == 0).all()  # exactly +0
    bad = [[-1, 1, 2], [0, N, 2], [0, 1, 1 << 40], [-(1 << 40), 0, 1], [N + 5, N + 6, N + 7]]
    for where in ("start", "middle", "end"):
        i = {"start": 0, "middle": len(f) // 2, "end": len(f)}[where]
        fb = np.concatenate([f[:i], bad, f[i:]])
        nb = check_normals(f"invalid_{where}", pos, fb)
        assert nb.tobytes() == n.tobytes()


@pytest.mark.gpu
def test_vertex_normals_empty_tiny_nonfinite_and_overflowing():
    rng = np.random.default_rng(14)
    check_normals("F0", rng.standard_normal((10, 3)), np.zeros((0, 3)))
    check_normals("N0_F0", np.zeros((0, 3)), np.zeros((0, 3)))
    check_normals("N0_F2", np.zeros((0, 3)), [[0, 0, 0], [1, 2, 3]])
    check_normals("N1", [[1.0, 2.0, 3.0]], [[0, 0, 0]])
    check_normals("N1_F0", [[1.0, 2.0, 3.0]], np.zeros((0, 3)))
    from deep_fem_uav_wing.gnn import synth

    mesh = synth.surface_tri_wing(2000, seed=15)
    pos = mesh["pos"].copy()
    pos[[3, 400, 1500], [0, 1, 2]] = [np.nan, np.inf, -np.inf]
    n = check_normals("nonfinite_pos", pos, mesh["faces"])
    assert (~np.isfinite(n)).any()
    pos = rng.uniform(-3e19, 3e19, (200, 3)).astype(np.float32)
    n = check_normals("coords_1e19", pos, rng.integers(0, 200, (400, 3)))
    assert (~np.isfinite(n)).any()  # products overflow


# ---- GPU: stress metrics ----------------------------------------------------------------------------------------------
MET_TOTALS = [0, 1, 1023, 1024, 1025, 606_207, 606_208, 606_209, 2_000_003, 20_000_003]   # 606 208 = 592 blocks * 1024
MET_SHAPES = sorted({(-(-t // c), c) for t in MET_TOTALS for c in (1, 3)})


def _met_masks(rng, N):
    m = {"none": None, "all_false": np.zeros(N, bool), "all_true": np.ones(N, bool), "random30": rng.random(N) < 0.3,
         "last_row": np.zeros(N, bool)}
    if N:
        m["last_row"][-1] = True
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [F32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("N,C", MET_SHAPES, ids=[f"N{n}xC{c}" for n, c in MET_SHAPES])
def test_stress_metrics_exact_and_bounded(N, C, dt):
    rng = np.random.default_rng(N * 3 + C)
    total = N * C
    # exact arithmetic: integer targets, |p - t| in {0..3}; every fp32 partial is an integer below 2^24
    t_int = rng.integers(-100, 101, (N, C)).astype(np.float32)
    d_int = rng.integers(-3, 4, (N, C)).astype(np.float32)
    exact = (_dev(t_int + d_int).to(dt), _dev(t_int).to(dt))
    # random: log-stress scale as the model predicts it
    tr = rng.standard_normal((N, C)).astype(np.float32) * 2 + 8
    rnd = (_dev(tr + rng.standard_normal((N, C)).astype(np.float32) * 0.3).to(dt), _dev(tr).to(dt))
    margins = {"mae": 0.0, "rmse": 0.0}
    for mname, m in _met_masks(rng, N).items():
        m_d = _dev(m.astype(np.uint8)) if m is not None else None
        got = run_metrics(*exact, m_d, N, C, False)
        ref, _ = metrics_ref(device_errors(*exact, False), m, C)
        assert got.tolist() == ref.tolist(), f"exact/{mname}: got {got.tolist()}, expected {ref.tolist()}"
        for log_scale in (False, True):
            e = device_errors(*rnd, log_scale)
            got = run_metrics(*rnd, m_d, N, C, log_scale)
            ref, sums = metrics_ref(e, m, C)
            for s in range(2):
                row = f"random/log{int(log_scale)}/{mname}/{('all', 'masked')[s]}"
                assert got[4 * s + 2] == ref[4 * s + 2] and got[4 * s + 3] == ref[4 * s + 3], f"{row}: max/count {got[4*s+2:4*s+4]} vs {ref[4*s+2:4*s+4]}"
                cnt = ref[4 * s + 3]
                for k, bound in ((0, mae_bound(total, sums[s][0], cnt)), (1, rmse_bound(total, sums[s][1], cnt))):
                    err = abs(got[4 * s + k] - ref[4 * s + k])
                    assert err <= bound, f"{row}/{('mae', 'rmse')[k]}: |{got[4*s+k]!r} - {ref[4*s+k]!r}| = {err:.3g} > bound {bound:.3g}"
                    if bound:
                        key = ("mae", "rmse")[k]
                        margins[key] = max(margins[key], err / bound)
    record(f"data_path/stress_metrics/{'f32' if dt == F32 else 'bf16'}/N{N}xC{C}", total=total, terms_per_thread=met_grid(total)[1],
           exact_mismatches=0, mae_err_over_bound=margins["mae"], rmse_err_over_bound=margins["rmse"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [F32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("C", [1, 3])
def test_stress_metrics_nonfinite(C, dt):
    """A NaN error anywhere (first, middle, last block) makes mae, rmse and max_error of its subset NaN; +-Inf gives Inf;
    Inf - Inf gives NaN; a NaN in a masked-out row leaves the masked statistics exactly as without it."""
    N = 606_209 // C + 1
    rng = np.random.default_rng(20 + C)
    t = rng.integers(-100, 101, (N, C)).astype(np.float32)
    p = t + rng.integers(-3, 4, (N, C)).astype(np.float32)
    mask = rng.random(N) < 0.5
    mask[[0, N // 2, N - 1]] = True
    off = np.flatnonzero(~mask)[[0, -1]]
    m_d = _dev(mask.astype(np.uint8))
    clean = run_metrics(_dev(p).to(dt), _dev(t).to(dt), m_d, N, C, False)
    assert np.isfinite(clean).all()
    for row in (0, N // 2, N - 1):  # selected rows
        for what, pv, tv, expect in (("nan_pred", np.nan, None, "nan"), ("nan_target", None, np.nan, "nan"), ("pinf", np.inf, None, "inf"),
                                     ("ninf_target", None, -np.inf, "inf"), ("inf_minus_inf", np.inf, np.inf, "nan")):
            pp, tt = p.copy(), t.copy()
            if pv is not None:
                pp[row, C - 1] = pv
            if tv is not None:
                tt[row, C - 1] = tv
            got = run_metrics(_dev(pp).to(dt), _dev(tt).to(dt), m_d, N, C, False)
            for s in range(2):
                v = got[4 * s:4 * s + 3]
                assert (np.isnan(v).all() if expect == "nan" else np.isposinf(v).all()), f"{what}/row{row}/{s}: {got.tolist()}"
                assert got[4 * s + 3] == clean[4 * s + 3]
    for row in off:  # masked-out rows: the masked half is untouched
        pp = p.copy()
        pp[row, 0] = np.nan
        got = run_metrics(_dev(pp).to(dt), _dev(t).to(dt), m_d, N, C, False)
        assert np.isnan(got[:3]).all() and got[3] == clean[3]
        assert got[4:].tolist() == clean[4:].tolist()
    record(f"data_path/stress_metrics/nonfinite/{'f32' if dt == F32 else 'bf16'}/C{C}", N=N, passed=1)


@pytest.mark.gpu
@pytest.mark.parametrize("log_scale", [True, False])
def test_stress_metrics_bf16_prediction_keeps_the_fp32_target(log_scale):
    """A bf16 prediction with an fp32 target gives the same 8 doubles as pred.float() with that target: the target is not
    rounded to bf16 (an error of up to 2^-8 relative in log space)."""
    from deep_fem_uav_wing.gnn import ops

    rng = np.random.default_rng(31)
    N = 200_003
    t = _dev((rng.standard_normal((N, 1)) * 2 + 12).astype(np.float32))
    p = (t + 0.05 * torch.randn_like(t)).to(BF16)
    m = _dev(rng.random(N) < 0.4)
    a = ops.stress_metrics(p, t, m, log_scale=log_scale).cpu()
    b = ops.stress_metrics(p.float(), t, m, log_scale=log_scale).cpu()
    assert a.tolist() == b.tolist(), f"{a.tolist()} != {b.tolist()}"


# ---- GPU: masked MSE fp32 ---------------------------------------------------------------------------------------------
MSE_N = [0, 1, 255, 256, 257, 151_553, 2_000_003, 20_000_003]


def run_mse(pred_d, targ_d, mask_d, N, C, mean):
    cabi = _cabi()
    ar = Arena()
    res = ar.out((2,), F32)
    gp = ar.out((N, C), F32)
    ws, wsb = ar.ws(cabi.lib.dfw_masked_mse_ws_bytes(N, C))
    gl = torch.tensor([G_LOSS], device="cuda")

    def call():
        cabi.check(cabi.lib.dfw_masked_mse_fwd(_ptr(pred_d), _ptr(targ_d), _ptr(mask_d), N, C, int(mean), cabi.DFW_F32, res.data_ptr(),
                                               ws.data_ptr(), wsb, _stream()))
        cabi.check(cabi.lib.dfw_masked_mse_bwd(_ptr(pred_d), _ptr(targ_d), _ptr(mask_d), res.data_ptr(), gl.data_ptr(), N, C, int(mean),
                                               cabi.DFW_F32, gp.data_ptr(), _stream()))

    _, names = launched_kernels(call)
    ar.check("masked_mse")
    assert_kernels("masked_mse", names, [re.escape("k_mse_fwd<float>")] + ([re.escape("k_mse_bwd<float>")] if N else []),
                   [] if N else [r"\bk_mse_bwd\b"])
    return res.cpu().numpy(), gp.cpu().numpy()


def check_mse(row, p, t, mask, C, mean, exact, res, g):
    """Returns (loss err/bound, gradient err/bound)."""
    sel = np.ones(p.shape[0], bool) if mask is None else mask
    d = p.astype(np.float64) - t.astype(np.float64)  # exact: the kernel's fp32 p - t is this value rounded once
    s = float(((p - t)[sel].astype(np.float64) ** 2).sum())
    cnt = int(sel.sum()) * C
    assert res[1] == np.float32(cnt), f"{row}: count {res[1]!r}, expected float32({cnt})"
    if cnt <= 2 ** 24:
        assert float(res[1]) == cnt
    loss_ref = s / max(cnt, 1) if mean else s
    if exact:
        assert res[0] == np.float32(loss_ref), f"{row}: loss {res[0]!r}, expected float32({loss_ref!r})"
        m_loss = 0.0
    else:
        err, bound = abs(float(res[0]) - loss_ref), mse_loss_bound(p.size, s, cnt, mean)
        assert err <= bound, f"{row}: loss {res[0]!r}, fp64 {loss_ref!r}, err {err:.3g} > bound {bound:.3g}"
        m_loss = err / bound if bound else 0.0
    # gradient: 2 g (p - t) / count with the fp32 count the forward reported; three roundings (divide, subtract, multiply)
    div = max(float(res[1]), 1.0) if mean else 1.0
    gref = 2.0 * G_LOSS * d / div
    gref[~sel] = 0.0
    err = np.abs(g.astype(np.float64) - gref)
    bound = ((1 + U) ** 3 - 1) * np.abs(gref) + 2.0 ** -149
    bad = ~(err <= bound)
    assert not bad.any(), f"{row}: {int(bad.sum())} gradient elements outside 3 roundings, first {np.argwhere(bad)[0].tolist()}"
    assert (g[~sel].view(np.uint32) == 0).all(), f"{row}: a masked-out gradient is not +0"
    return m_loss, float((err / bound).max()) if err.size else 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("mean", [True, False], ids=["mean", "sum"])
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("N", MSE_N)
def test_masked_mse_fp32_exact_and_bounded(N, C, mean):
    rng = np.random.default_rng(N + 7 * C + int(mean))
    t_int = rng.integers(-1000, 1001, (N, C)).astype(np.float32)
    p_int = t_int + rng.integers(-3, 4, (N, C)).astype(np.float32)
    t_r = rng.standard_normal((N, C), dtype=np.float32)
    p_r = t_r + rng.standard_normal((N, C), dtype=np.float32) * np.float32(0.5)
    worst = [0.0, 0.0]
    for mname, mask in (("none", None), ("random30", rng.random(N) < 0.3)):
        m_d = _dev(mask.astype(np.uint8)) if mask is not None else None
        for exact, (p, t) in ((True, (p_int, t_int)), (False, (p_r, t_r))):
            res, g = run_mse(_dev(p), _dev(t), m_d, N, C, mean)
            a, b = check_mse(f"mse/N{N}xC{C}/{'mean' if mean else 'sum'}/{mname}/{'exact' if exact else 'random'}", p, t, mask, C, mean, exact, res, g)
            worst = [max(worst[0], a), max(worst[1], b)]
    record(f"data_path/masked_mse/N{N}xC{C}/{'mean' if mean else 'sum'}", loss_err_over_bound=worst[0], grad_err_over_bound=worst[1],
           terms_per_thread=mse_grid(N * C)[1])


@pytest.mark.gpu
@pytest.mark.parametrize("mean", [True, False], ids=["mean", "sum"])
def test_masked_mse_fp32_nonfinite(mean):
    """NaN or Inf in masked-out rows changes neither the loss nor any gradient; in a selected row the loss is NaN."""
    N, C = 151_553, 3
    rng = np.random.default_rng(40)
    t = rng.standard_normal((N, C), dtype=np.float32)
    p = t + rng.standard_normal((N, C), dtype=np.float32)
    mask = rng.random(N) < 0.5
    m_d = _dev(mask.astype(np.uint8))
    res0, g0 = run_mse(_dev(p), _dev(t), m_d, N, C, mean)
    off, on = np.flatnonzero(~mask), np.flatnonzero(mask)
    pp, tt = p.copy(), t.copy()
    pp[off[:3], 0], tt[off[3:6], 1], pp[off[-1], C - 1], tt[off[-1], C - 1] = np.nan, np.inf, np.inf, np.inf
    res, g = run_mse(_dev(pp), _dev(tt), m_d, N, C, mean)
    assert res.tobytes() == res0.tobytes() and g.tobytes() == g0.tobytes()
    for v in (np.nan, np.inf):
        pp = p.copy()
        pp[on[len(on) // 2], 1] = v
        res, _ = run_mse(_dev(pp), _dev(t), m_d, N, C, mean)
        assert (np.isnan(res[0]) if v != v else np.isinf(res[0])) and res[1] == res0[1]


@pytest.mark.gpu
@pytest.mark.parametrize("reduction", ["mean", "sum"])
def test_masked_mse_empty_batch_backward(reduction):
    """An empty prediction has a null data pointer; its backward is a no-op, not an argument error."""
    from deep_fem_uav_wing.gnn.model import MaskedMSELoss

    pred = torch.zeros(0, 1, device="cuda", requires_grad=True)
    loss = MaskedMSELoss(reduction)(pred, torch.zeros(0, 1, device="cuda"), torch.zeros(0, dtype=torch.bool, device="cuda"))
    loss.backward()
    assert loss.item() == 0.0 and pred.grad is not None and pred.grad.shape == (0, 1)
