"""The glue between the kernels, checked stage by stage against fp64: every autograd Function of ``gnn/ops.py`` the model runs
(``SageConvFn``, ``LinearFn``, ``DecoderTailFn``, ``CastFn``, ``MaskedMSEFn``) and the one-call C entry points of
``csrc/dfw_layer.cu``.

Replay.  A training (or sensitivity) step of ``GraphSAGEModel`` runs with the five Functions' ``forward`` / ``backward``
wrapped.  Each call records what its kernels read - the compute-dtype weight copies and the ``agg``, ``pre``, ``stats``,
``act`` / ``hid`` tensors from ``ctx.saved_tensors`` - its outputs, the incoming gradient, the returned gradients and the
``g_y`` its epilogue backward produced.  Each stage is then restated in fp64 from the RECORDED inputs, so an error cannot
propagate from one layer to the next, and ReLU / dropout masks come from the kernel's own saved tensors and from
``oracle.sage_oracle.dropout_keep_scale``.  With u = 2^-24 the bounds are those of ``test_gpu_linear_bounds.py``:

  agg                        bit for bit against the gather oracle (a training step never takes the block aggregation)
  pre, stats, out, hid, row  fwd_reference (K-term fp32 reductions, LayerNorm propagation, bf16 stores)
  g_y of the SAGE tail       rstd (gh - mean(gh) - xh mean(gh xh)) with gh = g_out keep m gamma, short_bound over H terms;
                             an element whose z = xh gamma + beta lies within 2^-16 (|gamma xh| + |beta|) of 0 may take
                             either ReLU branch in fp32: it enters with m = 1/2 and its half-term d_j = |g_out keep gamma|/2
                             widens the row by rstd (d_i + (sum_j d_j + |xh_i| sum_j |xh_j| d_j) / H)
  g_y of ReLU / row dot      one product, mask from the saved activation (exact)
  dW, db, dgamma, ...        long_check (2^-16 S per element, rel_l2 within 4x CPU fp32)
  loss, g_pred               one long reduction / one product, from the unrounded target

The input gradient of a SAGE layer, g_x = (A^T D^-1 g_y) W_l + g_y W_r (+ g_out), is computed as the gather
t~ = aggregate_scaled(A^T, inv_deg[src], g_y) followed by one two-operand linear with the residual epilogue.  With the
source-side degree deg_t of a row and S_t = A^T D^-1 |g_y|, the gather adds deg_t terms in fp32 and may store bf16:

  |t~ - t| <= E_t = (deg_t + 8) 2u S_t  (+ 2^-8 (|t| + that) in bf16)

The linear then computes the exact product of what it read, t~ W_l + g_y W_r + g_out, to within a short-reduction bound
over 2H + 1 terms of S~ = |t~| |W_l| + |g_y| |W_r| + |g_out| <= S + E_t |W_l|, and |t~ W_l - t W_l| <= E_t |W_l|, so

  |g_x - r| <= (2H + 9) 2u (S + E_t |W_l|) + E_t |W_l|     (+ 2^-8 (|r| + that) for the bf16 store of g_x)

t is restated from the CSR by destination (``index_add`` over the edges), not from the transposed CSR the kernel read, so
the transpose build is checked on the way.  Every gradient is also bit-identical with and without the side-stream weight
gradient (``ops.OVERLAP_DW``) and across two runs.

One-call entry points.  ``dfw_sage_layer_fwd/bwd``, ``dfw_mlp2_fwd/bwd`` and ``dfw_graphsage_forward`` run through the raw C
ABI with every output and the workspace inside ``helpers.Arena`` guard bands; each case returns 0, equals the autograd path
bit for bit, writes nothing outside its ranges, succeeds with exactly the queried workspace and is refused with one byte less.

tests/test_gpu_linear_variants.py re-runs this file with the classic tensor-core linear and with every linear on SIMT."""
import os
import re
import zlib

import numpy as np
import pytest
import torch

from helpers import Arena, assert_bound, assert_no_rounding_bias, launched_kernels, record, rounding_bias
from test_gpu_linear_bounds import fwd_reference, long_check, short_bound, tc_dw_chain_bound

U = 2.0 ** -24
F32, BF16 = torch.float32, torch.bfloat16
SIMT = os.environ.get("DFW_FORCE_SIMT", "0")[:1] not in ("", "0")
_WEIGHT_GRAD_KERNELS = r"k_dw_|smallk_dw|k_colsum|k_epilogue_bwd_reduce"


def _seed(name):
    return zlib.crc32(name.encode()) & 0x7FFFFFFF


def keep_of(seed, N, H, p, device):
    """fp64 dropout factors (1/(1-p) or 0) the kernels draw for `seed`; all ones without dropout."""
    if not p:
        return torch.ones(N, H, dtype=torch.float64, device=device)
    from oracle.sage_oracle import dropout_keep_scale

    return torch.from_numpy(dropout_keep_scale(int(seed), N, H, p)).to(device).double()


def _bf16_store(r, E, bf16):
    return E + (2.0 ** -8 * (r.abs() + E) if bf16 else 0.0)


def no_store_bias(name, got, r, pre_store_bound):
    """The rounding-bias check of a bf16 store over the nonzero results (ReLU and dropout zeros carry no rounding); asserted
    where at least 20 000 elements qualify (the mean of 20 000 RNE errors has a standard deviation of 0.002 ulp)."""
    nz = r != 0
    bias, n = rounding_bias(got[nz], r[nz], pre_store_bound[nz])
    if n >= 20_000:
        assert abs(bias) < 0.05, f"{name}: mean signed bf16 store error {bias:+.4f} ulp over {n} elements (truncation gives -0.5)"
    return bias


def fwd_checks(name, got, ref, bf16):
    """got: {"pre", "out", "stats"} of a forward against fwd_reference's bounds."""
    m = {}
    for key in ("pre", "out"):
        if got.get(key) is not None:
            r, b, pre_store = ref[key]
            m[key] = assert_bound(f"{name}/{key}", got[key], r, b)
            if bf16:
                m[key + "_bias_ulp"] = no_store_bias(f"{name}/{key}", got[key], r, pre_store)
    if got.get("stats") is not None:
        m["mean"] = assert_bound(f"{name}/mean", got["stats"][:, 0], *ref["mean"])
        m["rstd"] = assert_bound(f"{name}/rstd", got["stats"][:, 1], *ref["rstd"])
    return m


def _long(name, got, a, b, dw_chain=None):
    """long_check of got = a^T b (a sum over nodes)."""
    r = a.double().T @ b.double()
    S = a.double().abs().T @ b.double().abs()
    cpu = a.float().cpu().T @ b.float().cpu()
    return long_check(name, got, r, S, cpu, chain_bound=dw_chain)[0]


def _colsum(name, got, r_rows, S_rows, cpu_rows, extra=None):
    chain = extra if (extra is not None and bool((extra > 0).any())) else None
    if chain is not None:  # an undecidable ReLU branch moves the sum by up to `extra`: widen the tensor-wide limit by twice that
        chain = 2 * chain + 4 * (cpu_rows.sum(0).to(r_rows.device).double() - r_rows.sum(0)).abs()
    return long_check(name, got, r_rows.sum(0), S_rows.sum(0), cpu_rows.sum(0), extra=extra, chain_bound=chain)[0]


def _dw_chain(g, a, Hout, k1, k2, dtype):
    """The tensor-core dW's own accumulation chain (test_gpu_linear_bounds.tc_dw_chain_bound) where that kernel runs."""
    e = 4 if dtype == F32 else 2
    if SIMT or Hout % 16 or (k1 * e) % 16 or (k2 * e) % 16 or k1 < 16:
        return None
    return tc_dw_chain_bound(g, a, Hout, k1, k2, dtype == F32)


# ---- fp64 restatements of each stage (device-agnostic: the CPU unit tests below run them on planted faults) -----------
def ln_tail_grad(pre, stats, gamma, beta, g_out, keep, dtype=torch.float64, mask=None):
    """g_y of LayerNorm -> ReLU -> dropout from the saved pre / stats, in `dtype`.  Returns (g_y, gg0, xh, mask, S_gy, amb)."""
    st = stats.to(dtype)
    mean, rstd = st[:, :1], st[:, 1:]
    g, b = gamma.to(dtype), beta.to(dtype)
    xh = (pre.to(dtype) - mean) * rstd
    amb = None
    if mask is None:
        z = xh * g + b
        amb = z.abs() < 2.0 ** -16 * ((g * xh).abs() + b.abs())
        mask = torch.where(amb, 0.5, (z > 0).to(dtype)).to(dtype)
    gg0 = g_out.to(dtype) * keep.to(dtype) * mask
    gh = gg0 * g
    gy = rstd * (gh - gh.mean(1, keepdim=True) - xh * (gh * xh).mean(1, keepdim=True))
    S = rstd * (gh.abs() + gh.abs().mean(1, keepdim=True) + xh.abs() * (gh * xh).abs().mean(1, keepdim=True))
    return gy, gg0, xh, mask, S, amb


def source_gather(graph, v, inv_deg):
    """t = A^T D^-1 v restated from the CSR by destination: t[src] += inv_deg[dst] v[dst]; also returns the source degrees."""
    rowptr, col = graph["rowptr"].long(), graph["col"].long()
    N = rowptr.numel() - 1
    E = int(rowptr[-1])
    dst = torch.repeat_interleave(torch.arange(N, device=v.device), rowptr[1:] - rowptr[:-1], output_size=E)
    src = col[:E].to(v.device)
    t = torch.zeros(N, v.shape[1], dtype=torch.float64, device=v.device)
    t.index_add_(0, src, inv_deg.double()[dst, None] * v.double()[dst])
    deg_t = torch.bincount(src, minlength=N).double()[:, None]
    return t, deg_t


def check_sage_bwd(name, rec):
    """One SageConvFn.backward with the fused tail.  `rec`: saved (x, agg, pre, stats, wl, wr, gamma, beta), graph
    {rowptr, col, inv_deg}, p, seed, g_out, g_y (what the epilogue produced), grads (g_x, dwl, dbl, dwr, dgamma, dbeta)."""
    x, agg, pre, stats, wl, wr, gamma, beta = rec["saved"]
    g_out, gy_k = rec["g_out"], rec["g_y"]
    g_x, dwl, dbl, dwr, dgamma, dbeta = rec["grads"][:6]
    N, H = g_out.shape
    dt = g_out.dtype
    bf16 = dt == BF16
    keep = keep_of(rec["seed"], N, H, rec["p"], g_out.device)
    gy, gg0, xh, mask, S_gy, amb = ln_tail_grad(pre, stats, gamma, beta, g_out, keep)
    rstd = stats.double()[:, 1:]
    d = torch.where(amb, 0.5 * (g_out.double() * keep * gamma.double()).abs(), 0.0)
    slack = rstd * (d + (d.sum(1, keepdim=True) + xh.abs() * (xh.abs() * d).sum(1, keepdim=True)) / H)
    Ef = short_bound(S_gy, H) + slack
    m = {"g_y": assert_bound(f"{name}/g_y", gy_k, gy, _bf16_store(gy, Ef, bf16)), "ambiguous_relu": int(amb.sum())}
    if bf16:
        m["g_y_bias_ulp"] = no_store_bias(f"{name}/g_y", gy_k, gy, Ef)
    want_params = dwl is not None
    if want_params:
        gy32, gg32, xh32, _, _, _ = ln_tail_grad(pre.float().cpu(), stats.cpu(), gamma.cpu(), beta.cpu(), g_out.float().cpu(),
                                                 keep.float().cpu(), torch.float32, mask.float().cpu())
        dg = torch.where(amb, 0.5 * (g_out.double() * keep).abs(), 0.0)
        m["dgamma"] = _colsum(f"{name}/dgamma", dgamma, gg0 * xh, (gg0 * xh).abs() * (1 + 4 * U), gg32 * xh32,
                              extra=(dg * xh.abs()).sum(0))
        m["dbeta"] = _colsum(f"{name}/dbeta", dbeta, gg0, gg0.abs(), gg32, extra=dg.sum(0))
        if dbl is not None:
            m["db_l"] = _colsum(f"{name}/db_l", dbl, gy, S_gy + Ef, gy32, extra=slack.sum(0))
        m["dW_l"] = _long(f"{name}/dW_l", dwl, gy_k, agg, _dw_chain(gy_k, agg, H, H, H, dt))
        m["dW_r"] = _long(f"{name}/dW_r", dwr, gy_k, x, _dw_chain(gy_k, x, H, H, H, dt))
    t, deg_t = source_gather(rec["graph"], gy_k, rec["graph"]["inv_deg"])
    St, _ = source_gather(rec["graph"], gy_k.abs(), rec["graph"]["inv_deg"])
    Et = _bf16_store(t, short_bound(St, deg_t), bf16)
    wl64, wr64 = wl.double(), wr.double()
    r = t @ wl64 + gy_k.double() @ wr64 + g_out.double()
    S = t.abs() @ wl64.abs() + gy_k.double().abs() @ wr64.abs() + g_out.double().abs()
    Etw = Et @ wl64.abs()
    Ex = short_bound(S + Etw, 2 * H + 1) + Etw
    m["g_x"] = assert_bound(f"{name}/g_x", g_x, r, _bf16_store(r, Ex, bf16))
    return m


def check_mse(name, pred, target, mask, mean, loss, count, g_loss, g_pred):
    """Masked MSE against fp64 on the unrounded inputs: the loss is one long reduction, the gradient one product."""
    p64, t64 = pred.double(), target.double().reshape(pred.shape)
    C = p64.numel() // max(p64.shape[0], 1)
    mk = torch.ones(p64.shape[0], dtype=torch.float64, device=p64.device) if mask is None else mask.reshape(-1).double()
    d = (p64 - t64).reshape(p64.shape[0], -1)
    cnt = float(mk.sum()) * C
    assert float(count) == cnt, f"{name}: count {float(count)} != {cnt}"
    div = max(cnt, 1.0) if mean else 1.0
    r_loss = ((d * d) * mk[:, None]).sum() / div
    cpu = (((pred.float().cpu() - target.float().cpu().reshape(pred.shape)).reshape(d.shape) ** 2) * mk.float().cpu()[:, None]).sum() / div
    m = {"loss": long_check(f"{name}/loss", loss.reshape(1), r_loss.reshape(1), r_loss.reshape(1), cpu.reshape(1))[0]}
    if g_pred is not None:
        r_g = 2 * float(g_loss) * d * mk[:, None] / div
        Ef = short_bound(r_g.abs(), 1) + 4 * U * r_g.abs()  # the fp32 scale 2 g / count carries two roundings of its own
        m["g_pred"] = assert_bound(f"{name}/g_pred", g_pred.reshape(d.shape), r_g, _bf16_store(r_g, Ef, g_pred.dtype == BF16))
    return m


# ---- CPU unit tests: the replay bounds accept the correct stage and reject each planted fault ------------------------------
def _cpu_sage_case(fault=None, N=300, H=32, p=0.2, seed=77):
    """fp32 restatement of SageConvFn.backward on CPU - the arithmetic the kernels do - with one fault planted on request."""
    from oracle.sage_oracle import csr_oracle

    gen = torch.Generator().manual_seed(5)
    rng = np.random.default_rng(5)
    E = 5 * N
    ei = np.stack([rng.integers(0, N, E), rng.integers(0, N, E)])
    rowptr, col, _, inv = csr_oracle(ei, N)
    graph = {"rowptr": torch.from_numpy(rowptr), "col": torch.from_numpy(col), "inv_deg": torch.from_numpy(inv)}
    x, agg = torch.randn(N, H, generator=gen), torch.randn(N, H, generator=gen)
    wl, wr = torch.randn(H, H, generator=gen) / H ** 0.5, torch.randn(H, H, generator=gen) / H ** 0.5
    pre = torch.randn(N, H, generator=gen) * 2 + 0.3
    stats = torch.stack([pre.mean(1), 1 / torch.sqrt(pre.var(1, unbiased=False) + 1e-5)], 1)
    gamma = (torch.rand(H, generator=gen) + 0.5) * torch.sign(torch.randn(H, generator=gen))
    beta = torch.randn(H, generator=gen) * 0.5
    g_out = torch.randn(N, H, generator=gen)
    keep = keep_of(seed + (fault == "seed"), N, H, p, "cpu").float()
    z = (pre - stats[:, :1]) * stats[:, 1:] * gamma + beta
    gy, gg0, xh, _, _, _ = ln_tail_grad(pre, stats, gamma, beta, g_out, keep, torch.float32, (z > 0).float())
    rp, cl = graph["rowptr"].long(), graph["col"].long()
    dst = torch.repeat_interleave(torch.arange(N), rp[1:] - rp[:-1])
    scale = inv[cl.numpy()] if fault == "inv_deg" else inv[dst.numpy()]  # source side: inv_deg of the row that sent g_y
    g_t = torch.zeros(N, H).index_add_(0, cl, torch.from_numpy(scale)[:, None] * gy[dst])
    g_x = g_t @ wl + gy @ wr + (0 if fault == "residual" else g_out)
    grads = (g_x, gy.T @ agg, gy.sum(0), gy.T @ x, (gg0 * xh).sum(0), gg0.sum(0))
    return {"saved": (x, agg, pre, stats, wl, wr, gamma, beta), "graph": graph, "p": p, "seed": seed, "g_out": g_out, "g_y": gy,
            "grads": grads}


def test_replay_bound_accepts_the_fp32_sage_backward():
    m = check_sage_bwd("cpu_sage", _cpu_sage_case())
    assert m["g_x"] <= 1 and m["g_y"] <= 1


@pytest.mark.parametrize("fault", ["residual", "seed", "inv_deg"])
def test_replay_bound_rejects_a_planted_sage_fault(fault):
    """A dropped residual addend of g_x, a dropout mask regenerated with seed + 1, and g_t scaled by the inv_deg of the
    destination of the transposed gather instead of the source."""
    with pytest.raises(AssertionError, match="outside the bound"):
        check_sage_bwd(f"cpu_sage_{fault}", _cpu_sage_case(fault))


def _cpu_mse(round_target, N=4096, mean=True):
    gen = torch.Generator().manual_seed(9)
    pred = (torch.randn(N, 1, generator=gen) * 3 + 5).to(BF16)
    target = torch.randn(N, 1, generator=gen) * 3 + 5
    mask = torch.rand(N, generator=gen) < 0.6
    t = target.to(BF16).float() if round_target else target
    d = pred.float() - t
    cnt = float(mask.sum())
    div = max(cnt, 1.0) if mean else 1.0
    loss = ((d * d)[mask].sum() / div).reshape(1)
    g = (2 * 0.5 * d * mask.float()[:, None] / div).to(BF16)
    return pred, target, mask, mean, loss, cnt, 0.5, g


@pytest.mark.parametrize("mean", [True, False])
def test_replay_mse_bound_accepts_fp32_and_rejects_a_target_rounded_to_bf16(mean):
    check_mse("cpu_mse", *_cpu_mse(False, mean=mean))
    with pytest.raises(AssertionError):
        check_mse("cpu_mse_rounded", *_cpu_mse(True, mean=mean))


def test_replay_mse_known_answer_on_cpu():
    """pred 17.0 (bf16) against 17.03 (fp32): F.mse_loss gives 9.0e-4; rounding the target to bf16 first gives 0."""
    pred, target = torch.tensor([[17.0]], dtype=BF16), torch.tensor([[17.03]])
    assert abs(float(torch.nn.functional.mse_loss(pred, target)) - 9.0e-4) < 1e-6
    loss = ((pred.float() - target) ** 2).reshape(1)
    check_mse("ka", pred, target, None, True, loss, 1, 1.0, None)
    with pytest.raises(AssertionError):
        check_mse("ka_rounded", pred, target, None, True, torch.zeros(1), 1, 1.0, None)


# ======================================== GPU: per-stage replay of the model =============================================
def _graph_dict(graph):
    return {"rowptr": graph.rowptr, "col": graph.col, "inv_deg": graph.inv_deg}


def _detached(v):
    if isinstance(v, (tuple, list)):
        return tuple(_detached(t) for t in v)
    return v.detach() if isinstance(v, torch.Tensor) else v


class Recorder:
    """Wraps forward / backward of the five Functions (and ops.epilogue_bwd, whose g_y the backward consumes)."""

    KINDS = ("SageConvFn", "LinearFn", "DecoderTailFn", "CastFn", "MaskedMSEFn")

    def __init__(self, monkeypatch):
        from deep_fem_uav_wing.gnn import ops

        self.calls, self.stack = [], []
        for kind in self.KINDS:
            cls = getattr(ops, kind)
            self._wrap(monkeypatch, cls, kind, cls.forward, cls.backward)
        real_eb = ops.epilogue_bwd

        def eb(*a, **k):
            res = real_eb(*a, **k)
            if self.stack:
                self.stack[-1]["g_y"] = res[0]
            return res

        monkeypatch.setattr(ops, "epilogue_bwd", eb)

    def _wrap(self, monkeypatch, cls, kind, fwd0, bwd0):
        def fwd(ctx, *args):
            out = fwd0(ctx, *args)
            rec = {"kind": kind, "args": _detached(args), "out": _detached(out)}
            ctx.replay_record = rec
            self.calls.append(rec)
            return out

        def bwd(ctx, *g):
            rec = ctx.replay_record
            rec["saved"], rec["g_in"] = _detached(ctx.saved_tensors), _detached(g)
            self.stack.append(rec)
            try:
                res = bwd0(ctx, *g)
            finally:
                self.stack.pop()
            rec["grads"] = _detached(res)
            return res

        monkeypatch.setattr(cls, "forward", staticmethod(fwd))
        monkeypatch.setattr(cls, "backward", staticmethod(bwd))


def check_sage_fwd(name, rec):
    from oracle import csr_aggregate_ex

    x_in, w_l, b_l, w_r, gamma, beta, graph, eps, p, seed, fused = rec["args"]
    x, agg, pre, stats, wl, wr, g64, b64 = rec["saved"]
    out = rec["out"]
    N, H = out.shape
    bf16 = x.dtype == BF16
    assert fused and float(eps) == 1e-5
    # the kernels read the compute-dtype copies of the fp32 master weights
    assert torch.equal(wl, w_l.detach().to(x.dtype)) and torch.equal(wr, w_r.detach().to(x.dtype))
    rp = graph.rowptr.cpu().numpy()
    ref = csr_aggregate_ex(rp, graph.col.cpu().numpy()[:int(rp[-1])], x.float().cpu().numpy(), row_scale=graph.inv_deg.cpu().numpy())
    ref = torch.from_numpy(ref).to(x.dtype)
    ib = torch.int32 if x.dtype == F32 else torch.int16
    mism = int((agg.cpu().view(ib) != ref.view(ib)).sum())
    assert mism == 0, f"{name}/agg: {mism} elements differ from the gather oracle"
    keep = keep_of(seed, N, H, p, out.device)
    fr = fwd_reference(agg, wl, x, wr, b_l.detach() if b_l is not None else None, (gamma.detach(), beta.detach()), True,
                       keep if p else None, x, None, None, bf16)
    return fwd_checks(name, {"pre": pre, "out": out, "stats": stats}, fr, bf16)


def check_linear(name, rec):
    x_in, w, b, relu, p, seed = rec["args"]
    x, wc, act = rec["saved"]
    out = rec["out"]
    N, Hout = out.shape
    bf16 = x.dtype == BF16
    assert torch.equal(wc, w.detach().to(x.dtype))
    keep = keep_of(seed, N, Hout, p, out.device) if p else None
    fr = fwd_reference(x, wc, None, None, b.detach() if b is not None else None, None, relu, keep, None, None, None, bf16)
    m = fwd_checks(name, {"out": out}, fr, bf16)
    g_out = rec["g_in"][0]
    g_x, dw, db = rec["grads"][:3]
    if relu or p:
        kp = keep if keep is not None else torch.ones_like(act, dtype=torch.float64)
        r_gy = g_out.double() * kp * (act.double() > 0)
        Ef = short_bound(r_gy.abs(), 1)
        m["g_y"] = assert_bound(f"{name}/g_y", rec["g_y"], r_gy, _bf16_store(r_gy, Ef, bf16))
        gy_k, r_db, S_db = rec["g_y"], r_gy, r_gy.abs() + Ef
    else:
        gy_k = g_out
        r_db, S_db = g_out.double(), g_out.double().abs()
    if dw is not None:
        m["dW"] = _long(f"{name}/dW", dw, gy_k, x, _dw_chain(gy_k, x, Hout, x.shape[1], 0, x.dtype))
        if db is not None:
            m["db"] = _colsum(f"{name}/db", db, r_db, S_db, r_db.float().cpu())
    if g_x is not None:
        r = gy_k.double() @ wc.double()
        Ex = short_bound(gy_k.double().abs() @ wc.double().abs(), Hout)
        m["g_x"] = assert_bound(f"{name}/g_x", g_x, r, _bf16_store(r, Ex, bf16))
    return m


def check_decoder(name, rec):
    h_in, w3, b3, w4, b4, p, seed = rec["args"]
    h, hid, w3c, w4f = rec["saved"]
    out = rec["out"]
    N, Hmid = hid.shape
    bf16 = h.dtype == BF16
    assert torch.equal(w3c, w3.detach().to(h.dtype)) and torch.equal(w4f, w4.detach().float().reshape(-1))
    keep = keep_of(seed, N, Hmid, p, out.device)
    b4f = b4.detach().float().reshape(-1) if b4 is not None else None
    fr = fwd_reference(h, w3c, None, None, b3.detach() if b3 is not None else None, None, True, keep if p else None, None, w4f, b4f, bf16)
    m = fwd_checks(name, {"out": hid}, fr, bf16)
    r_rd, E_rd = fr["rowdot"]
    m["row_dot"] = assert_bound(f"{name}/row_dot", out.reshape(-1), r_rd, _bf16_store(r_rd, E_rd, bf16))
    g_r = rec["g_in"][0].reshape(-1).float()
    g_h, dw3, db3, dw4, db4 = rec["grads"][:5]
    r_gy = g_r.double()[:, None] * w4f.double()[None, :] * keep * (hid.double() > 0)
    Ef = short_bound(r_gy.abs(), 1)
    gy_k = rec["g_y"]
    m["g_y"] = assert_bound(f"{name}/g_y", gy_k, r_gy, _bf16_store(r_gy, Ef, bf16))
    if dw3 is not None:
        m["dW3"] = _long(f"{name}/dW3", dw3, gy_k, h, _dw_chain(gy_k, h, Hmid, h.shape[1], 0, h.dtype))
        m["dw4"] = _long(f"{name}/dw4", dw4.reshape(-1, 1), hid, g_r[:, None])
        if db3 is not None:
            m["db3"] = _colsum(f"{name}/db3", db3, r_gy, r_gy.abs() + Ef, r_gy.float().cpu())
        if db4 is not None:
            m["db4"] = _colsum(f"{name}/db4", db4, g_r.double()[:, None], g_r.double().abs()[:, None], g_r.cpu()[:, None])
    if g_h is not None:
        r = gy_k.double() @ w3c.double()
        Ex = short_bound(gy_k.double().abs() @ w3c.double().abs(), Hmid)
        m["g_h"] = assert_bound(f"{name}/g_h", g_h, r, _bf16_store(r, Ex, bf16))
    return m


def check_cast(name, rec):
    t, dtype = rec["args"]
    assert torch.equal(rec["out"], t.detach().to(dtype)), f"{name}: forward cast is not round-to-nearest-even"
    g = rec["g_in"][0]
    assert torch.equal(rec["grads"][0], g.to(t.dtype)), f"{name}: backward cast differs from torch"
    return {}


def check_step(name, rec_calls, sens):
    """Every recorded stage of one step against its fp64 restatement; returns the margins per stage."""
    margins, counts = {}, {}
    for rec in rec_calls:
        kind = rec["kind"]
        i = counts[kind] = counts.get(kind, -1) + 1
        row = f"{name}/{kind}{i}"
        assert "grads" in rec, f"{row}: the backward of this Function never ran"
        if kind == "SageConvFn":
            m = check_sage_fwd(row, rec)
            x, agg, pre, stats, wl, wr, gamma, beta = rec["saved"]
            graph = rec["args"][6]
            m.update(check_sage_bwd(row, {"saved": rec["saved"], "graph": _graph_dict(graph), "p": rec["args"][8], "seed": rec["args"][9],
                                          "g_out": rec["g_in"][0].contiguous(), "g_y": rec["g_y"], "grads": rec["grads"]}))
            if sens:
                assert all(g is None for g in rec["grads"][1:6]), f"{row}: a parameter gradient was computed"
        elif kind == "LinearFn":
            m = check_linear(row, rec)
        elif kind == "DecoderTailFn":
            m = check_decoder(row, rec)
        elif kind == "CastFn":
            m = check_cast(row, rec)
        else:
            pred, target, mask, mean = rec["args"]
            loss, count = rec["out"]
            m = check_mse(row, pred, target, mask, mean, loss, count, rec["g_in"][0], rec["grads"][0])
        margins[f"{kind}{i}"] = m
    return margins


def _random_multigraph(n, seed, deg=6):
    """Directed multigraph: self loops, duplicate edges, a tenth of the nodes isolated (neither source nor destination)."""
    rng = np.random.default_rng(seed)
    live = rng.permutation(n)[: max(n - n // 10, 1)] if n else np.zeros(0, np.int64)
    E = deg * len(live)
    src, dst = rng.choice(live, E), rng.choice(live, E)
    k = E // 50
    src[:k] = dst[:k]                                     # self loops
    src[k:2 * k], dst[k:2 * k] = src[2 * k:3 * k], dst[2 * k:3 * k]  # duplicates
    return np.stack([src, dst]).astype(np.int64)


def _mesh(kind):
    from deep_fem_uav_wing.gnn import synth

    if kind == "tri":
        m = synth.surface_tri_wing(3000, seed=21)
    elif kind == "tet":
        m = synth.tet_lattice_wing(3000, seed=22)
    else:
        n = 20011 if kind == "multi" else int(kind[1:])
        rng = np.random.default_rng(n)
        m = {"x": rng.standard_normal((n, 10)).astype(np.float32), "edge_index": _random_multigraph(n, n),
             "y": (rng.random((n, 1)) * 8).astype(np.float32), "loss_mask": rng.random(n) < 0.8, "num_nodes": n}
    return m


# (compute dtype, mode, hidden, layers, out_channels, features, in_channels, graph)
REPLAY = [
    (F32, "p0.2", 64, 3, 1, "f32", 10, "tri"),
    (F32, "p0", 128, 1, 3, "f32", 24, "tet"),
    (F32, "sens", 256, 3, 1, "f32", 10, "multi"),
    (F32, "p0.2", 20, 3, 1, "f32", 10, "multi"),
    (F32, "p0.2", 36, 1, 3, "f32", 24, "tri"),
    (F32, "sens", 20, 1, 1, "f32", 24, "tet"),
    (F32, "p0.2", 128, 3, 1, "f32", 10, "n127"),
    (F32, "p0.2", 64, 1, 3, "f32", 10, "n129"),
    (F32, "p0.2", 128, 3, 1, "f32", 10, "n56909"),
    (BF16, "p0.2", 64, 3, 1, "f32", 10, "tri"),
    (BF16, "p0.2", 128, 3, 1, "bf16", 10, "multi"),
    (BF16, "p0", 256, 1, 3, "f32", 24, "tet"),
    (BF16, "sens", 128, 3, 1, "bf16", 10, "tet"),
    (BF16, "p0.2", 40, 3, 1, "f32", 10, "multi"),
    (BF16, "p0.2", 96, 1, 3, "bf16", 24, "tri"),
    (BF16, "sens", 96, 3, 1, "f32", 24, "multi"),
    (BF16, "p0", 40, 1, 1, "bf16", 10, "n128"),
    (BF16, "p0.2", 128, 3, 1, "bf16", 10, "n129"),
    (BF16, "p0.2", 256, 3, 1, "bf16", 10, "n56909"),
    (BF16, "p0.2", 64, 1, 3, "f32", 24, "n56909"),
]


def _rid(c):
    cd, mode, h, l, oc, feat, k, g = c
    return f"{'f32' if cd == F32 else 'bf16'}_{mode}_h{h}_l{l}_oc{oc}_{feat}feat_in{k}_{g}"


def _step(model, x, ei, y, mask, sens, seed):
    torch.manual_seed(seed)  # the model draws its dropout seed from torch's CPU generator
    from deep_fem_uav_wing.gnn.model import MaskedMSELoss

    xi = x.detach().clone().requires_grad_(sens)
    model.zero_grad(set_to_none=True)
    out = model(xi, ei)
    loss = MaskedMSELoss()(out, y, mask)
    return out, loss, xi


@pytest.mark.gpu
@pytest.mark.parametrize("case", REPLAY, ids=[_rid(c) for c in REPLAY])
def test_training_step_replays_against_fp64(case, monkeypatch):
    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    cd, mode, H, L, oc, feat, k, gname = case
    name = _rid(case)
    sens = mode == "sens"
    p = 0.2 if mode == "p0.2" else 0.0
    m = _mesh(gname)
    n = m["num_nodes"]
    x = torch.from_numpy(m["x"]).cuda()
    if k > 10:
        x = torch.cat([x, torch.randn(n, k - 10, generator=torch.Generator(device="cuda").manual_seed(3), device="cuda")], 1)
    if feat == "bf16":
        x = x.to(BF16)
    ei = torch.from_numpy(m["edge_index"]).cuda()
    y = torch.from_numpy(m["y"]).cuda().repeat(1, oc) + torch.arange(oc, device="cuda")
    mask = torch.from_numpy(np.asarray(m["loss_mask"])).cuda()
    torch.manual_seed(_seed(name))
    model = GraphSAGEModel(k, H, oc, L, dropout=p).cuda().set_compute_dtype(cd)
    with torch.no_grad():  # LayerNorm affine away from (1, 0), so gamma and beta take part in every restatement
        for norm in model.norms:
            norm.weight.copy_((torch.rand(H, device="cuda") + 0.5) * torch.sign(torch.randn(H, device="cuda")))
            norm.bias.copy_(torch.randn(H, device="cuda") * 0.5)
    if sens:
        model.eval().requires_grad_(False)
    else:
        model.train()
    graph = ops.get_graph(ei, n)

    rec = Recorder(monkeypatch)
    out, loss, xi = _step(model, x, ei, y, mask, sens, 1)
    bw_calls = []
    real_dw = ops.linear_bwd_weight
    monkeypatch.setattr(ops, "linear_bwd_weight", lambda *a, **kw: bw_calls.append(1) or real_dw(*a, **kw))
    _, names = launched_kernels(loss.backward)
    if sens:
        assert bw_calls == [], f"{name}: dfw_linear_bwd_weight ran in a step that wants no parameter gradient"
        bad = sorted({nm for nm in names if re.search(_WEIGHT_GRAD_KERNELS, nm)})
        assert not bad, f"{name}: weight-gradient kernels launched: {bad}"
        assert xi.grad is not None
    if gname == "multi":
        assert int(graph.status_t[2]) == 1, "the random multigraph must take the general transpose build"
    elif gname in ("tri", "tet"):
        assert int(graph.status_t[2]) == 0, "a mesh holds both directions of every edge: the transpose is a copy"
    kinds = [r["kind"] for r in rec.calls]
    assert kinds.count("SageConvFn") == L and kinds.count("MaskedMSEFn") == 1
    assert kinds.count("DecoderTailFn") == (oc == 1)
    assert kinds.count("CastFn") == (2 if (feat == "f32" and cd == BF16) else 0)
    margins = check_step(name, rec.calls, sens)
    record(f"layer_replay/{name}", margins=margins)

    def grads():
        return [xi.grad] if sens else [q.grad for q in model.parameters()]

    first = [g.clone() for g in grads()]
    assert all(g is not None for g in first)
    for overlap in (False, True):  # the side-stream weight gradient, off and on again (a second run)
        monkeypatch.setattr(ops, "OVERLAP_DW", overlap)
        out2, loss2, xi = _step(model, x, ei, y, mask, sens, 1)
        loss2.backward()
        assert torch.equal(out2, out)
        for a, b in zip(first, grads()):
            assert torch.equal(a, b), f"{name}: a gradient differs with OVERLAP_DW={overlap}"


# ======================================== GPU: masked MSE with mixed dtypes ==============================================
@pytest.mark.gpu
def test_masked_mse_known_answer_bf16_prediction_fp32_target():
    """F.mse_loss(bf16 17.0, fp32 17.03) = 9.0e-4 (the difference is taken in fp32); rounding the target first gives 0."""
    from deep_fem_uav_wing.gnn.model import MaskedMSELoss

    pred = torch.tensor([[17.0]], dtype=BF16, device="cuda", requires_grad=True)
    target = torch.tensor([[17.03]], device="cuda")
    loss = MaskedMSELoss()(pred, target)
    ref = torch.nn.functional.mse_loss(pred.detach().cpu(), target.cpu())
    assert loss.dtype == F32 and float(loss.detach()) == float(ref) and abs(float(loss.detach()) - 9.0e-4) < 1e-6
    loss.backward()
    g = 2 * (17.0 - float(target))
    assert pred.grad.dtype == BF16 and abs(float(pred.grad) - g) <= 2.0 ** -8 * abs(g)


@pytest.mark.gpu
@pytest.mark.parametrize("mean", [True, False], ids=["mean", "sum"])
@pytest.mark.parametrize("masked", [True, False], ids=["masked", "unmasked"])
def test_masked_mse_mixed_dtypes_against_fp64(mean, masked):
    from deep_fem_uav_wing.gnn.model import MaskedMSELoss

    N, C = 200003, 3
    gen = torch.Generator(device="cuda").manual_seed(31 + 2 * mean + masked)
    pred = (torch.randn(N, C, generator=gen, device="cuda") * 3 + 5).to(BF16).requires_grad_(True)
    target = torch.randn(N, C, generator=gen, device="cuda") * 3 + 5
    mask = (torch.rand(N, generator=gen, device="cuda") < 0.7) if masked else None
    crit = MaskedMSELoss("mean" if mean else "sum")
    loss = crit(pred, target, mask)
    (loss * 0.75).backward()
    m = check_mse(f"mse_mixed/{'mean' if mean else 'sum'}/{int(masked)}", pred.detach(), target, mask, mean, loss.detach(), crit.last_count,
                  0.75, pred.grad)
    assert pred.grad.dtype == BF16
    assert_no_rounding_bias("mse_mixed/g_pred", pred.grad, 2 * 0.75 * (pred.detach().double() - target.double())
                            * (mask.double()[:, None] if masked else 1.0) / ((float(crit.last_count) if mean else 1.0)), 0 * pred.grad.double())
    record(f"layer_replay/masked_mse_mixed/mean{int(mean)}/masked{int(masked)}", **m)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [F32, BF16], ids=["f32", "bf16"])
def test_masked_mse_equal_dtypes_unchanged(dt):
    """Equal dtypes take the same kernel call as before the mixed-dtype rule: the raw ABI on the same inputs, bit for bit."""
    from deep_fem_uav_wing.gnn import _cabi
    from deep_fem_uav_wing.gnn.model import MaskedMSELoss

    N, C = 50021, 1
    gen = torch.Generator(device="cuda").manual_seed(41)
    pred = torch.randn(N, C, generator=gen, device="cuda").to(dt).requires_grad_(True)
    target = torch.randn(N, C, generator=gen, device="cuda").to(dt)
    mask = torch.rand(N, generator=gen, device="cuda") < 0.5
    loss = MaskedMSELoss()(pred, target, mask)
    loss.backward()
    lib, s = _cabi.lib, torch.cuda.current_stream().cuda_stream
    res = torch.empty(2, device="cuda")
    ws = torch.empty(lib.dfw_masked_mse_ws_bytes(N, C), dtype=torch.uint8, device="cuda")
    m8 = mask.to(torch.uint8)
    d = int(dt == BF16)
    _cabi.check(lib.dfw_masked_mse_fwd(pred.data_ptr(), target.data_ptr(), m8.data_ptr(), N, C, 1, d, res.data_ptr(), ws.data_ptr(), ws.numel(), s))
    g = torch.empty_like(pred)
    one = torch.ones(1, device="cuda")
    _cabi.check(lib.dfw_masked_mse_bwd(pred.data_ptr(), target.data_ptr(), m8.data_ptr(), res.data_ptr(), one.data_ptr(), N, C, 1, d, g.data_ptr(), s))
    assert torch.equal(loss.detach(), res[0]) and torch.equal(pred.grad, g)


# ======================================== GPU: one-call entry points through the raw C ABI ===============================
NS = [0, 1, 129, 56909]


def _p(t):
    return None if t is None else t.data_ptr()


_SPARE = []


def _pn(t):
    """A valid address for an empty operand (N = 0): the ABI rejects NULL operands, torch reports 0 for empty tensors."""
    if t is None:
        return None
    if t.numel():
        return t.data_ptr()
    if not _SPARE:
        _SPARE.append(torch.empty(256, dtype=torch.uint8, device="cuda"))
    return _SPARE[0].data_ptr()


def _bits_equal(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(torch.uint8) if a.numel() else a, b.view(torch.uint8) if b.numel() else b)


def _ws_exact_and_short(name, call, nbytes):
    """call(ws_ptr, ws_bytes) -> rc.  Exactly `nbytes` inside guard bands succeeds; one byte less is refused."""
    from deep_fem_uav_wing.gnn import _cabi

    if nbytes > 0:
        ar = Arena()
        ws, _ = ar.ws(nbytes - 1)
        rc = call(ws.data_ptr(), nbytes - 1)
        assert rc != 0 and b"workspace" in _cabi.lib.dfw_last_error(), f"{name}: a workspace one byte short was not refused"
        ar.check(name + "/short")


def _rand_graph(n, seed):
    from types import SimpleNamespace

    from deep_fem_uav_wing.gnn import ops

    if n == 0:
        z = torch.zeros(0, dtype=torch.int32, device="cuda")
        return SimpleNamespace(rowptr=torch.zeros(1, dtype=torch.int32, device="cuda"), col=z, inv_deg=z.float(), num_edges=0)
    return ops.get_graph(torch.from_numpy(_random_multigraph(n, seed)).cuda(), n)


@pytest.mark.gpu
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("H", [64, 128, 256])
@pytest.mark.parametrize("dt", [F32, BF16], ids=["f32", "bf16"])
def test_one_call_sage_layer_over_its_matrix(dt, H, N):
    from deep_fem_uav_wing.gnn import _cabi, ops

    lib, s, d = _cabi.lib, torch.cuda.current_stream().cuda_stream, int(dt == BF16)
    graph = _rand_graph(N, 100 + H)
    gen = torch.Generator(device="cuda").manual_seed(H + N)
    x0 = torch.randn(N, H, generator=gen, device="cuda").to(dt)
    w_l = torch.randn(H, H, generator=gen, device="cuda") / H ** 0.5
    w_r = torch.randn(H, H, generator=gen, device="cuda") / H ** 0.5
    b0 = torch.randn(H, generator=gen, device="cuda")
    gamma = (torch.rand(H, generator=gen, device="cuda") + 0.5) * torch.sign(torch.randn(H, generator=gen, device="cuda"))
    beta = torch.randn(H, generator=gen, device="cuda") * 0.5
    g_out = torch.randn(N, H, generator=gen, device="cuda").to(dt)
    wl_c, wr_c = w_l.to(dt), w_r.to(dt)
    rp_t, col_t = graph.transpose() if N else (graph.rowptr, graph.col)
    for tail, p in ((False, 0.0), (True, 0.0), (True, 0.2)):
        for want_gx in (True, False):
            if want_gx and SIMT and N:
                continue  # the one-call backward's input gradient needs the tensor-core linear
            for has_bias in (True, False):
                row = f"sage_layer/{'bf16' if d else 'f32'}/h{H}/N{N}/tail{int(tail)}/p{p}/gx{int(want_gx)}/bias{int(has_bias)}"
                seed = 1000 + H
                flags = (_cabi.EP_LAYERNORM | _cabi.EP_RELU | _cabi.EP_RESIDUAL | (_cabi.EP_DROPOUT if p else 0)) if tail else 0
                b_l = b0 if has_bias else None
                ar = Arena()
                agg, out = ar.out((N, H), dt), ar.out((N, H), dt)
                pre = ar.out((N, H), dt) if tail else None
                stats = ar.out((N, 2), F32) if tail else None
                nb = lib.dfw_sage_layer_fwd_ws_bytes(N, H, H, d)
                ws, _ = ar.ws(nb)

                def fwd(wsp, wsb):
                    return lib.dfw_sage_layer_fwd(graph.rowptr.data_ptr(), _pn(graph.col), graph.inv_deg.data_ptr() if N else _pn(graph.inv_deg),
                                                  _pn(x0), wl_c.data_ptr(), _p(b_l), wr_c.data_ptr(), _p(gamma if tail else None),
                                                  _p(beta if tail else None), 1e-5, p, seed, flags, _pn(agg), _pn(pre), _pn(stats), _pn(out),
                                                  N, graph.num_edges, H, H, d, wsp, wsb, s)

                assert fwd(ws.data_ptr(), nb) == 0, lib.dfw_last_error()
                ar.check(row + "/fwd")
                _ws_exact_and_short(row + "/fwd", fwd, nb)
                ar2 = Arena()
                g_x = ar2.out((N, H), dt) if want_gx else None
                dw_l, dw_r = ar2.out((H, H), F32), ar2.out((H, H), F32)
                db_l = ar2.out((H,), F32) if has_bias else None
                dgamma = ar2.out((H,), F32) if tail else None
                dbeta = ar2.out((H,), F32) if tail else None
                nbb = lib.dfw_sage_layer_bwd_ws_bytes(N, H, H, d, int(want_gx))
                ws2, _ = ar2.ws(nbb)

                def bwd(wsp, wsb):
                    return lib.dfw_sage_layer_bwd(_pn(rp_t) if want_gx else None, _pn(col_t) if want_gx else None, _pn(graph.inv_deg),
                                                  _pn(x0), _pn(agg), _pn(pre), _pn(stats), wl_c.data_ptr(), wr_c.data_ptr(),
                                                  _p(gamma if tail else None), _p(beta if tail else None), _pn(g_out), p, seed, flags,
                                                  _pn(g_x), dw_l.data_ptr(), _p(db_l), dw_r.data_ptr(), _p(dgamma), _p(dbeta), N,
                                                  graph.num_edges, H, H, d, wsp, wsb, s)

                assert bwd(ws2.data_ptr(), nbb) == 0, lib.dfw_last_error()
                ar2.check(row + "/bwd")
                _ws_exact_and_short(row + "/bwd", bwd, nbb)
                params = [t for t in (dw_l, dw_r, db_l, dgamma, dbeta) if t is not None]
                if N == 0:
                    assert all(bool((t == 0).all()) for t in params), f"{row}: an empty batch must give zero parameter gradients"
                    continue
                # the autograd Function on the same inputs
                x = x0.clone().requires_grad_(want_gx)
                leaves = [t.clone().requires_grad_(True) if t is not None else None
                          for t in (w_l, b_l, w_r, gamma if tail else None, beta if tail else None)]
                ref = ops.SageConvFn.apply(x, leaves[0], leaves[1], leaves[2], leaves[3], leaves[4], graph, 1e-5, p, seed, tail)
                ref.backward(g_out)
                assert _bits_equal(out, ref.detach()), f"{row}: out differs from the autograd path"
                if want_gx:
                    assert _bits_equal(g_x, x.grad), f"{row}: g_x differs"
                for got, leaf in zip((dw_l, db_l, dw_r, dgamma, dbeta), leaves):
                    if leaf is not None:
                        assert _bits_equal(got, leaf.grad), f"{row}: a parameter gradient differs"


@pytest.mark.gpu
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("mode", ["encoder", "decoder"])
@pytest.mark.parametrize("dt", [F32, BF16], ids=["f32", "bf16"])
def test_one_call_mlp2_over_its_matrix(dt, mode, N):
    from deep_fem_uav_wing.gnn import _cabi, ops

    lib, s, d = _cabi.lib, torch.cuda.current_stream().cuda_stream, int(dt == BF16)
    enc = mode == "encoder"
    shapes = [(k, h) for k in (10, 24) for h in (64, 128, 256)] if enc else [(k, 64) for k in (64, 128, 256)]
    for K, Hx in shapes:
        Hmid, Hout = (64, Hx) if enc else (Hx, 1)
        gen = torch.Generator(device="cuda").manual_seed(K * 1000 + Hx + N)
        x0 = torch.randn(N, K, generator=gen, device="cuda").to(dt)
        w1 = torch.randn(Hmid, K, generator=gen, device="cuda") / K ** 0.5
        b1 = torch.randn(Hmid, generator=gen, device="cuda")
        w2 = torch.randn(Hout, Hmid, generator=gen, device="cuda") / Hmid ** 0.5
        b2 = torch.randn(Hout, generator=gen, device="cuda")
        g_o = torch.randn(N, Hout, generator=gen, device="cuda").to(dt)
        w1c = w1.to(dt)
        w2c = w2.to(dt) if enc else w2.reshape(-1).contiguous()
        for p in ((0.0,) if enc else (0.0, 0.2)):
            for want_gx in (True, False):
                for nb1, nb2 in ((False, False), (True, True)):
                    for save_hidden in ((True,) if enc else (True, False)):
                        row = f"mlp2/{mode}/{'bf16' if d else 'f32'}/k{K}/h{Hx}/N{N}/p{p}/gx{int(want_gx)}/nullbias{int(nb1)}/hid{int(save_hidden)}"
                        seed = 77 + K
                        bb1, bb2 = (None if nb1 else b1), (None if nb2 else b2)
                        ar = Arena()
                        hidden = ar.out((N, Hmid), dt) if save_hidden else None
                        out = ar.out((N, Hout), dt) if enc else ar.out((N,), F32)
                        nb = lib.dfw_mlp2_fwd_ws_bytes(N, K, Hmid, Hout, d)
                        ws, _ = ar.ws(nb)

                        def fwd(wsp, wsb):
                            return lib.dfw_mlp2_fwd(_pn(x0), w1c.data_ptr(), _p(bb1), w2c.data_ptr(), _p(bb2), p, seed, 0, 0 if enc else 1,
                                                    _pn(hidden), _pn(out), N, K, Hmid, Hout, d, wsp, wsb, s)

                        assert fwd(ws.data_ptr(), nb) == 0, lib.dfw_last_error()
                        ar.check(row + "/fwd")
                        _ws_exact_and_short(row + "/fwd", fwd, nb)
                        # the autograd path
                        x = x0.clone().requires_grad_(want_gx)
                        L1, L2 = w1.clone().requires_grad_(True), w2.clone().requires_grad_(True)
                        B1 = bb1.clone().requires_grad_(True) if bb1 is not None else None
                        B2 = bb2.clone().requires_grad_(True) if bb2 is not None else None
                        if N:
                            if enc:
                                h1 = ops.LinearFn.apply(x, L1, B1, True, 0.0, 0)
                                y = ops.LinearFn.apply(h1, L2, B2, True, 0.0, 0)
                                assert _bits_equal(out, y.detach()) and _bits_equal(hidden, h1.detach()), f"{row}: forward differs"
                                y.backward(g_o)
                            else:
                                y = ops.DecoderTailFn.apply(x, L1, B1, L2, B2, p, seed)
                                want = out.unsqueeze(1) if dt == F32 else ops.cast(out.unsqueeze(1), dt)
                                assert _bits_equal(want, y.detach()), f"{row}: row dot differs"
                                y.backward(g_o)
                        if not save_hidden:
                            continue  # inference: nothing to differentiate
                        ar2 = Arena()
                        g_x = ar2.out((N, K), dt) if want_gx else None
                        dw1, dw2 = ar2.out((Hmid, K), F32), ar2.out((Hout, Hmid) if enc else (Hmid,), F32)
                        db1 = ar2.out((Hmid,), F32) if bb1 is not None else None
                        db2 = ar2.out((Hout,), F32) if bb2 is not None else None
                        nbb = lib.dfw_mlp2_bwd_ws_bytes(N, K, Hmid, Hout, d, 0 if enc else 1, int(want_gx))
                        ws2, _ = ar2.ws(nbb)
                        g_in = g_o if enc else g_o.reshape(-1).float().contiguous()

                        def bwd(wsp, wsb):
                            return lib.dfw_mlp2_bwd(_pn(x0), _pn(hidden), _pn(out) if enc else None, w1c.data_ptr(), w2c.data_ptr(), _pn(g_in),
                                                    p, seed, 0, 0 if enc else 1, _pn(g_x), dw1.data_ptr(), _p(db1), dw2.data_ptr(), _p(db2),
                                                    N, K, Hmid, Hout, d, wsp, wsb, s)

                        assert bwd(ws2.data_ptr(), nbb) == 0, lib.dfw_last_error()
                        ar2.check(row + "/bwd")
                        _ws_exact_and_short(row + "/bwd", bwd, nbb)
                        params = [t for t in (dw1, db1, dw2, db2) if t is not None]
                        if N == 0:
                            assert all(bool((t == 0).all()) for t in params), f"{row}: an empty batch must give zero parameter gradients"
                            continue
                        if want_gx:
                            assert _bits_equal(g_x, x.grad), f"{row}: g_x differs"
                        for got, leaf in ((dw1, L1), (db1, B1), (dw2, L2), (db2, B2)):
                            if leaf is not None:
                                assert _bits_equal(got.reshape(leaf.grad.shape), leaf.grad), f"{row}: a parameter gradient differs"


FWD_HC = [(F32, 20), (BF16, 40)] + [(cd, h) for h in (64, 96, 128, 256) for cd in (F32, BF16)]


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 1, 4])
@pytest.mark.parametrize("cd,H", FWD_HC, ids=[f"{'f32' if c == F32 else 'bf16'}_h{h}" for c, h in FWD_HC])
def test_one_call_forward_over_its_matrix(cd, H, L):
    from deep_fem_uav_wing.gnn import _cabi, ops
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    lib, s, dtc = _cabi.lib, torch.cuda.current_stream().cuda_stream, int(cd == BF16)
    for N in (0, 1, 127, 129, 20011):
        graph = _rand_graph(N, 7 + N)
        for in_dim in (10, 24):
            for x_dt in ({F32, cd}):
                if SIMT and N and cd == BF16 and x_dt == F32 and in_dim <= 16:
                    continue  # the encoder's first linear stores bf16 directly (DFW_EP_OUT_BF16), which DFW_FORCE_SIMT refuses
                for null_bias in (False, True):
                    row = f"forward/{'bf16' if dtc else 'f32'}/h{H}/L{L}/N{N}/in{in_dim}/x{'bf16' if x_dt == BF16 else 'f32'}/nullbias{int(null_bias)}"
                    torch.manual_seed(_seed(row))
                    model = GraphSAGEModel(in_dim, H, 1, L, dropout=0.1).cuda().eval().set_compute_dtype(cd)
                    if null_bias:
                        for lin in [model.encoder[0], model.encoder[2], model.decoder[0], model.decoder[3]] + [c.lin_l for c in model.convs]:
                            lin.bias = None
                    x = torch.randn(N, in_dim, device="cuda").to(x_dt)
                    fw = model._forward_weights(x_dt, cd)
                    if null_bias:
                        assert sum(t is None for t in fw.tensors) == 4 + L
                    ar = Arena()
                    out = ar.out((N,), F32)
                    nb = lib.dfw_graphsage_forward_ws_bytes(N, in_dim, 64, H, 64, int(x_dt == BF16), dtc)
                    ws, _ = ar.ws(nb)

                    def call(wsp, wsb):
                        return lib.dfw_graphsage_forward(graph.rowptr.data_ptr(), _pn(graph.col), _pn(graph.inv_deg), _pn(x), int(x_dt == BF16),
                                                         fw.array, L, N, graph.num_edges, in_dim, 64, H, 64, 1e-5, dtc, _pn(out), wsp, wsb, s)

                    assert call(ws.data_ptr(), nb) == 0, lib.dfw_last_error()
                    ar.check(row)
                    _ws_exact_and_short(row, call, nb)
                    if N == 0:
                        continue
                    with torch.enable_grad():  # grad mode on: the piecewise path of autograd Functions
                        want = model(x, graph)
                    got = ops.cast(ops.cast(out.unsqueeze(1), cd), x_dt)  # as GraphSAGEModel hands the row dot over
                    assert _bits_equal(got, want.detach()), f"{row}: the one-call forward differs from the piecewise path"
