"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# Tolerances stated by BASELINE.json:north_star
TOL_FP32 = 1e-5
TOL_BF16 = 2e-2


def load_golden(name):
    """``<name>.npz``, merged with ``<name>.grads.npz`` where a model fixture keeps its gradients apart (every file stays
    under 1 MB)."""
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))
    grads = os.path.join(GOLDEN, name + ".grads.npz")
    if os.path.exists(grads):
        g.update(np.load(grads, allow_pickle=False))
    return g


def golden_state_dict(g):
    return {k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd/")}


def golden_grads(g):
    return {k[5:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("grad/")}


def rel_max(a, b):
    """max|a-b| / max|b|  (the forward-output metric of SURVEY 8d)."""
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    d = (a - b).abs().max().item() if a.numel() else 0.0
    return d / max(b.abs().max().item() if b.numel() else 0.0, 1e-30)


def rel_l2(a, b):
    """||a-b||_2 / ||b||_2  (the per-parameter gradient metric of SURVEY 8d)."""
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def canon_edges(ei):
    ei = np.asarray(ei)
    order = np.lexsort((ei[0], ei[1]))
    return ei[:, order]


def record(name, **vals):
    """Append the ACHIEVED numbers of a parity gate to ``gpurun_out/r02_parity_gates.jsonl`` (copied to ``profiles/`` after a
    GPU run) so that the margin of every tolerance is visible, not only pass/fail."""
    import json

    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "gpurun_out")
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "r02_parity_gates.jsonl"), "a") as f:
            f.write(json.dumps({"gate": name, **{k: (float(v) if isinstance(v, (int, float, np.floating)) else v) for k, v in vals.items()}}) + "\n")
    except OSError:
        pass


# ---- element-wise bounds against an fp64 reference (CPU, no device needed) -------------------------------------------
def bound_margin(got, r, bound):
    """(number of elements outside the bound, max |got - r| / bound).  An element with bound 0 must be exact; NaN fails."""
    err = (got.double() - r.double()).abs()
    bound = bound.double()
    bad = ~(err <= bound)
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0))
    return int(bad.sum().item()), (float(ratio.max().item()) if ratio.numel() else 0.0)


def assert_bound(name, got, r, bound):
    nbad, margin = bound_margin(got, r, bound)
    if nbad:
        err = (got.double() - r.double()).abs() - bound.double()
        i = int(torch.nan_to_num(err, nan=torch.inf).flatten().argmax())
        g, rr, b = got.flatten()[i].item(), r.flatten()[i].item(), bound.flatten()[i].item()
        raise AssertionError(f"{name}: {nbad} of {got.numel()} elements outside the bound (worst index {i}: got {g!r}, "
                             f"exact {rr!r}, bound {b!r}, max err/bound {margin:.3g})")
    return margin


def bf16_ulp(r):
    """One bf16 ulp at |r| (normal range)."""
    a = r.double().abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def rounding_bias(got, r, pre_store_bound):
    """Mean signed error of a bf16 store in ulps of r, signed toward |r| (a truncating store gives -0.5, RNE about 0),
    over the elements whose pre-store error bound is below 1/8 ulp, where the rounding is what decides the error."""
    r = r.double()
    use = (r != 0) & (pre_store_bound.double() < 0.125 * bf16_ulp(r))
    e = (got.double() - r) * torch.sign(r) / bf16_ulp(r)
    return float(e[use].mean().item()) if bool(use.any()) else 0.0, int(use.sum().item())


def assert_no_rounding_bias(name, got, r, pre_store_bound):
    if got.numel() < 100_000:
        return None
    bias, n = rounding_bias(got, r, pre_store_bound)
    assert n >= min(100_000, got.numel() // 2), f"{name}: only {n} elements qualify for the rounding-bias check"
    assert abs(bias) < 0.05, f"{name}: mean signed bf16 store error {bias:+.4f} ulp over {n} elements (truncation gives -0.5)"
    return bias


# ---- raw-ABI launches ----------------------------------------------------------------------------------------------------
class Arena:
    """Device buffers inside sentinel-filled guard bands: check() asserts that no byte outside the handed-out ranges
    changed.  The sentinel byte 0x7F reads as ~3.4e38 in fp32 and bf16, so an unwritten element fails its bound too."""

    G = 4096
    SENT = 0x7F

    def __init__(self):
        self.bufs = []

    def out(self, shape, dtype, fill=None):
        elt = torch.empty(0, dtype=dtype).element_size()
        n = int(np.prod(shape)) * elt
        raw = torch.full((n + 2 * self.G,), self.SENT, dtype=torch.uint8, device="cuda")
        t = raw[self.G:self.G + n].view(dtype).view(shape)
        if fill is not None:
            t.copy_(fill)
        self.bufs.append((raw, n))
        return t

    def ws(self, nbytes):
        return self.out((int(nbytes),), torch.uint8), int(nbytes)

    def check(self, name):
        torch.cuda.synchronize()
        for raw, n in self.bufs:
            lo, hi = raw[:self.G], raw[self.G + n:]
            assert bool((lo == self.SENT).all()) and bool((hi == self.SENT).all()), f"{name}: a byte outside an output or the workspace was written"


def launched_kernels(fn):
    """Run fn() under torch.profiler and return (fn's result, names of the CUDA kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if str(getattr(e, "device_type", "")).endswith("CUDA")]
    return res, names
