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
