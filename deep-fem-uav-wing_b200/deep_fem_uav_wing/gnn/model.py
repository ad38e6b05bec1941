"""GraphSAGE model for wing stress prediction - B200-native drop-in.

Mirrors the public surface of the reference's ``src/deep_fem_uav_wing/gnn/model.py``:

* ``GraphSAGEModel(in_channels=10, hidden_channels=128, out_channels=1, num_layers=4, dropout=0.1)``
  with ``forward(x, edge_index, batch=None)`` and ``predict(data)``        (``model.py:24-112``)
* ``MaskedMSELoss(reduction)``                                             (``model.py:115-153``)
* ``compute_metrics(pred, target, mask, log_scale)``                       (``model.py:156-216``)
* ``SAGEConv(in_channels, out_channels)`` - replaces ``torch_geometric.nn.SAGEConv`` as
  constructed at ``model.py:63`` (mean aggregation, root weight, bias), parameters
  ``lin_l.weight / lin_l.bias / lin_r.weight``.

``state_dict`` keys are identical to the reference's, so its checkpoints load here and ours
load there.  Unlike the reference (``model.py:11-19,219-233``) this module needs no PyTorch
Geometric.  All arithmetic runs in ``libdfw_b200.so`` (hand-written sm_100a CUDA reached
through a C ABI); inputs must be CUDA tensors - there is no CPU fallback.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from . import ops

HAS_TORCH_GEOMETRIC = False  # not needed; kept because callers of the reference may probe it


def _next_seed() -> int:
    # CPU generator: follows torch.manual_seed (train_gnn.py:128) without touching the device.  Under torchrun every rank
    # seeds that generator identically, so the rank is mixed in: ranks must not all drop the same units of their meshes.
    seed = int(torch.randint(0, 2**62, (1,)).item())
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        seed ^= (torch.distributed.get_rank() * 0x9E3779B97F4A7C15) & 0x3FFFFFFFFFFFFFFF
    return seed


class SAGEConv(nn.Module):
    r"""``out_i = W_l . mean_{j -> i} x_j + b_l + W_r . x_i``  (PyG ``SAGEConv`` defaults).

    ``forward(x, edge_index)`` returns the pre-normalisation tensor, like PyG's layer.  The
    CSR of ``edge_index`` is built on the device once per tensor and cached.
    """

    def __init__(self, in_channels: int, out_channels: int, bias: bool = True):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.lin_l = nn.Linear(in_channels, out_channels, bias=bias)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)
        self.reset_parameters()

    def reset_parameters(self):
        bound = 1.0 / math.sqrt(self.in_channels)
        nn.init.uniform_(self.lin_l.weight, -bound, bound)
        nn.init.uniform_(self.lin_r.weight, -bound, bound)
        if self.lin_l.bias is not None:
            nn.init.uniform_(self.lin_l.bias, -bound, bound)

    def forward(self, x: torch.Tensor, edge_index) -> torch.Tensor:
        graph = edge_index if isinstance(edge_index, ops.CSRGraph) else ops.get_graph(edge_index, x.shape[0])
        return ops.SageConvFn.apply(x, self.lin_l.weight, self.lin_l.bias, self.lin_r.weight, None, None, graph, 0.0, 0.0, 0,
                                    False)

    def extra_repr(self) -> str:
        return f"{self.in_channels}, {self.out_channels}, aggr=mean"


class GraphSAGEModel(nn.Module):
    """GraphSAGE model for node-level stress prediction (``model.py:24-112``).

    Args:
        in_channels: Input feature dimension (default: 10)
        hidden_channels: Hidden layer dimension (default: 128)
        out_channels: Output dimension (default: 1)
        num_layers: Number of SAGE layers (default: 4)
        dropout: Dropout rate (default: 0.1)
    """

    def __init__(self, in_channels: int = 10, hidden_channels: int = 128, out_channels: int = 1, num_layers: int = 4,
                 dropout: float = 0.1):
        super().__init__()
        if hidden_channels % 4 != 0 or hidden_channels > 256:
            raise ValueError("dfw_b200: hidden_channels must be a multiple of 4 and <= 256")
        self.in_channels = in_channels
        self.hidden_channels = hidden_channels
        self.out_channels = out_channels
        self.num_layers = num_layers
        self.dropout = dropout
        self.compute_dtype = torch.float32
        self.node_reorder = "auto"  # 'auto' | 'always' | 'never': k-d relabelling of large meshes for bf16 inference (ops.get_inference_graph)
        self.mesh_plan = "auto"  # large-mesh bf16 inference: prepare the mesh for the block aggregation 'always', 'never', or ('auto') from
        #                          the second forward on the same edge_index tensor - a graph seen once is not worth the one-time preparation
        self.device_seeds = None  # int64 CUDA tensor [num_layers + 1]: dropout seeds read by the kernels (CUDA-graph mode)

        self.encoder = nn.Sequential(
            nn.Linear(in_channels, 64), nn.ReLU(), nn.Linear(64, hidden_channels), nn.ReLU()
        )
        self.convs = nn.ModuleList()
        self.norms = nn.ModuleList()
        for _ in range(num_layers):
            self.convs.append(SAGEConv(hidden_channels, hidden_channels))
            self.norms.append(nn.LayerNorm(hidden_channels))
        self.decoder = nn.Sequential(
            nn.Linear(hidden_channels, 64), nn.ReLU(), nn.Dropout(dropout), nn.Linear(64, out_channels)
        )

    def set_compute_dtype(self, dtype: torch.dtype) -> "GraphSAGEModel":
        """fp32 (default) or bf16 activations; parameters stay fp32 master copies."""
        if dtype not in (torch.float32, torch.bfloat16):
            raise TypeError("compute dtype must be torch.float32 or torch.bfloat16")
        if dtype == torch.bfloat16 and self.hidden_channels % 8 != 0:  # 16-byte rows for the 128-bit gathers
            raise ValueError(f"dfw_b200: bf16 activations need hidden_channels % 8 == 0 (got {self.hidden_channels})")
        self.compute_dtype = dtype
        return self

    def forward(self, x, edge_index, batch=None):
        """``x [N, in_channels]``, ``edge_index [2, E]`` int64 -> ``[N, out_channels]``.
        ``batch`` is accepted and ignored, as in the reference (``model.py:74``)."""
        ops._require_cuda(x, "x")
        cd = self.compute_dtype
        out_dtype = x.dtype
        restore = None
        n_nodes = int(x.shape[0])
        if (cd == torch.bfloat16 and not torch.is_grad_enabled() and isinstance(edge_index, torch.Tensor)
                and self.hidden_channels in ops.TC_AGG_WIDTHS and n_nodes >= ops.TC_AGG_MIN_NODES
                and not torch.cuda.is_current_stream_capturing() and self.mesh_plan != "never"
                and (self.mesh_plan == "always" or ops.static_mesh_seen_before(edge_index))):
            # large static mesh, bf16 inference (BASELINE.json config 4): block plan for the tensor-core aggregation and,
            # where the given numbering has poor locality, a one-time k-d relabelling of the nodes - applied here to the
            # 10-wide input and undone on the 1-wide output, so no [N, H] tensor is ever permuted
            pos = x[:, :3] if (self.node_reorder != "never" and self.in_channels >= 3) else None
            ig = ops.get_inference_graph(edge_index, n_nodes, pos=pos, reorder=self.node_reorder)
            graph = ig.graph
            if ig.order is not None:
                x = x.index_select(0, ig.order)
                restore = ig.new_id
        else:
            graph = edge_index if isinstance(edge_index, ops.CSRGraph) else ops.get_graph(edge_index, n_nodes)
        if (not torch.is_grad_enabled() and not self.training and self.out_channels == 1 and graph.plan is None
                and x.dtype in (torch.float32, cd)
                and (cd == torch.float32 or not torch.cuda.is_current_stream_capturing())):
            # (under stream capture with bf16 activations the piecewise path stays: it casts the weights INSIDE the graph, so a
            # replay after a parameter update sees the new values; the cached bf16 copies below would be frozen into the graph)
            # inference: the whole forward behind one C call (dfw_graphsage_forward) - the same launches as below, bit-identical,
            # without ~0.5 ms of Python between them (graphs with a block plan keep the piecewise path: its aggregation differs)
            out = ops.graphsage_forward(graph, x, self._forward_weights(x.dtype, cd), cd, float(self.norms[0].eps) if self.num_layers else 1e-5)
            out = ops.cast(ops.cast(out, cd), out_dtype)  # (the piecewise path hands the decoder's fp32 row dot over in the compute dtype)
            return out if restore is None else out.index_select(0, restore)
        p = float(self.dropout) if self.training else 0.0
        if p > 0.0 and self.device_seeds is not None:  # seeds live on the device (see gnn/graphed.py)
            layer_seed = [self.device_seeds[i:i + 1] for i in range(self.num_layers)]
            dec_seed = self.device_seeds[self.num_layers:self.num_layers + 1]
        else:
            seed = _next_seed() if p > 0.0 else 0
            layer_seed = [seed + 0x632BE5AB * (i + 1) for i in range(self.num_layers)]
            dec_seed = seed + 0x7F4A7C15

        enc0, enc2 = self.encoder[0], self.encoder[2]
        # The first linear reads the 10 raw features in THEIR dtype: normalised positions rounded to bf16 (8 bits) move a
        # trained model's output by percents where the stress field is steep (wing tip), while the layer is 10-wide and
        # costs nothing in fp32; its 64-wide output is what enters the compute dtype.
        if (x.dtype == torch.float32 and cd == torch.bfloat16 and not torch.is_grad_enabled() and self.in_channels <= 16
                and enc0.out_features % 4 == 0):
            # inference: fp32 arithmetic, bf16 result in one launch (the bits dfw_cast would give, without the fp32 [N, 64] round trip)
            h, _, _, _ = ops.linear_fwd(x.contiguous(), ops._f32(enc0.weight.detach()), bias=ops._f32(enc0.bias.detach()) if enc0.bias is not None else None,
                                        relu=True, out_bf16=True)
        else:
            h = x if (x.dtype == torch.float32 and cd == torch.bfloat16) else ops.cast_ad(x, cd)
            h = ops.LinearFn.apply(h, enc0.weight, enc0.bias, True, 0.0, 0)
            h = ops.cast_ad(h, cd)
        h = ops.LinearFn.apply(h, enc2.weight, enc2.bias, True, 0.0, 0)

        for i, (conv, norm) in enumerate(zip(self.convs, self.norms)):
            h = ops.SageConvFn.apply(h, conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight, norm.weight, norm.bias, graph,
                                     float(norm.eps), p, layer_seed[i], True)

        dec0, dec3 = self.decoder[0], self.decoder[3]
        if self.out_channels == 1:
            out = ops.DecoderTailFn.apply(h, dec0.weight, dec0.bias, dec3.weight, dec3.bias, p, dec_seed)
        else:
            hid = ops.LinearFn.apply(h, dec0.weight, dec0.bias, True, p, dec_seed)
            out = ops.LinearFn.apply(hid, dec3.weight, dec3.bias, False, 0.0, 0)
        out = ops.cast_ad(out, out_dtype)
        return out if restore is None else out.index_select(0, restore)

    def _forward_weights(self, x_dtype: torch.dtype, cd: torch.dtype) -> "ops.ForwardWeights":
        """Parameters in the layout of ``dfw_graphsage_forward`` (compute-dtype copies of the matrices), rebuilt only when a parameter
        was modified or replaced since the last call."""
        params = list(self.parameters())
        key = (x_dtype, cd, tuple((q.data_ptr(), q._version) for q in params))
        cached = getattr(self, "_fw_cache", None)
        if cached is not None and cached[0] == key:
            return cached[1]
        f32 = lambda t: ops._f32(t.detach()) if t is not None else None  # noqa: E731
        enc0, enc2 = self.encoder[0], self.encoder[2]
        ts = [ops._w(enc0.weight, x_dtype if x_dtype == torch.float32 else cd), f32(enc0.bias), ops._w(enc2.weight, cd), f32(enc2.bias)]
        for conv, norm in zip(self.convs, self.norms):
            ts += [ops._w(conv.lin_l.weight, cd), f32(conv.lin_l.bias), ops._w(conv.lin_r.weight, cd), f32(norm.weight), f32(norm.bias)]
        dec0, dec3 = self.decoder[0], self.decoder[3]
        ts += [ops._w(dec0.weight, cd), f32(dec0.bias), f32(dec3.weight).reshape(-1), f32(dec3.bias).reshape(-1) if dec3.bias is not None else None]
        fw = ops.ForwardWeights(ts, (self.in_channels, int(enc0.out_features), self.hidden_channels, int(dec0.out_features), self.num_layers))
        object.__setattr__(self, "_fw_cache", (key, fw))
        return fw

    def predict(self, data):
        """Convenience method for inference (``model.py:101-112``)."""
        self.eval()
        with torch.no_grad():
            return self.forward(data.x, data.edge_index, getattr(data, "batch", None))


class MaskedMSELoss(nn.Module):
    """MSE loss with masking support for the root singularity band (``model.py:115-153``).

    One fused reduction kernel replaces the boolean indexing, so by default there is no host
    sync.  With an all-False mask the value is 0 as in the reference; the reference returns a
    fresh leaf there (no gradient reaches the model), here the gradient is exactly zero.  Pass
    ``strict_empty=True`` to reproduce the fresh-leaf behaviour (costs one host sync).

    As ``F.mse_loss``: a bf16 prediction against an fp32 target (a model fed bf16 features) is
    computed in fp32 from the unrounded target, and its gradient comes back in bf16.
    """

    def __init__(self, reduction: str = "mean", strict_empty: bool = False):
        super().__init__()
        if reduction not in ("mean", "sum"):
            raise ValueError(f"reduction must be 'mean' or 'sum', got {reduction!r}")  # F.mse_loss accepts 'none' too;
        self.reduction = reduction                                                         # the reference never uses it
        self.strict_empty = strict_empty
        self.last_count = None

    def forward(self, pred, target, mask=None):
        loss, count = ops.MaskedMSEFn.apply(pred, target, mask, self.reduction == "mean")
        self.last_count = count
        if self.strict_empty and mask is not None and float(count.item()) == 0.0:
            return torch.tensor(0.0, device=pred.device, requires_grad=True)
        return loss


def metrics_from_device(result: torch.Tensor) -> dict:
    """8 doubles of ``ops.stress_metrics`` -> the reference's nested dict (``model.py:206-216``).  One D2H copy."""
    r = result.detach().cpu().tolist()

    def sub(o):
        return {"mae": float(r[o]), "rmse": float(r[o + 1]), "max_error": float(r[o + 2]), "count": int(round(r[o + 3]))}

    return {"all_nodes": sub(0), "masked_nodes": sub(4)}


def compute_metrics(pred: torch.Tensor, target: torch.Tensor, mask: torch.Tensor | None = None,
                    log_scale: bool = True) -> dict:
    """MAE / RMSE / max error in the original scale for all and masked nodes (``model.py:156-216``).

    CUDA tensors are reduced on the device by ``dfw_stress_metrics`` and only the 8 resulting numbers cross to the
    host (the reference copies ``pred``/``target``/``mask`` in full, ``model.py:173-179``, once per validation batch,
    ``train_gnn.py:85``); CPU tensors take the reference's numpy path verbatim.  ``metrics_from_device`` turns the
    device result into the reference's dict, so callers can queue several batches and synchronise once."""
    if pred.is_cuda and pred.dtype in (torch.float32, torch.bfloat16):
        return metrics_from_device(ops.stress_metrics(pred, target, mask, log_scale))
    p = pred.detach().float().cpu().numpy().flatten()
    t = target.detach().float().cpu().numpy().flatten()
    m = mask.detach().cpu().numpy().flatten() if mask is not None else None
    if log_scale:
        p, t = np.expm1(p), np.expm1(t)

    def subset(pp, tt, mm):
        if mm is not None:
            pp, tt = pp[mm], tt[mm]
        if len(pp) == 0:
            return {"mae": 0.0, "rmse": 0.0, "max_error": 0.0, "count": 0}
        err = np.abs(pp - tt)
        return {"mae": float(np.mean(err)), "rmse": float(np.sqrt(np.mean(err**2))), "max_error": float(np.max(err)),
                "count": int(len(pp))}

    return {"all_nodes": subset(p, t, None), "masked_nodes": subset(p, t, m)}
