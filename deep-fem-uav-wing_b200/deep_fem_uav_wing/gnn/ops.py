"""Tensor-level wrappers and autograd Functions over the C ABI (``libdfw_b200.so``).

PyTorch is plumbing here: it owns device memory, streams and the autograd tape; every
arithmetic step of the GraphSAGE path is a hand-written sm_100a kernel reached through
``_cabi.lib``.  CUDA tensors only - there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import dataclasses
import weakref
from collections import OrderedDict
from dataclasses import dataclass, field

import torch

from . import _cabi
from ._cabi import DFW_BF16, DFW_F32, EP_DROPOUT, EP_LAYERNORM, EP_RELU, EP_RESIDUAL, EP_SEED_IS_PTR, EP_TRANSPOSE_W, check, lib

_DTYPES = {torch.float32: DFW_F32, torch.bfloat16: DFW_BF16}
LAUNCH_COUNTER = {"kernels": 0}  # kernels launched through the C ABI (bench.py's gpu_launches)


class KernelProfiler:
    """Optional per-call CUDA-event timing of the C-ABI launches (bench.py's roofline pass).
    Events are recorded on the stream the kernels are launched on."""

    def __init__(self):
        self.records = []

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, b, nbytes, flops in self.records:
            r = out.setdefault(name, {"calls": 0, "ms": 0.0, "bytes": 0, "flops": 0})
            r["calls"] += 1
            r["ms"] += a.elapsed_time(b)
            r["bytes"] += nbytes
            r["flops"] += flops
        return out


PROFILER: KernelProfiler | None = None


class _prof:
    __slots__ = ("name", "nbytes", "flops", "a")

    def __init__(self, name, nbytes=0, flops=0):
        self.name, self.nbytes, self.flops = name, nbytes, flops

    def __enter__(self):
        if PROFILER is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if PROFILER is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            PROFILER.records.append((self.name, self.a, b, self.nbytes, self.flops))
        return False


def _esz(t) -> int:
    return 4 if t.dtype == torch.float32 else 2


def _dt(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"dfw_b200 supports float32 and bfloat16 activations, got {t.dtype}") from None


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what} must be a CUDA tensor (got device {t.device}): deep_fem_uav_wing.gnn is the B200-native "
            "implementation and has no CPU fallback."
        )


def _seed_arg(seed):
    """Dropout seed by value (python int) or by reference (1-element int64 CUDA tensor, read by the kernel at run
    time - what a captured CUDA graph needs to draw a fresh mask on every replay)."""
    if isinstance(seed, torch.Tensor):
        return seed.data_ptr(), EP_SEED_IS_PTR
    return int(seed) & 0xFFFFFFFFFFFFFFFF, 0


def _f32(t):
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ----------------------------------------------------------------------------------------------
# (a) CSR
# ----------------------------------------------------------------------------------------------
@dataclass
class CSRGraph:
    """Device-resident canonical CSR of an ``edge_index`` (by destination) and, lazily, its
    transpose (by source) for the backward pass."""

    edge_index: torch.Tensor | None
    num_nodes: int
    num_edges: int
    rowptr: torch.Tensor
    col: torch.Tensor
    inv_deg: torch.Tensor
    perm: torch.Tensor | None = None
    status: torch.Tensor | None = None
    rowptr_t: torch.Tensor | None = None
    col_t: torch.Tensor | None = None
    _pending: list = field(default_factory=list)
    skipped_faces: torch.Tensor | None = None
    status_t: torch.Tensor | None = None  # int32 [3] of dfw_csr_transpose ([2] = 1: the graph was not symmetric)
    plan: "AggPlan | None" = None         # block plan for dfw_sage_aggregate_tc (large-mesh bf16 inference)
    edge_count: torch.Tensor | None = None  # int64 [1] on the device: exact E of a graph built with faces_to_graph(sync=False)

    def transpose(self):
        if self.rowptr_t is None:
            if self.edge_index is None:
                raise RuntimeError("CSRGraph: transposed CSR was not pre-built and edge_index is gone")
            self.rowptr_t, self.col_t, self.status_t = csr_transpose_raw(self.edge_index, self.num_nodes, self.rowptr, self.col)
        return self.rowptr_t, self.col_t

    def check(self) -> None:
        """Synchronously validate (raises IndexError on out-of-range endpoints)."""
        bad = int(self.status[0].item())
        if bad:
            raise IndexError(f"edge_index has {bad} edge(s) with an endpoint outside [0, {self.num_nodes})")

    @property
    def max_degree(self) -> int:
        return int(self.status[1].item())


def csr_build_raw(edge_index: torch.Tensor, num_nodes: int, by_src: bool = False, want_perm: bool = True,
                  want_inv_deg: bool = True):
    _require_cuda(edge_index, "edge_index")
    if edge_index.dim() != 2 or edge_index.shape[0] != 2:
        raise ValueError(f"edge_index must have shape [2, E], got {tuple(edge_index.shape)}")
    if edge_index.dtype != torch.int64:
        raise TypeError(f"edge_index must be int64 (torch.long), got {edge_index.dtype}")
    ei = edge_index.contiguous()
    E, N = int(ei.shape[1]), int(num_nodes)
    if E >= 2**31 - 1 or N >= 2**31 - 1:
        raise ValueError("dfw_b200 uses int32 CSR indices: E and N must be < 2^31")
    dev = ei.device
    rowptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
    col = torch.empty(E, dtype=torch.int32, device=dev)
    perm = torch.empty(E, dtype=torch.int32, device=dev) if want_perm else None
    inv_deg = torch.empty(N, dtype=torch.float32, device=dev) if want_inv_deg else None
    status = torch.empty(2, dtype=torch.int32, device=dev)
    ws_bytes = lib.dfw_csr_ws_bytes(E, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof("csr_build", 16 * E + 4 * E + 4 * (N + 1)):
        check(lib.dfw_csr_build(ei.data_ptr(), E, N, int(by_src), rowptr.data_ptr(), _ptr(col), _ptr(perm), _ptr(inv_deg),
                                status.data_ptr(), ws.data_ptr(), ws_bytes, _stream(ei)))
    LAUNCH_COUNTER["kernels"] += 7 if E > 0 else 3
    return rowptr, col, perm, inv_deg, status


def csr_transpose_raw(edge_index: torch.Tensor, num_nodes: int, rowptr: torch.Tensor, col: torch.Tensor):
    """CSR by source for the backward gather (``dfw_csr_transpose``): a copy of the CSR by destination when the graph
    holds both directions of every edge (checked on the device), the general build otherwise."""
    ei = edge_index.contiguous()
    E, N, dev = int(ei.shape[1]), int(num_nodes), ei.device
    rowptr_t = torch.empty(N + 1, dtype=torch.int32, device=dev)
    col_t = torch.empty(E, dtype=torch.int32, device=dev)
    status = torch.empty(3, dtype=torch.int32, device=dev)
    ws_bytes = lib.dfw_csr_ws_bytes(E, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof("csr_transpose", 16 * E + 4 * E + 4 * (N + 1)):
        check(lib.dfw_csr_transpose(ei.data_ptr(), E, N, rowptr.data_ptr(), _ptr(col), rowptr_t.data_ptr(), _ptr(col_t),
                                    status.data_ptr(), ws.data_ptr(), ws_bytes, _stream(ei)))
    LAUNCH_COUNTER["kernels"] += 9 if E > 0 else 5
    return rowptr_t, col_t, status


def faces_to_graph(faces: torch.Tensor, num_nodes: int, node_ids: torch.Tensor | None = None, want_edge_index: bool = True,
                   sync: bool = True):
    """Triangle faces -> (CSRGraph, edge_index) on the device (``dfw_faces_to_csr``; reference
    ``_faces_to_edge_index``, ``dataset.py:26-63``).

    ``faces``: int64 [F,3] of node ids; ``node_ids``: int64 [N] ids in node order (``npz["node_id"]``,
    ``dataset.py:94``), or None when the faces already hold 0-based indices.  One 8-byte D2H read (the edge count).
    The returned ``edge_index`` is registered with the graph cache, so ``model(x, edge_index)`` does not rebuild.
    ``sync=False`` (inference graphs, ``want_edge_index=False``): no D2H read at all - ``col`` keeps its capacity of 6F entries
    (``rowptr`` delimits the valid ones), ``num_edges`` is the closed-surface estimate 3F (the kernels use it as a sizing hint
    only) and the exact count stays on the device in ``graph.edge_count`` - so a screening loop never waits for the GPU."""
    if not sync and want_edge_index:
        raise ValueError("faces_to_graph(sync=False) cannot size edge_index: pass want_edge_index=False")
    _require_cuda(faces, "faces")
    if faces.dtype != torch.int64:
        raise TypeError(f"faces must be int64, got {faces.dtype}")
    f = faces.reshape(-1, 3).contiguous()
    F, N, dev = int(f.shape[0]), int(num_nodes), f.device
    if 6 * F >= 2**31 - 1 or N >= 2**31 - 1:
        raise ValueError("dfw_b200 uses int32 CSR indices: 6F and N must be < 2^31")
    sorted_ids = id_perm = None
    if node_ids is not None:
        ids = node_ids.to(device=dev, dtype=torch.int64).contiguous()
        if ids.numel() != N:
            raise ValueError(f"node_ids has {ids.numel()} entries for {N} nodes")
        if N > 1 and not bool((ids[1:] > ids[:-1]).all()):  # Gmsh surface ids come sorted (fem.py:611); else sort once
            sorted_ids, id_perm = torch.sort(ids)
            id_perm = id_perm.contiguous()
        else:
            sorted_ids = ids
    cap = max(6 * F, 1)
    rowptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
    col = torch.empty(cap, dtype=torch.int32, device=dev)
    inv_deg = torch.empty(N, dtype=torch.float32, device=dev)
    ei = torch.empty(2, cap, dtype=torch.int64, device=dev) if want_edge_index else None
    nedges = torch.zeros(1, dtype=torch.int64, device=dev)
    status = torch.empty(3, dtype=torch.int32, device=dev)
    ws_bytes = lib.dfw_faces_ws_bytes(F, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof("faces_to_csr", 24 * F + 4 * (N + 1)):
        check(lib.dfw_faces_to_csr(f.data_ptr(), F, _ptr(sorted_ids), _ptr(id_perm), N, rowptr.data_ptr(), col.data_ptr(),
                                   inv_deg.data_ptr(), _ptr(ei), nedges.data_ptr(), status.data_ptr(), ws.data_ptr(), ws_bytes,
                                   _stream(f)))
    LAUNCH_COUNTER["kernels"] += 13
    if sync:
        E = int(nedges.item())
        col = col[:E]
    else:
        E = min(3 * F, cap)
    edge_index = ei[:, :E].contiguous() if ei is not None else None
    g = CSRGraph(edge_index, N, E, rowptr, col, inv_deg, None, status[:2])
    g.edge_count = nedges
    g.rowptr_t, g.col_t = rowptr, col  # both directions of every edge are present: the transpose is the graph itself
    g.skipped_faces = status[2:3]
    if edge_index is not None:
        register_graph(edge_index, g)
    return g, edge_index


def node_features(pos: torch.Tensor, normal: torch.Tensor, stress: torch.Tensor | None, global_params, normalize_pos=True,
                  log_scale=True):
    """``dfw_node_features``: x [N,10] and y [N,1] of ``build_graph_data`` (``dataset.py:129-151``) on the device."""
    import ctypes

    _require_cuda(pos, "pos")
    pos = pos.to(torch.float32).contiguous()
    normal = normal.to(torch.float32).contiguous()
    N, dev = int(pos.shape[0]), pos.device
    x = torch.empty(N, 10, dtype=torch.float32, device=dev)
    y = None
    if stress is not None:
        stress = stress.to(torch.float32).contiguous()
        y = torch.empty(N, 1, dtype=torch.float32, device=dev)
    gp = (ctypes.c_float * 4)(*[float(v) for v in global_params])
    ws_bytes = lib.dfw_node_features_ws_bytes(N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof("node_features", 72 * N):
        check(lib.dfw_node_features(pos.data_ptr(), normal.data_ptr(), _ptr(stress), gp, int(bool(normalize_pos)), int(bool(log_scale)),
                                    x.data_ptr(), _ptr(y), N, ws.data_ptr(), ws_bytes, _stream(pos)))
    LAUNCH_COUNTER["kernels"] += 2
    return x, y


def node_features_batched(pos, normal, stress, global_params, case_ptr, max_case_rows: int, normalize_pos=True, log_scale=True):
    """``dfw_node_features_batched``: features of B concatenated cases in one launch pair.  ``global_params`` fp32 [B,4] (scaled,
    ``dataset.py:122-127``) and ``case_ptr`` int64 [B+1] are DEVICE tensors; per-case min-max normalisation of ``pos``."""
    _require_cuda(pos, "pos")
    pos = pos.to(torch.float32).contiguous()
    normal = normal.to(torch.float32).contiguous()
    N, dev, B = int(pos.shape[0]), pos.device, int(case_ptr.numel()) - 1
    x = torch.empty(N, 10, dtype=torch.float32, device=dev)
    y = None
    if stress is not None:
        stress = stress.to(torch.float32).contiguous()
        y = torch.empty(N, 1, dtype=torch.float32, device=dev)
    ws_bytes = lib.dfw_node_features_batched_ws_bytes(B)
    ws = torch.empty(max(ws_bytes, 8), dtype=torch.uint8, device=dev)
    gp = global_params.to(device=dev, dtype=torch.float32).contiguous()
    with torch.cuda.device(dev), _prof("node_features", 72 * N):
        check(lib.dfw_node_features_batched(pos.data_ptr(), normal.data_ptr(), _ptr(stress), gp.data_ptr(), case_ptr.data_ptr(), B, int(max_case_rows),
                                            int(bool(normalize_pos)), int(bool(log_scale)), x.data_ptr(), _ptr(y), ws.data_ptr(), ws.numel(), _stream(pos)))
    LAUNCH_COUNTER["kernels"] += 2
    return x, y


_CSR_CACHE: "OrderedDict[tuple, CSRGraph]" = OrderedDict()
_CSR_CACHE_SIZE = 16  # loaders create a new edge_index tensor per step: a long LRU only pins dead batches' CSRs in HBM


def _cache_key(edge_index: torch.Tensor, num_nodes: int):
    return (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, edge_index.device.index, int(num_nodes))


def get_graph(edge_index: torch.Tensor, num_nodes: int, validate: bool | None = None, want_perm: bool = False) -> CSRGraph:
    """CSR for ``edge_index`` - built once per (tensor identity, version) and cached.

    ``validate``: True = synchronous range check now (one host sync); None/False = the count of bad
    endpoints stays on the device (``graph.check()`` reads it)."""
    key = _cache_key(edge_index, num_nodes)
    g = _CSR_CACHE.get(key)
    if g is not None and g.edge_index is edge_index:
        _CSR_CACHE.move_to_end(key)
        return g
    rowptr, col, perm, inv_deg, status = csr_build_raw(edge_index, num_nodes, by_src=False, want_perm=want_perm)
    g = CSRGraph(edge_index, int(num_nodes), int(edge_index.shape[1]), rowptr, col, inv_deg, perm, status)
    if validate:
        g.check()
    _CSR_CACHE[key] = g
    while len(_CSR_CACHE) > _CSR_CACHE_SIZE:
        _CSR_CACHE.popitem(last=False)
    return g


def register_graph(edge_index: torch.Tensor, graph: CSRGraph) -> None:
    """Let a loader attach a pre-built CSR to the ``edge_index`` tensor it hands to the model."""
    _CSR_CACHE[_cache_key(edge_index, graph.num_nodes)] = graph
    graph.edge_index = edge_index
    while len(_CSR_CACHE) > _CSR_CACHE_SIZE:
        _CSR_CACHE.popitem(last=False)


def clear_graph_cache() -> None:
    _CSR_CACHE.clear()


# ----------------------------------------------------------------------------------------------
# thin kernel wrappers (no autograd)
# ----------------------------------------------------------------------------------------------
def aggregate(rowptr, col, row_scale, x, addend=None):
    _require_cuda(x, "x")
    x = x.contiguous()
    out = torch.empty_like(x)
    N, H = x.shape
    E = col.shape[0]
    amin = (2 + (addend is not None)) * N * H * _esz(x) + 4 * E + 4 * (N + 1)
    with torch.cuda.device(x.device), _prof("aggregate", amin):
        check(lib.dfw_sage_aggregate(rowptr.data_ptr(), col.data_ptr(), _ptr(row_scale), x.data_ptr(),
                                     _ptr(addend.contiguous() if addend is not None else None), out.data_ptr(), N, E, H, _dt(x),
                                     _stream(x)))
    LAUNCH_COUNTER["kernels"] += 1
    return out


def aggregate_rows(rowptr, col, row_scale, x_ext, n_rows: int):
    """Mean / sum aggregation whose SOURCE tensor has more rows than there are output rows: ``rowptr`` describes ``n_rows``
    destination rows, ``col`` indexes ``x_ext [n_ext, H]`` (own rows followed by halo rows: ``gnn/partition.py``)."""
    _require_cuda(x_ext, "x")
    x_ext = x_ext.contiguous()
    H = x_ext.shape[1]
    E = col.shape[0]
    out = torch.empty(n_rows, H, dtype=x_ext.dtype, device=x_ext.device)
    amin = (n_rows + x_ext.shape[0]) * H * _esz(x_ext) + 4 * E + 4 * (n_rows + 1)
    with torch.cuda.device(x_ext.device), _prof("aggregate", amin):
        check(lib.dfw_sage_aggregate(rowptr.data_ptr(), _ptr(col) if E else None, _ptr(row_scale), x_ext.data_ptr(), None, out.data_ptr(), n_rows, E, H,
                                     _dt(x_ext), _stream(x_ext)))
    LAUNCH_COUNTER["kernels"] += 1
    return out


def aggregate_scaled(rowptr, col, src_scale, x, label="aggregate_bwd"):
    """``out[i] = sum_k src_scale[col[k]] * x[col[k]]`` (``dfw_sage_aggregate_scaled``)."""
    _require_cuda(x, "x")
    x = x.contiguous()
    out = torch.empty_like(x)
    N, H = x.shape
    E = col.shape[0]
    amin = 2 * N * H * _esz(x) + 4 * E + 4 * (N + 1) + 4 * N
    with torch.cuda.device(x.device), _prof(label, amin):
        check(lib.dfw_sage_aggregate_scaled(rowptr.data_ptr(), col.data_ptr(), src_scale.data_ptr(), x.data_ptr(), out.data_ptr(),
                                            N, E, H, _dt(x), _stream(x)))
    LAUNCH_COUNTER["kernels"] += 1
    return out


@dataclass
class AggPlan:
    """Block plan of a CSR for ``dfw_sage_aggregate_tc`` (per 128-row block: distinct source rows + a 16-bit slot per edge)."""

    num_nodes: int
    blk_meta: torch.Tensor
    plan_src: torch.Tensor
    plan_rec: torch.Tensor
    plan_slot: torch.Tensor
    status: torch.Tensor          # uint64-as-int64 [2] on the device: [0] max edges of a block, [1] total staged rows
    usable: bool | None = None    # resolved by ``check()`` (one 16-byte D2H read): the plan is structurally valid
    profitable: bool = True       # cleared by get_inference_graph for low-degree graphs, where the gather kernel is faster
    staged_rows_per_row: float | None = None

    def check(self) -> bool:
        if self.usable is None:
            st = self.status.cpu().tolist()
            self.usable = int(st[0]) <= int(lib.dfw_agg_plan_max_block_edges())
            self.staged_rows_per_row = float(st[1]) / max(self.num_nodes, 1)
        return self.usable


def build_agg_plan(rowptr: torch.Tensor, col: torch.Tensor, num_nodes: int) -> AggPlan:
    """``dfw_agg_plan_build``: one-time preparation of a graph for the tensor-core aggregation (3 launches, no host sync)."""
    import ctypes

    N, E, dev = int(num_nodes), int(col.shape[0]), rowptr.device
    nb, sc, tc_ = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
    check(lib.dfw_agg_plan_sizes(N, E, ctypes.byref(nb), ctypes.byref(sc), ctypes.byref(tc_)))
    nb, sc, tc_ = nb.value, sc.value, tc_.value
    blk_meta = torch.empty(max(4 * nb, 4), dtype=torch.int32, device=dev)
    plan_src = torch.empty(sc, dtype=torch.int32, device=dev)
    plan_rec = torch.empty(max(136 * nb, 8), dtype=torch.int16, device=dev)
    plan_slot = torch.empty(tc_, dtype=torch.int16, device=dev)
    status = torch.zeros(2, dtype=torch.int64, device=dev)
    ws = torch.empty(max(8 * nb, 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof("agg_plan_build", 8 * E + 4 * (N + 1)):
        check(lib.dfw_agg_plan_build(rowptr.data_ptr(), _ptr(col), N, E, blk_meta.data_ptr(), plan_src.data_ptr(), plan_rec.data_ptr(),
                                     plan_slot.data_ptr(), status.data_ptr(), ws.data_ptr(), ws.numel(), _stream(rowptr)))
    LAUNCH_COUNTER["kernels"] += 3
    return AggPlan(N, blk_meta, plan_src, plan_rec, plan_slot, status)


def aggregate_tc(plan: AggPlan, row_scale, x, num_edges: int = 0, n_rows: int | None = None):
    """``dfw_sage_aggregate_tc``: mean (``row_scale = inv_deg``) or sum (None) of neighbour rows, bf16, H in {64, 128, 256}.
    ``n_rows``: the plan describes ``n_rows`` destination rows whose sources index a LONGER tensor ``x`` (own rows followed by
    halo rows, ``gnn/partition.py``): a block's own rows are the first ``n_rows`` rows of ``x``, every other source is a halo row."""
    _require_cuda(x, "x")
    if x.dtype != torch.bfloat16:
        raise TypeError(f"aggregate_tc takes bfloat16 rows, got {x.dtype}")
    x = x.contiguous()
    N, H = x.shape
    if n_rows is not None:
        if n_rows > N:
            raise ValueError(f"n_rows = {n_rows} exceeds the {N} rows of x")
        N = int(n_rows)
    if N != plan.num_nodes:
        raise ValueError(f"plan was built for {plan.num_nodes} rows, x has {N}")
    out = torch.empty(N, H, dtype=x.dtype, device=x.device)
    amin = 2 * N * H * 2 + 4 * num_edges + 4 * (N + 1)
    with torch.cuda.device(x.device), _prof("aggregate_tc", amin):
        check(lib.dfw_sage_aggregate_tc(plan.blk_meta.data_ptr(), plan.plan_src.data_ptr(), plan.plan_rec.data_ptr(), plan.plan_slot.data_ptr(),
                                        _ptr(row_scale), x.data_ptr(), out.data_ptr(), N, H, DFW_BF16, _stream(x)))
    LAUNCH_COUNTER["kernels"] += 1
    return out


def locality_order(pos: torch.Tensor, edge_index: torch.Tensor, leaf: int = 128, max_sample_edges: int = 1 << 22, fine_leaf: int = 8) -> torch.Tensor:
    """Node relabelling that makes blocks of ``leaf`` consecutive rows spatially compact: ``new_id[old_id]`` (int64, on the
    device of ``pos``).  One-time graph preparation for the blocked aggregation (``dfw_sage_aggregate_tc`` stages the union
    of a block's neighbours: 4.2 rows per output row on the config-4 lattice in its native numbering, 2.75 in this order,
    13.7 in a random numbering).

    k-d ordering by recursive MEDIAN bisection: every segment of the current order longer than ``leaf`` is sorted along the
    axis of its largest extent - measured in hops, i.e. coordinates divided by the mean coordinate difference along the mesh
    edges, so element anisotropy (thin wing sections) does not bias the choice - and cut at the multiple of ``leaf`` nearest
    its middle.  Splitting by RANK adapts to the node density (a Morton code of quantised coordinates does not: where the
    thickness tapers to zero whole columns fall into one cell).  The bisection continues INSIDE the leaves (exact halves, down
    to ``fine_leaf`` rows), so the order within a block is spatially coherent too and does not depend on the numbering the
    caller happened to use: a block's halo rows then sit in a few short runs of their neighbour blocks (on config 4 a randomly
    numbered mesh aggregated 22 % slower than the natively numbered one after relabelling until this was added - same staged
    rows, worse DRAM page locality).  log2(N / fine_leaf) rounds of two stable sorts, all on the device; the coordinates are
    the model's own input features ``x[:, :3]`` (normalised positions, reference ``dataset.py:130-145``), so the permutation
    is applied to the 10-wide input and undone on the 1-wide output."""
    n = int(pos.shape[0])
    dev = pos.device
    if n <= leaf:
        return torch.arange(n, device=dev)
    p = pos[:, :3].to(torch.float32)
    E = int(edge_index.shape[1])
    if E > 0:
        stride = max(1, E // max_sample_edges)
        es = edge_index[:, ::stride]
        hop = (p[es[0]] - p[es[1]]).abs().mean(dim=0)
        hop = torch.where(hop > 0, hop, torch.ones_like(hop))
        p = p / hop
    order = torch.arange(n, device=dev)
    bounds = torch.tensor([0, n], device=dev, dtype=torch.int64)
    while True:
        seg_len = bounds[1:] - bounds[:-1]
        big = seg_len > fine_leaf
        if not bool(big.any()):
            break
        nseg = int(seg_len.numel())
        seg = torch.repeat_interleave(torch.arange(nseg, device=dev), seg_len, output_size=n)
        cur = p[order]
        idx3 = seg[:, None].expand(-1, 3)
        mn = torch.full((nseg, 3), float("inf"), device=dev).scatter_reduce_(0, idx3, cur, "amin")
        mx = torch.full((nseg, 3), float("-inf"), device=dev).scatter_reduce_(0, idx3, cur, "amax")
        ax = torch.argmax(mx - mn, dim=1)
        coord = cur.gather(1, ax[seg][:, None]).squeeze(1)
        i1 = torch.argsort(coord, stable=True)
        i2 = torch.argsort(seg[i1], stable=True)
        order = order[i1[i2]]
        a, b = bounds[:-1][big], bounds[1:][big]
        half = (b - a) // 2
        half = torch.where(b - a > leaf, (half + leaf - 1) // leaf * leaf, half.clamp_min(1))  # block boundaries stay multiples of `leaf`
        mid = torch.minimum(a + half, b - 1)
        bounds = torch.sort(torch.cat([bounds, mid])).values
    new_id = torch.empty(n, dtype=torch.int64, device=dev)
    new_id[order] = torch.arange(n, device=dev)
    return new_id


TC_AGG_WIDTHS = (64, 128, 256)
TC_AGG_MIN_NODES = 1 << 17        # below this the gather kernel is launch / L2 bound anyway and the plan is not worth building
TC_AGG_REORDER_ABOVE = 3.2        # staged rows per output row above which a k-d relabelling is tried
TC_AGG_MIN_REUSE = 3.0            # edges per staged row below which the gather kernel wins (measured, tools/aggtc_small.py: surface
                                  # meshes, degree 6 / 3.0 staged = 2.0: gather 46 us vs block 54 us; tet, 13 / 3.35 = 3.9: 68 vs 55 us)


def aggregate_mean(graph: "CSRGraph", x):
    """Mean aggregation over ``graph``: the tensor-core block kernel when the graph carries a usable plan and the rows
    qualify (bf16, H in 64/128/256), the gather kernel otherwise.  Both are deterministic.  For finite inputs they differ by
    the order and rounding of the fp32 additions only (bounded relative to the sum of |terms|, not to the result: under
    cancellation the bound allows more than one bf16 ulp of the result).  A NaN or Inf row poisons only the rows that read it in the gather kernel,
    but every row of each 128-row block that stages it in the block kernel."""
    pl = graph.plan
    if pl is not None and pl.usable and pl.profitable and x.dtype == torch.bfloat16 and x.shape[1] in TC_AGG_WIDTHS:
        return aggregate_tc(pl, graph.inv_deg, x, graph.num_edges)
    return aggregate(graph.rowptr, graph.col, graph.inv_deg, x)


@dataclass
class InferenceGraph:
    """Graph prepared for large-mesh inference: CSR (+ block plan) of the possibly RELABELLED nodes.
    ``order[new] = old`` permutes input rows (``x.index_select(0, order)``), ``new_id[old] = new`` restores outputs."""

    graph: CSRGraph
    new_id: torch.Tensor | None = None
    order: torch.Tensor | None = None
    staged_rows_per_row_given: float | None = None
    staged_rows_per_row: float | None = None


_INF_CACHE: "OrderedDict[tuple, InferenceGraph]" = OrderedDict()


_SEEN_MESHES: "OrderedDict[int, weakref.ref]" = OrderedDict()


def static_mesh_seen_before(edge_index: torch.Tensor) -> bool:
    """True from the SECOND call with the same ``edge_index`` tensor object.  Preparing a mesh for the block aggregation (plan,
    k-d relabelling: ~100 ms for 2 M nodes, two small D2H reads) pays only when the mesh is used again; a screening loop that
    sees every graph once (BASELINE.json config 5) must not pay it per launch."""
    k = id(edge_index)
    r = _SEEN_MESHES.get(k)
    if r is not None and r() is edge_index:
        _SEEN_MESHES.move_to_end(k)
        return True
    _SEEN_MESHES[k] = weakref.ref(edge_index)
    while len(_SEEN_MESHES) > 16:
        _SEEN_MESHES.popitem(last=False)
    return False


def get_inference_graph(edge_index: torch.Tensor, num_nodes: int, pos: torch.Tensor | None = None, reorder: str = "auto") -> InferenceGraph:
    """One-time preparation of a large static mesh for bf16 inference (BASELINE.json config 4): CSR, block plan for
    ``dfw_sage_aggregate_tc`` and - ``reorder`` = 'auto' (when the given numbering stages more than
    ``TC_AGG_REORDER_ABOVE`` rows per output row and coordinates are available), 'always' or 'never' - the k-d node
    relabelling of ``locality_order``.  Cached per ``edge_index`` tensor.  Costs two 16-byte D2H reads (plan statistics)."""
    key = _cache_key(edge_index, num_nodes) + (reorder, pos is not None)
    ig = _INF_CACHE.get(key)
    if ig is not None and ig.graph is not None and (ig.graph.edge_index is edge_index or ig.new_id is not None):
        _INF_CACHE.move_to_end(key)
        return ig
    # the plan lives on a COPY of the cached CSR: ops.get_graph(edge_index) - what every other caller of this mesh gets -
    # must stay a plain graph (SageConvFn takes the block kernel whenever its graph carries a profitable plan)
    g = dataclasses.replace(get_graph(edge_index, num_nodes), _pending=[])
    g.plan = build_agg_plan(g.rowptr, g.col, num_nodes)
    ok = g.plan.check()
    ig = InferenceGraph(g, None, None, g.plan.staged_rows_per_row, g.plan.staged_rows_per_row)
    want = reorder == "always" or (reorder == "auto" and (not ok or g.plan.staged_rows_per_row > TC_AGG_REORDER_ABOVE))
    if want and pos is not None and num_nodes > 128:
        new_id = locality_order(pos, edge_index)
        ei2 = new_id[edge_index]
        rowptr, col, _, inv_deg, status = csr_build_raw(ei2, num_nodes, want_perm=False)
        g2 = CSRGraph(ei2, int(num_nodes), int(ei2.shape[1]), rowptr, col, inv_deg, None, status)
        g2.plan = build_agg_plan(rowptr, col, num_nodes)
        if g2.plan.check() and (not ok or g2.plan.staged_rows_per_row < 0.9 * g.plan.staged_rows_per_row):
            order = torch.empty_like(new_id)
            order[new_id] = torch.arange(num_nodes, device=new_id.device)
            ig = InferenceGraph(g2, new_id, order, g.plan.staged_rows_per_row, g2.plan.staged_rows_per_row)
    pl = ig.graph.plan
    if pl is not None and pl.usable and ig.graph.num_edges / max(num_nodes, 1) < TC_AGG_MIN_REUSE * pl.staged_rows_per_row:
        pl.profitable = False  # low-degree graph: every staged row would serve too few edges; aggregate_mean takes the gather kernel
    _INF_CACHE[key] = ig
    while len(_INF_CACHE) > 4:
        _INF_CACHE.popitem(last=False)
    return ig


def cfg4_aggregation_paths(edge_index, num_nodes, pos, x):
    """The aggregation paths bench.py times on BASELINE.json config 4: name -> (zero-argument callable running ONE mean
    aggregation of ``x`` over the graph, info dict).  One-time graph preparation happens here, outside the callables."""
    import time

    g = get_graph(edge_index, num_nodes)
    paths = {"gather": (lambda: aggregate(g.rowptr, g.col, g.inv_deg, x), {"what": "dfw_sage_aggregate on the CSR in the given numbering"})}
    if x.dtype == torch.bfloat16 and x.shape[1] in TC_AGG_WIDTHS:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plan = build_agg_plan(g.rowptr, g.col, num_nodes)
        ok = plan.check()
        t_plan = time.perf_counter() - t0
        if ok:
            paths["tensor_core_blocks"] = (lambda: aggregate_tc(plan, g.inv_deg, x, g.num_edges),
                                           {"what": "dfw_sage_aggregate_tc, given numbering", "staged_rows_per_row": round(plan.staged_rows_per_row, 3),
                                            "one_time_plan_ms": round(t_plan * 1e3, 2)})
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ig = get_inference_graph(edge_index, num_nodes, pos=pos, reorder="auto")
        torch.cuda.synchronize()
        t_prep = time.perf_counter() - t0
        if ig.order is not None:
            xp = x.index_select(0, ig.order)  # in the model the permutation is applied to the 10-wide input, not per layer
            g2 = ig.graph
            paths["tensor_core_blocks_kd_order"] = (
                lambda: aggregate_tc(g2.plan, g2.inv_deg, xp, g2.num_edges),
                {"what": "dfw_sage_aggregate_tc after the one-time k-d relabelling of the nodes (ops.locality_order, device)",
                 "staged_rows_per_row": round(ig.staged_rows_per_row, 3), "staged_rows_per_row_given_numbering": round(ig.staged_rows_per_row_given, 3),
                 "one_time_relabel_csr_plan_ms": round(t_prep * 1e3, 2)})
    return paths


def linear_fwd(a1, w1, a2=None, w2=None, bias=None, ln=None, eps=1e-5, relu=False, residual=None, dropout_p=0.0, seed=0,
               save_pre=False, rowdot=None, want_out=True, transpose_w=False, label="linear_fwd", out_bf16=False):
    """See ``dfw_linear_fwd``.  ``ln`` = (gamma, beta); ``rowdot`` = (w fp32 [Hout], b fp32 [1] or None).
    ``transpose_w``: ``w1``/``w2`` are ``[k, Hout]`` (a forward layer's weights used by its input gradient).
    ``out_bf16``: fp32 tiny-K linear whose result is stored as bf16 (``DFW_EP_OUT_BF16``: the encoder's first layer in bf16 mode)."""
    _require_cuda(a1, "input")
    N, k1 = a1.shape
    dev, dt = a1.device, a1.dtype
    flags = 0
    if transpose_w:
        Hout = w1.shape[1]
        k2_ = 0 if a2 is None else a2.shape[1]
        ptrs_ok = all(t is None or t.data_ptr() % 16 == 0 for t in (a1, a2, residual))
        if ptrs_ok and lib.dfw_linear_tc_eligible(N, Hout, k1, k2_, _dt(a1)):
            flags |= EP_TRANSPOSE_W  # the transposition rides in the weight-preparation launch
        else:
            w1 = w1.t().contiguous()
            w2 = w2.t().contiguous() if w2 is not None else None
    else:
        Hout = w1.shape[0]
    if relu:
        flags |= EP_RELU
    if ln is not None:
        flags |= EP_LAYERNORM
    if residual is not None:
        flags |= EP_RESIDUAL
    seed_v, seed_flag = _seed_arg(seed)
    if dropout_p > 0.0:
        flags |= EP_DROPOUT | seed_flag
    if out_bf16:
        flags |= _cabi.EP_OUT_BF16
    out = torch.empty(N, Hout, dtype=torch.bfloat16 if out_bf16 else dt, device=dev) if want_out else None
    pre = torch.empty(N, Hout, dtype=dt, device=dev) if save_pre else None
    stats = torch.empty(N, 2, dtype=torch.float32, device=dev) if (save_pre and ln is not None) else None
    rd_out = torch.empty(N, dtype=torch.float32, device=dev) if rowdot is not None else None
    k2 = 0 if a2 is None else a2.shape[1]
    es = _esz(a1)
    nbytes = N * (k1 + k2) * es + (N * Hout * es if (residual is not None and residual is not a2) else 0) \
        + N * Hout * es * (int(want_out) + int(save_pre)) + (8 * N if stats is not None else 0) + (4 * N if rowdot is not None else 0) \
        + Hout * (k1 + k2) * es
    ws_bytes = lib.dfw_linear_ws_bytes(Hout, k1, k2, _dt(a1))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof(label, nbytes, 2 * N * Hout * (k1 + k2)):
        check(lib.dfw_linear_fwd(
            a1.data_ptr(), w1.data_ptr(), k1, _ptr(a2), _ptr(w2), 0 if a2 is None else a2.shape[1], _ptr(bias),
            _ptr(ln[0]) if ln is not None else None, _ptr(ln[1]) if ln is not None else None, float(eps), _ptr(residual),
            float(dropout_p), seed_v, _ptr(out), _ptr(pre), _ptr(stats),
            _ptr(rowdot[0]) if rowdot is not None else None, _ptr(rowdot[1]) if rowdot is not None else None, _ptr(rd_out),
            N, Hout, flags, _dt(a1), ws.data_ptr(), ws_bytes, _stream(a1)))
    LAUNCH_COUNTER["kernels"] += 1
    return out, pre, stats, rd_out


def epilogue_bwd(g_out, N, Hout, dtype_like, *, g_rowdot=None, rowdot_w=None, pre=None, stats=None, act=None, ln=None,
                 relu=False, dropout_p=0.0, seed=0, want_bias_grad=False, want_param_grads=True):
    """``dfw_epilogue_bwd``.  ``want_param_grads=False``: the LayerNorm affine and row-dot parameter gradients come back as
    None and, with ``want_bias_grad=False``, the kernel skips its column pass (only ``g_y`` is computed)."""
    dev = dtype_like.device
    seed_v, seed_flag = _seed_arg(seed)
    flags = (EP_RELU if relu else 0) | (EP_LAYERNORM if ln is not None else 0) | ((EP_DROPOUT | seed_flag) if dropout_p > 0.0 else 0)
    g_y = torch.empty(N, Hout, dtype=dtype_like.dtype, device=dev)
    dgamma = dbeta = d_rw = d_rb = None
    if ln is not None and want_param_grads:
        dgamma = torch.empty(Hout, dtype=torch.float32, device=dev)
        dbeta = torch.empty(Hout, dtype=torch.float32, device=dev)
    if g_rowdot is not None and want_param_grads:
        d_rw = torch.empty(Hout, dtype=torch.float32, device=dev)
        d_rb = torch.empty(1, dtype=torch.float32, device=dev)
    d_bias = torch.empty(Hout, dtype=torch.float32, device=dev) if want_bias_grad else None
    ws_bytes = lib.dfw_epilogue_bwd_ws_bytes(N, Hout)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    es = 4 if dtype_like.dtype == torch.float32 else 2
    nbytes = N * Hout * es * (1 + int(g_out is not None) + int(pre is not None) + int(act is not None)) + (8 * N if stats is not None else 0)
    with torch.cuda.device(dev), _prof("epilogue_bwd", nbytes):
        check(lib.dfw_epilogue_bwd(
            _ptr(g_out), _ptr(g_rowdot), _ptr(rowdot_w), _ptr(pre), _ptr(stats), _ptr(act),
            _ptr(ln[0]) if ln is not None else None, _ptr(ln[1]) if ln is not None else None, float(dropout_p),
            seed_v, g_y.data_ptr(), _ptr(dgamma), _ptr(dbeta), _ptr(d_rw), _ptr(d_rb), _ptr(d_bias), N, Hout, flags,
            _DTYPES[dtype_like.dtype], ws.data_ptr(), ws_bytes, _stream(dtype_like)))
    LAUNCH_COUNTER["kernels"] += 2 if (dgamma is not None or d_rw is not None or want_bias_grad) else 1
    return g_y, dgamma, dbeta, d_rw, d_rb, d_bias


def linear_bwd_input(g_y, w, row_scale=None, addend=None):
    N, Hout = g_y.shape
    K = w.shape[1]
    g_a = torch.empty(N, K, dtype=g_y.dtype, device=g_y.device)
    nbytes = (N * Hout + N * K * (1 + int(addend is not None)) + Hout * K) * _esz(g_y)
    ws_bytes = lib.dfw_linear_ws_bytes(K, Hout, 0, _dt(g_y))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=g_y.device)
    with torch.cuda.device(g_y.device), _prof("linear_bwd_input", nbytes, 2 * N * Hout * K):
        check(lib.dfw_linear_bwd_input(g_y.data_ptr(), w.data_ptr(), _ptr(row_scale), _ptr(addend), g_a.data_ptr(), N, Hout, K,
                                       _dt(g_y), ws.data_ptr(), ws_bytes, _stream(g_y)))
    LAUNCH_COUNTER["kernels"] += 1
    return g_a


def linear_bwd_weight(g_y, a1, a2=None, want_bias=True):
    N, Hout = g_y.shape
    k1 = a1.shape[1]
    k2 = a2.shape[1] if a2 is not None else 0
    dev = g_y.device
    dw1 = torch.empty(Hout, k1, dtype=torch.float32, device=dev)
    dw2 = torch.empty(Hout, k2, dtype=torch.float32, device=dev) if a2 is not None else None
    db = torch.empty(Hout, dtype=torch.float32, device=dev) if want_bias else None
    ws_bytes = lib.dfw_linear_bwd_weight_ws_bytes(N, Hout, k1, k2)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    nbytes = N * (Hout + k1 + k2) * _esz(g_y) + 4 * Hout * (k1 + k2)
    with torch.cuda.device(dev), _prof("linear_bwd_weight", nbytes, 2 * N * Hout * (k1 + k2)):
        check(lib.dfw_linear_bwd_weight(g_y.data_ptr(), a1.data_ptr(), k1, _ptr(a2), k2, dw1.data_ptr(), _ptr(dw2), _ptr(db), N,
                                        Hout, _dt(g_y), 0, ws.data_ptr(), ws_bytes, _stream(g_y)))
    LAUNCH_COUNTER["kernels"] += 2
    return dw1, dw2, db


def stress_metrics(pred, target, mask=None, log_scale=True) -> torch.Tensor:
    """``dfw_stress_metrics``: 8 doubles on the device - [mae, rmse, max_error, count] for all nodes, then for the
    masked nodes (``compute_metrics``, reference ``model.py:156-216``).  No host synchronisation.  When the dtypes of
    ``pred`` and ``target`` differ, both are read in fp32: rounding an fp32 target to bf16 before ``expm1`` would cost up
    to 2^-8 relative in log space."""
    _require_cuda(pred, "pred")
    p, t = pred.detach(), target.detach()
    if p.dtype != t.dtype:
        p, t = p.float(), t.float()
    p, t = p.contiguous(), t.contiguous()
    N = p.shape[0] if p.dim() > 0 else 1
    C = p.numel() // max(N, 1) if N > 0 else 1
    m = None
    if mask is not None:
        m = mask.detach().reshape(-1).contiguous()
        m = m.view(torch.uint8) if m.dtype == torch.bool else m.to(torch.uint8)
        if m.numel() != N:
            raise ValueError(f"mask has {m.numel()} entries for {N} rows")
    result = torch.empty(8, dtype=torch.float64, device=p.device)
    ws_bytes = lib.dfw_stress_metrics_ws_bytes(N, C)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    with torch.cuda.device(p.device), _prof("stress_metrics", 2 * N * C * _esz(p) + (N if m is not None else 0)):
        check(lib.dfw_stress_metrics(p.data_ptr(), t.data_ptr(), _ptr(m), N, max(C, 1), int(bool(log_scale)), _dt(p),
                                     result.data_ptr(), ws.data_ptr(), ws_bytes, _stream(p)))
    LAUNCH_COUNTER["kernels"] += 1
    return result


def vertex_normals(pos: torch.Tensor, faces: torch.Tensor):
    """``dfw_vertex_normals``: area-weighted vertex normals fp32 [N,3] of a triangulated surface (reference ``fem.py:390-424``)
    and an int32 [1] device count of the faces skipped for an index outside [0, N).  ``faces`` int64 [F,3] of 0-based rows.
    Deterministic (ascending incidence order, no float atomics) and without host synchronisation."""
    _require_cuda(pos, "pos")
    _require_cuda(faces, "faces")
    if faces.dtype != torch.int64:
        raise TypeError(f"faces must be int64, got {faces.dtype}")
    pos = pos.to(torch.float32).contiguous()
    f = faces.reshape(-1, 3).contiguous()
    N, F, dev = int(pos.shape[0]), int(f.shape[0]), pos.device
    if 3 * F >= 2**31 - 1 or N >= 2**31 - 1:
        raise ValueError("dfw_vertex_normals uses int32 incidence lists: 3F and N must be < 2^31")
    normal = torch.empty(N, 3, dtype=torch.float32, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    ws_bytes = lib.dfw_vertex_normals_ws_bytes(F, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev), _prof("vertex_normals", 24 * F + 24 * N):
        check(lib.dfw_vertex_normals(pos.data_ptr(), N, f.data_ptr(), F, normal.data_ptr(), status.data_ptr(), ws.data_ptr(), ws_bytes,
                                     _stream(pos)))
    LAUNCH_COUNTER["kernels"] += 9 if F > 0 else 4
    return normal, status


def _case_ptr_arg(case_ptr: torch.Tensor, device, what: str) -> tuple[torch.Tensor, int]:
    if case_ptr.dtype != torch.int64 or case_ptr.device != device:
        raise TypeError(f"case_ptr must be an int64 tensor on the device of {what}")
    cp = case_ptr.contiguous()
    B = int(cp.numel()) - 1
    if B < 0:
        raise ValueError("case_ptr needs at least one entry")
    return cp, B


def _case_inputs(pred, pos, case_ptr, mask):
    """Checked, contiguous arguments of the per-case reductions over the model output: (pred, pos, case_ptr, mask, N, B)."""
    _require_cuda(pred, "pred")
    p = pred.detach().contiguous()
    N = int(p.shape[0]) if p.dim() > 0 else 1
    if p.numel() != N:
        raise ValueError(f"pred must be [N] or [N,1], got {tuple(pred.shape)}")
    pos = pos.to(torch.float32).contiguous()
    if tuple(pos.shape) != (N, 3):
        raise ValueError(f"pos must be [{N}, 3], got {tuple(pos.shape)}")
    cp, B = _case_ptr_arg(case_ptr, p.device, "pred")
    m = None
    if mask is not None:
        m = mask.detach().reshape(-1).contiguous()
        m = m.view(torch.uint8) if m.dtype == torch.bool else m.to(torch.uint8)
        if m.numel() != N:
            raise ValueError(f"mask has {m.numel()} entries for {N} rows")
    return p, pos, cp, m, N, B


def case_stress_summary(pred, pos, case_ptr, mask=None, root_band: float = 0.05, allowable_pa: float | None = None,
                        log_scale: bool = True) -> torch.Tensor:
    """``dfw_case_stress_summary``: float64 [B,8] on the device, one record per case of ``case_ptr`` (int64 [B+1], device):
    [rows, screened rows, max stress, its row within the case (-1: none), mean stress, max stress over all rows,
    screened rows above ``allowable_pa``, non-finite stresses].  Screened rows are ``mask`` (uint8/bool [N]) or, without
    it, ``pos_y > root_band * (max_y - min_y)`` of the case.  ``pred`` [N] or [N,1], fp32 or bf16, ``log1p(stress)`` when
    ``log_scale``.  Deterministic and independent of how cases are batched; no host synchronisation."""
    p, pos, cp, m, N, B = _case_inputs(pred, pos, case_ptr, mask)
    out = torch.empty(max(B, 0), 8, dtype=torch.float64, device=p.device)
    ws_bytes = lib.dfw_case_stress_summary_ws_bytes(N, B)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    allow = float(allowable_pa) if allowable_pa is not None else 0.0
    with torch.cuda.device(p.device), _prof("case_stress_summary", N * (_esz(p) + 12 + (1 if m is not None else 0)) + 8 * (B + 1) + 64 * B):
        check(lib.dfw_case_stress_summary(p.data_ptr(), _dt(p), pos.data_ptr(), _ptr(m), cp.data_ptr(), B, N, float(root_band), allow,
                                          int(bool(log_scale)), out.data_ptr(), ws.data_ptr(), ws_bytes, _stream(p)))
    LAUNCH_COUNTER["kernels"] += (3 if m is not None else 4) if B > 0 else 0
    return out


def case_ks_seed(pred, pos, case_ptr, mask=None, root_band: float = 0.05, rho: float = 100.0):
    """``dfw_case_ks_seed``: a smooth per-case peak of ``pred`` (log1p of the stress) and its gradient, on the device.

    Per case b, S_b is the set ``case_stress_summary`` takes ``max_stress_pa`` over (screened rows - ``mask`` or the root
    band - whose fp32 stress is finite).  With ``m_b = max u`` and ``s_b = sum exp(rho (u - m_b))`` over S_b, returns
    float64 [B,2] ``[KS_b = m_b + ln(s_b) / rho, |S_b|]`` (``[0, 0]`` for an empty set) and the seed fp32 [N]
    ``w = exp(rho (u - m_b)) / s_b`` on S_b, 0 elsewhere (``dKS_b / du``).  ``max u <= KS_b <= max u + ln|S_b| / rho``.
    Deterministic and independent of how cases are batched; no host synchronisation."""
    if not rho > 0.0 or rho == float("inf"):
        raise ValueError(f"rho must be positive and finite, got {rho}")
    p, pos, cp, m, N, B = _case_inputs(pred, pos, case_ptr, mask)
    out = torch.empty(max(B, 0), 2, dtype=torch.float64, device=p.device)
    seed = torch.empty(N, dtype=torch.float32, device=p.device)
    ws_bytes = lib.dfw_case_stress_summary_ws_bytes(N, B)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    with torch.cuda.device(p.device), _prof("case_ks_seed", N * (2 * _esz(p) + 2 * (12 if m is None else 1) + 4) + 8 * (B + 1) + 16 * B):
        check(lib.dfw_case_ks_seed(p.data_ptr(), _dt(p), pos.data_ptr(), _ptr(m), cp.data_ptr(), B, N, float(root_band), float(rho),
                                   out.data_ptr(), seed.data_ptr(), ws.data_ptr(), ws_bytes, _stream(p)))
    LAUNCH_COUNTER["kernels"] += (4 if m is not None else 5) if B > 0 else 0
    return out, seed


def case_column_sums(a, case_ptr, c0: int, nc: int) -> torch.Tensor:
    """``dfw_case_column_sums``: float64 [B,nc], the sums over each case's rows of columns ``c0 .. c0+nc-1`` of the fp32 [N,C]
    ``a`` (fp64, fixed order: independent of how cases are batched).  The screener passes the input gradient with
    ``c0 = 6, nc = 4``."""
    _require_cuda(a, "a")
    if a.dtype != torch.float32 or a.dim() != 2:
        raise TypeError(f"case_column_sums takes a float32 [N, C] tensor, got {a.dtype} {tuple(a.shape)}")
    a = a.detach().contiguous()
    N, C = int(a.shape[0]), int(a.shape[1])
    cp, B = _case_ptr_arg(case_ptr, a.device, "a")
    out = torch.empty(max(B, 0), int(nc), dtype=torch.float64, device=a.device)
    ws_bytes = lib.dfw_case_stress_summary_ws_bytes(N, B)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=a.device)
    with torch.cuda.device(a.device), _prof("case_column_sums", 4 * N * C + 8 * (B + 1) + 8 * B * int(nc)):
        check(lib.dfw_case_column_sums(a.data_ptr(), N, C, int(c0), int(nc), cp.data_ptr(), B, out.data_ptr(), ws.data_ptr(), ws_bytes,
                                       _stream(a)))
    LAUNCH_COUNTER["kernels"] += 1 + 2 * ((int(nc) + 4) // 5) if (B > 0 and nc > 0) else 0
    return out


def cast(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    if t.dtype == dtype:
        return t.contiguous()
    src = t.contiguous()
    dst = torch.empty_like(src, dtype=dtype)
    with torch.cuda.device(t.device):
        check(lib.dfw_cast(src.data_ptr(), _DTYPES[src.dtype], dst.data_ptr(), _DTYPES[dtype], src.numel(), _stream(src)))
    LAUNCH_COUNTER["kernels"] += 1
    return dst


class CastFn(torch.autograd.Function):
    """dtype conversion that stays on the autograd tape (bf16 activations <-> fp32 boundary)."""

    @staticmethod
    def forward(ctx, t, dtype):
        ctx.src_dtype = t.dtype
        return cast(t, dtype)

    @staticmethod
    def backward(ctx, g):
        return cast(g, ctx.src_dtype), None


def cast_ad(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    return t if t.dtype == dtype else CastFn.apply(t, dtype)


def _w(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """Weight in the compute dtype (detached; fp32 master weights stay in the Parameter)."""
    return cast(t.detach(), dtype)


def _grad_to(param: torch.Tensor, g):
    if g is None:
        return None
    return g if g.dtype == param.dtype else g.to(param.dtype)


def sage_layer_fwd(graph: "CSRGraph", x, w_l, b_l, w_r, ln=None, eps=1e-5, dropout_p=0.0, seed=0, residual=True, save=True):
    """One-call SAGE layer forward (``dfw_sage_layer_fwd``): ``h + dropout(relu(LayerNorm(lin_l(mean) + lin_r(h))))`` with
    ``ln = (gamma, beta)``, or the bare ``SAGEConv`` with ``ln = None``.  Returns ``(out, agg, pre, stats)``."""
    _require_cuda(x, "x")
    x = x.contiguous()
    N, Hin = x.shape
    Hout = w_l.shape[0]
    dev, dt = x.device, x.dtype
    seed_v, seed_flag = _seed_arg(seed)
    flags = 0
    if ln is not None:
        flags |= EP_LAYERNORM | EP_RELU | (EP_RESIDUAL if residual else 0) | ((EP_DROPOUT | seed_flag) if dropout_p > 0.0 else 0)
    agg = torch.empty_like(x)
    out = torch.empty(N, Hout, dtype=dt, device=dev)
    pre = torch.empty(N, Hout, dtype=dt, device=dev) if (save and ln is not None) else None
    stats = torch.empty(N, 2, dtype=torch.float32, device=dev) if (save and ln is not None) else None
    ws_bytes = lib.dfw_sage_layer_fwd_ws_bytes(N, Hin, Hout, _dt(x))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.dfw_sage_layer_fwd(graph.rowptr.data_ptr(), graph.col.data_ptr(), graph.inv_deg.data_ptr(), x.data_ptr(),
                                     w_l.data_ptr(), _ptr(b_l), w_r.data_ptr(), _ptr(ln[0]) if ln else None, _ptr(ln[1]) if ln else None,
                                     float(eps), float(dropout_p), seed_v, flags, agg.data_ptr(), _ptr(pre), _ptr(stats), out.data_ptr(),
                                     N, graph.num_edges, Hin, Hout, _dt(x), ws.data_ptr(), ws_bytes, _stream(x)))
    LAUNCH_COUNTER["kernels"] += 2
    return out, agg, pre, stats


def sage_layer_bwd(graph: "CSRGraph", x, agg, pre, stats, w_l, w_r, ln, g_out, dropout_p=0.0, seed=0, residual=True,
                   want_input_grad=True, has_bias=True):
    """One-call SAGE layer backward (``dfw_sage_layer_bwd``).  Returns ``(g_x, dw_l, db_l, dw_r, dgamma, dbeta)``."""
    g_out = g_out.contiguous()
    N, Hout = g_out.shape
    Hin = x.shape[1]
    dev = x.device
    seed_v, seed_flag = _seed_arg(seed)
    flags = 0
    if ln is not None:
        flags |= EP_LAYERNORM | EP_RELU | (EP_RESIDUAL if residual else 0) | ((EP_DROPOUT | seed_flag) if dropout_p > 0.0 else 0)
    f32 = dict(dtype=torch.float32, device=dev)
    g_x = torch.empty(N, Hin, dtype=x.dtype, device=dev) if want_input_grad else None
    dw_l, dw_r = torch.empty(Hout, Hin, **f32), torch.empty(Hout, Hin, **f32)
    db_l = torch.empty(Hout, **f32) if has_bias else None
    dgamma = torch.empty(Hout, **f32) if ln is not None else None
    dbeta = torch.empty(Hout, **f32) if ln is not None else None
    rp_t, col_t = graph.transpose() if want_input_grad else (None, None)
    ws_bytes = lib.dfw_sage_layer_bwd_ws_bytes(N, Hin, Hout, _dt(x), int(want_input_grad))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.dfw_sage_layer_bwd(_ptr(rp_t), _ptr(col_t), graph.inv_deg.data_ptr(), x.data_ptr(), agg.data_ptr(), _ptr(pre), _ptr(stats),
                                     w_l.data_ptr(), w_r.data_ptr(), _ptr(ln[0]) if ln else None, _ptr(ln[1]) if ln else None,
                                     g_out.data_ptr(), float(dropout_p), seed_v, flags, _ptr(g_x), dw_l.data_ptr(), _ptr(db_l),
                                     dw_r.data_ptr(), _ptr(dgamma), _ptr(dbeta), N, graph.num_edges, Hin, Hout, _dt(x),
                                     ws.data_ptr(), ws_bytes, _stream(x)))
    LAUNCH_COUNTER["kernels"] += 7 if want_input_grad else 4
    return g_x, dw_l, db_l, dw_r, dgamma, dbeta


class ForwardWeights:
    """The model's parameters as ``dfw_graphsage_forward`` takes them: a host array of device pointers (matrices in the compute
    dtype, vectors fp32) plus the tensors that keep those pointers alive.  Built by ``GraphSAGEModel`` and cached there until a
    parameter changes."""

    def __init__(self, tensors: list, dims: tuple):
        self.tensors = tensors  # order: see include/dfw_b200.h
        self.array = (ctypes.c_void_p * len(tensors))(*[(t.data_ptr() if t is not None else None) for t in tensors])
        self.in_dim, self.enc_mid, self.hidden, self.dec_mid, self.num_layers = dims


def graphsage_forward(graph: "CSRGraph", x, weights: ForwardWeights, compute_dtype: torch.dtype, eps: float = 1e-5) -> torch.Tensor:
    """``dfw_graphsage_forward``: the whole eval-mode forward (``model.py:74-99``) in ONE C call -> fp32 ``[N, 1]``."""
    _require_cuda(x, "x")
    x = x.contiguous()
    N, dev = int(x.shape[0]), x.device
    out = torch.empty(N, 1, dtype=torch.float32, device=dev)
    ws_bytes = lib.dfw_graphsage_forward_ws_bytes(N, weights.in_dim, weights.enc_mid, weights.hidden, weights.dec_mid, _dt(x), _DTYPES[compute_dtype])
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.dfw_graphsage_forward(graph.rowptr.data_ptr(), _ptr(graph.col), graph.inv_deg.data_ptr(), x.data_ptr(), _dt(x), weights.array,
                                        weights.num_layers, N, graph.num_edges, weights.in_dim, weights.enc_mid, weights.hidden, weights.dec_mid,
                                        float(eps), _DTYPES[compute_dtype], out.data_ptr(), ws.data_ptr(), ws_bytes, _stream(x)))
    LAUNCH_COUNTER["kernels"] += 3 + 2 * weights.num_layers + (1 if (x.dtype == torch.float32 and compute_dtype != torch.float32) else 0)
    return out


MLP2_ENCODER, MLP2_DECODER = 0, 1


def mlp2_fwd(x, w1, b1, w2, b2, mode, dropout_p=0.0, seed=0, save_hidden=True):
    """One-call encoder / decoder MLP forward (``dfw_mlp2_fwd``).  Encoder: ``relu(relu(x W1^T + b1) W2^T + b2)``;
    decoder (``out_channels = 1``): ``dropout(relu(x W1^T + b1)) . w2 + b2`` as fp32 ``[N]`` (``w2`` fp32 ``[Hmid]``, ``b2`` fp32 ``[1]``).
    Returns ``(out, hidden)``."""
    _require_cuda(x, "x")
    x = x.contiguous()
    N, K = x.shape
    Hmid = w1.shape[0]
    dev, dt = x.device, x.dtype
    seed_v, seed_flag = _seed_arg(seed)
    if mode == MLP2_ENCODER:
        Hout = w2.shape[0]
        out = torch.empty(N, Hout, dtype=dt, device=dev)
        save_hidden = True
    else:
        Hout = 1
        out = torch.empty(N, dtype=torch.float32, device=dev)
    hidden = torch.empty(N, Hmid, dtype=dt, device=dev) if save_hidden else None
    ws_bytes = lib.dfw_mlp2_fwd_ws_bytes(N, K, Hmid, Hout, _dt(x))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.dfw_mlp2_fwd(x.data_ptr(), w1.data_ptr(), _ptr(b1), w2.data_ptr(), _ptr(b2), float(dropout_p), seed_v, seed_flag, int(mode),
                               _ptr(hidden), out.data_ptr(), N, K, Hmid, Hout, _dt(x), ws.data_ptr(), ws_bytes, _stream(x)))
    LAUNCH_COUNTER["kernels"] += 2 if mode == MLP2_ENCODER else 1
    return out, hidden


def mlp2_bwd(x, hidden, out, w1, w2, g_out, mode, dropout_p=0.0, seed=0, want_input_grad=True, has_b1=True, has_b2=True):
    """One-call encoder / decoder MLP backward (``dfw_mlp2_bwd``).  Returns ``(g_x, dw1, db1, dw2, db2)``."""
    N, K = x.shape
    Hmid = w1.shape[0]
    dev = x.device
    seed_v, seed_flag = _seed_arg(seed)
    f32 = dict(dtype=torch.float32, device=dev)
    g_out = g_out.contiguous()
    if mode == MLP2_ENCODER:
        Hout = w2.shape[0]
        dw2, db2 = torch.empty(Hout, Hmid, **f32), (torch.empty(Hout, **f32) if has_b2 else None)
    else:
        Hout = 1
        dw2, db2 = torch.empty(Hmid, **f32), (torch.empty(1, **f32) if has_b2 else None)
    g_x = torch.empty(N, K, dtype=x.dtype, device=dev) if want_input_grad else None
    dw1, db1 = torch.empty(Hmid, K, **f32), (torch.empty(Hmid, **f32) if has_b1 else None)
    ws_bytes = lib.dfw_mlp2_bwd_ws_bytes(N, K, Hmid, Hout, _dt(x), int(mode), int(want_input_grad))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib.dfw_mlp2_bwd(x.data_ptr(), hidden.data_ptr(), _ptr(out), w1.data_ptr(), w2.data_ptr(), g_out.data_ptr(), float(dropout_p),
                               seed_v, seed_flag, int(mode), _ptr(g_x), dw1.data_ptr(), _ptr(db1), dw2.data_ptr(), _ptr(db2),
                               N, K, Hmid, Hout, _dt(x), ws.data_ptr(), ws_bytes, _stream(x)))
    LAUNCH_COUNTER["kernels"] += 10 if mode == MLP2_ENCODER else 5
    return g_x, dw1, db1, dw2, db2


# ----------------------------------------------------------------------------------------------
# autograd Functions
# ----------------------------------------------------------------------------------------------
# bench.py's roofline pass clears this while it times every kernel alone on its stream
OVERLAP_DW = True
_SIDE_STREAMS: dict = {}


class _fork_dw:
    """``with _fork_dw(t, enabled):`` runs the body on the device's side stream, ordered after everything issued so far
    on the current stream; ``join()`` makes the current stream wait for it.  (The weight gradient of a layer and its
    input gradient are independent: side by side they fill each other's partial last waves.)"""

    def __init__(self, like: torch.Tensor, enabled: bool):
        self.main = torch.cuda.current_stream(like.device)
        self.side = _side_stream(like.device) if (enabled and OVERLAP_DW) else None
        self.ctx = None

    def __enter__(self):
        if self.side is not None:
            self.side.wait_stream(self.main)
            self.ctx = torch.cuda.stream(self.side)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False

    def join(self):
        if self.side is not None:
            self.main.wait_stream(self.side)


def _side_stream(device) -> torch.cuda.Stream:
    key = torch.device(device).index
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return st



import threading

_TLS = threading.local()


class _Fn(torch.autograd.Function):
    """autograd.Function whose ``forward`` can ask whether the CALLER had grad mode on.  ``ctx.needs_input_grad`` reflects
    ``requires_grad`` of the inputs even under ``torch.no_grad()``, and inside ``forward`` grad mode is always off, so
    without this eval / ``predict()`` would still write the tensors only a backward needs (pre-LayerNorm values,
    statistics, the decoder's hidden layer) - extra HBM passes on the inference path."""

    @classmethod
    def apply(cls, *args):
        prev = getattr(_TLS, "grad", None)
        _TLS.grad = torch.is_grad_enabled()
        try:
            return super().apply(*args)
        finally:
            _TLS.grad = prev


def _caller_grad_enabled() -> bool:
    g = getattr(_TLS, "grad", None)
    return True if g is None else bool(g)


class SageConvFn(_Fn):
    """SAGEConv forward/backward (mean aggregation + lin_l + lin_r), optionally with the
    model's LayerNorm -> ReLU -> dropout -> residual tail fused in (``model.py:90-95``)."""

    @staticmethod
    def forward(ctx, x, w_l, b_l, w_r, gamma, beta, graph: CSRGraph, eps, dropout_p, seed, fused_tail):
        _require_cuda(x, "x")
        x = x.contiguous()
        dt = x.dtype
        wl, wr = _w(w_l, dt), _w(w_r, dt)
        bl = _f32(b_l.detach()) if b_l is not None else None
        agg = aggregate_mean(graph, x)  # the tensor-core block kernel when the graph carries a profitable plan (large-mesh bf16 inference)
        # needs_input_grad reflects requires_grad even under torch.no_grad(): without the grad-mode test eval / predict()
        # would still write the pre-LayerNorm tensor and the statistics of every layer
        needs_grad = _caller_grad_enabled() and any(ctx.needs_input_grad[:6])
        if fused_tail:
            ln = (_f32(gamma.detach()), _f32(beta.detach()))
            out, pre, stats, _ = linear_fwd(agg, wl, x, wr, bias=bl, ln=ln, eps=eps, relu=True, residual=x,
                                            dropout_p=dropout_p, seed=seed, save_pre=needs_grad)
        else:
            ln = None
            out, pre, stats, _ = linear_fwd(agg, wl, x, wr, bias=bl)
        if needs_grad:
            ctx.graph = graph
            ctx.fused_tail, ctx.eps, ctx.dropout_p, ctx.seed = fused_tail, eps, dropout_p, seed
            ctx.has_bias = b_l is not None
            ctx.save_for_backward(x, agg, pre, stats, wl, wr, ln[0] if ln else None, ln[1] if ln else None)
            ctx.param_dtypes = (w_l.dtype, w_r.dtype)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, agg, pre, stats, wl, wr, gamma, beta = ctx.saved_tensors
        graph: CSRGraph = ctx.graph
        g_out = g_out.contiguous()
        N, H = g_out.shape
        # no parameter gradient wanted (design sensitivities: only the input gradient): no weight-gradient work at all
        want_params = any(ctx.needs_input_grad[1:6])
        dgamma = dbeta = dbl = dwl = dwr = None
        if ctx.fused_tail:
            # the epilogue backward also emits the column sums of g_y = lin_l's bias gradient
            g_y, dgamma, dbeta, _, _, dbl = epilogue_bwd(g_out, N, H, g_out, pre=pre, stats=stats, ln=(gamma, beta), relu=True,
                                                         dropout_p=ctx.dropout_p, seed=ctx.seed,
                                                         want_bias_grad=ctx.has_bias and want_params, want_param_grads=want_params)
        else:
            g_y = g_out
        fork = _fork_dw(g_y, ctx.needs_input_grad[0] and want_params)
        if want_params:
            with fork:
                dwl, dwr, db_ = linear_bwd_weight(g_y, agg, x, want_bias=ctx.has_bias and not ctx.fused_tail)
            if not ctx.fused_tail:
                dbl = db_
        g_x = None
        if ctx.needs_input_grad[0]:
            # dL/dx = A^T D^-1 (g_y W_l) + g_y W_r (+ g_out) = (A^T D^-1 g_y) W_l + g_y W_r (+ g_out): aggregate the
            # gradient FIRST (scale on the source side), then ONE two-operand linear with the residual epilogue -
            # the forward's own kernel shape - instead of two contractions and an aggregation with an addend
            # (8 -> 6 passes over [N, H] tensors).
            rp_t, col_t = graph.transpose()
            g_t = aggregate_scaled(rp_t, col_t, graph.inv_deg, g_y)
            g_x, _, _, _ = linear_fwd(g_t, wl, g_y, wr, residual=g_out if ctx.fused_tail else None, transpose_w=True,
                                      label="linear_bwd_input")
        fork.join()
        return g_x, dwl, dbl, dwr, dgamma, dbeta, None, None, None, None, None


class LinearFn(_Fn):
    """``relu?(x W^T + b)`` (+ dropout): encoder / decoder linears (``model.py:52-57,67-72``)."""

    @staticmethod
    def forward(ctx, x, w, b, relu, dropout_p, seed):
        _require_cuda(x, "x")
        x = x.contiguous()
        dt = x.dtype
        wc = _w(w, dt)
        out, _, _, _ = linear_fwd(x, wc, bias=_f32(b.detach()) if b is not None else None, relu=relu, dropout_p=dropout_p,
                                  seed=seed)
        if _caller_grad_enabled() and any(ctx.needs_input_grad[:3]):
            ctx.relu, ctx.dropout_p, ctx.seed, ctx.has_bias = relu, dropout_p, seed, b is not None
            ctx.save_for_backward(x, wc, out if relu else None)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, wc, act = ctx.saved_tensors
        g_out = g_out.contiguous()
        N, H = g_out.shape
        want_params = any(ctx.needs_input_grad[1:3])
        dw = None
        if ctx.relu or ctx.dropout_p > 0.0:
            if H % 4 != 0:
                raise RuntimeError("dfw_b200: ReLU/dropout backward needs out_features % 4 == 0")
            g_y, _, _, _, _, db = epilogue_bwd(g_out, N, H, g_out, act=act, relu=ctx.relu, dropout_p=ctx.dropout_p, seed=ctx.seed,
                                               want_bias_grad=ctx.has_bias and want_params)
            want_db = False
        else:
            g_y, db, want_db = g_out, None, ctx.has_bias
        fork = _fork_dw(g_y, ctx.needs_input_grad[0] and want_params)
        if want_params:
            with fork:
                dw, _, db_ = linear_bwd_weight(g_y, x, None, want_bias=want_db)
            if want_db:
                db = db_
        g_x = linear_bwd_input(g_y, wc) if ctx.needs_input_grad[0] else None
        fork.join()
        return g_x, dw, db, None, None, None


class DecoderTailFn(_Fn):
    """``Linear(H,64) -> ReLU -> Dropout -> Linear(64,1)`` in one kernel (``model.py:67-72``):
    the 64 -> 1 projection is a row dot product in the epilogue of the first linear."""

    @staticmethod
    def forward(ctx, h, w3, b3, w4, b4, dropout_p, seed):
        _require_cuda(h, "h")
        h = h.contiguous()
        dt = h.dtype
        w3c = _w(w3, dt)
        w4f = _f32(w4.detach()).reshape(-1)
        needs_grad = _caller_grad_enabled() and any(ctx.needs_input_grad[:5])
        b4f = _f32(b4.detach()).reshape(-1) if b4 is not None else None
        hid, _, _, rd = linear_fwd(h, w3c, bias=_f32(b3.detach()) if b3 is not None else None, relu=True, dropout_p=dropout_p,
                                   seed=seed, rowdot=(w4f, b4f), want_out=needs_grad)
        out = rd.unsqueeze(1)
        if dt != torch.float32:
            out = cast(out, dt)
        if needs_grad:
            ctx.dropout_p, ctx.seed = dropout_p, seed
            ctx.has_b3, ctx.has_b4 = b3 is not None, b4 is not None
            ctx.save_for_backward(h, hid, w3c, w4f)
        return out

    @staticmethod
    def backward(ctx, g_out):
        h, hid, w3c, w4f = ctx.saved_tensors
        N = h.shape[0]
        Hmid = hid.shape[1]
        g_r = g_out.reshape(-1).float().contiguous()
        want_params = any(ctx.needs_input_grad[1:5])
        g_y, _, _, dw4, db4, db3 = epilogue_bwd(None, N, Hmid, hid, g_rowdot=g_r, rowdot_w=w4f, act=hid, relu=True,
                                                dropout_p=ctx.dropout_p, seed=ctx.seed, want_bias_grad=ctx.has_b3 and want_params,
                                                want_param_grads=want_params)
        fork = _fork_dw(g_y, ctx.needs_input_grad[0] and want_params)
        dw3 = None
        if want_params:
            with fork:
                dw3, _, _ = linear_bwd_weight(g_y, h, None, want_bias=False)
        g_h = linear_bwd_input(g_y, w3c) if ctx.needs_input_grad[0] else None
        fork.join()
        return (g_h, dw3, db3, dw4.reshape(1, -1) if dw4 is not None else None, (db4 if ctx.has_b4 and want_params else None),
                None, None)


class MaskedMSEFn(torch.autograd.Function):
    """When the dtypes of ``pred`` and ``target`` differ, both are read in fp32 (the upcast is exact; rounding an fp32
    target to bf16 would move the difference by up to 2^-9 |target|) and the fp32 gradient is rounded once to ``pred``'s
    dtype.  Equal dtypes are computed in that dtype."""

    @staticmethod
    def forward(ctx, pred, target, mask, reduction_mean):
        _require_cuda(pred, "pred")
        pred_c = pred.contiguous()
        target_c = target.contiguous()
        if pred_c.dtype != target_c.dtype:
            pred_c, target_c = _f32(pred_c), _f32(target_c)
        N = pred_c.shape[0]
        C = pred_c.numel() // max(N, 1) if N > 0 else 1
        m = None
        if mask is not None:
            m = mask.reshape(-1).to(torch.uint8).contiguous() if mask.dtype != torch.uint8 else mask.reshape(-1).contiguous()
            if mask.dtype == torch.bool:
                m = mask.reshape(-1).contiguous().view(torch.uint8)
        dev = pred.device
        result = torch.empty(2, dtype=torch.float32, device=dev)
        ws_bytes = lib.dfw_masked_mse_ws_bytes(N, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            check(lib.dfw_masked_mse_fwd(pred_c.data_ptr(), target_c.data_ptr(), _ptr(m), N, C, int(reduction_mean), _dt(pred_c),
                                         result.data_ptr(), ws.data_ptr(), ws_bytes, _stream(pred_c)))
        LAUNCH_COUNTER["kernels"] += 1
        ctx.save_for_backward(pred_c, target_c, m, result)
        ctx.reduction_mean = reduction_mean
        ctx.shape, ctx.pred_dtype = pred.shape, pred.dtype
        loss, count = result[0], result[1]
        ctx.mark_non_differentiable(count)
        return loss, count

    @staticmethod
    def backward(ctx, g_loss, _g_count):
        pred_c, target_c, m, result = ctx.saved_tensors
        N = pred_c.shape[0]
        C = pred_c.numel() // max(N, 1) if N > 0 else 1
        g = torch.empty_like(pred_c)
        gl = g_loss.float().reshape(1).contiguous()
        with torch.cuda.device(pred_c.device):
            check(lib.dfw_masked_mse_bwd(pred_c.data_ptr(), target_c.data_ptr(), _ptr(m), result.data_ptr(), gl.data_ptr(), N, C,
                                         int(ctx.reduction_mean), _dt(pred_c), g.data_ptr(), _stream(pred_c)))
        LAUNCH_COUNTER["kernels"] += 1
        return cast(g, ctx.pred_dtype).view(ctx.shape), None, None, None
