"""FEM-free design screening (BASELINE.json config 5): stress predicted from the geometry alone, batched, with a
per-case summary computed on the device.

A surrogate earns its keep on designs that have NOT been through FEM.  ``DesignScreener.screen`` takes cases with
positions, faces and the four wing parameters (``caseio.load_geometry_case``; the FEM case dicts of
``caseio.read_case`` / ``load_packed_case`` work too - their ``normal`` is used, their ``stress_vm`` ignored), packs
them into launches of up to ``max_nodes_per_launch`` nodes and per launch runs, without a host synchronisation:

    pinned staging + H2D on a copy stream, one launch ahead          (the cfg5 block of bench.py)
    dfw_vertex_normals                  when a case brings no normals (reference fem.py:390-424)
    dfw_node_features_batched           x [N,10] (dataset.py:129-151), per-case normalisation
    dfw_faces_to_csr                    graph of the disjoint union (dataset.py:26-63)
    dfw_graphsage_forward               the model, one C call
    dfw_case_stress_summary             [B,8] per case -> one 64-byte-per-case D2H copy into pinned memory

The host waits for the device only when the pinned result ring wraps and after the last launch, so the enqueue of
launch l+1 overlaps the GPU work of launch l.  Every kernel on the path is row-local with a fixed per-row order, so a
case's result does not depend on which cases share its launch.
"""
from __future__ import annotations

from collections import deque
from concurrent.futures import ThreadPoolExecutor
from typing import Any, Callable, Iterable, Iterator

import numpy as np
import torch

from . import ops

MAX_CASES_PER_LAUNCH = 65535  # dfw_node_features_batched: one grid row per case


def pack_launches(items: Iterable, size_of: Callable[[Any], int], max_nodes: int,
                  max_cases: int = MAX_CASES_PER_LAUNCH) -> Iterator[list]:
    """Greedy packing in input order: a launch takes cases until the next one would push it past ``max_nodes`` nodes or
    ``max_cases`` cases.  A case larger than ``max_nodes`` runs alone.  Consumes ``items`` lazily."""
    if max_nodes < 1 or max_cases < 1:
        raise ValueError("max_nodes and max_cases must be positive")
    group, nodes = [], 0
    for it in items:
        n = int(size_of(it))
        if group and (nodes + n > max_nodes or len(group) >= max_cases):
            yield group
            group, nodes = [], 0
        group.append(it)
        nodes += n
    if group:
        yield group


def faces_to_rows(node_id, faces) -> tuple[np.ndarray, int]:
    """Faces of node ids -> int64 [F', 3] rows into the case's node order, and the number of faces dropped because they
    name an unknown id (``inference_gnn._surface_faces``; a duplicated id maps to its last row, as the reference's
    ``node_id_to_idx`` dict does, ``dataset.py:106-109``)."""
    ids = np.asarray(node_id, dtype=np.int64).reshape(-1)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    n = ids.size
    if n == 0 or f.shape[0] == 0:
        return np.zeros((0, 3), np.int64), int(f.shape[0])
    if ids[-1] - ids[0] == n - 1 and (n == 1 or bool(np.all(ids[1:] > ids[:-1]))):
        rows = f - ids[0]  # consecutive ascending ids (the usual numbering): a subtraction
        if rows.min() >= 0 and rows.max() < n:
            return rows, 0
        ok = ((rows >= 0) & (rows < n)).all(axis=1)
        return np.ascontiguousarray(rows[ok]), int((~ok).sum())
    order = np.argsort(ids, kind="stable")
    s = ids[order]
    k = np.maximum(np.searchsorted(s, f, side="right") - 1, 0)
    ok = (s[k] == f).all(axis=1)
    return np.ascontiguousarray(order[k][ok]), int((~ok).sum())


def global_params(params: dict) -> np.ndarray:
    """The four scaled wing parameters of ``dataset.py:122-127``."""
    return np.array([(params["span_m"] - 1.0) / 1.0, (params["chord_m"] - 0.2) / 0.3, params["sweep_deg"] / 30.0,
                     (params["thickness_ratio"] - 0.05) / 0.10], dtype=np.float32)


class _Case:
    __slots__ = ("case_id", "node_id", "pos", "pos32", "normal", "rows", "skipped", "gp", "error")

    def __init__(self, c: dict):
        self.case_id, self.error = str(c.get("case_id", "")), None
        try:
            self.pos = np.asarray(c["pos"])
            if self.pos.ndim != 2 or self.pos.shape[1] != 3 or self.pos.shape[0] == 0:
                raise ValueError(f"pos must be a non-empty [N, 3] array, got shape {self.pos.shape}")
            n = self.pos.shape[0]
            self.node_id = np.asarray(c["node_id"], dtype=np.int64).reshape(-1)
            if self.node_id.size != n:
                raise ValueError(f"node_id has {self.node_id.size} entries for {n} nodes")
            self.pos32 = np.ascontiguousarray(self.pos, dtype=np.float32)
            normal = c.get("normal")
            self.normal = None if normal is None else np.ascontiguousarray(normal, dtype=np.float32).reshape(n, 3)
            self.rows, self.skipped = faces_to_rows(self.node_id, c["faces"])
            self.gp = global_params(c["params"])
        except (KeyError, ValueError, TypeError) as e:
            self.error = f"{type(e).__name__}: {e}"

    @property
    def n(self) -> int:
        return 0 if self.error else self.pos32.shape[0]


class DesignScreener:
    """Batched FEM-free stress screening with a trained ``GraphSAGEModel`` (``out_channels = 1``).

    ``screen(cases)`` returns one dict per input case, in input order: ``case_id``, ``status`` (``"success"`` /
    ``"failed"`` with ``reason``), ``n_nodes``, ``n_screened``, ``normals`` (``"case"`` / ``"computed"``),
    ``skipped_faces``, ``max_stress_pa`` over the screened nodes (outside the root band, or ``mask``), its
    ``max_stress_node_id`` and ``max_stress_pos`` (the case's own id and units), ``mean_stress_pa``,
    ``max_stress_all_nodes_pa`` and, with ``allowable_pa``, ``n_over_allowable`` and
    ``margin_of_safety = allowable / max - 1``.  A case whose prediction is not finite is ``"failed"``.
    fp32 or bf16 follows the model's ``set_compute_dtype``."""

    def __init__(self, model, max_nodes_per_launch: int = 320_000, root_band: float = 0.05, allowable_pa: float | None = None,
                 result_ring: int = 8, prep_threads: int = 4):
        if int(getattr(model, "out_channels", 1)) != 1:
            raise ValueError("DesignScreener needs a model with out_channels = 1 (one stress value per node)")
        if allowable_pa is not None and not allowable_pa > 0:
            raise ValueError("allowable_pa must be positive")
        self.model = model
        self.max_nodes = int(max_nodes_per_launch)
        self.root_band = float(root_band)
        self.allowable_pa = None if allowable_pa is None else float(allowable_pa)
        self.result_ring = max(1, int(result_ring))
        self.prep_threads = max(1, int(prep_threads))
        self.device = next(model.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("DesignScreener: the model must live on a CUDA device (deep_fem_uav_wing.gnn has no CPU fallback)")
        self._copy_stream = torch.cuda.Stream(device=self.device)

    # ---- per launch ---------------------------------------------------------------------------------------------------
    def _stage(self, group: list) -> dict:
        """Pinned staging and H2D of one launch on the copy stream."""
        good = [c for c in group if c.error is None]
        launch = {"group": group, "good": good}
        if not good:
            return launch
        B = len(good)
        N = sum(c.n for c in good)
        F = sum(c.rows.shape[0] for c in good)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True)  # noqa: E731
        pos, faces, gp, ptr = pin((N, 3), torch.float32), pin((F, 3), torch.int64), pin((B, 4), torch.float32), pin(B + 1, torch.int64)
        given = [c.normal is not None for c in good]
        normal = pin((N, 3), torch.float32) if any(given) else None
        pos_np, faces_np, gp_np, ptr_np = pos.numpy(), faces.numpy(), gp.numpy(), ptr.numpy()
        r = f = 0
        ptr_np[0] = 0
        for b, c in enumerate(good):
            n, nf = c.n, c.rows.shape[0]
            pos_np[r:r + n] = c.pos32
            if c.normal is not None:
                normal.numpy()[r:r + n] = c.normal
            np.add(c.rows, r, out=faces_np[f:f + nf])
            gp_np[b] = c.gp
            r, f = r + n, f + nf
            ptr_np[b + 1] = r
        dev = self.device
        with torch.cuda.stream(self._copy_stream):
            launch["pos"] = pos.to(dev, non_blocking=True)
            launch["faces"] = faces.to(dev, non_blocking=True)
            launch["gp"] = gp.to(dev, non_blocking=True)
            launch["case_ptr"] = ptr.to(dev, non_blocking=True)
            launch["normal"] = normal.to(dev, non_blocking=True) if normal is not None else None
            launch["staged"] = torch.cuda.Event()
            launch["staged"].record(self._copy_stream)
        launch.update(N=N, F=F, B=B, max_rows=max(c.n for c in good), given=given, ptr=ptr_np.copy())
        return launch

    def _run(self, launch: dict) -> None:
        """Normals, features, graph, forward and summary of one staged launch on the current stream; the [B,8] records go to
        pinned memory with one non-blocking copy."""
        if not launch["good"]:
            return
        stream = torch.cuda.current_stream(self.device)
        stream.wait_event(launch["staged"])
        for k in ("pos", "faces", "gp", "case_ptr", "normal"):
            if launch[k] is not None:
                launch[k].record_stream(stream)  # allocated on the copy stream, read on this one
        pos, faces, cp, given = launch["pos"], launch["faces"], launch["case_ptr"], launch["given"]
        if all(given):
            normal = launch["normal"]
        else:
            normal, _ = ops.vertex_normals(pos, faces)  # faces were mapped to rows on the host: no index is out of range
            if any(given):
                ptr = launch["ptr"]
                for b, g in enumerate(given):
                    if g:
                        normal[ptr[b]:ptr[b + 1]].copy_(launch["normal"][ptr[b]:ptr[b + 1]])
        x, _ = ops.node_features_batched(pos, normal, None, launch["gp"], cp, launch["max_rows"])
        graph, _ = ops.faces_to_graph(faces, launch["N"], want_edge_index=False, sync=False)
        with torch.no_grad():
            pred = self.model(x, graph)  # eval + no_grad + CSRGraph: the one-call dfw_graphsage_forward
        summary = ops.case_stress_summary(pred, pos, cp, None, self.root_band, self.allowable_pa, log_scale=True)
        res = torch.empty(launch["B"], 8, dtype=torch.float64, pin_memory=True)
        res.copy_(summary, non_blocking=True)
        launch["result"] = res
        launch["done"] = torch.cuda.Event()
        launch["done"].record(stream)
        for k in ("pos", "faces", "gp", "case_ptr", "normal", "staged"):
            launch.pop(k, None)

    def _records(self, launch: dict) -> list[dict]:
        """Per-case dicts of a finished launch (after its ``done`` event)."""
        if launch["good"]:
            launch["done"].synchronize()  # explicit wait: the ring wrapped, or the last launch
            rec = launch["result"].numpy()
        out, b = [], 0
        for c in launch["group"]:
            if c.error is not None:
                out.append({"case_id": c.case_id, "status": "failed", "reason": c.error})
                continue
            out.append(self._record(c, rec[b], launch["given"][b]))
            b += 1
        return out

    def _record(self, c: _Case, r: np.ndarray, given: bool) -> dict:
        d = {"case_id": c.case_id, "status": "success", "n_nodes": int(r[0]), "n_screened": int(r[1]),
             "normals": "case" if given else "computed", "skipped_faces": int(c.skipped)}
        if r[7] > 0:
            d.update(status="failed", reason=f"{int(r[7])} non-finite predicted stress value(s)")
            return d
        row = int(r[3])
        d["max_stress_pa"] = float(r[2])
        d["max_stress_node_id"] = int(c.node_id[row]) if row >= 0 else None
        d["max_stress_pos"] = [float(v) for v in c.pos[row]] if row >= 0 else None
        d["mean_stress_pa"] = float(r[4])
        d["max_stress_all_nodes_pa"] = float(r[5])
        if self.allowable_pa is not None:
            d["n_over_allowable"] = int(r[6])
            d["margin_of_safety"] = self.allowable_pa / float(r[2]) - 1.0 if r[2] > 0 else None
        return d

    def _prepare(self, cases: Iterable[dict]) -> Iterator[_Case]:
        """Host preparation of the cases (face ids -> rows, fp32 copies) on a few threads - numpy releases the GIL in these
        array passes - with a bounded look-ahead, in input order."""
        with ThreadPoolExecutor(self.prep_threads) as ex:
            q: deque = deque()
            for c in cases:
                q.append(ex.submit(_Case, c))
                if len(q) > 2 * self.prep_threads:
                    yield q.popleft().result()
            while q:
                yield q.popleft().result()

    # ---- public -------------------------------------------------------------------------------------------------------
    def iter_screen(self, cases: Iterable[dict]) -> Iterator[dict]:
        """``screen`` as a generator: results come out in input order as their launch's records are read back."""
        self.model.eval()
        prepared = self._prepare(cases)
        launches = pack_launches(prepared, lambda c: c.n, self.max_nodes)
        pending: deque = deque()
        with torch.cuda.device(self.device):
            nxt = next(launches, None)
            staged = self._stage(nxt) if nxt is not None else None
            while staged is not None:
                cur = staged
                nxt = next(launches, None)
                staged = self._stage(nxt) if nxt is not None else None  # H2D of the next launch overlaps this one
                self._run(cur)
                pending.append(cur)
                if len(pending) > self.result_ring:
                    yield from self._records(pending.popleft())
            while pending:
                yield from self._records(pending.popleft())

    def screen(self, cases: Iterable[dict]) -> list[dict]:
        return list(self.iter_screen(cases))
