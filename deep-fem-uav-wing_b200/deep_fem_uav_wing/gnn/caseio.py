"""Binary case format and batched report writer (SURVEY 8f-3).

The reference keeps a case in three files - ``data/raw/fem/<id>/surface_results.npz`` (``fem.py:642-650``),
``data/raw/mesh/<id>/boundary_sets.json`` whose ``surf_all_faces`` is a JSON list of ~100k ``[a, b, c]`` node-id
triples (``meshing.py:443-454``) and ``data/raw/geometry/<id>/params.json`` - and ``json.loads`` of the face list is
what a per-case inference spends its host time on once the forward takes under a millisecond.  ``pack_case`` folds
the three files into ONE uncompressed ``.npz`` (faces as an ``int32 [F, 3]`` array, the four wing parameters as
``float64 [4]``): it loads with a handful of ``memcpy``-speed array reads and goes to the GPU as is.  The reference's
files stay the interchange format - the packed file is a cache next to them (``data/packed/<id>.npz``) and
``build_graph_data*`` give bit-identical results from either (``tests/test_caseio.py``).

``ReportWriter`` collects the per-case ``inference_report.json`` payloads (reference schema,
``inference_gnn.py:314-326``) and writes them in one go at the end of a run, plus one merged JSON-lines file, instead
of one ``json.dumps`` + file open per case inside the inference loop.
"""
from __future__ import annotations

import json
import os
from pathlib import Path
from typing import Any

import numpy as np

PACK_VERSION = 1
_PARAM_KEYS = ("span_m", "chord_m", "sweep_deg", "thickness_ratio")
_NPZ_KEYS = ("node_id", "pos", "normal", "stress_vm", "disp", "loss_mask")


def read_case(surface_npz_path, boundary_sets_path, params_path) -> dict[str, Any]:
    """The reference's three files -> the raw arrays ``build_graph_data`` works on (``dataset.py:94-120``)."""
    npz = np.load(surface_npz_path)
    boundary_sets = json.loads(Path(boundary_sets_path).read_text(encoding="utf-8"))
    params = json.loads(Path(params_path).read_text(encoding="utf-8"))
    faces = boundary_sets["surf_all_faces"]
    faces = np.asarray(faces, dtype=np.int64).reshape(-1, 3) if len(faces) else np.zeros((0, 3), np.int64)
    raw = {k: np.asarray(npz[k]) for k in _NPZ_KEYS}
    raw["faces"] = faces
    raw["params"] = {k: params[k] for k in _PARAM_KEYS}
    raw["case_id"] = params["case_id"]
    return raw


def pack_case(surface_npz_path, boundary_sets_path, params_path, out_path) -> Path:
    """Write the packed single-file form of a case; returns ``out_path``."""
    raw = read_case(surface_npz_path, boundary_sets_path, params_path)
    faces = raw["faces"]
    small = faces.size == 0 or (int(faces.min()) >= -(2**31) and int(faces.max()) < 2**31)
    out_path = Path(out_path)
    out_path.parent.mkdir(parents=True, exist_ok=True)
    tmp = out_path.with_name(out_path.name + f".tmp{os.getpid()}")
    with open(tmp, "wb") as f:  # (a file object: np.savez would append ".npz" to a bare path)
        np.savez(
            f, pack_version=np.int64(PACK_VERSION), case_id=np.array(str(raw["case_id"])),
            params=np.array([raw["params"][k] for k in _PARAM_KEYS], dtype=np.float64),
            faces=faces.astype(np.int32 if small else np.int64), **{k: raw[k] for k in _NPZ_KEYS},
        )
    os.replace(tmp, out_path)  # atomic: a rank that reads while another packs never sees a partial file
    return out_path


def load_packed_case(path) -> dict[str, Any]:
    """Inverse of :func:`pack_case`: the same dict :func:`read_case` returns."""
    z = np.load(path, allow_pickle=False)
    version = int(z["pack_version"])
    if version != PACK_VERSION:
        raise ValueError(f"{path}: packed case version {version}, this build reads version {PACK_VERSION}")
    raw = {k: z[k] for k in _NPZ_KEYS}
    raw["faces"] = z["faces"].astype(np.int64).reshape(-1, 3)
    p = z["params"]
    # json round trip of a Python float is exact in float64, so the packed parameters equal the parsed ones bit for bit
    raw["params"] = {k: float(p[i]) for i, k in enumerate(_PARAM_KEYS)}
    raw["case_id"] = str(z["case_id"])
    return raw


GEOMETRY_VERSION = 1


def pack_geometry_case(out_path, case_id, node_id, pos, faces, params) -> Path:
    """Write the pre-FEM content of a case - surface node ids and positions, faces as node ids, the four wing parameters
    (a dict with ``span_m, chord_m, sweep_deg, thickness_ratio``) - as one uncompressed ``.npz``: what design screening
    (``gnn/screening.py``) needs of a design that has not been through FEM.  Arrays are stored with their dtypes as given,
    so :func:`load_geometry_case` returns them bit for bit.  Written atomically like :func:`pack_case`."""
    node_id, pos, faces = np.asarray(node_id), np.asarray(pos), np.asarray(faces)
    if pos.ndim != 2 or pos.shape[1] != 3 or node_id.shape != (pos.shape[0],):
        raise ValueError(f"pos must be [N, 3] and node_id [N], got {pos.shape} and {node_id.shape}")
    if faces.size % 3 or not np.issubdtype(faces.dtype, np.integer) or not np.issubdtype(node_id.dtype, np.integer):
        raise ValueError("faces must be an integer [F, 3] array of node ids and node_id an integer array")
    out_path = Path(out_path)
    out_path.parent.mkdir(parents=True, exist_ok=True)
    tmp = out_path.with_name(out_path.name + f".tmp{os.getpid()}")
    with open(tmp, "wb") as f:
        np.savez(f, geometry_version=np.int64(GEOMETRY_VERSION), case_id=np.array(str(case_id)), node_id=node_id, pos=pos,
                 faces=faces.reshape(-1, 3), params=np.array([float(params[k]) for k in _PARAM_KEYS], dtype=np.float64))
    os.replace(tmp, out_path)
    return out_path


def load_geometry_case(path) -> dict[str, Any]:
    """Inverse of :func:`pack_geometry_case`: ``{case_id, node_id, pos, faces, params}``, the case dict
    ``DesignScreener.screen`` takes."""
    z = np.load(path, allow_pickle=False)
    if "geometry_version" not in z.files:
        raise ValueError(f"{path}: not a geometry case (no geometry_version field)")
    version = int(z["geometry_version"])
    if version != GEOMETRY_VERSION:
        raise ValueError(f"{path}: geometry case version {version}, this build reads version {GEOMETRY_VERSION}")
    p = z["params"]
    return {"case_id": str(z["case_id"]), "node_id": z["node_id"], "pos": z["pos"], "faces": z["faces"],
            "params": {k: float(p[i]) for i, k in enumerate(_PARAM_KEYS)}}


def packed_path(root, case_id: str) -> Path:
    return Path(root) / "data" / "packed" / f"{case_id}.npz"


def pack_dataset(root, overwrite: bool = False) -> list[Path]:
    """Pack every complete case under ``<root>/data/raw`` into ``<root>/data/packed/<id>.npz``."""
    raw = Path(root) / "data" / "raw"
    fem_dir, mesh_dir, geometry_dir = raw / "fem", raw / "mesh", raw / "geometry"
    done = []
    if not fem_dir.is_dir():
        return done
    for case_dir in sorted(fem_dir.iterdir()):
        cid = case_dir.name
        src = (fem_dir / cid / "surface_results.npz", mesh_dir / cid / "boundary_sets.json", geometry_dir / cid / "params.json")
        if not case_dir.is_dir() or not all(p.exists() for p in src):
            continue
        dst = packed_path(root, cid)
        if overwrite or not dst.exists() or dst.stat().st_mtime < max(p.stat().st_mtime for p in src):
            pack_case(*src, dst)
        done.append(dst)
    return done


class ReportWriter:
    """Buffers per-case reports and writes them at ``flush()``: every ``<fem_dir>/<case>/inference_report.json`` in
    the reference's schema (``inference_gnn.py:314-326``) and, when ``merged_path`` is given, one JSON-lines file
    holding all of them (one line per case, the order they were added)."""

    def __init__(self, fem_dir, merged_path=None, indent: int | None = 2):
        self.fem_dir, self.merged_path, self.indent = Path(fem_dir), Path(merged_path) if merged_path else None, indent
        self._pending: list[dict] = []
        self.written = 0

    def add(self, report: dict) -> None:
        self._pending.append(report)

    def flush(self) -> int:
        lines = []
        for r in self._pending:
            case_dir = self.fem_dir / str(r["case_id"])
            if case_dir.is_dir():
                (case_dir / "inference_report.json").write_text(json.dumps(r, indent=self.indent), encoding="utf-8")
            lines.append(json.dumps(r))
        if self.merged_path is not None and lines:
            self.merged_path.parent.mkdir(parents=True, exist_ok=True)
            with open(self.merged_path, "a", encoding="utf-8") as f:
                f.write("\n".join(lines) + "\n")
        n = len(self._pending)
        self.written += n
        self._pending.clear()
        return n

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.flush()
        return False
