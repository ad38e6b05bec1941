"""Seeded synthetic wing meshes for benchmarks and parity tests.

The reference ships no data (``.gitignore:12``) and its mesh/FEM stages need external
binaries (gmsh, ccx), so every workload in BASELINE.json is synthesised here.  Two families:

* ``surface_tri_wing`` - the graph the reference actually trains on (SURVEY F5): the outer
  triangle surface of a NACA-00xx loft (recipe: ``blender/generate_wing.py:43-64``), a
  closed 2-manifold -> average degree ~6.  Optionally written to disk in the reference's
  three-file case format so ``build_graph_data`` (``gnn/dataset.py:66-164``) reads it.
* ``tet_lattice_wing`` - tet-volume connectivity (Kuhn 6-tet split of a hex lattice mapped
  into the wing) -> degree ~14, BASELINE.json config 4's "2M nodes / ~28M edges".

Both return a dict with ``x [N,10] f32``, ``edge_index [2,E] i64`` (symmetric, no self loops,
no duplicates, shuffled order - ``dataset.py:39-63`` emits Python-set order), ``y [N,1] f32``
(= log1p(stress), ``dataset.py:148-151``), ``loss_mask [N] bool`` (``fem.py:637-640``).
Wing parameter ranges: ``scripts/generate_geometry_dataset.py:26-30``.
"""

from __future__ import annotations

import json
from pathlib import Path

import numpy as np


def sample_wing_params(rng: np.random.Generator) -> dict:
    return {
        "span_m": float(rng.uniform(1.0, 2.0)),
        "chord_m": float(rng.uniform(0.2, 0.5)),
        "sweep_deg": float(rng.uniform(0.0, 30.0)),
        "thickness_ratio": float(rng.uniform(0.05, 0.15)),
    }


def _naca_half_thickness(xc: np.ndarray, t: float) -> np.ndarray:
    xc = np.clip(xc, 0.0, 1.0)
    return 5.0 * t * (0.2969 * np.sqrt(xc) - 0.1260 * xc - 0.3516 * xc**2 + 0.2843 * xc**3 - 0.1015 * xc**4)


def _global_features(p: dict) -> np.ndarray:
    # dataset.py:122-127
    return np.array(
        [
            (p["span_m"] - 1.0) / 1.0,
            (p["chord_m"] - 0.2) / 0.3,
            p["sweep_deg"] / 30.0,
            (p["thickness_ratio"] - 0.05) / 0.10,
        ],
        dtype=np.float32,
    )


def _assemble_features(pos: np.ndarray, normal: np.ndarray, p: dict) -> np.ndarray:
    # dataset.py:130-145
    pos = pos.astype(np.float32)
    lo, hi = pos.min(axis=0), pos.max(axis=0)
    rng_ = hi - lo
    rng_[rng_ < 1e-8] = 1.0
    pos_n = (pos - lo) / rng_
    normal = normal.astype(np.float32)
    ln = np.linalg.norm(normal, axis=1, keepdims=True)
    ln[ln < 1e-8] = 1.0
    g = np.tile(_global_features(p), (pos.shape[0], 1))
    return np.concatenate([pos_n, normal / ln, g], axis=1).astype(np.float32)


def _synthetic_stress(pos: np.ndarray, p: dict, rng: np.random.Generator) -> np.ndarray:
    """Smooth bending-like von Mises field with a root concentration (Pa)."""
    eta = np.clip(pos[:, 1] / p["span_m"], 0.0, 1.0)
    zc = np.abs(pos[:, 2]) / (0.5 * p["thickness_ratio"] * p["chord_m"] + 1e-9)
    sigma = 4.0e7 * (1.0 - eta) ** 2 * (0.25 + 0.75 * np.clip(zc, 0, 1.5))
    sigma *= 1.0 + 0.1 * rng.standard_normal(pos.shape[0])
    return np.abs(sigma).astype(np.float32)


def undirected_to_edge_index(und: np.ndarray, rng: np.random.Generator | None) -> np.ndarray:
    """[U,2] unique undirected pairs -> symmetric int64 [2, 2U], optionally shuffled."""
    u = und.shape[0]
    ei = np.empty((2, 2 * u), dtype=np.int64)
    ei[0, 0::2], ei[1, 0::2] = und[:, 0], und[:, 1]
    ei[0, 1::2], ei[1, 1::2] = und[:, 1], und[:, 0]
    if rng is not None:
        ei = ei[:, rng.permutation(2 * u)]
    return np.ascontiguousarray(ei)


def faces_to_undirected(faces: np.ndarray, n: int) -> np.ndarray:
    a = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]], axis=0).astype(np.int64)
    lo, hi = a.min(axis=1), a.max(axis=1)
    key = np.unique(lo * n + hi)
    return np.stack([key // n, key % n], axis=1)


def _grid_dims(n_nodes: int, aspect: float) -> tuple[int, int]:
    """(nu around the section, nv span stations) with nu*nv == n_nodes when possible."""
    target_nu = max(8, int(round(np.sqrt(n_nodes / aspect))))
    best = None
    for nu in range(max(8, target_nu // 2), target_nu * 2 + 1):
        if nu % 2 == 0 and n_nodes % nu == 0 and n_nodes // nu >= 2:
            if best is None or abs(nu - target_nu) < abs(best - target_nu):
                best = nu
    if best is None:
        best = target_nu + (target_nu % 2)
    return best, max(2, n_nodes // best)


def surface_tri_wing(n_nodes: int, seed: int = 42, shuffle_edges: bool = True, params: dict | None = None,
                     node_order: str = "native") -> dict:
    """Closed triangulated wing surface with ~``n_nodes`` nodes (exact when it factorises)."""
    rng = np.random.default_rng(seed)
    p = dict(params) if params is not None else sample_wing_params(rng)
    nu, nv = _grid_dims(n_nodes, aspect=0.8)
    half = nu // 2
    # section loop: TE -> (upper) -> LE -> (lower) -> back toward TE; cosine spacing
    th = np.arange(nu) * (2.0 * np.pi / nu)
    xc = 0.5 * (1.0 + np.cos(th))
    sign = np.where(np.arange(nu) <= half, 1.0, -1.0)
    zt = _naca_half_thickness(xc, p["thickness_ratio"]) * sign
    ys = np.linspace(0.0, p["span_m"], nv)
    sweep = np.tan(np.deg2rad(p["sweep_deg"]))
    X = xc[None, :] * p["chord_m"] + ys[:, None] * sweep
    Y = np.repeat(ys[:, None], nu, axis=1)
    Z = np.repeat(zt[None, :] * p["chord_m"], nv, axis=0)
    pos = np.stack([X, Y, Z], axis=-1).reshape(-1, 3)
    n = nu * nv
    idx = np.arange(n).reshape(nv, nu)
    # skin quads -> two triangles
    a = idx[:-1, :]
    b = np.roll(idx, -1, axis=1)[:-1, :]
    c = idx[1:, :]
    d = np.roll(idx, -1, axis=1)[1:, :]
    skin = np.concatenate([np.stack([a, b, d], -1).reshape(-1, 3), np.stack([a, d, c], -1).reshape(-1, 3)], axis=0)
    # root / tip caps: zig-zag strip between upper point i and lower point nu-i (no new nodes)
    caps = []
    for row, flip in ((idx[0], False), (idx[-1], True)):
        i = np.arange(1, half - 1)
        up0, up1 = row[i], row[i + 1]
        lo0, lo1 = row[nu - i], row[nu - i - 1]
        t1 = np.stack([up0, up1, lo0], -1)
        t2 = np.stack([up1, lo1, lo0], -1)
        ends = np.array([[row[0], row[1], row[nu - 1]], [row[half - 1], row[half], row[half + 1]]])
        tri = np.concatenate([t1, t2, ends], axis=0)
        caps.append(tri[:, ::-1] if flip else tri)
    faces = np.concatenate([skin] + caps, axis=0).astype(np.int64)
    # area-weighted vertex normals (fem.py:390-424 does the same on the real surface)
    fn = np.cross(pos[faces[:, 1]] - pos[faces[:, 0]], pos[faces[:, 2]] - pos[faces[:, 0]])
    normal = np.zeros_like(pos)
    for c in range(3):
        for k in range(3):
            normal[:, c] += np.bincount(faces[:, k], weights=fn[:, c], minlength=n)
    und = faces_to_undirected(faces, n)
    stress = _synthetic_stress(pos, p, rng)
    span = float(pos[:, 1].max() - pos[:, 1].min())
    mask = pos[:, 1] > 0.05 * span
    out = _finish(pos, normal, stress, mask, und, p, rng if shuffle_edges else None, node_order, rng)
    out["faces"] = faces if node_order == "native" else out["_relabel"][faces]
    out.pop("_relabel", None)
    out["case_id"] = f"synthtri_{seed:06d}"
    return out


def tet_lattice_wing(n_nodes: int, seed: int = 42, shuffle_edges: bool = True, params: dict | None = None,
                     node_order: str = "native", dims: tuple[int, int, int] | None = None) -> dict:
    """Tet-volume connectivity: hex lattice (thickness x chord x span) split into Kuhn tets."""
    rng = np.random.default_rng(seed)
    p = dict(params) if params is not None else sample_wing_params(rng)
    if dims is None:
        # thickness : chord : span ~ 1 : 3 : 12 cells
        s = (n_nodes / 36.0) ** (1.0 / 3.0)
        nx = max(2, int(round(s)))
        ny = max(2, int(round(3 * s)))
        nz = max(2, int(round(n_nodes / (nx * ny))))
    else:
        nx, ny, nz = dims
    n = nx * ny * nz
    ix, iy, iz = np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij")
    # node id: thickness fastest, then chord, then span  (banded like a swept Gmsh numbering)
    nid = (iz * ny + iy) * nx + ix
    und_list = []
    for dx, dy, dz in ((1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (0, 1, 1), (1, 0, 1), (1, 1, 1)):
        a = nid[: nx - dx, : ny - dy, : nz - dz].ravel()
        b = nid[dx:, dy:, dz:].ravel()
        und_list.append(np.stack([np.minimum(a, b), np.maximum(a, b)], axis=1))
    und = np.concatenate(und_list, axis=0).astype(np.int64)
    order = np.argsort(nid.ravel(), kind="stable")
    u = (iy.ravel()[order] / max(ny - 1, 1)).astype(np.float64)  # chordwise 0..1
    v = (iz.ravel()[order] / max(nz - 1, 1)).astype(np.float64)  # spanwise 0..1
    w = (ix.ravel()[order] / max(nx - 1, 1)).astype(np.float64) * 2.0 - 1.0  # thickness -1..1
    sweep = np.tan(np.deg2rad(p["sweep_deg"]))
    Y = v * p["span_m"]
    X = u * p["chord_m"] + Y * sweep
    Z = w * _naca_half_thickness(u, p["thickness_ratio"]) * p["chord_m"]
    pos = np.stack([X, Y, Z], axis=-1)
    normal = np.stack([0.2 * (u - 0.5), np.zeros_like(u), np.where(w >= 0, 1.0, -1.0)], axis=-1)
    stress = _synthetic_stress(pos, p, rng)
    mask = pos[:, 1] > 0.05 * float(pos[:, 1].max() - pos[:, 1].min())
    out = _finish(pos, normal, stress, mask, und, p, rng if shuffle_edges else None, node_order, rng)
    out.pop("_relabel", None)
    out["lattice_dims"] = (nx, ny, nz)
    out["case_id"] = f"synthtet_{seed:06d}"
    return out


def _finish(pos, normal, stress, mask, und, p, edge_rng, node_order, rng) -> dict:
    n = pos.shape[0]
    relabel = None
    if node_order == "random":
        relabel = rng.permutation(n)  # old id -> new id
        inv = np.empty(n, dtype=np.int64)
        inv[relabel] = np.arange(n)
        pos, normal, stress, mask = pos[inv], normal[inv], stress[inv], mask[inv]
        und = relabel[und]
        und = np.stack([und.min(axis=1), und.max(axis=1)], axis=1)
    elif node_order != "native":
        raise ValueError(node_order)
    x = _assemble_features(pos, normal, p)
    return {
        "x": x,
        "edge_index": undirected_to_edge_index(und, edge_rng),
        "y": np.log1p(stress).reshape(-1, 1).astype(np.float32),
        "loss_mask": mask.astype(bool),
        "pos": pos.astype(np.float32),
        "normal": normal.astype(np.float32),
        "stress_vm_raw": stress.astype(np.float32),
        "params": p,
        "num_nodes": n,
        "_relabel": relabel,
    }


def geometry_case(mesh: dict, node_id_base: int = 1) -> dict:
    """The pre-FEM content of a surface-tri mesh as the case dict ``DesignScreener.screen`` takes (node ids from
    ``node_id_base``, faces as node ids, no normals: screening computes them)."""
    n = mesh["num_nodes"]
    return {"case_id": mesh["case_id"], "node_id": np.arange(n, dtype=np.int64) + node_id_base, "pos": mesh["pos"],
            "faces": mesh["faces"].astype(np.int64) + node_id_base, "params": dict(mesh["params"])}


def write_geometry_case(mesh: dict, out_dir: Path, node_id_base: int = 1) -> Path:
    """Write a surface-tri mesh as a geometry case ``<out_dir>/<case_id>.npz`` (``caseio.pack_geometry_case``)."""
    from .caseio import pack_geometry_case

    c = geometry_case(mesh, node_id_base)
    return pack_geometry_case(Path(out_dir) / f"{c['case_id']}.npz", c["case_id"], c["node_id"], c["pos"], c["faces"], c["params"])


def write_case_files(mesh: dict, root: Path, node_id_base: int = 1) -> str:
    """Write a surface-tri mesh in the reference's on-disk case format:
    ``data/raw/fem/{id}/surface_results.npz`` (``fem.py:642-650``),
    ``data/raw/mesh/{id}/boundary_sets.json`` (only ``surf_all_faces`` is consumed,
    ``dataset.py:112``) and ``data/raw/geometry/{id}/params.json`` (``types.py:16-23``)."""
    root = Path(root)
    cid = mesh["case_id"]
    n = mesh["num_nodes"]
    node_id = np.arange(n, dtype=np.int64) + node_id_base
    for sub in ("fem", "mesh", "geometry"):
        (root / "data" / "raw" / sub / cid).mkdir(parents=True, exist_ok=True)
    np.savez_compressed(
        root / "data" / "raw" / "fem" / cid / "surface_results.npz",
        node_id=node_id,
        pos=mesh["pos"].astype(np.float64),
        normal=mesh["normal"].astype(np.float64),
        stress_vm=mesh["stress_vm_raw"].astype(np.float64),
        disp=np.zeros((n, 3), dtype=np.float64),
        loss_mask=mesh["loss_mask"].astype(bool),
    )
    faces = (mesh["faces"] + node_id_base).tolist()
    (root / "data" / "raw" / "mesh" / cid / "boundary_sets.json").write_text(
        json.dumps({"surf_all_faces": faces}), encoding="utf-8"
    )
    params = dict(mesh["params"])
    params["case_id"] = cid
    (root / "data" / "raw" / "geometry" / cid / "params.json").write_text(json.dumps(params), encoding="utf-8")
    return cid
