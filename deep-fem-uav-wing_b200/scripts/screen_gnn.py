#!/usr/bin/env python3
"""FEM-free design screening: predicted stress of many wing designs from their geometry alone (``gnn/screening.py``).

Cases come from geometry packs (``--cases-dir``, written by ``caseio.pack_geometry_case``), from the dataset's FEM case
files (``--all`` over ``data/raw``: their normals are used, their stress is not) or are generated (``--synthetic N``).
One JSON line per case goes to ``--out`` in input order, and the ``--top-k`` designs by peak stress are printed.
With ``torchrun`` the case list is sharded ``case_ids[rank::world]`` as in ``inference_gnn.py``; the data path has no
communication, and at the end a gloo group gathers the records to rank 0, which writes the one output file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from pathlib import Path

PKG_ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(PKG_ROOT))
sys.path.insert(0, str(Path(__file__).resolve().parent))

import torch  # noqa: E402


def case_list(args, root: Path) -> list:
    """(kind, key) per case, in input order."""
    if args.synthetic:
        return [("synthetic", args.seed + i) for i in range(args.synthetic)]
    if args.cases_dir:
        return [("geometry", str(p)) for p in sorted(Path(args.cases_dir).glob("*.npz"))]
    fem = root / "data" / "raw" / "fem"
    return [("raw", d.name) for d in sorted(fem.iterdir()) if d.is_dir()] if fem.is_dir() else []


def load_case(kind: str, key, args, root: Path) -> dict:
    from deep_fem_uav_wing.gnn import caseio, synth

    if kind == "synthetic":
        return synth.geometry_case(synth.surface_tri_wing(args.synthetic_nodes, seed=key))
    if kind == "geometry":
        return caseio.load_geometry_case(key)
    raw = root / "data" / "raw"
    src = (raw / "fem" / key / "surface_results.npz", raw / "mesh" / key / "boundary_sets.json", raw / "geometry" / key / "params.json")
    missing = [p.name for p in src if not p.exists()]
    if missing:
        return {"case_id": key, "error": f"{missing[0]} not found"}
    return caseio.read_case(*src)


def main():
    p = argparse.ArgumentParser(description="FEM-free design screening with a trained GNN surrogate (B200-native)")
    p.add_argument("--checkpoint", type=str, default="checkpoints/best_model.pt", help="relative to --root, as in inference_gnn.py")
    p.add_argument("--root", type=str, default=os.environ.get("DFW_PROJECT_ROOT", str(Path.cwd())))
    src = p.add_mutually_exclusive_group(required=True)
    src.add_argument("--cases-dir", type=str, help="directory of geometry packs (caseio.pack_geometry_case)")
    src.add_argument("--all", action="store_true", help="every case under <root>/data/raw")
    src.add_argument("--synthetic", type=int, default=0, metavar="N", help="N generated wing surfaces (gnn/synth.py)")
    p.add_argument("--seed", type=int, default=0, help="first seed of --synthetic")
    p.add_argument("--synthetic-nodes", type=int, default=20000)
    p.add_argument("--dtype", choices=["fp32", "bf16"], default="fp32")
    p.add_argument("--allowable-mpa", type=float, default=None, help="allowable von Mises stress, MPa")
    p.add_argument("--root-band", type=float, default=0.05)
    p.add_argument("--max-nodes-per-launch", type=int, default=320_000)
    p.add_argument("--top-k", type=int, default=10)
    p.add_argument("--out", type=str, default="screening.jsonl", help="JSON lines, one per case in input order (relative to --root)")
    args = p.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("deep_fem_uav_wing (B200 build) is CUDA-only: no CPU fallback exists")
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)

    from inference_gnn import load_model

    from deep_fem_uav_wing.gnn.screening import DesignScreener

    root = Path(args.root)
    model = load_model(root / args.checkpoint, device)
    if args.dtype == "bf16":
        model.set_compute_dtype(torch.bfloat16)
    allowable = args.allowable_mpa * 1e6 if args.allowable_mpa is not None else None
    screener = DesignScreener(model, max_nodes_per_launch=args.max_nodes_per_launch, root_band=args.root_band, allowable_pa=allowable)
    cases = case_list(args, root)
    mine = list(range(len(cases)))[rank::world]

    errors = {}

    def stream():
        for i in mine:
            c = load_case(*cases[i], args, root)
            if "error" in c:  # screened as a failed case, in its place
                errors[i] = c.pop("error")
            yield c

    records = []
    for i, r in zip(mine, screener.iter_screen(stream())):
        if i in errors:
            r["reason"] = errors[i]
        records.append(dict(r, index=i))
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("gloo")
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(records, gathered, dst=0)
        dist.destroy_process_group()
        if rank != 0:
            return
        records = sorted((r for part in gathered for r in part), key=lambda r: r["index"])
    out = root / args.out
    out.parent.mkdir(parents=True, exist_ok=True)
    with open(out, "w", encoding="utf-8") as f:
        for r in records:
            r.pop("index", None)
            f.write(json.dumps(r) + "\n")
    ok = [r for r in records if r["status"] == "success"]
    print(f"[Screen] {len(ok)}/{len(records)} case(s) screened ({args.dtype}) -> {out}")
    ranked = sorted(ok, key=lambda r: r["max_stress_pa"], reverse=True)[: max(args.top_k, 0)]
    for k, r in enumerate(ranked, 1):
        line = f"[Screen] #{k} {r['case_id']}: max {r['max_stress_pa'] / 1e6:.2f} MPa at node {r['max_stress_node_id']}"
        if "margin_of_safety" in r and r["margin_of_safety"] is not None:
            line += f", margin of safety {r['margin_of_safety']:+.3f} ({r['n_over_allowable']} node(s) over allowable)"
        print(line)


if __name__ == "__main__":
    main()
