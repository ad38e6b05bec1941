#!/usr/bin/env python3
"""Generate the golden fixtures in ``tests/golden/`` by running the REFERENCE's own code.

Run in the build container only (it reads ``/root/reference``, which does not exist on the
GPU box):  ``python tests/golden/make_golden.py``.  The fixtures it writes are committed.

What is executed from the reference (imported, never copied):
* ``src/deep_fem_uav_wing/gnn/dataset.py``: ``_faces_to_edge_index`` (``:26-63``) and
  ``build_graph_data`` (``:66-164``) - pure numpy, import as they are.
* ``src/deep_fem_uav_wing/gnn/model.py``: ``GraphSAGEModel`` (``:24-112``), ``MaskedMSELoss``
  (``:115-153``), ``compute_metrics`` (``:156-216``).  That module needs
  ``torch_geometric.nn.SAGEConv``, which is not installed and cannot be (no network), so a
  shim module named ``torch_geometric`` is registered whose ``SAGEConv`` is the oracle's
  ``SAGEConvRef`` restatement.  Everything else (encoder, LayerNorm/ReLU/dropout/residual
  wiring, decoder, loss, metrics) is the reference's own code.  Consequently the fixtures
  PIN the wiring, the loss and the metrics; the SAGEConv op stays "parity unpinned".
"""
from __future__ import annotations

import importlib
import sys
import tempfile
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
REPO = HERE.parent.parent
REF_SRC = Path("/root/reference/src")
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "deep-fem-uav-wing_b200"))

from oracle.sage_oracle import SAGEConvRef  # noqa: E402

# our own synthetic generator (loaded under a private name so that the package name
# ``deep_fem_uav_wing`` stays free for the reference import below)
_spec = importlib.util.spec_from_file_location(
    "dfw_synth", REPO / "deep-fem-uav-wing_b200" / "deep_fem_uav_wing" / "gnn" / "synth.py"
)
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)


def import_reference():
    tg = types.ModuleType("torch_geometric")
    tg_nn = types.ModuleType("torch_geometric.nn")
    tg_data = types.ModuleType("torch_geometric.data")
    tg_nn.SAGEConv = SAGEConvRef
    tg_nn.global_mean_pool = lambda x, batch: x.mean(0, keepdim=True)

    class Data:  # minimal stand-in; only needed so that ``dataset.py`` imports its PyG branch
        def __init__(self, **kw):
            self.__dict__.update(kw)

    class InMemoryDataset:
        pass

    tg_data.Data, tg_data.InMemoryDataset = Data, InMemoryDataset
    tg.nn, tg.data = tg_nn, tg_data
    sys.modules.update({"torch_geometric": tg, "torch_geometric.nn": tg_nn, "torch_geometric.data": tg_data})
    sys.path.insert(0, str(REF_SRC))
    for k in [k for k in sys.modules if k.startswith("deep_fem_uav_wing")]:
        del sys.modules[k]
    ref_model = importlib.import_module("deep_fem_uav_wing.gnn.model")
    ref_dataset = importlib.import_module("deep_fem_uav_wing.gnn.dataset")
    assert str(REF_SRC) in ref_model.__file__, ref_model.__file__
    assert ref_model.HAS_TORCH_GEOMETRIC
    return ref_model, ref_dataset


def sd_to_np(sd, prefix):
    return {f"{prefix}{k}": v.detach().cpu().numpy() for k, v in sd.items()}


def model_case(ref_model, name, mesh, hidden, layers, seed):
    torch.manual_seed(seed)
    model = ref_model.GraphSAGEModel(10, hidden, 1, layers, dropout=0.0)
    model.train()
    x = torch.from_numpy(mesh["x"])
    ei = torch.from_numpy(mesh["edge_index"])
    y = torch.from_numpy(mesh["y"])
    m = torch.from_numpy(mesh["loss_mask"])
    out = model(x, ei, None)
    loss = ref_model.MaskedMSELoss()(out, y, m)
    loss.backward()
    metrics = ref_model.compute_metrics(out, y, m)
    rec = {
        "x": mesh["x"], "edge_index": mesh["edge_index"], "y": mesh["y"], "loss_mask": mesh["loss_mask"],
        "hidden": np.int64(hidden), "layers": np.int64(layers),
        "out": out.detach().numpy(), "loss": np.float64(loss.item()),
        "metrics": np.array([metrics["all_nodes"]["mae"], metrics["all_nodes"]["rmse"], metrics["all_nodes"]["max_error"],
                             metrics["all_nodes"]["count"], metrics["masked_nodes"]["mae"], metrics["masked_nodes"]["rmse"],
                             metrics["masked_nodes"]["max_error"], metrics["masked_nodes"]["count"]], dtype=np.float64),
    }
    rec.update(sd_to_np(model.state_dict(), "sd/"))
    grads = {f"grad/{k}": p.grad.detach().numpy() for k, p in model.named_parameters()}
    # eval-mode forward with the constructor-default dropout (must equal dropout-free forward)
    model.eval()
    with torch.no_grad():
        rec["out_eval"] = model(x, ei).numpy()
    np.savez_compressed(HERE / f"{name}.npz", **rec)
    np.savez_compressed(HERE / f"{name}.grads.npz", **grads)  # apart, so that every file stays under 1 MB
    print(f"{name}: N={x.shape[0]} E={ei.shape[1]} loss={loss.item():.6f}")


def box_wing_mesh():
    """The 12-triangle box wing of ``geometry.py:82-102`` (8 nodes, 18 undirected edges)."""
    faces = np.array([[0, 1, 5], [0, 5, 4], [3, 7, 6], [3, 6, 2], [0, 3, 2], [0, 2, 1],
                      [4, 5, 6], [4, 6, 7], [0, 4, 7], [0, 7, 3], [1, 2, 6], [1, 6, 5]])
    return faces


def main():
    ref_model, ref_dataset = import_reference()
    rng = np.random.default_rng(7)

    # ---- graph construction: reference functions on written case files -----------------
    mesh = synth.surface_tri_wing(600, seed=11)
    with tempfile.TemporaryDirectory() as td:
        cid = synth.write_case_files(mesh, Path(td), node_id_base=101)
        raw = Path(td) / "data" / "raw"
        g = ref_dataset.build_graph_data(raw / "fem" / cid / "surface_results.npz",
                                         raw / "mesh" / cid / "boundary_sets.json",
                                         raw / "geometry" / cid / "params.json")
        np.savez_compressed(HERE / "build_graph_case.npz",
                            in_node_id=np.arange(mesh["num_nodes"]) + 101, in_pos=mesh["pos"].astype(np.float64),
                            in_normal=mesh["normal"].astype(np.float64), in_stress=mesh["stress_vm_raw"].astype(np.float64),
                            in_loss_mask=mesh["loss_mask"], in_faces=mesh["faces"] + 101,
                            in_params=np.array([mesh["params"][k] for k in ("span_m", "chord_m", "sweep_deg", "thickness_ratio")]),
                            x=g["x"], edge_index=g["edge_index"], y=g["y"], loss_mask=g["loss_mask"], pos=g["pos"],
                            stress_vm_raw=g["stress_vm_raw"], global_params=g["global_params"],
                            global_params_raw=g["global_params_raw"])
        print("build_graph_case:", g["x"].shape, g["edge_index"].shape)

    box = box_wing_mesh()
    ids = {i + 10: i for i in range(8)}
    e_box = ref_dataset._faces_to_edge_index((box + 10).tolist(), ids)
    e_skip = ref_dataset._faces_to_edge_index((box + 10).tolist() + [[10, 11, 999]], ids)  # unknown id -> face skipped
    e_empty = ref_dataset._faces_to_edge_index([], ids)
    np.savez_compressed(HERE / "faces_to_edge_index.npz", faces=box + 10, e_box=e_box, e_skip=e_skip, e_empty=e_empty)
    print("faces_to_edge_index:", e_box.shape, e_skip.shape, e_empty.shape)

    # ---- model fixtures: the reference's GraphSAGEModel on tiny meshes ------------------
    # (a) the box wing as a "real" tiny mesh
    xb = rng.standard_normal((8, 10)).astype(np.float32)
    box_mesh = {"x": xb, "edge_index": e_box, "y": rng.standard_normal((8, 1)).astype(np.float32),
                "loss_mask": np.array([0, 1, 1, 0, 1, 1, 1, 1], dtype=bool)}
    model_case(ref_model, "model_box_h16_l2", box_mesh, hidden=16, layers=2, seed=42)
    # (b) config-1 architecture (H=64, L=3) on a 600-node surface-tri wing
    model_case(ref_model, "model_tri600_h64_l3", synth.surface_tri_wing(600, seed=42), hidden=64, layers=3, seed=42)
    # (c) default architecture (H=128, L=4) on a small tet lattice with an isolated node and
    #     a duplicate + self-loop + one-directional edge appended
    tet = synth.tet_lattice_wing(500, seed=5)
    n = tet["num_nodes"]
    tet["x"] = np.concatenate([tet["x"], rng.standard_normal((1, 10)).astype(np.float32)])  # isolated node n
    tet["y"] = np.concatenate([tet["y"], np.zeros((1, 1), np.float32)])
    tet["loss_mask"] = np.concatenate([tet["loss_mask"], [True]])
    extra = np.array([[3, 3, 7, 0], [9, 9, 7, n - 1]], dtype=np.int64)  # dup 3->9 twice, self loop 7, one-way 0->n-1
    tet["edge_index"] = np.concatenate([tet["edge_index"], extra], axis=1)
    model_case(ref_model, "model_tet500_h128_l4", tet, hidden=128, layers=4, seed=43)

    # ---- loss / metric fixtures ---------------------------------------------------------
    pred = torch.from_numpy(rng.standard_normal((50, 1)).astype(np.float32) + 3.0).requires_grad_(True)
    targ = torch.from_numpy(rng.standard_normal((50, 1)).astype(np.float32) + 3.0)
    mask = torch.from_numpy(rng.random(50) > 0.4)
    rec = {"pred": pred.detach().numpy(), "target": targ.numpy(), "mask": mask.numpy()}
    for red in ("mean", "sum"):
        for mname, mm in (("mask", mask), ("none", None), ("allfalse", torch.zeros(50, dtype=torch.bool))):
            pred.grad = None
            l = ref_model.MaskedMSELoss(red)(pred, targ, mm)
            rec[f"loss_{red}_{mname}"] = np.float64(l.item())
            rec[f"loss_{red}_{mname}_requires_grad"] = np.bool_(l.requires_grad)
            if mname != "allfalse":
                l.backward()
                rec[f"grad_{red}_{mname}"] = pred.grad.numpy().copy()
    for mname, mm in (("mask", mask), ("none", None), ("allfalse", torch.zeros(50, dtype=torch.bool))):
        for ls in (True, False):
            met = ref_model.compute_metrics(pred, targ, mm, log_scale=ls)
            rec[f"metrics_{mname}_{int(ls)}"] = np.array(
                [met[a][b] for a in ("all_nodes", "masked_nodes") for b in ("mae", "rmse", "max_error", "count")], dtype=np.float64)
    np.savez_compressed(HERE / "loss_metrics.npz", **rec)
    print("loss_metrics written")


if __name__ == "__main__":
    main()
