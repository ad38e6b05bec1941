#!/usr/bin/env python3
"""Design-screening throughput (BASELINE.json config 5 through gnn/screening.py) and the time of its two new kernels.

Workload: ``--n-cases`` synthetic ``--nodes``-node wing surfaces (48 distinct per run, cycled as bench.py's cfg5 block
does: generating 10k meshes on the host would take minutes), GraphSAGE H = 128, L = 4, fp32 and bf16, three arms:
  (a) normals given with the case - the same input as bench.py's cfg5 block, so the two rates compare directly;
  (b) geometry only - normals computed on the device (dfw_vertex_normals);
  (c) the input of (a) with design sensitivities (``sensitivities=True``: grad-mode forward, dfw_case_ks_seed, the
      input-gradient backward, dfw_case_column_sums), with the observed ks_stress_pa / max_stress_pa at the default rho.
The screening rate is host wall time around ``DesignScreener.screen`` (host preparation included), which ends in an
explicit device wait.  Kernel times: CUDA events around ``--kernel-iters`` back-to-back calls on one 320k-node launch
(16 x 20k nodes; its working set fits in L2, so these are L2-resident times), the new kernels included.  The GPU name and power limit are read in
the same run.  Prints one JSON line (and writes it to ``--out``).
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO / "deep-fem-uav-wing_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_info() -> dict:
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def kernel_times(meshes, iters: int) -> dict:
    from deep_fem_uav_wing.gnn import ops

    pos = np.concatenate([m["pos"] for m in meshes])
    offs = np.cumsum([0] + [m["num_nodes"] for m in meshes])
    faces = np.concatenate([m["faces"].astype(np.int64) + o for m, o in zip(meshes, offs[:-1])])
    pos_d, faces_d = torch.from_numpy(pos).cuda(), torch.from_numpy(faces).cuda()
    cp = torch.from_numpy(offs.astype(np.int64)).cuda()
    pred = torch.log1p(torch.rand(len(pos), device="cuda") * 5e7)
    N, F = len(pos), len(faces)
    pred_bf16 = pred.bfloat16()
    g_x = torch.randn(N, 10, device="cuda")
    out = {"launch_nodes": N, "launch_faces": F, "launch_cases": len(meshes), "iters": iters}
    for name, fn, nbytes in (("vertex_normals", lambda: ops.vertex_normals(pos_d, faces_d), 24 * F + 24 * N),
                             ("case_stress_summary_fp32", lambda: ops.case_stress_summary(pred, pos_d, cp), 16 * N),
                             ("case_stress_summary_bf16", lambda: ops.case_stress_summary(pred.bfloat16(), pos_d, cp), 14 * N),
                             # reads pred and the y column twice (max pass, then the seed pass), writes the fp32 seed
                             ("case_ks_seed_fp32", lambda: ops.case_ks_seed(pred, pos_d, cp), 2 * 16 * N + 4 * N),
                             ("case_ks_seed_bf16", lambda: ops.case_ks_seed(pred_bf16, pos_d, cp), 2 * 14 * N + 4 * N),
                             # the screener's call: columns 6..9 of the fp32 [N, 10] input gradient (whole 40-byte rows)
                             ("case_column_sums_gx", lambda: ops.case_column_sums(g_x, cp, 6, 4), 40 * N)):
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / iters
        out[name] = {"us_per_call": round(us, 2), "algorithmic_bytes": nbytes, "GB_per_s": round(nbytes / (us * 1e-6) / 1e9, 1),
                     "note": "includes the op wrapper's workspace allocation and (bf16) the cast of pred"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-cases", type=int, default=10000)
    ap.add_argument("--nodes", type=int, default=20000)
    ap.add_argument("--distinct", type=int, default=48)
    ap.add_argument("--kernel-iters", type=int, default=200)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("screen_bench measures on a CUDA device; none found")
    from deep_fem_uav_wing.gnn import synth
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    torch.cuda.set_device(0)
    res = {"metric": "design screening (config 5) through DesignScreener", **gpu_info(), "n_cases": args.n_cases,
           "nodes_per_case": args.nodes, "hidden": 128, "layers": 4, "max_nodes_per_launch": 320_000}
    meshes = [synth.surface_tri_wing(args.nodes, seed=1000 + i) for i in range(args.distinct)]
    geometry = [synth.geometry_case(m) for m in meshes]
    given = [dict(c, normal=m["normal"]) for c, m in zip(geometry, meshes)]
    arms = {"normals_given": (given, False), "normals_computed": (geometry, False), "sensitivities_normals_given": (given, True)}
    for dtype in (torch.float32, torch.bfloat16):
        torch.manual_seed(42)
        model = GraphSAGEModel(10, 128, 1, 4).cuda().eval().set_compute_dtype(dtype)
        for arm, (cases, sens) in arms.items():
            screener = DesignScreener(model, sensitivities=sens)
            screener.screen(cases[i % len(cases)] for i in range(64))  # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = screener.screen(cases[i % len(cases)] for i in range(args.n_cases))
            dt = time.perf_counter() - t0
            assert len(out) == args.n_cases and all(r["status"] == "success" for r in out), "a screened case failed"
            r = {"cases_per_s": round(args.n_cases / dt, 1), "nodes_per_s": round(args.n_cases * args.nodes / dt), "s_total": round(dt, 3)}
            if sens:
                ratio = np.array([c["ks_stress_pa"] / c["max_stress_pa"] for c in out[:len(cases)]])
                r.update(ks_rho=screener.ks_rho, ks_over_max_stress={"min": round(float(ratio.min()), 5),
                                                                     "median": round(float(np.median(ratio)), 5),
                                                                     "max": round(float(ratio.max()), 5), "cases": len(ratio)})
            res[f"{arm}_{'fp32' if dtype == torch.float32 else 'bf16'}"] = r
    res["kernels_320k_launch"] = kernel_times(meshes[:16], args.kernel_iters)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
