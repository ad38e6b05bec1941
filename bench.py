#!/usr/bin/env python3
"""Headline benchmark: GraphSAGE fwd+bwd+AdamW training throughput (meshes/s) on BASELINE.json
config 2 - 200 synthetic 50k-node wing meshes, hidden 128, 4 layers, fp32, batch 4 - at N GPUs,
data-parallel by mesh (weak scaling: every rank steps through its own 4-mesh batches).

    python bench.py --gpus 1 --steps 50 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the CPU path (oracle port of the PyG model) on host cores

One JSON line on rank 0.  `value` = device-resident throughput (pre-collated batches, CSR cached);
`e2e` = the same steps through the public API from pinned HOST batches (H2D + on-device CSR build +
fwd/bwd/AdamW + loss.item() per step).  `roofline` = dominant kernel of the step by measured time
(CUDA events on the launching stream, separate instrumented pass over the same steps), algorithmic
bytes or flops per launch / average duration, against MEASURED_PEAKS.json.  `cpu_baseline` = the
oracle on the box's host cores on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the timed device-resident training step computed in its last step
(its loss and the parameters its AdamW update left in the model, float32) as DIR/<name>.npy.  Every
input is seeded, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [REPO, os.path.join(REPO, "deep-fem-uav-wing_b200")]

HIDDEN, LAYERS, BATCH, NODES, N_MESHES, DROPOUT = 128, 4, 4, 50000, 200, 0.1
LR, WD = 1e-3, 1e-4  # train_gnn.py:167
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


# --------------------------------------------------------------------------------------------
# workload
# --------------------------------------------------------------------------------------------
def _synth():
    """gnn/synth.py imported BY FILE PATH: it is pure numpy, and importing it through the package would load libdfw_b200.so
    into the CPU arm's process too."""
    import importlib.util

    mod = sys.modules.get("_dfw_synth")
    if mod is None:
        spec = importlib.util.spec_from_file_location("_dfw_synth", os.path.join(REPO, "deep-fem-uav-wing_b200", "deep_fem_uav_wing", "gnn", "synth.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules["_dfw_synth"] = mod
        spec.loader.exec_module(mod)
    return mod


def make_meshes(ids, kind="tri"):
    synth = _synth()
    gen = synth.surface_tri_wing if kind == "tri" else synth.tet_lattice_wing
    out = []
    for i in ids:
        m = gen(NODES, seed=42 + i)
        out.append({k: m[k] for k in ("x", "edge_index", "y", "loss_mask", "num_nodes")})
    return out


def to_data(m):
    from deep_fem_uav_wing.gnn.loader import Data

    return Data(x=torch.from_numpy(m["x"]), edge_index=torch.from_numpy(m["edge_index"]), y=torch.from_numpy(m["y"]),
                loss_mask=torch.from_numpy(m["loss_mask"]))


class ClockSampler:
    """nvidia-smi style clock / throttle-reason samples during the timed region (via NVML)."""

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.ok = [], set(), False, False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks": 0x2}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self.stop_flag = True
        if self.ok:
            self.t.join(timeout=2)
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": float(self.max),
                    "reasons": sorted(self.reasons), "samples": len(self.samples)}
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}


def dump_outputs(out_dir, loss, model):
    """The last timed training step's loss and the parameters it left in ``model``, one float32 ``.npy`` per array
    (``loss.npy``, ``param.<name>.npy``): about 0.6 MB for the benchmarked model."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().reshape(1)}
    arrays.update({f"param.{k}": p.detach() for k, p in model.named_parameters()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def timed_region(step_fn, steps, dist_on, device):
    """barrier + synchronize on both sides, CUDA events on the launching stream, MAX over ranks."""
    import torch.distributed as dist

    if dist_on:
        dist.barrier()
    torch.cuda.synchronize(device)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        step_fn(i)
    b.record()
    torch.cuda.synchronize(device)
    if dist_on:
        dist.barrier()
    ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=device)
    if dist_on:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


# --------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference's PyG model)
# --------------------------------------------------------------------------------------------
def cpu_training_throughput(meshes, steps, warmup, threads=None):
    """The reference's training step (train_gnn.py:50-60) on the host cores: oracle port of the PyG model, torch CPU fp32.
    ``threads`` = None: every core of the box, set EXPLICITLY (torchrun exports OMP_NUM_THREADS=1)."""
    from oracle.sage_oracle import GraphSAGEModelRef, MaskedMSELossRef

    torch.set_num_threads(threads if threads else (os.cpu_count() or 1))
    torch.manual_seed(42)
    model = GraphSAGEModelRef(10, HIDDEN, 1, LAYERS, DROPOUT).train()
    opt = torch.optim.AdamW(model.parameters(), lr=LR, weight_decay=WD)
    crit = MaskedMSELossRef()
    batches = []
    for s in range(0, len(meshes) - BATCH + 1, BATCH):
        off, xs, eis, ys, ms = 0, [], [], [], []
        for m in meshes[s:s + BATCH]:
            xs.append(torch.from_numpy(m["x"])); eis.append(torch.from_numpy(m["edge_index"]) + off)
            ys.append(torch.from_numpy(m["y"])); ms.append(torch.from_numpy(m["loss_mask"])); off += m["num_nodes"]
        batches.append((torch.cat(xs), torch.cat(eis, 1), torch.cat(ys), torch.cat(ms)))

    def step(i):
        x, ei, y, m = batches[i % len(batches)]
        opt.zero_grad()
        loss = crit(model(x, ei, None), y, m)
        loss.backward()
        opt.step()
        return loss.item()

    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(warmup + i)
    dt = time.perf_counter() - t0
    return BATCH * steps / dt, dt / steps * 1e3


def cpu_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"os_cpu_count": os.cpu_count(), "torch_threads": torch.get_num_threads(), "cpu_model": model}


def run_reference(args, rank, world, emit):
    """Reference arm: the reference's own CPU implementation of the path (oracle port - PyG is not installable here) on ALL
    host cores, on this arm's config/metric/unit.  A step = one 4 x 50k-node batch (the per-GPU batch of the config) through
    fwd + bwd + AdamW: a bounded sample of the workload (~2 s per step on 16 cores).  --steps / --warmup are honoured; under
    torchrun rank 0 alone runs (with every core: the thread count is set explicitly), the other ranks exit 0."""
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    meshes = make_meshes(range(BATCH * min(4, steps)), args.mesh)
    value, ms = cpu_training_throughput(meshes, steps, warmup)
    info = cpu_info()
    sample = (f"{warmup} warm-up + {steps} timed fwd+bwd+AdamW steps, each on one 4x50k-node batch (cycling {len(meshes) // BATCH} batch(es)); "
              f"oracle port of the PyG model, torch CPU fp32, {info['torch_threads']} threads")
    line = {
        "impl": "reference", "metric": "train_meshes_per_sec", "value": value, "unit": "meshes/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "meshes/s", "cores": info["torch_threads"], "kind": "port", "sample": sample, **info},
        "e2e": {"value": value, "unit": "meshes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args, world):
    return {
        "workload": f"cfg2: GraphSAGE fwd+bwd+AdamW, {N_MESHES} synthetic {NODES}-node {'surface-triangle' if args.mesh == 'tri' else 'tet-lattice'} "
                    f"wing meshes, hidden {HIDDEN}, {LAYERS} SAGE layers, fp32, dropout {DROPOUT}, batch {BATCH} meshes/step/GPU",
        "hidden": HIDDEN, "layers": LAYERS, "batch_meshes_per_gpu": BATCH, "nodes_per_mesh": NODES, "global_batch_meshes": BATCH * world,
        "parallelism": f"dp{world} by mesh" if world > 1 else "single GPU",
        "l2_policy": "no flush: every step reads a different 4-mesh batch and streams > 1.5 GB of activations (L2 = 126 MB)",
    }


# --------------------------------------------------------------------------------------------
# parity gates printed with the perf numbers (SURVEY 8d) - the oracle is used as the CHECKER only, next to the CPU baseline
# --------------------------------------------------------------------------------------------
def parity_gates(device):
    """CSR bit-exact, forward max|d|/max|ref| and the worst per-parameter gradient rel-L2 of the product path against the
    oracle on identical weights and one identical 20k-node mesh (config 1's size), dropout 0, H/L of the benchmarked model."""
    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel, MaskedMSELoss
    from oracle import csr_oracle_c
    from oracle.sage_oracle import GraphSAGEModelRef, MaskedMSELossRef

    mesh = _synth().surface_tri_wing(20000, seed=4242)
    x, ei = torch.from_numpy(mesh["x"]), torch.from_numpy(mesh["edge_index"])
    y, m = torch.from_numpy(mesh["y"]), torch.from_numpy(mesh["loss_mask"])
    torch.manual_seed(42)
    ref = GraphSAGEModelRef(10, HIDDEN, 1, LAYERS, dropout=0.0)
    model = GraphSAGEModel(10, HIDDEN, 1, LAYERS, dropout=0.0)
    model.load_state_dict(ref.state_dict(), strict=True)
    model = model.to(device)
    g = ops.get_graph(ei.to(device), x.shape[0], want_perm=True)
    o = csr_oracle_c(mesh["edge_index"], x.shape[0])
    csr_ok = bool(torch.equal(g.rowptr.cpu(), torch.from_numpy(o[0])) and torch.equal(g.col.cpu(), torch.from_numpy(o[1]))
                  and torch.equal(g.perm.cpu(), torch.from_numpy(o[2])))
    out_ref = ref(x, ei)
    MaskedMSELossRef()(out_ref, y, m).backward()
    out = model(x.to(device), ei.to(device))
    MaskedMSELoss()(out, y.to(device), m.to(device)).backward()
    fwd = ((out.detach().cpu() - out_ref.detach()).abs().max() / out_ref.detach().abs().max()).item()
    ref64 = GraphSAGEModelRef(10, HIDDEN, 1, LAYERS, dropout=0.0).double()
    ref64.load_state_dict({k: v.double() for k, v in ref.state_dict().items()})
    MaskedMSELossRef()(ref64(x.double(), ei), y.double(), m).backward()
    rel = lambda a, b: ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()
    worst32 = max(rel(p.grad.cpu(), pr.grad) for p, pr in zip(model.parameters(), ref.parameters()))
    worst64 = max(rel(p.grad.cpu(), p64.grad) for p, p64 in zip(model.parameters(), ref64.parameters()))
    oracle64 = max(rel(pr.grad, p64.grad) for pr, p64 in zip(ref.parameters(), ref64.parameters()))
    ops.clear_graph_cache()
    return {"csr_bit_exact": csr_ok, "fwd_rel_err": fwd, "grad_rel_l2_worst_vs_fp32_oracle": worst32,
            "grad_rel_l2_worst_vs_fp64_oracle": worst64, "fp32_oracle_grad_rel_l2_vs_fp64": oracle64, "tolerance_fp32": 1e-5,
            "mesh": "surface-tri 20k nodes, seed 4242", "hidden": HIDDEN, "layers": LAYERS,
            "pass": bool(csr_ok and fwd < 1e-5 and worst64 < max(1e-5, 3 * oracle64))}


# --------------------------------------------------------------------------------------------
# BASELINE.json config 4: aggregation roofline on the 2M-node / 27M-edge tet lattice (N = 1 only)
# --------------------------------------------------------------------------------------------
CFG4_DIMS = (38, 114, 462)  # thickness x chord x span nodes: 2 001 384 nodes, 27.3 M directed edges


def cfg4_lattice_device(dims, device, order="native", seed=42):
    """The graph of ``synth.tet_lattice_wing(dims=...)`` (Kuhn 6-tet split of a hex lattice mapped into the wing: 14
    neighbours per interior node; node id = (iz*ny + iy)*nx + ix) and its normalised positions, generated on the device
    (27 M edges take ~20 s of numpy on the host).  ``order='random'``: nodes relabelled by a random permutation.
    Same edge SET as the numpy generator (tests/test_bench_helpers.py)."""
    nx, ny, nz = dims
    n = nx * ny * nz
    idx = torch.arange(n, device=device, dtype=torch.int64).view(nz, ny, nx)
    parts = []
    for dx, dy, dz in ((1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (0, 1, 1), (1, 0, 1), (1, 1, 1)):
        a = idx[: nz - dz, : ny - dy, : nx - dx].reshape(-1)
        b = idx[dz:, dy:, dx:].reshape(-1)
        parts += [torch.stack([a, b]), torch.stack([b, a])]
    ei = torch.cat(parts, dim=1)
    g = torch.Generator(device=device).manual_seed(seed)
    ei = ei[:, torch.randperm(ei.shape[1], device=device, generator=g)]  # edge order carries no information (dataset.py:39-63)
    ix = (idx % nx).reshape(-1).double()
    iy = ((idx // nx) % ny).reshape(-1).double()
    iz = (idx // (nx * ny)).reshape(-1).double()
    u, v, w = iy / max(ny - 1, 1), iz / max(nz - 1, 1), ix / max(nx - 1, 1) * 2.0 - 1.0
    span, chord, sweep, tc = 1.5, 0.35, 15.0, 0.10
    uc = u.clamp(0.0, 1.0)
    naca = 5.0 * tc * (0.2969 * uc.sqrt() - 0.1260 * uc - 0.3516 * uc ** 2 + 0.2843 * uc ** 3 - 0.1015 * uc ** 4)
    Y = v * span
    pos = torch.stack([u * chord + Y * float(np.tan(np.deg2rad(sweep))), Y, w * naca * chord], dim=1).float()
    lo, hi = pos.min(dim=0).values, pos.max(dim=0).values
    rng_ = torch.where(hi - lo < 1e-8, torch.ones_like(lo), hi - lo)
    pos_n = (pos - lo) / rng_  # dataset.py:130-136
    if order == "random":
        relabel = torch.randperm(n, device=device, generator=g)  # old id -> new id
        inv = torch.empty_like(relabel)
        inv[relabel] = torch.arange(n, device=device)
        ei = relabel[ei]
        pos_n = pos_n[inv]
    elif order != "native":
        raise ValueError(order)
    return ei.contiguous(), pos_n.contiguous(), n


def aggregation_cfg4(device, pk, iters=20):
    """north_star's aggregation target (>= 60 % of HBM peak) is scored on config 4: one mean-aggregation launch over the
    2M-node lattice, H = 256 bf16, native and random node order, L2 flushed between launches, CUDA events.
    ``A_min = 2*N*H*b + 4*E + 4*(N+1)`` (SURVEY 8d)."""
    from deep_fem_uav_wing.gnn import ops

    H = 256
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    out = {"hidden": H, "dtype": "bf16", "lattice": list(CFG4_DIMS), "l2": "flushed between launches (256 MB write)", "iters": iters}
    for order in ("native", "random"):
        ei, pos_n, n = cfg4_lattice_device(CFG4_DIMS, device, order)
        E = int(ei.shape[1])
        x = torch.randn(n, H, device=device, generator=torch.Generator(device=device).manual_seed(1)).bfloat16()
        amin = 2 * n * H * 2 + 4 * E + 4 * (n + 1)
        ent = {"N": n, "E": E, "A_min_MB": round(amin / 1e6, 1), "A_gather_MB": round((E * H * 2 + n * H * 2 + 4 * E + 4 * (n + 1)) / 1e6, 1)}
        # the path the model takes is timed FIRST: timed right behind the slow comparison paths (2.1 / 2.8 ms per launch on the randomly
        # numbered lattice, 60+ launches) the same kernel measured 600-625 us instead of 495-503 us (tools/cfg4_random_probe.py)
        for name, (fn, info) in reversed(list(ops.cfg4_aggregation_paths(ei, n, pos_n, x).items())):
            if os.environ.get("DFW_BENCH_VERBOSE"):
                print(f"[cfg4] {order} {name}", file=sys.stderr, flush=True)
            for _ in range(3):
                fn()
            ts = []
            for _ in range(iters):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize(device)
                ts.append(a.elapsed_time(b) * 1e-3)
            ts.sort()
            med = ts[len(ts) // 2]
            ent[name] = {"us": round(med * 1e6, 1), "p10_us": round(ts[len(ts) // 10] * 1e6, 1), "p90_us": round(ts[-1 - len(ts) // 10] * 1e6, 1),
                         "achieved_GBps": round(amin / med / 1e9, 1), "frac": round(amin / med / 1e9 / pk["hbm_gbs"], 4), **info}
        best = min((k for k in ent if isinstance(ent[k], dict)), key=lambda k: ent[k]["us"])
        ent["best"] = {"path": best, "us": ent[best]["us"], "frac": ent[best]["frac"]}
        # the whole config-4 forward through the public API (GraphSAGEModel, H = 256, L = 3, bf16, eval): the first call
        # prepares the graph (CSR, block plan, k-d relabelling where it pays: one-time per mesh), later calls reuse it
        from deep_fem_uav_wing.gnn.model import GraphSAGEModel

        ops.clear_graph_cache()
        ops._INF_CACHE.clear()
        torch.manual_seed(0)
        model = GraphSAGEModel(10, H, 1, 3).to(device).eval().set_compute_dtype(torch.bfloat16)
        model.mesh_plan = "always"  # a static mesh: prepare it on the first call ('auto' would on the second)
        nrm = torch.nn.functional.normalize(torch.randn(n, 3, device=device, generator=torch.Generator(device=device).manual_seed(2)), dim=1)
        feats = torch.cat([pos_n, nrm, torch.full((n, 4), 0.5, device=device)], dim=1).contiguous()
        with torch.no_grad():
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            model(feats, ei)
            torch.cuda.synchronize(device)
            first_ms = (time.perf_counter() - t0) * 1e3
            fts = []
            for _ in range(5):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                model(feats, ei)
                b.record()
                torch.cuda.synchronize(device)
                fts.append(a.elapsed_time(b))
        fts.sort()
        ent["forward_L3"] = {"ms": round(fts[len(fts) // 2], 3), "nodes_per_sec": n / (fts[len(fts) // 2] * 1e-3), "first_call_incl_graph_preparation_ms": round(first_ms, 1),
                             "what": "GraphSAGEModel(10, 256, 1, 3) bf16 eval forward on the prepared graph (median of 5, L2 flushed)"}
        del model, feats, nrm
        out[order] = ent
        del ei, pos_n, x
        ops.clear_graph_cache()
        torch.cuda.empty_cache()
    out["peak_GBps"] = pk["hbm_gbs"]
    out["peak_source"] = pk["_source"]
    return out


def partitioned_cfg4(device, rank, world, iters=5):
    """SURVEY 8f-4: the config-4 mesh (2 M nodes, H = 256, L = 3, bf16, eval) as ONE forward partitioned over the ranks -
    1-D node partition in k-d order, one NCCL all-to-all of halo rows per SAGE layer (gnn/partition.py).  STRONG scaling of a
    single mesh (the training arms of this line are weak scaling); time = max over ranks."""
    import torch.distributed as dist

    from deep_fem_uav_wing.gnn.model import GraphSAGEModel
    from deep_fem_uav_wing.gnn.partition import PartitionedMeshInference

    ei, pos_n, n = cfg4_lattice_device(CFG4_DIMS, device, "native")
    nrm = torch.nn.functional.normalize(torch.randn(n, 3, device=device, generator=torch.Generator(device=device).manual_seed(2)), dim=1)
    feats = torch.cat([pos_n, nrm, torch.full((n, 4), 0.5, device=device)], dim=1).contiguous()
    torch.manual_seed(0)
    model = GraphSAGEModel(10, 256, 1, 3).to(device).eval().set_compute_dtype(torch.bfloat16)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    pm = PartitionedMeshInference(model, feats, ei)
    torch.cuda.synchronize(device)
    prep_ms = (time.perf_counter() - t0) * 1e3
    del ei, feats, nrm
    for _ in range(2):
        pm()
    ts = []
    for _ in range(iters):
        dist.barrier()
        torch.cuda.synchronize(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = pm()
        b.record()
        torch.cuda.synchronize(device)
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=device)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ts.append(float(ms.item()))
    ts.sort()
    halo = torch.tensor([float(pm.halo_rows)], device=device)
    dist.all_reduce(halo, op=dist.ReduceOp.MAX)
    res = {"ms": round(ts[len(ts) // 2], 3), "nodes_per_sec": n / (ts[len(ts) // 2] * 1e-3), "N": n, "ranks": world, "hidden": 256, "layers": 3, "dtype": "bf16",
           "max_halo_rows_per_rank": int(halo.item()), "rows_per_rank": pm.part.n_own, "one_time_partitioning_ms": round(prep_ms, 1),
           "scaling": "strong (one mesh)", "exchange": "all_to_all_single of halo rows per SAGE layer (NCCL)", "finite": bool(torch.isfinite(out).all())}
    del pm, model
    torch.cuda.empty_cache()
    return res


# --------------------------------------------------------------------------------------------
# BASELINE.json config 1: the reference's own CPU-runnable case - ONE 20k-node mesh, H = 64, L = 3, fp32, eval (inference_gnn.py:224-328)
def cfg1_block(device, with_cpu=True, iters=50):
    """Latency of one inference forward on a 20k-node mesh (surface-tri and tet lattice): launched from Python through the public
    API (``model(x, edge_index)``, CSR cached after the first call: eval + no_grad takes ``dfw_graphsage_forward``), replayed from a
    CUDA graph, and the oracle port on the host cores beside it.  Wall-clock per call incl. the host side (synchronised)."""
    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.graphed import GraphedForward
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    synth = _synth()
    out = {"hidden": 64, "layers": 3, "dtype": "f32", "nodes": 20000, "iters": iters}
    for kind, gen in (("tri", synth.surface_tri_wing), ("tet", synth.tet_lattice_wing)):
        m = gen(20000, seed=42)
        x, ei = torch.from_numpy(m["x"]).to(device), torch.from_numpy(m["edge_index"]).to(device)
        torch.manual_seed(42)
        model = GraphSAGEModel(10, 64, 1, 3).to(device).eval()

        def wall(fn):
            for _ in range(5):
                fn()
            torch.cuda.synchronize(device)
            ts = []
            for _ in range(iters):
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize(device)
                ts.append(time.perf_counter() - t0)
            ts.sort()
            return ts[len(ts) // 2] * 1e3

        with torch.no_grad():
            eager_ms = wall(lambda: model(x, ei))
            replay, _ = GraphedForward(model).capture_resident(x, ops.get_graph(ei, x.shape[0]))
            graph_ms = wall(replay)
        ent = {"N": int(x.shape[0]), "E": int(ei.shape[1]), "eager_ms": round(eager_ms, 4), "cuda_graph_ms": round(graph_ms, 4),
               "nodes_per_sec_graph": x.shape[0] / (graph_ms * 1e-3)}
        if with_cpu:
            from oracle.sage_oracle import GraphSAGEModelRef

            torch.set_num_threads(os.cpu_count() or 1)
            ref = GraphSAGEModelRef(10, 64, 1, 3, dropout=0.0).eval()
            ref.load_state_dict({k: v.cpu() for k, v in model.state_dict().items()}, strict=True)
            xc, ec = x.cpu(), ei.cpu()
            with torch.no_grad():
                ref(xc, ec)
                cs = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    o_ref = ref(xc, ec)
                    cs.append(time.perf_counter() - t0)
                got = model(x, ei).cpu()
            cs.sort()
            ent["cpu_oracle_ms"] = round(cs[len(cs) // 2] * 1e3, 3)
            ent["fwd_rel_err_vs_oracle"] = float((got - o_ref).abs().max() / o_ref.abs().max())
            torch.set_num_threads(1)
        out[kind] = ent
        ops.clear_graph_cache()
    return out


# BASELINE.json config 5: design-screening batch inference, case list sharded over the ranks, no communication
# --------------------------------------------------------------------------------------------
def cfg5_block(device, rank, world, dist_on, n_cases=10000, nodes=20000, per_launch=16, distinct=48):
    """Every rank takes ``case_ids[rank::world]`` (inference_gnn.py:380-398 loops the cases independently).  Per launch
    ``per_launch`` packed cases (pos, normal, faces, globals - the content of the reference's three case files) go from
    pinned host memory to the device, the graph is built there (``dfw_faces_to_csr`` + ``dfw_node_features_batched``), one
    forward (H = 128, L = 4) runs and the per-case mean prediction comes back to the host.  ``distinct`` different synthetic
    cases per rank are cycled (generating 10k on the host would take minutes); everything else is per case.
    fp32 is the headline (`value`); the same loop with bf16 activations is reported beside it."""
    import torch.distributed as dist

    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    synth = _synth()
    mine = len(range(rank, n_cases, world))
    cases = []
    for i in range(min(distinct, mine)):
        m = synth.surface_tri_wing(nodes, seed=1000 + rank * distinct + i)
        p = m["params"]
        gp = [(p["span_m"] - 1.0) / 1.0, (p["chord_m"] - 0.2) / 0.3, p["sweep_deg"] / 30.0, (p["thickness_ratio"] - 0.05) / 0.10]  # dataset.py:122-127
        cases.append({"pos": torch.from_numpy(m["pos"]).pin_memory(), "normal": torch.from_numpy(m["normal"]).pin_memory(),
                      "faces": torch.from_numpy(m["faces"].astype(np.int64)).pin_memory(), "n": m["num_nodes"],
                      "gp": torch.tensor(gp, dtype=torch.float32).pin_memory()})
    copy_stream = torch.cuda.Stream(device=device)
    n_launch = (mine + per_launch - 1) // per_launch
    res_pin = torch.zeros(n_launch + 2, per_launch, dtype=torch.float32).pin_memory()  # every case's mean prediction, read after the loop
    groups = [[cases[(l * per_launch + j) % len(cases)] for j in range(min(per_launch, mine - l * per_launch))] for l in range(n_launch)]
    counters = {"h2d": 0}

    def stage(group):
        with torch.cuda.stream(copy_stream):
            dev = []
            for c in group:
                dev.append((c["pos"].to(device, non_blocking=True), c["normal"].to(device, non_blocking=True),
                            c["faces"].to(device, non_blocking=True), c["n"], c["gp"].to(device, non_blocking=True)))
                counters["h2d"] += c["pos"].numel() * 4 + c["normal"].numel() * 4 + c["faces"].numel() * 8 + 16
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return dev, ev

    def run(model, dev, slot):
        fs, off, ptr = [], 0, [0]
        for _, _, faces, n, _ in dev:
            fs.append(faces + off)
            off += n
            ptr.append(off)
        # ONE feature launch pair (per-case min-max normalisation, dataset.py:130-136) and ONE graph build for the whole launch (the
        # faces of the disjoint union), neither with a host read: the host runs ahead of the device for the whole screening loop
        x, _ = ops.node_features_batched(torch.cat([d[0] for d in dev]), torch.cat([d[1] for d in dev]), None, torch.stack([d[4] for d in dev]),
                                         torch.tensor(ptr, dtype=torch.int64).pin_memory().to(device, non_blocking=True), max(d[3] for d in dev))
        g, _ = ops.faces_to_graph(torch.cat(fs), off, want_edge_index=False, sync=False)
        with torch.no_grad():
            out = model(x, g)  # eval + no_grad: ONE C call (dfw_graphsage_forward)
        nc = len(dev)
        if all(ptr[i + 1] - ptr[i] == ptr[1] for i in range(nc)):
            means = out.float().view(nc, -1).mean(dim=1)
        else:
            means = torch.stack([out[ptr[i]:ptr[i + 1]].float().mean() for i in range(nc)])
        res_pin[slot, :nc].copy_(means, non_blocking=True)

    def measure(dtype):
        torch.manual_seed(42)
        model = GraphSAGEModel(10, HIDDEN, 1, LAYERS).to(device).eval().set_compute_dtype(dtype)
        for l in range(2):  # warm-up
            dev, ev = stage(groups[l % n_launch])
            torch.cuda.current_stream(device).wait_event(ev)
            run(model, dev, n_launch + l)
        torch.cuda.synchronize(device)
        counters["h2d"] = 0
        k0 = ops.LAUNCH_COUNTER["kernels"]
        if dist_on:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        nxt = stage(groups[0])
        for l in range(n_launch):
            dev, ev = nxt
            if l + 1 < n_launch:
                nxt = stage(groups[l + 1])  # H2D of the next launch (copy stream) overlaps this launch's graph build + forward
            torch.cuda.current_stream(device).wait_event(ev)
            run(model, dev, l)
        b.record()
        torch.cuda.synchronize(device)
        assert bool(torch.isfinite(res_pin[:n_launch]).all()), "config 5: a case produced a non-finite mean prediction"
        ms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=device)
        if dist_on:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), ops.LAUNCH_COUNTER["kernels"] - k0

    ms32, launches = measure(torch.float32)
    h2d = counters["h2d"]
    ms16, _ = measure(torch.bfloat16)
    return {"value": n_cases / (ms32 * 1e-3), "unit": "meshes/s", "n_cases": n_cases, "cases_per_rank": mine, "nodes_per_case": nodes,
            "nodes_per_sec": n_cases * nodes / (ms32 * 1e-3), "ms_total": ms32, "cases_per_launch": per_launch, "hidden": HIDDEN,
            "layers": LAYERS, "dtype": "f32", "h2d_bytes_per_case": h2d // max(mine, 1), "d2h_bytes_per_case": 4,
            "gpu_launches": launches, "sharding": "case_ids[rank::world], no communication",
            "bf16": {"value": n_cases / (ms16 * 1e-3), "unit": "meshes/s", "ms_total": ms16, "what": "same loop, bf16 activations (fp32 first layer, fp32 accumulation)"},
            "path": "packed case (pos, normal, faces) in pinned host memory -> H2D -> dfw_node_features_batched + dfw_faces_to_csr (copy stream, "
                    "one launch ahead) -> GraphSAGEModel forward (dfw_graphsage_forward, one C call) -> per-case mean prediction D2H", "data": f"{len(cases)} distinct synthetic cases per rank, cycled"}


# --------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mesh", default="tri", choices=["tri", "tet"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the tet-batch, config-4 aggregation and config-5 blocks")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels one by one instead of replaying CUDA graphs (both arms)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed training step's loss and parameters to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner) write to fd 1 too, so
    # everything else is routed to stderr and the JSON line goes to the saved descriptor.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        run_reference(args, rank, world, emit)
        return

    import torch.distributed as dist

    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.ddp import MeshDataParallel
    from deep_fem_uav_wing.gnn.loader import Batch, DataLoader
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel, MaskedMSELoss

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device: the product path has no CPU fallback")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    dist_on = world > 1
    if dist_on:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    assert world == args.gpus or not dist_on, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    # ---- parity gates, printed with the perf numbers (rank 0; the oracle is the checker) ----------
    gates = parity_gates(device) if (rank == 0 and not args.no_cpu_baseline) else None
    # The oracle above spins up torch's CPU intra-op pool (one OpenMP worker per core, busy-waiting between parallel regions); left
    # that wide, those workers compete with the loader's prefetch thread for the host cores in the end-to-end arm (measured: e2e
    # 1272 instead of 1540-1630 meshes/s).  The GPU arms need no CPU intra-op parallelism; the CPU arms set their own thread count.
    torch.set_num_threads(1)

    # ---- data: this rank's shard of the 200 meshes (mesh id = rank + k*world) -----------------
    steps, warmup = args.steps, args.warmup
    n_local = min(N_MESHES // world, BATCH * (steps + warmup))
    n_local = max(BATCH, n_local // BATCH * BATCH)
    ids = [rank + k * world for k in range(n_local)]
    meshes = make_meshes(ids, args.mesh)
    datas = [to_data(m) for m in meshes]
    n_batches = n_local // BATCH

    torch.manual_seed(42)
    model = GraphSAGEModel(10, HIDDEN, 1, LAYERS, DROPOUT).to(device).train()
    ddp = MeshDataParallel(model) if dist_on else None
    opt = torch.optim.AdamW(model.parameters(), lr=LR, weight_decay=WD, fused=True, capturable=True)
    crit = MaskedMSELoss()

    def train_step(b, read_loss=False, return_loss=False, graph=None):
        if ddp is not None:
            ddp.zero_grad()
        else:
            opt.zero_grad(set_to_none=True)
        out = model(b.x, graph if graph is not None else b.edge_index, b.batch)
        loss = crit(out, b.y, b.loss_mask)
        if ddp is not None:
            ddp.scale_loss(loss, crit.last_count).backward()
            ddp.finish()
        else:
            loss.backward()
        opt.step()
        if return_loss:
            return loss.detach()
        return loss.item() if read_loss else None

    # ---- arm 1: device-resident batches, CSR cached (one-time build per batch) -----------------
    resident = [Batch.from_data_list(datas[i * BATCH:(i + 1) * BATCH]).to(device) for i in range(n_batches)]
    graphs = [ops.get_graph(b.edge_index, b.x.shape[0]) for b in resident]  # one-time CSR builds, held here: "CSR cached" does
    for g_ in graphs:                                                        # not depend on the size of ops.get_graph's LRU
        g_.transpose()
    for i in range(warmup):
        train_step(resident[i % n_batches], graph=graphs[i % n_batches])
    # One CUDA graph per resident batch (captured ON the batch's tensors: no staging copies, the cached CSR stays outside
    # the graph): a step costs one launch, so the device-resident number is not bounded by Python's ~2 ms of launch work
    # per step (--no-graph: kernels launched one by one).
    replays = None
    if not args.no_graph:
        from deep_fem_uav_wing.gnn.graphed import GraphedTrainStep

        rstep = GraphedTrainStep(model, crit, opt, ddp=ddp)
        replays, rlosses = zip(*[rstep.capture_resident(b.x, g_, b.y, b.loss_mask) for b, g_ in zip(resident, graphs)])
        for i in range(min(3, n_batches)):
            replays[i]()
    sampler = ClockSampler(local_rank)
    sampler.start()
    k0 = ops.LAUNCH_COUNTER["kernels"]
    if replays is not None:
        ms_total = timed_region(lambda i: replays[(warmup + i) % n_batches](), steps, dist_on, device)
        last_loss = rlosses[(warmup + steps - 1) % n_batches]
    else:
        eager_loss = [None]

        def eager_step(i):
            j = (warmup + i) % n_batches
            eager_loss[0] = train_step(resident[j], return_loss=True, graph=graphs[j])

        ms_total = timed_region(eager_step, steps, dist_on, device)
        last_loss = eager_loss[0]
    launches = ops.LAUNCH_COUNTER["kernels"] - k0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_loss, model)  # before the later arms step the model further
    value = BATCH * steps * world / (ms_total * 1e-3)

    # ---- inference arm (BASELINE metric: "train/infer"): eval-mode forward over the same resident batches ----
    model.eval()
    with torch.no_grad():
        for i in range(3):
            model(resident[i % n_batches].x, graphs[i % n_batches])
        if not args.no_graph:  # one CUDA graph per resident batch, like the training arm: 13 launches per forward are host-bound otherwise
            from deep_fem_uav_wing.gnn.graphed import GraphedForward

            fwd = GraphedForward(model)
            ireplays = [fwd.capture_resident(b.x, g_)[0] for b, g_ in zip(resident, graphs)]
            for r_ in ireplays[:3]:
                r_()
            ms_inf = timed_region(lambda i: ireplays[(warmup + i) % n_batches](), steps, dist_on, device)
        else:
            ms_inf = timed_region(lambda i: model(resident[(warmup + i) % n_batches].x, graphs[(warmup + i) % n_batches]), steps,
                                  dist_on, device)
    model.train()
    infer = {"value": BATCH * steps * world / (ms_inf * 1e-3), "unit": "meshes/s", "ms_per_step": ms_inf / steps,
             "nodes_per_sec": BATCH * steps * world * NODES / (ms_inf * 1e-3), "cuda_graph": not args.no_graph,
             "what": "eval-mode forward, device-resident batches, CSR cached"}

    # ---- roofline pass: same steps with per-launch CUDA events ---------------------------------
    prof_steps = min(steps, 8)
    ops.PROFILER = ops.KernelProfiler()
    overlap, ops.OVERLAP_DW = ops.OVERLAP_DW, False  # every kernel alone on its stream while its duration is measured
    for i in range(prof_steps):
        train_step(resident[i % n_batches], graph=graphs[i % n_batches])
    summ = ops.PROFILER.summary()
    ops.PROFILER = None
    ops.OVERLAP_DW = overlap
    pk = peaks()
    tot_ms = sum(r["ms"] for r in summ.values())
    kernels = {}
    for name, r in summ.items():
        avg_s = r["ms"] * 1e-3 / r["calls"]
        ent = {"calls_per_step": r["calls"] / prof_steps, "avg_us": round(avg_s * 1e6, 2), "share_of_kernel_time": round(r["ms"] / tot_ms, 4),
               "achieved_GBps": round(r["bytes"] / r["calls"] / avg_s / 1e9, 1),
               "hbm_frac": round(r["bytes"] / r["calls"] / avg_s / 1e9 / pk["hbm_gbs"], 4)}
        if r["flops"]:
            ent["achieved_TFLOPs"] = round(r["flops"] / r["calls"] / avg_s / 1e12, 2)
        kernels[name] = ent
    dom = max(summ, key=lambda k: summ[k]["ms"])
    d = kernels[dom]
    # DRAM traffic per launch of the same kernel on the same shapes, from the committed `ncu --set full` captures
    # (tools/ncu_capture_all.sh -> tools/ncu_summary.py --json); null when no capture of that kernel is on file
    traffic, traffic_src = None, None
    # (an EARLIER capture on another box: `_capture` in that file names the commit and date it was taken at; the DRAM bytes
    # of a kernel depend on its shapes and tiling, not on the box, so they stay valid until the kernel's tiling changes)
    tpath = next((q for q in (os.path.join(REPO, "profiles", f) for f in ("r02_ncu_traffic.json", "r01_ncu_traffic.json")) if os.path.exists(q)), None)
    cap = {"aggregate": "agg_cfg2", "aggregate_bwd": "aggs_cfg2", "linear_fwd": "lin_fwd_fp32",
           "linear_bwd_input": "lin_fwd_fp32", "linear_bwd_weight": "dw_fp32", "epilogue_bwd": "epi_bwd_fp32"}
    if tpath is not None:
        tj = json.load(open(tpath))
        find = lambda key: next((v for k, v in tj.items() if isinstance(v, dict) and k.endswith(key)), None) if key else None
        for name, ent in kernels.items():
            c = find(cap.get(name))
            if c:
                ent["ncu_dram_bytes_per_launch"] = c["dram_bytes"]
        c = find(cap.get(dom))
        if c:
            traffic = c["dram_bytes"]
            traffic_src = {"file": os.path.relpath(tpath, REPO), "entry": cap[dom], "capture": tj.get("_capture", "round 1 (r01b captures, commit 5c226f5 era)")}
    roofline = {"kernel": dom, "bound": "hbm", "achieved": d["achieved_GBps"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": d["hbm_frac"], "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": summ[dom]["bytes"] / summ[dom]["calls"], "peak_source": pk["_source"],
                "note": "algorithmic bytes per launch (DESIGN.md) / mean CUDA-event duration; every kernel of the step is listed under `kernels`"}

    # ---- arm 2: end to end through the public API from pinned host memory ----------------------
    e2e, gstep = None, None
    if not args.no_e2e:
        # (build_graph=True - the batch's CSR built by the prefetch worker on the copy stream - was measured: 2.74 vs 2.75 ms per
        # step once the caching allocator has settled, and 3.9 ms while it still grows; the CSR build stays inside the captured step)
        host_loader = DataLoader(datas, batch_size=BATCH, shuffle=False, device=device)
        h2d = sum(int(getattr(datas[j], k).numel() * getattr(datas[j], k).element_size()) for j in range(BATCH)
                  for k in ("x", "edge_index", "y", "loss_mask")) + 8 * (BATCH + 1)

        def epoch_iter():
            while True:
                for b in host_loader:
                    yield b

        it = epoch_iter()
        ops.clear_graph_cache()
        for _ in range(warmup):
            train_step(next(it), read_loss=True)
        # every step's loss is read back on the host inside the timed region; the read of step i happens after
        # step i+1 has been enqueued (one-step software pipeline), so the GPU is never idle while Python launches
        loss_pin = torch.empty(steps, dtype=torch.float32).pin_memory()
        loss_evs, loss_vals = [], []

        use_graph = not args.no_graph
        if use_graph:
            from deep_fem_uav_wing.gnn.graphed import GraphedTrainStep

            gstep = GraphedTrainStep(model, crit, opt, eager_steps=2, ddp=ddp)
            for _ in range(4):  # first calls of the shape run eagerly, then the step is captured
                b = next(it)
                gstep(b.x, b.edge_index, b.y, b.loss_mask, graph=getattr(b, "graph", None))

        def e2e_step(i):
            if use_graph:
                b = next(it)
                loss = gstep(b.x, b.edge_index, b.y, b.loss_mask, graph=getattr(b, "graph", None))
            else:
                loss = train_step(next(it), return_loss=True)
            loss_pin[i:i + 1].copy_(loss.reshape(1).float(), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            loss_evs.append(ev)
            if i > 0:
                loss_evs[i - 1].synchronize()
                loss_vals.append(float(loss_pin[i - 1]))
            if i == steps - 1:
                ev.synchronize()
                loss_vals.append(float(loss_pin[i]))

        ms_e2e = timed_region(e2e_step, steps, dist_on, device)
        assert len(loss_vals) == steps and all(np.isfinite(loss_vals)), "e2e losses were not all read back"
        e2e = {"value": BATCH * steps * world / (ms_e2e * 1e-3), "unit": "meshes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e / steps, "cuda_graph": bool(use_graph),
               "path": "DataLoader(pinned host Data, device=cuda) -> H2D on a copy stream (1 batch prefetch) -> GraphSAGEModel(x, edge_index, batch) "
                       "incl. on-device CSR build -> MaskedMSELoss -> backward -> AdamW (one CUDA graph per batch shape, gradient all-reduce captured with it) -> loss copied to pinned host memory and read "
                       "(every step, one step behind the launch front)"}

    # ---- the other graph family of config 2 (BASELINE.md scores both): tet-lattice batch, degree ~14 ----------------------
    tet = None
    if args.mesh == "tri" and not args.no_extras:
        tdatas = [to_data(m) for m in make_meshes([5000 + rank * 2 * BATCH + i for i in range(2 * BATCH)], "tet")]
        tres = [Batch.from_data_list(tdatas[i * BATCH:(i + 1) * BATCH]).to(device) for i in range(2)]
        for b in tres:
            ops.get_graph(b.edge_index, b.x.shape[0]).transpose()
        for i in range(3):
            train_step(tres[i % 2])
        tsteps = min(steps, 20)
        if not args.no_graph:
            treplays = [rstep.capture_resident(b.x, b.edge_index, b.y, b.loss_mask)[0] for b in tres]
            for r_ in treplays:
                r_()
            ms_tet = timed_region(lambda i: treplays[i % 2](), tsteps, dist_on, device)
        else:
            ms_tet = timed_region(lambda i: train_step(tres[i % 2]), tsteps, dist_on, device)
        tet = {"value": BATCH * tsteps * world / (ms_tet * 1e-3), "unit": "meshes/s", "ms_per_step": ms_tet / tsteps, "steps": tsteps,
               "nodes_per_batch": int(tres[0].x.shape[0]), "edges_per_batch": int(tres[0].edge_index.shape[1]),
               "what": "same training step, device-resident, on 4 x 50k-node TET-lattice meshes (degree ~14), 2 batches cycled"}

    # ---- config 5 (every N), config 4's aggregation roofline (N = 1), config 4 partitioned over the ranks (N > 1) ---------
    cfg5 = agg4 = part4 = cfg1 = None
    if not args.no_extras:
        cfg5 = cfg5_block(device, rank, world, dist_on)
        if rank == 0 and world == 1:
            cfg1 = cfg1_block(device, with_cpu=not args.no_cpu_baseline)
        if world == 1:
            agg4 = aggregation_cfg4(device, pk)
        else:
            part4 = partitioned_cfg4(device, rank, world)

    # ---- CPU baseline (rank 0, N=1 only) ---------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, ms = cpu_training_throughput(meshes[:2 * BATCH], steps=8, warmup=2)
        info = cpu_info()
        v1, ms1 = cpu_training_throughput(meshes[:BATCH], steps=1, warmup=0, threads=1)
        cpu = {"value": v, "unit": "meshes/s", "cores": info["torch_threads"], "kind": "port", "ms_per_step": ms,
               "sample": "2 warm-up + 8 timed fwd+bwd+AdamW steps over the first two 4x50k-node batches of this workload (oracle port of the PyG model, torch CPU fp32, all host threads)",
               "one_thread": {"value": v1, "unit": "meshes/s", "ms_per_step": ms1, "sample": "1 timed step, torch.set_num_threads(1)"},
               **info}

    if rank == 0:
        line = {
            "metric": "train_meshes_per_sec", "value": value, "unit": "meshes/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, world),
            "nodes_per_sec": value * NODES, "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "infer": infer,
            "aggregation": {"kernel": "dfw_sage_aggregate (forward mean, this workload)", "achieved_GBps": kernels.get("aggregate", {}).get("achieved_GBps"),
                            "hbm_frac": kernels.get("aggregate", {}).get("hbm_frac")},
            "aggregation_cfg4": agg4, "partitioned_cfg4": part4, "cfg1": cfg1, "cfg5": cfg5, "tet_batch": tet, "parity": gates,
            "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu,
        }
        emit(line)
    if dist_on:
        # the captured steps hold NCCL work: release the graphs, agree that everybody is done, and leave without
        # tearing the communicator down (destroying a communicator that graphs still reference can block)
        gstep = rstep = replays = None
        import gc

        gc.collect()
        torch.cuda.synchronize(device)
        dist.barrier()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
