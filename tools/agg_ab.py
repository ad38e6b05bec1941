#!/usr/bin/env python3
"""Timing of the gather aggregation on the config-2 batch shapes."""
import json, os, sys, torch
REPO = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path[:0] = [REPO, os.path.join(REPO, "deep-fem-uav-wing_b200")]
import bench
from deep_fem_uav_wing.gnn import ops, synth
from deep_fem_uav_wing.gnn.loader import Batch
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
def t(fn, iters=30):
    for _ in range(3): fn()
    ts = []
    for _ in range(iters):
        flush.zero_(); a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b) * 1e3)
    ts.sort(); return round(ts[len(ts) // 2], 1)
res = {}
for kind in ("tri", "tet"):
    b = Batch.from_data_list([bench.to_data(m) for m in bench.make_meshes(range(4), kind)]).to("cuda")
    g = ops.get_graph(b.edge_index, b.x.shape[0]); rp_t, col_t = g.transpose()
    for H, dt in ((128, torch.float32), (128, torch.bfloat16)):
        x = torch.randn(b.x.shape[0], H, device="cuda").to(dt)
        amin = 2 * x.numel() * x.element_size() + 4 * g.num_edges + 4 * (x.shape[0] + 1)
        f = t(lambda: ops.aggregate(g.rowptr, g.col, g.inv_deg, x)); bw = t(lambda: ops.aggregate_scaled(rp_t, col_t, g.inv_deg, x))
        res[f"{kind} {str(dt)[6:]}"] = {"fwd_us": f, "fwd_frac": round(amin / f / 1e3 / 6542.1, 3), "bwd_us": bw}
print(json.dumps(res))
