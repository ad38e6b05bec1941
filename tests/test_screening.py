"""FEM-free design screening (gnn/screening.py, scripts/screen_gnn.py): the two device kernels against numpy oracles,
batch independence, the screener against the existing per-case inference path, and the CLI on one and two GPUs."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from helpers import record
from test_gpu_data_path_exact import normals_f32_oracle

REPO = Path(__file__).resolve().parent.parent
PKG = REPO / "deep-fem-uav-wing_b200"


# ---- numpy oracles ---------------------------------------------------------------------------------------------------
def normals_oracle(pos, faces):
    """fp64 area-weighted vertex normals over the given (fp32) positions, and per vertex the sum of |face normal| of its
    incident faces (the scale of the fp32 rounding error)."""
    p = np.asarray(pos, dtype=np.float64)
    f = np.asarray(faces, dtype=np.int64)
    fn = np.cross(p[f[:, 1]] - p[f[:, 0]], p[f[:, 2]] - p[f[:, 0]])
    fa = np.linalg.norm(fn, axis=1)
    n, scale = np.zeros_like(p), np.zeros(len(p))
    for k in range(3):
        for c in range(3):
            n[:, c] += np.bincount(f[:, k], weights=fn[:, c], minlength=len(p))
        scale += np.bincount(f[:, k], weights=fa, minlength=len(p))
    return n, scale


def summary_oracle(pa, pos_y, case_ptr, mask=None, root_band=0.05, allowable=None):
    """[B,8] records of dfw_case_stress_summary from the fp32 stresses ``pa`` (the same expm1f values), in fp64."""
    out = []
    for b in range(len(case_ptr) - 1):
        r0, r1 = int(case_ptr[b]), int(case_ptr[b + 1])
        v, y = pa[r0:r1], pos_y[r0:r1]
        if mask is not None:
            scr = mask[r0:r1].astype(bool)
        elif r1 > r0:
            scr = y.astype(np.float64) > root_band * (float(y.max()) - float(y.min()))
        else:
            scr = np.zeros(0, bool)
        fin = np.isfinite(v)
        sel = scr & fin
        vs = v[sel].astype(np.float64)
        rows = np.nonzero(sel)[0]
        rec = [r1 - r0, int(scr.sum()), 0.0, -1, 0.0, float(v[fin].max()) if fin.any() else 0.0, 0, int((~fin).sum())]
        if vs.size:
            k = int(np.argmax(vs))  # first maximum = lowest row
            rec[2], rec[3], rec[4] = float(vs[k]), int(rows[k]), float(vs.sum() / vs.size)
            rec[6] = int((vs > allowable).sum()) if allowable else 0
        out.append(rec)
    return np.array(out, dtype=np.float64).reshape(-1, 8)


def _model(hidden=128, layers=4, seed=0, dtype=torch.float32):
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel

    torch.manual_seed(seed)
    return GraphSAGEModel(10, hidden, 1, layers).cuda().eval().set_compute_dtype(dtype)


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_pack_launches_order_budget_oversize_and_case_cap():
    from deep_fem_uav_wing.gnn.screening import MAX_CASES_PER_LAUNCH, pack_launches

    sizes = [100, 200, 50, 700, 30, 30, 1000, 10]
    groups = list(pack_launches(iter(sizes), lambda s: s, 300))
    assert [s for g in groups for s in g] == sizes  # input order kept, nothing lost
    assert groups == [[100, 200], [50], [700], [30, 30], [1000], [10]]  # oversize cases alone
    assert all(sum(g) <= 300 for g in groups if len(g) > 1)
    assert MAX_CASES_PER_LAUNCH == 65535
    many = list(pack_launches(iter([1] * 70000), lambda s: s, 10**9))
    assert [len(g) for g in many] == [65535, 70000 - 65535]
    with pytest.raises(ValueError):
        next(pack_launches([1], lambda s: s, 0))


def test_faces_to_rows_drops_unknown_ids():
    from deep_fem_uav_wing.gnn.screening import faces_to_rows

    rows, skipped = faces_to_rows(np.arange(5) + 1, np.array([[1, 2, 3], [3, 4, 5], [5, 6, 1], [0, 1, 2]]))
    assert rows.tolist() == [[0, 1, 2], [2, 3, 4]] and skipped == 2
    ids = np.array([40, 10, 30, 20])  # not consecutive, not sorted
    rows, skipped = faces_to_rows(ids, np.array([[10, 20, 30], [40, 10, 99]]))
    assert rows.tolist() == [[1, 3, 2]] and skipped == 1
    rows, _ = faces_to_rows(np.array([7, 8, 7]), np.array([[7, 8, 8]]))  # duplicated id: its last row, as the reference's dict
    assert rows.tolist() == [[2, 1, 1]]


def test_geometry_case_round_trip_and_version(tmp_path):
    from deep_fem_uav_wing.gnn import caseio, synth

    mesh = synth.surface_tri_wing(600, seed=3)
    path = synth.write_geometry_case(mesh, tmp_path)
    c = caseio.load_geometry_case(path)
    ref = synth.geometry_case(mesh)
    assert c["case_id"] == ref["case_id"] == mesh["case_id"] and c["params"] == mesh["params"]
    for k in ("node_id", "pos", "faces"):
        assert c[k].dtype == ref[k].dtype and c[k].tobytes() == ref[k].tobytes(), k
    z = dict(np.load(path))
    z["geometry_version"] = np.int64(caseio.GEOMETRY_VERSION + 1)
    bad = tmp_path / "bad.npz"
    np.savez(bad, **z)
    with pytest.raises(ValueError, match="version"):
        caseio.load_geometry_case(bad)
    synth.write_case_files(mesh, tmp_path / "root")
    fem = tmp_path / "root" / "data" / "raw"
    cid = mesh["case_id"]
    packed = caseio.pack_case(fem / "fem" / cid / "surface_results.npz", fem / "mesh" / cid / "boundary_sets.json",
                              fem / "geometry" / cid / "params.json", tmp_path / "packed.npz")
    with pytest.raises(ValueError, match="not a geometry case"):
        caseio.load_geometry_case(packed)


def test_new_entry_points_validate_before_any_cuda_call():
    from deep_fem_uav_wing.gnn import _cabi

    lib = _cabi.lib
    assert lib.dfw_vertex_normals_ws_bytes(-1, 5) == 0 and lib.dfw_case_stress_summary_ws_bytes(5, -1) == 0
    assert lib.dfw_vertex_normals_ws_bytes(1000, 500) >= 16 * 3000 + 4 * 501
    assert lib.dfw_case_stress_summary_ws_bytes(100_000, 16) > lib.dfw_case_stress_summary_ws_bytes(1000, 16) > 0
    fake = 256  # never dereferenced: every call below must fail its argument checks first
    rc = lib.dfw_vertex_normals(None, -1, None, 0, None, None, None, 0, None)
    assert rc != 0 and b"negative" in lib.dfw_last_error()
    rc = lib.dfw_vertex_normals(None, 10, fake, 4, fake, fake, fake, 1 << 30, None)
    assert rc != 0 and b"null input" in lib.dfw_last_error()
    rc = lib.dfw_vertex_normals(fake, 10, fake, 4, fake, None, fake, 1 << 30, None)
    assert rc != 0 and b"null output" in lib.dfw_last_error()
    rc = lib.dfw_vertex_normals(fake, 10, fake, 4, fake, fake, fake, 16, None)
    assert rc != 0 and b"workspace too small" in lib.dfw_last_error()
    rc = lib.dfw_case_stress_summary(fake, 0, fake, None, fake, -2, 10, 0.05, 0.0, 1, fake, fake, 1 << 30, None)
    assert rc != 0 and b"negative" in lib.dfw_last_error()
    rc = lib.dfw_case_stress_summary(fake, 5, fake, None, fake, 2, 10, 0.05, 0.0, 1, fake, fake, 1 << 30, None)
    assert rc != 0 and b"dtype" in lib.dfw_last_error()
    rc = lib.dfw_case_stress_summary(None, 0, fake, None, fake, 2, 10, 0.05, 0.0, 1, fake, fake, 1 << 30, None)
    assert rc != 0 and b"null pred" in lib.dfw_last_error()
    rc = lib.dfw_case_stress_summary(fake, 0, fake, None, None, 2, 10, 0.05, 0.0, 1, fake, fake, 1 << 30, None)
    assert rc != 0 and b"null case_ptr" in lib.dfw_last_error()
    rc = lib.dfw_case_stress_summary(fake, 0, fake, None, fake, 2, 10, 0.05, 0.0, 1, fake, fake, 8, None)
    assert rc != 0 and b"workspace too small" in lib.dfw_last_error()


def test_screener_refuses_multi_output_and_cpu_models():
    from deep_fem_uav_wing.gnn.model import GraphSAGEModel
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    with pytest.raises(ValueError, match="out_channels = 1"):
        DesignScreener(GraphSAGEModel(10, 16, 2, 1))
    with pytest.raises(RuntimeError, match="CUDA"):
        DesignScreener(GraphSAGEModel(10, 16, 1, 1))


def test_screen_cli_is_cuda_only(tmp_path):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=str(PKG))
    r = subprocess.run([sys.executable, str(PKG / "scripts" / "screen_gnn.py"), "--root", str(tmp_path), "--synthetic", "1"], env=env,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "CUDA-only: no CPU fallback exists" in r.stderr


# ---- GPU: kernels ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("order", ["native", "random"])
def test_vertex_normals_against_fp64_oracle(order):
    from deep_fem_uav_wing.gnn import ops, synth

    mesh = synth.surface_tri_wing(20000, seed=11, node_order=order)
    pos, faces = mesh["pos"], mesh["faces"].astype(np.int64)
    n_ref, scale = normals_oracle(pos, faces)
    pos_d, faces_d = torch.from_numpy(pos).cuda(), torch.from_numpy(faces).cuda()
    n1, st = ops.vertex_normals(pos_d, faces_d)
    n2, _ = ops.vertex_normals(pos_d, faces_d)
    assert torch.equal(n1.view(torch.int32), n2.view(torch.int32))  # bitwise run to run
    assert int(st.item()) == 0
    # bit for bit against the float32 oracle that repeats the kernel's products and its ascending incidence order
    n_f32, _ = normals_f32_oracle(pos, faces)
    assert n1.cpu().numpy().view(np.uint32).tobytes() == n_f32.view(np.uint32).tobytes()
    record("screen_vertex_normals", order=order, bit_mismatches=0)
    # features: columns 3-5 from the computed normals, everything else bit-identical to the given-normal features
    cp = torch.tensor([0, len(pos)], dtype=torch.int64, device="cuda")
    gp = torch.zeros(1, 4, device="cuda")
    x_c, _ = ops.node_features_batched(pos_d, n1, None, gp, cp, len(pos))
    x_g, _ = ops.node_features_batched(pos_d, torch.from_numpy(mesh["normal"]).cuda(), None, gp, cp, len(pos))
    x_c, x_g = x_c.cpu().numpy(), x_g.cpu().numpy()
    cols = [0, 1, 2, 6, 7, 8, 9]
    assert x_c[:, cols].tobytes() == x_g[:, cols].tobytes()
    nn_ref = np.linalg.norm(n_ref, axis=1)
    good = nn_ref >= 1e-3 * scale  # skins that nearly cancel (trailing edge) are ill-conditioned in direction
    unit = n_ref[good] / nn_ref[good, None]
    ferr = np.abs(x_c[good, 3:6] - unit).max()
    record("screen_normal_features", order=order, max_abs_err=float(ferr), excluded_vertices=int((~good).sum()))
    assert ferr <= 1e-5 and good.mean() > 0.99
    # bad faces are skipped and counted; the others give the same bits; a case's normals do not depend on its neighbours
    bad = np.array([[0, 1, len(pos)], [-1, 2, 3], [4, 5, 1 << 40]], dtype=np.int64)
    n3, st3 = ops.vertex_normals(pos_d, torch.from_numpy(np.concatenate([faces[:100], bad, faces[100:]])).cuda())
    assert int(st3.item()) == 3 and torch.equal(n3.view(torch.int32), n1.view(torch.int32))
    other = synth.surface_tri_wing(3000, seed=12)
    both_pos = torch.from_numpy(np.concatenate([other["pos"], pos])).cuda()
    both_faces = torch.from_numpy(np.concatenate([other["faces"].astype(np.int64), faces + len(other["pos"])])).cuda()
    n4, _ = ops.vertex_normals(both_pos, both_faces)
    assert torch.equal(n4[len(other["pos"]):].view(torch.int32), n1.view(torch.int32))


def _ragged_case(seed=5):
    """1, 7, 20k, 300k, 0 and 50 rows; case 5 has every y equal (nothing screened); ties, NaN and Inf injected."""
    rng = np.random.default_rng(seed)
    sizes = [1, 7, 20000, 300000, 0, 50]
    ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    N = int(ptr[-1])
    pos = rng.uniform(0.0, 1.5, size=(N, 3)).astype(np.float32)
    pos[ptr[5]:ptr[6], 1] = 0.0  # max_y - min_y = 0: no y exceeds the band
    pred = rng.uniform(10.0, 18.0, size=N).astype(np.float32)  # log1p(stress): ~2e4 .. 7e7 Pa
    for b, rows in ((2, [300, 7000, 19999]), (3, [1000, 150000, 299000])):  # ties at the top, across chunks
        r = ptr[b] + np.array(rows)
        pos[r, 1] = 1.4
        pred[r] = 18.5
    pred[ptr[3] + 5] = np.nan
    pred[ptr[3] + 200000] = np.inf
    pred[ptr[3] + 250000] = -np.inf
    pred[ptr[1] + 3] = np.nan
    return pos, pred, ptr


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_case_stress_summary_against_oracle(dtype):
    from deep_fem_uav_wing.gnn import ops

    pos, pred, ptr = _ragged_case()
    pos_d, cp = torch.from_numpy(pos).cuda(), torch.from_numpy(ptr).cuda()
    pred_d = torch.from_numpy(pred).cuda().to(dtype)
    pa = torch.expm1(pred_d.float()).cpu().numpy()  # the same fp32 expm1f values the kernel reduces
    allow = float(np.median(pa[np.isfinite(pa)]))
    got = ops.case_stress_summary(pred_d.reshape(-1, 1), pos_d, cp, allowable_pa=allow).cpu().numpy()
    ref = summary_oracle(pa, pos[:, 1], ptr, allowable=allow)
    exact = [0, 1, 2, 3, 5, 6, 7]
    assert np.array_equal(got[:, exact], ref[:, exact]), (got, ref)
    rel = np.abs(got[:, 4] - ref[:, 4]) / np.maximum(np.abs(ref[:, 4]), 1e-300)
    record("screen_summary_mean", dtype=str(dtype), max_rel=float(rel.max()))
    assert rel.max() <= 1e-12
    # lowest tied row wins; NaN and +Inf are counted (log1p -inf is -1 Pa: finite)
    assert got[3, 3] == 1000 and got[2, 3] == 300 and got[3, 7] == 2 and got[1, 7] == 1
    assert got[5, 1] == 0 and got[5, 3] == -1 and got[5, 2] == 0 and got[5, 4] == 0 and got[4, 0] == 0
    # an explicit mask equal to the band gives the same bits; an arbitrary mask follows the oracle
    band = np.zeros(len(pred), np.uint8)
    for b in range(len(ptr) - 1):
        y = pos[ptr[b]:ptr[b + 1], 1]
        if y.size:
            band[ptr[b]:ptr[b + 1]] = y.astype(np.float64) > 0.05 * (float(y.max()) - float(y.min()))
    got_m = ops.case_stress_summary(pred_d, pos_d, cp, mask=torch.from_numpy(band).cuda(), allowable_pa=allow).cpu().numpy()
    assert got_m.tobytes() == got.tobytes()
    rmask = (np.random.default_rng(1).random(len(pred)) < 0.3)
    got_r = ops.case_stress_summary(pred_d, pos_d, cp, mask=torch.from_numpy(rmask).cuda()).cpu().numpy()
    ref_r = summary_oracle(pa, pos[:, 1], ptr, mask=rmask)
    assert np.array_equal(got_r[:, exact], ref_r[:, exact])
    # every case alone gives the same record, bitwise
    for b in range(len(ptr) - 1):
        r0, r1 = int(ptr[b]), int(ptr[b + 1])
        alone = ops.case_stress_summary(pred_d[r0:r1], pos_d[r0:r1], torch.tensor([0, r1 - r0], device="cuda"), allowable_pa=allow)
        assert alone.cpu().numpy().tobytes() == got[b:b + 1].tobytes(), b


# ---- GPU: the screener -------------------------------------------------------------------------------------------------
def _geometry_cases(sizes, seed0=100):
    from deep_fem_uav_wing.gnn import synth

    return [synth.geometry_case(synth.surface_tri_wing(n, seed=seed0 + i)) for i, n in enumerate(sizes)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_screener_records_do_not_depend_on_the_launch(dtype):
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    sizes = [600, 4000, 1200, 9000, 800, 2500, 700, 5200, 3000, 640, 7000, 1500, 900, 2000, 6000, 1000]
    cases = _geometry_cases(sizes)
    model = _model(dtype=dtype)
    together = DesignScreener(model, max_nodes_per_launch=10**6, allowable_pa=5e6).screen(cases)
    alone = DesignScreener(model, max_nodes_per_launch=1, allowable_pa=5e6).screen(cases)
    assert [r["case_id"] for r in together] == [c["case_id"] for c in cases]
    assert all(r["status"] == "success" and r["normals"] == "computed" and r["skipped_faces"] == 0 for r in together)
    assert together == alone  # every float compared exactly


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_screener_matches_the_per_case_inference_path(tmp_path, dtype):
    from deep_fem_uav_wing.gnn import caseio, ops, synth
    from deep_fem_uav_wing.gnn.dataset import graph_from_raw_device
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    raws = []
    for i, n in enumerate((3000, 8000, 20000)):
        cid = synth.write_case_files(synth.surface_tri_wing(n, seed=40 + i, node_order="random" if i == 1 else "native"), tmp_path)
        d = tmp_path / "data" / "raw"
        raws.append(caseio.read_case(d / "fem" / cid / "surface_results.npz", d / "mesh" / cid / "boundary_sets.json",
                                     d / "geometry" / cid / "params.json"))
    model = _model(seed=3, dtype=dtype)
    res = DesignScreener(model).screen(raws)
    for raw, r in zip(raws, res):
        g = graph_from_raw_device(raw, device="cuda")
        with torch.no_grad():
            pred = model(g["x"], g["edge_index"])
        pa = torch.expm1(pred.float()).cpu().numpy().reshape(-1)
        pos = raw["pos"].astype(np.float32)
        ref = summary_oracle(pa, pos[:, 1], [0, len(pa)])[0]
        dev = ops.case_stress_summary(pred, g["pos"], torch.tensor([0, len(pa)], device="cuda")).cpu().numpy()[0]
        assert r["status"] == "success" and r["normals"] == "case"
        assert r["max_stress_pa"] == ref[2] and r["max_stress_node_id"] == int(raw["node_id"][int(ref[3])])
        assert r["max_stress_pos"] == [float(v) for v in raw["pos"][int(ref[3])]]
        assert r["mean_stress_pa"] == dev[4] and abs(r["mean_stress_pa"] - ref[4]) <= 1e-12 * ref[4]
        assert r["n_screened"] == int(raw["loss_mask"].sum())  # the band rule is the dataset's loss_mask


@pytest.mark.gpu
def test_computed_normals_rank_like_given_normals():
    from deep_fem_uav_wing.gnn import synth
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    meshes = [synth.surface_tri_wing(20000, seed=200 + i) for i in range(12)]
    computed = [synth.geometry_case(m) for m in meshes]
    given = [dict(c, normal=m["normal"]) for c, m in zip(computed, meshes)]
    for dtype in (torch.float32, torch.bfloat16):
        s = DesignScreener(_model(seed=1, dtype=dtype))
        a, b = s.screen(given), s.screen(computed)
        assert all(r["normals"] == "case" for r in a) and all(r["normals"] == "computed" for r in b)
        ma, mb = np.array([r["max_stress_pa"] for r in a]), np.array([r["max_stress_pa"] for r in b])
        record("screen_computed_vs_given_normals", dtype=str(dtype), max_rel_diff_max_stress=float((np.abs(ma - mb) / ma).max()))
        assert np.argsort(-ma, kind="stable").tolist() == np.argsort(-mb, kind="stable").tolist()


@pytest.mark.gpu
def test_screen_enqueues_without_implicit_synchronisation(monkeypatch):
    from deep_fem_uav_wing.gnn import ops
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    cases = _geometry_cases([1500 + 37 * i for i in range(40)], seed0=300)
    cases[7] = dict(cases[7], normal=np.ones((len(cases[7]["pos"]), 3), np.float32))  # one launch mixes given and computed normals
    model = _model()
    screener = DesignScreener(model, max_nodes_per_launch=12_000, result_ring=2)  # several launches; the ring wraps
    ref = screener.screen(cases)
    calls = []
    real = ops.graphsage_forward
    monkeypatch.setattr(ops, "graphsage_forward", lambda *a, **k: calls.append(1) or real(*a, **k))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = screener.screen(cases)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(calls) >= 6  # one dfw_graphsage_forward call per launch
    assert got == ref and got[7]["normals"] == "case" and got[8]["normals"] == "computed"


# ---- GPU: the CLI ------------------------------------------------------------------------------------------------------
def _checkpoint(root: Path):
    m = _model(seed=9)
    (root / "checkpoints").mkdir(parents=True, exist_ok=True)
    cfg = {"in_channels": 10, "hidden_channels": 128, "out_channels": 1, "num_layers": 4, "dropout": 0.1}
    torch.save({"model_config": cfg, "model_state_dict": {k: v.cpu() for k, v in m.state_dict().items()}}, root / "checkpoints" / "m.pt")
    return m


def _cli(root, *extra, prefix=()):
    env = dict(os.environ, PYTHONPATH=str(PKG))
    cmd = [*prefix, str(PKG / "scripts" / "screen_gnn.py"), "--root", str(root), "--checkpoint", "checkpoints/m.pt",
           "--synthetic", "20", "--seed", "500", "--synthetic-nodes", "3000", "--allowable-mpa", "30", "--top-k", "3", *extra]
    r = subprocess.run(cmd if prefix else [sys.executable, *cmd], env=env, capture_output=True, text=True, timeout=540)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r


@pytest.mark.gpu
def test_screen_cli_synthetic_matches_the_api(tmp_path):
    from deep_fem_uav_wing.gnn import synth
    from deep_fem_uav_wing.gnn.screening import DesignScreener

    model = _checkpoint(tmp_path)
    r = _cli(tmp_path, "--out", "one.jsonl")
    recs = [json.loads(line) for line in (tmp_path / "one.jsonl").read_text().splitlines()]
    assert len(recs) == 20 and "#1 " in r.stdout and "margin of safety" in r.stdout
    api = DesignScreener(model, allowable_pa=30e6).screen(synth.geometry_case(synth.surface_tri_wing(3000, seed=500 + i)) for i in range(20))
    assert [x["max_stress_pa"] for x in recs] == [x["max_stress_pa"] for x in api]
    assert [x["case_id"] for x in recs] == [x["case_id"] for x in api]


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_screen_cli_two_gpus_merges_the_same_records(tmp_path):
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, found {torch.cuda.device_count()}")
    _checkpoint(tmp_path)
    _cli(tmp_path, "--out", "one.jsonl")
    port = 29700 + (os.getpid() % 1500)
    _cli(tmp_path, "--out", "two.jsonl", prefix=(sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                                                 "--master-addr", "127.0.0.1", "--master-port", str(port)))
    assert (tmp_path / "two.jsonl").read_text() == (tmp_path / "one.jsonl").read_text()
