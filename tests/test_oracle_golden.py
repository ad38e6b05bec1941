"""The oracle is only trustworthy once pinned: replay the fixtures recorded from the reference's own
code (tests/golden/make_golden.py) and hand-derived known answers for the un-pinned SAGEConv."""
import numpy as np
import pytest
import torch

from helpers import golden_grads, golden_state_dict, load_golden, rel_l2, rel_max
from oracle import csr_aggregate_c, csr_oracle_c
from oracle.sage_oracle import (GraphSAGEModelRef, MaskedMSELossRef, SAGEConvRef, compute_metrics_ref, csr_oracle,
                                faces_to_edge_index_ref)

CASES = ["model_box_h16_l2", "model_tri600_h64_l3", "model_tet500_h128_l4"]
# The model fixtures were recorded with 8 CPU intra-op threads.  MKL's fp32 product of the decoder's last layer (64 -> 1)
# sums in an order that depends on the thread count, so the outputs are bit-equal at that thread count only.
RECORDED_THREADS = 8


@pytest.fixture
def recorded_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(RECORDED_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", CASES)
def test_oracle_model_matches_reference_fixture(name, recorded_threads):
    g = load_golden(name)
    model = GraphSAGEModelRef(10, int(g["hidden"]), 1, int(g["layers"]), dropout=0.0)
    model.load_state_dict(golden_state_dict(g), strict=True)
    model.train()
    x, ei = torch.from_numpy(g["x"]), torch.from_numpy(g["edge_index"])
    y, m = torch.from_numpy(g["y"]), torch.from_numpy(g["loss_mask"])
    out = model(x, ei, None)
    loss = MaskedMSELossRef()(out, y, m)
    loss.backward()
    assert torch.equal(out.detach(), torch.from_numpy(g["out"]))  # same arithmetic, same machine class: bit-equal
    assert abs(loss.item() - float(g["loss"])) <= 1e-6 * abs(float(g["loss"]))
    assert sorted(golden_grads(g)) == sorted(k for k, _ in model.named_parameters())  # every gradient is on file
    for k, gr in golden_grads(g).items():
        got = dict(model.named_parameters())[k].grad
        assert rel_l2(got, gr) < 1e-6, k
    met = compute_metrics_ref(out, y, m)
    flat = [met[a][b] for a in ("all_nodes", "masked_nodes") for b in ("mae", "rmse", "max_error", "count")]
    np.testing.assert_allclose(flat, g["metrics"], rtol=1e-6)
    model.eval()
    with torch.no_grad():
        assert rel_max(model(x, ei), g["out_eval"]) < 1e-6


def test_oracle_loss_and_metrics_fixture():
    g = load_golden("loss_metrics")
    pred = torch.from_numpy(g["pred"]).requires_grad_(True)
    targ, mask = torch.from_numpy(g["target"]), torch.from_numpy(g["mask"])
    for red in ("mean", "sum"):
        for mname, mm in (("mask", mask), ("none", None), ("allfalse", torch.zeros(50, dtype=torch.bool))):
            pred.grad = None
            l = MaskedMSELossRef(red)(pred, targ, mm)
            assert abs(l.item() - float(g[f"loss_{red}_{mname}"])) <= 1e-6 * max(1.0, abs(float(g[f"loss_{red}_{mname}"])))
            assert bool(l.requires_grad) == bool(g[f"loss_{red}_{mname}_requires_grad"])
            if mname != "allfalse":
                l.backward()
                np.testing.assert_allclose(pred.grad.numpy(), g[f"grad_{red}_{mname}"], rtol=1e-6, atol=1e-7)
    for mname, mm in (("mask", mask), ("none", None), ("allfalse", torch.zeros(50, dtype=torch.bool))):
        for ls in (True, False):
            met = compute_metrics_ref(pred, targ, mm, log_scale=ls)
            flat = [met[a][b] for a in ("all_nodes", "masked_nodes") for b in ("mae", "rmse", "max_error", "count")]
            np.testing.assert_allclose(flat, g[f"metrics_{mname}_{int(ls)}"], rtol=1e-6)


def test_faces_to_edge_index_restatement_matches_reference_fixture():
    from helpers import canon_edges

    g = load_golden("faces_to_edge_index")
    ids = {i + 10: i for i in range(8)}
    mine = faces_to_edge_index_ref(g["faces"].tolist(), ids)
    assert np.array_equal(canon_edges(mine), canon_edges(g["e_box"]))
    assert g["e_box"].shape == (2, 36)  # 18 undirected edges of the 12-triangle box (SURVEY 8c)
    mine_skip = faces_to_edge_index_ref(g["faces"].tolist() + [[10, 11, 999]], ids)
    assert np.array_equal(canon_edges(mine_skip), canon_edges(g["e_skip"]))
    assert faces_to_edge_index_ref([], ids).shape == (2, 0) and g["e_empty"].shape == (2, 0)


# ---- hand-derived known answers for SAGEConv (un-pinned upstream: PyG is absent) -------------------
def _conv(h_in, h_out):
    c = SAGEConvRef(h_in, h_out)
    with torch.no_grad():
        c.lin_l.weight.copy_(torch.eye(h_out, h_in))
        c.lin_l.bias.zero_()
        c.lin_r.weight.copy_(2.0 * torch.eye(h_out, h_in))
    return c


def test_known_answer_path_and_direction():
    # 0 -> 1 -> 2 (one-directional): node 0 has no incoming edge -> mean 0
    x = torch.tensor([[1.0, 10.0], [2.0, 20.0], [4.0, 40.0]])
    ei = torch.tensor([[0, 1], [1, 2]])
    out = _conv(2, 2)(x, ei)
    exp = torch.tensor([[0.0 + 2, 0.0 + 20], [1.0 + 4, 10.0 + 40], [2.0 + 8, 20.0 + 80]])
    assert torch.equal(out, exp)


def test_known_answer_star_isolated_duplicate_selfloop():
    # star: leaves 1..4 -> centre 0 ; node 5 isolated ; duplicate edge 1->0 ; self loop 2->2
    x = torch.arange(6, dtype=torch.float32).unsqueeze(1) + 1.0  # [[1],[2],[3],[4],[5],[6]]
    ei = torch.tensor([[1, 2, 3, 4, 1, 2], [0, 0, 0, 0, 0, 2]])
    out = _conv(1, 1)(x, ei)
    mean0 = (2 + 3 + 4 + 5 + 2) / 5.0  # duplicate counted with multiplicity
    exp = torch.tensor([[mean0 + 2 * 1], [0 + 2 * 2], [3 + 2 * 3], [0 + 2 * 4], [0 + 2 * 5], [0 + 2 * 6]])
    assert torch.allclose(out, exp, atol=1e-6)


def test_known_answer_disjoint_union_equals_separate_runs():
    torch.manual_seed(0)
    c = SAGEConvRef(4, 4)
    xa, xb = torch.randn(5, 4), torch.randn(3, 4)
    ea = torch.tensor([[0, 1, 2, 3, 4], [1, 2, 3, 4, 0]])
    eb = torch.tensor([[0, 1, 2], [2, 0, 1]])
    joint = c(torch.cat([xa, xb]), torch.cat([ea, eb + 5], dim=1))
    assert torch.allclose(joint, torch.cat([c(xa, ea), c(xb, eb)]), atol=1e-6)


def test_oracle_gradcheck_fp64():
    torch.manual_seed(1)
    m = GraphSAGEModelRef(10, 8, 1, 2, dropout=0.0).double()
    x = torch.randn(7, 10, dtype=torch.float64, requires_grad=True)
    ei = torch.tensor([[0, 1, 2, 3, 4, 5, 5, 2], [1, 2, 3, 4, 5, 0, 5, 0]])
    assert torch.autograd.gradcheck(lambda xx: m(xx, ei), (x,), eps=1e-6, atol=1e-5)


# ---- CSR oracle: numpy lexsort vs the plain-C restatement -------------------------------------------
@pytest.mark.parametrize("n,e,seed", [(1, 0, 0), (5, 0, 1), (50, 400, 2), (1000, 20000, 3), (3, 64, 4)])
@pytest.mark.parametrize("by", ["dst", "src"])
def test_csr_oracles_agree(n, e, seed, by):
    rng = np.random.default_rng(seed)
    ei = rng.integers(0, n, size=(2, e)).astype(np.int64)
    a = csr_oracle(ei, n, by)
    b = csr_oracle_c(ei, n, by)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


def test_csr_oracle_known_answer():
    ei = np.array([[2, 0, 1, 2, 2], [1, 1, 0, 1, 0]], dtype=np.int64)  # dup 2->1 at positions 0 and 3
    rowptr, col, perm, inv = csr_oracle(ei, 4)
    assert rowptr.tolist() == [0, 2, 5, 5, 5]
    assert col.tolist() == [1, 2, 0, 2, 2]
    assert perm.tolist() == [2, 4, 1, 0, 3]  # stable among equal (dst, src)
    np.testing.assert_allclose(inv, [0.5, 1 / 3, 1.0, 1.0])
    with pytest.raises(IndexError):
        csr_oracle_c(np.array([[0], [9]], dtype=np.int64), 4)


def test_c_aggregate_matches_torch_oracle():
    rng = np.random.default_rng(0)
    n, e, h = 300, 2500, 24
    ei = rng.integers(0, n, size=(2, e)).astype(np.int64)
    x = rng.standard_normal((n, h)).astype(np.float32)
    rowptr, col, _, inv = csr_oracle_c(ei, n)
    got = csr_aggregate_c(rowptr, col, inv, x)
    ref = SAGEConvRef.mean_aggregate(torch.from_numpy(x), torch.from_numpy(ei)).numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-6)
