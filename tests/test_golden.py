"""Golden fixtures (tests/golden/, made by make_golden.py): the oracle must keep reproducing them, and the
graph derived from the reference's own LockBit traces must label exactly the files the reference lists as
encrypted (benchmarks/m{0,1}/results/file_list.txt, stored as m{0,1}_encrypted_files.txt)."""
import os

import numpy as np
import pytest
import torch

from oracle import sage_ref, lstm_ref, mcts_ref, rewards_ref

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "golden_hotpath.npz"))


def test_oracle_sage_reproduces_golden(gold):
    P = sage_ref.make_params(32, 128, 2, seed=1)
    t = lambda k: torch.from_numpy(gold[k])
    h, sc, el = sage_ref.forward(P, t("sage_x"), t("sage_rowptr"), t("sage_col"), t("sage_ew"), edge_logits=True)
    assert np.allclose(h.numpy(), gold["sage_h"], rtol=1e-5, atol=1e-6)
    assert np.allclose(sc.numpy(), gold["sage_score"], atol=1e-6) and np.allclose(el.numpy(), gold["sage_edge_logit"], rtol=1e-5, atol=1e-5)


def test_oracle_lstm_reproduces_golden(gold):
    LP = lstm_ref.make_params(16, 256, 2, seed=3)
    got = lstm_ref.forward(LP, torch.from_numpy(gold["lstm_seq"]), torch.from_numpy(gold["lstm_len"]))
    assert np.allclose(got.numpy(), gold["lstm_probs"], atol=1e-6)


def test_oracle_planner_reproduces_golden_bit_exact(gold):
    p, size, cost = gold["act_p"], gold["act_size"], gold["act_cost"]
    s = rewards_ref.score(gold["rw_states"], p, size, cost)
    assert np.array_equal(s.view(np.uint32), gold["rw_score"].view(np.uint32))
    r = mcts_ref.search(p, size, cost, R=64, D=10, T=12, seed=9)
    assert np.array_equal(r["root_n"], gold["mcts_root_n"])
    assert np.array_equal(r["root_w"].view(np.uint32), gold["mcts_root_w"].view(np.uint32))
    assert r["best"] == int(gold["mcts_best"]) and r["num_nodes"] == int(gold["mcts_num_nodes"])


def test_reference_trace_graph_labels_match_file_list():
    tr = np.load(os.path.join(GOLD, "golden_m1_graph.npz"))
    for name, n_enc in (("m0", 25), ("m1", 45)):            # benchmarks/m{0,1}/results/metadata.json: 25 / 45 files
        label = tr[f"{name}_label"]; listed = tr[f"{name}_is_listed_encrypted"]
        assert int(label.sum()) == n_enc and np.array_equal(label.astype(bool), listed)
        rp = tr[f"{name}_rowptr"]
        assert rp[0] == 0 and rp[-1] == tr[f"{name}_col"].shape[0] and (np.diff(rp) >= 0).all()
        assert int((tr[f"{name}_kind"] == 1).sum()) == 1     # one ransomware process node


def test_golden_graph_is_current_with_reference():
    """The graph constructor still derives the stored graphs from the reference's traces (stored next to them)."""
    from nerrf_b200 import graph as G
    tr = np.load(os.path.join(GOLD, "golden_m1_graph.npz"))
    for name in ("m0", "m1"):
        g = G.graph_from_jsonl(os.path.join(GOLD, f"{name}_trace.jsonl"))
        assert np.array_equal(g.rowptr, tr[f"{name}_rowptr"]) and np.array_equal(g.col, tr[f"{name}_col"])
        assert np.allclose(g.x, tr[f"{name}_x"])
        enc = set(open(os.path.join(GOLD, f"{name}_encrypted_files.txt")).read().split())
        assert np.array_equal(np.array([n in enc for n in g.meta["names"]]), tr[f"{name}_is_listed_encrypted"])
