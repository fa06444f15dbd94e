"""Generate the committed golden fixtures (run in the authoring container, CPU only):

    python tests/golden/make_golden.py

* golden_hotpath.npz   seeded inputs + ORACLE outputs for GraphSAGE-T / LSTM / rewards / MCTS.
                       The reference ships no golden vectors for this path (SURVEY.md 8c): these
                       pin the oracle against drift and give the GPU tests a fixed target.
* golden_m1_graph.npz  the temporal graph DERIVED from the reference's own LockBit traces
                       (benchmarks/m{0,1}/results/m{0,1}_trace.jsonl, stored here as m{0,1}_trace.jsonl)
                       by nerrf_b200.graph (arrays only: CSR, features, labels); the encrypted files
                       the reference lists (benchmarks/m{0,1}/results/file_list.txt) are stored here as
                       m{0,1}_encrypted_files.txt.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from nerrf_b200 import graph as G                      # noqa: E402
from oracle import sage_ref, lstm_ref, mcts_ref, rewards_ref    # noqa: E402


def main():
    out = {}
    g = G.synthetic_graph(N=300, E=2500, seed=42)
    P = sage_ref.make_params(32, 128, 2, seed=1)
    t = lambda a: torch.from_numpy(a)
    h, sc, el = sage_ref.forward(P, t(g.x), t(g.rowptr), t(g.col), t(g.ew), edge_logits=True)
    out.update(sage_x=g.x, sage_rowptr=g.rowptr, sage_col=g.col, sage_ew=g.ew, sage_h=h.numpy(), sage_score=sc.numpy(),
               sage_edge_logit=el.numpy())
    LP = lstm_ref.make_params(16, 256, 2, seed=3)
    gen = torch.Generator().manual_seed(5)
    seq = torch.randn(5, 9, 16, generator=gen); lengths = torch.tensor([9, 1, 4, 9, 6])
    out.update(lstm_seq=seq.numpy(), lstm_len=lengths.numpy(), lstm_probs=lstm_ref.forward(LP, seq, lengths).numpy())
    rng = np.random.default_rng(2)
    A = 40
    p = rng.beta(0.5, 0.5, A).astype(np.float32); size = rng.lognormal(np.log(2.0), 1.0, A).astype(np.float32)
    cost = rng.choice([1.0, 10.0, 100.0], A, p=[.9, .09, .01]).astype(np.float32)
    applied = rng.random((33, A)) < 0.3
    st = rewards_ref.pack_bits(np.concatenate([applied, np.ones((33, 1024 - A), bool)], 1))
    r = mcts_ref.search(p, size, cost, R=64, D=10, T=12, seed=9)
    out.update(act_p=p, act_size=size, act_cost=cost, rw_states=st, rw_score=rewards_ref.score(st, p, size, cost),
               mcts_root_n=r["root_n"], mcts_root_w=r["root_w"], mcts_best=np.int32(r["best"]),
               mcts_num_nodes=np.int32(r["num_nodes"]))
    np.savez_compressed(os.path.join(HERE, "golden_hotpath.npz"), **out)
    print("golden_hotpath.npz:", {k: v.shape for k, v in out.items()})

    tr = {}
    for name in ("m0", "m1"):
        trace = os.path.join(HERE, f"{name}_trace.jsonl")
        gg = G.graph_from_jsonl(trace)
        enc = set(open(os.path.join(HERE, f"{name}_encrypted_files.txt")).read().split())
        names = gg.meta["names"]
        # the same trace with OBSERVABLE features only (simulator annotations folded onto openat/write/rename):
        # what ai/train.py trains on and what a wire-format trace of the same activity would give
        go = G.graph_from_jsonl(trace, observable=True)
        assert np.array_equal(go.rowptr, gg.rowptr) and np.array_equal(go.col, gg.col)
        tr[f"{name}_x_obs"] = go.x
        tr.update({f"{name}_rowptr": gg.rowptr, f"{name}_col": gg.col, f"{name}_ew": gg.ew, f"{name}_x": gg.x,
                   f"{name}_label": gg.meta["label"], f"{name}_kind": gg.meta["node_kind"],
                   f"{name}_size_mb": gg.meta["size_mb"],
                   f"{name}_is_listed_encrypted": np.array([n in enc for n in names])})
        print(name, gg.num_nodes, "nodes", gg.num_edges, "edges", int(gg.meta["label"].sum()), "attacked,", len(enc), "listed encrypted")
    np.savez_compressed(os.path.join(HERE, "golden_m1_graph.npz"), **tr)


if __name__ == "__main__":
    main()
