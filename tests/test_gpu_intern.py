"""Device-side node interning (csrc/intern_device.cu: hash table, rename-alias forest, creating-mention scan) against the
host routine nerrf_trace_intern (csrc/ingest.cu), which is the spec: identical node ids, kinds and naming events."""
import json
import os

import numpy as np
import pytest

from nerrf_b200 import ingest, stream, trace_sim

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _same(cols, order=None, merge=True):
    want = ingest.intern_nodes(cols, order, merge)
    got = ingest.intern_nodes_device(cols, order, merge)
    for name, a, b in zip(("node_p", "node_f", "node_g", "kind", "name_event", "name_which"), got, want):
        assert np.array_equal(a, b), f"{name} differs (merge_renames={merge})"
    return want


def _cols(events):
    return ingest.decode_event_batch(ingest.encode_event_batch(events))


@pytest.mark.parametrize("merge", [True, False])
def test_simulated_lockbit_traces(merge):
    for seed in (0, 3):
        cols = _cols(trace_sim.lockbit_trace(n_files=40, seed=seed, benign_files=60))
        order = np.argsort(cols.timestamp, kind="stable")
        _same(cols, order, merge)
        _same(cols, None, merge)


def _ev(t, pid, event, path, new_path=""):
    return {"timestamp": float(t), "pid": pid, "event": event, "path": path, "new_path": new_path, "size": 10}


@pytest.mark.parametrize("merge", [True, False])
def test_renames_aliases_and_chains(merge):
    """Real renames (a.dat -> a.dat.lockbit3), rename CHAINS (b -> c -> d), a rename target whose key is already a node
    (no merge then), two files sharing a stem, events on the new name after the rename, several pids."""
    ev = [
        _ev(0, 7, "openat", "/d/a.dat"), _ev(1, 7, "write", "/d/a.dat"),
        _ev(2, 7, "rename", "/d/a.dat", "/d/a.dat.lockbit3"),            # target key "/d/a.dat" is new: aliased
        _ev(3, 7, "write", "/d/a.dat.lockbit3"),                         # lands on the same node, names the rollback
        _ev(4, 8, "openat", "/d/b.txt"), _ev(5, 8, "rename", "/d/b.txt", "/d/c.txt.bak"),
        _ev(6, 8, "rename", "/d/c.txt.bak", "/d/e.x.y"),                 # chain: key "/d/c.txt" -> key "/d/e.x"
        _ev(7, 9, "openat", "/d/e.x.z"),                                 # stem "/d/e.x": reaches the chain's root
        _ev(8, 9, "openat", "/d/q.dat"), _ev(9, 9, "openat", "/d/r.dat"),
        _ev(10, 9, "rename", "/d/q.dat", "/d/r.lockbit3"),               # target key "/d/r" already a node: no merge
        _ev(11, 9, "write", "/d/r.lockbit3"),
        _ev(12, 7, "openat", "/d/noext"), _ev(13, 7, "rename", "/d/noext", "/d/noext"),
        _ev(14, 8, "openat", "/d/dir.v2/file"), _ev(15, 8, "openat", "/d/dir.v2/file.tmp"),
    ]
    cols = _cols(ev)
    node_p, node_f, node_g, kind, ne, nw = _same(cols, None, merge)
    if merge:
        assert node_f[0] == node_f[2] == node_f[3] and node_f[4] == node_f[5] == node_f[6] == node_f[7]
        assert node_f[8] != node_f[9] and node_f[10] == node_f[8] and node_f[11] == node_f[9]
    rng = np.random.default_rng(0)
    _same(cols, rng.permutation(cols.n), merge)                           # any processing order: same as the host in that order


def test_random_paths_fuzz():
    """Random short paths over a tiny alphabet (many shared stems, many rename targets that already exist)."""
    rng = np.random.default_rng(5)
    names = ["/r/" + "".join(rng.choice(list("ab."), size=int(rng.integers(1, 6)))) for _ in range(60)]
    for trial in range(20):
        ev = []
        for t in range(int(rng.integers(1, 300))):
            g = str(rng.choice(names)) if rng.random() < 0.3 else ""
            ev.append(_ev(t, int(rng.integers(1, 6)), "rename" if g else "write", str(rng.choice(names)), g))
        cols = _cols(ev)
        for merge in (True, False):
            _same(cols, None, merge)
            _same(cols, rng.permutation(cols.n), merge)


def test_reference_traces():
    """The reference's own LockBit traces (benchmarks/m{0,1}/results/m{0,1}_trace.jsonl, stored under tests/golden/)."""
    for m in ("m0", "m1"):
        ev = [json.loads(l) for l in open(os.path.join(GOLD, f"{m}_trace.jsonl"))]
        _same(_cols(ev), None, True)


def test_fleet_scale_and_tracker_style():
    """A 100k-event fleet trace (many pids, placeholder-patched paths) and the tracker-style form of a trace (write events
    carry no path: resolve_columns gives them the pid's open file first)."""
    cols, _ = stream.fleet_columns(1000, 10, seed=1)
    order = np.argsort(cols.timestamp, kind="stable")
    want = _same(cols, order, True)
    assert want[3].shape[0] > 90_000
    ev = trace_sim.lockbit_trace(n_files=20, seed=2, benign_files=10)
    for e in ev:
        if e["event"] in ("write", "file_encrypt_start"):
            e["path"] = ""
    cols = ingest.resolve_columns(_cols(ev))
    _same(cols, np.argsort(cols.timestamp, kind="stable"), True)


def test_empty_and_single():
    cols = _cols([_ev(0, 1, "openat", "/x")])
    _same(cols, None, True)
    got = ingest.intern_nodes_device(_cols([]), None, True)
    assert got[0].shape[0] == 0 and got[3].shape[0] == 0
