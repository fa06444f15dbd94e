"""ctypes wrapper of the C restatement of the planner oracle (oracle/c/planner_oracle.c) -- TEST INFRASTRUCTURE.

Built by build() with gcc into oracle/_build/ (git-ignored); when that library is missing or stale, lib() compiles it
into a temporary directory that is removed once the library is loaded, so a run never writes into the tree.  Used by
tests/test_oracle_c.py to pin the numpy oracle bit for bit against a second, independent implementation, and by
bench.py as the all-host-cores CPU baseline of the MCTS half of the metric.  Never imported by the product
(nerrf_b200/)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from . import rewards_ref as RW
from .mcts_ref import ln_table, best_child

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "c", "planner_oracle.c")
OUT_DIR = os.path.join(_HERE, "_build")
LIB = os.path.join(OUT_DIR, "libplanner_oracle.so")
_lib = None


def _stale(out):
    return not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(SRC)


def build(force=False, out_dir=OUT_DIR):
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, os.path.basename(LIB))
    if force or _stale(out):
        cmd = ["gcc", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", SRC, "-o", out, "-lm"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("gcc failed on the C oracle:\n" + r.stdout + r.stderr)
    return out


def lib():
    global _lib
    if _lib is None:
        if _stale(LIB):
            with tempfile.TemporaryDirectory(prefix="nerrf_planner_oracle_") as d:
                h = C.CDLL(build(out_dir=d))
        else:
            h = C.CDLL(LIB)
        h.nerrf_oracle_mcts.restype = C.c_int
        _lib = h
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def philox(c0, c1, c2, c3, k0, k1):
    out = np.zeros(4, np.uint32)
    lib().nerrf_oracle_philox(C.c_uint32(c0), C.c_uint32(c1), C.c_uint32(c2), C.c_uint32(c3), C.c_uint32(k0), C.c_uint32(k1), _p(out))
    return tuple(int(v) for v in out)


def _guard(guard):
    return None if guard is None else np.ascontiguousarray(guard, np.int32)


def score(states, p, size, cost, guard=None):
    p = np.ascontiguousarray(p, np.float32); size = np.ascontiguousarray(size, np.float32); cost = np.ascontiguousarray(cost, np.float32)
    A = p.shape[0]
    nw = RW.layout(A)[3]
    st = np.ascontiguousarray(states, np.uint32).reshape(-1, nw)
    out = np.zeros(st.shape[0], np.float32)
    g = _guard(guard)
    lib().nerrf_oracle_score(_p(st), C.c_int64(st.shape[0]), _p(p), _p(size), _p(cost), _p(g) if g is not None else None,
                             C.c_int(A), _p(out))
    return out


def search(p, size, cost, R=4096, D=50, T=64, seed=0, c=np.sqrt(2.0), root_state=None, threads=None, guard=None):
    p = np.ascontiguousarray(p, np.float32); size = np.ascontiguousarray(size, np.float32); cost = np.ascontiguousarray(cost, np.float32)
    A = p.shape[0]
    _, _, A_pad, nw = RW.layout(A)
    root = RW.empty_state(A) if root_state is None else (np.asarray(root_state, np.uint32) | RW.empty_state(A))
    root = np.ascontiguousarray(root, np.uint32)
    lo, inv = RW.reward_bounds(p, size, cost, root, guard)
    g = _guard(guard)
    lnN = ln_table(T, R)
    root_n = np.zeros(A_pad, np.int32); root_w = np.zeros(A_pad, np.float32); nn = np.zeros(1, np.int32)
    if threads:
        os.environ["OMP_NUM_THREADS"] = str(threads)
    lib().nerrf_oracle_mcts(_p(p), _p(size), _p(cost), _p(g) if g is not None else None, C.c_int(A), _p(root), C.c_int(R), C.c_int(D), C.c_int(T), C.c_uint64(seed),
                            C.c_float(np.float32(c)), C.c_float(lo), C.c_float(inv), _p(lnN), _p(root_n), _p(root_w), _p(nn))
    return {"root_n": root_n[:A].copy(), "root_w": root_w[:A].copy(), "best": best_child(root_n[:A], root_w[:A]),
            "num_nodes": int(nn[0]), "lo": lo, "inv_range": inv}
