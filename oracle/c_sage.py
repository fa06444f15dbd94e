"""ctypes wrapper of the C/OpenMP restatement of the GraphSAGE-T oracle (oracle/c/sage_oracle.c) -- TEST INFRASTRUCTURE.

Two uses, both on the checker side of the fence:
  * tests: a second, independent witness of oracle/sage_ref.py (PyTorch) -- tests/test_oracle_c_sage.py pins the
    two against each other, and the full-size cfg-2 parity test uses it because it finishes in seconds;
  * bench.py: the all-host-cores CPU arm (`--impl reference`, `cpu_baseline`) over the FULL graph.
Never imported by the product (nerrf_b200/).

Built by build() with gcc -O3 -march=native into oracle/_build/.  The file name carries a hash of this host's CPU
flags, so a library built on another host is not reused: lib() then compiles it (about a second) into a temporary
directory that is removed once the library is loaded, so a run never writes into the tree, which may be read-only."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "c", "sage_oracle.c")
OUT_DIR = os.path.join(_HERE, "_build")
_lib = None


def _cpu_tag():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return hashlib.sha1(line.encode()).hexdigest()[:10]
    except OSError:
        pass
    return "generic"


def lib_path(out_dir=OUT_DIR):
    return os.path.join(out_dir, f"libsage_oracle_{_cpu_tag()}.so")


def _stale(out):
    return not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(SRC)


def build(force=False, out_dir=OUT_DIR):
    os.makedirs(out_dir, exist_ok=True)
    out = lib_path(out_dir)
    if force or _stale(out):
        base = ["gcc", "-O3", "-fopenmp", "-fno-fast-math", "-shared", "-fPIC", SRC, "-lm"]
        tmp = out + f".{os.getpid()}.tmp"
        r = subprocess.run(base + ["-march=native", "-o", tmp], capture_output=True, text=True)
        if r.returncode != 0:                                   # an exotic host: portable build
            r = subprocess.run(base + ["-o", tmp], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("gcc failed on the C sage oracle:\n" + r.stdout + r.stderr)
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        if _stale(lib_path()):
            with tempfile.TemporaryDirectory(prefix="nerrf_sage_oracle_") as d:
                h = C.CDLL(build(out_dir=d))
        else:
            h = C.CDLL(lib_path())
        for n in ("nerrf_oracle_sage_layer", "nerrf_oracle_sage_aggregate", "nerrf_oracle_sage_node_head",
                  "nerrf_oracle_sage_forward", "nerrf_oracle_sage_threads"):
            getattr(h, n).restype = C.c_int
        _lib = h
    return _lib


def threads():
    return int(lib().nerrf_oracle_sage_threads())


def set_threads(n):
    lib().nerrf_oracle_sage_set_threads(C.c_int(int(n)))
    return threads()


def tune_threads(fwd: "Forward", candidates=(8, 16, 32, 64, 128)):
    """The host may expose more logical CPUs than it grants cycles (cgroup quota) or memory bandwidth: pick the thread
    count at which one full forward runs fastest.  Returns (threads, seconds)."""
    import time
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best = (None, float("inf"))
    for c in sorted({c for c in candidates if c <= ncpu} | {min(ncpu, 8)}):
        set_threads(c)
        fwd.run()
        t0 = time.perf_counter(); fwd.run(); dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (c, dt)
    set_threads(best[0])
    return best


def _np(a, dt):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a, dt)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _rp(rowptr):
    if hasattr(rowptr, "detach"):
        rowptr = rowptr.detach().cpu().numpy()
    rowptr = np.asarray(rowptr)
    if rowptr.dtype == np.int64:
        return np.ascontiguousarray(rowptr), 1
    return np.ascontiguousarray(rowptr, np.int32), 0


def aggregate(x, rowptr, col, ew, row_begin=0, row_end=None):
    x = _np(x, np.float32); col = _np(col, np.int32); ew = _np(ew, np.float32)
    rp, is64 = _rp(rowptr)
    N, F = x.shape
    row_end = N if row_end is None else row_end
    m = np.empty((row_end - row_begin, F), np.float32)
    rc = lib().nerrf_oracle_sage_aggregate(_p(x), C.c_int64(N), C.c_int(F), _p(rp), C.c_int(is64), _p(col), _p(ew),
                                           C.c_int64(row_begin), C.c_int64(row_end), _p(m))
    if rc:
        raise ValueError(f"nerrf_oracle_sage_aggregate rc={rc}")
    return m


def layer(x, rowptr, col, ew, W, b, relu=True, row_begin=0, row_end=None, out=None):
    x = _np(x, np.float32); col = _np(col, np.int32); ew = _np(ew, np.float32)
    W = _np(W, np.float32); b = _np(b, np.float32)
    rp, is64 = _rp(rowptr)
    N, F = x.shape
    H = W.shape[1]
    assert W.shape[0] == 2 * F and b.shape[0] == H
    row_end = N if row_end is None else row_end
    if out is None:
        out = np.empty((row_end - row_begin, H), np.float32)
    rc = lib().nerrf_oracle_sage_layer(_p(x), C.c_int64(N), C.c_int(F), _p(rp), C.c_int(is64), _p(col), _p(ew), _p(W), _p(b),
                                       C.c_int(H), C.c_int(int(relu)), C.c_int64(row_begin), C.c_int64(row_end), _p(out))
    if rc:
        raise ValueError(f"nerrf_oracle_sage_layer rc={rc}")
    return out


def node_head(h, node_w, node_b):
    h = _np(h, np.float32); node_w = _np(node_w, np.float32)
    score = np.empty(h.shape[0], np.float32)
    lib().nerrf_oracle_sage_node_head(_p(h), C.c_int64(h.shape[0]), C.c_int(h.shape[1]), _p(node_w),
                                      C.c_float(float(np.asarray(_np(node_b, np.float32)).reshape(-1)[0])), _p(score))
    return score


class Forward:
    """Prepared whole forward (arrays converted once, buffers allocated once) so that bench.py times only the C call."""

    def __init__(self, params, x, rowptr, col, ew):
        self.x = _np(x, np.float32); self.col = _np(col, np.int32); self.ew = _np(ew, np.float32)
        self.rp, self.is64 = _rp(rowptr)
        self.W = [_np(w, np.float32) for w, _ in params["layers"]]
        self.b = [_np(b, np.float32) for _, b in params["layers"]]
        self.node_w = _np(params["node_w"], np.float32)
        self.node_b = float(np.asarray(_np(params["node_b"], np.float32)).reshape(-1)[0])
        self.N, self.F = self.x.shape
        self.H = self.W[0].shape[1]
        self.L = len(self.W)
        self.h = np.empty((self.N, self.H), np.float32)
        self.tmp = np.empty((self.N, self.H), np.float32) if self.L > 1 else None
        self.score = np.empty(self.N, np.float32)
        self._Wp = (C.c_void_p * self.L)(*[w.ctypes.data for w in self.W])
        self._bp = (C.c_void_p * self.L)(*[b.ctypes.data for b in self.b])

    def run(self):
        rc = lib().nerrf_oracle_sage_forward(_p(self.x), C.c_int64(self.N), C.c_int(self.F), _p(self.rp), C.c_int(self.is64),
                                             _p(self.col), _p(self.ew), C.c_int(self.L), self._Wp, self._bp, C.c_int(self.H),
                                             _p(self.node_w), C.c_float(self.node_b), _p(self.h),
                                             _p(self.tmp) if self.tmp is not None else None, _p(self.score))
        if rc:
            raise ValueError(f"nerrf_oracle_sage_forward rc={rc}")
        return self.h, self.score


def forward(params, x, rowptr, col, ew):
    """Same contract as oracle.sage_ref.forward (without edge logits): returns (h [N,H], node_score [N]) as numpy."""
    return Forward(params, x, rowptr, col, ew).run()
