"""Synthetic LockBit-style trace generator emitting the reference simulator's TRACE schema.

Schema (keys / event names / phases) follows benchmarks/m1/scripts/sim_lockbit_m1.py:24-36 and
the shipped fixtures benchmarks/m{0,1}/results/*_trace.jsonl: timestamp (ISO), event, path,
size, pid, phase, file_type; phases reconnaissance -> preparation (file_created) -> attack
(file_encrypt_start on x.dat, file_encrypt_complete on x.lockbit3) -> ransom note.
Used for tests and for the cfg-5 style end-to-end example; the real m0/m1 traces are stored under
tests/golden/ (m{0,1}_trace.jsonl).
"""
from __future__ import annotations

from datetime import datetime, timedelta

import numpy as np

_TYPES = ("document", "database", "spreadsheet", "media")
_STEMS = ("contract", "invoice", "report", "memo", "inventory", "audio", "archive", "product")


def lockbit_trace(n_files=45, seed=0, pid=454, benign_files=0, start="2025-08-30T14:07:06"):
    rng = np.random.default_rng(seed)
    t = datetime.fromisoformat(start)
    ev = []

    def emit(event, path, size=0, phase="attack", ftype="document", dt=0.2):
        nonlocal t
        t = t + timedelta(seconds=float(dt))
        ev.append({"timestamp": t.isoformat(), "event": event, "path": path, "size": int(size), "pid": pid,
                   "phase": phase, "file_type": ftype})

    emit("simulation_start", "/app/uploads", phase="initial")
    for name in ("process", "network", "user", "disk", "mount"):
        emit(f"{name}_enum", f"/tmp/{name}.txt", phase="reconnaissance", dt=0.5)
    files = []
    emit("seed_start", "/app/uploads", phase="preparation")
    for i in range(n_files + benign_files):
        ftype = _TYPES[int(rng.integers(len(_TYPES)))]
        stem = f"/app/uploads/{_STEMS[int(rng.integers(len(_STEMS)))]}_{i:03d}"
        size = int(rng.integers(2 << 20, 5 << 20))
        files.append((stem, size, ftype))
        emit("file_created", stem + ".dat", size, "preparation", ftype, dt=0.3)
    emit("seed_complete", "/app/uploads", sum(s for _, s, _ in files), phase="preparation")
    emit("encryption_start", "/app/uploads", dt=2.0)
    for stem, size, ftype in files[:n_files]:
        emit("file_encrypt_start", stem + ".dat", size, "attack", ftype, dt=0.01)
        emit("file_encrypt_complete", stem + ".lockbit3", size, "attack", ftype, dt=1.4)
    emit("ransom_note_created", "/app/uploads/README_LOCKBIT.txt", 512)
    emit("encryption_complete", "/app/uploads")
    emit("simulation_complete", "/app/uploads", phase="complete")
    return ev
