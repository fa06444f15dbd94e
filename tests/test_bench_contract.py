"""bench.py driver contract, the parts that need no GPU: the reference arm (the CPU oracle port timed on the host
cores) prints ONE JSON line with the agreed keys, and the N=1 arm refuses to run without a CUDA device instead of
falling back to the CPU."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True,
                          timeout=600)


def test_reference_arm_prints_the_contract_line(tmp_path):
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "graphsage_t_edges_per_sec" and d["unit"] == "edges/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["config"]["nodes"] == 1_000_000 and d["config"]["edges"] == 10_000_000 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # --dump-outputs: every node score and a fixed sample of embedding rows, float32, well under 64 MB
    score, h = np.load(tmp_path / "score.npy"), np.load(tmp_path / "h_sample.npy")
    assert sorted(p.name for p in tmp_path.iterdir()) == ["h_sample.npy", "score.npy"]
    assert score.dtype == h.dtype == np.float32 and score.shape == (1_000_000,) and h.shape == (32768, 128)
    assert np.isfinite(score).all() and np.isfinite(h).all() and score.std() > 0 and h.std() > 0
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _run("--steps", "1", "--warmup", "0")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
