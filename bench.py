#!/usr/bin/env python
"""bench.py -- headline benchmark of the NERRF AI hot path on B200 (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): GraphSAGE-T edges/sec (+ MCTS rollouts/sec, reported under "mcts") on the
1M-node / 10M-edge synthetic temporal graph, 3-layer inference (configs[1]).  One "step" = one
full GraphSAGE_T.forward (3 fused gather+aggregate+GEMM layers + node head) over the graph.

  value      graph resident in HBM, CUDA-event timed, whole job (all ranks), max over ranks
  e2e        the same forward from HOST buffers: N=1 through nerrf_sage_session_forward_host (pinned host graph -> H2D
             -> forward -> D2H node scores, every step); N>1 every rank uploads only ITS rows / edge block and the
             ranks complete each other's features over NVLink (nerrf_b200.dist.ShardedSage.sharded_upload)
  roofline   dominant kernel = the F=128 fused layer (layers 2 and 3): algorithmic bytes
             E*(8+4F) + N*(4+4F+4H) per launch / its CUDA-event duration inside the timed region,
             against MEASURED_PEAKS.json hbm_gbs; "variants" holds the same for hub-destination and uniform graphs
  parity     every number in this line is the timing of a CHECKED computation: the forward is compared with the
             oracle over the full graph (C/OpenMP restatement, oracle/c/sage_oracle.c) and -- N>1 -- the sharded forward
             with the single-GPU forward bit for bit on every rank (own rows + every remotely produced row it reads);
             a failed check makes the process exit non-zero
  cpu_baseline / --impl reference   the oracle's C/OpenMP restatement over the FULL graph on the box's host cores
             (kind "port": the reference ships no implementation of this path, SURVEY.md 0)
N > 1: weak scaling -- the graph grows to N x (1M nodes, 10M edges), 1-D edge-block sharded with row-aligned cuts, one
embedding exchange per layer fused into the layer kernel (nerrf_b200/dist.py).  Extra objects of the N>1 line:
"trace_graph" (trace-structured graph, component-aware cuts), "cfg4" (BASELINE configs[3]: 10M / 100M strong-scaled
over the N GPUs), "cfg5" (configs[4]: the streamed LockBit fleet trace end to end), "nvlink" (achieved GB/s).

--dump-outputs DIR (single process): after the timed steps, what the forward returned in the LAST timed step, as float32
.npy files: DIR/score.npy (the node score of every node, [N]) and DIR/h_sample.npy (the final embeddings of a fixed
seeded sample of DUMP_ROWS nodes, [DUMP_ROWS, 128]; the full [N, 128] array is 512 MB).  The graph and the weights are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # a run writes nothing into the tree, which may be read-only

N_NODES, N_EDGES, F_IN, HIDDEN, LAYERS = 1_000_000, 10_000_000, 32, 128, 3
MCTS_CFG = dict(A=1024, R=4096, D=50, T=64)
GRAPH_SEED = 20250115
DUMP_ROWS, DUMP_SEED = 32768, 0


def algorithmic_bytes_layer(E, N, F, H=HIDDEN, s_rp=4):
    """SURVEY.md 8d: col + w + gathered source row per edge; rowptr + self row + output row per node."""
    return E * (8 + 4 * F) + N * (s_rp + 4 * F + 4 * H)


def algorithmic_bytes_forward(E, N):
    b, F = 0, F_IN
    for _ in range(LAYERS):
        b += algorithmic_bytes_layer(E, N, F)
        F = HIDDEN
    return b + 4 * N


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons via NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.002)
        except Exception as e:       # NVML missing: report it rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def workload_config(n_gpus):
    gen = ("numpy PCG64 seed %d" % GRAPH_SEED) if n_gpus == 1 else ("torch CUDA generator seed %d, random vertex relabeling" % GRAPH_SEED)
    return {"workload": f"GraphSAGE-T {LAYERS}-layer inference, {n_gpus}x(1M-node / 10M-edge) synthetic temporal graph "
                        f"({gen}, src=floor(N*u^3), dst~U), F_in={F_IN}, H={HIDDEN}",
            "nodes": N_NODES * n_gpus, "edges": N_EDGES * n_gpus, "layers": LAYERS,
            "parallelism": "single GPU" if n_gpus == 1 else f"1-D edge-block shards x{n_gpus}, one embedding exchange per layer",
            "l2": "inputs exceed L2 (graph 0.2 GB + activations 0.5 GB/layer per GPU vs 126 MB); no flush"}


def dump_rows(n):
    """The rows of h written by --dump-outputs: a fixed seeded sample, sorted."""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(n, DUMP_ROWS), replace=False))


def write_outputs(out_dir, h_sample, score):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("h_sample", h_sample), ("score", score)):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


# ------------------------------------------------------------------------------------------ oracle side (checker / CPU arm)
def oracle_check(model, rowptr, col, ew, x, h_gpu, score_gpu, k=64):
    """The C/OpenMP oracle (oracle/c/sage_oracle.c) over the FULL graph on the host cores vs a GPU forward: every element
    of h, every score, the top-k anomalous-node ranking.  The oracle is the checker here, never the product path."""
    from oracle import c_sage
    # torchrun exports OMP_NUM_THREADS=1: give the checker the cores the box grants (cgroup quota: 16 of the 128 logical CPUs)
    c_sage.set_threads(min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))
    t0 = time.perf_counter()
    hw, sw = c_sage.forward(model.oracle_params(), x.cpu().numpy(), rowptr.cpu().numpy(), col.cpu().numpy(), ew.cpu().numpy())
    dt = time.perf_counter() - t0
    hg = h_gpu.cpu().numpy(); sg = score_gpu.cpu().numpy()
    rms = float(np.sqrt((hw.astype(np.float64) ** 2).mean()))
    err = np.abs(hg - hw)
    bad = int((err > 1e-4 * np.abs(hw) + 1e-5 * rms).sum())
    s_err = float(np.abs(sg - sw).max())
    top_g = np.argsort(-sg, kind="stable")[:k]; top_o = np.argsort(-sw, kind="stable")[:k]
    # rankings may differ only by swaps of nodes whose ORACLE scores are within 4 * s_err (near ties at fp32 resolution)
    rank_ok = bool(np.abs(sw[top_g].astype(np.float64) - sw[top_o].astype(np.float64)).max() <= 4 * s_err + 1e-12)
    out = {"max_abs_err_over_rms": float(err.max() / rms), "elements_out_of_tolerance": bad, "elements": int(hw.size),
           "tolerance": "|got-want| <= 1e-4*|want| + 1e-5*rms (north star: 1e-4 rel fp32)", "score_max_abs_err": s_err,
           f"top{k}_indices_identical": bool(np.array_equal(top_g, top_o)), f"top{k}_ranking_ok": rank_ok,
           "oracle": "oracle/c/sage_oracle.c (C/OpenMP), full graph", "oracle_seconds": dt}
    out["ok"] = bad == 0 and s_err < 1e-5 and rank_ok
    return out


def cpu_arm_forward(params, x, rowptr, col, ew, steps, warmup):
    """Times the C/OpenMP oracle forward over the full graph with the thread count at which it runs fastest.  Returns
    (mean seconds, threads, the Forward holding the outputs of the last timed step)."""
    from oracle import c_sage
    f = c_sage.Forward(params, x, rowptr, col, ew)
    threads, _ = c_sage.tune_threads(f)
    for _ in range(warmup):
        f.run()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter(); f.run(); ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)), threads, f


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference ships none (SURVEY.md 0), so
    this is the oracle's C/OpenMP restatement (kind "port") over the FULL graph of the product arm's config -- N x (1M, 10M)
    at --gpus N -- on the host cores.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import sage_ref as S
    n = args.gpus
    if n == 1:
        from nerrf_b200.graph import synthetic_graph
        g = synthetic_graph(N_NODES, N_EDGES, seed=GRAPH_SEED)
        x, rp, col, ew = g.x, g.rowptr, g.col, g.ew
    else:           # the product arm's N x graph comes from the torch CUDA generator: build the same one (data only)
        import torch
        from nerrf_b200.dist import gpu_synthetic_graph
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
        rp, col, ew, x = (t.cpu().numpy() for t in gpu_synthetic_graph(N_NODES * n, N_EDGES * n, GRAPH_SEED, dev, relabel=True))
        torch.cuda.empty_cache()
    params = S.make_params(F_IN, HIDDEN, LAYERS, seed=1)
    dt, threads, f = cpu_arm_forward(params, x, rp, col, ew, args.steps, max(args.warmup, 1))
    if args.dump_outputs:
        write_outputs(args.dump_outputs, f.h[dump_rows(f.N)], f.score)
    E = int(col.shape[0])
    eps = E / dt
    sample = f"the full {LAYERS}-layer forward over the whole graph ({E} edges, {rp.shape[0] - 1} nodes), {args.steps} steps"
    line = {"impl": "reference", "metric": "graphsage_t_edges_per_sec", "value": eps, "unit": "edges/s",
            "n_gpus": n, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n),
            "cpu_baseline": {"value": eps, "unit": "edges/s", "cores": threads, "kind": "port", "sample": sample,
                             "impl": "oracle/c/sage_oracle.c (C + OpenMP, -O3 -march=native), thread count auto-tuned"},
            "e2e": {"value": eps, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        line, ok = run_multi(args, world, rank, local_rank, dev)
        if rank == 0:
            print(json.dumps(line), flush=True)
        dist.barrier()
        dist.destroy_process_group()
    else:
        line, ok = run_single(args, dev, local_rank)
        print(json.dumps(line), flush=True)
    if not ok:
        sys.stderr.write("bench.py: a parity check FAILED (see the \"parity\" objects of the line above)\n")
        raise SystemExit(3)


def run_single(args, dev, local_rank):
    import torch
    from nerrf_b200.graph import synthetic_graph
    from nerrf_b200.ai.models import GraphSAGE_T
    from nerrf_b200.ai.models.graphsage_t import HostSession
    K, W = args.steps, max(args.warmup, 3)
    model = GraphSAGE_T(F_IN, HIDDEN, LAYERS, algo=args.algo).to(dev)
    g = synthetic_graph(N_NODES, N_EDGES, seed=GRAPH_SEED)
    pin = lambda a: torch.from_numpy(a).pin_memory()
    hx, hrp, hcol, hew = pin(g.x), pin(g.rowptr), pin(g.col), pin(g.ew)
    x, rp, col, ew = (t.to(dev) for t in (hx, hrp, hcol, hew))
    N, E = g.num_nodes, g.num_edges
    h_a = torch.empty(N, HIDDEN, device=dev); h_b = torch.empty(N, HIDDEN, device=dev)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(LAYERS + 1)] for _ in range(K)]
    score = torch.empty(N, device=dev)

    def step(i=None):
        inp, bufs = x, (h_a, h_b)
        if i is not None: ev[i][0].record()
        for l in range(LAYERS):
            out = bufs[l & 1]
            # the node head is fused into the last layer's epilogue
            model.layer_forward(l, inp, rp, col, ew, out=out, score_out=score if l == LAYERS - 1 else None, reuse_long_scan=l > 0)
            if i is not None: ev[i][l + 1].record()
            inp = out
        return inp, score

    for _ in range(W):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(physical_gpu_index(local_rank)); sampler.start()
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t_start.record()
    for i in range(K):
        h_last, score_last = step(i)
    t_end.record()
    torch.cuda.synchronize()
    clocks = sampler.result()
    if args.dump_outputs:
        rows = torch.from_numpy(dump_rows(N)).to(dev)
        write_outputs(args.dump_outputs, h_last.index_select(0, rows).cpu().numpy(), score_last.cpu().numpy())
        del rows
    total_ms = t_start.elapsed_time(t_end)
    layer_ms = np.array([[ev[i][l].elapsed_time(ev[i][l + 1]) for l in range(LAYERS)] for i in range(K)])
    ms_per_step = total_ms / K
    value = E / (ms_per_step * 1e-3)

    # roofline of the dominant kernel: the F=128 fused layer (middle layer: no fused head)
    peak, peak_src = measured_peaks()
    dom_ms = float(layer_ms[:, 1:LAYERS - 1].mean()) if LAYERS > 2 else float(layer_ms[:, 1:].mean())
    dom_bytes = algorithmic_bytes_layer(E, N, HIDDEN)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    traffic = traffic_l1 = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("sage_layer_F128_dram_bytes_per_launch")
        traffic_l1 = json.load(open(tp)).get("sage_layer_F32_dram_bytes_per_launch")
    l1_bytes = algorithmic_bytes_layer(E, N, F_IN)
    l1_ms = float(layer_ms[:, 0].mean())
    roofline = {"bound": "hbm", "kernel": "fused GraphSAGE-T layer F=128 (gather+aggregate+GEMM)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "ncu --set full capture of the same kernel and graph (profiles/traffic.json); not measured in this run",
                "layer_F32": {"kernel": "the same kernel at F=32 (layer 1, quad-mode gather)", "algorithmic_bytes_per_launch": l1_bytes,
                              "kernel_ms": l1_ms, "achieved": l1_bytes / (l1_ms * 1e-3) / 1e9, "frac": l1_bytes / (l1_ms * 1e-3) / 1e9 / peak,
                              "traffic": traffic_l1},
                "peak_source": peak_src, "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms,
                "per_layer_ms": [float(v) for v in layer_ms.mean(0)],
                "forward": {"algorithmic_bytes": algorithmic_bytes_forward(E, N),
                            "achieved": algorithmic_bytes_forward(E, N) / (ms_per_step * 1e-3) / 1e9,
                            "frac": algorithmic_bytes_forward(E, N) / (ms_per_step * 1e-3) / 1e9 / peak}}

    # parity of exactly what was timed: the full forward against the oracle over the full graph
    h_fin, sc_fin = step()
    parity = {"single_gpu_vs_oracle": oracle_check(model, rp, col, ew, x, h_fin, sc_fin)}
    ok = parity["single_gpu_vs_oracle"]["ok"]

    # e2e through the host-buffer C-ABI call
    sess = HostSession(model, N, E)
    score_host = torch.empty(N).pin_memory()
    for _ in range(2):
        sess.forward(hx, hrp, hcol, hew, score_host)
    t0 = time.perf_counter()
    for _ in range(K):
        sess.forward(hx, hrp, hcol, hew, score_host)
    e2e_s = (time.perf_counter() - t0) / K
    h2d = int(hx.numel() * 4 + hrp.numel() * 4 + hcol.numel() * 4 + hew.numel() * 4)
    # the same K steps as a stream of graphs: nerrf_sage_session_submit_host / _wait, two steps in flight (the upload of
    # step i+1 runs under the layers of step i; every step still copies ITS inputs H2D and ITS scores D2H)
    score_pipe = [torch.empty(N).pin_memory() for _ in range(2)]
    for _ in range(2):
        sess.wait(sess.submit(hx, hrp, hcol, hew, score_pipe[0]))
    for sp in score_pipe:
        sp.zero_()
    t0 = time.perf_counter()
    prev = None
    for i in range(K):
        tk = sess.submit(hx, hrp, hcol, hew, score_pipe[i % 2])
        if prev is not None:
            sess.wait(prev)
        prev = tk
    sess.wait(prev)
    pipe_s = (time.perf_counter() - t0) / K
    e2e = {"value": E / pipe_s, "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(N * 4),
           "ms_per_step": pipe_s * 1e3,
           "api": "nerrf_sage_session_submit_host + nerrf_sage_session_wait (HostSession.submit / wait): K steps streamed "
                  "through the session with two in flight; every step uploads its own inputs from pinned host memory and "
                  "reads its own scores back",
           "single_call": {"value": E / e2e_s, "ms_per_step": e2e_s * 1e3,
                           "api": "nerrf_sage_session_forward_host (HostSession.forward): one blocking call per step, no overlap "
                                  "between steps"},
           "pcie_floor_ms": h2d / 55e9 * 1e3}
    sess.close()
    parity["host_session_equals_device_path"] = bool(torch.equal(score_host, sc_fin.cpu()))
    parity["pipelined_session_equals_device_path"] = bool(all(torch.equal(sp, sc_fin.cpu()) for sp in score_pipe[:min(K, 2)]))
    ok = ok and parity["host_session_equals_device_path"] and parity["pipelined_session_equals_device_path"]

    variants = run_graph_variants(dev, model, peak)
    del h_a, h_b
    mcts_info = run_mcts_bench(dev, args)
    lstm_info = run_lstm_bench(dev)
    graph_info = run_graph_build_bench(dev, rp, col)
    cfg5 = run_cfg5(dev, None) if not args.no_cfg5 else None
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import sage_ref as S
        dt, th, _ = cpu_arm_forward(S.make_params(F_IN, HIDDEN, LAYERS, seed=1), g.x, g.rowptr, g.col, g.ew, 3, 1)
        cpu = {"value": E / dt, "unit": "edges/s", "cores": th, "kind": "port", "seconds": dt,
               "sample": f"oracle/c/sage_oracle.c (C + OpenMP), the full {LAYERS}-layer forward over the whole graph ({E} edges), mean of 3, "
                         f"thread count auto-tuned (host exposes {os.cpu_count()} logical CPUs)"}
    line = {"metric": "graphsage_t_edges_per_sec", "value": value, "unit": "edges/s", "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(1), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": K * LAYERS, "clocks": clocks, "parity": parity, "variants": variants, "mcts": mcts_info,
            "lstm": lstm_info, "graph_build": graph_info, "cfg5": cfg5, "algo": args.algo}
    if cfg5 is not None:
        ok = ok and cfg5.get("ok", True)
    return line, ok


def run_graph_variants(dev, model, peak, reps=5):
    """SURVEY.md 8d asks for the hub-DESTINATION variant next to the headline generator; the uniform-source graph has no
    hub rows for the L2 to hold (every gathered row is a DRAM read).  Same size as cfg 2, generated on the GPU."""
    import torch
    from nerrf_b200.dist import gpu_synthetic_graph
    out = {}
    for fam in ("hub_dst", "uniform"):
        rp, col, ew, x = gpu_synthetic_graph(N_NODES, N_EDGES, GRAPH_SEED, dev, family=fam)
        bufs = [torch.empty(N_NODES, HIDDEN, device=dev) for _ in range(2)]
        score = torch.empty(N_NODES, device=dev)

        def step(ev=None):
            inp = x
            for l in range(LAYERS):
                if ev: ev[l].record()
                model.layer_forward(l, inp, rp, col, ew, out=bufs[l & 1], score_out=score if l == LAYERS - 1 else None, reuse_long_scan=l > 0)
                inp = bufs[l & 1]
            if ev: ev[LAYERS].record()
        for _ in range(3): step()
        torch.cuda.synchronize()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(LAYERS + 1)] for _ in range(reps)]
        for i in range(reps): step(evs[i])
        torch.cuda.synchronize()
        ms = [float(np.mean([evs[i][l].elapsed_time(evs[i][l + 1]) for i in range(reps)])) for l in range(LAYERS)]
        fwd = sum(ms)
        out[fam] = {"per_layer_ms": ms, "forward_ms": fwd, "edges_per_s": N_EDGES / (fwd * 1e-3),
                    "max_in_degree": int((rp[1:] - rp[:-1]).max()),
                    "roofline_frac_F128_layer": algorithmic_bytes_layer(N_EDGES, N_NODES, HIDDEN) / (ms[1] * 1e-3) / 1e9 / peak,
                    "roofline_frac_forward": algorithmic_bytes_forward(N_EDGES, N_NODES) / (fwd * 1e-3) / 1e9 / peak}
        del rp, col, ew, x, bufs, score
    return out


def run_multi(args, world, rank, local_rank, dev):
    """N > 1: weak scaling on the relabelled random graph (headline), + trace-structured graph, cfg 4, cfg 5."""
    import torch
    import torch.distributed as dist
    from nerrf_b200 import dist as nd
    from nerrf_b200.ai.models import GraphSAGE_T
    K, W = args.steps, max(args.warmup, 3)
    model = GraphSAGE_T(F_IN, HIDDEN, LAYERS, algo=args.algo).to(dev)
    peak, peak_src = measured_peaks()
    mk_sampler = lambda: ClockSampler(physical_gpu_index(local_rank))
    ok = True

    # ---------------------------------------------------------------- headline: N x (1M, 10M), random relabelled
    N, E = N_NODES * world, N_EDGES * world
    rowptr, col, ew, x = nd.gpu_synthetic_graph(N, E, GRAPH_SEED, dev, relabel=True)
    ss = nd.ShardedSage(model, rowptr, col, ew, rank, world, dev, exchange=args.exchange)
    ss.set_x(x)
    tr = nd.timed_sharded_run(ss, K, W, mk_sampler)
    ms_per_step, clocks = tr["ms_per_step"], tr["clocks"]
    sh = ss.shard
    e_loc, r_loc = sh.edge_end - sh.edge_base, sh.row_end - sh.row_begin
    dom_bytes = algorithmic_bytes_layer(e_loc, r_loc, HIDDEN)
    dom_ms = tr["compute_ms"][1]
    eg, ing = ss.exchange_bytes_per_layer()
    layer_wall = [tr["compute_ms"][l] + tr["exchange_ms"][l] for l in range(LAYERS)]
    nvlink = {"egress_bytes_per_layer_rank0": eg, "mean_ingress_bytes_per_layer": ing,
              "achieved_egress_gbps_per_exchanged_layer": [eg / (layer_wall[l] * 1e-3) / 1e9 for l in range(LAYERS - 1)],
              "peak_per_direction_gbps": 900.0, "measured_peer_copy_gbps": 770.0,
              "bound_ms_per_exchanged_layer": max(eg, ing) / 900e9 * 1e3,
              "bound_ms_per_exchanged_layer_at_measured_peer_copy": max(eg, ing) / 770e9 * 1e3,
              "weak_scaling_ceiling": "random vertex relabeling makes every rank read the same hub-heavy ~55 % of all rows: a rank must "
                                      "RECEIVE that many 512-byte rows per exchanged layer whatever the transport (P2P, multicast), so "
                                      "step time >= 2 x ingress / link rate + the last layer; trace_graph is the same metric on the workload "
                                      "the metric names (a trace: components with no cut)",
              "note": "the exchange is fused into the layer kernel: its rows travel while the next tiles are gathered, so the "
                      "layer's wall time (compute + barrier segments) is what the bytes are divided by"}
    par, (h_ref, sc_ref) = ss.parity_vs_single_gpu(rowptr, col, ew, x)
    parity = {"sharded_vs_single_gpu": par}
    chk = oracle_check(model, rowptr, col, ew, x, h_ref, sc_ref) if rank == 0 else None
    parity["single_gpu_vs_oracle"] = chk
    flag = torch.tensor([int(par["own_rows_bit_exact"] and par["read_rows_bit_exact"] and (chk["ok"] if chk else True))], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = ok and bool(flag)
    del h_ref, sc_ref

    # ---- e2e: every rank's inputs come from pinned host memory every step; x is uploaded SHARDED and completed over NVLink
    hx_own = x[sh.row_begin:sh.row_end].cpu().pin_memory()
    hrp_own = sh.rowptr[sh.row_begin:sh.row_end + 1].cpu().pin_memory()
    hcol, hew = sh.col.cpu().pin_memory(), sh.ew.cpu().pin_memory()
    hscore = torch.empty(r_loc).pin_memory()
    x_keep = x

    def e2e_step():
        ss.sharded_upload(hx_own, hrp_own, hcol, hew)
        ss.step()
        hscore.copy_(ss.score[sh.row_begin:sh.row_end], non_blocking=True)
        torch.cuda.synchronize()
    e2e_step(); e2e_step(); dist.barrier()
    te = time.perf_counter()
    for _ in range(K):
        e2e_step()
    dist.barrier()
    e2e_s = torch.tensor([(time.perf_counter() - te) / K], device=dev)
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    # the sharded upload delivered exactly the resident features, on every row this rank reads (own rows + sources of its edges)
    reads = torch.zeros(N, dtype=torch.bool, device=dev); reads[sh.col.long()] = True; reads[sh.row_begin:sh.row_end] = True
    ridx = reads.nonzero().squeeze(1)
    e2e_same = bool(torch.equal(ss.x[ridx], x_keep[ridx]))
    del reads, ridx
    flag = torch.tensor([int(e2e_same)], device=dev); dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    parity["sharded_upload_delivers_every_row_read"] = bool(flag)
    ok = ok and bool(flag)
    h2d = int(hx_own.numel() * 4 + hrp_own.numel() * hrp_own.element_size() + hcol.numel() * 4 + hew.numel() * 4)
    e2e = {"value": E / float(e2e_s), "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(r_loc * 4),
           "ms_per_step": float(e2e_s) * 1e3,
           "api": "nerrf_b200.dist.ShardedSage.sharded_upload + step: per-rank pinned inputs (bytes are per rank); each rank uploads "
                  "its own rows of x and its edge block, peers receive the rows they reference over NVLink"}
    ss.set_x(x_keep)
    exchange_desc = ss.describe()
    headline_roofline = {"bound": "hbm", "kernel": "fused GraphSAGE-T layer F=128 (rank 0's edge block)",
                         "achieved": dom_bytes / (dom_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": dom_bytes / (dom_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "per_layer_compute_ms": tr["compute_ms"], "per_layer_exchange_ms": tr["exchange_ms"],
                         "per_rank_segments_ms": tr["per_rank_segments_ms"], "exchange_bytes_per_layer": int(N * HIDDEN * 4)}
    del ss, rowptr, col, ew, x, x_keep, hx_own, hcol, hew
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- trace-structured graph (component-aware cuts)
    trace_graph = run_trace_graph(model, world, rank, dev, K, W, peak)
    ok = ok and trace_graph["parity"]["own_rows_bit_exact"] and trace_graph["parity"]["read_rows_bit_exact"]
    # ---------------------------------------------------------------- cfg 4: 10M / 100M, strong-scaled over the N GPUs
    cfg4 = run_cfg4(model, args, world, rank, dev, K, W) if not args.no_cfg4 else None
    if cfg4 is not None:
        ok = ok and cfg4["ok"]
    # ---------------------------------------------------------------- MCTS root-parallel
    mcts_local = run_mcts_bench(dev, args, seed=rank)
    roll = torch.tensor([mcts_local["value"], mcts_local["e2e_value"]], device=dev)
    dist.all_reduce(roll, op=dist.ReduceOp.SUM)
    mcts_local.update({"value": float(roll[0]), "e2e_value": float(roll[1]),
                       "note": "root-parallel: sum over ranks of independent trees (seed = rank), no collective"})
    # ---------------------------------------------------------------- cfg 5: streamed fleet trace end to end on N GPUs
    cfg5 = run_cfg5(dev, (rank, world)) if not args.no_cfg5 else None
    if cfg5 is not None:
        ok = ok and cfg5.get("ok", True)
    flag = torch.tensor([int(ok)], device=dev); dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    ok = bool(flag)
    line = {"metric": "graphsage_t_edges_per_sec", "value": E / (ms_per_step * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (torch CUDA generator, same distribution as the N=1 graph, random vertex relabeling for shard balance)",
            "config": dict(workload_config(world), exchange=exchange_desc), "roofline": headline_roofline, "cpu_baseline": None,
            "e2e": e2e, "gpu_launches": K * LAYERS, "clocks": clocks, "parity": parity, "nvlink": nvlink,
            "trace_graph": trace_graph, "cfg4": cfg4, "cfg5": cfg5, "mcts": mcts_local, "algo": args.algo}
    return line, ok


def run_trace_graph(model, world, rank, dev, K, W, peak):
    """The workload the metric names is a 1M-node TRACE: a fleet of processes each touching its own files.  Weak scaling:
    world x 15625 components of 64 nodes (1M nodes, ~10M edges per GPU), node ids contiguous per component, cuts aligned to
    components -- the per-layer exchange has nothing to send and only the barriers remain."""
    import torch
    from nerrf_b200 import dist as nd
    n_comp = 15625 * world
    rowptr, col, ew, x, S = nd.gpu_trace_graph(n_comp, dev)
    N, E = rowptr.numel() - 1, col.numel()
    ss = nd.ShardedSage(model, rowptr, col, ew, rank, world, dev, exchange="p2p", align=S)
    ss.set_x(x)
    tr = nd.timed_sharded_run(ss, K, W)
    par, _ = ss.parity_vs_single_gpu(rowptr, col, ew, x)
    # the same graph on ONE GPU at 1/world of the size is the weak-scaling reference point: time it on every rank
    rp1, col1, ew1, x1, _ = nd.gpu_trace_graph(15625, dev)
    bufs = [torch.empty(rp1.numel() - 1, HIDDEN, device=dev) for _ in range(2)]
    sc1 = torch.empty(rp1.numel() - 1, device=dev)

    def one():
        inp = x1
        for l in range(LAYERS):
            model.layer_forward(l, inp, rp1, col1, ew1, out=bufs[l & 1], score_out=sc1 if l == LAYERS - 1 else None, reuse_long_scan=l > 0)
            inp = bufs[l & 1]
    for _ in range(3): one()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K): one()
    e1.record(); torch.cuda.synchronize()
    ms1 = e0.elapsed_time(e1) / K
    v1 = col1.numel() / (ms1 * 1e-3)
    vN = E / (tr["ms_per_step"] * 1e-3)
    return {"metric": "graphsage_t_edges_per_sec", "value": vN, "unit": "edges/s", "ms_per_step": tr["ms_per_step"], "nodes": int(N),
            "edges": int(E), "scaling": "weak", "single_gpu_same_per_gpu_size": {"value": v1, "ms_per_step": ms1, "edges": int(col1.numel())},
            "weak_scaling_efficiency": vN / (world * v1), "exchange": ss.describe(), "component_nodes": S,
            "per_layer_compute_ms": tr["compute_ms"], "per_layer_exchange_ms": tr["exchange_ms"], "parity": par,
            "workload": f"trace-structured graph: {n_comp} components x (1 process + {S - 1} files), 3..7 events per file, "
                        "process<->file edges, cuts aligned to components"}


def run_cfg4(model, args, world, rank, dev, K, W):
    """BASELINE configs[3]: 10M-node / 100M-edge graph 1-D edge-sharded over the N GPUs (strong form), one embedding exchange
    per layer.  Parity: sharded == single-GPU bit for bit on every rank; single-GPU vs the oracle over the full graph (rank 0)."""
    import torch
    import torch.distributed as dist
    from nerrf_b200 import dist as nd
    N, E = 10_000_000, 100_000_000
    rowptr, col, ew, x = nd.gpu_synthetic_graph(N, E, GRAPH_SEED + 4, dev, relabel=True)
    ss = nd.ShardedSage(model, rowptr, col, ew, rank, world, dev, exchange=args.exchange)
    ss.set_x(x)
    Kc = max(3, min(K, 5))
    tr = nd.timed_sharded_run(ss, Kc, 3)
    par, (h_ref, sc_ref) = ss.parity_vs_single_gpu(rowptr, col, ew, x)
    chk = oracle_check(model, rowptr, col, ew, x, h_ref, sc_ref) if rank == 0 else None
    flag = torch.tensor([int(par["own_rows_bit_exact"] and par["read_rows_bit_exact"] and (chk["ok"] if chk else True))], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    eg, ing = ss.exchange_bytes_per_layer()
    out = {"metric": "graphsage_t_edges_per_sec", "value": E / (tr["ms_per_step"] * 1e-3), "unit": "edges/s", "n_gpus": world,
           "ms_per_step": tr["ms_per_step"], "steps": Kc, "nodes": N, "edges": E, "scaling": "strong", "exchange": ss.describe(),
           "per_layer_compute_ms": tr["compute_ms"], "per_layer_exchange_ms": tr["exchange_ms"],
           "egress_bytes_per_layer_rank0": eg, "parity": {"sharded_vs_single_gpu": par, "single_gpu_vs_oracle": chk}, "ok": bool(flag),
           "workload": "BASELINE configs[3]: 10M-node / 100M-edge synthetic temporal graph (same generator family as cfg 2), "
                       f"1-D edge-block shards x{world}"}
    del ss, rowptr, col, ew, x, h_ref, sc_ref
    torch.cuda.empty_cache()
    return out


def run_cfg5(dev, dist_rw, n_procs=10400, n_attacked=40):
    """BASELINE configs[4]: end-to-end LockBit trace -- streamed events -> sliding-window temporal graph (GPU constructor)
    -> GraphSAGE_T anomaly scores -> top-A files -> lstm -> MCTS plan, tick by tick (nerrf_b200.stream).  Fleet trace in the
    m1 simulator's schema (SURVEY.md 8d cfg 5: m1 replicated to >= 1M nodes): n_procs processes, n_attacked of them
    ransomware.  Plan correctness = the union of the ticks' plans renames back exactly the encrypted files."""
    import torch
    from nerrf_b200 import stream, pipeline
    from nerrf_b200.ai import train as T
    from nerrf_b200.ai.models import GraphSAGE_T
    from nerrf_b200.ai.models.lstm import LSTMScorer
    multi = bool(dist_rw and dist_rw[1] > 1)
    lead = not multi or dist_rw[0] == 0
    t0 = time.perf_counter()
    torch.manual_seed(0)
    model, scorer = GraphSAGE_T(F_IN, HIDDEN, 2), LSTMScorer()
    if lead:                                                       # ai/train.py on the GPU (not timed): GraphSAGE-T forward + backward through
        T.train(model, scorer, T.toy_set(range(100, 104)), epochs=25, lr=3e-3, device=dev)   # the library's kernels; N>1: rank 0 trains,
    model.to(dev); scorer.to(dev)                                  # the weights are broadcast
    if multi:
        import torch.distributed as dist
        for p_ in list(model.parameters()) + list(scorer.parameters()):
            dist.broadcast(p_.data, 0)
    t_train = time.perf_counter() - t0
    t0 = time.perf_counter()
    cols, encrypted, bad_pids = stream.fleet_columns(n_procs, n_attacked, seed=5, return_pids=True) if lead else (None, set(), set())
    t_gen = time.perf_counter() - t0
    ctx = pipeline.DistContext(dist_rw[0], dist_rw[1]) if multi else None
    sp = stream.StreamingPlanner(model, scorer, window_s=60.0, tick_s=30.0, top_a=4096, n_rollouts=1024, depth=32, iterations=8,
                                 commit_per_search=64, kill_candidates=True, device=str(dev), dist_ctx=ctx)
    t0 = time.perf_counter()
    ticks = sp.run(cols)
    torch.cuda.synchronize()
    t_run = time.perf_counter() - t0
    if not lead:                                                   # the plan (names) lives on rank 0
        return {"ok": True}
    planned = set(sp.reverted)
    tp = len(planned & encrypted)
    big = max(ticks, key=lambda t: t.nodes)
    stage = {}
    for t in ticks:
        for k, v in t.timings_ms.items():
            stage[k] = stage.get(k, 0.0) + float(v)
    out = {"workload": f"fleet trace: {n_procs} processes x 95 files (m1 simulator schema), {n_attacked} ransomware processes x 45 encrypted "
                       f"files; 60 s sliding window, one tick per 30 s of trace time" +
                       ("; host-side ingest on rank 0, device graph / sequences broadcast, GNN sharded, LSTM batch split, MCTS root-parallel" if multi else ""),
           "events": int(cols.n), "events_per_s_end_to_end": cols.n / t_run, "ticks": len(ticks), "seconds_total": t_run,
           "largest_window": {"events": big.events, "nodes": big.nodes, "edges": big.edges, "timings_ms": {k: float(v) for k, v in big.timings_ms.items()}},
           "stage_ms_sum_over_ticks": stage, "n_gpus": dist_rw[1] if dist_rw else 1,
           "plan": {"reversions": len(planned), "encrypted_files": len(encrypted), "true_positives": tp,
                    "precision": tp / max(len(planned), 1), "recall": tp / max(len(encrypted), 1),
                    "exact": planned == encrypted, "truncated_ticks": int(sum(t.truncated for t in ticks)),
                    "process_kills": len(sp.killed), "ransomware_processes": len(bad_pids),
                    "kills_correct": len(sp.killed & bad_pids), "kills_wrong": len(sp.killed - bad_pids),
                    "note": "planner spec v1: a reversion only sticks once the process that wrote the file is killed (cost 10), so the "
                            "plan interleaves process kills and file reversions; <= 32 kill candidates per tick"},
           "stream_upload_ms": float(getattr(sp, "ingest_ms", 0.0)),
           "constructor": "device-resident stream (nerrf_b200.stream.DeviceStream): columns uploaded once (stream_upload_ms, inside "
                          "seconds_total); per tick the window is a slice of the time-sorted index array and node interning (hash "
                          "table), per-node features, edge assembly and the CSR sort run on the GPU",
           "not_timed": {"train_s": t_train, "trace_generation_s": t_gen,
                         "train": "ai/train.py, 25 epochs on the GPU: GraphSAGE-T layers forward (tcgen05) and backward (csrc/sage_bwd.cu) through the C-ABI"},
           "ok": True}
    return out


def run_mcts_bench(dev, args, seed=0):
    """cfg 3: A=1024, R=4096 leaf-parallel rollouts, depth 50; T=64 iterations (headline) and SURVEY.md 8d's T=16."""
    import torch
    from nerrf_b200.ai.planner import mcts
    from nerrf_b200.ai.planner.rewards import Actions
    rng = np.random.default_rng(2)
    A, R, D, T = (MCTS_CFG[k] for k in "ARDT")
    act = Actions(rng.beta(0.5, 0.5, A), rng.lognormal(np.log(2.0), 1.0, A),
                  rng.choice([1.0, 10.0, 100.0], A, p=[.9, .09, .01]))
    out_T = {}
    for Tn in (16, T):
        ctx = mcts.SearchContext(act, R, D, Tn, device=dev)
        ctx.search(seed)                                                       # warm-up
        torch.cuda.synchronize()
        reps = 7
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for i in range(reps):
            evs[i][0].record(); lo_inv = ctx.launch(seed + i); evs[i][1].record()
        torch.cuda.synchronize()
        out_T[Tn] = (float(np.median([a.elapsed_time(b) for a, b in evs])), ctx, lo_inv)
    ms, ctx, lo_inv = out_T[T]
    r = ctx.fetch(*lo_inv)
    # through the public call incl. result read-back, and through the host-buffer C-ABI session
    reps = 5
    t0 = time.perf_counter()
    for i in range(reps):
        ctx.search(seed + i)
    api_s = (time.perf_counter() - t0) / reps
    sess = mcts.HostSession(A, T, R, device=dev)
    mcts.search(act, None, R, D, seed, iterations=T, host_call=sess)
    t0 = time.perf_counter()
    for i in range(reps):
        mcts.search(act, None, R, D, seed + i, iterations=T, host_call=sess)
    e2e_s = (time.perf_counter() - t0) / reps
    sess.close()
    cpu = None
    if int(os.environ.get("WORLD_SIZE", "1")) == 1 and (args is None or not getattr(args, "no_cpu_baseline", False)):
        # the C restatement of the oracle (oracle/c/planner_oracle.c, OpenMP over the rollouts of an iteration; it is
        # bit-identical to the numpy oracle, tests/test_oracle_c.py): the same search, 5 times, at the fastest thread count
        from oracle import c_oracle
        best = (None, float("inf"))
        for th in (8, 16, 32, 64):
            if th > (os.cpu_count() or 1):
                continue
            c_oracle.search(act.p, act.size, act.cost, R=R, D=D, T=2, seed=seed, threads=th)            # build + warm
            t0 = time.perf_counter()
            for i in range(3):
                c_oracle.search(act.p, act.size, act.cost, R=R, D=D, T=T, seed=seed + i, threads=th)
            dt = (time.perf_counter() - t0) / 3
            if dt < best[1]:
                best = (th, dt)
        cpu = {"value": T * R / best[1], "unit": "rollouts/s", "cores": best[0], "kind": "port", "seconds": best[1],
               "sample": f"oracle/c/planner_oracle.c (OpenMP over the {R} rollouts of an iteration), the full {T}-iteration search x3, "
                         "thread count auto-tuned"}
    ms16 = out_T[16][0]
    return {"metric": "mcts_rollouts_per_sec", "value": R * T / (ms * 1e-3), "unit": "rollouts/s", "ms_per_search": ms,
            "us_per_iteration": ms / T * 1e3, "cpu_baseline": cpu,
            "cfg3_T16": {"value": R * 16 / (ms16 * 1e-3), "ms_per_search": ms16, "rollouts_per_search": R * 16,
                         "note": "SURVEY.md 8d cfg 3 as written: 16 iterations x 4096 rollouts"},
            "api_value": R * T / api_s, "e2e_value": R * T / e2e_s,
            "config": {"actions": A, "rollouts_per_iteration": R, "depth": D, "iterations": T,
                       "note": "headline uses T=64 iterations (4x the rollouts of SURVEY.md's cfg 3, which is reported under cfg3_T16)"},
            "best_action": r.best,
            "note": "value: device time (CUDA events) of one search, inputs resident; api_value: SearchContext.search incl. "
                    "result read-back; e2e_value: nerrf_mcts_session_search_host (H2D + search + D2H inside the call, "
                    "device buffers owned by the session handle)"}


def run_lstm_bench(dev, B=4096, T=100):
    """BiLSTM(256 x 2 layers) over B candidate-file sequences of T=100 events (SURVEY.md 8a a4)."""
    import torch
    from nerrf_b200.ai.models import lstm
    model = lstm.LSTMScorer().to(dev)
    seq = torch.randn(B, T, 16, device=dev)
    lengths = torch.randint(T // 2, T + 1, (B,), device=dev)
    model(seq, lengths); torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); model(seq, lengths); model(seq, lengths); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 2
    flops = B * T * 2.0 * (2 * 1024 * (16 + 256) + 2 * 1024 * (512 + 256))      # both directions, both layers
    return {"metric": "lstm_sequences_per_sec", "value": B / (ms * 1e-3), "unit": "sequences/s", "ms": ms,
            "tflops_fp32_equivalent": flops / (ms * 1e-3) / 1e12, "config": {"batch": B, "T": T, "hidden": 256, "layers": 2},
            "algo": lstm.default_algo()}


def run_graph_build_bench(dev, rowptr, col, reps=3):
    """Device graph constructor (SURVEY.md 8f rank 1): the workload's own edges as a shuffled edge list -> CSR."""
    import torch
    from nerrf_b200.graph import build_csr_device, WINDOW
    N, E = rowptr.numel() - 1, col.numel()
    gen = torch.Generator(device=dev).manual_seed(7)
    dst = torch.repeat_interleave(torch.arange(N, device=dev, dtype=torch.int32), (rowptr[1:] - rowptr[:-1]).long())
    perm = torch.randperm(E, generator=gen, device=dev)
    src, dst = col[perm].contiguous(), dst[perm].contiguous()
    t = torch.rand(E, generator=gen, device=dev) * WINDOW
    conf = 0.5 + 0.5 * torch.rand(E, generator=gen, device=dev)
    del perm
    rp2, _, _ = build_csr_device(src, dst, t, conf, N)
    assert torch.equal(rp2, rowptr), "device constructor rowptr differs"
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        build_csr_device(src, dst, t, conf, N)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # the shape the pipeline produces: an event stream is in time order, so the sort only needs the destination bits
    order = torch.argsort(t)
    src_s, dst_s, t_s, conf_s = src[order].contiguous(), dst[order].contiguous(), t[order].contiguous(), conf[order].contiguous()
    del order
    rp3, _, _ = build_csr_device(src_s, dst_s, t_s, conf_s, N)
    assert torch.equal(rp3, rowptr), "device constructor rowptr differs (time-ordered input)"
    e0.record()
    for _ in range(reps):
        build_csr_device(src_s, dst_s, t_s, conf_s, N)
    e1.record(); torch.cuda.synchronize()
    ms_sorted = e0.elapsed_time(e1) / reps
    alg = 24.0 * E + 4.0 * (N + 1)          # read src,dst,t,conf; write col,ew; write rowptr
    own = not os.environ.get("NERRF_GRAPH_SORT", "").startswith("c")
    return {"metric": "graph_build_edges_per_sec", "value": E / (ms * 1e-3), "unit": "edges/s", "ms": ms,
            "algorithmic_gbps": alg / (ms * 1e-3) / 1e9,
            "time_ordered_input": {"value": E / (ms_sorted * 1e-3), "ms": ms_sorted,
                                   "note": "edge list already in time order (what a trace window is): destination bits only, 3 passes"},
            "config": {"nodes": N, "edges": E,
                       "sort": ("own stable LSD radix sort (csrc/radix_sort.cuh), 52-bit key, 7 passes (edge list in random time order)" if own
                                else "cub::DeviceRadixSort (NERRF_GRAPH_SORT=cub), 52-bit key")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="auto", choices=["auto", "ffma", "umma", "umma2"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true", help="N>1: skip the 10M/100M strong-scaling run")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the streamed fleet-trace end-to-end run")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "p2p-all", "multicast", "allgather", "broadcast", "allreduce"],
                    help="N>1: per-layer embedding exchange: p2p = fused into the layer kernel (epilogue stores to "
                         "peer-mapped buffers over NVLink, only the rows a peer references); p2p-all = same, every row "
                         "to every peer; multicast = NVSwitch multimem.st; allgather / broadcast / allreduce = NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one to DIR as float32 .npy (see the module "
                         "docstring); single process only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs needs a single-process run")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
