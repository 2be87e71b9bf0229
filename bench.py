#!/usr/bin/env python
"""Benchmark of the GNAN hot path (BASELINE.json metric: fwd+bwd graphs/s on graph tasks & nodes/s on node tasks, 1-8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload mol|mutag|cora|pubmed|arxiv] [--impl reference] [--dump-outputs DIR] ...

`--steps K` is the number of timed steps of both GPU legs (device-resident and e2e) of every workload; the per-kernel attribution
pass runs min(K, 10) steps, and the CPU reference arm runs at least 2 steps within its time budget.

A step is forward + loss + backward + Adam step (trainer.py:48-67). Workloads = BASELINE.json configs:
  mol     configs[4]  32768 molecule-shaped graphs (10-100 nodes) per step and rank, GPU all-pairs hop preprocessing of the
                      batch INSIDE the step; data-parallel over ranks (one gradient all-reduce). Weak scaling.
  mutag   configs[0]  4337 Mutagenicity-shaped graphs per step and rank, packed block-diagonal form, data-parallel.
  cora    configs[1]  2708 nodes x 1434 features, 7 classes; replicas only (does not shard).
  pubmed  configs[2]  19717 nodes x 501 features, 3 classes; hop rows sharded over ranks (strong scaling).
  arxiv   configs[3]  169343 nodes x 129 features, 40 classes, 28.7 GB of hop bytes; hop rows sharded over ranks.

Default (no --workload): the HEADLINE line is `mol`, the configuration that shards at every N (so that the 1-2-4-8 scaling
run measures a real data-parallel step with a collective in it), and the same JSON line carries `sub_records` for the other
configs: at N = 1 cora (the node-task half of the metric), mutag, pubmed and arxiv, each with its own value / e2e /
roofline / cpu_baseline; at N > 1 the row-sharded arxiv step (all-gather of S + reduce-scatter of dS + gradient all-reduce,
strong scaling) with per-step collective times, plus `parity_vs_single_gpu` (data-parallel and row-sharded results against
the single-GPU computation of the same problem).

`value` times the step with inputs resident in HBM (CUDA events per step, L2 flushed between steps); `e2e` times the same
step through the module API from pinned HOST buffers (copied every step, loss read back every step). `roofline` describes
the dominant kernel of the step (largest CUDA-event time among the library's ops, measured live on the launching stream).
`cpu_baseline` / `--impl reference` time the reference's CPU path on the box's host cores: the UNMODIFIED reference modules
when a copy is importable (baseline/_ref or /root/reference, through oracle/pyg_shim.py), else the oracle's port of them
(oracle/gnan_port.py; the reference is pure Python and does not travel to the GPU box).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, L = 64, 3   # run.sh:10-11
MOL_NBINS = 48 # fixed level-table width of the in-step BFS of the molecule workload (47 hop levels + the unreachable bin)


# ---------------------------------------------------------------------------------------------------------------------
# synthetic workloads (SURVEY.md §8d)
# ---------------------------------------------------------------------------------------------------------------------
def random_simple_graph(rng, n, n_undirected_edges, n_isolated):
    m = n - n_isolated
    need = n_undirected_edges
    got = np.zeros((0, 2), dtype=np.int64)
    while got.shape[0] < need:
        s = rng.integers(0, m, size=2 * (need - got.shape[0]) + 16)
        d = rng.integers(0, m, size=s.shape[0])
        e = np.stack([np.minimum(s, d), np.maximum(s, d)], 1)[s != d]
        got = np.unique(np.concatenate([got, e]), axis=0)
    got = got[rng.permutation(got.shape[0])[:need]]
    return np.concatenate([got, got[:, ::-1]]).T.copy()


def make_node_workload(name, seed=0, classes=None):
    rng = np.random.default_rng(seed)
    if name == "cora":
        n, k_raw, c, e_und, iso, dens = 2708, 1433, 7, 5278, 54, 0.0127
        x = (rng.random((n, k_raw)) < dens).astype(np.float32)
        x /= np.maximum(x.sum(1, keepdims=True), 1.0)                       # row-normalised bag of words (datasets.py:94)
        desc = "cora-shape TensorGNAN node classification (BASELINE.json configs[1])"
    elif name == "arxiv":
        n, k_raw, c, e_und, iso = 169343, 128, 40, 583121, 0        # 1 166 243 directed edges ~ 583 k undirected pairs
        x = rng.normal(size=(n, k_raw)).astype(np.float32)
        desc = "ogbn-arxiv-shape TensorGNAN node classification (BASELINE.json configs[3]), 28.7 GB uint8 hop matrix"
    else:
        n, k_raw, c, e_und, iso, dens = 19717, 500, 3, 44338, 0, 0.10
        x = ((rng.random((n, k_raw)) < dens) * rng.random((n, k_raw)) * 0.1).astype(np.float32)
        desc = "pubmed-shape TensorGNAN node classification (BASELINE.json configs[2])"
    if classes:
        c = classes
    x = np.concatenate([x, np.ones((n, 1), np.float32)], 1)                 # pre_process_datasets.py:127
    ei = random_simple_graph(rng, n, e_und, iso)
    y = rng.integers(0, c, size=n)
    mask = np.zeros(n, bool)
    mask[rng.permutation(n)[:140]] = True
    return SimpleNamespace(kind="node", name=name, desc=desc, n=n, K=k_raw + 1, C=c, x=torch.from_numpy(x),
                           edge_index=torch.from_numpy(ei), y=torch.from_numpy(y), train_mask=torch.from_numpy(mask),
                           unit="nodes/s", units_per_step=n, evals_per_step=n * (k_raw + 1))


def make_graph_workload(seed=0, n_graphs=4337):
    """Mutagenicity-shaped batch: n_g = clip(round(N(30.3, 20)), 4, 120), random tree + ceil(n/10) extra edges, one-hot over
    14 atom types + the constant column (K = 15), binary labels, C = 1 (main.py:347-349)."""
    rng = np.random.default_rng(seed)
    sizes = np.clip(np.round(rng.normal(30.3, 20.0, size=n_graphs)), 4, 120).astype(np.int64)
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    src, dst = [], []
    for g, n in enumerate(sizes):
        par = np.array([rng.integers(0, v) for v in range(1, n)], dtype=np.int64)
        e = set(zip(par.tolist(), range(1, n)))
        extra = int(np.ceil(n / 10))
        while extra > 0:
            a, b = int(rng.integers(0, n)), int(rng.integers(0, n))
            if a != b and (min(a, b), max(a, b)) not in e:
                e.add((min(a, b), max(a, b))); extra -= 1
        e = np.array(sorted(e), dtype=np.int64) + node_off[g]
        src += [e[:, 0], e[:, 1]]; dst += [e[:, 1], e[:, 0]]
    ei = np.stack([np.concatenate(src), np.concatenate(dst)])
    tot = int(node_off[-1])
    x = np.zeros((tot, 15), np.float32)
    x[np.arange(tot), rng.integers(0, 14, size=tot)] = 1.0
    x[:, 14] = 1.0
    y = rng.integers(0, 2, size=n_graphs).astype(np.float32)
    return SimpleNamespace(kind="graph", name="mutag", desc="Mutagenicity-shape TensorGNAN graph classification, 4337 graphs per "
                           "step in packed block-diagonal form (BASELINE.json configs[0])", n=tot, K=15, C=1,
                           x=torch.from_numpy(x), edge_index=torch.from_numpy(ei), node_off=torch.from_numpy(node_off),
                           sizes=sizes, y=torch.from_numpy(y), unit="graphs/s", units_per_step=n_graphs, evals_per_step=tot * 15)


def make_mol_workload(seed=0, n_graphs=32768, n_lo=10, n_hi=100):
    """BASELINE.json configs[4]: molecular graphs with n ~ U{10..100}, random tree + ceil(n/10) extra edges, one-hot over 14
    types + constant column, C = 1. Generated vectorised; one step = one batch of `n_graphs` graphs INCLUDING the GPU
    all-pairs hop-distance preprocessing of that batch (edge list -> packed hop blocks + level counts)."""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(n_lo, n_hi + 1, size=n_graphs).astype(np.int64)
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    tot = int(node_off[-1])
    gid = np.repeat(np.arange(n_graphs), sizes)
    local = np.arange(tot) - node_off[gid]
    child = np.nonzero(local > 0)[0]
    parent = node_off[gid[child]] + np.floor(rng.random(child.shape[0]) * local[child]).astype(np.int64)
    n_extra = np.ceil(sizes / 10).astype(np.int64)
    eg = np.repeat(np.arange(n_graphs), n_extra)
    ea = node_off[eg] + np.floor(rng.random(eg.shape[0]) * sizes[eg]).astype(np.int64)
    eb = node_off[eg] + np.floor(rng.random(eg.shape[0]) * sizes[eg]).astype(np.int64)
    a = np.concatenate([parent, np.minimum(ea, eb)]); b = np.concatenate([child, np.maximum(ea, eb)])
    keep = a != b
    und = np.unique(np.stack([a[keep], b[keep]], 1), axis=0)            # simple graph: drop self loops and duplicates
    ei = np.concatenate([und, und[:, ::-1]]).T.copy()
    x = np.zeros((tot, 15), np.float32)
    x[np.arange(tot), rng.integers(0, 14, size=tot)] = 1.0
    x[:, 14] = 1.0
    y = rng.integers(0, 2, size=n_graphs).astype(np.float32)
    return SimpleNamespace(kind="graph", name="mol", desc=f"molecule-shape TensorGNAN graph classification (BASELINE.json configs[4]): "
                           f"{n_graphs} graphs of {n_lo}-{n_hi} nodes per step, GPU APSP preprocessing of the batch inside the step",
                           n=tot, K=15, C=1, x=torch.from_numpy(x), edge_index=torch.from_numpy(ei), node_off=torch.from_numpy(node_off),
                           sizes=sizes, y=torch.from_numpy(y), unit="graphs/s", units_per_step=n_graphs, evals_per_step=tot * 15)


def flops_per_eval(C):
    return 2 * H + (L - 2) * 2 * H * H + 2 * H * C      # forward FLOPs of one shape-function evaluation (SURVEY §8d)


# ---------------------------------------------------------------------------------------------------------------------
def clocks_sampler():
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        return subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                 "-i", os.environ.get("LOCAL_RANK", "0")], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return None


def clocks_summary(proc):
    if proc is None:
        return None
    proc.terminate()
    try:
        out, _ = proc.communicate(timeout=5)
    except Exception:
        return None
    sm, mx, reasons = [], 0.0, set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in out.strip().splitlines():
        f = [t.strip() for t in line.split(",")]
        if len(f) < 9:
            continue
        try:
            sm.append(float(f[1])); mx = max(mx, float(f[2]))
        except ValueError:
            continue
        for nme, v in zip(names, f[5:9]):
            if v.lower().startswith("active"):
                reasons.add(nme)
    if not sm:
        return None
    return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json: hbm_gbs for HBM-bound kernels, bf16_tflops_sustained for tensor-bound ones)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"



def workload_config(wl, where, world=1):
    shard = "hop rows sharded over ranks: all-gather of S, reduce-scatter of dS, all-reduce of the parameter gradients"
    dp = "data-parallel graphs: one all-reduce of the flat gradient buffer per step"
    par = {"cora": "replicas only (SURVEY.md §8e: small node-level graph)", "pubmed": shard, "arxiv": shard, "mutag": dp, "mol": dp}[wl.name]
    return {"workload": wl.desc, "nodes": wl.n, "features": wl.K, "classes": wl.C, "hidden": H, "n_layers": L,
            "step": "forward + loss + backward + Adam", "normalize_rho": True, "dropout": 0.0,
            "timing": "CUDA events per step; 256 MiB L2 flush between timed steps" if where == "gpu" else "perf_counter",
            "parallelism": par if world > 1 else "single GPU"}


def make_workload(name, seed=0, classes=0):
    if name == "mutag":
        return make_graph_workload(seed=seed)
    if name == "mol":
        return make_mol_workload(seed=seed)
    return make_node_workload(name, classes=classes)


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU path on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def find_reference():
    """Directory holding the unmodified reference modules, or None (the GPU box has none: /root/reference does not travel)."""
    for d in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if os.path.exists(os.path.join(d, "GNAN.py")) and os.path.exists(os.path.join(d, "models.py")):
            return d
    return None


def reference_step_fn(wl, seed=0):
    """Returns (step_fn, n_threads, units_per_call, note, kind). kind = "reference": the unmodified GNAN.py / models.py
    modules driven through their own forward; kind = "port": oracle.gnan_port (same op order, pinned to the reference's outputs)."""
    from oracle import apsp as oapsp
    torch.manual_seed(seed)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    ref_dir = find_reference()
    node = wl.kind == "node"
    if ref_dir is not None:
        from oracle import pyg_shim
        gnan_py, models_py, _, _ = pyg_shim.import_reference(ref_dir)
        if node:
            cls = gnan_py.TensorGNAN if wl.name == "cora" else gnan_py.GNAN
            m = (cls(wl.K, wl.C, L, H, normalize_rho=True, is_graph_task=False) if wl.name == "cora"
                 else cls(wl.K, wl.C, L, H, normalize_rho=True, rho_per_feature=True))
        else:
            m = models_py.TensorGNAN(wl.K, wl.C, L, H, normalize_rho=True, is_graph_task=True, readout_n_layers=0)
        with torch.no_grad():                                       # same O(1)-scale weights as the GPU arm (cost does not depend on them)
            for n_, p in m.named_parameters():
                if "weight" in n_:
                    torch.nn.init.xavier_normal_(p, gain=1.0)
        params = list(m.parameters())
        kind, src = "reference", f"unmodified reference modules from {ref_dir}"
        fwd_full = lambda x, nd, nm: m(SimpleNamespace(x=x, edge_index=None, node_distances=nd, normalization_matrix=nm))
        fwd_rows = lambda x, nd, nm, rows: m(SimpleNamespace(x=x, edge_index=None, node_distances=nd, normalization_matrix=nm), node_ids=rows)
    else:
        from oracle import gnan_port
        from oracle import params as P
        if node:
            from gnan_b200.GNAN import TensorGNAN
            g = TensorGNAN(wl.K, wl.C, L, H, normalize_rho=True, is_graph_task=False)
        else:
            from gnan_b200.models import TensorGNAN
            g = TensorGNAN(wl.K, wl.C, L, H, normalize_rho=True, is_graph_task=True, readout_n_layers=0)
        g.fs.xavier_normal_(1.0); g.rho.xavier_normal_(1.0)
        sd = {k: v.detach().numpy() for k, v in g.state_dict().items()}
        fs = gnan_port.to_torch(P.stack_mlps(sd, [f"fs.{k}" for k in range(wl.K)], L, 3), torch.float32, True)
        rho = gnan_port.to_torch(P.stack_mlps(sd, ["rho"], L, 2, node), torch.float32, True)
        params = [t for d in (fs, rho) for t in d.values() if t is not None and t.requires_grad]
        kind, src = "port", "oracle/gnan_port.py (port of the reference modules; no reference copy on this box)"
        if node:
            fwd_full = lambda x, nd, nm: gnan_port.tensor_gnan_gnanpy(fs, rho, x, nd, nm, True, False)
        else:
            fwd_full = lambda x, nd, nm: gnan_port.tensor_gnan_models(fs, rho, x, nd, nm, True, True, None)
        fwd_rows = lambda x, nd, nm, rows: gnan_port.gnan_rowloop(fs, rho, x, nd, nm, True, rows)
    opt = torch.optim.Adam(params, lr=1e-3)
    if wl.name == "cora":
        hop = oapsp.apsp(wl.edge_index.numpy(), wl.n)
        nd, nm = (torch.from_numpy(t) for t in oapsp.reference_format(hop, oapsp.level_counts(hop)))
        loss_fn = torch.nn.CrossEntropyLoss()

        def step():
            opt.zero_grad()
            out = fwd_full(wl.x, nd, nm)                                                   # GNAN.py:55-79, full graph
            loss = loss_fn(out[wl.train_mask], wl.y[wl.train_mask])
            loss.backward(); opt.step()
            return float(loss.item())
        return step, threads, wl.n, f"full {wl.name}-shape step (fwd+CE+bwd+Adam), GNAN.py TensorGNAN; {src}", kind
    if wl.name in ("pubmed", "arxiv"):          # the shipped TensorGNAN cannot run at this shape (99.5 GB activation): row loop on 64 rows
        rows = 64
        hop = oapsp.apsp_rows(wl.edge_index.numpy(), wl.n, rows)       # BFS from the first 64 sources only
        cnt = oapsp.level_counts(hop)
        nd, nm = (torch.from_numpy(t) for t in oapsp.reference_format(hop, cnt))
        loss_fn = torch.nn.CrossEntropyLoss()

        def step():
            opt.zero_grad()
            out = fwd_rows(wl.x, nd, nm, list(range(rows)))                                # GNAN.py:146-172 on a [64,N] slice
            loss = loss_fn(out, wl.y[:rows])
            loss.backward(); opt.step()
            return float(loss.item())
        return (step, threads, rows, "GNAN.forward(node_ids=range(64)) on a [64,N] slice: rows/s, NOT a full step (full shape not "
                f"runnable on a CPU); {src}", kind)
    # graph tasks: one graph per step (datasets.py:339-341, batch_size=1), models.TensorGNAN (what main.py builds); the
    # per-graph Dijkstra preprocessing the reference does once per dataset is NOT in the timed step
    graphs = []
    for g_ in range(min(200, len(wl.sizes))):
        b, e = int(wl.node_off[g_]), int(wl.node_off[g_ + 1])
        sel = (wl.edge_index[0] >= b) & (wl.edge_index[0] < e)
        hop = oapsp.apsp((wl.edge_index[:, sel] - b).numpy(), e - b)
        nd, nm = (torch.from_numpy(t) for t in oapsp.reference_format(hop, oapsp.level_counts(hop)))
        graphs.append((wl.x[b:e], nd, nm, wl.y[g_:g_ + 1]))
    loss_fn = torch.nn.BCEWithLogitsLoss()
    state = {"i": 0}

    def step():
        x, nd, nm, y = graphs[state["i"] % len(graphs)]
        state["i"] += 1
        opt.zero_grad()
        out = fwd_full(x, nd, nm)                                                          # models.py:358-384
        loss = loss_fn(out.flatten(), y)
        loss.backward(); opt.step()
        return float(loss.item())
    return step, threads, 1, f"one graph per step (batch_size=1 as datasets.py:339), models.py TensorGNAN, fwd+BCE+bwd+Adam; {src}", kind


def time_reference(wl, steps, warmup, budget_s, group=1):
    """group > 1: one timed step = `group` consecutive reference steps (graph tasks: a bounded sample of `group` single-graph
    steps, so that `--steps K` keeps its meaning while a step stays long enough to time)."""
    step1, threads, units, note, kind = reference_step_fn(wl)
    if group > 1:
        units, note = units * group, f"{group} x [{note}] per step"

        def step():
            for _ in range(group):
                step1()
    else:
        step = step1
    t_begin = time.perf_counter()
    w_done = 0
    for _ in range(warmup):
        if w_done >= 1 and time.perf_counter() - t_begin > budget_s / 3:
            break
        step(); w_done += 1
    times = []
    for _ in range(steps):
        t0 = time.perf_counter(); step(); times.append(time.perf_counter() - t0)
        if len(times) >= 2 and time.perf_counter() - t_begin > budget_s:
            break
    ms = 1e3 * sum(times) / len(times)
    extras = {}                                        # side figures merged into the cpu_baseline record
    if wl.kind == "graph":
        # the shipped trainer wraps every epoch in torch.autograd.set_detect_anomaly(True) (trainer.py:24): the same steps as the
        # reference really runs them, reported next to the plain figure (SURVEY §8d-i); `value` stays the faster, plain one
        n_an = 40
        with torch.autograd.set_detect_anomaly(True):
            step1()
            t0 = time.perf_counter()
            for _ in range(n_an):
                step1()
            extras["value_with_anomaly_mode"] = n_an * (units // group) / (time.perf_counter() - t0)
    return units / (ms / 1e3), ms, len(times), w_done, threads, note, kind, extras


def reference_apsp_record(wl, n_graphs=100):
    """The reference's own hop preprocessing (pre_process_datasets.py:104-122: scipy Dijkstra + the per-entry normaliser loop) on the
    first `n_graphs` graphs of a graph workload, timed on one core as the reference runs it (SURVEY §8d-iv). Reported NEXT TO the
    model step: the GPU step of the molecule workload contains its preprocessing, the reference's `value` does not. None when no
    copy of the unmodified reference is importable (the oracle's C BFS is a different algorithm and is not timed in its place)."""
    ref_dir = find_reference()
    if ref_dir is None or wl.kind != "graph":
        return None
    import contextlib
    import io
    import tempfile
    from oracle import pyg_shim
    _, _, pre_py, _ = pyg_shim.import_reference(ref_dir)
    graphs = []
    for g_ in range(min(n_graphs, len(wl.sizes))):
        b, e = int(wl.node_off[g_]), int(wl.node_off[g_ + 1])
        sel = (wl.edge_index[0] >= b) & (wl.edge_index[0] < e)
        graphs.append(SimpleNamespace(x=wl.x[b:e, :-1].clone(), edge_index=(wl.edge_index[:, sel] - b).clone()))   # pre_process appends the constant column
    with tempfile.TemporaryDirectory() as tmp, contextlib.redirect_stdout(io.StringIO()):
        t0 = time.perf_counter()
        pre_py.pre_process(graphs, True, "bench_sample", processed_data_dir=tmp)
        dt = time.perf_counter() - t0
    return {"value": len(graphs) / dt, "unit": "graphs/s", "cores": 1, "kind": "reference",
            "sample": f"unmodified pre_process_datasets.pre_process on the first {len(graphs)} graphs of the batch ({1e3 * dt / len(graphs):.1f} ms per graph, "
                      "incl. writing its processed_data file)"}


def with_apsp(rec, wl):
    """adds the reference's preprocessing rate and the combined rate (model step + preprocessing per graph) to a cpu_baseline record,
    (on top of time_reference's side figures, already merged by the caller)"""
    try:
        ap = reference_apsp_record(wl) if wl.name == "mol" else None
    except Exception as exc:                                   # an extra figure: never costs the line
        rec["apsp_preprocessing"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
        return rec
    if ap is not None:
        rec["apsp_preprocessing"] = ap
        rec["value_incl_apsp"] = 1.0 / (1.0 / rec["value"] + 1.0 / ap["value"])
    return rec


def cpu_baseline_record(wl, budget_s):
    graph = wl.kind == "graph"
    val, ms, n, w, threads, note, kind, extras = time_reference(wl, 50 if graph else 2, 5 if graph else 1, budget_s)
    return with_apsp({"value": val, "unit": wl.unit if wl.name in ("cora", "mutag", "mol") else "rows/s", "cores": threads, "kind": kind,
                      "sample": f"{n} timed steps after {w} warm-up ({ms:.1f} ms each): {note}", **extras}, wl)


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    wl = make_workload(args.workload or "mol", classes=args.classes)
    # graph tasks: the reference trains one graph at a time (a few ms each); a bench step is a bounded sample of 50 of them
    val, ms, n, w, threads, note, kind, extras = time_reference(wl, max(args.steps, 2), max(args.warmup, 1), 300.0, group=50 if wl.kind == "graph" else 1)
    print(json.dumps({
        "impl": "reference", "metric": f"GNAN fwd+bwd {wl.unit} ({wl.name}-shape TensorGNAN)", "value": val, "unit": wl.unit,
        "n_gpus": args.gpus, "steps": n, "warmup": w, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(wl, "cpu"),
        "cpu_baseline": with_apsp({"value": val, "unit": wl.unit, "cores": threads, "kind": kind,
                                   "sample": f"{n} steps after {w} warm-up: {note}", **extras}, wl),
        "e2e": {"value": val, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# one workload on the GPUs of this job -> one record
# ---------------------------------------------------------------------------------------------------------------------
KERNEL_NAMES = {
    "mlp_bwd": "mlp_tc_bwd_kernel / mlp_bwd_kernel", "mlp_fwd": "mlp_tc_fwd_kernel / mlp_fwd_kernel",
    "mlp_entries_bwd": "mlp_entries_bwd_small_kernel (<= 96 entries per feature on average) | mlp_tc_bwd_kernel / mlp_bwd_kernel (entries mode)", "mlp_entries_fwd": "mlp_fwd_kernel (entries mode)",
    "aggregate_rows_fwd_save": "agg_tc_fwd_kernel (+ colmax / digits pre-pass) | agg_rows_bins_kernel",
    "aggregate_rows_bwd_saved": "agg_tc_ds_kernel (+ row compaction, digits, dT kernels) | agg_rows_ds_kernel",
    "aggregate_blockdiag_fwd": "agg_bd_graph_fwd_kernel | agg_blockdiag_fwd_rows_kernel",
    "aggregate_blockdiag_bwd": "agg_bd_graph_ds/dt kernels | agg_blockdiag_bwd_global_kernel",
    "apsp_bfs_batched": "apsp_batched_v3_kernel (+ bv3_classify_kernel)", "build_csr": "csr_degree/fill/duplicates kernels + cub scan",
}
COLLECTIVES = ("allgather_rows", "reduce_scatter_rows", "allreduce_gradients")


DUMP_SAMPLE = 1 << 20   # elements kept of a larger dumped array
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes each tensor as <out_dir>/<name>.npy, float64 as float64 and anything else as float32. An array of more than DUMP_SAMPLE
    elements is reduced to a fixed seeded sample of its flattened values: the same positions in every run, so that two builds can be
    compared output for output. Refuses to write more than DUMP_MAX_BYTES in all."""
    out = {}
    for nm, t in arrays.items():
        a = t.detach().cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        out[nm] = a
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for nm, a in out.items():
        np.save(os.path.join(out_dir, nm + ".npy"), a)


def run_workload(args, env, name, *, steps, warmup, classes=0, compare_legs=False, cpu_budget_s=60.0, dump_dir=None):
    import torch.distributed as dist
    from gnan_b200 import ops
    from gnan_b200 import dist as gdist
    from gnan_b200.preprocess import HopData, LocalEdges, PackedBatch, apsp, apsp_batched
    from gnan_b200.sparse import compress_features
    from gnan_b200.packed import HostBundle
    from gnan_b200.trainer import CapturedStep
    from gnan_b200.optim import Adam as FusedAdam
    world, rank, dev, flush, lib = env.world, env.rank, env.dev, env.flush, env.lib
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    wl = make_workload(name, seed=rank, classes=classes)

    torch.manual_seed(0)
    if wl.kind == "node":
        from gnan_b200.GNAN import TensorGNAN
        model = TensorGNAN(wl.K, wl.C, L, H, normalize_rho=True, is_graph_task=False, device=dev).to(dev)
    else:
        from gnan_b200.models import TensorGNAN
        model = TensorGNAN(wl.K, wl.C, L, H, normalize_rho=True, is_graph_task=True, readout_n_layers=0, device=dev).to(dev)
    model.fs.xavier_normal_(1.0); model.rho.xavier_normal_(1.0)
    model.precision = args.precision
    model.dedup = args.dedup == "on" and wl.name != "arxiv"         # arxiv features are continuous: nothing to share
    opt = FusedAdam(model.parameters(), lr=1e-3)               # torch.optim.Adam semantics, one launch for all tensors (csrc/train.cu)
    sharded = wl.name in ("pubmed", "arxiv") and world > 1
    scaling = "strong" if sharded else "weak"
    fg = gdist.FlatGradients(model.parameters()) if world > 1 and wl.name != "cora" else None
    zero_grads = (lambda: fg.zero()) if fg is not None else (lambda: opt.zero_grad(set_to_none=True))
    last_out = [None]                                           # the model output of the latest step (a captured step rewrites it)

    # ---- device-resident inputs and the step ------------------------------------------------------------------------
    if wl.kind == "node":
        loss_fn = torch.nn.CrossEntropyLoss(reduction="sum")
        if sharded:
            blocks = [gdist.row_block(wl.n, r, world) for r in range(world)]
            sizes = [e - b for b, e in blocks]
            b0, e0 = blocks[rank]
            hd = apsp(wl.edge_index, wl.n, device=dev, row_begin=b0, row_end=e0)
        else:
            b0, e0, sizes = 0, wl.n, [wl.n]
            hd = apsp(wl.edge_index, wl.n, device=dev)                  # GPU preprocessing (not part of the timed step)
        x_h = wl.x[b0:e0].contiguous()
        big = hd.hop.numel() > (2 << 30)            # do not stage tens of GB in pinned host memory: no hop copy in the e2e leg
        hop_h = None if big else hd.hop.cpu()
        cnt_h = hd.level_counts.cpu()
        idx_d = wl.train_mask[b0:e0].nonzero().flatten().to(dev)
        yl_d = wl.y[b0:e0].to(dev)[idx_d]
        n_train = float(wl.train_mask.sum())
        n_train_local = int(idx_d.numel())
        x_d = x_h.to(dev)
        cx = compress_features(x_d) if model.dedup else None                           # once per dataset (per row shard), like the hop matrix
        cx_h = None if cx is None else cx.compact_host()      # narrow index arrays on the host side
        data_d = SimpleNamespace(x=x_d, hop_data=hd, x_compressed=cx)
        x_bytes = x_h.numel() * 4 if cx is None else cx_h.nbytes()
        h2d = x_bytes + (0 if big else hop_h.numel()) + cnt_h.numel() * 4

        host_parts = ([x_h] if cx is None else cx_h._tensors()) + ([] if big else [hop_h]) + [cnt_h]

        def assemble(views):                                           # the step's input object over typed views of a staging buffer
            it = iter(views)
            xx = next(it) if cx is None else None
            c = None if cx is None else cx_h._map(lambda t: next(it))
            hop_d = hd.hop if big else next(it)
            return SimpleNamespace(x=xx, hop_data=HopData(hop_d, next(it), wl.n, b0), x_compressed=c)

        def widen(d):                                                  # eager steps read the compact copy through widened tensors
            return d if d.x_compressed is None else SimpleNamespace(x=d.x, hop_data=d.hop_data, x_compressed=d.x_compressed.to(dev))

        def loss_of(data):
            if sharded:
                out = gdist.row_sharded_forward(model, data.x, data.hop_data, sizes, x_compressed=data.x_compressed)
            else:
                out = model.forward(data)
            last_out[0] = out.detach()
            # masked cross entropy: value and the [N,C] output gradient from one kernel (trainer.py:52-66)
            return ops.cross_entropy_rows(out, yl_d, rows=idx_d, scale=1.0 / n_train)
        after_bwd = (lambda: fg.all_reduce()) if sharded else None
        rows_local = e0 - b0
        in_step_apsp = False
    else:
        loss_fn = torch.nn.BCEWithLogitsLoss()
        in_step_apsp = wl.name == "mol"
        node_off_h = wl.node_off.numpy()
        pk = apsp_batched(wl.edge_index, node_off_h, device=dev, x=wl.x.to(dev), y=wl.y.to(dev))
        lc_h = pk.level_counts.cpu()
        lc_max = int(lc_h.max()) if lc_h.numel() else 0                 # the level sizes cross PCIe in the narrowest type that holds them
        lc_h = lc_h.to(torch.uint8 if lc_max < 256 else torch.int16 if lc_max < 32768 else torch.int32)
        host = PackedBatch(wl.x, pk.hop.cpu(), pk.hop_off.cpu(), pk.node_off.cpu(), lc_h, wl.y, pk.max_nodes)
        cx = compress_features(pk.x) if model.dedup else None
        cx_h = None if cx is None else cx.compact_host()      # narrow index arrays on the host side
        pk.x_compressed = cx
        data_d = pk
        x_bytes = host.x.numel() * 4 if cx is None else cx_h.nbytes()
        h2d = x_bytes + sum(t.numel() * t.element_size() for t in (host.hop, host.hop_off, host.node_off, host.level_counts, host.y))
        if in_step_apsp:                                                # the step starts from the raw edge list
            noff_d, hoff_d, x_d, y_d = pk.node_off, pk.hop_off, wl.x.to(dev), wl.y.to(dev)
            # the batch's edge list in its transfer form: uint8 endpoints inside their graph + per-graph edge offsets (2 bytes per
            # directed edge cross PCIe). --edge-format local (default): the step consumes it as it is (the BFS kernel builds each
            # graph's adjacency in shared memory: no CSR builder); int64: the step starts from PyG's int64 [2,E] edge_index
            # (gnan_edges_from_local rebuilds it on the device in the e2e leg, then gnan_build_csr + BFS)
            ei_h = LocalEdges.from_edge_index(wl.edge_index, node_off_h)
            local_edges = args.edge_format == "local"
            pair_stats = local_edges and args.pair_stats
            ei_d = ei_h.to(dev) if local_edges else wl.edge_index.to(dev)
            noff_h, hoff_h = pk.node_off.cpu(), pk.hop_off.cpu()
            data_d = (ei_d, noff_d, hoff_d, x_d, y_d, cx)
            h2d = x_bytes + ei_h.nbytes() + sum(t.numel() * t.element_size() for t in (noff_h, hoff_h, host.y))
            apsp_status = []

        feat_parts = [host.x] if cx is None else cx_h._tensors()
        if in_step_apsp:
            host_parts = [ei_h.src, ei_h.dst, ei_h.edge_off, noff_h, hoff_h] + feat_parts + [host.y]
        else:
            host_parts = feat_parts + [host.hop, host.hop_off, host.node_off, host.level_counts, host.y]

        def assemble(views):
            it = iter(views)
            if in_step_apsp:
                le, no, ho = LocalEdges(next(it), next(it), next(it)), next(it), next(it)
            xx = next(it) if cx is None else None
            c = None if cx is None else cx_h._map(lambda t: next(it))
            if in_step_apsp:
                return (le, no, ho, xx, next(it), c)
            b = PackedBatch(xx, next(it), next(it), next(it), next(it), next(it), host.max_nodes)
            b.x_compressed = c
            return b

        def widen(d):
            if in_step_apsp:
                e = d[0].expand(d[1]) if isinstance(d[0], LocalEdges) and not local_edges else d[0]
                return (e, d[1], d[2], d[3], d[4], None if d[5] is None else d[5].to(dev))
            if getattr(d, "x_compressed", None) is not None:
                d.x_compressed = d.x_compressed.to(dev)
            if d.level_counts is not None and d.level_counts.dtype != torch.int32:
                d.level_counts = d.level_counts.to(torch.int32)
            return d

        def loss_of(data):
            if in_step_apsp:                                            # GPU BFS of the batch (pre_process_datasets.py:106-122); the graph
                e, no, ho, xx, yy, c = data                             # boundaries are host metadata of the loader, like the batch size
                # fixed-width level table (48 levels; deeper batches raise the overflow flag, checked after the timed loop):
                # no host synchronisation inside the step, so CSR build + BFS + model step replay as ONE CUDA graph
                # hop bytes + fused normaliser table, one-pass readout kernel; with --pair-stats the BFS accumulates the pair statistics
                # of the graph readout itself (undirected molecules) and the model never reads the hop bytes
                data = apsp_batched(e, node_off_h, device=dev, x=xx, y=yy, node_off_device=no, hop_off_device=ho, nbins=MOL_NBINS,
                                    rscale=not pair_stats, pair_stats=pair_stats)
                data.x_compressed = c
                apsp_status[:] = [data.status]
            out = model(data)
            last_out[0] = out.detach()
            return ops.bce_with_logits(out.flatten(), data.y)           # model(data): [B,1]; BCEWithLogitsLoss, value + gradient in one kernel
        after_bwd = (lambda: fg.all_reduce(average=True)) if world > 1 else None
        rows_local = wl.n
        n_train_local = None

    def step(data):
        zero_grads()
        loss = loss_of(data)
        loss.backward()
        if after_bwd is not None:
            after_bwd()
        opt.step()
        return loss

    for _ in range(warmup):
        step(data_d)
    torch.cuda.synchronize()

    # ---- capture the whole step (forward + loss + backward [+ collectives] + Adam) into one CUDA graph ----------------------
    graphed, launches_per_step = None, None
    if not args.no_cuda_graph:
        try:
            scx = None if cx is None else cx.to(dev).clone_tensors()
            if wl.kind == "node":
                hop_static = data_d.hop_data.hop if big else data_d.hop_data.hop.clone()
                static_hop = HopData(hop_static, data_d.hop_data.level_counts.clone(), wl.n, b0)
                static_hop.static_level_counts = True          # the level counts are refreshed with the same values only (see trainer.CapturedStep)
                static_in = SimpleNamespace(x=None if cx is not None else data_d.x.clone(), hop_data=static_hop, x_compressed=scx)
            elif in_step_apsp:
                ei_s = LocalEdges(ei_d.src.clone(), ei_d.dst.clone(), ei_d.edge_off.clone()) if local_edges else ei_d.clone()
                static_in = (ei_s, noff_d.clone(), hoff_d.clone(), None if cx is not None else x_d.clone(), y_d.clone(), scx)
            else:
                static_in = PackedBatch(None if cx is not None else data_d.x.clone(), data_d.hop.clone(), data_d.hop_off.clone(),
                                        data_d.node_off.clone(), data_d.level_counts.clone(), data_d.y.clone(), data_d.max_nodes)
                static_in.x_compressed = scx
                static_in.static_level_counts = True
            cap = CapturedStep(lambda: loss_of(static_in), opt, warmup=2, after_backward=after_bwd, zero_grad=zero_grads)
            graphed, launches_per_step = (cap, static_in), cap.kernel_launches
            for _ in range(3):
                cap()
            torch.cuda.synchronize()
        except Exception as exc:                                    # pragma: no cover
            print(f"[bench] {name}: CUDA graph capture failed, running eagerly: {exc!r}", file=sys.stderr)
            graphed = None
            torch.cuda.synchronize()

    inputs_consumed = torch.cuda.Event()                            # recorded once a step no longer reads the tensors handed to it

    refresh_graphs = {}                                             # id(staged input object) -> CUDA graph of its refresh copies

    def refresh(data):
        """static inputs of the captured step <- a staged batch (typed views of a device staging buffer; widens the compact types)"""
        sin = graphed[1]
        if in_step_apsp:
            for dst, src in zip(sin[1:5], data[1:5]):
                if dst is not None:
                    dst.copy_(src, non_blocking=True)
            if local_edges:
                for dst, src in zip((sin[0].src, sin[0].dst, sin[0].edge_off), (data[0].src, data[0].dst, data[0].edge_off)):
                    dst.copy_(src, non_blocking=True)
            else:
                data[0].expand(sin[1], out=sin[0])                  # LocalEdges -> int64 [2,E]
            if sin[5] is not None:
                sin[5].copy_tensors_(data[5])
        else:
            if sin.x is not None:
                sin.x.copy_(data.x, non_blocking=True)
            else:
                sin.x_compressed.copy_tensors_(data.x_compressed)
            if wl.kind == "node":
                if not big:
                    sin.hop_data.hop.copy_(data.hop_data.hop, non_blocking=True)
                sin.hop_data.level_counts.copy_(data.hop_data.level_counts, non_blocking=True)
            else:
                for f in ("hop", "hop_off", "node_off", "level_counts", "y"):
                    getattr(sin, f).copy_(getattr(data, f), non_blocking=True)

    def run_step(data):
        if graphed is None:
            out = step(widen(data))
            inputs_consumed.record()
            return out
        cap, sin = graphed
        if data is not sin:                                         # e2e leg: refresh the static inputs from the fresh copy
            g = refresh_graphs.get(id(data))
            if g is not None:
                g.replay()                                          # the ~20 small copy kernels as one launch
            else:
                refresh(data)
        inputs_consumed.record()                                    # the replay reads the static inputs only
        return cap()
    if graphed is not None:
        data_d = graphed[1]

    # ---- device-resident timing ---------------------------------------------------------------------------------------
    launches0 = lib.gnan_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier(); torch.cuda.synchronize()
    for a, b in ev:
        flush.fill_(1)                                              # evict L2 (126 MB) between timed steps
        a.record(); loss = run_step(data_d); b.record()
    torch.cuda.synchronize(); barrier()
    if dump_dir is not None and rank == 0:                          # before the passes below move the weights again
        named = list(model.named_parameters())
        dump_outputs(dump_dir, {"loss": loss, "output": last_out[0], **{f"grad.{k}": p.grad for k, p in named if p.grad is not None},
                                **{f"param.{k}": p for k, p in named}})
    launches = lib.gnan_launch_count() - launches0
    if graphed is not None:
        launches = launches_per_step * steps                        # replayed launches are not seen by the library's counter
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    # per-kernel / per-collective CUDA events live in the Python op wrappers, which a graph replay bypasses: an eager pass of
    # the same step (same process, same inputs, L2 flushed between steps) attributes the time
    n_attr = min(steps, 10)
    ops.enable_timing(True)
    for _ in range(n_attr):
        flush.fill_(1)
        step(data_d)
    kt = ops.timing_results()
    ops.enable_timing(False)
    per_step = {k: v[1] / n_attr for k, v in kt.items()}

    def timed_variant(setup, restore, in_data):
        """the same step under another model setting: eager per-kernel pass + (captured if possible) timed pass"""
        setup()
        for _ in range(3):
            step(in_data)
        ops.enable_timing(True)
        for _ in range(n_attr):
            flush.fill_(1)
            step(in_data)
        vkt = {k: v[1] / n_attr for k, v in ops.timing_results().items()}
        ops.enable_timing(False)
        run, mode = (lambda: step(in_data)), "eager"
        if graphed is not None:
            try:
                run, mode = CapturedStep(lambda: loss_of(in_data), opt, warmup=1, after_backward=after_bwd, zero_grad=zero_grads), "cuda graph"
            except Exception as exc:                                # pragma: no cover
                print(f"[bench] variant capture failed, timing it eagerly: {exc!r}", file=sys.stderr)
        vev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_attr)]
        for a, b in vev:
            flush.fill_(1)
            a.record(); run(); b.record()
        torch.cuda.synchronize()
        restore()
        return float(np.median([a.elapsed_time(b) for a, b in vev])), vkt, mode

    strict, dense = None, None
    if compare_legs and world == 1:
        if args.precision != "fp32":                                # the 1e-5 parity mode: FFMA kernels only
            ms_, kt_, mode_ = timed_variant(lambda: setattr(model, "precision", "fp32"), lambda: setattr(model, "precision", args.precision), data_d)
            strict = {"ms_per_step": ms_, "value": wl.units_per_step / (ms_ / 1e3), "unit": wl.unit, "kernel_ms_per_step": kt_, "mode": mode_,
                      "note": "same step with precision='fp32' (FFMA shape-function kernels only, every golden case within 1.5e-6 of the reference)"}
        if cx is not None and wl.kind == "node":                    # every (node, feature) pair evaluated: the regime of dropout training
            dense_in = SimpleNamespace(x=x_d, hop_data=data_d.hop_data, x_compressed=None)
            ms_, kt_, mode_ = timed_variant(lambda: setattr(model, "dedup", False), lambda: setattr(model, "dedup", True), dense_in)
            dflops = 2.0 * flops_per_eval(wl.C) * rows_local * wl.K
            dbwd = kt_.get("mlp_bwd", 0.0)
            dense = {"ms_per_step": ms_, "value": wl.units_per_step / (ms_ / 1e3), "unit": wl.unit, "mode": mode_, "kernel_ms_per_step": kt_,
                     "dominant_kernel": "mlp_tc_bwd_kernel" if args.precision != "fp32" else "mlp_bwd_kernel",
                     "dominant_kernel_tflops": dflops / (dbwd / 1e3) / 1e12 if dbwd > 0 else None,
                     "note": "--dedup off: all nodes x features evaluations executed (the regime of dropout training)"}
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / steps
    total_units = wl.units_per_step * (1 if (sharded or wl.name == "cora" and False) else world)
    value = total_units / (ms_per_step / 1e3)

    # ---- end to end from pinned host buffers ----------------------------------------------------------------------------
    # Every step's inputs are copied host -> device inside the timed region and its loss is read back; the copy of step i+1
    # is issued on a second stream before the host blocks on step i's loss, so PCIe transfers overlap the previous step's
    # kernels (double-buffered inputs; CUDA streams + events, no host-side prefetch outside the timed region).
    # The host side of a batch is ONE pinned buffer (packed.HostBundle): one cudaMemcpyAsync per step into one of two device
    # staging buffers; run_step then refreshes the captured step's static inputs from typed views of it (widening the compact
    # index types on the way).
    copy_stream = torch.cuda.Stream()
    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    bundle = HostBundle(host_parts)
    assert bundle.payload_bytes == h2d, (bundle.payload_bytes, h2d)
    stage_bufs = [bundle.device_buffer(dev) for _ in range(2)]
    staged = [assemble(bundle.views(b)) for b in stage_bufs]
    copies = [0]
    if graphed is not None:
        # the refresh of the static inputs from each of the two staging buffers is a CUDA graph of its own: one launch instead of
        # ~20 eager copy kernels whose host cost (~0.15 ms) exceeded a whole Mutagenicity-shaped step
        from gnan_b200.trainer import _no_gc_during_capture
        try:
            for d, buf in zip(staged, stage_bufs):
                bundle.copy_to(buf)                                 # real data: the refresh gathers through the staged index arrays
                refresh(d)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with _no_gc_during_capture(), torch.cuda.graph(g, capture_error_mode="thread_local" if world > 1 else "global"):
                    refresh(d)
                refresh_graphs[id(d)] = g
        except Exception as exc:                                    # pragma: no cover
            print(f"[bench] refresh capture failed, copying eagerly: {exc!r}", file=sys.stderr)
            refresh_graphs.clear()
            torch.cuda.synchronize()

    def issue_copy():
        k = copies[0] & 1
        copies[0] += 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(inputs_consumed)                 # staging buffer k was last read by the step before last
            bundle.copy_to(stage_bufs[k])
            e = torch.cuda.Event()
            e.record(copy_stream)
        return staged[k], e

    def e2e_loop(n):
        """Software pipeline of depth 2: while step i runs, the host has already issued the copy of step i+1 and reads the loss
        of step i-1 (its 4 bytes were copied to pinned host memory right behind that step; every step's loss is read)."""
        nxt = issue_copy()
        last, pending = 0.0, None
        for i in range(n):
            d, e = nxt
            torch.cuda.current_stream().wait_event(e)
            loss = run_step(d)
            hb, done = loss_host[i & 1], torch.cuda.Event()
            hb.copy_(loss.detach().reshape(1), non_blocking=True)   # device -> host read of this step's loss
            done.record()
            if i + 1 < n:
                nxt = issue_copy()                                  # overlaps this step's kernels
            if pending is not None:
                pending[1].synchronize()
                last = float(pending[0][0])
            pending = (hb, done)
            del d
        pending[1].synchronize()
        return float(pending[0][0])

    e2e_loop(3)
    barrier(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    e2e_loop(steps)
    b.record(); torch.cuda.synchronize(); barrier()
    t = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = total_units * steps / (float(t.item()) / 1e3)

    rec = None
    if rank == 0:
        hbm, tflops, peak_src = measured_peaks()
        if dense is not None and dense.get("dominant_kernel_tflops"):
            dense["dominant_kernel_frac_of_bf16_peak"] = dense["dominant_kernel_tflops"] / tflops
        # ---- roofline of the DOMINANT kernel of this step (largest CUDA-event time among the library's ops) ----------------
        kernels_only = {k: v for k, v in per_step.items() if k not in COLLECTIVES}
        dom = max(kernels_only, key=kernels_only.get) if kernels_only else "mlp_bwd"
        dur_ms = kernels_only.get(dom, 0.0)
        n_entries = None if cx is None else int(cx.num_entries)
        evals = rows_local * wl.K if cx is None else n_entries          # shape-function evaluations actually executed per pass
        pairs = float((wl.sizes.astype(np.float64) ** 2).sum()) if wl.kind == "graph" else float(rows_local) * wl.n
        prof = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        traffic = json.load(open(prof)).get(f"{wl.name}:{dom}:{args.precision}") if os.path.exists(prof) else None

        def hbm_roof(op, alg_bytes, what):
            d = per_step.get(op, 0.0)
            ach = alg_bytes / (d / 1e3) / 1e9 if d > 0 else 0.0
            return {"kernel": KERNEL_NAMES.get(op, op), "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                    "traffic": json.load(open(prof)).get(f"{wl.name}:{op}:{args.precision}") if os.path.exists(prof) else None,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "algorithmic_bytes": what, "avg_launch_ms": d}
        if dom.startswith("mlp"):
            # backward = 2x the forward FLOPs; recompute and padded tile rows are not counted (SURVEY.md §8d: with shared
            # evaluations the count is the evaluations actually executed)
            alg = (2.0 if "bwd" in dom else 1.0) * flops_per_eval(wl.C) * evals
            achieved = alg / (dur_ms / 1e3) / 1e12 if dur_ms > 0 else 0.0
            roof = {"kernel": KERNEL_NAMES.get(dom, dom), "bound": "tensor", "achieved": achieved, "peak": tflops, "unit": "TFLOP/s",
                    "frac": achieved / tflops, "traffic": traffic, "peak_source": peak_src, "algorithmic_flops_per_launch": alg,
                    "evaluations_per_launch": evals, "avg_launch_ms": dur_ms}
        elif dom == "aggregate_rows_bwd_saved":
            roof = hbm_roof(dom, float(n_train_local) * wl.n, "1 hop byte per (row with a loss, column): rows whose output gradient is zero are skipped")
        elif dom == "apsp_bfs_batched":
            # the kernel's outputs: the hop blocks and the fixed-width normaliser table (fp32 [nodes, MOL_NBINS], written in full)
            roof = hbm_roof(dom, pairs + 4.0 * wl.n * MOL_NBINS, "1 hop byte written per ordered pair + 4 bytes per (node, level) of the "
                            + ("pair-statistics" if pair_stats else "normaliser") + f" table ({MOL_NBINS} levels)")
        elif dom == "build_csr":
            roof = hbm_roof(dom, 16.0 * wl.edge_index.shape[1], "16 bytes read per edge")
        elif dom == "aggregate_blockdiag_fwd" and in_step_apsp:
            roof = hbm_roof(dom, pairs + 4.0 * wl.n * MOL_NBINS, "1 hop byte read per ordered pair + 4 bytes per (node, level) of the normaliser "
                            "table; the backward reads neither (it reuses the forward's pair statistics)")
        else:
            roof = hbm_roof(dom, pairs, "1 hop byte per ordered pair per pass (SURVEY.md §8d)")
        roof["kernel_ms_per_step"] = per_step
        agg = None
        if wl.kind == "node":           # the hop-matrix passes of this step against the HBM roofline, whatever the dominant kernel is
            fwd = hbm_roof("aggregate_rows_fwd_save", pairs, "1 hop byte per ordered pair")
            if wl.C >= 2 and fwd["avg_launch_ms"] > 0:
                # tensor-core form (csrc/agg_tc.cu): every hop byte expands to NB one-hot int8 values contracted against NP digit
                # columns of S; with many channels the int8 tensor pipe, not HBM, bounds the pass. Peak = 2x the measured bf16 rate.
                nbv = int(hd.nbins)
                nb_lanes = 8 if nbv <= 8 else (16 if nbv <= 16 else 32)
                c4, c5 = -(-wl.C // 4), -(-wl.C // 5)
                np_cols = 16 * c4 if c4 == c5 else 16 * c5
                ops_exec = 2.0 * pairs * nb_lanes * np_cols
                ach = ops_exec / (fwd["avg_launch_ms"] / 1e3) / 1e12
                fwd["tensor_view"] = {"bound": "tensor (int8)", "executed_ops_per_launch": ops_exec, "achieved": ach, "unit": "TOP/s",
                                      "peak": 2.0 * tflops, "frac": ach / (2.0 * tflops), "lanes_per_row": nb_lanes, "digit_columns": np_cols,
                                      "note": "executed one-hot int8 MACs (not algorithmic FLOPs); see profiles/ for the ncu tensor-pipe utilisation"}
            agg = {"forward": fwd,
                   "backward": hbm_roof("aggregate_rows_bwd_saved", float(n_train_local) * wl.n,
                                        "1 hop byte per (row with a loss, column); rows with zero output gradient are skipped"),
                   "rows_with_loss": n_train_local, "hop_bytes": pairs}
        rec = {
            "metric": f"GNAN fwd+bwd {wl.unit} ({wl.name}-shape TensorGNAN)", "value": value, "unit": wl.unit, "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32x3": "f32 (shape-function hidden layers as 3xTF32 split on tcgen05, fp32 accumulate; aggregation: exact int32 "
                      "accumulation of 8-bit digits of S on tcgen05 kind::i8)", "tf32": "tf32"}[args.precision],
            "data": "synthetic", "config": dict(workload_config(wl, "gpu", world), **({"edge_input": (
                "LocalEdges (uint8 endpoints inside their graph + per-graph edge offsets): the BFS kernel builds each graph's adjacency itself"
                + (" and accumulates the pair statistics of the graph readout (undirected graphs)" if pair_stats else "")
                if local_edges else "int64 [2,E] edge_index: gnan_build_csr + BFS")} if in_step_apsp else {})),
            "e2e": {"value": e2e_val, "unit": wl.unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": steps,
                    "note": "hop matrix kept device-resident in the e2e leg (too large to stage in pinned host memory)" if (wl.kind == "node" and big) else None},
            "gpu_launches": int(launches), "cuda_graph": graphed is not None,
            "roofline": roof, "aggregation": agg, "strict_fp32": strict, "dense_kernels": dense,
            "dedup": None if cx is None else {
                "entries": n_entries, "dense_evaluations": rows_local * wl.K, "exception_density": cx.density(),
                "note": "rows with equal values in a feature column share one shape-function evaluation (exact; dropout is 0 here); "
                        "the compressed form is built once per dataset like the hop matrix. --dedup off runs the dense kernels"},
        }
        if world > 1:
            rec["collectives_ms_per_step"] = {k: per_step.get(k, 0.0) for k in COLLECTIVES if k in per_step}
            rec["collectives_note"] = "CUDA-event time of each collective in an eager pass of the step on rank 0 (includes waiting for the slowest rank)"
        if not args.no_cpu_baseline and world == 1:
            rec["cpu_baseline"] = cpu_baseline_record(wl, cpu_budget_s)
    # release this workload's memory before the next one
    del graphed, data_d, model, opt
    import gc
    gc.collect(); torch.cuda.empty_cache()
    return rec


# ---------------------------------------------------------------------------------------------------------------------
# multi-GPU results against the single-GPU computation of the same problem (the 2-GPU pytest is skipped on 1-GPU boxes)
# ---------------------------------------------------------------------------------------------------------------------
def parity_vs_single_gpu(env):
    import torch.distributed as dist
    from gnan_b200 import dist as gdist
    from gnan_b200.preprocess import apsp, apsp_batched
    world, rank, dev = env.world, env.rank, env.dev
    rel = lambda a, c: float((a.double() - c.double()).norm() / c.double().norm().clamp_min(1e-300))
    out = {}
    # (1) row-sharded node task vs one GPU holding all rows
    from gnan_b200.GNAN import TensorGNAN
    rng = np.random.default_rng(5)
    n, K, C = 4000, 24, 5
    ei = random_simple_graph(rng, n, 7000, 30)
    x = torch.tensor(rng.normal(size=(n, K))).float().to(dev)
    w = torch.tensor(rng.normal(size=(n, C))).float().to(dev)
    w[torch.tensor(rng.random(n) > 0.05).to(dev)] = 0.0                # a 5 % "train mask"
    torch.manual_seed(1)
    m = TensorGNAN(K, C, L, H, normalize_rho=True, device=dev).to(dev)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    gdist.broadcast_parameters(m)
    full = m(SimpleNamespace(x=x, hop_data=apsp(torch.tensor(ei), n, device=dev)))
    (full * w).sum().backward()
    g_full = [p.grad.clone() for p in m.parameters()]
    fg = gdist.FlatGradients(m.parameters())
    fg.zero()
    blocks = [gdist.row_block(n, r, world) for r in range(world)]
    b, e = blocks[rank]
    hd = apsp(torch.tensor(ei), n, device=dev, row_begin=b, row_end=e)
    o = gdist.row_sharded_forward(m, x[b:e].contiguous(), hd, [q - p for p, q in blocks])
    (o * w[b:e]).sum().backward()
    fg.all_reduce()
    per = {k: rel(p.grad, g) for (k, p), g in zip(m.named_parameters(), g_full)}
    worst = max(per, key=per.get)
    errs = torch.tensor([rel(o, full[b:e].detach()) if e > b else 0.0, per[worst]], device=dev, dtype=torch.float64)
    dist.all_reduce(errs, op=dist.ReduceOp.MAX)
    out["row_sharded"] = {"nodes": n, "out_rel_err": float(errs[0]), "max_param_grad_rel_err": float(errs[1]), "worst_param_rank0": worst}
    # (2) data-parallel graph batches vs one GPU holding the union batch
    from gnan_b200.models import TensorGNAN as GraphGNAN
    torch.manual_seed(2)
    gm = GraphGNAN(15, 1, L, H, normalize_rho=True, is_graph_task=True, readout_n_layers=0, device=dev).to(dev)
    gm.fs.xavier_normal_(1.0); gm.rho.xavier_normal_(1.0)
    gdist.broadcast_parameters(gm)
    loss_fn = torch.nn.BCEWithLogitsLoss()
    wls = [make_mol_workload(seed=100 + r, n_graphs=256) for r in range(world)]

    def loss_on(wl_list):
        off, eis, xs, ys, noffs = 0, [], [], [], [np.zeros(1, np.int64)]
        for wl in wl_list:
            eis.append(wl.edge_index + off); xs.append(wl.x); ys.append(wl.y); noffs.append(wl.node_off.numpy()[1:] + off)
            off += wl.n
        pk = apsp_batched(torch.cat(eis, 1), np.concatenate(noffs), device=dev, x=torch.cat(xs).to(dev), y=torch.cat(ys).to(dev))
        return loss_fn(gm(pk).flatten(), pk.y)
    gm.zero_grad(set_to_none=True)
    loss_on(wls).backward()
    g_union = [p.grad.clone() for p in gm.parameters()]
    fg2 = gdist.FlatGradients(gm.parameters())
    fg2.zero()
    loss_on([wls[rank]]).backward()
    fg2.all_reduce(average=True)
    err = torch.tensor([max(rel(p.grad, g) for p, g in zip(gm.parameters(), g_union))], device=dev, dtype=torch.float64)
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    out["data_parallel"] = {"graphs_per_rank": 256, "max_param_grad_rel_err": float(err[0])}
    out["note"] = "max over ranks; the single-GPU result is computed on every rank from the same seeded problem"
    return out


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="gnan_b200", choices=["gnan_b200", "reference"])
    ap.add_argument("--pair-stats", action="store_true",
                    help="molecule workload with --edge-format local: the BFS accumulates the readout's pair statistics itself and the model "
                         "skips the hop-byte pass (measured a tie on B200: +0.13 ms in the BFS, -0.14 ms in the readout; off by default)")
    ap.add_argument("--edge-format", default="local", choices=["local", "int64"],
                    help="molecule workload: the step's edge-list input (LocalEdges transfer form, or PyG's int64 edge_index)")
    ap.add_argument("--workload", default=None, choices=["mol", "mutag", "cora", "pubmed", "arxiv"],
                    help="one workload only; default: headline = mol plus sub-records for the other BASELINE configs")
    ap.add_argument("--classes", type=int, default=0, help="override the number of classes (arxiv: 40, or 1 = the reference's hard-coded value)")
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32x3", "tf32"])
    ap.add_argument("--dedup", default="on", choices=["on", "off"],
                    help="share shape-function evaluations between rows with equal feature values (gnan_b200.sparse; exact, dropout is 0 here)")
    ap.add_argument("--headline-only", action="store_true", help="no sub-records and no comparison legs (used for the ncu launch list)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true", help="run the step eagerly instead of replaying a captured CUDA graph")
    ap.add_argument("--subs", default=None, help="comma-separated sub-record workloads (default: cora,mutag,pubmed,arxiv at N=1; arxiv at N>1)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps of the headline workload, write what its last timed step computed (loss, model output, "
                         "parameter gradients, updated parameters) as DIR/<name>.npy; arrays over 1 Mi elements as a fixed seeded sample; "
                         "with row-sharded ranks, the output is rank 0's rows, as row_sharded_forward returns them there")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from gnan_b200 import _lib
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    env = SimpleNamespace(world=world, rank=rank, dev=dev, flush=torch.empty(256 << 20, dtype=torch.uint8, device=dev), lib=_lib.load())
    clk = clocks_sampler() if rank == 0 else None                  # sampled over the whole run (all under load)

    primary = args.workload or "mol"
    line = run_workload(args, env, primary, steps=args.steps, warmup=args.warmup, classes=args.classes,
                        compare_legs=(primary == "cora" and not args.headline_only), cpu_budget_s=90.0, dump_dir=args.dump_outputs)
    subs, parity = {}, None
    if args.workload is None and not args.headline_only:
        names = (args.subs.split(",") if args.subs else (["cora", "mutag", "pubmed", "arxiv"] if world == 1 else ["arxiv"]))
        for nm in [n for n in names if n]:
            try:
                subs[nm] = run_workload(args, env, nm, steps=args.steps, warmup=3, compare_legs=(nm == "cora"), cpu_budget_s=45.0)
            except Exception as exc:                                # pragma: no cover
                print(f"[bench] sub-record {nm} failed: {exc!r}", file=sys.stderr)
                subs[nm] = {"error": repr(exc)}
                torch.cuda.synchronize()
        if world > 1:
            try:
                parity = parity_vs_single_gpu(env)
            except Exception as exc:                                # pragma: no cover
                print(f"[bench] parity_vs_single_gpu failed: {exc!r}", file=sys.stderr)
                parity = {"error": repr(exc)}
    clocks = clocks_summary(clk)
    if rank == 0:
        line["clocks"] = clocks
        if subs:
            line["sub_records"] = subs
            line["sub_records_note"] = ("the other BASELINE.json configs measured in the same process, same rules (device-timed value, e2e from "
                                        "host buffers, roofline of the dominant kernel); at N > 1 node tasks are row-sharded (strong scaling)")
        if parity is not None:
            line["parity_vs_single_gpu"] = parity
        print(json.dumps(line), flush=True)
    if world > 1:
        # captured graphs holding NCCL work were released with each workload (run_workload frees them); tear the group down with a
        # watchdog so that a communicator that still refuses to finalise cannot hang the job after the line is out
        import threading
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        threading.Timer(30.0, lambda: os._exit(0)).start()
        dist.destroy_process_group()
        os._exit(0)


if __name__ == "__main__":
    main()
