"""Measurement of gnan_b200.interpret.explain on bench.py's workloads: per-kernel time (CUDA events around each launch, ops timing
labels explain_*), the whole call, exception lookups per second and output bytes per second.

    python tests/tools/bench_explain.py [--out profiles/explain_b200.json] [--iters 5]

Workloads: the Cora shape (all 2 708 rows), the PubMed shape (all 19 717 rows), the 32 768-graph molecule batch (deferred: the
fused BFS + readout supplies colw) and the 4 337-graph Mutagenicity-shaped batch. Two untimed calls warm every shape up. The L2 is
overwritten (a 256 MB fill) before every timed call, so each call starts from HBM. The card name and power limit are read in the
same process."""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..")
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from gnan_b200 import interpret, ops  # noqa: E402

DEV = "cuda"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


def node_workload(name):
    from gnan_b200.GNAN import TensorGNAN
    from gnan_b200.preprocess import apsp
    wl = bench.make_node_workload(name)
    torch.manual_seed(0)
    m = TensorGNAN(wl.K, wl.C, bench.L, bench.H, normalize_rho=True, is_graph_task=False, device=DEV).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    inputs = SimpleNamespace(x=wl.x.to(DEV), hop_data=apsp(wl.edge_index, wl.n, device=DEV))
    return m, inputs, wl


def graph_workload(name):
    from gnan_b200.models import TensorGNAN
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    wl = bench.make_mol_workload() if name == "mol" else bench.make_graph_workload()
    torch.manual_seed(0)
    m = TensorGNAN(wl.K, wl.C, bench.L, bench.H, normalize_rho=True, is_graph_task=True, readout_n_layers=0, device=DEV).to(DEV)
    m.fs.xavier_normal_(1.0); m.rho.xavier_normal_(1.0)
    node_off = wl.node_off.numpy()
    if name == "mol":
        pk = apsp_batched(LocalEdges.from_edge_index(wl.edge_index, node_off), node_off, device=DEV, x=wl.x.to(DEV),
                          nbins=bench.MOL_NBINS, rscale=True)
        assert pk.deferred
    else:
        pk = apsp_batched(wl.edge_index, node_off, device=DEV, x=wl.x.to(DEV))
    return m, pk, wl


def lookups(inputs, graph, e):
    """(row, exception) pairs the kernel visits: node rows x exceptions of the graph; graph rows: every exception once"""
    from gnan_b200.sparse import compress_features
    x = inputs.x
    cx = compress_features(x, max_density=None)
    n_exc = cx.num_entries - cx.num_features
    return n_exc if graph else e.features.shape[0] * n_exc


def run(name, iters):
    graph = name in ("mol", "mutag")
    m, inputs, wl = graph_workload(name) if graph else node_workload(name)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    for _ in range(2):
        e = interpret.explain(m, inputs)
    torch.cuda.synchronize()
    ops.enable_timing(True)
    total = 0.0
    for _ in range(iters):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e = interpret.explain(m, inputs)
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    kernels = {k: {"calls_per_explain": v[0] / iters, "ms_per_explain": v[1] / iters} for k, v in ops.timing_results().items()}
    ops.enable_timing(False)
    lk = lookups(inputs, graph, e)
    kname = "explain_graph_features" if graph else "explain_rows_features"
    kms = kernels[kname]["ms_per_explain"]
    out_bytes = e.features.numel() * 4
    return {"workload": name, "rows": int(e.features.shape[0]), "K": int(e.features.shape[1]), "C": int(e.features.shape[2]),
            "explain_ms": total / iters, "kernels": kernels, "feature_kernel": kname, "exception_lookups": int(lk),
            "lookups_per_s": lk / (kms * 1e-3), "output_bytes": out_bytes, "output_bytes_per_s": out_bytes / (kms * 1e-3),
            "max_abs_sum_minus_out": float((e.features.double().sum(1) - e.out.double()).abs().max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("workloads", nargs="*", default=["cora", "pubmed", "mol", "mutag"])
    args = ap.parse_args()
    res = {"card": card(), "l2_flushed": True, "warmup_calls": 2, "iters": args.iters, "results": []}
    for w in args.workloads:
        r = run(w, args.iters)
        print(json.dumps(r), flush=True)
        res["results"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
