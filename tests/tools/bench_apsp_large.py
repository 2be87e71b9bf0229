"""Batched BFS on datasets with graphs of more than 128 nodes (apsp_batched_large_kernel). Needs a GPU.

    python tests/tools/bench_apsp_large.py [--out result.json] [--reps 20]

(a) PackedDataset.from_graphs against the per-graph `apsp` loop of preprocess.pre_process, on a Mutagenicity-shaped set (4337 graphs,
    bench.py's sizes plus a tail of 20 graphs of 257..417 nodes) and a PROTEINS-shaped one (1113 graphs, mean about 39 nodes, tail to
    620). Host clock around work that ends in a device synchronise; one warm-up call each first.
(b) the Mutagenicity-shaped batch in the fixed-width mode (nbins=64, no host synchronisation) with and without its tail: CUDA events
    over --reps calls; the difference is about the large-graph kernel's own time, which torch.profiler also reports in a separate run.
(c) 1000 graphs of 257..1024 nodes: graphs/s and GB/s of hop bytes written (fixed-width mode, CUDA events).
(d) batches whose largest graph has 129..256 nodes: d1 = 4000 molecule-like graphs of 129..256 nodes (about 150 MB of hop bytes,
    more than L2), d2 = the PROTEINS-shaped size draw without its tail (4..256 nodes) four times over. Fixed-width calls (nbins=64,
    CUDA events, three windows of --reps calls) and PackedDataset.from_graphs (host clock), each also with one extra edgeless
    257-node graph appended, and that graph alone. The extra graph costs one CTA of the large kernel, three chunks of one level.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
sys.path.insert(0, ROOT)

from tests.test_gpu_batched_large_graphs import molecule_like_graphs, mutagenicity_sizes  # noqa: E402

DEV = "cuda"


def proteins_sizes(rng, n_graphs=1113, n_tail=12):
    sizes = np.clip(np.round(rng.lognormal(3.4, 0.6, size=n_graphs)), 4, 256).astype(np.int64)
    if n_tail:
        sizes[-n_tail:] = rng.integers(257, 621, size=n_tail)
        sizes[-1] = 620
    return sizes


def packed_inputs(graphs):
    sizes = np.array([int(g.x.shape[0]) for g in graphs], dtype=np.int64)
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    ei = torch.cat([g.edge_index + int(node_off[i]) for i, g in enumerate(graphs)], dim=1)
    return ei, node_off, sizes


def host_time(fn, reps=1):
    fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best


def event_time_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def kernel_time_ms(fn, name):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = 0.0
    for e in prof.key_averages():
        if name in e.key:
            tot += getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0))
    return tot / 1000.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_apsp_large needs a GPU"
    from gnan_b200.packed import PackedDataset
    from gnan_b200.preprocess import apsp, apsp_batched, check_batched_status
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
    res = {"card": card}

    rng = np.random.default_rng(0)
    sets = {"mutagenicity_shaped": molecule_like_graphs(rng, mutagenicity_sizes(rng)),
            "proteins_shaped": molecule_like_graphs(rng, proteins_sizes(rng))}
    for name, graphs in sets.items():
        ei, node_off, sizes = packed_inputs(graphs)
        t_packed = host_time(lambda: PackedDataset.from_graphs(graphs, device=DEV), reps=3)

        def per_graph():
            for g in graphs:
                apsp(g.edge_index, int(g.x.shape[0]), device=DEV)
        t_loop = host_time(per_graph)
        ds = PackedDataset.from_graphs(graphs, device=DEV)
        res[name] = {"graphs": len(graphs), "mean_nodes": float(sizes.mean()), "max_nodes": int(sizes.max()),
                     "graphs_over_256": int((sizes > 256).sum()), "nbins": ds.nbins,
                     "from_graphs_s": t_packed, "per_graph_apsp_loop_s": t_loop, "speedup": t_loop / t_packed}
        print(name, res[name], flush=True)

    # (b) with and without the large tail, fixed-width mode
    graphs = sets["mutagenicity_shaped"]
    ei, node_off, sizes = packed_inputs(graphs)
    small = [g for g in graphs if g.x.shape[0] <= 256]
    ei_s, node_off_s, sizes_s = packed_inputs(small)
    nb = 64
    eid, eid_s = ei.to(DEV), ei_s.to(DEV)
    pk = apsp_batched(eid, node_off, device=DEV, nbins=nb)
    check_batched_status(pk.status)
    t_all = event_time_ms(lambda: apsp_batched(eid, node_off, device=DEV, nbins=nb), args.reps)
    t_small = event_time_ms(lambda: apsp_batched(eid_s, node_off_s, device=DEV, nbins=nb), args.reps)
    k_large = kernel_time_ms(lambda: apsp_batched(eid, node_off, device=DEV, nbins=nb), "apsp_batched_large_kernel")
    tail_pairs = int((sizes[sizes > 256] ** 2).sum())
    res["tail_of_mutagenicity_shaped"] = {"nbins": nb, "call_ms_with_tail": t_all, "call_ms_without_tail": t_small,
                                          "difference_ms": t_all - t_small, "large_kernel_ms_profiler": k_large,
                                          "tail_pairs": tail_pairs, "large_kernel_pairs_per_s": tail_pairs / (k_large / 1e3) if k_large else None}
    print(res["tail_of_mutagenicity_shaped"], flush=True)

    # (c) 1000 graphs of 257..1024 nodes
    rng = np.random.default_rng(1)
    big = molecule_like_graphs(rng, rng.integers(257, 1025, size=1000))
    ei_b, node_off_b, sizes_b = packed_inputs(big)
    eid_b = ei_b.to(DEV)
    pk = apsp_batched(eid_b, node_off_b, device=DEV, nbins=nb)
    check_batched_status(pk.status)
    reps_c = max(3, args.reps // 4)
    t_big = event_time_ms(lambda: apsp_batched(eid_b, node_off_b, device=DEV, nbins=nb), reps_c)
    k_big = kernel_time_ms(lambda: apsp_batched(eid_b, node_off_b, device=DEV, nbins=nb), "apsp_batched_large_kernel")
    hop_bytes = int((sizes_b ** 2).sum())
    res["large_graphs_1000"] = {"nbins": nb, "mean_nodes": float(sizes_b.mean()), "hop_bytes": hop_bytes, "call_ms": t_big,
                                "graphs_per_s": 1000 / (t_big / 1e3), "hop_GB_per_s_call": hop_bytes / (t_big / 1e3) / 1e9,
                                "large_kernel_ms_profiler": k_big,
                                "hop_GB_per_s_kernel": hop_bytes / (k_big / 1e3) / 1e9 if k_big else None}
    print(res["large_graphs_1000"], flush=True)

    # (d) largest graph of 129..256 nodes, alone and with one edgeless 257-node graph
    rng = np.random.default_rng(2)
    mid = {"d1_129_to_256": molecule_like_graphs(rng, rng.integers(129, 257, size=4000)),
           "d2_proteins_shaped_no_tail_x4": molecule_like_graphs(rng, np.tile(proteins_sizes(rng, n_tail=0), 4))}
    extra = SimpleNamespace(x=torch.zeros(257, 14), edge_index=torch.zeros(2, 0, dtype=torch.int64), y=torch.tensor([0.0]))
    for name, graphs in mid.items():
        r = {}
        for key, gs in (("", graphs), ("_plus_257", graphs + [extra]), ("_257_alone", [extra])):
            ei, node_off, sizes = packed_inputs(gs)
            eid = ei.to(DEV)
            pk = apsp_batched(eid, node_off, device=DEV, nbins=nb)
            check_batched_status(pk.status)
            r["graphs" + key] = len(gs)
            r["hop_bytes" + key] = int((sizes ** 2).sum())
            r["call_ms" + key] = [event_time_ms(lambda: apsp_batched(eid, node_off, device=DEV, nbins=nb), args.reps) for _ in range(3)]
            r["bfs_kernels_ms_profiler" + key] = kernel_time_ms(lambda: apsp_batched(eid, node_off, device=DEV, nbins=nb), "apsp_batched_")
            r["from_graphs_s" + key] = host_time(lambda: PackedDataset.from_graphs(gs, device=DEV), reps=3)
        res[name] = r
        print(name, r, flush=True)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
