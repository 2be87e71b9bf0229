"""Training step on batches with graphs of more than 128 nodes, preprocessed inside the step. Needs a GPU.

    python tests/tools/bench_deferred_large.py [--out profiles/deferred_large_b200.json] [--reps 30]

Workloads (tests/tools/bench_apsp_large.py's synthetic graphs: random tree + n/10 extra edges, both directions, 14 one-hot features):
  mutagenicity_shaped  4 337 graphs, bench.py's molecule size draw plus a tail of 20 graphs of 257..417 nodes, as one batch;
  proteins_shaped      1 113 graphs, lognormal sizes of 4..256 nodes plus 12 of 257..620, as one batch;
and each without its graphs of more than 128 nodes, which prices them. models.TensorGNAN (K = 14, C = 1, normalize_rho, nbins = 48) takes a step of
forward, fused BCE loss, backward and Adam(capturable), captured in a CUDA graph (trainer.CapturedStep). Three ways to get the
distances inside the step:
  (a) deferred: apsp_batched(LocalEdges int16, nbins, rscale=True); the BFS and the readout are one kernel per size class;
  (b) rscale:   apsp_batched(int64 edge_index, nbins, rscale=True) (CSR, BFS writing hop bytes + 1/count), then the one-pass readout;
  (c) counts:   apsp_batched(int64 edge_index, nbins) (CSR, BFS writing hop bytes + int32 counts), level_rscale, one-pass readout;
(c) is the only one that took such batches before the fused kernel went past 128 nodes. CUDA events around each replay, with
a 256 MB buffer overwritten between replays so that no step finds the last one's data in L2; median and spread over --reps.
Kernel times come from torch.profiler in a separate run. Bytes per step: the edge list in each transfer width (uint8 only where
every graph has at most 256 nodes) and as int64. The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
sys.path.insert(0, ROOT)

from tests.test_gpu_batched_large_graphs import molecule_like_graphs, mutagenicity_sizes  # noqa: E402
from tests.tools.bench_apsp_large import packed_inputs, proteins_sizes  # noqa: E402

DEV = "cuda"
NBINS = 48


def make_step(mode, graphs):
    from gnan_b200 import ops, trainer
    from gnan_b200.models import TensorGNAN
    from gnan_b200.preprocess import LocalEdges, apsp_batched
    ei, node_off, sizes = packed_inputs(graphs)
    x = torch.cat([g.x for g in graphs]).to(DEV)
    y = torch.cat([g.y for g in graphs]).to(DEV)
    no_d = torch.tensor(node_off, dtype=torch.int32, device=DEV)
    ho_d = torch.tensor(np.concatenate([[0], np.cumsum(sizes.astype(np.int64) ** 2)]), dtype=torch.int64, device=DEV)
    le = LocalEdges.from_edge_index(ei, node_off, dtype=torch.int16).to(DEV)
    eid = ei.to(DEV)
    torch.manual_seed(0)
    m = TensorGNAN(x.shape[1], 1, 3, 64, normalize_rho=True, is_graph_task=True, readout_n_layers=0, device=DEV).to(DEV)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, capturable=True)

    def closure():
        if mode == "deferred":
            pk = apsp_batched(le, node_off, device=DEV, x=x, y=y, node_off_device=no_d, hop_off_device=ho_d, nbins=NBINS, rscale=True)
        elif mode == "rscale":
            pk = apsp_batched(eid, node_off, device=DEV, x=x, y=y, node_off_device=no_d, hop_off_device=ho_d, nbins=NBINS, rscale=True)
        else:
            pk = apsp_batched(eid, node_off, device=DEV, x=x, y=y, node_off_device=no_d, hop_off_device=ho_d, nbins=NBINS)
        return ops.bce_with_logits(m(pk).flatten(), pk.y)
    return trainer.CapturedStep(closure, opt, warmup=2), closure


def time_steps(step, reps):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for _ in range(3):
        step()
    for a, b in ev:
        flush.fill_(1)
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    t = np.array([a.elapsed_time(b) for a, b in ev])
    return {"median_ms": float(np.median(t)), "min_ms": float(t.min()), "max_ms": float(t.max())}


def kernel_times(step):
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0))
        for key in ("bfs_readout_large_kernel", "apsp_batched_v3_kernel", "apsp_batched_large_kernel", "agg_bd_graph_fwd",
                    "build_csr", "level_rscale"):
            if key in e.key and t > 0:
                out[key] = out.get(key, 0.0) + t / 1000.0
    return out


def transfer_bytes(graphs):
    from gnan_b200.preprocess import LocalEdges
    ei, node_off, sizes = packed_inputs(graphs)
    r = {"edges": int(ei.shape[1]), "int64_edge_index": int(ei.numel() * 8),
         "int16": LocalEdges.from_edge_index(ei, node_off, dtype=torch.int16).nbytes()}
    r["uint8"] = LocalEdges.from_edge_index(ei, node_off).nbytes() if sizes.max() <= 256 else None
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_deferred_large needs a GPU"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
    res = {"card": card, "nbins": NBINS, "reps": args.reps}
    rng = np.random.default_rng(0)
    sets = {"mutagenicity_shaped": molecule_like_graphs(rng, mutagenicity_sizes(rng)),
            "proteins_shaped": molecule_like_graphs(rng, proteins_sizes(rng))}
    for name, graphs in sets.items():
        small = [g for g in graphs if g.x.shape[0] <= 128]
        for tag, gs in ((name, graphs), (name + "_at_most_128_nodes", small)):
            sizes = np.array([g.x.shape[0] for g in gs])
            r = {"graphs": len(gs), "nodes": int(sizes.sum()), "max_nodes": int(sizes.max()), "graphs_over_128": int((sizes > 128).sum()),
                 "bytes_per_step": transfer_bytes(gs)}
            losses = {}
            for mode in ("deferred", "rscale", "counts"):
                step, _ = make_step(mode, gs)
                losses[mode] = float(step())
                r[mode] = time_steps(step, args.reps)
                r[mode]["kernels_ms_profiler"] = kernel_times(step)
            r["first_replay_losses"] = losses
            res[tag] = r
            print(tag, json.dumps(r), flush=True)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
