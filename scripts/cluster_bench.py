"""Device graph partitioner and ClusterLoader (dgg_b200.samplers.partition / ClusterData / ClusterLoader): partition
time, cut fraction, coarse levels and largest part against the cap, and ms per ClusterLoader batch, at

  pubmed  N = 19 717, 44 324 undirected edges (bench.chung_lu_graph with Pubmed's sizes), 64 parts
  reddit  N = 232 965, 114 615 892 edges generated on the device, 1 500 parts (PyG's Cluster-GCN Reddit setting)

ClusterLoader batches draw batch_size = 20 shuffled parts.  Reddit-shape edges are random (source, target) pairs with
targets within 3 000 ids of the source, from a fixed seed; only the sizes follow the dataset.  Timing: host clock
around work that ends in a device synchronise (the partitioner reads a few values per level back to the host), after
one warm-up call of the same shape.  For context it also times the NumPy restatement (tests/cluster_ref.py) on the
Pubmed-shape partition on the host cores and checks that the GPU result equals it.  Prints the card name and power
limit with the numbers; --out also writes them as JSON.

    python scripts/cluster_bench.py [--batches 50] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from scripts.neighbor_sample_bench import card  # noqa: E402


def _pubmed():
    import bench

    idx, _ = bench.chung_lu_graph(19717, 4.5, 171, seed=0)
    return idx.cuda(), 19717


def _reddit(e=114615892):
    n = 232965
    gen = torch.Generator(device="cuda").manual_seed(0)
    ei = torch.randint(0, n, (2, e), generator=gen, device="cuda")
    ei[1] = (ei[0] + torch.randint(-3000, 3000, (e,), generator=gen, device="cuda")).clamp_(0, n - 1)
    return ei, n


def run_shape(name, ei, n, k, batches):
    from dgg_b200 import samplers

    samplers._partition_parts(ei, n, k, ei.device)            # warm-up: module load, allocator, sort plans
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    part, levels = samplers._partition_parts(ei, n, k, ei.device)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    perm, partptr = samplers.partition(ei, k, num_nodes=n)
    torch.cuda.synchronize()
    dt_full = time.perf_counter() - t0
    u, v = ei[0], ei[1]
    keep = u != v
    cut = int((part[u[keep]] != part[v[keep]]).sum())
    sizes = partptr[1:] - partptr[:-1]
    data = samplers.SubgraphBatch(edge_index=ei, num_nodes=n)
    cd = samplers.ClusterData(data, num_parts=k, log=False)
    loader = samplers.ClusterLoader(cd, batch_size=20, shuffle=True)
    torch.manual_seed(0)
    it = iter(loader)
    next(it)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    done = edges = 0
    while done < batches:
        try:
            b = next(it)
        except StopIteration:
            it = iter(loader)
            continue
        edges += b.num_edges
        done += 1
    torch.cuda.synchronize()
    dtb = time.perf_counter() - t0
    return perm, partptr, dict(shape=name, n=n, e=int(ei.shape[1]), num_parts=k, partition_ms=1e3 * dt,
                               partition_with_perm_ms=1e3 * dt_full, levels=levels,
                               cut_fraction_of_directed_edges=cut / max(1, int(keep.sum())),
                               max_part=int(sizes.max()), min_part=int(sizes.min()),
                               cap=(103 * n + 100 * k - 1) // (100 * k), loader_batch_size=20,
                               loader_ms_per_batch=1e3 * dtb / batches, loader_edges_per_batch=edges / batches)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batches", type=int, default=50)
    ap.add_argument("--shapes", default="pubmed,reddit")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cluster_bench.py measures the GPU partitioner: no CUDA device")
    result = dict(card=card(), shapes=[])
    for name in a.shapes.split(","):
        if name == "pubmed":
            ei, n = _pubmed()
            perm, partptr, r = run_shape(name, ei, n, 64, a.batches)
            from tests import cluster_ref as R

            t0 = time.perf_counter()
            want = R.partition(ei.cpu().numpy(), n, 64)
            r.update(restatement_ms=1e3 * (time.perf_counter() - t0), host_cpus=os.cpu_count(),
                     gpu_equals_restatement=bool(np.array_equal(perm.cpu().numpy(), want[0])
                                                 and np.array_equal(partptr.cpu().numpy(), want[1])))
        else:
            ei, n = _reddit()
            perm, partptr, r = run_shape(name, ei, n, 1500, a.batches)
        result["shapes"].append(r)
        print(json.dumps(dict(card=result["card"], **r)), flush=True)
        del ei, perm, partptr
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    if not all(r.get("gpu_equals_restatement", True) for r in result["shapes"]):
        raise SystemExit("the GPU partition differs from the restatement")


if __name__ == "__main__":
    main()
