"""Device-side k-hop neighbour sampling (dgg_b200.samplers.neighbor_sample): ms per batch, sampled edges/s, kernel
launches and device->host reads per batch, at the two shapes the reference's mini-batch drivers use:

  pubmed  N = 19 717, 88 648 edges, num_neighbors [50, 50], 1 024 seeds per batch (train_pubmed.py:370-375)
  reddit  N = 232 965, 114 615 892 edges generated on the device, num_neighbors [25, 10], 1 024 seeds per batch

Edges are uniform random (source, target) pairs from a fixed seed; only the sizes follow the datasets.  Timing: host
clock around `--batches` calls ended by a device synchronise (the sampler reads two values per hop back to the host,
so a call cannot run ahead of the device anyway), after `--warmup` calls.  Launch and read counts come from one
torch.profiler pass of its own.  For context it also times tests/neighbor_ref.py (the sequential restatement the GPU
output is checked against) on one Pubmed batch on the host cores, and checks that batch bit for bit.  Prints the card
name and power limit with the numbers; --out also writes them as JSON.

    python scripts/neighbor_sample_bench.py [--batches 200] [--warmup 20] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPES = {
    "pubmed": dict(n=19717, e=88648, num_neighbors=[50, 50], batch=1024),
    "reddit": dict(n=232965, e=114615892, num_neighbors=[25, 10], batch=1024),
}


def card():
    out = dict(name=torch.cuda.get_device_name(0), power_limit_w=None, sm_max_mhz=None)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        p, c = [s.strip() for s in q.strip().split(",")]
        out.update(power_limit_w=float(p), sm_max_mhz=float(c))
    except Exception as exc:          # the card name still identifies the measurement
        out["nvidia_smi"] = f"unavailable: {exc}"
    return out


def make_csc(n, e, seed):
    """Uniform random edges on the device -> the CSC as a CSRGraph over in-neighbours."""
    from dgg_b200 import CSRGraph

    gen = torch.Generator(device="cuda").manual_seed(seed)
    src = torch.randint(0, n, (e,), generator=gen, device="cuda")
    dst = torch.randint(0, n, (e,), generator=gen, device="cuda")
    perm = torch.argsort(dst * n + src, stable=True)
    csc = CSRGraph.from_indices(torch.stack([dst[perm], src[perm]]), n)
    del src, dst, perm
    torch.cuda.empty_cache()
    return csc


def run_shape(name, batches, warmup):
    from dgg_b200 import lib, samplers

    s = SHAPES[name]
    n, b, fan = s["n"], s["batch"], s["num_neighbors"]
    csc = make_csc(n, s["e"], seed=1)
    order = torch.randperm(n, generator=torch.Generator().manual_seed(2)).to(torch.int32).cuda()
    seeds = [order[(i * b) % (n - b):][:b] for i in range(batches + warmup)]
    for i in range(warmup):
        samplers.neighbor_sample(csc, seeds[i], fan, seed=1000 + i)
    torch.cuda.synchronize()
    L = lib()
    l0 = L.dggb_kernel_launches()
    edges = 0
    t0 = time.perf_counter()
    for i in range(warmup, warmup + batches):
        *_, ne = samplers.neighbor_sample(csc, seeds[i], fan, seed=1000 + i)
        edges += sum(ne)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    lib_launches = (L.dggb_kernel_launches() - l0) / batches

    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(4):
            samplers.neighbor_sample(csc, seeds[i], fan, seed=1000 + i)
        torch.cuda.synchronize()
    gpu_events = [ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
    kernels = sum(1 for ev in gpu_events if not ev.name.startswith(("Memcpy", "Memset")))
    reads = sum(1 for ev in gpu_events if ev.name.startswith("Memcpy DtoH"))
    return csc, dict(shape=name, n=n, e=s["e"], num_neighbors=fan, batch=b, batches=batches,
                     ms_per_batch=1e3 * dt / batches, sampled_edges_per_batch=edges / batches,
                     sampled_edges_per_s=edges / dt, dggb_launches_per_batch=lib_launches,
                     gpu_kernels_per_batch=kernels / 4, device_to_host_reads_per_batch=reads / 4)


def restatement_timing(csc):
    """One Pubmed batch through tests/neighbor_ref.py on the host, and the same batch on the GPU."""
    from dgg_b200 import samplers
    from tests.neighbor_ref import neighbor_sample_ref

    s = SHAPES["pubmed"]
    colptr, row = csc.rowptr.cpu().numpy(), csc.col.cpu().numpy()
    seeds = torch.randperm(s["n"], generator=torch.Generator().manual_seed(3))[:s["batch"]]
    t0 = time.perf_counter()
    want = neighbor_sample_ref(colptr, row, seeds.numpy(), s["num_neighbors"], seed=77)
    dt = time.perf_counter() - t0
    got = samplers.neighbor_sample(csc, seeds.to(torch.int32).cuda(), s["num_neighbors"], seed=77)
    same = all(np.array_equal(np.asarray(g.cpu() if torch.is_tensor(g) else g).astype(np.int64),
                              np.asarray(w).astype(np.int64)) for g, w in zip(got, want))
    return dict(restatement_ms_per_pubmed_batch=1e3 * dt, gpu_equals_restatement=bool(same),
                host_cpus=os.cpu_count())


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batches", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--shapes", default="pubmed,reddit")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("neighbor_sample_bench.py measures the GPU sampler: no CUDA device")
    result = dict(card=card(), shapes=[])
    for name in a.shapes.split(","):
        csc, r = run_shape(name, a.batches, a.warmup)
        if name == "pubmed":
            r.update(restatement_timing(csc))
        result["shapes"].append(r)
        print(json.dumps(dict(card=result["card"], **r)), flush=True)
        del csc
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    if not all(r.get("gpu_equals_restatement", True) for r in result["shapes"]):
        raise SystemExit("the GPU batch differs from the restatement")


if __name__ == "__main__":
    main()
