"""bench.py -- DGG forward+backward throughput (nodes/s) at Pubmed shape on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload pubmed]
                    [--dump-outputs DIR]

One "step" = one ``DGG.forward`` + backward (gradients for every DGG parameter) over one Pubmed-shape
graph batch (N=19 717 nodes, F=500, h=64, E~108 k incl. self loops; BASELINE.json configs[2],
SURVEY.md 8d).  At --gpus N > 1 (torchrun) every rank processes its own graph batch per step and the
DGG weight gradients are all-reduced over NCCL (weak scaling, the way the reference's mini-batch
drivers would be data-parallelised); value = nodes all ranks processed / max-over-ranks device time.

Prints ONE JSON line (see the task contract): value (inputs resident in HBM), e2e (host buffers,
H2D/D2H inside the timed region, through the public ``dgm.DGG`` module), roofline of the dominant
kernel, cpu_baseline (the CPU oracle port timed on this box's host cores), clocks, gpu_launches.

``--impl reference`` times the CPU oracle port of the reference algorithm (the reference itself is
Python that cannot travel to the GPU box, and is the dense O(N^2 log N) algorithm) on host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

PUBMED = dict(n=19717, f=500, h=64, mean_deg=4.5, max_deg=171)
REDDIT = dict(n=232965, f=602, h=64, kc=32)   # BASELINE.json configs[3]: row-sharded all-pairs scores
METRIC = "dgg_fwd_bwd_nodes_per_s"
N_SETS = 6  # rotating input sets: 6 x ~50 MB touched per step > 126 MB L2


# --------------------------------------------------------------------------- synthetic workload
def chung_lu_graph(n, mean_deg, max_deg, seed):
    """Power-law (Chung-Lu) undirected graph + self loops -> coalesced COO (idx int64 [2,E], val).
    SURVEY.md 8d: Pubmed-shape stand-in when the real ind.pubmed.graph is not on the box."""
    g = torch.Generator().manual_seed(seed)
    w = (torch.rand(n, generator=g) * (1 - 1e-3) + 1e-3) ** (-1.0 / 1.6)      # Pareto tail
    w = w.clamp(max=float(max_deg))
    w = w * (mean_deg * n / w.sum())
    m = int(mean_deg * n / 2)
    p = w / w.sum()
    src = torch.multinomial(p, m, replacement=True, generator=g)
    dst = torch.multinomial(p, m, replacement=True, generator=g)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    loops = torch.arange(n)
    i = torch.cat([src, dst, loops])
    j = torch.cat([dst, src, loops])
    a = torch.sparse_coo_tensor(torch.stack([i, j]), torch.ones(i.numel()), (n, n)).coalesce()
    return a.indices().contiguous(), torch.ones(a._nnz())


def make_set(shape, seed):
    idx, val = chung_lu_graph(shape["n"], shape["mean_deg"], shape["max_deg"], seed)
    g = torch.Generator().manual_seed(1000 + seed)
    x = torch.rand(shape["n"], shape["f"], generator=g)
    x = x / x.sum(-1, keepdim=True)                     # == T.NormalizeFeatures (train_small_graphs.py:345)
    g_vals = torch.randn(idx.shape[1], generator=g)     # upstream gradient of the adjacency values
    g_xenc = torch.randn(shape["n"], shape["h"], generator=g) * 0.01
    return dict(idx=idx, val=val, x=x, g_vals=g_vals, g_xenc=g_xenc)


def dgg_args():
    return argparse.Namespace(extra_edge_dim=0)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm))


# --------------------------------------------------------------------------- CPU oracle leg
def induced_sample(s, n_sample):
    """The first n_sample nodes' induced subgraph of an input set (the whole set when n_sample == N)."""
    idx = s["idx"]
    if n_sample < s["x"].shape[0]:
        keep = (idx[0] < n_sample) & (idx[1] < n_sample)
        return dict(idx=idx[:, keep].contiguous(), val=s["val"][keep], x=s["x"][:n_sample],
                    g_vals=s["g_vals"][keep], g_xenc=s["g_xenc"][:n_sample])
    return s


def cpu_oracle_fwd_bwd(sets, state, n_sample, want_result=False):
    """One DGG fwd+bwd of the CPU oracle (dense reference algorithm) on the first n_sample nodes'
    induced subgraph of set 0.  Returns seconds (and, on request, what it computed: the parity leg)."""
    from oracle import dgg_oracle as O

    s = induced_sample(sets[0], n_sample)
    idx, g_vals, x = s["idx"], s["g_vals"], s["x"]
    p = {k: v.detach().clone().requires_grad_(True) for k, v in state.items()}
    t0 = time.perf_counter()
    r = O.dgg_forward(x, idx, n_sample, p)
    vals = r["out"][idx[0], idx[1]]
    near = None
    if want_result:
        # parity leg: entries whose score is within 1e-5 (relative) of a row neighbour can swap ranks under another
        # fp32 summation order; they are left out of the loss on BOTH sides (clock paused for this bookkeeping)
        from tests.helpers import near_tie_entries

        t1 = time.perf_counter()
        near = near_tie_entries(idx, r["R"].detach(), n_sample)
        g_vals = g_vals * ~near
        t0 += time.perf_counter() - t1
    torch.autograd.backward([vals, r["x_enc"]], [g_vals, s["g_xenc"]])
    dt = time.perf_counter() - t0
    if not want_result:
        return dt
    return dt, dict(vals=vals.detach(), R=r["R"].detach(), x_enc=r["x_enc"].detach(), near=near,
                    grads={k: v.grad for k, v in p.items()})


def parity_vs_oracle(m, host_set, n_sample, ref, dev):
    """The GPU module on the SAME inputs the cpu_baseline leg just ran the oracle on: what the JSON line's
    ``parity`` field reports (tests/test_gpu_bench_shapes.py asserts the same quantities)."""
    from tests.helpers import sparse_ranks

    s = induced_sample(host_set, n_sample)
    idx = s["idx"]
    near = ref["near"]
    for q in m.parameters():
        q.grad = None
    adj = torch.sparse_coo_tensor(idx.to(dev), s["val"].to(dev), (n_sample, n_sample), is_coalesced=True)
    out, x_enc = m(s["x"].to(dev), adj)
    torch.autograd.backward([out._dgg_vals, x_enc], [(s["g_vals"] * ~near).to(dev), s["g_xenc"].to(dev)])
    vals = out._dgg_vals.detach().cpu()
    rank_ref = sparse_ranks(idx, ref["R"], n_sample)
    mism = (m.last_rank.cpu().long() != rank_ref) & ~near
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    grads = {k: rel(q.grad.cpu(), ref["grads"][k]) for k, q in m.named_parameters()}
    return dict(nodes=int(n_sample), edges=int(idx.shape[1]),
                support_equal=bool(torch.equal(out.coalesce().indices().cpu(), idx)),
                max_abs=float((vals - ref["vals"])[~near].abs().max()),
                max_abs_x_enc=float((x_enc.detach().cpu() - ref["x_enc"]).abs().max()),
                rank_mismatch_rows=int(torch.unique(idx[0][mism]).numel()),
                near_tie_entries=int(near.sum()),
                grad_max_rel_err=max(grads.values()), grad_rel_err=grads,
                note="entries whose score is within 1e-5 (relative) of a row neighbour can swap ranks under another "
                     "fp32 summation order: they are excluded from max_abs / rank_mismatch_rows and from the loss "
                     "whose gradients are compared (on both sides); grad_rel_err = max|d| / max|ref| per parameter")


def pick_sample(sets, state, budget_s, n_full):
    """Largest node count whose dense O(N^2) oracle step fits the time budget (calibrated live)."""
    n0 = min(2048, n_full)
    cpu_oracle_fwd_bwd(sets, state, min(512, n_full))          # warm the thread pool
    t0 = cpu_oracle_fwd_bwd(sets, state, n0)
    c = t0 / (n0 * n0)
    n = int(min(n_full, (budget_s / c) ** 0.5))
    return max(256, n)


# --------------------------------------------------------------------------- main arms
def run_reference(args, rank):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count())
    shape = PUBMED
    sets = [make_set(shape, 0)]
    torch.manual_seed(0)
    state = ref_state(shape)
    total_budget = 150.0
    n_s = pick_sample(sets, state, total_budget / max(1, args.steps + args.warmup), shape["n"])
    for _ in range(args.warmup):
        cpu_oracle_fwd_bwd(sets, state, n_s)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_oracle_fwd_bwd(sets, state, n_s)
    value = n_s * args.steps / t
    sample = (f"CPU oracle port of dgm.py:1758-1815 (dense N^2 scatter + row sort), fwd+bwd on the {n_s}-node "
              f"induced subgraph of the Pubmed-shape graph; dense cost grows ~N^2 so nodes/s at the full "
              f"{shape['n']} nodes is lower")
    line = dict(metric=METRIC, value=value, unit="nodes/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * t / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference",
                config=dict(workload="pubmed-shape DGG fwd+bwd", n=shape["n"], f=shape["f"], h=shape["h"]),
                cpu_baseline=dict(value=value, unit="nodes/s", cores=os.cpu_count(), kind="port", sample=sample),
                e2e=dict(value=value, unit="nodes/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line), flush=True)


def ref_state(shape):
    """Random-init DGG weights with the reference's parameter names (dgm.py:1741-1752)."""
    import torch.nn as nn

    torch.manual_seed(0)
    ne, ee, dd = nn.Linear(shape["f"], shape["h"]), nn.Linear(shape["h"], shape["h"]), nn.Linear(1, 1)
    with torch.no_grad():
        ne.weight.mul_(8.0)          # spread the scores (default init on row-normalised x is near-constant)
        dd.weight.fill_(0.9)
        dd.bias.fill_(0.4)
    return {"node_encoder.0.weight": ne.weight.detach(), "node_encoder.0.bias": ne.bias.detach(),
            "edge_encoder.0.weight": ee.weight.detach(), "edge_encoder.0.bias": ee.bias.detach(),
            "degree_decoder.0.weight": dd.weight.detach(), "degree_decoder.0.bias": dd.bias.detach()}


def time_region(fn, steps, world):
    """barrier + sync, CUDA events around `steps` calls on the current stream, max over ranks -> ms."""
    import torch.distributed as dist

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def run_ours(args, rank, local_rank, world):
    import torch.distributed as dist

    import dgg_b200
    import dgm
    from dgg_b200 import CSRGraph

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shape = PUBMED
    L = dgg_b200.lib()

    host_sets = [make_set(shape, 100 * rank + s) for s in range(N_SETS)]
    state = ref_state(shape)
    m = dgm.DGG(in_dim=shape["f"], latent_dim=shape["h"], args=dgg_args())
    m.load_state_dict(state)
    m = m.to(dev)
    params = [p for p in m.parameters()]

    # ---- device-resident inputs (the `value` arm) ----
    dsets = []
    for s in host_sets:
        adj = torch.sparse_coo_tensor(s["idx"].to(dev), s["val"].to(dev), (shape["n"], shape["n"]),
                                      is_coalesced=True)
        CSRGraph.from_coo(adj)  # CSR handle cached on the tensor, as a training loop holding adj would
        dsets.append(dict(adj=adj, x=s["x"].to(dev), g_vals=s["g_vals"].to(dev), g_xenc=s["g_xenc"].to(dev)))
    flat_grads = None

    def eager_step(s):
        for p in params:            # zero_grad(set_to_none=True): the backward's own buffers become the .grad tensors
            p.grad = None           # (no fill, no accumulation kernels); a captured graph returns them as outputs
        out, x_enc = m(s["x"], s["adj"])
        torch.autograd.backward([out._dgg_vals, x_enc], [s["g_vals"], s["g_xenc"]])
        return out._dgg_vals, x_enc, [p.grad for p in params]

    # one captured CUDA graph per resident input set (a training loop that holds its mini-batches on the
    # device replays its step); --no-graph times the eager path instead
    graphed, peer_ar, flat_grads, grad_sync = None, None, None, "none (single GPU)"
    if not args.no_graph:
        from dgg_b200.sharding import PeerAllReduce

        n_par = sum(p.numel() for p in params)
        if world > 1 and PeerAllReduce.available() and not os.environ.get("DGGB_NO_PEER_AR"):
            try:    # the step's gradients are packed into symmetric (peer-mapped) memory by ONE copy kernel and summed
                    # by a captured kernel; two buffers, alternated by the graphs: no end barrier
                peer_ar = [PeerAllReduce(n_par, end_barrier=False) for _ in range(2)]
                grad_sync = ("in-graph one-shot all-reduce kernel over NVLink peer memory, double-buffered"
                             + (" (NVSwitch multicast reduction)" if peer_ar[0].multicast else " (P2P loads)"))
            except Exception as e:   # symmetric memory not available on this fabric: captured NCCL all-reduce
                peer_ar = None
                grad_sync = f"NCCL all_reduce captured in the step graph (symmetric memory unavailable: {repr(e)[:80]})"
        if peer_ar is None and world > 1:
            flat_grads = torch.zeros(n_par, dtype=torch.float32, device=dev)
            if grad_sync.startswith("none"):
                grad_sync = "NCCL all_reduce captured in the step graph"

        def graph_body(s, j):
            out, x_enc, grads = eager_step(s)
            if world > 1:       # one batched copy instead of a fill + one accumulation kernel per parameter
                flat = peer_ar[j % 2].buffer if peer_ar is not None else flat_grads
                torch.cat([g.reshape(-1) for g in grads], out=flat)
                if peer_ar is not None:
                    return out, x_enc, peer_ar[j % 2]()
                dist.all_reduce(flat)
                return out, x_enc, flat
            return out, x_enc, grads

        graphed = []
        for j, s in enumerate(dsets):       # N_SETS is even: consecutive replays alternate between the two buffers
            graphed.append(dgg_b200.GraphedStep(lambda s=s, j=j: graph_body(s, j)))

    replay_no = [0]     # a running index (not the caller's): consecutive replays must alternate the gradient buffers
    last = [None]       # (edge values, x_enc, weight gradients) of the latest step: what --dump-outputs writes

    def step_resident(i):
        if graphed is not None:
            last[0] = graphed[replay_no[0] % N_SETS]()
            replay_no[0] += 1
        else:
            last[0] = eager_step(dsets[i % N_SETS])
            if world > 1:
                flat = torch.cat([p.grad.flatten() for p in params])
                dist.all_reduce(flat)
                last[0] = last[0][:2] + (flat,)

    # ---- host-buffer inputs (the `e2e` arm): what train_small_graphs.py does every call ----
    pinned = [dict(idx=s["idx"].pin_memory(), val=s["val"].pin_memory(), x=s["x"].pin_memory()) for s in host_sets]
    out_host = torch.empty(max(s["idx"].shape[1] for s in host_sets), dtype=torch.float32).pin_memory()
    gsum_host = torch.empty(1, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in pinned[0].values())
    d2h = pinned[0]["idx"].shape[1] * 4 + 4

    # Every step copies ITS inputs host -> device (pinned memory) and reads its result back; the copy of step
    # i+1 is issued on a side stream while step i computes (what a prefetching training loop does), so the
    # timed region still contains every H2D/D2H byte but PCIe and the SMs overlap.
    copy_stream = torch.cuda.Stream()
    staged = {}

    def prefetch(i):
        hs = pinned[i % N_SETS]
        with torch.cuda.stream(copy_stream):
            bufs = (hs["idx"].to(dev, non_blocking=True), hs["val"].to(dev, non_blocking=True),
                    hs["x"].to(dev, non_blocking=True))
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        staged[i] = (bufs, ev)

    def step_e2e(i):
        s = dsets[i % N_SETS]
        if i not in staged:
            prefetch(i)
        (idx, val, x), ev = staged.pop(i)
        prefetch(i + 1)
        torch.cuda.current_stream().wait_event(ev)
        for t_ in (idx, val, x):
            t_.record_stream(torch.cuda.current_stream())
        for p in params:
            p.grad = None
        adj = torch.sparse_coo_tensor(idx, val, (shape["n"], shape["n"]), is_coalesced=True)
        out, x_enc = m(x, adj)
        torch.autograd.backward([out._dgg_vals, x_enc], [s["g_vals"], s["g_xenc"]])
        if world > 1:
            flat = torch.cat([p.grad.flatten() for p in params])
            dist.all_reduce(flat)
        e = out._dgg_vals.numel()
        out_host[:e].copy_(out._dgg_vals.detach(), non_blocking=True)
        gsum_host.copy_(params[0].grad.sum().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the caller reads the result on the host

    for i in range(max(3, args.warmup)):
        step_resident(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = L.dggb_kernel_launches()
    ms = time_region(step_resident, args.steps, world)
    launches = int(L.dggb_kernel_launches() - l0)
    outputs = step_outputs(last[0], m) if args.dump_outputs and rank == 0 else None
    if graphed is not None:   # replayed graphs launch the kernels recorded at capture time
        launches = sum(graphed[i % N_SETS].dggb_launches_per_replay for i in range(args.steps))
        assert N_SETS % 2 == 0
    for i in range(max(3, args.warmup)):
        step_e2e(i)
    staged.clear()          # the timed region starts with nothing prefetched
    torch.cuda.synchronize()
    ms_e2e = time_region(step_e2e, args.steps, world)
    clocks = sampler.stop() if rank == 0 else None

    nodes = shape["n"] * world * args.steps
    value = nodes / (ms * 1e-3)
    e2e_value = nodes / (ms_e2e * 1e-3)
    reddit = None
    if not os.environ.get("DGGB_BENCH_NO_REDDIT"):
        try:        # all ranks take part (collectives); a failure here must not cost the headline line
            reddit = reddit_record(rank, world, dev)
        except Exception as e:
            reddit = dict(error=repr(e)[:300])

    if rank != 0:
        finish(world)
        return

    roofline = kernel_roofline(m, dsets, shape)
    try:    # the whole step against the same peak: algorithmic bytes of its launches / the replayed step time
        step_keys = [k for k in roofline["others"]
                     if k.startswith(("linear_tf32x3_kernel<chained y>", "gemm_tn_tf32x3_kernel: dWn",
                                      "linear_tf32x3_kernel: d pre", "dgg_fwd_fused2_kernel", "dgg_bwd_fused2_kernel"))]
        if len(step_keys) == 5 and world == 1:
            sb = sum(roofline["others"][k]["algorithmic_bytes"] for k in step_keys)
            # the edge kernels' gathered rows are L2-resident at this size: second figure with their COMPULSORY bytes
            sc = sum(roofline["others"][k].get("compulsory_bytes", roofline["others"][k]["algorithmic_bytes"])
                     for k in step_keys)
            st = ms / args.steps * 1e-3
            roofline["step"] = dict(algorithmic_bytes=int(sb), compulsory_bytes=int(sc), ms=st * 1e3,
                                    gbps=sb / st / 1e9, frac=sb / st / 1e9 / roofline["peak"],
                                    frac_compulsory=sc / st / 1e9 / roofline["peak"], launches=step_keys)
    except Exception as e:      # reporting only
        roofline["step"] = dict(error=repr(e)[:120])
    epoch = full_model_epoch(dsets, shape, dev) if world == 1 else None
    if epoch is not None and not os.environ.get("DGGB_BENCH_NO_CONFIGS"):
        epoch["configs"] = config_epochs(dev, dsets)
    cpu, parity = None, None
    if world == 1:
        torch.set_num_threads(os.cpu_count())
        n_s = pick_sample(host_sets, state, 12.0, shape["n"])
        t, ref = cpu_oracle_fwd_bwd(host_sets, state, n_s, want_result=True)
        cpu = dict(value=n_s / t, unit="nodes/s", cores=os.cpu_count(), kind="port",
                   sample=f"CPU oracle (dense reference algorithm, dgm.py:1758-1815) fwd+bwd on the {n_s}-node "
                          f"induced subgraph of set 0, 1 run, {t:.1f} s")
        parity = parity_vs_oracle(m, host_sets[0], n_s, ref, dev)
        del ref

    line = dict(metric=METRIC, value=value, unit="nodes/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic",
                config=dict(workload="pubmed-shape DGG fwd+bwd", n=shape["n"], f=shape["f"], h=shape["h"],
                            edges=int(host_sets[0]["idx"].shape[1]), graphs_per_step_per_gpu=1,
                            l2=f"rotating {N_SETS} input sets (> 126 MB L2)",
                            launch=("eager" if args.no_graph else "CUDA-graph replay of the captured fwd+bwd step"),
                            parallelism=(f"dp{world} (one graph batch per rank; weight-gradient sum: {grad_sync})"
                                         if world > 1 else "single GPU")),
                e2e=dict(value=e2e_value, unit="nodes/s", ms_per_step=ms_e2e / args.steps,
                         h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h)),
                gpu_launches=launches, roofline=roofline, cpu_baseline=cpu, parity=parity, clocks=clocks, epoch=epoch,
                reddit=reddit)
    if outputs is not None:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    print(json.dumps(line), flush=True)
    finish(world)


def step_outputs(res, m):
    """What a caller of the timed step receives, copied to the host as float32: the DGG edge values (in the order of
    the input's coalesced support), x_enc, and every parameter's gradient (summed over the ranks when several GPUs
    take part).  About 6 MB at Pubmed shape."""
    vals, x_enc, grads = res
    named = list(m.named_parameters())
    if torch.is_tensor(grads):      # one flat all-reduced buffer
        grads = grads.split([q.numel() for _, q in named])
    out = dict(out_values=vals, x_enc=x_enc)
    out.update({f"grad.{k}": g.reshape(q.shape) for (k, q), g in zip(named, grads)})
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def finish(world):
    """Every rank leaves together and without the process-group / symmetric-memory teardown (which can block when
    the peers are already gone): rank 0 still runs the single-GPU legs (roofline, parity) after the others are done."""
    if world > 1:
        import torch.distributed as dist

        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


def reddit_record(rank, world, dev, steps=4, warmup=2):
    """BASELINE.json configs[3] inside every bench line: Reddit-shape (N = 232 965, F = 602, 41 classes) row-sharded
    ``SAGE_DGG``-style training step -- all-pairs DGG (all_gather(z) -> tcgen05 score GEMM + streaming top-K on the
    rank's row block, in-kernel Philox Gumbel noise) + two mean-aggregation layers (all_gather(p) -> CSR SpMM on
    local rows -> reduce_scatter in the backward) + loss + backward + weight-gradient all-reduce.  STRONG scaling:
    the graph is fixed, rank r owns rows [r ceil(N / R), ...).  Also reports shard parity: four random 1 024-row
    blocks recomputed on their own (different row offset: the kernel's tiles fall elsewhere) must equal the rows of
    the sharded result bit for bit, and one block is checked against a dense fp32 restatement with an injected
    Gumbel slice (SURVEY 8d)."""
    import torch.distributed as dist
    import torch.nn.functional as F

    from dgg_b200 import functional as K
    from dgg_b200 import sharding as S

    shape = REDDIT
    n, f, h, kc, nclass = shape["n"], shape["f"], shape["h"], shape["kc"], 41
    rb, cnt, _ = S.row_block(n, world, rank)
    torch.manual_seed(0)                                     # replicated weights: same seed on every rank
    m = S.RowShardedSAGE_DGG(f, h, nclass, d=h, kc=kc).to(dev)
    params = [p for p in m.parameters()]
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    x = torch.randn(cnt, f, generator=gen, device=dev)
    labels = torch.randint(0, nclass, (cnt,), generator=gen, device=dev)

    def step(i):
        for p in params:
            p.grad = None
        logp, idx, ahat = m(x, n, seed=i)
        loss = F.nll_loss(logp, labels, reduction="sum") / n
        loss.backward()
        if world > 1:
            S.all_reduce_grads(params)
        return logp, idx, ahat

    m.train()
    for i in range(warmup):
        step(i)
    ms = time_region(step, steps, world)
    # ---- shard parity
    m.eval()
    with torch.no_grad():
        z_local = m.input_project(x)
        z_all = S.all_gather_rows(z_local, n) if world > 1 else z_local
        t = m.t.detach()
        full_i, full_v = K.allpairs_topk(z_all, t, None, kc, 3, rb, cnt, seed=7, noise_scale=1.0)
        g2 = torch.Generator().manual_seed(5 + rank)
        bitwise, offs = True, []
        for _ in range(4):
            off = int(torch.randint(0, max(1, cnt - 1024), (1,), generator=g2))
            rows = min(1024, cnt - off)
            i2, v2 = K.allpairs_topk(z_all, t, None, kc, 3, rb + off, rows, seed=7, noise_scale=1.0)
            bitwise &= bool(torch.equal(i2, full_i[off:off + rows]) and torch.equal(v2, full_v[off:off + rows]))
            offs.append(rb + off)
        rows = min(1024, cnt)
        gn = torch.Generator(device=dev).manual_seed(99 + rank)
        noise = -torch.log(-torch.log(torch.rand(rows, n, generator=gn, device=dev).clamp_min(1e-20)))
        ii, vv = K.allpairs_topk(z_all, t, noise, kc, 3, rb, rows)
        dd = torch.cdist(z_all[rb:rb + rows], z_all, compute_mode="donot_use_mm_for_euclid_dist")
        dd[torch.arange(rows, device=dev), torch.arange(rb, rb + rows, device=dev)] = 0.0
        yy = -t * dd + noise
        tv, ti = torch.topk(yy, kc + 1, dim=-1)
        ok = ((tv[:, :-1] - tv[:, 1:]) > 2e-5).all(-1)
        idx_match = float((ii.long()[ok] == ti[ok][:, :kc]).float().mean()) if bool(ok.any()) else 1.0
        max_abs = float((vv - tv[:, :kc]).abs().max())
        flags = torch.tensor([float(bitwise), idx_match, max_abs], device=dev)
        if world > 1:
            mins = flags.clone()
            dist.all_reduce(mins, op=dist.ReduceOp.MIN)
            maxs = flags.clone()
            dist.all_reduce(maxs, op=dist.ReduceOp.MAX)
            flags = torch.stack([mins[0], mins[1], maxs[2]])
        parity = dict(blocks=4, rows_per_block=1024, bitwise_equal=bool(flags[0] > 0.5),
                      dense_idx_match_on_separated_rows=float(flags[1]), dense_max_abs=float(flags[2]),
                      tolerance="indices exact on rows whose selected scores are > 2e-5 apart; values atol 2e-5 "
                                "(3xTF32 distances vs fp32 direct differences)")
        # ---- dominant kernels timed alone on this rank's block
        def timed(fn, it=3):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(it):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / it * 1e-3
        t_ap = timed(lambda: K.allpairs_topk(z_all, t, None, kc, 3, rb, cnt, seed=3, noise_scale=1.0))
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(peaks_path)) if os.path.isfile(peaks_path) else dict(bf16_tflops_sustained=1400.0, hbm_gbs=6650.0)
    flops = 2.0 * cnt * n * h
    rec = dict(workload="reddit-shape row-sharded SAGE_DGG-style train step (all-pairs DGG + 2 mean-aggregation layers)",
               n=n, f=f, d=h, kc=kc, classes=nclass, scaling="strong", n_gpus=world, steps=steps,
               ms_per_step=ms / steps, nodes_per_s=n * steps / (ms * 1e-3),
               collectives="all_gather(z), all_gather(s^-1/2), all_gather(p) per layer; reduce_scatter of the column-side "
                           "gradients in the backward; one flat all_reduce of the replicated weight gradients (NCCL)",
               shard_parity=parity,
               roofline=dict(bound="tensor", kernel="allpairs_topk2_kernel (score GEMM + top-K, this rank's row block)",
                             achieved=flops / t_ap / 1e12, peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                             frac=flops / t_ap / 1e12 / peaks["bf16_tflops_sustained"], kernel_ms=t_ap * 1e3,
                             pair_scores_per_s=cnt * n / t_ap,
                             simt_issue=dict(instr_per_pair=20.9, peak_pairs_per_s=148 * 128 * 1.965e9 / 20.9,
                                             frac=cnt * n / t_ap / (148 * 128 * 1.965e9 / 20.9),
                                             source="profiles/r02c_allpairs_ncu.md: 334 SASS instructions per "
                                                    "16-column chunk of the streaming loop, 128 lanes x 148 SMs"),
                             note="the SIMT epilogue (distance, Philox word, one ex2 candidate test per scored pair; "
                                  "the Gumbel logs only for candidates) bounds this kernel, not the tensor pipe; "
                                  "3xTF32 issues 3x the algorithmic flops"))
    del m, x, z_all
    torch.cuda.empty_cache()
    return rec


def full_model_epoch(dsets, shape, dev, iters=20):
    """BASELINE.json's second number, "epoch ms": one GCN_DGG_00 training step (forward, nll loss, backward,
    Adam with the script's two parameter groups) at Pubmed shape, and the script epoch = 1 train step + 2
    evaluation forwards (train_small_graphs.py:429-440).  Eager launches, device-resident inputs."""
    import torch.nn.functional as F

    import model as models

    args = argparse.Namespace(extra_edge_dim=0, dgg_adj_input="input_adj")
    torch.manual_seed(0)
    net = models.GCN_DGG_00(nfeat=shape["f"], nlayers=2, nhidden=shape["h"], nclass=3, dropout=0.5, lamda=0.5,
                            alpha=0.1, variant=False, args=args).to(dev)
    with torch.no_grad():
        net.conv1.W.mul_(0.1)
        net.conv2.W.mul_(0.1)
    # the script's two parameter groups (train_small_graphs.py:407-414); fused=True: one Adam kernel per group
    opt = torch.optim.Adam([dict(params=net.params1, weight_decay=5e-4), dict(params=net.params2, weight_decay=0.0)],
                           lr=0.01, fused=True)
    n = shape["n"]
    labels = torch.randint(0, 3, (n,), device=dev)
    mask = torch.zeros(n, dtype=torch.bool, device=dev)
    mask[:60] = True

    def train_step(i):
        s = dsets[i % N_SETS]
        net.train()
        opt.zero_grad()
        out, _, _ = net(s["x"], s["adj"])
        F.nll_loss(out[mask], labels[mask]).backward()
        opt.step()

    def script_epoch(i):
        train_step(i)
        net.eval()
        with torch.no_grad():
            for _ in range(2):
                net(dsets[i % N_SETS]["x"], dsets[i % N_SETS]["adj"])

    def timed(fn):
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    t_step, t_epoch = timed(train_step), timed(script_epoch)
    res = dict(model="GCN_DGG_00", shape="pubmed", train_step_ms=t_step, script_epoch_ms=t_epoch,
               nodes_per_s_train_step=n / (t_step * 1e-3),
               reference_cpu="BASELINE.md: 125 s per train step on 8 CPU cores (dense D A D normalisation, N^3)")
    # the same train step replayed as a CUDA graph (capturable Adam, one graph per resident batch)
    try:
        import dgg_b200

        opt_g = torch.optim.Adam([dict(params=net.params1, weight_decay=5e-4),
                                  dict(params=net.params2, weight_decay=0.0)], lr=0.01, capturable=True,
                                 fused=True)
        idx_train = mask.nonzero().flatten()
        y_train = labels[idx_train]

        def graph_body(s):
            net.train()
            opt_g.zero_grad(set_to_none=True)
            out, _, _ = net(s["x"], s["adj"])
            loss = F.nll_loss(out[idx_train], y_train)
            loss.backward()
            opt_g.step()
            return loss

        graphs = [dgg_b200.GraphedStep(lambda s=s: graph_body(s)) for s in dsets]
        res["train_step_graph_ms"] = timed(lambda i: graphs[i % N_SETS]())
    except Exception as e:   # capture is an optimisation, never a reason to lose the bench line
        res["train_step_graph_ms"] = None
        res["train_step_graph_error"] = repr(e)[:200]
    return res


def _step_timer(fn, iters=10, warm=3):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _sparse_features(n, f, density, seed):
    """Bag-of-words style features (Cora 1.3 % / Citeseer 0.9 % dense), row-normalised like T.NormalizeFeatures."""
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(n, f, generator=g) < density).float()
    x[torch.arange(n), torch.randint(0, f, (n,), generator=g)] = 1.0
    return x / x.sum(-1, keepdim=True)


def config_epochs(dev, pubmed_sets):
    """BASELINE.json configs[0..2] as training steps (forward, nll loss, backward, the script's Adam groups) on
    synthetic graphs of the named shapes, eager and as a CUDA-graph replay, next to the CPU oracle's fwd+bwd of the
    same model (dense reference algorithm, this box's host cores):
      Cora-shape  GCN_DGG   (DGG_LearnableK_debug: u-v-deg, k-net x, k_times_edge_prob)   N = 2 708, F = 1 433
      Citeseer-shape GCNII_DGG, 64 layers, 2 DGG layers                                  N = 3 327, F = 3 703
      Pubmed-shape GAT_DGG_00, 8 heads + 1 (GPU only: the dense reference needs ~40 GB per backward)"""
    import torch.nn.functional as F

    import dgg_b200
    import model as models
    from oracle import dgg_oracle as O

    out = []
    lk = dict(extra_edge_dim=2, extra_k_dim=1, dgg_hard=False, deg_mean=3.899, deg_std=5.288,
              dgg_mode_edge_net="u-v-deg", dgg_mode_k_net="x", dgg_mode_k_select="k_times_edge_prob", debug_step=3,
              perturb_edge_prob=False, symmetric_noise=True, stochastic_k=False, dgg_adj_input="input_adj",
              n_dgg_layers=2)

    def build_graph(n, mean_deg, seed):
        idx, val = chung_lu_graph(n, mean_deg, 60, seed)
        keep = idx[0] != idx[1]                     # the scripts pass the graph WITHOUT self loops
        return idx[:, keep].contiguous(), val[keep]

    def run(name, cls, n, f, c, density, mean_deg, layers, args, hidden=64, lr=0.01, cpu=None):
        idx, val = build_graph(n, mean_deg, 7)
        x = _sparse_features(n, f, density, 8)
        g = torch.Generator().manual_seed(9)
        labels = torch.randint(0, c, (n,), generator=g)
        train_idx = torch.arange(140)
        torch.manual_seed(0)
        net = models.__dict__[cls](nfeat=f, nlayers=layers, nhidden=hidden, nclass=c, dropout=0.6, lamda=0.5,
                                   alpha=0.1, variant=False, args=argparse.Namespace(**args))
        state = {k: v.detach().clone() for k, v in net.state_dict().items()}
        net = net.to(dev)
        adj = torch.sparse_coo_tensor(idx.to(dev), val.to(dev), (n, n)).coalesce()
        dgg_b200.CSRGraph.from_coo(adj)
        xd, yd, ti = x.to(dev), labels.to(dev), train_idx.to(dev)
        def groups():      # fresh dicts per optimiser (Adam writes its defaults, incl. capturable, into them)
            return ([dict(params=net.params1, weight_decay=0.01), dict(params=net.params2, weight_decay=5e-4)]
                    if "II" in cls else
                    [dict(params=net.params1, weight_decay=5e-4), dict(params=net.params2, weight_decay=0)])
        rec = dict(model=cls, shape=name, n=n, f=f, layers=layers, edges=int(idx.shape[1]))

        def make_step(opt):
            def step(_i=0):
                net.train()
                opt.zero_grad(set_to_none=True)
                res = net(xd, adj)
                logp = res[0] if isinstance(res, tuple) else res
                loss = F.nll_loss(logp[ti], yd[ti])
                loss.backward()
                opt.step()
                return loss
            return step

        rec["train_step_ms"] = _step_timer(make_step(torch.optim.Adam(groups(), lr=lr, fused=True)))
        try:
            gs = dgg_b200.GraphedStep(make_step(torch.optim.Adam(groups(), lr=lr, capturable=True, fused=True)))
            rec["train_step_graph_ms"] = _step_timer(lambda i: gs(), iters=20)
        except Exception as e:
            rec["train_step_graph_ms"], rec["train_step_graph_error"] = None, repr(e)[:200]
        if cpu is not None:
            torch.set_num_threads(os.cpu_count())
            cpu(x, idx, val, n, state, labels, train_idx)                       # warm the thread pool
            t0 = time.perf_counter()
            cpu(x, idx, val, n, state, labels, train_idx)
            rec["cpu_oracle_fwd_bwd_ms"] = (time.perf_counter() - t0) * 1e3
            rec["cpu_cores"] = os.cpu_count()
        out.append(rec)

    def cpu_gcn_dgg(x, idx, val, n, state, labels, ti):
        p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
        a = O.add_self_loops_dense(idx, val, n).to_sparse().coalesce()
        d = O.learnable_k_forward(x, a.indices(), a.values(), n, {k[7:]: v for k, v in p.items() if k.startswith("dggs.0.")},
                                  "u-v-deg", "x", "k_times_edge_prob")
        na = O.normalize_adj(d["out"])
        hh = O.gcn_conv(O.gcn_conv(x, na, p["conv1.W"]), na, p["conv2.W"])
        F.nll_loss(F.log_softmax(hh, -1)[ti], labels[ti]).backward()

    def cpu_gcnii_dgg(x, idx, val, n, state, labels, ti):
        p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
        a = O.add_self_loops_dense(idx, val, n).to_sparse().coalesce()
        h0 = torch.relu(F.linear(x, p["fcs.0.weight"], p["fcs.0.bias"]))
        hh, na = h0, None
        n_layers = sum(1 for k in p if k.startswith("convs.") and k.endswith(".weight"))
        for i in range(n_layers):
            if i < 2:
                d = O.learnable_k_forward(x, a.indices(), a.values(), n,
                                          {k[len(f"dggs.{i}."):]: v for k, v in p.items() if k.startswith(f"dggs.{i}.")},
                                          "u-v-deg", "x", "k_times_edge_prob")
                na = O.normalize_adj(d["out"])
            hh = torch.relu(O.gcnii_conv(hh, na, h0, p[f"convs.{i}.weight"], 0.5, 0.1, i + 1))
        logits = F.linear(hh, p["fcs.1.weight"], p["fcs.1.bias"])
        F.nll_loss(F.log_softmax(logits, 1)[ti], labels[ti]).backward()

    for spec in (dict(name="cora", cls="GCN_DGG", n=2708, f=1433, c=7, density=0.013, mean_deg=3.9, layers=2, args=lk,
                      cpu=cpu_gcn_dgg),
                 dict(name="citeseer", cls="GCNII_DGG", n=3327, f=3703, c=6, density=0.009, mean_deg=2.8, layers=64,
                      args=lk, cpu=cpu_gcnii_dgg)):
        try:
            run(**spec)
        except Exception as e:
            out.append(dict(model=spec["cls"], shape=spec["name"], error=repr(e)[:300]))
    # ---- config 3 as literally written: Pubmed-shape GAT_DGG_00 (class DGG + 8 attention heads + 1)
    try:
        shape = PUBMED
        n = shape["n"]
        torch.manual_seed(0)
        net = models.GAT_DGG_00(nfeat=shape["f"], nlayers=2, nhidden=shape["h"], nclass=3,
                                args=argparse.Namespace(extra_edge_dim=0, dgg_adj_input="input_adj")).to(dev)
        opt = torch.optim.Adam(net.parameters(), lr=0.005, weight_decay=5e-4, fused=True)      # train_small_graphs.py:417
        labels = torch.randint(0, 3, (n,), device=dev)
        ti = torch.arange(60, device=dev)
        sets = []
        for s_ in pubmed_sets:
            ii = s_["adj"].indices()
            nl = ii[:, ii[0] != ii[1]].contiguous()
            a_ = torch.sparse_coo_tensor(nl, torch.ones(nl.shape[1], device=dev), (n, n)).coalesce()
            sets.append((s_["x"], a_, nl))

        def gat_step(i, o=None):
            o = opt if o is None else o
            xg, ag, eg = sets[i % len(sets)]
            net.train()
            o.zero_grad(set_to_none=True)
            logp, _, _ = net(xg, ag, edge_index=eg)
            loss = F.nll_loss(logp[ti], labels[ti])
            loss.backward()
            o.step()
            return loss

        eager_ms = _step_timer(gat_step, iters=10)
        graph_ms, graph_err = None, None
        try:      # one captured step per resident input set (two sets: the 9-head step holds ~0.3 GB of activations)
            opt_g = torch.optim.Adam(net.parameters(), lr=0.005, weight_decay=5e-4, capturable=True, fused=True)
            gsteps = [dgg_b200.GraphedStep(lambda j=j: gat_step(j, opt_g)) for j in range(2)]
            graph_ms = _step_timer(lambda i: gsteps[i % 2](), iters=20)
        except Exception as e:
            graph_err = repr(e)[:200]
        out.append(dict(model="GAT_DGG_00", shape="pubmed", n=n, f=shape["f"], heads="8 + 1",
                        train_step_ms=eager_ms, train_step_graph_ms=graph_ms,
                        **({"train_step_graph_error": graph_err} if graph_err else {}),
                        reference_cpu="not runnable: 9 heads x dense [N, N] fp32 attention = 1.55 GB each, ~40 GB live in "
                                      "the backward (SURVEY 3.3)"))
    except Exception as e:
        out.append(dict(model="GAT_DGG_00", shape="pubmed", error=repr(e)[:300]))
    return out


def kernel_roofline(m, dsets, shape, iters=30):
    """Time each hand-written kernel of the step alone (CUDA events on the launch stream, rotating
    input sets) and report the dominant one against the measured HBM peak."""
    import ctypes

    import torch.nn.functional as F

    from dgg_b200 import CSRGraph
    from dgg_b200 import functional as K

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    lin, dd = m.edge_encoder[0], m.degree_decoder[0]
    prepared = []
    with torch.no_grad():
        for s in dsets:
            g, _ = CSRGraph.from_coo(s["adj"])
            y = F.linear(m.node_encoder(s["x"]), lin.weight)
            prepared.append((g, y, s["g_vals"]))
    n, h = shape["n"], shape["h"]
    E = prepared[0][0].nnz

    def timed(fn, reps=24):
        """Average duration of one call of fn: `reps` calls (rotating input sets) captured into ONE CUDA graph and
        replayed back to back, CUDA events around the replays -- the same launch mechanism as the timed step (an eager
        loop of 10-20 us kernels measures the host's launch rate instead)."""
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(N_SETS):
                fn(i)
        torch.cuda.current_stream().wait_stream(side)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for i in range(reps):
                fn(i)
        t_end = time.perf_counter() + 0.05      # >= 50 ms of replays first: the clocks have dropped while the host
        while time.perf_counter() < t_end:      # was busy, let them ramp up again
            gr.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            gr.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (iters * reps) * 1e-3

    from dgg_b200._lib import check, i32, lib, p, stream

    dev = prepared[0][1].device
    R = torch.empty(E + 64, device=dev)
    rank = torch.empty(E + 64, dtype=torch.int32, device=dev)
    s_row, k_row = torch.empty(n, device=dev), torch.empty(n, device=dev)
    out = torch.empty(E + 64, device=dev)
    dy = torch.zeros(n, h, device=dev)
    small = torch.zeros(h + 4 + n, device=dev)
    dw, db = dd.weight.detach().reshape(-1), dd.bias.detach().reshape(-1)
    be = lin.bias.detach()

    fused = all(0 < g.max_row_nnz <= K._FUSED_MAX_ROW for g, _, _ in prepared)   # what the modules dispatch to

    def fwd(i):   # the forward launch(es) of the edge ranker through the C-ABI, outputs preallocated
        g, y, _ = prepared[i % N_SETS]
        if fused:
            check(lib().dggb_dgg_edge_fwd_fused(p(g.rowptr), p(g.erow), p(g.col), i32(n), i32(g.nnz),
                                                i32(g.max_row_nnz), i32(h), p(y), p(be), p(dw), p(db), p(None),
                                                i32(-1), p(R), p(rank), p(s_row), p(k_row), p(out), p(None),
                                                ctypes.c_int64(0), stream()), "fwd")
            return
        check(lib().dggb_dgg_edge_fwd(p(g.rowptr), p(g.erow), p(g.col), i32(n), i32(g.nnz), i32(h), p(y), p(be),
                                      p(dw), p(db), p(None), i32(-1), p(R), p(rank), p(s_row), p(k_row), p(out),
                                      p(None), stream()), "fwd")

    def bwd(i):   # the backward launch(es); R/rank/s/k of the last forward stand in
        g, y, gv = prepared[i % N_SETS]
        if fused:
            check(lib().dggb_dgg_edge_bwd_fused(p(g.rowptr), p(g.erow), p(g.col), i32(n), i32(g.nnz),
                                                i32(g.max_row_nnz), i32(h), p(y), p(be), p(dw), p(db), p(None),
                                                i32(-1), p(R), p(rank), p(s_row), p(k_row), p(gv), p(small[h + 4:]),
                                                p(dy), p(small[:h]), p(small[h:h + 2]), stream()), "bwd")
            return
        check(lib().dggb_dgg_edge_bwd(p(g.rowptr), p(g.erow), p(g.col), i32(n), i32(g.nnz), i32(h), p(y), p(be),
                                      p(dw), p(db), p(None), i32(-1), p(R), p(rank), p(s_row), p(k_row), p(gv),
                                      p(small[h + 4:]), p(dy), p(small[:h]), p(small[h:h + 2]), stream()), "bwd")

    t_fwd = timed(fwd)
    t_bwd = timed(bwd)

    # the two tensor-core GEMM kernels of the node encoder (forward, weight gradient), outputs preallocated
    f_in = shape["f"]
    enc = m.node_encoder[0]
    w_enc, b_enc = enc.weight.detach().contiguous(), enc.bias.detach().contiguous()
    xs = [s["x"] for s in dsets]
    x_out = torch.empty(n, h, device=dev)
    ws_lin = torch.empty(2 * h * f_in + 2 * h * h, device=dev)
    dpre = torch.randn(n, h, device=dev)
    dw_out = torch.zeros(h * f_in + h, device=dev)
    L = lib()
    ws_tn_bytes = int(L.dggb_gemm_tn_tc_workspace_bytes(i32(n), i32(h)))
    ws_tn = torch.empty(ws_tn_bytes // 4, device=dev)

    # what one training step launches for the encoder (functional._EncodeProject): forward = weight split + GEMM with
    # the chained y = x_enc We^T; backward = d pre (leaving its transposed TF32 split and g_y's) + ONE weight-gradient
    # launch (dWn = dpre^T x, dWe = g_y^T x_enc)
    we = lin.weight.detach().contiguous()
    y_out = torch.empty(n, h, device=dev)
    wet = torch.empty(2 * h * h, device=dev)
    zb = torch.zeros(h * h + h * f_in + h, device=dev)
    npad = (n + 31) // 32 * 32
    tsp = torch.zeros(4, h, npad, device=dev)
    g_y, g_xe, x_enc_s = torch.randn(n, h, device=dev), torch.randn(n, h, device=dev), torch.randn(n, h, device=dev)

    def lin_plain(i):
        check(L.dggb_linear_act_fwd(p(xs[i % N_SETS]), p(w_enc), p(b_enc), ctypes.c_float(0.01), i32(n), i32(f_in),
                                    i32(h), p(x_out), p(ws_lin), ctypes.c_int64(ws_lin.numel() * 4), stream()), "lin")

    def enc_fwd(i):
        check(L.dggb_encoder_fwd(p(xs[i % N_SETS]), p(w_enc), p(b_enc), ctypes.c_float(0.01), i32(n), i32(f_in), i32(h),
                                 p(x_out), p(we), p(y_out), p(ws_lin), ctypes.c_int64(ws_lin.numel() * 4), p(wet),
                                 p(zb), ctypes.c_int64(zb.numel()), stream()), "encoder_fwd")

    def enc_dpre(i):
        check(L.dggb_encoder_bwd_dpre(p(g_y), p(wet), p(g_xe), p(x_enc_s), ctypes.c_float(0.01), i32(n), i32(h), p(None),
                                      p(tsp[0]), p(tsp[1]), i32(npad), p(zb[h * h + h * f_in:]), p(tsp[2]), p(tsp[3]),
                                      stream()), "encoder_bwd_dpre")

    def tn(i):
        check(L.dggb_gemm_tn_tc_presplit(p(tsp[0]), p(tsp[1]), i32(npad), p(xs[i % N_SETS]), i32(n), i32(h), i32(f_in),
                                         p(zb[h * h:h * h + h * f_in]), p(tsp[2]), p(tsp[3]), p(x_enc_s), i32(h),
                                         p(zb[:h * h]), stream()), "gemm_tn_tc_presplit")

    enc_fwd(0)          # leaves the pre-split We^T the d pre launch reads
    t_lin = timed(lin_plain)
    t_enc = timed(enc_fwd)
    t_dpre = timed(enc_dpre)
    t_tn = timed(tn)
    # algorithmic bytes (DESIGN.md section 4; int32 CSR, fp32)
    b_fwd = E * (4 + 4 * h) + n * (4 * h + 12) + E * 12
    b_bwd = E * (4 + 4 * h + 12) + E * 4 * h + n * (4 * h * 2 + 12)
    b_lin = n * f_in * 4 + n * h * 4 + h * f_in * 4
    b_enc = n * f_in * 4 + 2 * n * h * 4 + h * f_in * 4 + h * h * 4
    b_dpre = 3 * n * h * 4 + 4 * h * npad * 4
    b_tn = n * f_in * 4 + n * h * 4 + 4 * h * npad * 4 + h * f_in * 4
    v2 = not os.environ.get("DGGB_FUSED_V1")
    cands = [("linear_tf32x3_kernel<chained y> (+ split_w): encoder forward, x_enc and y", t_enc, b_enc),
             ("gemm_tn_tf32x3_kernel: dWn = dpre^T x and dWe = g_y^T x_enc in one launch", t_tn, b_tn),
             ("linear_tf32x3_kernel: d pre + transposed TF32 splits of d pre and g_y + bias gradient", t_dpre, b_dpre),
             (("dgg_fwd_fused2_kernel" if v2 else "dgg_fwd_fused_kernel") if fused
              else "dgg_edge_score_kernel + dgg_row_rank_kernel", t_fwd, b_fwd),
             (("dgg_bwd_fused2_kernel" if v2 else "dgg_bwd_fused_kernel") if fused
              else "dgg_row_dk_kernel + dgg_edge_grad_kernel", t_bwd, b_bwd),
             ("linear_tf32x3_kernel (+ split_w): plain node encoder, as in r01", t_lin, b_lin)]
    name, t, b = max(cands, key=lambda c: c[1])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tpath):
        traffic = json.load(open(tpath)).get(name)
    others = {c[0]: dict(us=c[1] * 1e6, algorithmic_bytes=int(c[2]), gbps=c[2] / c[1] / 1e9,
                         frac=c[2] / c[1] / 1e9 / peak) for c in cands}
    # the gathered rows of the edge kernels are L2-resident at this size (y is 5 MB): next to the un-cached
    # algorithmic bytes above, the fraction against the COMPULSORY bytes (every array touched once)
    comp_fwd = E * 8 + n * h * 4 + E * 12 + n * 12
    comp_bwd = E * 8 + n * h * 4 + E * 16 + n * h * 4 + n * 12
    for key, tt, cb in ((cands[3][0], t_fwd, comp_fwd), (cands[4][0], t_bwd, comp_bwd)):
        others[key].update(compulsory_bytes=int(cb), frac_compulsory=cb / tt / 1e9 / peak)

    # ---- selection and aggregation kernels the conv layers / DGG_LearnableK_debug / GAT use (north_star: "achieved HBM
    # GB/s against B200 peak for selection and SpMM"), same graphs, F = h
    from dgg_b200 import functional as K

    feats = [torch.randn(n, h, device=dev) for _ in range(N_SETS)]
    gys = torch.randn(n, h, device=dev)
    vals = [torch.rand(g.nnz, device=dev) + 0.1 for g, _, _ in prepared]
    ks = torch.rand(n, device=dev) * 8 + 1
    w64 = torch.randn(h, h, device=dev) / 8
    heads = 8
    hd = torch.randn(n, heads * h, device=dev)
    pq = torch.randn(n, heads, 2, device=dev)
    gat_out = torch.empty(n, heads * h, device=dev)
    mz = torch.empty(2, n, heads, device=dev)
    y_sp, dval, dx = torch.empty(n, h, device=dev), torch.empty(E + 64, device=dev), torch.zeros(n, h, device=dev)
    rk, fo = torch.empty(E + 64, dtype=torch.int32, device=dev), torch.empty(E + 64, device=dev)
    dsc, dk = torch.empty(E + 64, device=dev), torch.empty(n, device=dev)
    s_out = torch.empty(n, h, device=dev)

    def G(i):
        return prepared[i % N_SETS][0]

    extra = [
        ("spmm_fwd_kernel (F=64)", lambda i: check(L.dggb_spmm_csr_fwd(p(G(i).rowptr), p(G(i).col), p(vals[i % N_SETS]), n, p(feats[i % N_SETS]), h, None, p(y_sp), stream()), "spmm"),
         E * (8 + h * 4) + n * h * 4 + n * 4),
        ("spmm_bwd_kernel (F=64, dA + dX)", lambda i: check(L.dggb_spmm_csr_bwd(p(G(i).rowptr), p(G(i).col), p(vals[i % N_SETS]), n, p(feats[i % N_SETS]), h, None, p(gys), p(dval), p(dx), stream()), "spmm_bwd"),
         E * (8 + h * 4) + n * h * 4 + E * (h * 4 + 4) + n * 4),
        ("spmm_gemm_fwd_kernel (SpMM + W 64x64 + ReLU)", lambda i: check(L.dggb_spmm_gemm_fwd(p(G(i).rowptr), p(G(i).col), p(vals[i % N_SETS]), n, p(feats[i % N_SETS]), h, None, None, 1.0, 0.0, p(w64), h, 1.0, 0.0, None, 1, None, p(y_sp), p(s_out), stream()), "spmm_gemm"),
         E * (8 + h * 4) + 2 * n * h * 4 + n * 4 + h * h * 4),
        ("row_firstk_fwd_kernel (in-row rank + soft first-k)", lambda i: check(L.dggb_row_firstk_fwd(p(G(i).rowptr), n, p(vals[i % N_SETS]), p(ks), 0, p(rk), p(fo), None, stream()), "firstk"),
         E * 12 + n * 8),
        ("row_firstk_bwd_kernel", lambda i: check(L.dggb_row_firstk_bwd(p(G(i).rowptr), n, p(vals[i % N_SETS]), p(ks), 0, p(rk), p(fo), p(dsc), p(dk), stream()), "firstk_bwd"),
         E * 20 + n * 12),
        ("gat_fwd_kernel (8 heads x F=64, dense-background softmax)", lambda i: check(L.dggb_gat_aggregate_fwd(p(G(i).rowptr), p(G(i).col), n, G(i).nnz, heads, h, p(hd), heads * h, p(pq), p(vals[i % N_SETS]), None, p(hd[0]), None, 0.2, float(n), p(gat_out), heads * h, p(mz[0]), p(mz[1]), stream()), "gat"),
         heads * (E * (h * 4 + 8) + 2 * n * h * 4 + n * 16) + E * 8),
    ]
    for nm, fn, nbytes in extra:
        tt = timed(fn)
        others[nm] = dict(us=tt * 1e6, algorithmic_bytes=int(nbytes), gbps=nbytes / tt / 1e9, frac=nbytes / tt / 1e9 / peak)
    return dict(bound="hbm", kernel=name, achieved=b / t / 1e9, peak=peak, unit="GB/s", frac=b / t / 1e9 / peak,
                traffic=traffic, peak_source=peak_src, algorithmic_bytes=int(b), kernel_us=t * 1e6, others=others)


# --------------------------------------------------------------------------- Reddit-shape all-pairs arm
def run_reddit(args, rank, local_rank, world):
    """Row-sharded all-pairs DGG (legacy ``DGG_LearnableK_SDD`` formula, dgm.py:259-351) fwd+bwd at Reddit
    shape: N=232 965, F=602, d=64, Kc=32, in-kernel Philox Gumbel(0,1) noise (an injected N x N tensor
    would be 217 GB).  Strong scaling: rank r owns rows [r N/R, (r+1) N/R) and scores them against the
    all-gathered embeddings; column-side gradients come back through a reduce-scatter; weight gradients
    are all-reduced."""
    import torch.distributed as dist
    import torch.nn.functional as F

    import dgg_b200
    import dgm
    from dgg_b200 import functional as K
    from dgg_b200 import sharding as S

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shape = REDDIT
    n, f, h, kc = shape["n"], shape["f"], shape["h"], shape["kc"]
    L = dgg_b200.lib()
    rb, cnt, _ = S.row_block(n, world, rank)
    m = dgm.DGG_LearnableK_SDD(in_dim=f, latent_dim=h, dist_fn="metric")
    with torch.no_grad():
        m.k_net.k_project.bias.fill_(9.0)        # k ~ 10 -> window ~ 22.6 <= Kc
        m.k_net.k_project.weight.mul_(0.1)
        m.t.fill_(4.0)
    m = m.to(dev)
    params = list(m.parameters())
    gen = torch.Generator().manual_seed(rank)
    x_host = torch.randn(cnt, f, generator=gen).pin_memory()
    g_host = torch.randn(cnt, kc, generator=gen)
    x_dev, g_dev = x_host.to(dev), g_host.to(dev)
    r = torch.arange(kc, device=dev, dtype=torch.float32).reshape(1, kc)
    out_host = torch.empty(cnt, kc).pin_memory()
    idx_host = torch.empty(cnt, kc, dtype=torch.int32).pin_memory()

    def fwd_bwd(x, step):
        for p in params:
            p.grad = None
        z = m.input_project(x)
        k = m.k_net(x) + m.k_bias
        if world > 1:
            idx, y = S.sharded_allpairs_topk(z, m.t, n, kc, seed=step, noise_scale=1.0)
        else:
            idx, y = K.allpairs_topk(z, m.t, None, kc, 3, seed=step, noise_scale=1.0)
        vals = y * torch.sigmoid(m.hs_start - m.interval * r + (k - 1) * m.interval)
        vals.backward(g_dev)
        if world > 1:
            S.all_reduce_grads(params)
        return idx, vals

    def step_resident(i):
        fwd_bwd(x_dev, i)

    def step_e2e(i):
        x = x_host.to(dev, non_blocking=True)
        idx, vals = fwd_bwd(x, i)
        out_host.copy_(vals.detach(), non_blocking=True)
        idx_host.copy_(idx, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for i in range(max(3, args.warmup)):
        step_resident(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = L.dggb_kernel_launches()
    ms = time_region(step_resident, args.steps, world)
    launches = int(L.dggb_kernel_launches() - l0)
    for i in range(3):
        step_e2e(i)
    ms_e2e = time_region(step_e2e, args.steps, world)
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # dominant kernel: the fused score GEMM + top-K, timed alone on this rank's row block
    with torch.no_grad():
        z_all = torch.softmax(torch.randn(n, h, device=dev), -1)
        tt = m.t.detach()
        for i in range(2):
            K.allpairs_topk(z_all, tt, None, kc, 3, rb, cnt, seed=i, noise_scale=1.0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        it = 5
        for i in range(it):
            K.allpairs_topk(z_all, tt, None, kc, 3, rb, cnt, seed=i, noise_scale=1.0)
        e1.record()
        torch.cuda.synchronize()
        t_k = e0.elapsed_time(e1) / it * 1e-3
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks_path))["bf16_tflops_sustained"] if os.path.isfile(peaks_path) else 1400.0
    flops = 2.0 * cnt * n * h
    roofline = dict(bound="tensor", kernel="allpairs_topk_kernel (+ split_tf32 pre-pass)", achieved=flops / t_k / 1e12,
                    peak=peak, unit="TFLOP/s", frac=flops / t_k / 1e12 / peak, traffic=None,
                    peak_source="MEASURED_PEAKS.json bf16_tflops_sustained" if os.path.isfile(peaks_path) else "fallback",
                    algorithmic_flops=flops, kernel_ms=t_k * 1e3, pair_scores_per_s=cnt * n / t_k,
                    note="SIMT epilogue (norms, sqrt, Philox Gumbel, selection) over rows x N scores bounds this "
                         "kernel, not the tensor pipe (SURVEY 8d caveat); 3xTF32 issues 3x the algorithmic flops")
    value = n * args.steps / (ms * 1e-3)
    line = dict(metric=METRIC, value=value, unit="nodes/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32",
                data="synthetic",
                config=dict(workload="reddit-shape all-pairs DGG fwd+bwd (row-sharded scores)", n=n, f=f, d=h, kc=kc,
                            noise="in-kernel Philox Gumbel(0,1)", precision="3xTF32 tcgen05, fp32 accumulate",
                            l2="inputs (x 561 MB, z 60 MB) exceed the 126 MB L2",
                            parallelism=f"rows/{world} + all_gather(z) + reduce_scatter(dz) over NCCL"),
                e2e=dict(value=n * args.steps / (ms_e2e * 1e-3), unit="nodes/s", ms_per_step=ms_e2e / args.steps,
                         h2d_bytes_per_step=int(x_host.numel() * 4 * world),
                         d2h_bytes_per_step=int(cnt * kc * 8 * world)),
                gpu_launches=launches, roofline=roofline, cpu_baseline=None, clocks=clocks)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _bind_to_gpu_numa_node(local_rank):
    """Multi-rank runs: keep this rank's host threads (and therefore its pinned staging buffers, first touch) on the
    CPUs next to its GPU -- eight ranks staging 41.6 MB per step through one socket's memory halve the end-to-end
    rate.  Best effort: silently skipped where NVML / sched_setaffinity are unavailable."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [i for i in range(os.cpu_count()) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pubmed", choices=["pubmed", "reddit"])
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (edge values, x_enc, weight "
                         "gradients) as DIR/<name>.npy; the inputs depend on the arguments only, so two builds can "
                         "be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "pubmed"):
        ap.error("--dump-outputs covers the pubmed workload of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl != "reference" and world > 1:
        _bind_to_gpu_numa_node(local_rank)
    if args.impl == "reference":
        run_reference(args, rank)
    elif args.workload == "reddit":
        run_reddit(args, rank, local_rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
