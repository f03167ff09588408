"""Time the fused DGG edge launches alone at the Pubmed shape of bench.py, each captured `reps` times into one CUDA
graph over the 6 rotating input sets (the launch mechanism of the timed step), CUDA events around the replays.

    fwd       dggb_dgg_edge_fwd_fused         (no branch mask)
    fwd_mask  dggb_dgg_edge_fwd_fused_mask    (writes the branch mask: what a training step launches)
    bwd       dggb_dgg_edge_bwd_fused         (builds with the mask entry points: the two-launch backward from y)
    bwd_mask  dggb_dgg_edge_bwd_fused_mask    (reads the mask: what a training step launches)

Entries a build does not export are reported as null, so the same script times a build without the mask entry
points.  Prints one JSON line (microseconds per launch, best of --rounds) with the card's name and power limit."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402
import dgm  # noqa: E402
from dgg_b200 import CSRGraph  # noqa: E402
from dgg_b200._lib import check, i32, lib, p, stream  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=24)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda")
    shape = bench.PUBMED
    m = dgm.DGG(in_dim=shape["f"], latent_dim=shape["h"], args=bench.dgg_args())
    m.load_state_dict(bench.ref_state(shape))
    m = m.to(dev)
    lin, dd = m.edge_encoder[0], m.degree_decoder[0]
    n, h = shape["n"], shape["h"]
    sets = []
    with torch.no_grad():
        for s in range(bench.N_SETS):
            hs = bench.make_set(shape, s)
            adj = torch.sparse_coo_tensor(hs["idx"].to(dev), hs["val"].to(dev), (n, n), is_coalesced=True)
            g, _ = CSRGraph.from_coo(adj)
            y = F.linear(m.node_encoder(hs["x"].to(dev)), lin.weight).contiguous()
            sets.append((g, y, hs["g_vals"].to(dev)))
    E = max(g.nnz for g, _, _ in sets)
    assert all(0 < g.max_row_nnz <= 512 for g, _, _ in sets)
    be = lin.bias.detach()
    dw, db = dd.weight.detach().reshape(-1), dd.bias.detach().reshape(-1)
    R, out = torch.empty(E, device=dev), torch.empty(E, device=dev)
    rank = torch.empty(E, dtype=torch.int32, device=dev)
    s_row, k_row = torch.empty(n, device=dev), torch.empty(n, device=dev)
    mask = torch.empty(E, (h + 31) // 32, dtype=torch.int32, device=dev)
    dy = torch.zeros(n, h, device=dev)
    small = torch.zeros(h + 4 + n, device=dev)
    L = lib()
    has_mask = hasattr(L, "dggb_dgg_edge_bwd_fused_mask")

    def head(g, y):
        return (p(g.rowptr), p(g.erow), p(g.col), i32(n), i32(g.nnz), i32(g.max_row_nnz), i32(h), p(y), p(be))

    def fwd(i):
        g, y, _ = sets[i % len(sets)]
        check(L.dggb_dgg_edge_fwd_fused(*head(g, y), p(dw), p(db), None, i32(-1), p(R), p(rank), p(s_row), p(k_row),
                                        p(out), None, ctypes.c_int64(0), stream()), "fwd")

    def fwd_mask(i):
        g, y, _ = sets[i % len(sets)]
        check(L.dggb_dgg_edge_fwd_fused_mask(*head(g, y), p(dw), p(db), None, i32(-1), p(R), p(rank), p(s_row),
                                             p(k_row), p(out), p(mask), None, None, ctypes.c_int64(0), stream()),
              "fwd_mask")

    def bwd(i):
        g, y, gv = sets[i % len(sets)]
        check(L.dggb_dgg_edge_bwd_fused(*head(g, y), p(dw), p(db), None, i32(-1), p(R), p(rank), p(s_row), p(k_row),
                                        p(gv), p(small[h + 4:]), p(dy), p(small[:h]), p(small[h:h + 2]), stream()),
              "bwd")

    def bwd_mask(i):
        g, y, gv = sets[i % len(sets)]
        check(L.dggb_dgg_edge_bwd_fused_mask(p(g.rowptr), p(g.erow), p(g.col), i32(n), i32(g.nnz), i32(g.max_row_nnz),
                                             i32(h), p(dw), p(db), None, i32(-1), p(R), p(rank), p(s_row), p(k_row),
                                             p(mask), None, p(gv), p(small[h + 4:]), p(dy), p(small[:h]),
                                             p(small[h:h + 2]), stream()), "bwd_mask")

    def graph_of(fn):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(len(sets)):
                fn(i)
        torch.cuda.current_stream().wait_stream(side)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for i in range(args.reps):
                fn(i)
        return gr

    def time_graph(gr):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            gr.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (args.iters * args.reps) * 1e3

    # the mask the backward reads comes from a masked forward of the same set (rank / s / k too); the timed backward
    # rotates over the sets, like the unmasked one, with the last forward's per-entry arrays standing in
    if has_mask:
        fwd_mask(0)
    else:
        fwd(0)
    fns = {"fwd": fwd, "fwd_mask": fwd_mask if has_mask else None, "bwd": bwd, "bwd_mask": bwd_mask if has_mask else None}
    graphs = {k: graph_of(f) for k, f in fns.items() if f is not None}
    t_end = time.perf_counter() + 0.2          # let the clocks ramp up
    while time.perf_counter() < t_end:
        for gr in graphs.values():
            gr.replay()
    torch.cuda.synchronize()
    best = {k: None for k in fns}
    for _ in range(args.rounds):              # interleaved rounds, best of each
        for k, gr in graphs.items():
            t = time_graph(gr)
            best[k] = t if best[k] is None else min(best[k], t)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e!r})"
    print(json.dumps(dict(us_per_launch={k: (None if v is None else round(v, 3)) for k, v in best.items()},
                          E=E, n=n, h=h, reps=args.reps, iters=args.iters, rounds=args.rounds, gpu=q)))


if __name__ == "__main__":
    main()
