"""Every launch path of the DGG edge family (csrc/dgg_edge.cu) against one fp64 reference.

Dispatch rules (h = hidden width, E = entries, max_row = the longest row):

* Lanes per entry: L = the smallest power of two with 16 L >= h, capped at 32; T = ceil(h / 4 L) rounded up to 1, 2 or
  4 (``dispatch_T``), so T = 1 only at h = 4 and T = 2 only at h = 8.  The fused kernels are specialised
  ``<4, LC>`` for h = 16 LC (LC in 1, 2, 4, 8, 16, 32) and use the runtime-L ``<T, 0>`` otherwise: ``<1,0>`` at h = 4,
  ``<2,0>`` at h = 8, ``<4,0>`` for every other h (12, 20, 36, 100, 260, 508, ...), with ``c < h`` guards.
* Python ``functional._DGGEdge`` takes the fused path when 0 < max_row <= 512 and E > 0, the two-launch path otherwise.
* Two-launch forward: ``dgg_edge_score_kernel<T>`` (skipped when E = 0), ``dgg_row_rank_kernel``, and, when a row is
  longer than 1 024 entries (Python then passes the ``long_ws`` list), ``long_row_rank_kernel`` in mode 2 (soft) or
  3 (hard_k >= 0).  Without ``long_ws`` such a row is swept by its warp straight from global memory.  Rows of at most
  32 entries are ranked with shuffles, rows of 33 .. 1 024 from the warp's shared-memory slice.
* Two-launch backward: ``dgg_row_dk_kernel`` (soft mode only), then ``dgg_edge_grad_kernel<T>``; nothing when E = 0.
* ``row_firstk_fwd_kernel`` (mode 0 k_times_edge_prob, 1 k_only), ``long_row_rank_kernel`` in the same mode for rows
  longer than 1 024, then ``row_firstk_bwd_kernel``.  Nothing runs on a graph without entries.
* Fused forward: ``dgg_fwd_fused2_kernel``.  Block b owns the rows that start in the entry interval
  [b epb, (b + 1) epb); blocks = min(ceil(E / min_epb), 148 x occupancy), epb = ceil(E / blocks),
  min_epb = DGGB_FUSED_EPB or 128.  It reads its score window of cap = min(epb + max_row, 12 288) entries from shared
  memory and re-reads entries beyond it from global memory.
* Fused backward: ``dgg_bwd_fused2_kernel`` when cap = epb + max_row <= 6 144, ``dgg_bwd_fused_kernel`` otherwise
  (each on the grid of its own occupancy).  ``dgg_bwd_fused_kernel`` keeps ds of the first 1 024 rows of a block in
  shared memory and reads further rows' ds back from ``ds_ws``.  ``dgg_bwd_fused2_kernel`` adds dbe with vector
  reductions when dbe is 16-byte aligned and with scalar atomics otherwise.

``PATHS`` maps each case to the launches of the family it makes, in order (forward, then backward); a ``[m]`` suffix
is the runtime mode of the kernel, which the profiler does not show.  ``test_dispatch_launches_the_tabled_kernels``
checks the table against the profiler and ``test_path_table_reaches_every_instantiation`` checks that the cases reach
all 38 kernels and the edges listed there.

Inputs keep the LeakyReLU kinks out of rounding reach by construction: y lies on a dyadic grid of step q and be on
the same grid offset by q / 2, so every y_u - y_v + be is exact and at least q / 2 away from 0.  q shrinks with h so
that z stays mostly below ~8 (one case scales it by 16 to saturate R to 1.0f).  deg_b is chosen from the data so that
w s + b is away from 0 on every row and takes both signs; the setup asserts that margin.  Two nodes of each graph
share their y row, which makes exact ties in every row that holds both.

Reference: the same computation in fp64 with ``index_add_`` over the entry list (no dense N x N), LeakyReLU slope =
the exact value of 0.01f.  Forward checks:

* self-consistency, exact: rank is the stable descending rank of the kernel's own fp32 R (ties: lower column first);
  out = R (fk(rank - k) + 1) from the kernel's own R / rank / k, within tanhf's few ulp (U R (|rank - k| + 12)), and
  out = (rank < hard_k ? R : 0) bit for bit in hard mode;
* against fp64, with u = 2^-24 and bounds from the data:
  z: u (h + 4) sum_c |LeakyReLU(pre_c)|;  R1 = sigmoid(z): R1 (1 - R1) zb + 6 u R1;  with noise
  R = sigmoid(R1 + noise): R (1 - R) (R1b + u |R1 + noise|) + 6 u R;
  s: sum_row Rb + u (deg + 2) sum_row R;  w s + b: |w| sb + 2 u (|w s| + |w s + b|);  k: slope (that) + u |k|;
  rank: exact wherever the entry's fp64 gap to both neighbours in its row exceeds the sum of their R bounds.

Backward: fp64 autograd of sum(g out) with the kernel's ranks held fixed (nothing is left out of the loss).  Each
gradient term carries the forward error of the values it uses plus u times the number of rounded terms:
  T_e = g R sech^2(r - k) / 2: |g| (Rb sech^2 + R (2 |tanh| (sech^2 kb + 4 u + sech^2 u |t|) + 4 u)) / 2 + 6 u |T|;
  dk_i = sum_row T: sum Tb + u (deg + 4) sum |T|;  ds_i = dk lr w: lr |w| dkb + 3 u |ds|;
  d deg_w, d deg_b: the row terms' bounds + u (n + 8) sum |terms|;
  dR_e = g (fk + 1) + ds_u: |g| FKb + dsb_u + 2 u (|g (fk + 1)| + |ds_u|), FKb = (sech^2 kb + 4 u + sech^2 u |t|) / 2
  + 4 u; through the noise sigmoid dRb R (1 - R) + |dR| |1 - 2 R| Rb + 3 u |.|; dz = dR R1 (1 - R1): dRb R1 (1 - R1)
  + |dR| |1 - 2 R1| R1b + 3 u |dz|;  dy: the entry bounds of every entry at the node + u (in-degree + out-degree + 8)
  sum |d pre|;  dbe: sum of the entry bounds + u (E + 16) sum |d pre|.  Bounds are doubled for the linearisation.
In hard mode d deg_w and d deg_b are exactly 0.
"""
import ctypes
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

U = 2.0 ** -24
SLOPE = float(np.float32(0.01))        # kLeaky = 0.01f, exactly
SMS = 148
FUSED_MAX_ROW, RANK_CAP, BWD2_CAP, FWD_CAP = 512, 1024, 6144, 12288
W = 0.75                               # deg_w (deg_b follows from the data)

# mode: "auto" (the Python dispatch), "two" (fused path switched off); epb: DGGB_FUSED_EPB
Dgg = namedtuple("Dgg", "graph h hard_k noise mode epb sat seed")
FirstK = namedtuple("FirstK", "graph k_only seed")


def _d(graph, h, hard_k=-1, noise=False, mode="auto", epb=None, sat=False, seed=0):
    return Dgg(graph, h, hard_k, noise, mode, epb, sat, seed)


PATHS = [
    # ---- fused, second generation (default) ----
    (_d("mixed", 64, seed=1), ["fused2_fwd<4,4>", "fused2_bwd<4,4>"]),
    (_d("mixed", 16, 3, seed=2), ["fused2_fwd<4,1>", "fused2_bwd<4,1>"]),
    (_d("blocks", 32, noise=True, epb=64, seed=3), ["fused2_fwd<4,2>", "fused2_bwd<4,2>"]),
    (_d("blocks", 128, 0, epb=64, seed=4), ["fused2_fwd<4,8>", "fused2_bwd<4,8>"]),
    (_d("mixed512", 256, seed=5), ["fused2_fwd<4,16>", "fused2_bwd<4,16>"]),
    (_d("mixed", 512, 1, noise=True, seed=6), ["fused2_fwd<4,32>", "fused2_bwd<4,32>"]),
    (_d("one", 4, seed=7), ["fused2_fwd<1,0>", "fused2_bwd<1,0>"]),
    (_d("mixed", 8, noise=True, seed=8), ["fused2_fwd<2,0>", "fused2_bwd<2,0>"]),
    (_d("blocks", 12, epb=64, seed=9), ["fused2_fwd<4,0>", "fused2_bwd<4,0>"]),
    (_d("mixed", 100, 600, seed=10), ["fused2_fwd<4,0>", "fused2_bwd<4,0>"]),
    (_d("mixed", 260, 1, noise=True, seed=29), ["fused2_fwd<4,0>", "fused2_bwd<4,0>"]),
    (_d("mixed", 64, sat=True, seed=11), ["fused2_fwd<4,4>", "fused2_bwd<4,4>"]),             # R == 1.0f ties
    # window > 12 288 (global re-read) and cap > 6 144: dgg_bwd_fused_kernel, > 1 024 rows per block
    (_d("wide", 20, epb=16000, seed=12), ["fused2_fwd<4,0>", "fused_bwd<4,0>"]),
    (_d("wide", 36, epb=16000, seed=28), ["fused2_fwd<4,0>", "fused_bwd<4,0>"]),
    # the largest second-generation backward window (epb + max_row = 6 138: 48 KB of scores and terms)
    (_d("wide", 64, epb=6080, seed=14), ["fused2_fwd<4,4>", "fused2_bwd<4,4>"]),
    # natural size, no override: the default grid's window exceeds 6 144 entries
    (_d("natural", 4, seed=13), ["fused2_fwd<1,0>", "fused_bwd<1,0>"]),
    # two blocks of ~10 000 entries (cap > 6 144, > 1 024 rows per block): every dgg_bwd_fused_kernel instantiation
    (_d("mixed512", 4, 1, noise=True, epb=16000, seed=20), ["fused2_fwd<1,0>", "fused_bwd<1,0>"]),
    (_d("mixed", 8, noise=True, epb=16000, seed=21), ["fused2_fwd<2,0>", "fused_bwd<2,0>"]),
    (_d("mixed", 16, 3, epb=16000, seed=22), ["fused2_fwd<4,1>", "fused_bwd<4,1>"]),
    (_d("mixed512", 32, epb=16000, seed=23), ["fused2_fwd<4,2>", "fused_bwd<4,2>"]),
    (_d("mixed", 64, 1, noise=True, epb=16000, seed=24), ["fused2_fwd<4,4>", "fused_bwd<4,4>"]),
    (_d("mixed512", 128, noise=True, epb=16000, seed=25), ["fused2_fwd<4,8>", "fused_bwd<4,8>"]),
    (_d("mixed", 256, epb=16000, seed=26), ["fused2_fwd<4,16>", "fused_bwd<4,16>"]),
    (_d("mixed512", 512, 0, epb=16000, seed=27), ["fused2_fwd<4,32>", "fused_bwd<4,32>"]),
    # ---- two launches ----
    (_d("hubs", 4, seed=30), ["score<1>", "row_rank", "long_rank[2]", "row_dk", "edge_grad<1>"]),
    (_d("hubs", 8, 3, seed=31), ["score<2>", "row_rank", "long_rank[3]", "edge_grad<2>"]),
    (_d("hubs", 64, noise=True, seed=32), ["score<4>", "row_rank", "long_rank[2]", "row_dk", "edge_grad<4>"]),
    (_d("hubs", 508, 0, noise=True, seed=33), ["score<4>", "row_rank", "long_rank[3]", "edge_grad<4>"]),
    (_d("hub513", 12, seed=34), ["score<4>", "row_rank", "row_dk", "edge_grad<4>"]),
    (_d("hub1024", 36, 5000, seed=35), ["score<4>", "row_rank", "edge_grad<4>"]),
    (_d("mixed", 16, mode="two", seed=36), ["score<4>", "row_rank", "row_dk", "edge_grad<4>"]),
    (_d("one", 8, mode="two", seed=37), ["score<2>", "row_rank", "row_dk", "edge_grad<2>"]),
    (_d("blocks", 4, 1, noise=True, mode="two", seed=38), ["score<1>", "row_rank", "edge_grad<1>"]),
    (_d("empty", 64, seed=39), ["row_rank"]),                                                   # no entries
    # ---- first-k ----
    (FirstK("hubs", False, 40), ["firstk_fwd[0]", "long_rank[0]", "firstk_bwd"]),
    (FirstK("hubs", True, 41), ["firstk_fwd[1]", "long_rank[1]", "firstk_bwd"]),
    (FirstK("mixed512", False, 42), ["firstk_fwd[0]", "firstk_bwd"]),
    (FirstK("hub1024", True, 43), ["firstk_fwd[1]", "firstk_bwd"]),
    (FirstK("one", False, 44), ["firstk_fwd[0]", "firstk_bwd"]),
    (FirstK("empty", False, 45), []),
]


def _path_id(case):
    c, launches = case
    head = launches[0] if launches else "nolaunch"
    if isinstance(c, FirstK):
        return f"firstk-{c.graph}-{'konly' if c.k_only else 'kxp'}-{head}"
    extra = (f"-hk{c.hard_k}" if c.hard_k >= 0 else "") + ("-noise" if c.noise else "") + ("-sat" if c.sat else "")
    extra += f"-{c.mode}" + (f"-epb{c.epb}" if c.epb else "")
    return f"dgg-{c.graph}-h{c.h}{extra}-{head}"


# ---------------------------------------------------------------------------------------------------------------
# graphs
# ---------------------------------------------------------------------------------------------------------------
def _csr(n, row, col):
    k = torch.unique(row * n + col)
    row, col = k // n, k % n
    rowptr = torch.zeros(n + 1, dtype=torch.long)
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
    return rowptr, row, col


def _random_graph(n, max_deg, exact, seed, long_frac=0.0, fixed_deg=None):
    """Random rows of 1 .. max_deg entries (or fixed_deg), a fraction long_frac of rows with 33 .. 60 entries, the
    rows of ``exact`` with exactly that many distinct columns, self loops on 40 rows, and the twin nodes (n // 7,
    n // 7 + 1) together in 30 rows."""
    gen = torch.Generator().manual_seed(seed)
    if fixed_deg is not None:
        deg = torch.full((n,), fixed_deg, dtype=torch.long)
    else:
        deg = torch.randint(1, max_deg + 1, (n,), generator=gen)
        if long_frac:
            deg = torch.where(torch.rand(n, generator=gen) < long_frac, torch.randint(33, 61, (n,), generator=gen),
                              deg)
    deg[list(exact)] = 0
    row = torch.repeat_interleave(torch.arange(n), deg)
    col = torch.randint(0, n, (row.numel(),), generator=gen)
    free = torch.ones(n, dtype=torch.bool)
    free[list(exact)] = False
    cand = torch.nonzero(free).flatten()
    loops = cand[torch.randperm(cand.numel(), generator=gen)[:40]]
    tw = cand[torch.randperm(cand.numel(), generator=gen)[:30]]
    t1 = n // 7
    rows = [row, loops, tw, tw]
    cols = [col, loops, torch.full_like(tw, t1), torch.full_like(tw, t1 + 1)]
    for r, d in exact.items():
        rows.append(torch.full((d,), r, dtype=torch.long))
        cols.append(torch.randperm(n, generator=gen)[:d])
    return _csr(n, torch.cat(rows), torch.cat(cols))


def _blocks_graph(seed):
    """Entry count a multiple of 64 (with DGGB_FUSED_EPB = 64 every block owns exactly 64 entries): leading empty rows,
    runs of empty rows that start exactly at a block boundary (the walk-back of ``fused_row_range``), a 320-entry row
    whose span holds four block boundaries (four blocks own no row), rows of 1, 32, 33 and 64 entries, trailing empty
    rows.  The twins (n // 7, n // 7 + 1) share the 64-entry rows."""
    unit = [0, 0, 0] + [16] * 4 + [0] * 3 + [16] * 4 + [320] + [33, 31] + [1] * 64 + [0, 0] + [32, 32] + [5, 59] + [64]
    degs = unit * 4 + [0] * 40
    n = len(degs)
    assert sum(degs) % 64 == 0 and n >= 320
    gen = torch.Generator().manual_seed(seed)
    t1 = n // 7
    rows, cols = [], []
    for r, d in enumerate(degs):
        if d == 0:
            continue
        c = torch.randperm(n, generator=gen)[:d]
        if d == 64:
            c = torch.unique(torch.cat([c[:62], torch.tensor([t1, t1 + 1])]))
            c = torch.cat([c, torch.tensor([x for x in range(n) if x not in set(c.tolist())][:64 - c.numel()], dtype=torch.long)])
        if d == 16:
            c[0] = r                                      # self loops
            c = torch.unique(c)
            if c.numel() < 16:
                c = torch.cat([c, torch.tensor([x for x in range(n) if x not in set(c.tolist())][:16 - c.numel()],
                                                 dtype=torch.long)])
        rows.append(torch.full((d,), r, dtype=torch.long))
        cols.append(c)
    rowptr, row, col = _csr(n, torch.cat(rows), torch.cat(cols))
    assert torch.equal(rowptr[1:] - rowptr[:-1], torch.tensor(degs))
    return rowptr, row, col


def _base_exact(n):
    e = {0: 0, 1: 0, 2: 0, 3: 1, 4: 32, 5: 33, n // 3: 64, n - 1: 0, n - 2: 0, n - 3: 0}
    e.update({r: 0 for r in range(n // 2, n // 2 + 10)})
    return e


_GRAPHS = {}


def _graph(name):
    """(rowptr, row, col) int64 on the CPU."""
    if name in _GRAPHS:
        return _GRAPHS[name]
    if name == "mixed":
        g = _random_graph(3000, 12, _base_exact(3000), 1)
    elif name == "mixed512":
        g = _random_graph(3000, 12, {**_base_exact(3000), 100: 512, 101: 511}, 2)
    elif name == "hub513":
        g = _random_graph(3000, 12, {**_base_exact(3000), 10: 513}, 3)
    elif name == "hub1024":
        g = _random_graph(3000, 12, {**_base_exact(3000), 10: 1024, 11: 1000}, 4)
    elif name == "hubs":       # several hub rows: 1 025, 2 049, 2 500 and 4 100 entries
        g = _random_graph(5000, 12, {**_base_exact(5000), 7: 1025, 8: 2500, 2000: 4100, 4000: 2049}, 5)
    elif name == "wide":
        g = _random_graph(20000, 12, _base_exact(20000), 6, long_frac=0.05)
    elif name == "natural":
        n = 1_000_000
        g = _random_graph(n, 8, {0: 0, n // 2: 0, n - 1: 0}, 7, fixed_deg=8)
    elif name == "blocks":
        g = _blocks_graph(8)
    elif name == "one":
        g = (torch.tensor([0, 1]), torch.zeros(1, dtype=torch.long), torch.zeros(1, dtype=torch.long))
    elif name == "empty":
        g = (torch.zeros(51, dtype=torch.long), torch.zeros(0, dtype=torch.long), torch.zeros(0, dtype=torch.long))
    else:
        raise KeyError(name)
    _GRAPHS[name] = g
    return g


def _info(name):
    rowptr = _graph(name)[0]
    deg = rowptr[1:] - rowptr[:-1]
    return int(rowptr[-1]), int(deg.max()) if deg.numel() else 0, deg


# ---------------------------------------------------------------------------------------------------------------
# the dispatch restated
# ---------------------------------------------------------------------------------------------------------------
def _lanes(h):
    L = 1
    while L < 32 and 16 * L < h:
        L *= 2
    t = -(-h // (4 * L))
    return L, (1 if t == 1 else (2 if t == 2 else 4))


def _inst(h):
    L, t = _lanes(h)
    return f"<4,{L}>" if h == 16 * L else f"<{t},0>"


def _bwd2_fits(nnz, max_row, epb_env):
    """cap = epb + max_row <= 6 144 for every occupancy the grid could see (1 .. 8 blocks of 256 threads per SM)."""
    min_epb = epb_env if (epb_env or 0) >= 1 else 128
    b = -(-nnz // min_epb)
    if b <= SMS:
        lo = hi = -(-nnz // b)
    else:
        lo, hi = -(-nnz // (SMS * 8)), -(-nnz // SMS)
    assert (hi + max_row <= BWD2_CAP) or (lo + max_row > BWD2_CAP), "the dispatch depends on the occupancy"
    return lo + max_row <= BWD2_CAP


def _expected(c):
    nnz, mx, _ = _info(c.graph)
    if isinstance(c, FirstK):
        if nnz == 0:
            return []
        m = 1 if c.k_only else 0
        return [f"firstk_fwd[{m}]"] + ([f"long_rank[{m}]"] if mx > RANK_CAP else []) + ["firstk_bwd"]
    t = _lanes(c.h)[1]
    if c.mode != "two" and 0 < mx <= FUSED_MAX_ROW and nnz > 0:
        inst = _inst(c.h)
        return ["fused2_fwd" + inst, ("fused2_bwd" if _bwd2_fits(nnz, mx, c.epb) else "fused_bwd") + inst]
    out = ([f"score<{t}>"] if nnz > 0 else []) + ["row_rank"]
    if mx > RANK_CAP:
        out.append(f"long_rank[{3 if c.hard_k >= 0 else 2}]")
    if nnz > 0:
        out += (["row_dk"] if c.hard_k < 0 else []) + [f"edge_grad<{t}>"]
    return out


def _epb_window(c):
    """(epb, fwd cap, rows per block at most) of a fused case whose grid does not depend on the occupancy."""
    nnz, mx, _ = _info(c.graph)
    min_epb = c.epb or 128
    b = -(-nnz // min_epb)
    assert b <= SMS
    epb = -(-nnz // b)
    return epb, min(epb + mx, FWD_CAP)


def test_path_table_reaches_every_instantiation():
    for c, launches in PATHS:
        assert _expected(c) == launches, (c, _expected(c), launches)
    got = {name.split("[")[0] for _, launches in PATHS for name in launches}
    insts = ["<4,1>", "<4,2>", "<4,4>", "<4,8>", "<4,16>", "<4,32>", "<1,0>", "<2,0>", "<4,0>"]
    want = {f"score<{t}>" for t in (1, 2, 4)} | {f"edge_grad<{t}>" for t in (1, 2, 4)}
    want |= {"row_rank", "long_rank", "row_dk", "firstk_fwd", "firstk_bwd"}
    want |= {f + i for f in ("fused2_fwd", "fused2_bwd", "fused_bwd") for i in insts}
    assert len(want) == 38
    assert got == want, (want - got, got - want)
    modes = {name for _, launches in PATHS for name in launches if "[" in name}
    assert modes == {"long_rank[0]", "long_rank[1]", "long_rank[2]", "long_rank[3]", "firstk_fwd[0]",
                     "firstk_fwd[1]"}
    # the runtime-L kernels at several h that are not 16 L
    assert {c.h for c, _ in PATHS if isinstance(c, Dgg) and c.mode != "two" and _inst(c.h) == "<4,0>"} >= {
        12, 20, 36, 100, 260}
    # row lengths and placements
    lens = set()
    for name in {c.graph for c, _ in PATHS}:
        lens |= set(_info(name)[2].tolist())
    assert {0, 1, 32, 33, 512, 513, 1024, 1025} <= lens
    assert any(d > 2048 and d % 256 for d in lens)
    hub_rows = (_info("hubs")[2] > RANK_CAP).sum()
    assert hub_rows >= 3
    for name in ("mixed", "blocks", "hubs"):
        deg = _info(name)[2]
        assert deg[0] == 0 and deg[-1] == 0 and (deg[len(deg) // 2:] == 0).any()
    # blocks of 64 entries: empty runs that start on a boundary, blocks that own no row
    rowptr = _graph("blocks")[0]
    empty_at = rowptr[:-1][(rowptr[1:] - rowptr[:-1]) == 0]
    assert ((empty_at % 64 == 0) & (empty_at > 0) & (empty_at < rowptr[-1])).any()
    starts = set((rowptr[:-1] // 64).tolist())
    assert len(set(range(int(rowptr[-1]) // 64)) - starts) >= 4
    # modes
    dggs = [c for c, _ in PATHS if isinstance(c, Dgg) and _info(c.graph)[0] > 0]
    assert {c.hard_k for c in dggs if c.hard_k >= 0 and c.hard_k < 600} == {0, 1, 3}
    assert any(c.hard_k >= _info(c.graph)[1] for c in dggs)
    assert {(c.noise, c.hard_k >= 0) for c in dggs} == {(False, False), (False, True), (True, False), (True, True)}
    assert any(c.sat for c in dggs)
    # large windows reach both backward kernels by the window rule: dgg_bwd_fused2_kernel up to 6 144 entries (big2
    # below), dgg_bwd_fused_kernel above in every instantiation, each overridden grid with > 1 024 rows in one block
    big1 = [c for c, launches in PATHS if isinstance(c, Dgg) and launches[-1].startswith("fused_bwd")]
    assert {_inst(c.h) for c in big1} == set(insts)
    for c in big1:
        if c.epb:
            epb, _ = _epb_window(c)
            assert epb + _info(c.graph)[1] > BWD2_CAP
            assert int(torch.bincount(_graph(c.graph)[0][:-1] // epb).max()) > RANK_CAP
    # fused2 forward re-read (epb + max_row > 12 288)
    wide = [c for c in dggs if c.graph == "wide" and c.epb == 16000]
    # windows beyond 48 KB of shared memory, the default per-block limit: forward 12 288 floats, backward 2 x 6 138
    big2 = [c for c, launches in PATHS if isinstance(c, Dgg) and c.epb and launches[-1].startswith("fused2_bwd")]
    assert any(8 * (_epb_window(c)[0] + _info(c.graph)[1]) > 48 * 1024 - 2048 for c in big2)
    assert any(4 * _epb_window(c)[1] == 48 * 1024 for c in wide)
    rowptr, _, _ = _graph("wide")
    deg = rowptr[1:] - rowptr[:-1]
    for c in wide:
        epb, _ = _epb_window(c)
        assert epb + _info(c.graph)[1] > FWD_CAP
        blk = rowptr[:-1] // epb                         # the block that owns each row
        nb = int(blk.max()) + 1
        assert int(torch.bincount(blk, minlength=nb).max()) > RANK_CAP
        assert int(torch.bincount(blk[deg > 32], minlength=nb).max()) > 32


# ---------------------------------------------------------------------------------------------------------------
# test graphs on the device and the fp64 reference
# ---------------------------------------------------------------------------------------------------------------
class G:
    def __init__(self, name):
        from dgg_b200 import CSRGraph

        rowptr, row, col = _graph(name)
        self.n, self.nnz = rowptr.numel() - 1, int(rowptr[-1])
        self.csr = CSRGraph(self.n, rowptr.to(torch.int32).cuda(), col.to(torch.int32).cuda())
        self.rowptr, self.row, self.col = rowptr.cuda(), row.cuda(), col.cuda()
        self.deg = (rowptr[1:] - rowptr[:-1]).double().cuda()
        self.indeg = torch.bincount(col, minlength=self.n).double().cuda()
        self.max_row = int(self.deg.max()) if self.n else 0

    def row_sum(self, v):
        return torch.zeros(self.n, dtype=v.dtype, device=v.device).index_add_(0, self.row, v)


def _within(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = int(torch.where(bad, (err - bound) / bound.clamp_min(1e-300), -1.0).reshape(-1).argmax())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} entries beyond the bound; worst at flat "
                             f"index {i}: got {float(got.reshape(-1)[i])}, want {float(want.reshape(-1)[i])}, "
                             f"bound {float(bound.reshape(-1)[i])}")


def _stable_rank(g, vals):
    """0-based descending rank inside each row, ties by lower position (= lower column) first."""
    o = torch.sort(vals, descending=True, stable=True).indices
    o = o[torch.sort(g.row[o], stable=True).indices]
    pos = torch.empty_like(o)
    pos[o] = torch.arange(o.numel(), device=o.device)
    return pos - g.rowptr[g.row], o


def _inputs(c, g):
    """fp32 y, be, noise and the upstream gradient of case c (y on the dyadic grid, twins equal)."""
    h, n = c.h, g.n
    gen = torch.Generator().manual_seed(1000 + c.seed)
    q = 2.0 ** -math.ceil(math.log2(0.7 * h)) * (16.0 if c.sat else 1.0)
    m = torch.randint(-8, 9, (n, h), generator=gen) + torch.randint(-4, 5, (n, 1), generator=gen)
    if n > 8:
        m[n // 7 + 1] = m[n // 7]
    y = m.float() * q
    be = (torch.randint(-4, 4, (h,), generator=gen).float() + 0.5) * q
    noise = (torch.rand(g.nnz, generator=gen) * 2 - 1) if c.noise else None
    gout = torch.randn(g.nnz, generator=gen)
    return y.cuda(), be.cuda(), None if noise is None else noise.cuda(), gout.cuda()


class Fwd64:
    """fp64 forward up to s (independent of deg_w / deg_b) with bounds; deg_b is then chosen from s."""

    def __init__(self, g, y, be, noise):
        self.g = g
        yd, bd = y.double(), be.double()
        pre = yd[g.row] - yd[g.col] + bd
        assert bool((pre.abs() > 0).all())
        self.lg = torch.where(pre > 0, 1.0, SLOPE).to(torch.float64)
        lz = pre * self.lg
        h = y.shape[1]
        self.z = lz.sum(1)
        zb = U * (h + 4) * lz.abs().sum(1)
        self.R1 = torch.sigmoid(self.z)
        self.R1b = self.R1 * (1 - self.R1) * zb + 6 * U * self.R1
        if noise is not None:
            x2 = self.R1 + noise.double()
            self.R = torch.sigmoid(x2)
            self.Rb = self.R * (1 - self.R) * (self.R1b + U * x2.abs()) + 6 * U * self.R
        else:
            self.R, self.Rb = self.R1, self.R1b
        self.s = g.row_sum(self.R)
        self.sb = g.row_sum(self.Rb) + U * (g.deg + 2) * self.s

    def choose_b(self, w=W):
        """deg_b (an fp32 value) such that w s + b keeps clear of 0 on every row and takes both signs."""
        g = self.g
        v = torch.unique(self.s[g.deg > 0]) if g.nnz else self.s[:0]
        if v.numel() == 0:
            mid = 0.25
        elif v.numel() == 1:
            mid = float(v[0]) / 2
        else:
            lo = int(0.005 * (v.numel() - 1))
            hi = max(int(0.995 * (v.numel() - 1)), lo + 1)
            gaps = v[lo + 1:hi + 1] - v[lo:hi]
            i = lo + int(gaps.argmax())
            mid = float(v[i] + v[i + 1]) / 2
        b = float(np.float32(-w * mid))
        self.w, self.b = w, b
        kin = w * self.s + b
        self.kin_b = abs(w) * self.sb + 2 * U * ((w * self.s).abs() + kin.abs())
        assert bool((kin.abs() > 4 * self.kin_b).all()), "w s + b too close to 0 on some row"
        if g.nnz and g.n > 1:
            assert bool((kin > 0).any()) and bool((kin < 0).any())
        self.lr = torch.where(kin > 0, 1.0, SLOPE).to(torch.float64)
        self.k = kin * self.lr
        self.kb = self.lr * self.kin_b + U * self.k.abs()
        return b


def _ref64(g, y, be, w, b, noise, rank, hard_k):
    """fp64 out of the DGG edge op at the leaves (y, be, w, b), with the given ranks held fixed."""
    pre = y[g.row] - y[g.col] + be
    z = torch.where(pre > 0, pre, SLOPE * pre).sum(1)
    R = torch.sigmoid(z)
    if noise is not None:
        R = torch.sigmoid(R + noise.double())
    if hard_k >= 0:
        return R * (rank < hard_k).double()
    s = g.row_sum(R)
    kin = w * s + b
    k = torch.where(kin > 0, kin, SLOPE * kin)
    th = torch.tanh(rank.double() - k[g.row])
    return R * (2.0 - 0.5 * (1.0 + th))


def check_forward(g, f, hard_k, R, rank, k, s, out, sat=False):
    """Self-consistency (exact up to tanhf) and the fp64 checks of R, s, k, rank."""
    E = g.nnz
    want_rank, _ = _stable_rank(g, R)
    assert torch.equal(rank.long(), want_rank), "rank is not the stable descending rank of the kernel's own R"
    if hard_k >= 0:
        assert torch.equal(out, torch.where(rank < hard_k, R, torch.zeros_like(R))), "hard-k out"
    elif E:
        t = rank.double() - k.double()[g.row]
        want = R.double() * (2.0 - 0.5 * (1.0 + torch.tanh(t)))
        _within(out, want, U * R.double() * (t.abs() + 12), "out (from the kernel's own R, rank, k)")
    _within(R, f.R, 2 * f.Rb, "R")
    _within(s, f.s, 2 * f.sb, "s")
    _within(k, f.k, 2 * f.kb, "k")
    if E == 0:
        return
    r64, o = _stable_rank(g, f.R)
    sv, sr, sbd = f.R[o], g.row[o], f.Rb[o]
    same = sr[1:] == sr[:-1]
    sep = (sv[:-1] - sv[1:]) > (sbd[:-1] + sbd[1:])
    clear = torch.ones(E, dtype=torch.bool, device=R.device)
    clear[:-1] &= ~same | sep
    clear[1:] &= ~same | sep
    ok = torch.empty_like(clear)
    ok[o] = clear
    assert torch.equal(rank.long()[ok], r64[ok]), "rank differs from the fp64 rank on a well-separated entry"
    if not sat:
        assert float(ok.float().mean()) > 0.5, float(ok.float().mean())


def grad_bounds(g, f, hard_k, noise, rank, gout, yd, bed):
    """fp64 gradients at the kernel's ranks, and their bounds: (dy, dbe, dw, db), (dyb, dbeb, dwb, dbb)."""
    ld = [yd.clone().requires_grad_(True), bed.clone().requires_grad_(True),
          torch.tensor(f.w, dtype=torch.float64, device=yd.device, requires_grad=True),
          torch.tensor(f.b, dtype=torch.float64, device=yd.device, requires_grad=True)]
    if g.nnz == 0:
        z = torch.zeros_like
        return (z(yd), z(bed), 0.0, 0.0), (z(yd), z(bed), 0.0, 0.0)
    out = _ref64(g, ld[0], ld[1], ld[2], ld[3], noise, rank, hard_k)
    grads = torch.autograd.grad((out * gout.double()).sum(), ld, allow_unused=True)
    dy, dbe, dw, db = [0.0 if q is None else q.detach() for q in grads]
    ga, R, Rb, R1, R1b = gout.double().abs(), f.R, f.Rb, f.R1, f.R1b
    r = rank.double()
    if hard_k >= 0:
        dR = gout.double() * (rank < hard_k).double()
        dRb = torch.zeros_like(dR)
        dwb = dbb = 0.0
    else:
        t = r - f.k[g.row]
        th = torch.tanh(t)
        sech2 = 1 - th * th
        kb = f.kb[g.row]
        T = gout.double() * R * 0.5 * sech2
        Tb = ga * 0.5 * (Rb * sech2 + R * (2 * th.abs() * (sech2 * kb + 4 * U + sech2 * U * t.abs()) + 4 * U)) \
            + 6 * U * T.abs()
        dk = g.row_sum(T)
        dkb = g.row_sum(Tb) + U * (g.deg + 4) * g.row_sum(T.abs())
        ds = dk * f.lr * f.w
        dsb = f.lr * abs(f.w) * dkb + 3 * U * ds.abs()
        dwb = float((f.lr * (dkb * f.s.abs() + dk.abs() * f.sb)).sum() + U * (g.n + 8) * (dk * f.lr * f.s).abs().sum())
        dbb = float((f.lr * dkb).sum() + U * (g.n + 8) * (dk * f.lr).abs().sum())
        fk1 = 2.0 - 0.5 * (1.0 + th)
        fkb = 0.5 * (sech2 * kb + 4 * U + sech2 * U * t.abs()) + 4 * U
        dR = gout.double() * fk1 + ds[g.row]
        dRb = ga * fkb + dsb[g.row] + 2 * U * ((gout.double() * fk1).abs() + ds[g.row].abs())
    if noise is not None:
        q2 = R * (1 - R)
        dRb = dRb * q2 + dR.abs() * (1 - 2 * R).abs() * Rb + 3 * U * (dR * q2).abs()
        dR = dR * q2
    q1 = R1 * (1 - R1)
    dz = dR * q1
    dzb = dRb * q1 + dR.abs() * (1 - 2 * R1).abs() * R1b + 3 * U * dz.abs()
    dpa = dz.abs()[:, None] * f.lg                      # |d pre|
    dpb = dzb[:, None] * f.lg + U * dpa
    off = g.row != g.col
    n, h = yd.shape
    node = torch.zeros(n, h, dtype=torch.float64, device=yd.device)
    dyb = node.index_add(0, g.row[off], dpb[off]).index_add_(0, g.col[off], dpb[off])
    touch = node.index_add(0, g.row[off], dpa[off]).index_add_(0, g.col[off], dpa[off])
    dyb = dyb + U * (g.deg + g.indeg + 8)[:, None] * touch
    dbeb = dpb.sum(0) + U * (g.nnz + 16) * dpa.sum(0)
    return (dy, dbe, dw, db), (2 * dyb, 2 * dbeb, 2 * dwb, 2 * dbb)


def check_grads(got, ref, bounds, hard_k):
    (dy, dbe, dw, db), (dyb, dbeb, dwb, dbb) = ref, bounds
    gy, gbe, gw, gb = got
    _within(gy, dy, dyb, "dy")
    _within(gbe, dbe, dbeb, "dbe")
    if hard_k >= 0:
        assert float(gw.reshape(-1)[0]) == 0.0 and float(gb.reshape(-1)[0]) == 0.0, "hard mode: d deg_w / d deg_b"
    else:
        dev = gy.device
        _within(gw.reshape(1), torch.tensor([float(dw)], dtype=torch.float64, device=dev),
                torch.tensor([dwb], dtype=torch.float64, device=dev), "d deg_w")
        _within(gb.reshape(1), torch.tensor([float(db)], dtype=torch.float64, device=dev),
                torch.tensor([dbb], dtype=torch.float64, device=dev), "d deg_b")


def _set_path(monkeypatch, c):
    from dgg_b200 import functional as K

    monkeypatch.setattr(K, "_FUSED_MAX_ROW", 0 if c.mode == "two" else FUSED_MAX_ROW)
    if c.epb:
        monkeypatch.setenv("DGGB_FUSED_EPB", str(c.epb))
    else:
        monkeypatch.delenv("DGGB_FUSED_EPB", raising=False)


def _prepare(c):
    g = G(c.graph)
    y, be, noise, gout = _inputs(c, g)
    f = Fwd64(g, y, be, noise)
    b = f.choose_b()
    return g, y, be, noise, gout, f, b


def _run_dgg(c, g, y, be, noise, gout, b, monkeypatch, backward=True):
    from dgg_b200 import functional as K

    _set_path(monkeypatch, c)
    leaves = [y.clone().requires_grad_(True), be.clone().requires_grad_(True),
              torch.full((1, 1), W, device="cuda", requires_grad=True),
              torch.full((1,), b, device="cuda", requires_grad=True)]
    out, k, R, rank = K.dgg_edge(*leaves, g.csr, noise=noise, hard_k=c.hard_k)
    s = out.grad_fn.saved_tensors[7]
    if backward:
        (out * gout).sum().backward()
    return out.detach(), k, R, rank, s, leaves


@gpu
@pytest.mark.parametrize("case", [c for c in PATHS if isinstance(c[0], Dgg)],
                         ids=[_path_id(c) for c in PATHS if isinstance(c[0], Dgg)])
def test_dgg_path_matches_fp64(case, monkeypatch):
    c, _ = case
    g, y, be, noise, gout, f, b = _prepare(c)
    out, k, R, rank, s, leaves = _run_dgg(c, g, y, be, noise, gout, b, monkeypatch)
    check_forward(g, f, c.hard_k, R, rank, k, s, out, sat=c.sat)
    if g.n > 8 and noise is None and g.nnz:                     # the twins: equal R, the lower column first
        t1 = g.n // 7
        row, col, Rc, rc = g.row.cpu(), g.col.cpu(), R.cpu(), rank.cpu()
        away = (row != t1) & (row != t1 + 1)
        e1 = {int(row[e]): int(e) for e in torch.nonzero((col == t1) & away).flatten()}
        e2 = {int(row[e]): int(e) for e in torch.nonzero((col == t1 + 1) & away).flatten()}
        pairs = [(e1[r], e2[r]) for r in e1 if r in e2]
        assert len(pairs) >= 3
        for a, bb in pairs:
            assert float(Rc[a]) == float(Rc[bb]) and int(rc[a]) < int(rc[bb])
    ref, bounds = grad_bounds(g, f, c.hard_k, noise, rank, gout, y.double(), be.double())
    check_grads([q.grad for q in leaves], ref, bounds, c.hard_k)


# ---------------------------------------------------------------------------------------------------------------
# first-k
# ---------------------------------------------------------------------------------------------------------------
def _firstk_inputs(c, g):
    gen = torch.Generator().manual_seed(2000 + c.seed)
    score = torch.randint(1, 200, (g.nnz,), generator=gen).float() / 256.0        # dyadic, many exact ties
    k = torch.rand(g.n, generator=gen) * (g.deg.cpu().float() + 2)
    gout = torch.randn(g.nnz, generator=gen)
    return score.cuda(), k.cuda(), gout.cuda()


def _run_firstk(c, g, score, k, gout):
    from dgg_b200 import functional as K

    sc = score.clone().requires_grad_(not c.k_only)
    kk = k.clone().requires_grad_(True)
    out, rank = K.row_firstk(sc, kk, g.csr, k_only=c.k_only, return_rank=True)
    (out * gout).sum().backward()
    return out.detach(), rank, sc, kk


@gpu
@pytest.mark.parametrize("case", [c for c in PATHS if isinstance(c[0], FirstK)],
                         ids=[_path_id(c) for c in PATHS if isinstance(c[0], FirstK)])
def test_firstk_path_matches_fp64(case):
    """rank: the stable descending rank of the scores, exactly; out, dscore and dk against fp64 at those ranks."""
    c, _ = case
    g = G(c.graph)
    score, k, gout = _firstk_inputs(c, g)
    out, rank, sc, kk = _run_firstk(c, g, score, k, gout)
    want_rank, _ = _stable_rank(g, score)
    assert torch.equal(rank.long(), want_rank)
    r = rank.double()
    t = r - k.double()[g.row]
    th = torch.tanh(t)
    sech2 = 1 - th * th
    fk = 1.0 - 0.5 * (1.0 + th)
    sd = score.double()
    fkb = 0.5 * (4 * U + sech2 * U * t.abs()) + 3 * U
    if c.k_only:
        _within(out, fk, fkb, "out")
        assert sc.grad is None
        terms = gout.double() * 0.5 * sech2
        tb = gout.double().abs() * 0.5 * (2 * th.abs() * (4 * U + sech2 * U * t.abs()) + 4 * U) + 4 * U * terms.abs()
    else:
        _within(out, sd * fk, sd * fkb + U * (sd * fk).abs(), "out")
        gfk = gout.double() * fk
        _within(sc.grad, gfk, gout.double().abs() * fkb + U * gfk.abs(), "dscore")
        terms = gout.double() * sd * 0.5 * sech2
        tb = (gout.double() * sd).abs() * 0.5 * (2 * th.abs() * (4 * U + sech2 * U * t.abs()) + 4 * U) \
            + 4 * U * terms.abs()
    dk = g.row_sum(terms)
    _within(kk.grad, dk, 2 * (g.row_sum(tb) + U * (g.deg + 4) * g.row_sum(terms.abs())), "dk")


# ---------------------------------------------------------------------------------------------------------------
# dispatch against the profiler
# ---------------------------------------------------------------------------------------------------------------
_SHORT = {"dgg_edge_score_kernel": "score", "dgg_row_rank_kernel": "row_rank", "long_row_rank_kernel": "long_rank",
          "dgg_row_dk_kernel": "row_dk", "dgg_edge_grad_kernel": "edge_grad", "row_firstk_fwd_kernel": "firstk_fwd",
          "row_firstk_bwd_kernel": "firstk_bwd", "dgg_fwd_fused2_kernel": "fused2_fwd",
          "dgg_bwd_fused2_kernel": "fused2_bwd", "dgg_bwd_fused_kernel": "fused_bwd"}


def _kernel_launches(trace_path):
    import json
    import re

    with open(trace_path) as fh:
        ev = json.load(fh)["traceEvents"]
    names = []
    for e in sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        m = re.search(r"\b(\w+_kernel)\b(<[^>]*>)?", e["name"])
        if m and m.group(1) in _SHORT:
            t = "" if m.group(2) is None else "<" + ",".join(re.findall(r"\d+", m.group(2))) + ">"
            names.append(_SHORT[m.group(1)] + t)
    return names


@gpu
def test_dispatch_launches_the_tabled_kernels(monkeypatch, tmp_path):
    """The profiler's kernel names, in launch order, are the table's (so the table is the dispatch, not a guess)."""
    from torch.profiler import ProfilerActivity, profile

    runs = []
    for c, _ in PATHS:
        if isinstance(c, Dgg):
            g, y, be, noise, gout, _, b = _prepare(c)
            runs.append((c, g, y, be, noise, gout, b))
        else:
            g = G(c.graph)
            runs.append((c, g) + _firstk_inputs(c, g))
    for run in runs:
        run[1].csr.erow                                  # built before the trace starts
    want = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # A profiler session that is not the process's first can lose its first few kernel records (2 or 3 of
        # them late in a full GPU test session): untracked kernels absorb the loss before the tabled launches.
        for _ in range(32):
            torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        for run, (_, launches) in zip(runs, PATHS):
            c = run[0]
            if isinstance(c, Dgg):
                _run_dgg(c, *run[1:], monkeypatch)
            else:
                _run_firstk(c, *run[1:])
            want += [name.split("[")[0] for name in launches]
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(tmp_path / "trace.json"))
    assert _kernel_launches(tmp_path / "trace.json") == want


# ---------------------------------------------------------------------------------------------------------------
# fused against two launches, inference against training, a second backward
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("graph,h,mode,epb", [("mixed", 64, "auto", None), ("blocks", 12, "auto", 64),
                                              ("mixed512", 8, "auto", None), ("wide", 36, "auto", 16000),
                                              ("wide", 100, "auto", 16000), ("one", 4, "auto", None)])
def test_fused_R_and_rank_equal_two_launch_bit_for_bit(graph, h, mode, epb, monkeypatch):
    """The fused kernels compute each R exactly as the score kernel does, and the rank is a count: both are the
    two-launch results bit for bit (s, k and out differ by the order of the row sums)."""
    c = _d(graph, h, mode=mode, epb=epb, seed=50)
    g, y, be, noise, gout, f, b = _prepare(c)
    fa = _run_dgg(c, g, y, be, noise, gout, b, monkeypatch, backward=False)
    fb = _run_dgg(c._replace(mode="two"), g, y, be, noise, gout, b, monkeypatch, backward=False)
    assert torch.equal(fa[2], fb[2]) and torch.equal(fa[3], fb[3])


@gpu
@pytest.mark.parametrize("graph,h,hard_k", [("mixed", 64, -1), ("blocks", 20, 3), ("hubs", 16, -1)])
def test_inference_forward_and_second_backward(graph, h, hard_k, monkeypatch):
    """A forward without autograd (no zero_ws to clear) equals the training forward bit for bit; a second backward
    through the same node (its buffer no longer cleared by the forward) gives the first one's gradients."""
    from dgg_b200 import functional as K

    c = _d(graph, h, hard_k, epb=64 if graph == "blocks" else None, seed=60)
    g, y, be, noise, gout, f, b = _prepare(c)
    _set_path(monkeypatch, c)
    leaves = [y.clone().requires_grad_(True), be.clone().requires_grad_(True),
              torch.full((1, 1), W, device="cuda", requires_grad=True),
              torch.full((1,), b, device="cuda", requires_grad=True)]
    train = K.dgg_edge(*leaves, g.csr, hard_k=hard_k)
    with torch.no_grad():
        infer = K.dgg_edge(*[q.detach() for q in leaves], g.csr, hard_k=hard_k)
    for a, bb in zip(train, infer):
        assert torch.equal(a.detach(), bb)
    loss = (train[0] * gout).sum()
    first = torch.autograd.grad(loss, leaves, retain_graph=True)
    second = torch.autograd.grad(loss, leaves)
    ref, bounds = grad_bounds(g, f, hard_k, None, train[3], gout, y.double(), be.double())
    check_grads(first, ref, bounds, hard_k)
    check_grads(second, ref, bounds, hard_k)


# ---------------------------------------------------------------------------------------------------------------
# entry points called directly
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("path", ["fused2", "fused2-misaligned-dbe", "large-window", "fused-unmasked", "two"])
def test_backward_entry_points_accumulate(path, monkeypatch):
    """dy, dbe and ddeg pre-filled with random values come back as the pre-fill plus the gradient ("accumulated
    into"); ds_ws pre-filled with NaN does not leak.  The masked fused backward runs dgg_bwd_fused2_kernel on the
    default grid (with a dbe that is not 16-byte aligned: its scalar-atomic flush) and dgg_bwd_fused_kernel for a
    window above 6 144 entries (> 1 024 rows per block: ds read back from ds_ws); the unmasked fused entry point and
    the two-launch one run dggb_dgg_edge_bwd."""
    from dgg_b200._lib import check, lib, p, stream
    from tests.test_gpu_dgg_edge_mask import _fwd

    c = _d("mixed", 64, epb=16000 if path == "large-window" else None, seed=70)
    g, y, be, noise, gout, f, b = _prepare(c)
    _set_path(monkeypatch, c)
    assert _bwd2_fits(g.nnz, g.max_row, c.epb) == (path != "large-window")
    R, rank, s, k, out, mask, _ = _fwd(g, y, be, b, None, -1, masked=True)
    ref, bounds = grad_bounds(g, f, -1, None, rank, gout, y.double(), be.double())
    gen = torch.Generator().manual_seed(71)
    n, h = y.shape
    pre_y = torch.randn(n, h, generator=gen).cuda()
    pre_b = torch.randn(h + 1, generator=gen).cuda()
    pre_d = torch.randn(2, generator=gen).cuda()
    dy, ddeg = pre_y.clone(), pre_d.clone()
    dbe_buf = pre_b.clone()
    dbe = dbe_buf[1:] if path.endswith("misaligned-dbe") else dbe_buf[:h]
    assert (dbe.data_ptr() % 16 == 0) != path.endswith("misaligned-dbe")
    pre_dbe = dbe.clone()
    ds_ws = torch.full((n,), float("nan"), device="cuda")
    wt, bt = torch.full((1,), W, device="cuda"), torch.full((1,), b, device="cuda")
    head = (p(g.csr.rowptr), p(g.csr.erow), p(g.csr.col), n, g.nnz)
    fwd_out = (p(R), p(rank), p(s), p(k))
    grads = (p(gout), p(ds_ws), p(dy), p(dbe), p(ddeg), stream())
    if path == "two":
        check(lib().dggb_dgg_edge_bwd(*head, h, p(y), p(be), p(wt), p(bt), None, -1, *fwd_out, *grads), "dgg_edge_bwd")
    elif path == "fused-unmasked":
        check(lib().dggb_dgg_edge_bwd_fused(*head, g.max_row, h, p(y), p(be), p(wt), p(bt), None, -1, *fwd_out,
                                            *grads), "dgg_edge_bwd_fused")
    else:
        check(lib().dggb_dgg_edge_bwd_fused_mask(*head, g.max_row, h, p(wt), p(bt), None, -1, *fwd_out, p(mask), None,
                                                 *grads), "dgg_edge_bwd_fused_mask")
    torch.cuda.synchronize()
    (dy64, dbe64, dw64, db64), (dyb, dbeb, dwb, dbb) = ref, bounds

    def acc(got, pre, want, bound, what):
        pre = pre.double()
        _within(got, pre + want, bound + 2 * U * (pre.abs() + (pre + want).abs()), what)

    acc(dy, pre_y, dy64, dyb, "dy (accumulated)")
    acc(dbe, pre_dbe, dbe64, dbeb, "dbe (accumulated)")
    dev = dy.device
    acc(ddeg, pre_d, torch.tensor([float(dw64), float(db64)], dtype=torch.float64, device=dev),
        torch.tensor([dwb, dbb], dtype=torch.float64, device=dev), "ddeg (accumulated)")
    nb = 0 if path.endswith("misaligned-dbe") else h             # the float next to dbe stays as it was
    assert float(dbe_buf[nb]) == float(pre_b[nb])


@gpu
def test_long_rows_without_long_ws_match_the_listed_path():
    """long_ws = NULL: a warp sweeps its hub row (1 025 .. 4 100 entries) straight from global memory; with the list
    the grid-wide kernel ranks it.  Both give the same ranks and values (dggb_dgg_edge_fwd and dggb_row_firstk_fwd)."""
    from dgg_b200._lib import check, lib, p, stream

    c = _d("hubs", 16, seed=80)
    g, y, be, noise, gout, f, b = _prepare(c)
    assert g.max_row > 2000
    n, E = g.n, g.nnz
    wt = torch.full((1,), W, device="cuda")
    bt = torch.full((1,), b, device="cuda")
    res = []
    for listed in (True, False):
        R, out = torch.empty(E, device="cuda"), torch.empty(E, device="cuda")
        rank = torch.empty(E, dtype=torch.int32, device="cuda")
        s, k = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
        ws = torch.zeros(n + 1, dtype=torch.int32, device="cuda") if listed else None
        check(lib().dggb_dgg_edge_fwd(p(g.csr.rowptr), p(g.csr.erow), p(g.csr.col), n, E, 16, p(y), p(be), p(wt),
                                      p(bt), None, -1, p(R), p(rank), p(s), p(k), p(out), p(ws), stream()), "fwd")
        check_forward(g, f, -1, R, rank, k, s, out)
        score, kf, _ = _firstk_inputs(FirstK("hubs", False, 81), g)
        fr, fo = torch.empty(E, dtype=torch.int32, device="cuda"), torch.empty(E, device="cuda")
        ws = torch.zeros(n + 1, dtype=torch.int32, device="cuda") if listed else None
        check(lib().dggb_row_firstk_fwd(p(g.csr.rowptr), n, p(score), p(kf), 0, p(fr), p(fo), p(ws), stream()),
              "firstk")
        res.append((R, rank, s, k, out, fr, fo))
    a, bb = res
    for i in (0, 1, 2, 3, 5):
        assert torch.equal(a[i], bb[i]), i
    for i in (4, 6):           # one formula in two kernels: a contraction may differ by an ulp
        _within(a[i], bb[i].double(), 4 * U * bb[i].double().abs(), "out")


@gpu
def test_graph_with_no_entries(monkeypatch):
    """K.dgg_edge, K.row_firstk and dgm.DGG on a graph without entries: empty outputs, k = LeakyReLU(deg_b) on every
    row, zero gradients, and no launch where there is nothing to do."""
    import argparse

    import dgm
    from dgg_b200 import CSRGraph
    from dgg_b200 import functional as K
    from dgg_b200._lib import lib

    n, h = 50, 16
    g = CSRGraph(n, torch.zeros(n + 1, dtype=torch.int32, device="cuda"), torch.zeros(0, dtype=torch.int32,
                                                                                        device="cuda"))
    for b in (0.375, -0.375):
        for hard_k in (-1, 2):
            leaves = [torch.randn(n, h, device="cuda", requires_grad=True),
                      torch.randn(h, device="cuda", requires_grad=True),
                      torch.full((1, 1), W, device="cuda", requires_grad=True),
                      torch.full((1,), b, device="cuda", requires_grad=True)]
            out, k, R, rank = K.dgg_edge(*leaves, g, hard_k=hard_k)
            assert out.numel() == 0 and R.numel() == 0 and rank.numel() == 0
            want_k = b if b > 0 else float(np.float32(np.float32(b) * np.float32(0.01)))
            assert bool((k == want_k).all()), (k, want_k)
            torch.cuda.synchronize()
            before = int(lib().dggb_kernel_launches())
            out.sum().backward()
            torch.cuda.synchronize()
            assert int(lib().dggb_kernel_launches()) == before
            for q in leaves:
                assert bool((q.grad == 0).all())
    score = torch.zeros(0, device="cuda", requires_grad=True)
    kk = torch.rand(n, device="cuda", requires_grad=True)
    before = int(lib().dggb_kernel_launches())
    out, rank = K.row_firstk(score, kk, g, return_rank=True)
    out.sum().backward()
    torch.cuda.synchronize()
    assert int(lib().dggb_kernel_launches()) == before
    assert out.numel() == 0 and rank.numel() == 0 and bool((kk.grad == 0).all()) and score.grad.numel() == 0
    # the module: an adjacency without entries
    args = argparse.Namespace(extra_edge_dim=0)
    m = dgm.DGG(in_dim=8, latent_dim=h, args=args).cuda()
    x = torch.randn(n, 8, device="cuda")
    adj = torch.sparse_coo_tensor(torch.zeros(2, 0, dtype=torch.long), torch.zeros(0), (n, n)).coalesce().cuda()
    a, x_enc = m(x, adj)
    assert a._nnz() == 0 and x_enc.shape == (n, h)
    (a.coalesce().values().sum() + x_enc.sum()).backward()
    for q in (m.degree_decoder[0].weight, m.degree_decoder[0].bias, m.edge_encoder[0].weight, m.edge_encoder[0].bias):
        assert q.grad is not None and bool((q.grad == 0).all())
    db = m.degree_decoder[0].bias.detach()
    assert torch.equal(m.last_k, torch.where(db > 0, db, db * SLOPE).expand(n))


# ---------------------------------------------------------------------------------------------------------------
# argument checks (CPU: every call below is rejected before anything touches memory or the GPU)
# ---------------------------------------------------------------------------------------------------------------
def test_edge_entry_points_reject_bad_arguments():
    import dgg_b200

    L = dgg_b200.lib()
    one = ctypes.c_void_p(16)          # never dereferenced
    null = None
    BAD_ARG, BAD_SHAPE, UNSUPPORTED = -1, -2, -3

    def fwd(n=4, nnz=8, h=16, R=one, rowptr=one, erow=one, s=one, y=one):
        return L.dggb_dgg_edge_fwd(rowptr, erow, one, n, nnz, h, y, one, one, one, null, -1, R, one, s, one, one,
                                   null, null)

    assert fwd(rowptr=null) == BAD_ARG
    assert fwd(y=null) == BAD_ARG
    assert fwd(s=null) == BAD_ARG
    assert fwd(R=null) == BAD_ARG                      # entries but no R
    assert fwd(erow=null) == BAD_ARG
    assert fwd(n=-1) == BAD_ARG and fwd(nnz=-1) == BAD_ARG and fwd(h=0) == BAD_ARG
    assert fwd(h=6) == BAD_SHAPE and fwd(h=516) == BAD_SHAPE
    assert fwd(nnz=0, R=null, erow=null, h=6) == BAD_SHAPE       # NULL entry arrays are accepted without entries

    def bwd(n=4, nnz=8, h=16, g=one, ds=one, dbe=one):
        return L.dggb_dgg_edge_bwd(one, one, one, n, nnz, h, one, one, one, one, null, -1, one, one, one, one, g, ds,
                                   one, dbe, one, null)

    assert bwd(g=null) == BAD_ARG and bwd(ds=null) == BAD_ARG and bwd(dbe=null) == BAD_ARG
    assert bwd(n=-1) == BAD_ARG and bwd(h=10) == BAD_SHAPE
    assert bwd(nnz=0, g=null, h=10) == BAD_SHAPE

    def ffwd(nnz=8, mx=4, h=16, R=one, zc=0):
        return L.dggb_dgg_edge_fwd_fused(one, one, one, 4, nnz, mx, h, one, one, one, one, null, -1, R, one, one, one,
                                         one, null, zc, null)

    assert ffwd(R=null) == BAD_ARG and ffwd(mx=-1) == BAD_ARG and ffwd(zc=-1) == BAD_ARG
    assert ffwd(h=6) == BAD_SHAPE
    assert ffwd(mx=513) == UNSUPPORTED and ffwd(nnz=0) == UNSUPPORTED

    def fbwd(nnz=8, mx=4, h=16, ds=one):
        return L.dggb_dgg_edge_bwd_fused(one, one, one, 4, nnz, mx, h, one, one, one, one, null, -1, one, one, one,
                                         one, one, ds, one, one, one, null)

    assert fbwd(ds=null) == BAD_ARG and fbwd(h=6) == BAD_SHAPE
    assert fbwd(mx=513) == UNSUPPORTED and fbwd(nnz=0) == UNSUPPORTED
    assert L.dggb_row_firstk_fwd(one, 4, one, one, 2, one, one, null, null) == UNSUPPORTED
    assert L.dggb_row_firstk_fwd(one, 4, null, one, 0, one, one, null, null) == BAD_ARG
    assert L.dggb_row_firstk_fwd(one, -1, one, one, 0, one, one, null, null) == BAD_ARG
    assert L.dggb_row_firstk_bwd(one, 4, one, one, 5, one, one, one, one, null) == UNSUPPORTED
    assert L.dggb_row_firstk_bwd(one, 4, one, one, 0, one, one, null, one, null) == BAD_ARG
    assert L.dggb_csr_expand_rows(null, 4, one, null) == BAD_ARG
