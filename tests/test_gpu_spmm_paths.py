"""Every launch path of the SpMM family (csrc/spmm.cu) against one fp64 reference.

Dispatch rules (F = feature width; for the conv layer Fin / Fout):

* ``dispatch_vec`` (``dggb_spmm_csr_fwd`` / ``_bwd``, ``spmm_fwd_kernel<VEC,T>`` / ``spmm_bwd_kernel<VEC,T>``): VEC = 4
  if F % 4 == 0, else 2 if F % 2 == 0, else 1; chunks = ceil(F / VEC); L = the smallest power of two with 4 L >= chunks,
  capped at 32; T = ceil(chunks / L) rounded up to 1, 2 or 4.  Past 4 chunks per lane (L = 32) the row is covered in
  passes of VEC * 128 columns: VEC 4 from F = 516, VEC 2 from F = 258, VEC 1 from F = 129.
  T = 2 needs exactly two chunks at L = 1, i.e. F = 2 VEC; F = 4 (VEC 2) and F = 2 (VEC 1) take a wider vector, so
  ``<2,2>`` and ``<1,2>`` are unreachable.  Reachable: (4,1) F = 4, (4,2) F = 8, (4,4), (2,1) F = 2, (2,4), (1,1) F = 1,
  (1,4).
* ``spmm_gemm_lanes`` (edge kernels and the conv layer's gathers): chunks = F / 4 (F % 4 == 0), L and T as above:
  T = 1 at F = 4, T = 2 at F = 8, T = 4 from F = 12.  F <= 512 (edge) and Fin <= 128 (conv) never need a second pass.
* ``edge_run_len``: a group of L lanes walks a run of r = nnz // (148 * 4 * 8 * G) entries clamped to 1..8, G = 32 / L.
  At F = 64 (G = 8) r >= 2 from nnz = 75 776 and r = 8 from 303 104; at F = 4 / 8 (G = 32) from 303 104 and
  1 212 416; at F = 512 (G = 1) r = 8 from 37 888.  A row wholly inside one run is written with a plain store, a row
  cut by a run boundary is combined with vector reductions.
* Python ``functional._Spmm``: the edge kernels when F % 4 == 0, F <= 512 and 0 < nnz <= 64 n (and
  ``_NO_EDGE_SPMM`` is off), the CSR kernels otherwise.
* Conv layer (``dggb_spmm_gemm_fwd`` / ``_bwd``): RB = 4 rows per warp iteration when n >= kSmallGraphRows =
  8 * 148 * 8 = 9 472, RB = 1 below.  Forward Q by Fout (<= 32: 1, <= 64: 2, else 4), backward Q by Fin (the columns of
  ds).  Forward with RB = 1 runs ``spmm_gemm_fwd_row_kernel<Q>`` unless DGGB_SPMM_GEMM_NO_ROW is set, which selects
  ``spmm_gemm_fwd_kernel<T,Q,1>``.  The backward has no row kernel.  T and Q both follow Fin in the backward, so only
  (T,Q) = (1,1), (2,1), (4,1), (4,2), (4,4) are reachable there: Fin = 4 or 8 means Q = 1.  ``functional.spmm_gemm``
  takes n < ``_FUSED_CONV_MAX_N`` only (8 192), so the tests raise that limit to reach RB = 4.
* ``gcnii_stack_fwd_kernel<Q>``: F = 32 Q, Q in {1, 2, 4}; OWN = 32, 16, 8 entries per round.

``PATHS`` maps each case to the launches of the family it makes, in order (forward, then backward);
``test_dispatch_launches_the_tabled_kernels`` checks the table against the kernels the profiler sees, and
``test_path_table_reaches_every_instantiation`` checks that the cases reach every reachable instantiation (and every run
length class of the edge kernels).

Reference: the same computation in fp64 with ``index_add_`` over the entry list (no dense N x N).  Bounds come from the
data: the same computation on absolute values (|A| |X|, |s| |W|, ...) times u = 2^-24 times the number of rounded
terms plus a small slack (the row length, the column in-degree for dx, Fin / Fout for the dense parts).  A dropped,
duplicated or misrouted entry misses such a bound by orders of magnitude.  ReLU: gradient entries whose fp64
pre-activation lies within its bound of 0 are left out of the loss on both sides.
"""
import ctypes
from collections import namedtuple

import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
SMS = 148
SMALL_GRAPH_ROWS = 8 * SMS * 8
C1, C2, THETA, BETA = 0.875, 0.125, 0.375, 0.625     # dyadic: the kernels see exactly these values

# grads: which leaves require a gradient ("vx": values and x; "v" / "x": one of them -> dx / dval NULL)
Spmm = namedtuple("Spmm", "n f deg seed rs no_edge grads")
# mode: "row" (default dispatch), "ep" (DGGB_SPMM_GEMM_NO_ROW); RB follows n.  opts: h0 res relu keep rs beta
Conv = namedtuple("Conv", "n fin fout deg seed mode opts grads")
Stack = namedtuple("Stack", "n f layers deg seed keep")

PATHS = [
    # ---- CSR (warp per row) ----
    (Spmm(2000, 4, 6, 1, True, True, "vx"), ["csr_fwd<4,1>", "csr_bwd<4,1>"]),
    (Spmm(1001, 8, 5, 2, False, True, "v"), ["csr_fwd<4,2>", "csr_bwd<4,2>"]),
    (Spmm(3001, 64, 7, 3, True, True, "x"), ["csr_fwd<4,4>", "csr_bwd<4,4>"]),
    (Spmm(1500, 516, 6, 4, True, False, "vx"), ["csr_fwd<4,4>", "csr_bwd<4,4>"]),       # two passes
    (Spmm(400, 64, 150, 5, False, False, "vx"), ["csr_fwd<4,4>", "csr_bwd<4,4>"]),      # nnz > 64 n
    (Spmm(50, 64, 0, 6, False, False, "vx"), []),                                        # nnz = 0: Y = 0, no launch
    (Spmm(1200, 2, 6, 7, False, False, "vx"), ["csr_fwd<2,1>", "csr_bwd<2,1>"]),
    (Spmm(999, 6, 5, 8, True, False, "vx"), ["csr_fwd<2,4>", "csr_bwd<2,4>"]),
    (Spmm(1100, 258, 6, 9, False, False, "vx"), ["csr_fwd<2,4>", "csr_bwd<2,4>"]),      # two passes
    (Spmm(1, 1, 1, 10, True, False, "vx"), ["csr_fwd<1,1>", "csr_bwd<1,1>"]),           # n = 1
    (Spmm(2500, 1, 8, 11, True, False, "vx"), ["csr_fwd<1,1>", "csr_bwd<1,1>"]),
    (Spmm(777, 3, 6, 12, False, False, "vx"), ["csr_fwd<1,4>", "csr_bwd<1,4>"]),
    (Spmm(1300, 129, 6, 13, True, False, "vx"), ["csr_fwd<1,4>", "csr_bwd<1,4>"]),      # two passes
    # ---- edge-parallel ----
    (Spmm(2000, 4, 6, 14, True, False, "vx"), ["edge_fwd<1>", "edge_bwd<1>"]),          # run 1
    (Spmm(20000, 4, 25, 15, False, False, "vx"), ["edge_fwd<1>", "edge_bwd<1>"]),       # run 3
    (Spmm(40000, 4, 34, 16, True, False, "vx"), ["edge_fwd<1>", "edge_bwd<1>"]),        # run 8
    (Spmm(1999, 8, 6, 17, False, False, "v"), ["edge_fwd<2>", "edge_bwd<2>"]),          # run 1
    (Spmm(20000, 8, 25, 18, True, False, "x"), ["edge_fwd<2>", "edge_bwd<2>"]),         # run 3
    (Spmm(40000, 8, 34, 19, True, False, "vx"), ["edge_fwd<2>", "edge_bwd<2>"]),        # run 8
    (Spmm(3000, 64, 7, 20, True, False, "vx"), ["edge_fwd<4>", "edge_bwd<4>"]),         # run 1
    (Spmm(10000, 64, 13, 21, False, False, "vx"), ["edge_fwd<4>", "edge_bwd<4>"]),      # run 3
    (Spmm(20000, 64, 17, 22, True, False, "vx"), ["edge_fwd<4>", "edge_bwd<4>"]),       # run 8
    (Spmm(3000, 512, 14, 23, True, False, "vx"), ["edge_fwd<4>", "edge_bwd<4>"]),       # run 8, L = 32
    (Spmm(1, 12, 1, 24, False, False, "vx"), ["edge_fwd<4>", "edge_bwd<4>"]),           # n = 1
    (Spmm(4001, 12, 6, 25, False, False, "vx"), ["edge_fwd<4>", "edge_bwd<4>"]),
    # ---- conv layer, RB = 4 (n >= 9 472) ----
    (Conv(9472, 4, 32, 6, 30, "row", "rs relu", "all"), ["conv_fwd<1,1,4>", "conv_bwd<1,1,4>"]),
    (Conv(10007, 4, 64, 6, 31, "row", "h0 keep", "v"), ["conv_fwd<1,2,4>", "conv_bwd<1,1,4>"]),
    (Conv(9500, 4, 100, 6, 32, "row", "res relu", "x"), ["conv_fwd<1,4,4>", "conv_bwd<1,1,4>"]),
    (Conv(9601, 8, 8, 6, 33, "row", "h0 beta relu keep rs", "all"), ["conv_fwd<2,1,4>", "conv_bwd<2,1,4>"]),
    (Conv(9473, 8, 48, 6, 34, "row", "res", "all"), ["conv_fwd<2,2,4>", "conv_bwd<2,1,4>"]),
    (Conv(9800, 8, 128, 6, 35, "row", "relu rs", "all"), ["conv_fwd<2,4,4>", "conv_bwd<2,1,4>"]),
    (Conv(12001, 12, 3, 6, 36, "row", "relu h0", "all"), ["conv_fwd<4,1,4>", "conv_bwd<4,1,4>"]),
    (Conv(12000, 64, 64, 6, 37, "row", "h0 beta relu keep", "all"), ["conv_fwd<4,2,4>", "conv_bwd<4,2,4>"]),
    (Conv(9473, 128, 128, 6, 38, "row", "h0 beta relu rs res", "all"), ["conv_fwd<4,4,4>", "conv_bwd<4,4,4>"]),
    (Conv(10000, 64, 128, 6, 39, "ep", "relu", "all"), ["conv_fwd<4,4,4>", "conv_bwd<4,2,4>"]),   # env ignored
    (Conv(9999, 128, 16, 6, 40, "row", "res keep", "all"), ["conv_fwd<4,1,4>", "conv_bwd<4,4,4>"]),
    # ---- conv layer, RB = 1, entry-parallel forward (DGGB_SPMM_GEMM_NO_ROW) ----
    (Conv(1, 4, 32, 1, 41, "ep", "relu", "all"), ["conv_fwd<1,1,1>", "conv_bwd<1,1,1>"]),
    (Conv(3001, 4, 64, 6, 42, "ep", "rs keep", "all"), ["conv_fwd<1,2,1>", "conv_bwd<1,1,1>"]),
    (Conv(2000, 4, 128, 6, 43, "ep", "h0", "x"), ["conv_fwd<1,4,1>", "conv_bwd<1,1,1>"]),
    (Conv(2999, 8, 8, 6, 44, "ep", "beta h0 relu", "all"), ["conv_fwd<2,1,1>", "conv_bwd<2,1,1>"]),
    (Conv(37, 8, 64, 4, 45, "ep", "res", "all"), ["conv_fwd<2,2,1>", "conv_bwd<2,1,1>"]),
    (Conv(4000, 8, 100, 6, 46, "ep", "relu rs", "v"), ["conv_fwd<2,4,1>", "conv_bwd<2,1,1>"]),
    (Conv(5000, 32, 32, 6, 47, "ep", "beta h0 relu keep", "all"), ["conv_fwd<4,1,1>", "conv_bwd<4,1,1>"]),
    (Conv(9471, 64, 64, 6, 48, "ep", "beta h0 relu keep rs", "all"), ["conv_fwd<4,2,1>", "conv_bwd<4,2,1>"]),
    (Conv(1234, 128, 128, 6, 49, "ep", "beta h0 relu res", "all"), ["conv_fwd<4,4,1>", "conv_bwd<4,4,1>"]),
    # ---- conv layer, RB = 1, row kernel ----
    (Conv(1, 64, 64, 1, 50, "row", "beta h0 relu", "all"), ["conv_row<2>", "conv_bwd<4,2,1>"]),
    (Conv(3327, 36, 7, 6, 51, "row", "relu rs", "all"), ["conv_row<1>", "conv_bwd<4,2,1>"]),
    (Conv(2708, 128, 100, 6, 52, "row", "h0 keep relu", "all"), ["conv_row<4>", "conv_bwd<4,4,1>"]),
    (Conv(500, 4, 16, 6, 53, "row", "relu", "all"), ["conv_row<1>", "conv_bwd<1,1,1>"]),
    (Conv(9471, 12, 64, 6, 54, "row", "res rs", "all"), ["conv_row<2>", "conv_bwd<4,1,1>"]),
    # ---- GCNII stack ----
    (Stack(1000, 32, 2, 8, 60, True), ["stack<1>"]),
    (Stack(1000, 32, 96, 8, 61, False), ["stack<1>"]),
    (Stack(2000, 64, 96, 6, 62, True), ["stack<2>"]),
    (Stack(1, 64, 2, 1, 63, False), ["stack<2>"]),
    (Stack(1001, 128, 2, 10, 64, True), ["stack<4>"]),
    (Stack(1001, 128, 96, 6, 65, False), ["stack<4>"]),
]


def _path_id(case):
    c, launches = case
    kind = type(c).__name__.lower()
    extra = ""
    if isinstance(c, Spmm):
        extra = f"-f{c.f}-{c.grads}" + ("-rs" if c.rs else "") + ("-noedge" if c.no_edge else "")
    elif isinstance(c, Conv):
        extra = f"-{c.fin}x{c.fout}-{c.mode}-{c.grads}-" + c.opts.replace(" ", "+")
    else:
        extra = f"-f{c.f}-L{c.layers}" + ("-keep" if c.keep else "")
    return f"{kind}-{launches[0] if launches else 'nolaunch'}-n{c.n}{extra}"


# ---------------------------------------------------------------------------------------------------------------
# graphs and the dispatch restated
# ---------------------------------------------------------------------------------------------------------------
_GRAPHS = {}


def _graph(n, deg, seed):
    """(rowptr, row, col) int64 on the CPU of a coalesced graph, asymmetric, out-degree skewed towards low rows.
    Mixed in where n allows: empty rows at the start, middle and end; rows of exactly 1, 32, 33 and 64 entries; a hub
    row of more than 1 024 entries; a column with an in-degree in the thousands.  deg = 0: no entries at all."""
    key = (n, deg, seed)
    if key in _GRAPHS:
        return _GRAPHS[key]
    gen = torch.Generator().manual_seed(seed)
    if n == 1:
        row = col = torch.zeros(deg, dtype=torch.long)
    else:
        m = n * deg
        row = (torch.rand(m, generator=gen) ** 1.5 * n).long().clamp_max(n - 1)
        col = torch.randint(0, n, (m,), generator=gen)
        if deg > 0 and n >= 2000:                   # column n // 5: in-degree ~ min(n, 3000)
            hot_rows = torch.randperm(n, generator=gen)[:min(n, 3000)]
            row = torch.cat([row, hot_rows])
            col = torch.cat([col, torch.full_like(hot_rows, n // 5)])
        exact = {}
        if deg > 0 and n >= 8:
            exact.update({0: 0, n // 2: 0, n - 1: 0})
        if deg > 0 and n >= 100:
            exact.update({1: 1, 2: 32, 3: 33, n // 3: 64, n // 2 + 1: 32, n - 2: 33})
        if deg > 0 and n >= 1100:
            exact[n // 4] = min(n, 1100 + seed % 300)
        if exact:
            drop = torch.zeros(n, dtype=torch.bool)
            drop[list(exact)] = True
            keep = ~drop[row]
            row, col = row[keep], col[keep]
            for r, d in exact.items():
                row = torch.cat([row, torch.full((d,), r, dtype=torch.long)])
                col = torch.cat([col, torch.randperm(n, generator=gen)[:d]])
        k = torch.unique(row * n + col)
        row, col = k // n, k % n
    rowptr = torch.zeros(n + 1, dtype=torch.long)
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
    _GRAPHS[key] = (rowptr, row, col)
    return _GRAPHS[key]


def _lanes(chunks):
    L = 1
    while L < 32 and 4 * L < chunks:
        L *= 2
    t = -(-chunks // L)
    return L, (4 if t > 2 else (2 if t == 2 else 1))


def _csr_vec_t(f):
    vec = 4 if f % 4 == 0 else (2 if f % 2 == 0 else 1)
    L, t = _lanes(-(-f // vec))
    return vec, t, -(-f // (vec * L * t))           # (VEC, T, passes)


def _edge_run(nnz, f):
    L, _ = _lanes(f // 4)
    r = nnz // (SMS * 4 * 8 * (32 // L))
    return max(1, min(8, r))


def _uses_edge(c, nnz):
    return (not c.no_edge) and c.f % 4 == 0 and c.f <= 512 and 0 < nnz <= 64 * c.n


def _expected(c):
    """The launches of the family the dispatch rules above give for case c."""
    if isinstance(c, Spmm):
        nnz = int(_graph(c.n, c.deg, c.seed)[0][-1])
        if nnz == 0:
            return []
        if _uses_edge(c, nnz):
            t = _lanes(c.f // 4)[1]
            return [f"edge_fwd<{t}>", f"edge_bwd<{t}>"]
        vec, t, _ = _csr_vec_t(c.f)
        return [f"csr_fwd<{vec},{t}>", f"csr_bwd<{vec},{t}>"]
    if isinstance(c, Conv):
        t = _lanes(c.fin // 4)[1]
        qf = 1 if c.fout <= 32 else (2 if c.fout <= 64 else 4)
        qb = 1 if c.fin <= 32 else (2 if c.fin <= 64 else 4)
        rb = 4 if c.n >= SMALL_GRAPH_ROWS else 1
        fwd = f"conv_row<{qf}>" if (rb == 1 and c.mode == "row") else f"conv_fwd<{t},{qf},{rb}>"
        return [fwd, f"conv_bwd<{t},{qb},{rb}>"]
    return [f"stack<{c.f // 32}>"]


def test_path_table_reaches_every_instantiation():
    for c, launches in PATHS:
        assert _expected(c) == launches, (c, _expected(c), launches)
    got = {name for _, launches in PATHS for name in launches}
    want = {f"csr_{d}<{v},{t}>" for d in ("fwd", "bwd") for v, t in ((4, 1), (4, 2), (4, 4), (2, 1), (2, 4), (1, 1),
                                                                      (1, 4))}
    want |= {f"edge_{d}<{t}>" for d in ("fwd", "bwd") for t in (1, 2, 4)}
    want |= {f"conv_row<{q}>" for q in (1, 2, 4)}
    want |= {f"conv_fwd<{t},{q},{rb}>" for t in (1, 2, 4) for q in (1, 2, 4) for rb in (1, 4)}
    want |= {f"conv_bwd<{t},{q},{rb}>" for t, q in ((1, 1), (2, 1), (4, 1), (4, 2), (4, 4)) for rb in (1, 4)}
    want |= {f"stack<{q}>" for q in (1, 2, 4)}
    assert got == want, (want - got, got - want)
    # a multi-pass CSR case for each VEC; run lengths 1, 2..7 and 8 for each edge T; the shapes of the issue
    passes = {}
    runs = {}
    for c, launches in PATHS:
        if not isinstance(c, Spmm):
            continue
        nnz = int(_graph(c.n, c.deg, c.seed)[0][-1])
        if not launches:
            continue
        if launches[0].startswith("csr"):
            vec, _, ps = _csr_vec_t(c.f)
            passes.setdefault(vec, set()).add(ps)
        else:
            r = _edge_run(nnz, c.f)
            runs.setdefault(_lanes(c.f // 4)[1], set()).add(1 if r == 1 else (8 if r == 8 else 2))
    assert all(max(passes[v]) > 1 for v in (4, 2, 1)), passes
    assert runs == {1: {1, 2, 8}, 2: {1, 2, 8}, 4: {1, 2, 8}}, runs
    stacks = [c for c, _ in PATHS if isinstance(c, Stack)]
    assert {c.layers for c in stacks} == {2, 96}


# ---------------------------------------------------------------------------------------------------------------
# fp64 reference
# ---------------------------------------------------------------------------------------------------------------
class G:
    """A test graph on the device: CSRGraph handle, entry rows / columns, row lengths and column in-degrees."""

    def __init__(self, n, deg, seed):
        from dgg_b200 import CSRGraph

        rowptr, row, col = _graph(n, deg, seed)
        self.n, self.nnz = n, int(rowptr[-1])
        self.csr = CSRGraph(n, rowptr.to(torch.int32).cuda(), col.to(torch.int32).cuda())
        self.row, self.col = row.cuda(), col.cuda()
        self.deg = (rowptr[1:] - rowptr[:-1]).double().cuda().unsqueeze(1)
        self.indeg = torch.bincount(col, minlength=n).double().cuda().unsqueeze(1)


def _spmm64(g, vals, x, rs=None):
    y = torch.zeros(g.n, x.shape[1], dtype=x.dtype, device=x.device).index_add_(0, g.row, vals[:, None] * x[g.col])
    return y if rs is None else y * rs[:, None]


def _within(got, want, bound, what):
    err = (got.double() - want).abs()
    bad = err > bound
    if bool(bad.any()):
        i = int(((err - bound) / bound.clamp_min(1e-300)).argmax())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} entries beyond the bound; worst at flat "
                             f"index {i}: got {float(got.reshape(-1)[i])}, want {float(want.reshape(-1)[i])}, "
                             f"bound {float(bound.reshape(-1)[i])}")


def _grad_pair(fn, leaves, gy):
    """fp64 autograd of fn at the leaves and of fn on their absolute values at |gy| (the error scale of each grad)."""
    ls = [None if t is None else t.detach().double().requires_grad_(True) for t in leaves]
    out = fn(ls, False)
    live = [t for t in ls if t is not None]
    grads = torch.autograd.grad(out, live, gy.double(), allow_unused=True)
    la = [None if t is None else t.detach().double().abs().requires_grad_(True) for t in leaves]
    out_a = fn(la, True)
    grads_a = torch.autograd.grad(out_a, [t for t in la if t is not None], gy.double().abs(), allow_unused=True)
    it, ia = iter(grads), iter(grads_a)
    return out.detach(), out_a.detach(), [None if t is None else (next(it), next(ia)) for t in leaves]


def _data(n, f, seed):
    gen = torch.Generator().manual_seed(seed + 1000)
    return gen, torch.randn(n, f, generator=gen)


@pytest.mark.parametrize("case", [c for c in PATHS if isinstance(c[0], Spmm)],
                         ids=[_path_id(c) for c in PATHS if isinstance(c[0], Spmm)])
def test_spmm_path_matches_fp64(case, monkeypatch):
    from dgg_b200 import functional as K

    c, _ = case
    monkeypatch.setattr(K, "_NO_EDGE_SPMM", c.no_edge)
    g = G(c.n, c.deg, c.seed)
    gen, x = _data(c.n, c.f, c.seed)
    vals = torch.randn(g.nnz, generator=gen)
    rs = (torch.rand(c.n, generator=gen) * 2.0 - 0.5) if c.rs else None
    gy = torch.randn(c.n, c.f, generator=gen).cuda()
    v_ = vals.cuda().requires_grad_("v" in c.grads)
    x_ = x.cuda().requires_grad_("x" in c.grads)
    rs_ = None if rs is None else rs.cuda()
    y = K.spmm(v_, x_, g.csr, rs_)
    (y * gy).sum().backward()

    def fn(ls, absval):
        v, xx = ls
        r = None if rs_ is None else (rs_.double().abs() if absval else rs_.double())
        return _spmm64(g, v, xx, r)

    want, want_abs, grads = _grad_pair(fn, [vals.cuda(), x.cuda()], gy)
    _within(y.detach(), want, U * (g.deg + 4) * want_abs, "y")
    (dv, dv_abs), (dx, dx_abs) = grads
    if "v" in c.grads:
        _within(v_.grad, dv, U * (c.f + 4) * dv_abs, "dval")
    else:
        assert v_.grad is None
    if "x" in c.grads:
        _within(x_.grad, dx, U * (g.indeg + 4) * dx_abs, "dx")
    else:
        assert x_.grad is None


def _conv_inputs(c, g):
    gen, x = _data(c.n, c.fin, c.seed)
    opts = c.opts.split()
    t = dict(vals=torch.randn(g.nnz, generator=gen), x=x,
             w=torch.randn(c.fin, c.fout, generator=gen) / c.fin ** 0.5)
    t["h0"] = torch.randn(c.n, c.fin, generator=gen) if "h0" in opts else None
    t["res"] = torch.randn(c.n, c.fout, generator=gen) if "res" in opts else None
    t["rs"] = (torch.rand(c.n, generator=gen) * 2.0 - 0.5) if "rs" in opts else None
    t["keep"] = ((torch.rand(c.n, c.fout, generator=gen) > 0.2).float() * 1.25) if "keep" in opts else None
    t["gy"] = torch.randn(c.n, c.fout, generator=gen)
    return {k: (None if v is None else v.cuda()) for k, v in t.items()}, "relu" in opts, \
        (BETA if "beta" in opts else 0.0), (THETA if "beta" in opts else 1.0 - BETA)


def _conv64(g, ls, absval, rs, keep, theta, beta, relu, c2):
    """(y, z) of act(theta (s W) + beta s + resid) * keep, s = c1 rs (A x) + c2 h0; the absolute-value form drops the
    ReLU (1-Lipschitz) and takes |.| of every constant."""
    vals, x, w, h0, res = ls
    a = abs if absval else (lambda v: v)
    r = None if rs is None else a(rs.double())
    s = a(C1) * _spmm64(g, vals, x, r)
    if h0 is not None:
        s = s + a(c2) * h0
    z = a(theta) * (s @ w) + (a(beta) * s if beta else 0.0)
    if res is not None:
        z = z + res
    y = torch.relu(z) if (relu and not absval) else z
    if keep is not None:
        y = y * a(keep.double())
    return y, z, s


class ConvRef:
    """fp64 forward of a conv case with its bounds, and the backward at a given gy (ReLU-ambiguous entries zeroed)."""

    def __init__(self, g, t, relu, beta, theta, c2=C2):
        self.g, self.t, self.relu, self.beta, self.theta, self.c2 = g, t, relu, beta, theta, c2
        self.leaves = [t["vals"], t["x"], t["w"], t["h0"], t["res"]]
        ls = [None if v is None else v.double() for v in self.leaves]
        la = [None if v is None else v.double().abs() for v in self.leaves]
        self.y, self.z, self.s = self._fwd(ls, False)
        _, self.z_abs, self.s_abs = self._fwd(la, True)
        fin = t["x"].shape[1]
        kabs = 1.0 if t["keep"] is None else t["keep"].double().abs()
        self.z_bound = U * (g.deg + fin + 10) * self.z_abs
        self.y_bound = self.z_bound * kabs + U * self.y.abs()
        self.s_bound = U * (g.deg + 6) * abs(theta) * self.s_abs
        # gradient entries whose pre-activation lies within its bound of 0: left out of the loss on both sides
        self.gy = t["gy"].clone()
        if relu:
            self.gy[self.z.abs() <= self.z_bound] = 0.0

    def _fwd(self, ls, absval):
        t = self.t
        return _conv64(self.g, ls, absval, t["rs"], t["keep"], self.theta, self.beta, self.relu, self.c2)

    def grads(self):
        mask = (self.z > 0).double() if self.relu else None

        def fn(ls, absval):
            y = self._fwd(ls, absval)[0]
            return y * mask if (absval and mask is not None) else y

        _, _, gr = _grad_pair(fn, self.leaves, self.gy)
        return gr

    def check_grads(self, got, names=("dval", "dx", "dw", "dh0", "dres"), scale=(1, 1, 1, 1, 1)):
        """got: kernel gradients in leaf order (None: not computed)."""
        g = self.g
        fin, fout = self.t["x"].shape[1], self.t["w"].shape[1]
        terms = [fout + fin + 10, fout + g.indeg + 10, g.n + float(g.deg.max()) + fin + 10, fout + 6, 2]
        for name, gk, ref, k, sc in zip(names, got, self.grads(), terms, scale):
            if gk is None or ref is None:
                continue
            want, want_abs = ref
            _within(gk, sc * want, U * k * abs(sc) * want_abs, name)


def _set_mode(monkeypatch, mode):
    if mode == "ep":
        monkeypatch.setenv("DGGB_SPMM_GEMM_NO_ROW", "1")
    else:
        monkeypatch.delenv("DGGB_SPMM_GEMM_NO_ROW", raising=False)


def _run_conv(c, g, t, relu, beta, theta, monkeypatch):
    """Forward and backward through functional.spmm_gemm (autograd wiring included) -> (y, grads in leaf order)."""
    from dgg_b200 import functional as K

    monkeypatch.setattr(K, "_FUSED_CONV_MAX_N", 10 ** 9)
    monkeypatch.setattr(K, "_NO_FUSED_CONV", False)
    _set_mode(monkeypatch, c.mode)
    need = {"all": "vals x w h0 res", "v": "vals", "x": "x"}[c.grads].split()
    leaves = {k: (None if t[k] is None else t[k].clone().requires_grad_(k in need)) for k in ("vals", "x", "w", "h0",
                                                                                            "res")}
    y = K.spmm_gemm(leaves["vals"], leaves["x"], leaves["w"], g.csr, h0=leaves["h0"], resid=leaves["res"],
                    row_scale=t["rs"], c1=C1, c2=C2, theta=theta, beta=beta, relu=relu, out_keep=t["keep"])
    assert y is not None
    return y, leaves


@pytest.mark.parametrize("case", [c for c in PATHS if isinstance(c[0], Conv)],
                         ids=[_path_id(c) for c in PATHS if isinstance(c[0], Conv)])
def test_conv_path_matches_fp64(case, monkeypatch):
    c, _ = case
    g = G(c.n, c.deg, c.seed)
    t, relu, beta, theta = _conv_inputs(c, g)
    ref = ConvRef(g, t, relu, beta, theta)
    y, leaves = _run_conv(c, g, t, relu, beta, theta, monkeypatch)
    _within(y.detach(), ref.y, ref.y_bound, "y")
    (y * ref.gy).sum().backward()
    got = [None if leaves[k] is None else leaves[k].grad for k in ("vals", "x", "w", "h0", "res")]
    need = {"all": 5, "v": 1, "x": 1}[c.grads]
    assert sum(q is not None for q in got) == min(need, sum(v is not None for v in leaves.values()))
    ref.check_grads(got)


# ---------------------------------------------------------------------------------------------------------------
# conv backward entry point called directly: accumulate bits, dval / dx alone, gy_masked, the zero_ws clear, s_out
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3001, 9472], ids=["rb1", "rb4"])
@pytest.mark.parametrize("parts", ["all", "dval", "dx"])
def test_conv_backward_entry_point_outputs(n, parts, monkeypatch):
    """dggb_spmm_gemm_bwd with accumulate = 3 on pre-filled dval / ds_out (they must come back as prefill + gradient),
    dval or dx alone (the other NULL), gy_masked = gy keep relu'(y), and zero_ws (filled with NaN, a length that is
    not a multiple of 4) cleared.  The forward's s_out = theta s is checked too."""
    from dgg_b200._lib import check, lib, p, stream

    monkeypatch.delenv("DGGB_SPMM_GEMM_NO_ROW", raising=False)
    c = Conv(n, 64, 64, 6, 70 + n, "row", "h0 beta relu keep rs", "all")
    g = G(c.n, c.deg, c.seed)
    t, relu, beta, theta = _conv_inputs(c, g)
    ref = ConvRef(g, t, relu, beta, theta)
    f = 64
    y = torch.empty(n, f, device="cuda")
    s = torch.empty(n, f, device="cuda")
    check(lib().dggb_spmm_gemm_fwd(p(g.csr.rowptr), p(g.csr.col), p(t["vals"]), n, p(t["x"]), f, p(t["rs"]), p(t["h0"]),
                                   C1, C2, p(t["w"]), f, theta, beta, None, 1, p(t["keep"]), p(y), p(s), stream()),
          "spmm_gemm_fwd")
    _within(y, ref.y, ref.y_bound, "y")
    _within(s, theta * ref.s, ref.s_bound, "s_out")
    gen = torch.Generator().manual_seed(n)
    pre_v = torch.randn(g.nnz, generator=gen).cuda()
    pre_s = torch.randn(n, f, generator=gen).cuda()
    dval = pre_v.clone() if parts != "dx" else None
    ds = pre_s.clone() if parts == "all" else None
    dx = torch.zeros(n, f, device="cuda") if parts != "dval" else None
    zero_ws = torch.full((f * f + 3,), float("nan"), device="cuda")
    gm = torch.full((n, f), float("nan"), device="cuda")
    gy = ref.gy.contiguous()
    check(lib().dggb_spmm_gemm_bwd(p(g.csr.rowptr), p(g.csr.col), p(t["vals"]), n, p(t["x"]), f, p(t["rs"]), C1,
                                   p(t["w"]), f, theta, beta, p(gy), p(dval), p(dx), p(ds), C2, p(zero_ws),
                                   zero_ws.numel(), p(y), p(gm), p(t["keep"]), 3, stream()), "spmm_gemm_bwd")
    assert bool((zero_ws == 0).all())
    want_gm = gy * t["keep"] * (y > 0)
    assert torch.equal(gm, want_gm)
    gr = ref.grads()
    if dval is not None:
        want, want_abs = gr[0]
        _within(dval, pre_v.double() + want, U * (2 * f + 10) * want_abs + U * (pre_v.double().abs() + want.abs()),
                "dval (accumulated)")
    if ds is not None:
        want, want_abs = gr[3]
        _within(ds, pre_s.double() + want, U * (f + 6) * want_abs + U * (pre_s.double().abs() + want.abs()),
                "ds_out = c2 ds (accumulated)")
    if dx is not None:
        want, want_abs = gr[1]
        _within(dx, want, U * (f + g.indeg + 10) * want_abs, "dx")


def test_entry_points_with_no_entries():
    """nnz = 0 on the edge entry points (the Python layer never sends an empty graph there): success, nothing
    written.  The CSR kernels on a graph whose rows are all empty: Y = 0, dval / dx untouched.  K.spmm on a graph
    without entries: zeros and zero gradients."""
    from dgg_b200 import CSRGraph
    from dgg_b200 import functional as K
    from dgg_b200._lib import check, lib, p, stream

    n, f = 50, 64
    rowptr = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
    col = torch.zeros(4, dtype=torch.int32, device="cuda")
    val = torch.ones(4, device="cuda")
    x = torch.randn(n, f, device="cuda")
    y = torch.full((n, f), 7.0, device="cuda")
    check(lib().dggb_spmm_edge_fwd(p(rowptr), p(col), p(col), p(val), n, 0, p(x), f, None, p(y), stream()),
          "spmm_edge_fwd")
    dval = torch.full((4,), 7.0, device="cuda")
    dx = torch.full((n, f), 7.0, device="cuda")
    check(lib().dggb_spmm_edge_bwd(p(col), p(col), p(val), 0, p(x), f, None, p(x), p(dval), p(dx), stream()),
          "spmm_edge_bwd")
    torch.cuda.synchronize()
    assert bool((y == 7).all()) and bool((dval == 7).all()) and bool((dx == 7).all())
    for fc in (64, 6, 1):
        xc = torch.randn(n, fc, device="cuda")
        yc = torch.full((n, fc), 7.0, device="cuda")
        dxc = torch.full((n, fc), 7.0, device="cuda")
        check(lib().dggb_spmm_csr_fwd(p(rowptr), p(col), p(val), n, p(xc), fc, None, p(yc), stream()), "spmm_csr_fwd")
        check(lib().dggb_spmm_csr_bwd(p(rowptr), p(col), p(val), n, p(xc), fc, None, p(xc), p(dval), p(dxc),
                                      stream()), "spmm_csr_bwd")
        torch.cuda.synchronize()
        assert bool((yc == 0).all()) and bool((dval == 7).all()) and bool((dxc == 7).all())
    g = CSRGraph(n, rowptr, col[:0])
    xg = x.clone().requires_grad_(True)
    vg = val[:0].clone().requires_grad_(True)
    out = K.spmm(vg, xg, g, torch.rand(n, device="cuda"))
    out.sum().backward()
    assert bool((out == 0).all()) and bool((xg.grad == 0).all()) and vg.grad.numel() == 0


# ---------------------------------------------------------------------------------------------------------------
# GCNII stack
# ---------------------------------------------------------------------------------------------------------------
def _stack_inputs(c, g):
    gen, x0 = _data(c.n, c.f, c.seed)
    # |A| row sums ~ 0.75 and |W| row sums ~ 0.8: the error bound stays of the order of the values over 96 layers
    vals = (torch.rand(g.nnz, generator=gen) * 2.0 - 1.0) * 1.5 / g.deg.cpu()[g.row.cpu(), 0].float()
    h0 = torch.randn(c.n, c.f, generator=gen)
    ws = [torch.randn(c.f, c.f, generator=gen) / c.f for _ in range(c.layers)]
    thetas = [float(torch.randint(32, 161, (1,), generator=gen)) / 256.0 for _ in range(c.layers)]
    keep = ((torch.rand(c.layers, c.n, c.f, generator=gen) > 0.2).float() * 1.25) if c.keep else None
    return vals.cuda(), x0.cuda(), h0.cuda(), [w.cuda() for w in ws], thetas, None if keep is None else keep.cuda()


def _run_stack(c, g, vals, x0, h0, ws, thetas, keep):
    """dggb_gcnii_stack_fwd called directly: every layer's output and theta * s, not only the last layer's."""
    from dgg_b200._lib import check, lib, p, stream

    nl, n, f = c.layers, c.n, c.f
    assert n <= int(lib().dggb_gcnii_stack_max_rows(f))
    y = torch.empty(nl, n, f, device="cuda")
    s = torch.empty(nl, n, f, device="cuda")
    bar = torch.zeros(1, dtype=torch.int32, device="cuda")
    wp = (ctypes.c_void_p * nl)(*[w.data_ptr() for w in ws])
    th = (ctypes.c_float * nl)(*thetas)
    check(lib().dggb_gcnii_stack_fwd(p(g.csr.rowptr), p(g.csr.col), p(vals), n, p(x0), p(h0), f, nl,
                                     ctypes.cast(wp, ctypes.c_void_p), ctypes.cast(th, ctypes.c_void_p), C1, C2,
                                     p(keep), p(y), p(s), p(bar), stream()), "gcnii_stack_fwd")
    torch.cuda.synchronize()
    return y, s


@pytest.mark.parametrize("case", [c for c in PATHS if isinstance(c[0], Stack)],
                         ids=[_path_id(c) for c in PATHS if isinstance(c[0], Stack)])
def test_stack_matches_fp64(case):
    """Layer by layer in fp64 with the bound carried along: E_k = |keep_k| (E_s (|theta_k| |W_k| + |1 - theta_k|)
    + u (f + 10) Z_abs_k) + u |y_k|, E_s = c1 |A| E_{k-1} + u (row length + 6) S_abs_k (ReLU is 1-Lipschitz)."""
    c, _ = case
    g = G(c.n, c.deg, c.seed)
    vals, x0, h0, ws, thetas, keep = _stack_inputs(c, g)
    y, s = _run_stack(c, g, vals, x0, h0, ws, thetas, keep)
    va, h0d = vals.double(), h0.double()
    prev, prev_abs, E = x0.double(), x0.double().abs(), torch.zeros_like(h0d)
    for k in range(c.layers):
        th, be = thetas[k], 1.0 - thetas[k]
        w = ws[k].double()
        sk = C1 * _spmm64(g, va, prev) + C2 * h0d
        sa = C1 * _spmm64(g, va.abs(), prev_abs) + C2 * h0d.abs()
        zk = th * (sk @ w) + be * sk
        za = th * (sa @ w.abs()) + be * sa
        yk = torch.relu(zk)
        kabs = 1.0
        if keep is not None:
            yk = yk * keep[k].double()
            kabs = keep[k].double()
        Es = C1 * _spmm64(g, va.abs(), E) + U * (g.deg + 6) * sa
        _within(s[k], th * sk, th * Es + U * th * sa, f"s_out layer {k}")
        E = kabs * (th * (Es @ w.abs()) + be * Es + U * (c.f + 10) * za) + U * yk.abs()
        _within(y[k], yk, E, f"y layer {k}")
        prev, prev_abs = yk, yk.abs()


# ---------------------------------------------------------------------------------------------------------------
# dispatch against the profiler
# ---------------------------------------------------------------------------------------------------------------
_SHORT = {"spmm_fwd_kernel": "csr_fwd", "spmm_bwd_kernel": "csr_bwd", "spmm_edge_fwd_kernel": "edge_fwd",
          "spmm_edge_bwd_kernel": "edge_bwd", "spmm_gemm_fwd_row_kernel": "conv_row",
          "spmm_gemm_fwd_kernel": "conv_fwd", "spmm_gemm_bwd_kernel": "conv_bwd", "gcnii_stack_fwd_kernel": "stack"}


def _kernel_launches(trace_path):
    import json
    import re

    with open(trace_path) as fh:
        ev = json.load(fh)["traceEvents"]
    names = []
    for e in sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        m = re.search(r"\b(\w+_kernel)<([^>]*)>", e["name"])
        if m and m.group(1) in _SHORT:
            names.append(_SHORT[m.group(1)] + "<" + ",".join(re.findall(r"\d+", m.group(2))) + ">")
    return names


def test_dispatch_launches_the_tabled_kernels(monkeypatch, tmp_path):
    """The profiler's kernel names, in launch order, are the table's (so the table is the dispatch, not a guess)."""
    from torch.profiler import ProfilerActivity, profile

    from dgg_b200 import functional as K

    runs = []
    for c, _ in PATHS:
        g = G(c.n, c.deg, c.seed)
        if isinstance(c, Spmm):
            gen, x = _data(c.n, c.f, c.seed)
            runs.append((c, g, x.cuda(), torch.randn(g.nnz, generator=gen).cuda()))
        elif isinstance(c, Conv):
            runs.append((c, g) + _conv_inputs(c, g))
        else:
            runs.append((c, g, _stack_inputs(c, g)))
    want = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # A profiler session that is not the process's first can lose its first few kernel records (2 or 3 of
        # them late in a full GPU test session): untracked kernels absorb the loss before the tabled launches.
        for _ in range(32):
            torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        for run, (_, launches) in zip(runs, PATHS):
            c, g = run[:2]
            if isinstance(c, Spmm):
                monkeypatch.setattr(K, "_NO_EDGE_SPMM", c.no_edge)
                x, v = run[2].requires_grad_(True), run[3].requires_grad_(True)
                K.spmm(v, x, g.csr).sum().backward()
            elif isinstance(c, Conv):
                t, relu, beta, theta = run[2:]
                y, _ = _run_conv(c, g, t, relu, beta, theta, monkeypatch)
                (y * t["gy"]).sum().backward()
            else:
                _run_stack(c, g, *run[2])
            want += launches
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(tmp_path / "trace.json"))
    assert _kernel_launches(tmp_path / "trace.json") == want


# ---------------------------------------------------------------------------------------------------------------
# sym_normalize, which produces the values every SpMM above consumes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,deg", [(5000, 6), (1, 1), (777, 40)])
def test_sym_normalize_matches_fp64_autograd(n, deg):
    """out_e = d_i v_e d_j with d = (row sums)^-1/2 on an asymmetric graph (hub rows, a column of in-degree ~3000,
    every node with a self loop so that every row sum is positive) and non-uniform values; the backward's column-side
    sums T_i = sum_{row i} g v d_col + sum_{col i} g v d_row against fp64 autograd."""
    from dgg_b200 import CSRGraph
    from dgg_b200 import functional as K

    rowptr, row, col = _graph(n, deg, 80 + n)
    k = torch.unique(torch.cat([row * n + col, torch.arange(n) * (n + 1)]))
    row, col = k // n, k % n
    rowptr = torch.zeros(n + 1, dtype=torch.long)
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
    gen = torch.Generator().manual_seed(n)
    vals = 0.05 + torch.rand(row.numel(), generator=gen) ** 3 * 4.0
    gy = torch.randn(row.numel(), generator=gen)
    g = CSRGraph(n, rowptr.to(torch.int32).cuda(), col.to(torch.int32).cuda())
    v = vals.cuda().requires_grad_(True)
    out = K.sym_normalize(v, g)
    (out * gy.cuda()).sum().backward()
    row, col = row.cuda(), col.cuda()
    vd = vals.cuda().double().requires_grad_(True)
    d = torch.zeros(n, dtype=torch.float64, device="cuda").index_add_(0, row, vd) ** -0.5
    want = d[row] * vd * d[col]
    (want * gy.cuda().double()).sum().backward()
    deg_r = torch.bincount(row, minlength=n).double()
    deg_c = torch.bincount(col, minlength=n).double()
    # d_i: a row sum of deg_i positive terms, then 1 / sqrtf (relative error deg_i / 2 + 2 roundings)
    rel_d = U * (deg_r / 2 + 3)
    _within(out.detach(), want.detach(), want.detach().abs() * (rel_d[row] + rel_d[col] + 3 * U), "out")
    dd = d.detach()
    ga, va = gy.cuda().double().abs(), vals.cuda().double()
    t_abs = torch.zeros(n, dtype=torch.float64, device="cuda").index_add_(0, row, ga * va * dd[col])
    t_abs.index_add_(0, col, ga * va * dd[row])
    nb = torch.zeros(n, dtype=torch.float64, device="cuda")      # largest relative error of a d in T_i's terms
    nb.scatter_reduce_(0, row, rel_d[col], "amax").scatter_reduce_(0, col, rel_d[row], "amax")
    terms = (deg_r + deg_c + 8)[row] * U + 3 * rel_d[row] + nb[row]
    bound = ga * dd[row] * dd[col] * (rel_d[row] + rel_d[col] + 3 * U) + 0.5 * dd[row] ** 3 * t_abs[row] * terms
    _within(v.grad, vd.grad, bound, "dval")
