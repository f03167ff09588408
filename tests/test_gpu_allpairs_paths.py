"""Every launch path of the all-pairs selector (csrc/allpairs.cu) against one fp64 dense reference.

``dggb_allpairs_topk_after_fwd`` sends a call to one template instantiation:

* ``v2<KB, SP, NM>`` (``allpairs_topk2_kernel``, two epilogue groups): kc <= 32, no continuation bound, and either
  DGGB_AP_V1 unset or the "big" tile shape (KB = 4 at 3xTF32, i.e. d = 65..128 with precision 3);
* ``v2c<4, 3, NM>`` (its continuation instantiation): the big shape with kc = 33..64 (two launches, the second
  bounded by the first one's last entry) or with a continuation bound;
* ``v1<KB, SP, NM>`` (``allpairs_topk_kernel``): everything else -- kc = 33..64, continuation passes, DGGB_AP_V1=1.

KB = dpad / 32 with dpad = d rounded up to 32 (96 -> 128); SP = precision (1: one TF32 pass, 3: 3xTF32); NM = noise
mode (0 none, 1 injected tensor, 2 in-kernel Philox Gumbel, 3 none + the evaluation normaliser ``out_rowsum``).
``PATHS`` maps each case to the launches the rule above gives, and ``test_dispatch_launches_the_tabled_kernels``
checks that table against the kernels the profiler sees.

Reference: y = -t D + G in fp64 (D = fp64 pairwise distance, G = the injected tensor or the host restatement of the
Philox noise), stable descending sort (value descending, column ascending).  Value bound of a kernel score: d2 carries
an absolute error eps (3xTF32 ~ a few 1e-6 |z|^2, single TF32 pass ~ 1e-3; |z|^2 <= 1 here), so
|dy| <= t min(sqrt(eps), eps / (2 D)) = t eps / max(sqrt(eps), 2 D), plus 1e-5 of fp32 rounding; the diagonal is
pinned to d2 = 0 by the kernel and gets 1e-5 alone.  Philox adds 5e-5 for the kernel's fast-math logs.  Indices must
match the reference exactly on rows whose top-(kc+1) reference gaps exceed twice the bounds of both neighbours."""
import json
import math
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

EPS = {3: 4e-6, 1: 1e-3}
T = 3.0
SEED = 0x5EED1234ABCD
SCALE = 0.3


def _z(n, d, seed, dup=False):
    gen = torch.Generator().manual_seed(seed)
    z = torch.softmax(torch.randn(n, d, generator=gen) * 2.0, -1)
    if dup:     # points 5m + 1 repeat points 5m: columns whose scores tie exactly in every row
        z[1::5] = z[0::5][:len(z[1::5])]
    return z


def _noise(nm, n, rows, seed, row_begin=0):
    """(injected tensor or None, dense G [rows, n] of the reference or None)."""
    if nm == 1:
        gen = torch.Generator().manual_seed(seed + 1)
        u = torch.rand(rows, n, generator=gen).clamp_(1e-9, 1 - 1e-7)
        g = SCALE * -torch.log(-torch.log(u))
        return g, g
    if nm == 2:
        from tests.philox_ref import gumbel_matrix
        return None, gumbel_matrix(rows, n, SEED, SCALE, row_begin)
    return None, None


def _call(z, nm, kc, prec, noise=None, row_begin=0, row_count=None, inv_temp=1.0, after=None):
    from dgg_b200 import functional as K

    kw = dict(row_begin=row_begin, row_count=row_count, after=after)
    if nm == 1:
        kw["noise"] = noise.cuda()
    elif nm == 2:
        kw.update(seed=SEED, noise_scale=SCALE)
    elif nm == 3:
        kw["inv_temp"] = inv_temp
    out = K.allpairs_topk(z.cuda(), torch.tensor([T], device="cuda"), kc=kc, precision=prec, **kw)
    return tuple(o.cpu() for o in out)


def _passes(z, nm, kc, prec, noise=None):
    """kc > 64: ceil(kc / 64) continuation passes, concatenated (as DGG_LearnableK_SDD._select does)."""
    outs, after = [], None
    for p0 in range(0, kc, 64):
        i, v = _call(z, nm, min(64, kc - p0), prec, noise, after=after)[:2]
        outs.append((i, v))
        after = (v[:, -1].cuda().contiguous(), i[:, -1].cuda().contiguous())
    return torch.cat([a for a, _ in outs], 1), torch.cat([b for _, b in outs], 1)


class Ref:
    """fp64 scores of rows [row_begin, row_begin + rows) against all n columns."""

    def __init__(self, z, G, prec, nm, row_begin=0, rows=None):
        n = z.shape[0]
        rows = n - row_begin if rows is None else rows
        zd = z.double().cuda()
        self.D = torch.cdist(zd[row_begin:row_begin + rows], zd, compute_mode="donot_use_mm_for_euclid_dist")
        self.y = -T * self.D + (0.0 if G is None else G.double().cuda())
        self.diag = torch.zeros_like(self.D, dtype=torch.bool)
        r = torch.arange(rows, device="cuda")
        self.diag[r, r + row_begin] = True
        eps = EPS[prec]
        self.tol = torch.where(self.diag, 0.0, T * eps / (2 * self.D).clamp_min(eps ** 0.5)) + 1e-5 + \
            (5e-5 if nm == 2 else 0.0)
        self.srt, self.order = torch.sort(self.y, dim=-1, descending=True, stable=True)
        self.n = n

    def rowsum(self, inv_temp):
        """sum_j exp(y_ij inv_temp) and its bound: the kernel's score error (tol) through exp, __expf's
        2 + 1.173 |x| ulp (CUDA C Programming Guide, intrinsic functions), the fp32 rounding of x = y inv_temp and of
        inv_temp itself, and two fp32 running sums of n / 2 positive terms each (<= n / 2 + 1 roundings of 2^-24)."""
        x = self.y * inv_temp
        e = torch.exp(x)
        s = e.sum(-1)
        rel = torch.expm1(self.tol * abs(inv_temp)) + (2 + 1.173 * x.abs()) * 2.0 ** -23 + x.abs() * 2.0 ** -23
        return s, (e * rel).sum(-1) + s * (self.n / 2 + 1) * 2.0 ** -24

    def check(self, idx, val, kc, min_exact=0.5, exact_ties=False):
        idx, val = idx.cuda().long(), val.cuda()
        rows, n = self.y.shape
        m = min(kc, n)
        assert idx.shape == (rows, kc) and val.shape == (rows, kc)
        # unused slots (n < kc): idx -1, val 0; used ones hold distinct columns
        assert bool((idx[:, m:] == -1).all()) and bool((val[:, m:] == 0).all())
        idx, val = idx[:, :m], val[:, :m]
        assert bool(((idx >= 0) & (idx < n)).all())
        s = idx.sort(-1).values
        assert bool((s[:, 1:] != s[:, :-1]).all()), "a column selected twice"
        # kernel order: value descending, column ascending among equal values
        ordered = (val[:, :-1] > val[:, 1:]) | ((val[:, :-1] == val[:, 1:]) & (idx[:, :-1] < idx[:, 1:]))
        assert bool(ordered.all()), "list not in (value desc, column asc) order"
        # values at the columns the kernel picked
        tol_p = torch.gather(self.tol, 1, idx)
        err = (val.double() - torch.gather(self.y, 1, idx)).abs() - tol_p
        assert float(err.max()) <= 0, float(err.max())
        # bit-exact indices away from ties: rank r is pinned when the reference gaps to ranks r - 1 and r + 1 both
        # exceed twice the two entries' bounds (then the sets of the first r and r + 1 entries are determined)
        k1 = min(m + 1, n)
        st = torch.gather(self.tol, 1, self.order[:, :k1])
        clear = (self.srt[:, :k1 - 1] - self.srt[:, 1:k1]) > 2 * (st[:, :-1] + st[:, 1:])
        yes = torch.ones(rows, 1, dtype=torch.bool, device=clear.device)
        clear = torch.cat([yes, clear, yes], 1)[:, :m + 1]
        pinned = clear[:, :-1] & clear[:, 1:]
        assert float(pinned.double().mean()) >= min_exact, float(pinned.double().mean())
        bad = pinned & (idx != self.order[:, :m])
        assert not bool(bad.any()), (int(bad.sum()), bad.nonzero()[:4])
        # a top-m set: nothing outside the list beats the m-th kept value by more than the two bounds
        if m < n:
            outside = torch.ones_like(self.y, dtype=torch.bool).scatter_(1, idx, False)
            kth = val[:, -1:].double()
            excess = (self.y - kth - self.tol - tol_p[:, -1:]).masked_fill(~outside, -1e30)
            assert float(excess.max()) <= 0, float(excess.max())
        if exact_ties:      # duplicated points: some rows must hold exactly tied scores, so the tie order is exercised
            assert int((val[:, :-1] == val[:, 1:]).sum()) > rows // 2


# (n, d, kc, precision, noise mode, DGGB_AP_V1, duplicated points) -> launches in order
PATHS = [
    ((1000, 20, 8, 3, 0, False, True), ["v2<1,3,0>"]),
    ((700, 32, 32, 3, 1, False, False), ["v2<1,3,1>"]),
    ((1301, 20, 1, 3, 2, False, False), ["v2<1,3,2>"]),
    ((1000, 32, 32, 3, 3, False, False), ["v2<1,3,3>"]),
    ((700, 20, 32, 1, 0, False, False), ["v2<1,1,0>"]),
    ((1000, 32, 8, 1, 1, False, False), ["v2<1,1,1>"]),
    ((333, 32, 32, 1, 2, False, False), ["v2<1,1,2>"]),
    ((1000, 20, 8, 1, 3, False, False), ["v2<1,1,3>"]),
    ((1000, 48, 32, 3, 0, False, False), ["v2<2,3,0>"]),
    ((1301, 64, 8, 3, 1, False, False), ["v2<2,3,1>"]),
    ((700, 64, 32, 3, 2, False, False), ["v2<2,3,2>"]),
    ((1000, 48, 8, 3, 3, False, True), ["v2<2,3,3>"]),
    ((45, 64, 8, 1, 0, False, False), ["v2<2,1,0>"]),
    ((700, 48, 32, 1, 1, False, False), ["v2<2,1,1>"]),
    ((1000, 64, 1, 1, 2, False, False), ["v2<2,1,2>"]),
    ((1000, 64, 32, 1, 3, False, False), ["v2<2,1,3>"]),
    ((1000, 96, 32, 3, 0, False, True), ["v2<4,3,0>"]),
    ((700, 128, 8, 3, 1, False, False), ["v2<4,3,1>"]),
    ((1000, 128, 32, 3, 2, False, False), ["v2<4,3,2>"]),
    ((1000, 96, 8, 3, 3, False, False), ["v2<4,3,3>"]),
    ((700, 128, 8, 3, 0, True, False), ["v2<4,3,0>"]),        # the big shape ignores DGGB_AP_V1
    ((1000, 128, 32, 1, 0, False, False), ["v2<4,1,0>"]),
    ((333, 96, 8, 1, 1, False, False), ["v2<4,1,1>"]),
    ((700, 128, 32, 1, 2, False, False), ["v2<4,1,2>"]),
    ((1000, 128, 8, 1, 3, False, False), ["v2<4,1,3>"]),
    ((1000, 128, 64, 3, 0, False, True), ["v2c<4,3,0>"] * 2),
    ((700, 96, 33, 3, 1, False, False), ["v2c<4,3,1>"] * 2),
    ((1000, 128, 64, 3, 2, False, False), ["v2c<4,3,2>"] * 2),
    ((1000, 96, 64, 3, 3, False, False), ["v2c<4,3,3>"] * 2),
    ((1000, 32, 33, 3, 0, False, True), ["v1<1,3,0>"]),
    ((700, 20, 8, 3, 1, True, False), ["v1<1,3,1>"]),
    ((1000, 32, 64, 3, 2, False, False), ["v1<1,3,2>"]),
    ((1000, 20, 32, 3, 3, True, False), ["v1<1,3,3>"]),
    ((1000, 20, 64, 1, 0, False, False), ["v1<1,1,0>"]),
    ((1000, 32, 33, 1, 1, False, False), ["v1<1,1,1>"]),
    ((700, 32, 8, 1, 2, True, False), ["v1<1,1,2>"]),
    ((1000, 20, 64, 1, 3, False, False), ["v1<1,1,3>"]),
    ((1000, 64, 64, 3, 0, False, False), ["v1<2,3,0>"]),
    ((700, 48, 33, 3, 1, False, False), ["v1<2,3,1>"]),
    ((1000, 64, 8, 3, 2, True, False), ["v1<2,3,2>"]),
    ((1000, 64, 64, 3, 3, False, True), ["v1<2,3,3>"]),
    ((700, 64, 32, 1, 0, True, False), ["v1<2,1,0>"]),
    ((1000, 48, 64, 1, 1, False, False), ["v1<2,1,1>"]),
    ((1000, 64, 33, 1, 2, False, False), ["v1<2,1,2>"]),
    ((1000, 48, 33, 1, 3, False, False), ["v1<2,1,3>"]),
    ((1000, 128, 64, 1, 0, False, False), ["v1<4,1,0>"]),
    ((700, 96, 32, 1, 1, True, False), ["v1<4,1,1>"]),
    ((1000, 128, 33, 1, 2, False, False), ["v1<4,1,2>"]),
    ((1000, 96, 64, 1, 3, False, True), ["v1<4,1,3>"]),
]


def _path_id(case):
    (n, d, kc, prec, nm, v1, dup), launches = case
    return f"{launches[0]}-n{n}-d{d}-kc{kc}" + ("-V1" if v1 else "") + ("-dup" if dup else "")


def test_path_table_reaches_every_instantiation():
    got = {name for _, launches in PATHS for name in launches}
    want = {f"v2<{kb},{sp},{nm}>" for kb in (1, 2, 4) for sp in (1, 3) for nm in range(4)}
    want |= {f"v1<{kb},{sp},{nm}>" for kb, sp in ((1, 3), (1, 1), (2, 3), (2, 1), (4, 1)) for nm in range(4)}
    want |= {f"v2c<4,3,{nm}>" for nm in range(4)}
    assert got == want, (want - got, got - want)


@pytest.mark.parametrize("case", PATHS, ids=[_path_id(c) for c in PATHS])
def test_path_matches_fp64_reference(case, monkeypatch):
    (n, d, kc, prec, nm, v1, dup), _ = case
    if v1:
        monkeypatch.setenv("DGGB_AP_V1", "1")
    else:
        monkeypatch.delenv("DGGB_AP_V1", raising=False)
    z = _z(n, d, n * 7 + d + kc, dup)
    noise, G = _noise(nm, n, n, n + d)
    out = _call(z, nm, kc, prec, noise)
    ref = Ref(z, G, prec, nm)
    min_exact = 0.5 if prec == 3 and not dup else 0.0   # one TF32 pass widens the tie zone past the typical gap
    ref.check(out[0], out[1], kc, min_exact, exact_ties=dup)
    if nm == 3:
        s, tol = ref.rowsum(1.0)
        assert float(((out[2].cuda().double() - s).abs() - tol).max()) <= 0


def _kernel_launches(trace_path):
    with open(trace_path) as f:
        ev = json.load(f)["traceEvents"]
    names = []
    for e in sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        m = re.search(r"allpairs_topk(2?)_kernel<(?:\(int\))?(\d+), (?:\(int\))?(\d+), (?:\(int\))?(\d+)"
                      r"(?:, (?:\(bool\))?(\w+))?>", e["name"])
        if m:
            cont = m.group(5) in ("true", "1")
            names.append(("v2c" if cont else ("v2" if m.group(1) else "v1")) + f"<{m.group(2)},{m.group(3)},{m.group(4)}>")
    return names


def test_dispatch_launches_the_tabled_kernels(monkeypatch, tmp_path):
    """The profiler's kernel names, in launch order, are the table's (so the table is the dispatch, not a guess)."""
    from torch.profiler import ProfilerActivity, profile

    want = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for (n, d, kc, prec, nm, v1, _dup), launches in PATHS:
            if v1:
                monkeypatch.setenv("DGGB_AP_V1", "1")
            else:
                monkeypatch.delenv("DGGB_AP_V1", raising=False)
            _call(torch.rand(n, d), nm, kc, prec, torch.zeros(n, n) if nm == 1 else None)
            want += launches
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(tmp_path / "trace.json"))
    assert _kernel_launches(tmp_path / "trace.json") == want


# n = 1 and n = 20 with kc = 32 / 64 on each kernel: every column in order, unused slots idx -1 / val 0
@pytest.mark.parametrize("n", [1, 20])
@pytest.mark.parametrize("kc", [32, 64])
@pytest.mark.parametrize("d,prec,nm", [(64, 3, 2), (128, 3, 1), (20, 1, 3), (96, 3, 0)])
def test_fewer_columns_than_kc(n, kc, d, prec, nm):
    z = _z(n, d, 11 * n + kc)
    noise, G = _noise(nm, n, n, 3)
    out = _call(z, nm, kc, prec, noise)
    ref = Ref(z, G, prec, nm)
    ref.check(out[0], out[1], kc, min_exact=0.0)
    if nm == 3:
        s, tol = ref.rowsum(1.0)
        assert float(((out[2].cuda().double() - s).abs() - tol).max()) <= 0


@pytest.mark.parametrize("d,kc,v1", [(64, 16, False), (64, 16, True), (32, 40, False), (128, 64, False),
                                     (128, 16, False)], ids=["v2", "v1-forced", "v1", "v2c", "v2-big"])
@pytest.mark.parametrize("inv_temp", [0.1, 1.0, 10.0])
def test_rowsum_matches_fp64(d, kc, v1, inv_temp, monkeypatch):
    """out_rowsum = sum_j exp(y_ij inv_temp) over all n columns, n = 1000 = 16 key tiles (both v2 epilogue groups
    contribute, and their partial sums are merged), within the bound derived in ``Ref.rowsum``."""
    if v1:
        monkeypatch.setenv("DGGB_AP_V1", "1")
    else:
        monkeypatch.delenv("DGGB_AP_V1", raising=False)
    n = 1000
    z = _z(n, d, 5 + d)
    idx, val, rs = _call(z, 3, kc, 3, inv_temp=inv_temp)
    ref = Ref(z, None, 3, 3)
    ref.check(idx, val, kc)
    s, tol = ref.rowsum(inv_temp)
    err = (rs.cuda().double() - s).abs()
    assert float((err - tol).max()) <= 0, (float(err.max()), float(tol.min()))


@pytest.mark.parametrize("d,kc,nm,v1", [(64, 16, 2, False), (64, 16, 3, True), (128, 64, 1, False),
                                        (64, 40, 0, False), (128, 16, 3, False), (20, 8, 1, False)])
@pytest.mark.parametrize("row_begin", [37, 300])
def test_row_block_equals_full_run(d, kc, nm, v1, row_begin, monkeypatch):
    """Rows [row_begin, n) -- a start that is not a multiple of 128 and a ragged last CTA -- give the full run's bits."""
    if v1:
        monkeypatch.setenv("DGGB_AP_V1", "1")
    else:
        monkeypatch.delenv("DGGB_AP_V1", raising=False)
    n = 1000
    rows = n - row_begin
    z = _z(n, d, 17 + d + kc)
    noise, G = _noise(nm, n, n, 9)
    full = _call(z, nm, kc, 3, noise)
    part = _call(z, nm, kc, 3, None if noise is None else noise[row_begin:], row_begin, rows)
    for a, b in zip(full, part):
        assert torch.equal(a[row_begin:], b)
    Ref(z, None if G is None else G[row_begin:], 3, nm, row_begin, rows).check(part[0], part[1], kc)


@pytest.mark.parametrize("n,d,nm", [(1000, 64, 1), (1000, 64, 2), (1000, 128, 1), (1000, 128, 2), (50, 64, 0),
                                    (50, 128, 0)])
def test_continuation_passes_match_reference(n, d, nm):
    """kc = 100 as a pass of 64 and a continuation pass of 36 (d = 64: v1; d = 128: the v2 continuation instantiation).
    n = 50: the first pass runs out of columns, so the continuation pass returns only empty slots."""
    kc = 100
    z = _z(n, d, 23 + d + nm)
    noise, G = _noise(nm, n, n, 4)
    idx, val = _passes(z, nm, kc, 3, noise)
    Ref(z, G, 3, nm).check(idx, val, kc, min_exact=0.5 if n > kc else 0.0)


@pytest.mark.parametrize("d", [24, 30, 64, 100, 128])
@pytest.mark.parametrize("kc", [8, 40, 64])
def test_pair_backward_matches_fp64_autograd(d, kc):
    """dz, dt of sum(w * y) over the selected pairs of rows [37, 37 + rows) against fp64 autograd of the same pairs.
    n = 50 with kc = 64 leaves -1 slots (their upstream gradient must be ignored); point 9 duplicates point 5, whose
    pair has D = 0 off the diagonal and gets zero gradient, as torch.cdist gives."""
    from dgg_b200 import functional as K

    n = 50 if kc == 64 else 400
    rb = 37
    rows = n - rb - 3
    gen = torch.Generator().manual_seed(d * 100 + kc)
    z0 = torch.softmax(torch.randn(n, d, generator=gen) * 2.0, -1)
    z0[rb + 9] = z0[rb + 5]
    G = torch.randn(rows, n, generator=gen) * 0.1
    G[5, rb + 9] = G[9, rb + 5] = 50.0              # the duplicate pair is selected in both of its rows
    w = torch.randn(rows, kc, generator=gen)
    z = z0.cuda().requires_grad_(True)
    t = torch.tensor([1.7], device="cuda", requires_grad=True)
    idx, val = K.allpairs_topk(z, t, G.cuda(), kc, 3, rb, rows)
    (val * w.cuda()).sum().backward()
    j = idx.cpu().long()
    assert int((j < 0).sum()) == (rows * (kc - n) if kc > n else 0)
    assert bool((j[5] == rb + 9).any()) and bool((j[9] == rb + 5).any())
    zr = z0.double().requires_grad_(True)
    tr = torch.tensor([1.7], dtype=torch.float64, requires_grad=True)
    i = torch.arange(rb, rb + rows).reshape(rows, 1).expand(rows, kc)
    keep = j >= 0
    diff = zr[i[keep]] - zr[j[keep]]
    d2 = (diff * diff).sum(-1)
    nz = d2 > 0
    dist = torch.where(nz, d2, torch.ones_like(d2)).sqrt() * nz      # zero gradient where D == 0
    rr = torch.arange(rows).reshape(rows, 1).expand(rows, kc)
    (w[keep].double() * (-tr * dist + G[rr[keep], j[keep]].double())).sum().backward()
    torch.testing.assert_close(z.grad.cpu().double(), zr.grad, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(t.grad.cpu().double(), tr.grad, rtol=1e-4, atol=1e-4)


# ---------------------------------------------------------------------------------------------------------------
# DGG_LearnableK_SDD
# ---------------------------------------------------------------------------------------------------------------
def _module(f, h, k_bias):
    import dgm

    m = dgm.DGG_LearnableK_SDD(in_dim=f, latent_dim=h)
    m.k_bias.fill_(k_bias)
    with torch.no_grad():
        m.t.fill_(20.0)         # a trained temperature: at t = 1 the initial z are too close for any tie-free row
    state = {k: v.clone() for k, v in m.state_dict().items()}
    return m.cuda(), state


@pytest.mark.parametrize("h", [64, 128])
@pytest.mark.parametrize("k_bias,bucket", [(10.0, 32), (40.0, 64), (100.0, 128)])
def test_module_matches_oracle(h, k_bias, bucket):
    """Training forward (injected noise) and the evaluation branch against oracle.allpairs_metric_forward in fp64, on
    rows whose reference order has no near-tie inside the selection window.

    Error budget of a score y_ij = -t D_ij (+ G_ij): the kernel's bound t eps / max(sqrt(eps), 2 D) + 1e-5 (module
    docstring) plus t (|dz_i| + |dz_j|) for the fp32 encoder's z (dz = its row error against the fp64 oracle, measured).
    Training: out = y first_k(rank, k), so |d out| <= dy + 1.75 |dk| |y| (the sigmoid's slope is interval / 4).
    Evaluation: out = p first_k with p = exp(y / temp) / Z, so |dp| / p <= expm1(dy / temp + log sum_j p_j e^(dy_j / temp))
    plus __expf's 2 + 1.173 |x| ulp and the fp32 row sum (n / 2 + 1 roundings of 2^-24)."""
    from oracle import dgg_oracle as O

    n, f = 300, 24
    gen = torch.Generator().manual_seed(h + bucket)
    x = torch.rand(n, f, generator=gen) * 10.0
    G = -torch.log(-torch.log(torch.rand(n, n, generator=gen).clamp(1e-9, 1 - 1e-7)))
    m, state = _module(f, h, k_bias)
    m.exact_kc = True
    p = {k: v.double() for k, v in state.items()}
    t = float(p["t"])
    for noise, temp in ((True, 1.0), (False, 0.5)):
        if noise:
            m.set_noise(G.cuda())
        with torch.no_grad():
            adj, k = m(x.cuda(), temp=temp, noise=noise)
            z = m.input_project(x.cuda()).cpu().double()
        assert m._kc_last == bucket
        r = O.allpairs_metric_forward(x.double(), p, G.double() if noise else None, temp=temp, k_bias=k_bias)
        k = k[0].cpu().double()
        torch.testing.assert_close(k, r["k"], rtol=1e-5, atol=1e-4)
        got = adj.to_dense().cpu().double()
        D = torch.cdist(r["z"], r["z"], compute_mode="donot_use_mm_for_euclid_dist")
        ez = torch.linalg.vector_norm(z - r["z"], dim=-1)
        eps = EPS[3]
        dy = torch.where(torch.eye(n, dtype=torch.bool), 0.0,
                         t * (eps / (2 * D).clamp_min(eps ** 0.5) + ez[:, None] + ez[None, :])) + 1e-5
        dk = float((k - r["k"]).abs().max())
        if noise:
            key, dkey = r["y"], dy
            tol = dy + 2.0 * dk * r["y"].abs()
        else:
            key, dkey = (-t * D) / temp, dy / temp
            pr = r["y"]
            dlogz = torch.log((pr * torch.exp(dkey)).sum(-1, keepdim=True))
            x_abs = key.abs()
            rel = torch.expm1(dkey + dlogz) + (2 + 1.173 * x_abs) * 2.0 ** -23 + (n / 2 + 1) * 2.0 ** -24
            tol = pr * rel + 2.0 * dk * pr
        # tie-free rows: every gap of the reference's top-(bucket + 1) exceeds twice the bounds of its two entries, so
        # the kernel's ranks (and with them the first-k weights) are the reference's
        srt, order = torch.sort(key, dim=-1, descending=True, stable=True)
        st = torch.gather(dkey, 1, order[:, :bucket + 1])
        ok = ((srt[:, :bucket] - srt[:, 1:bucket + 1]) > 2 * (st[:, :-1] + st[:, 1:])).all(-1)
        assert float(ok.double().mean()) > 0.15, float(ok.double().mean())
        err = (got - r["out"]).abs() - tol
        assert float(err[ok].max()) <= 0, float(err[ok].max())


@pytest.mark.parametrize("n", [6, 13])
def test_module_small_graph_selects_every_column(n):
    """n below the window: kc == n every time (no spurious K overflow), each row holds all n columns."""
    m, _ = _module(16, 64, 30.0)
    x = torch.rand(n, 16, device="cuda")
    for _ in range(4):
        with torch.no_grad():
            adj, _k = m(x, temp=1.0, noise=True)
        assert not m.overflowed()
        ind = adj.coalesce().indices()
        assert ind.shape[1] == n * n


def test_module_window_overflow_contract():
    """k grows past the window the selector ran with: overflowed() reports it, the next forward raises once (and
    enlarges the window), the one after runs."""
    import dgg_b200

    n = 400
    m, _ = _module(16, 64, 5.0)
    x = torch.rand(n, 16, device="cuda")
    with torch.no_grad():
        m(x, temp=1.0, noise=True)
        assert not m.overflowed()
        kc0 = m._kc_last
        m.k_bias.fill_(float(kc0) + 10.0)      # rows now need more than kc0 entries
        m(x, temp=1.0, noise=True)
        assert m.overflowed()
        with pytest.raises(dgg_b200.DggbError):
            m(x, temp=1.0, noise=True)
        adj, k = m(x, temp=1.0, noise=True)
        assert m._kc_last >= math.ceil(float(k.max()) + m.k_window)
        assert not m.overflowed()
