"""The k-block-streamed all-pairs instantiations (d > 128) against the fp64 reference of test_gpu_allpairs_paths.

For dpad = d rounded up to 32 above 128, ``dggb_allpairs_topk_after_fwd`` runs ``allpairs_topk_kernel<0, SP, NM>``
(``v1<0,SP,NM>`` below): v1's tile shape, warp roles and epilogue, with the query tile streamed by 32-feature
k-block together with the key tile instead of kept resident.  It runs unsplit and ignores DGGB_AP_V1 / DGGB_AP_PARTS.

Score bound.  ``Ref`` takes an absolute d2 error of EPS[prec] (|z|^2 <= 1), set at d <= 128, i.e. at most 4 k-blocks.
What grows with d is fp32 accumulation: every k-block adds SP x 4 tcgen05.mma results (8 products each; products of
TF32 values are exact in fp32) into the fp32 accumulator, each add rounding by at most 1 ulp (2^-23 relative) of a
running sum bounded by sum_k |z_ik z_jk| <= 1, and d2 takes -2 S; the squared norms from the split pre-pass add one
more fp32 add per k-block and lane for each of |z_i|^2 and |z_j|^2 (2^-24 each).  Hence, for kb = dpad / 32 > 4,
    eps(prec, d) = EPS[prec] + (kb - 4) (2 SP 4 2^-23 + 2 2^-24)
(3xTF32: 8.7e-5 at d = 1024; one TF32 pass: 1.03e-3), which ``WideRef`` puts into Ref's tolerance model."""
import pytest
import torch

from tests.test_gpu_allpairs_paths import EPS, T, Ref, _call, _kernel_launches, _noise, _passes, _z

pytestmark = pytest.mark.gpu


def eps_wide(prec, d):
    kb = -(-d // 32)
    return EPS[prec] + max(0, kb - 4) * (2 * prec * 4 * 2.0 ** -23 + 2 * 2.0 ** -24)


class WideRef(Ref):
    """Ref with the d2 bound eps_wide(prec, d) in place of EPS[prec] (same score model, see Ref)."""

    def __init__(self, z, G, prec, nm, row_begin=0, rows=None):
        super().__init__(z, G, prec, nm, row_begin, rows)
        eps = eps_wide(prec, z.shape[1])
        self.tol = torch.where(self.diag, 0.0, T * eps / (2 * self.D).clamp_min(eps ** 0.5)) + 1e-5 + \
            (5e-5 if nm == 2 else 0.0)


# (n, d, kc, precision, noise mode, duplicated points) -> launches in order
PATHS = [
    ((1000, 129, 8, 3, 0, True), ["v1<0,3,0>"]),
    ((700, 130, 32, 3, 1, False), ["v1<0,3,1>"]),      # rows of z 520 B apart: not 16-byte aligned
    ((1301, 160, 1, 3, 2, False), ["v1<0,3,2>"]),
    ((1000, 256, 33, 3, 3, False), ["v1<0,3,3>"]),
    ((1000, 200, 32, 3, 0, False), ["v1<0,3,0>"]),
    ((1000, 160, 64, 3, 0, False), ["v1<0,3,0>"]),
    ((1000, 512, 64, 3, 1, False), ["v1<0,3,1>"]),
    ((700, 384, 8, 3, 1, False), ["v1<0,3,1>"]),
    ((1301, 1024, 32, 3, 2, False), ["v1<0,3,2>"]),
    ((45, 500, 64, 3, 2, False), ["v1<0,3,2>"]),       # below one key tile, fewer columns than kc
    ((1000, 256, 64, 3, 3, True), ["v1<0,3,3>"]),
    ((45, 200, 8, 1, 0, False), ["v1<0,1,0>"]),
    ((700, 1024, 33, 1, 0, False), ["v1<0,1,0>"]),
    ((1000, 384, 64, 1, 1, False), ["v1<0,1,1>"]),
    ((700, 500, 32, 1, 2, False), ["v1<0,1,2>"]),
    ((1000, 512, 8, 1, 3, False), ["v1<0,1,3>"]),
    ((1301, 129, 1, 1, 3, False), ["v1<0,1,3>"]),
]


def _path_id(case):
    (n, d, kc, prec, nm, dup), launches = case
    return f"{launches[0]}-n{n}-d{d}-kc{kc}" + ("-dup" if dup else "")


def test_path_table_reaches_every_wide_instantiation():
    got = {name for _, launches in PATHS for name in launches}
    assert got == {f"v1<0,{sp},{nm}>" for sp in (1, 3) for nm in range(4)}
    assert {c[0][1] for c in PATHS} >= {129, 130, 160, 200, 256, 384, 500, 512, 1024}
    assert {c[0][2] for c in PATHS} >= {1, 8, 32, 33, 64}
    assert {c[0][0] for c in PATHS} >= {45, 700, 1000, 1301}


@pytest.mark.parametrize("case", PATHS, ids=[_path_id(c) for c in PATHS])
def test_wide_path_matches_fp64_reference(case):
    (n, d, kc, prec, nm, dup), _ = case
    z = _z(n, d, n * 7 + d + kc, dup)
    noise, G = _noise(nm, n, n, n + d)
    out = _call(z, nm, kc, prec, noise)
    ref = WideRef(z, G, prec, nm)
    min_exact = 0.5 if prec == 3 and not dup and n > kc else 0.0
    ref.check(out[0], out[1], kc, min_exact, exact_ties=dup)
    if nm == 3:
        s, tol = ref.rowsum(1.0)
        assert float(((out[2].cuda().double() - s).abs() - tol).max()) <= 0


# d <= 128 controls: the resident-tile kernels keep their calls
CONTROLS = [
    ((1000, 128, 32, 3, 2), ["v2<4,3,2>"]),
    ((1000, 128, 64, 3, 0), ["v2c<4,3,0>"] * 2),
    ((1000, 64, 64, 3, 1), ["v1<2,3,1>"]),
    ((700, 128, 8, 1, 3), ["v2<4,1,3>"]),
]


def test_dispatch_launches_the_wide_kernel(monkeypatch, tmp_path):
    """Every wide row launches v1<0,SP,NM> once per call, whatever DGGB_AP_V1 / DGGB_AP_PARTS say; the d <= 128
    controls launch their resident-tile kernels."""
    from torch.profiler import ProfilerActivity, profile

    monkeypatch.setenv("DGGB_AP_PARTS", "4")
    rows = [c[:5] + (v1,) for (c, l) in PATHS for v1 in (False, True)] + [c + (False,) for c, _ in CONTROLS]
    launches = [l for (_, l) in PATHS for _v1 in (False, True)] + [l for _, l in CONTROLS]
    want = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # A profiler session that is not the process's first can lose its first few kernel records: untracked
        # kernels absorb the loss before the tabled launches.
        for _ in range(32):
            torch.ones(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        for (n, d, kc, prec, nm, v1), ls in zip(rows, launches):
            if v1:
                monkeypatch.setenv("DGGB_AP_V1", "1")
            else:
                monkeypatch.delenv("DGGB_AP_V1", raising=False)
            _call(torch.rand(n, d), nm, kc, prec, torch.zeros(n, n) if nm == 1 else None)
            want += ls
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(tmp_path / "trace.json"))
    assert _kernel_launches(tmp_path / "trace.json") == want


@pytest.mark.parametrize("d", [256, 512])
@pytest.mark.parametrize("nm", [1, 2, 3])
@pytest.mark.parametrize("row_begin", [37, 300])
def test_wide_row_block_equals_full_run(d, nm, row_begin):
    """Rows [row_begin, n) -- a start that is not a multiple of 128 and a ragged last CTA -- give the full run's bits."""
    n, kc = 1000, 32
    rows = n - row_begin
    z = _z(n, d, 17 + d + nm)
    noise, G = _noise(nm, n, n, 9)
    full = _call(z, nm, kc, 3, noise)
    part = _call(z, nm, kc, 3, None if noise is None else noise[row_begin:], row_begin, rows)
    for a, b in zip(full, part):
        assert torch.equal(a[row_begin:], b)
    # without noise, d = 512 leaves near-ties in about 3 of 4 reference ranks (a property of the inputs)
    WideRef(z, None if G is None else G[row_begin:], 3, nm, row_begin, rows).check(part[0], part[1], kc,
                                                                                  0.25 if nm == 3 else 0.5)


@pytest.mark.parametrize("n,d,nm", [(1000, 256, 1), (1000, 256, 2), (1000, 512, 1), (1000, 512, 2), (50, 256, 0),
                                    (50, 512, 2)])
def test_wide_continuation_passes_match_reference(n, d, nm):
    """kc = 100 as a pass of 64 and a continuation pass of 36.  n = 50: the first pass runs out of columns, so the
    continuation pass returns only empty slots."""
    kc = 100
    z = _z(n, d, 23 + d + nm)
    noise, G = _noise(nm, n, n, 4)
    idx, val = _passes(z, nm, kc, 3, noise)
    WideRef(z, G, 3, nm).check(idx, val, kc, min_exact=0.5 if n > kc else 0.0)
    if n < kc:
        assert bool((idx[:, 64:] == -1).all())


@pytest.mark.parametrize("inv_temp", [0.1, 1.0, 10.0])
def test_wide_rowsum_matches_fp64(inv_temp):
    """out_rowsum = sum_j exp(y_ij inv_temp) over all n columns within the bound derived in ``Ref.rowsum``."""
    n, d, kc = 1000, 256, 32
    z = _z(n, d, 5 + d)
    idx, val, rs = _call(z, 3, kc, 3, inv_temp=inv_temp)
    ref = WideRef(z, None, 3, 3)
    ref.check(idx, val, kc)
    s, tol = ref.rowsum(inv_temp)
    err = (rs.cuda().double() - s).abs()
    assert float((err - tol).max()) <= 0, (float(err.max()), float(tol.min()))


@pytest.mark.parametrize("n", [1, 20])
@pytest.mark.parametrize("kc", [32, 64])
@pytest.mark.parametrize("prec,nm", [(3, 2), (3, 1), (1, 3), (3, 0)])
def test_wide_fewer_columns_than_kc(n, kc, prec, nm):
    d = 200
    z = _z(n, d, 11 * n + kc)
    noise, G = _noise(nm, n, n, 3)
    out = _call(z, nm, kc, prec, noise)
    ref = WideRef(z, G, prec, nm)
    ref.check(out[0], out[1], kc, min_exact=0.0)
    if nm == 3:
        s, tol = ref.rowsum(1.0)
        assert float(((out[2].cuda().double() - s).abs() - tol).max()) <= 0


def test_wide_many_tiles_phase_wraparound():
    """n = 37 888 (592 key tiles, 8 k-blocks each: the stage, norm-ring and accumulator phases wrap many times) with
    Philox noise; 512 rows spread over the grid against the reference of each one's 128-row block."""
    n, d, kc = 37888, 256, 32
    z = _z(n, d, 99)
    idx, val = _call(z, 2, kc, 3)
    for rb in (0, 9344, 18944, 37760):           # first, middle and last row blocks of the grid
        _, G = _noise(2, n, 128, 0, rb)
        WideRef(z, G, 3, 2, rb, 128).check(idx[rb:rb + 128], val[rb:rb + 128], kc)


@pytest.mark.parametrize("d", [130, 256, 512])
@pytest.mark.parametrize("kc", [8, 64])
def test_wide_pair_backward_matches_fp64_autograd(d, kc):
    """dz, dt of sum(w * y) over the selected pairs of rows [37, 37 + rows) against fp64 autograd of the same pairs
    (dggb_allpairs_pair_bwd at widths above one 128-feature chunk).  n = 50 with kc = 64 leaves -1 slots; point 9
    duplicates point 5, whose pair has D = 0 off the diagonal and gets zero gradient, as torch.cdist gives."""
    from dgg_b200 import functional as K

    n = 50 if kc == 64 else 400
    rb = 37
    rows = n - rb - 3
    gen = torch.Generator().manual_seed(d * 100 + kc)
    z0 = torch.softmax(torch.randn(n, d, generator=gen) * 2.0, -1)
    z0[rb + 9] = z0[rb + 5]
    G = torch.randn(rows, n, generator=gen) * 0.1
    G[5, rb + 9] = G[9, rb + 5] = 50.0
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
    dist = torch.where(nz, d2, torch.ones_like(d2)).sqrt() * nz
    rr = torch.arange(rows).reshape(rows, 1).expand(rows, kc)
    (w[keep].double() * (-tr * dist + G[rr[keep], j[keep]].double())).sum().backward()
    torch.testing.assert_close(z.grad.cpu().double(), zr.grad, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(t.grad.cpu().double(), tr.grad, rtol=1e-4, atol=1e-4)


# ---------------------------------------------------------------------------------------------------------------
# DGG_LearnableK_SDD at latent_dim > 128
# ---------------------------------------------------------------------------------------------------------------
def _module(f, h, k_bias):
    import dgm

    m = dgm.DGG_LearnableK_SDD(in_dim=f, latent_dim=h)
    m.k_bias.fill_(k_bias)
    with torch.no_grad():
        m.t.fill_(20.0)         # a trained temperature: at t = 1 the initial z are too close for any tie-free row
    state = {k: v.clone() for k, v in m.state_dict().items()}
    return m.cuda(), state


def _tie_free(key, dkey, bucket, r0):
    """Rows whose reference gaps between ranks r0 - 1 .. bucket all exceed twice the bounds of their two entries: the
    set of the first r0 entries of the row and every rank from r0 on are then the kernel's.  Inside the first r0 ranks
    (first_k >= sigmoid(16) there, see _plateau) an order the bounds cannot resolve changes out by the first_k spread
    alone, which _plateau adds to the tolerance.  (At d > 128 the wider score bound leaves few rows whose whole
    top-129 is resolved, as test_module_matches_oracle asks at d <= 128.)"""
    srt, order = torch.sort(key, dim=-1, descending=True, stable=True)
    st = torch.gather(dkey, 1, order[:, :bucket + 1])
    clear = (srt[:, :bucket] - srt[:, 1:bucket + 1]) > 2 * (st[:, :-1] + st[:, 1:])
    gap = torch.arange(bucket).reshape(1, bucket)
    return (clear | (gap < r0 - 1)).all(-1)


def _plateau(k, hs_start=2.0, interval=7.0):
    """(r0, 1 - first_k(r0 - 1)) per row: r0 = max(0, floor(k) - 3), the ranks before it carry first_k weights within
    1 - sigmoid(16) of 1 and of each other."""
    k = k.reshape(-1, 1)
    r0 = (torch.floor(k) - 3).clamp_min(0)
    return r0, torch.where(r0 > 0, 1 - torch.sigmoid(hs_start - interval * (r0 - 1) + (k - 1) * interval), 0.0)


@pytest.mark.parametrize("k_bias,bucket", [(10.0, 32), (100.0, 128)])
def test_wide_module_matches_oracle(k_bias, bucket):
    """latent_dim = 256: the training forward (injected noise) with its backward, and the evaluation branch, against
    oracle.allpairs_metric_forward in fp64 on tie-free rows (the error budget of test_module_matches_oracle with
    eps_wide); encoder and t gradients for the one-pass bucket.  bucket = 128 runs _select's two passes."""
    from oracle import dgg_oracle as O

    n, f, h = 300, 24, 256
    gen = torch.Generator().manual_seed(h + bucket)
    x = torch.rand(n, f, generator=gen) * 10.0
    G = -torch.log(-torch.log(torch.rand(n, n, generator=gen).clamp(1e-9, 1 - 1e-7)))
    w_out = torch.randn(n, n, generator=gen)
    m, state = _module(f, h, k_bias)
    m.exact_kc = True
    p = {k: v.double().requires_grad_(v.is_floating_point()) for k, v in state.items()}
    t = float(state["t"])
    eps = eps_wide(3, h)
    for noise, temp in ((True, 1.0), (False, 0.5)):
        if noise:
            m.set_noise(G.cuda())
            m.zero_grad()
            adj, k = m(x.cuda(), temp=temp, noise=True)
            with torch.no_grad():
                z = m.input_project(x.cuda()).cpu().double()
        else:
            with torch.no_grad():
                adj, k = m(x.cuda(), temp=temp, noise=False)
        assert m._kc_last == bucket
        r = O.allpairs_metric_forward(x.double(), p, G.double() if noise else None, temp=temp, k_bias=k_bias)
        kk = k[0].detach().cpu().double()
        torch.testing.assert_close(kk, r["k"].detach(), rtol=1e-5, atol=1e-4)
        got = adj.to_dense().detach().cpu().double()
        zr, yr = r["z"].detach(), r["y"].detach()
        D = torch.cdist(zr, zr, compute_mode="donot_use_mm_for_euclid_dist")
        ez = torch.linalg.vector_norm(z - zr, dim=-1)
        dy = torch.where(torch.eye(n, dtype=torch.bool), 0.0,
                         t * (eps / (2 * D).clamp_min(eps ** 0.5) + ez[:, None] + ez[None, :])) + 1e-5
        dk = float((kk - r["k"].detach()).abs().max())
        if noise:
            key, dkey = yr, dy
            tol = dy + 2.0 * dk * yr.abs()
        else:
            key, dkey = (-t * D) / temp, dy / temp
            dlogz = torch.log((yr * torch.exp(dkey)).sum(-1, keepdim=True))
            rel = torch.expm1(dkey + dlogz) + (2 + 1.173 * key.abs()) * 2.0 ** -23 + (n / 2 + 1) * 2.0 ** -24
            tol = yr * rel + 2.0 * dk * yr
        r0, spread = _plateau(r["k"].detach())
        tol = tol + yr.abs() * spread
        ok = _tie_free(key, dkey, bucket, r0)
        # at least 15 of the 300 rows (without noise, d = 256 leaves near-ties in most rows' top ranks)
        assert float(ok.double().mean()) >= 0.05, (noise, float(ok.double().mean()))
        err = (got - r["out"].detach()).abs() - tol
        assert float(err[ok].max()) <= 0, float(err[ok].max())
        if noise and bucket <= 64:
            # gradients of sum(w_out * out) of the encoder and t (the ones that flow through the selector's pair
            # backward), on the rows the forward pinned (the others are masked out of the loss on both sides so that
            # near-ties do not pick different entries).  k_net's gradient, sum_r y_r first_k'(r), carries the score
            # error dy without a bound derived here, and is left out.
            mask = ok.double()[:, None] * w_out.double()
            (adj.to_dense() * mask.float().cuda()).sum().backward()
            (r["out"] * mask).sum().backward()
            for name, q in m.named_parameters():
                if name.startswith("k_net."):
                    continue
                ref_g = p[name].grad
                if ref_g is None:           # a parameter the metric forward does not use (k_net's stochastic head)
                    assert q.grad is None, name
                    continue
                torch.testing.assert_close(q.grad.cpu().double(), ref_g, rtol=2e-3, atol=2e-4, msg=name)
