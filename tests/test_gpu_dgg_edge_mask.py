"""The branch mask of the fused DGG edge kernels (dggb_dgg_edge_fwd_fused_mask / dggb_dgg_edge_bwd_fused_mask).

The forward stores, per entry, one bit per channel (pre_c = y_u - y_v + be > 0, bit c % 32 of word c / 32) and, with
ablation noise, the pre-noise sigmoid r1; the backward reads them instead of gathering y.  Checked here:

* the mask against a torch recomputation of pre (exact: the inputs of test_gpu_dgg_edge_paths keep every pre_c at
  least q / 2 away from 0), for h = 4, 12, 64, 100 and 512, with and without noise, with hard_k; r1 against the R of
  the same forward without noise, bit for bit; and R, rank, s, k, out against the forward without a mask, bit for bit;
* the masked backward against the unmasked entry point (which runs the two-launch backward from y): both within the
  fp64 bounds of test_gpu_dgg_edge_paths, on dgg_bwd_fused2_kernel and on dgg_bwd_fused_kernel, which takes windows
  above 6 144 entries;
* argument checks of the two entry points (CPU).
"""
import ctypes

import numpy as np
import pytest
import torch

from tests.test_gpu_dgg_edge_paths import W, _bwd2_fits, _d, _prepare, _set_path, check_grads, grad_bounds

gpu = pytest.mark.gpu


def _mask_ref(g, y, be):
    """[E, ceil(h / 32)] uint32 words of (y_u - y_v + be > 0), computed in fp32 (exact on the dyadic inputs)."""
    h = y.shape[1]
    bits = ((y[g.row] - y[g.col] + be) > 0).cpu().numpy().astype(np.uint64)
    nw = (h + 31) // 32
    padded = np.zeros((bits.shape[0], nw * 32), dtype=np.uint64)
    padded[:, :h] = bits
    shifts = np.arange(32, dtype=np.uint64)
    return (padded.reshape(-1, nw, 32) << shifts).sum(axis=2).astype(np.uint32)


def _fwd(g, y, be, b, noise, hard_k, masked):
    """One fused forward through the C-ABI: (R, rank, s, k, out, mask or None, r1 or None)."""
    from dgg_b200._lib import check, i64, lib, p, stream

    n, h = y.shape
    E = g.nnz
    dev = y.device
    R, out = torch.empty(E, device=dev), torch.empty(E, device=dev)
    rank = torch.empty(E, dtype=torch.int32, device=dev)
    s, k = torch.empty(n, device=dev), torch.empty(n, device=dev)
    wt, bt = torch.full((1,), W, device=dev), torch.full((1,), b, device=dev)
    head = (p(g.csr.rowptr), p(g.csr.erow), p(g.csr.col), n, E, g.max_row, h, p(y), p(be), p(wt), p(bt), p(noise),
            hard_k, p(R), p(rank), p(s), p(k), p(out))
    mask = r1 = None
    if masked:
        mask = torch.full((E, (h + 31) // 32), -1, dtype=torch.int32, device=dev)
        r1 = torch.full((E,), float("nan"), device=dev) if noise is not None else None
        check(lib().dggb_dgg_edge_fwd_fused_mask(*head, p(mask), p(r1), None, i64(0), stream()), "fwd_mask")
    else:
        check(lib().dggb_dgg_edge_fwd_fused(*head, None, i64(0), stream()), "fwd")
    torch.cuda.synchronize()
    return R, rank, s, k, out, mask, r1


MASK_CASES = [
    # (h, hard_k, noise, mode): every lane layout of the fused kernels (L = 1 .. 32, T = 1, 2, 4, h not 16 L)
    (4, -1, False, "auto"), (4, -1, True, "auto"),
    (12, 3, False, "auto"), (12, -1, True, "auto"),
    (64, -1, False, "auto"), (64, -1, True, "auto"), (64, 1, False, "auto"),
    (100, -1, False, "auto"), (100, 3, True, "auto"),
    (512, -1, False, "auto"), (512, 0, True, "auto"),
]


@gpu
@pytest.mark.parametrize("h,hard_k,noise,mode", MASK_CASES,
                         ids=[f"h{h}-hk{k}-{'noise' if z else 'plain'}-{m}" for h, k, z, m in MASK_CASES])
def test_forward_mask_and_r1(h, hard_k, noise, mode, monkeypatch):
    c = _d("mixed", h, hard_k, noise=noise, mode=mode, seed=90 + h)
    g, y, be, nz, gout, f, b = _prepare(c)
    _set_path(monkeypatch, c)
    R, rank, s, k, out, mask, r1 = _fwd(g, y, be, b, nz, hard_k, masked=True)
    want = _mask_ref(g, y, be)
    got = mask.cpu().numpy().view(np.uint32)
    bad = np.nonzero(got != want)
    assert bad[0].size == 0, f"{bad[0].size} mask words differ, first at entry {bad[0][0]} word {bad[1][0]}: " \
                             f"got {got[bad][0]:#010x}, want {want[bad][0]:#010x}"
    # the mask and r1 change nothing else
    plain = _fwd(g, y, be, b, nz, hard_k, masked=False)
    for name, a, bb in zip(("R", "rank", "s", "k", "out"), (R, rank, s, k, out), plain[:5]):
        assert torch.equal(a, bb), name
    if nz is not None:   # r1 is the R of the same forward without noise
        R_plain = _fwd(g, y, be, b, None, hard_k, masked=False)[0]
        assert torch.equal(r1, R_plain)
        want = torch.sigmoid(r1.double() + nz.double())    # R = sigmoid(r1 + noise), a few ulp of sigmoidf_
        assert bool(((R.double() - want).abs() <= 8 * 2.0 ** -24).all())


def _bwd(g, y, be, b, nz, hard_k, R, rank, s, k, gout, mask, r1):
    from dgg_b200._lib import check, lib, p, stream

    n, h = y.shape
    dev = y.device
    dy, dbe, ddeg = torch.zeros(n, h, device=dev), torch.zeros(h, device=dev), torch.zeros(2, device=dev)
    ds_ws = torch.full((n,), float("nan"), device=dev)
    wt, bt = torch.full((1,), W, device=dev), torch.full((1,), b, device=dev)
    head = (p(g.csr.rowptr), p(g.csr.erow), p(g.csr.col), n, g.nnz, g.max_row, h)
    tail = (p(nz), hard_k, p(R), p(rank), p(s), p(k))
    if mask is not None:
        check(lib().dggb_dgg_edge_bwd_fused_mask(*head, p(wt), p(bt), *tail, p(mask), p(r1), p(gout), p(ds_ws),
                                                 p(dy), p(dbe), p(ddeg), stream()), "bwd_mask")
    else:
        check(lib().dggb_dgg_edge_bwd_fused(*head, p(y), p(be), p(wt), p(bt), *tail, p(gout), p(ds_ws), p(dy),
                                            p(dbe), p(ddeg), stream()), "bwd")
    torch.cuda.synchronize()
    return dy, dbe, ddeg[0:1], ddeg[1:2]


BWD_CASES = [
    # (graph, h, hard_k, noise, mode, epb, backward kernel of the masked entry point)
    ("mixed", 64, -1, False, "auto", None, "fused2"),
    ("mixed", 64, -1, True, "auto", None, "fused2"),
    ("mixed", 100, 3, False, "auto", None, "fused2"),
    ("blocks", 16, -1, True, "auto", 64, "fused2"),
    ("mixed", 8, 1, True, "auto", 16000, "fused"),        # windows above 6 144 entries: dgg_bwd_fused_kernel
    ("mixed", 512, -1, False, "auto", 16000, "fused"),
    ("wide", 20, -1, False, "auto", 16000, "fused"),
    ("wide", 64, 2, True, "auto", 16000, "fused"),
]


@gpu
@pytest.mark.parametrize("graph,h,hard_k,noise,mode,epb,kernel", BWD_CASES,
                         ids=[f"{c[0]}-h{c[1]}-hk{c[2]}-{'noise' if c[3] else 'plain'}-{c[4]}-{c[6]}"
                              for c in BWD_CASES])
def test_masked_backward_matches_the_unmasked_entry_point(graph, h, hard_k, noise, mode, epb, kernel, monkeypatch):
    c = _d(graph, h, hard_k, noise=noise, mode=mode, epb=epb, seed=95 + h)
    g, y, be, nz, gout, f, b = _prepare(c)
    _set_path(monkeypatch, c)
    assert _bwd2_fits(g.nnz, g.max_row, epb) == (kernel == "fused2")
    R, rank, s, k, out, mask, r1 = _fwd(g, y, be, b, nz, hard_k, masked=True)
    ref, bounds = grad_bounds(g, f, hard_k, nz, rank, gout, y.double(), be.double())
    new = _bwd(g, y, be, b, nz, hard_k, R, rank, s, k, gout, mask, r1)
    old = _bwd(g, y, be, b, nz, hard_k, R, rank, s, k, gout, None, None)
    check_grads(new, ref, bounds, hard_k)
    check_grads(old, ref, bounds, hard_k)
    # one against the other: within the sum of both bounds
    dyb, dbeb = bounds[0], bounds[1]
    assert bool(((new[0].double() - old[0].double()).abs() <= 2 * dyb).all())
    assert bool(((new[1].double() - old[1].double()).abs() <= 2 * dbeb).all())


def test_mask_entry_points_reject_bad_arguments():
    import dgg_b200

    L = dgg_b200.lib()
    one = ctypes.c_void_p(16)          # never dereferenced
    null = None
    BAD_ARG, BAD_SHAPE, UNSUPPORTED = -1, -2, -3

    def ffwd(nnz=8, mx=4, h=16, noise=null, mask=one, r1=null, R=one):
        return L.dggb_dgg_edge_fwd_fused_mask(one, one, one, 4, nnz, mx, h, one, one, one, one, noise, -1, R, one, one,
                                              one, one, mask, r1, null, 0, null)

    assert ffwd(noise=one) == BAD_ARG                  # noise and a mask: the backward needs r1
    assert ffwd(R=null) == BAD_ARG and ffwd(mx=-1) == BAD_ARG
    assert ffwd(h=6) == BAD_SHAPE
    assert ffwd(mx=513) == UNSUPPORTED and ffwd(nnz=0) == UNSUPPORTED
    assert ffwd(noise=one, mask=null, mx=513) == UNSUPPORTED    # no mask: r1 is not needed
    assert ffwd(noise=one, r1=one, mx=513) == UNSUPPORTED

    def fbwd(nnz=8, mx=4, h=16, noise=null, mask=one, r1=null, ds=one):
        return L.dggb_dgg_edge_bwd_fused_mask(one, one, one, 4, nnz, mx, h, one, one, noise, -1, one, one, one, one,
                                              mask, r1, one, ds, one, one, one, null)

    assert fbwd(mask=null) == BAD_ARG and fbwd(ds=null) == BAD_ARG
    assert fbwd(noise=one) == BAD_ARG                  # noise without r1
    assert fbwd(h=6) == BAD_SHAPE
    assert fbwd(mx=513) == UNSUPPORTED and fbwd(nnz=0) == UNSUPPORTED
    assert fbwd(noise=one, r1=one, mx=513) == UNSUPPORTED
