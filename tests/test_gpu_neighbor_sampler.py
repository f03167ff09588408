"""The device-side k-hop neighbour sampler (csrc/neighbor.cu, dgg_b200.samplers.neighbor_sample / NeighborLoader).

PyG's NeighborLoader (train_pubmed.py:370-375) is not in the reference tree and not installed, and its samples differ
from these by design (another RNG stream, another within-target order of Floyd's picks): the GPU output is bit-exact
against the sequential restatement in tests/neighbor_ref.py only.  Properties that do not depend on the restatement
(parent edges, per-target counts, distinct picks, unique n_id, determinism, uniform picks) are checked on their own.
The tests without the gpu mark check argument validation and never touch the device."""
import ctypes
import types

import numpy as np
import pytest
import torch

from tests.neighbor_ref import neighbor_sample_ref

gpu = pytest.mark.gpu


def _edges(n, avg_deg, seed, isolated=3, loops=5, multi=7, hub_deg=0):
    """int64 [2, E] (source, target): random edges, the last `isolated` nodes without in-edges, `loops` self loops,
    `multi` repeated edges and, with hub_deg > 0, node 0 as the target of hub_deg edges."""
    gen = torch.Generator().manual_seed(seed)
    m = n * avg_deg
    src = torch.randint(0, n, (m,), generator=gen)
    dst = torch.randint(0, n - isolated, (m,), generator=gen)
    lo = torch.randint(0, n - isolated, (loops,), generator=gen)
    dup = torch.randint(0, m, (multi,), generator=gen)
    src, dst = torch.cat([src, lo, src[dup]]), torch.cat([dst, lo, dst[dup]])
    if hub_deg:
        src = torch.cat([src, torch.randint(0, n, (hub_deg,), generator=gen)])
        dst = torch.cat([dst, torch.zeros(hub_deg, dtype=torch.long)])
    perm = torch.randperm(src.numel(), generator=gen)            # callers' edge ids are in no particular order
    return torch.stack([src[perm], dst[perm]])


def _csc_host(ei, n):
    perm = np.argsort((ei[1] * n + ei[0]).numpy(), kind="stable")
    colptr = np.concatenate([[0], np.cumsum(np.bincount(ei[1].numpy(), minlength=n))])
    return colptr, ei[0].numpy()[perm], perm


def _csc_device(ei, n):
    from dgg_b200 import CSRGraph

    eic = ei.cuda()
    perm = torch.argsort(eic[1] * n + eic[0], stable=True)
    return CSRGraph.from_indices(eic.flip(0)[:, perm].contiguous(), n)


def _seeds(n, b, seed, first=()):
    rest = [int(v) for v in torch.randperm(n, generator=torch.Generator().manual_seed(seed)) if int(v) not in first]
    return np.array(list(first) + rest[:b - len(first)], dtype=np.int64)


def _run(csc, seeds, num_neighbors, seed, replace=False):
    from dgg_b200 import samplers

    n_id, ei, pos, nn, ne = samplers.neighbor_sample(csc, torch.as_tensor(seeds, dtype=torch.int32).cuda(),
                                                     num_neighbors, seed, replace)
    return n_id.cpu().numpy().astype(np.int64), ei.cpu().numpy(), pos.cpu().numpy().astype(np.int64), nn, ne


# (n, avg in-degree, hub in-degree, seeds, num_neighbors, replace)
CASES = {
    "floyd": (300, 12, 0, 20, [5, 3], False),
    "all_entries": (300, 6, 0, 15, [-1, 40], False),
    "zero_fanout": (300, 8, 0, 20, [0, 4], False),
    "zero_fanout_last": (300, 8, 0, 20, [3, 0], False),
    "replace": (300, 8, 0, 20, [6, 4], True),
    "replace_all": (300, 8, 0, 20, [-1, 9], True),
    "hub_1024": (3000, 2, 5000, 12, [1024, 2], False),
    "hub_1024_replace": (3000, 2, 5000, 12, [1024], True),
    "one_hop": (400, 10, 0, 30, [4], False),
    "three_hops": (400, 10, 0, 30, [4, 3, 2], False),
    "no_hops": (50, 3, 0, 5, [], False),
    "no_new_nodes": (60, 4, 0, 60, [3, 2], False),          # every node is a seed: hop 0 finds nothing new
    "few_new_nodes": (60, 6, 0, 55, [-1, 2, 2], False),     # later hops emit edges but discover no node
}


@gpu
@pytest.mark.parametrize("case", list(CASES))
def test_matches_the_restatement_bit_for_bit(case):
    n, deg, hub, b, fanout, replace = CASES[case]
    ei = _edges(n, deg, seed=len(case), hub_deg=hub)
    colptr, row, _ = _csc_host(ei, n)
    # an isolated target (no in-edges) among the seeds, and the hub when there is one
    seeds = _seeds(n, b, seed=b, first=((0,) if hub else ()) + (n - 1,))
    seed = 0x0123_4567_89AB_CDEF ^ len(case)
    got = _run(_csc_device(ei, n), seeds, fanout, seed, replace)
    want = neighbor_sample_ref(colptr, row, seeds, fanout, seed, replace)
    for g, w, what in zip(got, want, ("n_id", "edge_index", "pos", "num_sampled_nodes", "num_sampled_edges")):
        assert np.array_equal(np.asarray(g), np.asarray(w)), what
    assert sum(got[4]) > 0 or not fanout or fanout[0] == 0


@gpu
def test_no_seeds_give_an_empty_sample():
    n_id, ei, pos, nn, ne = _run(_csc_device(_edges(50, 3, seed=6), 50), np.zeros(0, dtype=np.int64), [4, 2], 1)
    assert n_id.shape == (0,) and ei.shape == (2, 0) and pos.shape == (0,) and nn == [0, 0, 0] and ne == [0, 0]


@gpu
def test_properties_independent_of_the_restatement():
    n, k = 2000, [10, 5]
    ei = _edges(n, 8, seed=1)
    colptr, row, perm = _csc_host(ei, n)
    csc = _csc_device(ei, n)
    seeds = _seeds(n, 64, seed=2, first=(n - 1, n - 2))
    n_id, sei, pos, nn, ne = _run(csc, seeds, k, seed=99)
    # n_id unique, seeds first; counts consistent
    assert len(np.unique(n_id)) == len(n_id) and np.array_equal(n_id[:len(seeds)], seeds)
    assert sum(nn) == len(n_id) and sum(ne) == sei.shape[1] == len(pos)
    # every sampled edge is a parent edge: the caller's edge id maps back to (n_id[src], n_id[dst])
    e_id = perm[pos]
    assert np.array_equal(n_id[sei[0]], ei[0].numpy()[e_id]) and np.array_equal(n_id[sei[1]], ei[1].numpy()[e_id])
    # per target: min(d, k) entries, all distinct positions, inside the target's own CSC range
    hop_of = np.repeat(np.arange(len(k)), ne)
    starts = np.cumsum([0] + nn)
    for h, kh in enumerate(k):
        for t in range(starts[h], starts[h + 1]):
            mine = pos[(hop_of == h) & (sei[1] == t)]
            v = n_id[t]
            assert len(mine) == min(colptr[v + 1] - colptr[v], kh)
            assert len(np.unique(mine)) == len(mine)
            assert ((mine >= colptr[v]) & (mine < colptr[v + 1])).all()
    # determinism: the same seed twice (and after another seed in between) is bitwise equal
    _run(csc, seeds, k, seed=100)
    again = _run(csc, seeds, k, seed=99)
    for a, b in zip((n_id, sei, pos), again[:3]):
        assert np.array_equal(a, b)


@gpu
def test_floyd_picks_are_uniform():
    """4 000 targets with 40 in-edges each, 10 picks without replacement: every position within the target is
    picked with probability 1/4.  An off-by-one in the draw range skews the last positions by a quarter or more."""
    from scipy.stats import chisquare

    t, d, k = 4000, 40, 10
    n = t + d
    src = torch.arange(t, t + d).repeat(t)                     # the same 40 sources for every target
    dst = torch.arange(t).repeat_interleave(d)
    ei = torch.stack([src, dst])
    colptr, _, _ = _csc_host(ei, n)
    n_id, sei, pos, _, _ = _run(_csc_device(ei, n), np.arange(t), [k], seed=2024)
    q = pos - colptr[n_id[sei[1]]]
    hist = np.bincount(q, minlength=d)
    assert hist.sum() == t * k
    assert chisquare(hist).pvalue > 1e-3, hist
    # the pairs are uniform too: the first pick of a target (its smallest position) follows C(d-1-p, k-1) / C(d, k)
    first = q.reshape(t, k).min(1)
    from math import comb
    expect = np.array([comb(d - 1 - p, k - 1) / comb(d, k) for p in range(d - k + 1)]) * t
    obs = np.bincount(first, minlength=d - k + 1)
    keep = expect >= 5
    f_obs = np.append(obs[keep], obs[~keep].sum())
    f_exp = np.append(expect[keep], expect[~keep].sum())
    assert chisquare(f_obs, f_exp * f_obs.sum() / f_exp.sum()).pvalue > 1e-3


@gpu
def test_repeated_or_invalid_seeds_raise_and_leave_the_workspace_usable():
    from dgg_b200 import samplers

    n = 300
    ei = _edges(n, 6, seed=4)
    colptr, row, _ = _csc_host(ei, n)
    csc = _csc_device(ei, n)
    for bad in ([3, 7, 3], [3, n], [-1, 2]):
        with pytest.raises(ValueError):
            samplers.neighbor_sample(csc, torch.tensor(bad, dtype=torch.int32, device="cuda"), [4, 2], 5)
    with pytest.raises(ValueError):
        samplers.neighbor_sample(csc, torch.tensor([1], dtype=torch.int32, device="cuda"), [1025], 5)
    seeds = _seeds(n, 10, seed=3)
    got = _run(csc, seeds, [4, 2], 5)
    want = neighbor_sample_ref(colptr, row, seeds, [4, 2], 5)
    for g, w in zip(got, want):
        assert np.array_equal(np.asarray(g), np.asarray(w))


def _data(n=500, deg=6, f=8, seed=0):
    gen = torch.Generator().manual_seed(seed)
    ei = _edges(n, deg, seed=seed)
    e = ei.shape[1]
    return types.SimpleNamespace(x=torch.randn(n, f, generator=gen), y=torch.randint(0, 3, (n,), generator=gen),
                                 train_mask=torch.rand(n, generator=gen) < 0.3, edge_index=ei,
                                 edge_attr=torch.randn(e, 2, generator=gen), num_nodes=n)


def _check_batch(batch, data, num_neighbors):
    n_id, e_id = batch.n_id.cpu(), batch.e_id.cpu()
    assert torch.equal(batch.x.cpu(), data.x[n_id]) and torch.equal(batch.y.cpu(), data.y[n_id])
    assert torch.equal(batch.train_mask.cpu(), data.train_mask[n_id])
    assert torch.equal(batch.edge_attr.cpu(), data.edge_attr[e_id])
    assert torch.equal(n_id[batch.edge_index.cpu()], data.edge_index[:, e_id])
    assert batch.num_nodes == n_id.numel() == sum(batch.num_sampled_nodes)
    assert batch.num_sampled_nodes[0] == batch.batch_size
    assert len(batch.num_sampled_edges) == len(num_neighbors) and sum(batch.num_sampled_edges) == e_id.numel()


@gpu
@pytest.mark.parametrize("kind", ["mask", "index", "none"])
@pytest.mark.parametrize("drop_last", [False, True])
def test_loader_input_nodes_and_partial_batches(kind, drop_last):
    from dgg_b200.samplers import NeighborLoader

    data = _data()
    inputs = {"mask": data.train_mask, "index": torch.randperm(500, generator=torch.Generator().manual_seed(1))[:70],
              "none": None}[kind]
    want = {"mask": data.train_mask.nonzero().view(-1), "index": inputs, "none": torch.arange(500)}[kind]
    bs = 32
    loader = NeighborLoader(data, num_neighbors=[5, 3], input_nodes=inputs, batch_size=bs, drop_last=drop_last,
                            num_workers=4, persistent_workers=True)
    full, rest = divmod(want.numel(), bs)
    assert rest > 0 and len(loader) == full + (0 if drop_last else 1)
    seen = []
    for batch in loader:
        _check_batch(batch, data, [5, 3])
        seen.append(batch.n_id[:batch.batch_size].cpu())
    sizes = [s.numel() for s in seen]
    assert sizes == [bs] * full + ([] if drop_last else [rest])
    assert torch.equal(torch.cat(seen), want[:sum(sizes)])


@gpu
def test_loader_is_reproducible_under_manual_seed():
    from dgg_b200.samplers import NeighborLoader

    data = _data(seed=3)
    loader = NeighborLoader(data, num_neighbors=[4, 4], batch_size=50, shuffle=True)

    def epoch():
        torch.manual_seed(7)
        return [(b.n_id.cpu(), b.edge_index.cpu(), b.e_id.cpu()) for b in loader]

    a, b = epoch(), epoch()
    assert len(a) == len(b) == 10
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            assert torch.equal(u, v)
    assert not torch.equal(torch.cat([x[0][:50] for x in a]), torch.arange(500))      # shuffled
    assert torch.equal(torch.cat([x[0][:50] for x in a]).sort().values, torch.arange(500))


@gpu
def test_gcn_dgg_00_training_step_on_a_sampled_batch():
    import argparse

    import model
    from dgg_b200.samplers import NeighborLoader

    n, f, h, c = 3000, 32, 32, 4
    data = _data(n=n, deg=5, f=f, seed=5)
    data.y = data.y % c
    loader = NeighborLoader(data, num_neighbors=[10, 5], input_nodes=data.train_mask, batch_size=128, shuffle=True)
    torch.manual_seed(0)
    net = model.GCN_DGG_00(nfeat=f, nhidden=h, nclass=c,
                           args=argparse.Namespace(extra_edge_dim=0, dgg_adj_input="input_adj")).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-2)
    batch = next(iter(loader))
    m = batch.num_nodes
    adj = torch.sparse_coo_tensor(batch.edge_index.flip(0), torch.ones(batch.edge_index.shape[1], device="cuda"),
                                  (m, m)).coalesce()
    out, _, _ = net(batch.x, adj)
    loss = torch.nn.functional.nll_loss(out[:batch.batch_size], batch.y[:batch.batch_size])
    opt.zero_grad()
    loss.backward()
    assert out.shape == (m, c) and torch.isfinite(out).all() and torch.isfinite(loss)
    grads = [q.grad for q in net.parameters() if q.grad is not None]
    assert grads and all(torch.isfinite(g).all() for g in grads)
    opt.step()


def test_entry_points_reject_bad_arguments_without_touching_the_gpu():
    import dgg_b200

    L = dgg_b200.lib()
    null, one = ctypes.c_void_p(0), ctypes.c_void_p(16)      # `one` is never dereferenced: the checks fire first
    bad_arg, bad_shape = -1, -2
    assert L.dggb_neighbor_seed(null, 4, 10, one, one, None) == bad_arg
    assert L.dggb_neighbor_seed(one, -1, 10, one, one, None) == bad_arg
    assert L.dggb_neighbor_seed(one, 4, 10, one, null, None) == bad_arg
    assert L.dggb_neighbor_count(null, 10, one, 4, 5, 0, one, None) == bad_arg
    assert L.dggb_neighbor_count(one, 10, one, -1, 5, 0, one, None) == bad_arg
    assert L.dggb_neighbor_count(one, 10, one, 4, 1025, 0, one, None) == bad_shape
    args = [one, one, one, 4, 5, 0, 0, 1, 0, one, one, one, one, one, None]
    for i in (0, 1, 2, 9, 10, 11, 12, 13):
        assert L.dggb_neighbor_sample(*(args[:i] + [null] + args[i + 1:])) == bad_arg, i
    assert L.dggb_neighbor_sample(*(args[:3] + [-1] + args[4:])) == bad_arg
    assert L.dggb_neighbor_sample(*(args[:4] + [1025] + args[5:])) == bad_shape
    assert L.dggb_neighbor_sample(*(args[:6] + [255] + args[7:])) == bad_shape
    assert L.dggb_neighbor_flag(one, null, 4, one, one, one, None) == bad_arg
    assert L.dggb_neighbor_flag(one, one, -2, one, one, one, None) == bad_arg
    assert L.dggb_neighbor_assign(one, one, 4, null, one, 0, one, one, None) == bad_arg
    assert L.dggb_neighbor_assign(one, one, -1, one, one, 0, one, one, None) == bad_arg
    assert L.dggb_neighbor_edges(one, one, one, -1, one, one, None) == bad_arg
    assert L.dggb_neighbor_edges(one, one, one, 4, one, null, None) == bad_arg
    assert L.dggb_neighbor_reset(null, 4, 10, one, one, None) == bad_arg
    assert L.dggb_neighbor_reset(one, -3, 10, one, one, None) == bad_arg


def test_loader_rejects_unsupported_options_before_touching_the_gpu():
    from dgg_b200.samplers import NeighborLoader

    data = _data(n=40, deg=2)
    with pytest.raises(NotImplementedError):
        NeighborLoader(data, [2], directed=False)
    with pytest.raises(NotImplementedError):
        NeighborLoader(data, [2], disjoint=True)
    with pytest.raises(NotImplementedError):
        NeighborLoader(data, [2], time_attr="time")
    with pytest.raises(NotImplementedError):
        NeighborLoader(data, {("paper", "cites", "paper"): [2]})
    with pytest.raises(NotImplementedError):
        NeighborLoader(data, [2], input_nodes=("paper", torch.arange(3)))
    with pytest.raises(ValueError):
        NeighborLoader(data, [2], input_nodes=torch.tensor([1, 5, 1]))
    with pytest.raises(ValueError):
        NeighborLoader(data, [2], input_nodes=torch.tensor([1, 40]))
    with pytest.raises(ValueError):
        NeighborLoader(data, [2], input_nodes=torch.ones(39, dtype=torch.bool))


def test_restatement_follows_the_stated_rules():
    """The restatement itself on a hand-checked graph: target 0 has in-neighbours 1, 2, 3; node 3 has 0 and 3."""
    colptr = np.array([0, 3, 3, 3, 5])
    row = np.array([1, 2, 3, 0, 3])
    n_id, ei, pos, nn, ne = neighbor_sample_ref(colptr, row, [0], [-1, -1], seed=1)
    assert n_id.tolist() == [0, 1, 2, 3] and nn == [1, 3, 0] and ne == [3, 2]
    assert ei.tolist() == [[1, 2, 3, 0, 3], [0, 0, 0, 3, 3]] and pos.tolist() == [0, 1, 2, 3, 4]
