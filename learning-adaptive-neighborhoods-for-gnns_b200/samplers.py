"""Device-side sub-graph samplers for the mini-batch drivers (SURVEY 8f rank 2).

``train_large_graphs.py:402-413`` / ``train_reddit.py:400-411`` build their mini-batches with
``torch_geometric.loader.GraphSAINTRandomWalkSampler(data, batch_size=, walk_length=, num_steps=, sample_coverage=,
save_dir=, num_workers=)`` -- third-party, CPU, worker processes; every batch is then moved to the device and converted
edge list -> scipy -> torch sparse (train_large_graphs.py:226-233).  ``GraphSAINTRandomWalkSampler`` here keeps the
constructor and the batch attribute surface (``x``, ``y``, ``edge_index``, the ``*_mask`` / edge attributes of the
parent, ``node_norm`` / ``edge_norm`` when ``sample_coverage > 0``, ``num_nodes``, ``.to(device)``) but samples on the
GPU from the int32 CSR the rest of the path uses: ``dggb_random_walk`` (one thread per walker, Philox uniforms) and
``dggb_induced_subgraph_count/fill``.  A maintainer swaps ``import torch_geometric.loader as dataloaders`` for
``import dgg_b200.samplers as dataloaders``.

Semantics restated from PyG 2.1 ``GraphSAINTSampler`` / torch_sparse (neither is in the reference tree: parity is
pinned only against the Python restatement in tests/test_gpu_sampler.py, i.e. **unpinned** against the library):
start nodes ``torch.randint(0, N, (batch_size,))`` from the global CPU generator (what ``torch.manual_seed(args.seed)``
of the scripts seeds), uniform neighbour choice per step, walkers on a node without out-edges stay, the batch is the
sub-graph induced by the sorted unique visited nodes with all parent edges between them in row-major order, and the
normalisation statistics are visit counts over pre-sampled batches (``edge_norm = node_count[row] / edge_count``
clamped to 1e4, ``node_norm = num_samples / node_count / N``).

``train_pubmed.py:370-375`` feeds its mini-batches from ``torch_geometric.loader.NeighborLoader(data,
num_neighbors=[50, 50], ...)``.  ``NeighborLoader`` here follows the PyG 2.x constructor and batch surface for
homogeneous graphs (``n_id``, ``e_id``, ``batch_size``, ``num_sampled_nodes``, ``num_sampled_edges``, node / edge
attributes sliced by them) and samples on the GPU with ``neighbor_sample`` over ``dggb_neighbor_*``
(csrc/neighbor.cu): a without-replacement draw per target (Floyd's algorithm, as torch_sparse) or k draws with
replacement, then the de-duplication and relabelling of the sampled nodes in torch_sparse's sequential order.  Samples
are NOT PyG's samples for the same seed: the RNG stream differs (Philox keyed on the batch seed, the hop, the frontier
slot and the draw) and so does the within-target order of Floyd's picks (ascending here).  Parity is pinned only
against the restatement in tests/neighbor_ref.py.

The Cluster-GCN branch of ``train_large_graphs.py`` uses ``torch_geometric.loader.ClusterData`` (METIS on host cores
through torch_sparse) and ``ClusterLoader``.  ``ClusterData`` / ``ClusterLoader`` here follow the PyG 2.1 surface and
partition on the GPU with ``partition`` over ``dggb_partition_*`` (csrc/partition.cu): a deterministic multilevel k-way
partitioner (size-constrained label-propagation coarsening, a BFS-order split of the coarsest graph, label-propagation
refinement and an exact rebalance), every part non-empty and at most ``ceil(1.03 N / num_parts)`` nodes.  The parts
are NOT METIS's: parity is pinned only against the restatement in tests/cluster_ref.py.
"""
from __future__ import annotations

import torch

from ._lib import check, i32, i64, lib, p, stream
from .graph import CSRGraph


class SubgraphBatch:
    """Attribute bag standing in for ``torch_geometric.data.Data`` (``.to`` / ``.num_nodes`` / ``.keys()``)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def keys(self):
        return [k for k in self.__dict__ if not k.startswith("_")]

    def to(self, device, non_blocking=False):
        for k, v in list(self.__dict__.items()):
            if torch.is_tensor(v):
                setattr(self, k, v.to(device, non_blocking=non_blocking))
        return self

    @property
    def num_edges(self):
        return int(self.edge_index.shape[1])


def _data_items(data):
    keys = data.keys() if callable(getattr(data, "keys", None)) else getattr(data, "keys", None)
    if keys is None:
        keys = [k for k in vars(data) if not k.startswith("_")]
    return [(k, getattr(data, k)) for k in keys]


def _split_attrs(data, n, e, dev):
    """-> (node attributes [n, ...] on dev, edge attributes [e, ...] on dev, everything else), by leading size."""
    node_attrs, edge_attrs, other = {}, {}, {}
    for k, v in _data_items(data):
        if k in ("edge_index", "num_nodes"):
            continue
        if torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == n:
            node_attrs[k] = v.to(dev)
        elif torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == e:
            edge_attrs[k] = v.to(dev)
        else:
            other[k] = v
    return node_attrs, edge_attrs, other


def induced_subgraph(graph: CSRGraph, nodes: torch.Tensor):
    """Sub-graph induced by the sorted unique int32 node list -> (CSRGraph over len(nodes) nodes, eid int32 [E'] =
    positions of the kept entries in ``graph``).  One device->host read (the entry count sizes the outputs)."""
    assert nodes.is_cuda and nodes.dtype == torch.int32 and nodes.dim() == 1
    m = int(nodes.numel())
    dev = nodes.device
    relabel = torch.empty(graph.n, dtype=torch.int32, device=dev)
    counts = torch.empty(m + 1, dtype=torch.int32, device=dev)
    L = lib()
    check(L.dggb_induced_subgraph_count(p(graph.rowptr), p(graph.col), i32(graph.n), p(nodes), i32(m), p(relabel),
                                        p(counts), stream()), "induced_subgraph_count")
    sub_rowptr = torch.zeros(m + 1, dtype=torch.int32, device=dev)
    torch.cumsum(counts[:m], 0, out=sub_rowptr[1:])
    nnz = int(sub_rowptr[-1].item())
    sub_col = torch.empty(nnz, dtype=torch.int32, device=dev)
    sub_eid = torch.empty(nnz, dtype=torch.int32, device=dev)
    check(L.dggb_induced_subgraph_fill(p(graph.rowptr), p(graph.col), p(nodes), i32(m), p(relabel), p(sub_rowptr),
                                       p(sub_col), p(sub_eid), stream()), "induced_subgraph_fill")
    return CSRGraph(m, sub_rowptr, sub_col), sub_eid


def random_walk(graph: CSRGraph, start: torch.Tensor, walk_length: int, seed: int, walker_offset: int = 0):
    """-> int32 [len(start), walk_length + 1] (column 0 = start)."""
    assert start.is_cuda and start.dtype == torch.int32
    b = int(start.numel())
    walk = torch.empty(b, walk_length + 1, dtype=torch.int32, device=start.device)
    check(lib().dggb_random_walk(p(graph.rowptr), p(graph.col), i32(graph.n), p(start), i32(b), i32(walk_length),
                                 int(seed) & 0xFFFFFFFFFFFFFFFF, i64(walker_offset), p(walk), stream()), "random_walk")
    return walk


class GraphSAINTRandomWalkSampler:
    """``for batch in loader`` yields ``num_steps`` sub-graphs per epoch (``__len__ == num_steps``)."""

    def __init__(self, data, batch_size, walk_length, num_steps=1, sample_coverage=0, save_dir=None, log=True,
                 device=None, **kwargs):
        assert data.edge_index is not None
        self.data = data
        self.walk_length = int(walk_length)
        self.num_steps = int(num_steps)
        self.batch_size = int(batch_size)
        self.sample_coverage = sample_coverage
        dev = torch.device(device) if device is not None else (
            data.edge_index.device if data.edge_index.is_cuda else torch.device("cuda"))
        self.device = dev
        self.N = int(getattr(data, "num_nodes", None) or data.x.shape[0])
        ei = data.edge_index.to(dev)
        self.E = int(ei.shape[1])
        # parent adjacency in CSR order; perm maps a CSR position to the caller's edge id (edge attributes follow it)
        key = ei[0] * self.N + ei[1]
        self.perm = torch.argsort(key, stable=True)
        self.graph = CSRGraph.from_indices(ei[:, self.perm].contiguous(), self.N)
        self._node_attrs, self._edge_attrs, self._other = _split_attrs(data, self.N, self.E, dev)
        self.node_norm = self.edge_norm = None
        if self.sample_coverage > 0:
            self.node_norm, self.edge_norm = self._compute_norm()

    def __len__(self):
        return self.num_steps

    # -------------------------------------------------------------------------------------------- sampling
    def _sample(self):
        """-> (node_idx int32 sorted unique, sub CSRGraph, eid int32 positions in the parent CSR)."""
        start = torch.randint(0, self.N, (self.batch_size,), dtype=torch.long)       # global CPU generator, as PyG
        seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.long))
        walk = random_walk(self.graph, start.to(self.device, dtype=torch.int32), self.walk_length, seed)
        node_idx = torch.unique(walk.reshape(-1))                                    # sorted ascending
        sub, eid = induced_subgraph(self.graph, node_idx.to(torch.int32))
        return node_idx, sub, eid

    def _compute_norm(self):
        node_count = torch.zeros(self.N, dtype=torch.float32, device=self.device)
        edge_count = torch.zeros(self.E, dtype=torch.float32, device=self.device)
        num_samples = total = 0
        while total < self.N * self.sample_coverage:
            node_idx, _, eid = self._sample()
            node_count[node_idx.long()] += 1
            edge_count[eid.long()] += 1
            total += int(node_idx.numel())
            num_samples += 1
        row = self.graph.erow.long()
        edge_norm = (node_count[row] / edge_count).clamp_(0, 1e4)
        edge_norm[torch.isnan(edge_norm)] = 0.1
        node_count[node_count == 0] = 0.1
        node_norm = num_samples / node_count / self.N
        return node_norm, edge_norm        # edge_norm is indexed by CSR position

    def _collate(self, node_idx, sub, eid):
        nl, el = node_idx.long(), eid.long()
        batch = SubgraphBatch(num_nodes=int(node_idx.numel()), edge_index=sub.coo_indices())
        for k, v in self._node_attrs.items():
            setattr(batch, k, v[nl])
        orig = self.perm[el]
        for k, v in self._edge_attrs.items():
            setattr(batch, k, v[orig])
        for k, v in self._other.items():
            setattr(batch, k, v)
        if self.node_norm is not None:
            batch.node_norm = self.node_norm[nl]
            batch.edge_norm = self.edge_norm[el]
        batch._csr = sub           # consumers inside this package skip the edge list -> CSR conversion
        return batch

    def __iter__(self):
        for _ in range(self.num_steps):
            yield self._collate(*self._sample())


# ------------------------------------------------------------------------------------------------ neighbour sampling
_MAX_FANOUT, _MAX_HOPS, _INT32_MAX = 1024, 255, 2 ** 31 - 1


def _neighbor_workspace(csc: CSRGraph):
    """(local int32 [N] = -1, claim int32 [N] = INT32_MAX), allocated once per graph; every call puts back the entries
    it touched."""
    ws = csc.aux.get("neighbor_ws")
    if ws is None:
        dev = csc.col.device
        ws = (torch.full((csc.n,), -1, dtype=torch.int32, device=dev),
              torch.full((csc.n,), _INT32_MAX, dtype=torch.int32, device=dev))
        csc.aux["neighbor_ws"] = ws
    return ws


def neighbor_sample(csc: CSRGraph, seeds: torch.Tensor, num_neighbors, seed: int, replace: bool = False):
    """k-hop neighbour sampling on the device (the contract of ``dggb_neighbor_*`` in include/dggb.h).

    ``csc``: the parent graph over in-neighbours, as a CSRGraph whose ``rowptr`` is the CSC colptr and whose ``col``
    holds the sources: the entries of target v are the u of the edges u -> v, sorted by u.  ``seeds``: unique int32
    node ids on the device.  ``num_neighbors``: fanout per hop, -1 for every in-neighbour, at most 1024.  ``seed``:
    the 64-bit Philox key.

    Returns ``(n_id, edge_index, pos, num_sampled_nodes, num_sampled_edges)``: ``n_id`` int32 [M] with the seeds first
    and then each hop's new nodes in discovery order; ``edge_index`` int64 [2, E] of local ids (row 0 the source, row 1
    the target); ``pos`` int32 [E], the CSC position of every sampled entry; the two per-hop count lists.

    Two device->host reads per hop with a non-empty frontier: the hop's emission total (it sizes the outputs) and its
    number of new nodes (it sizes the next frontier).  The workspace (2 x int32 [N]) is allocated once per graph in
    ``csc.aux``; each call resets only the entries of the nodes it sampled, so calls that share a graph must run on
    one stream.
    """
    assert seeds.is_cuda and seeds.dtype == torch.int32 and seeds.dim() == 1
    num_neighbors = [int(k) for k in num_neighbors]
    if len(num_neighbors) > _MAX_HOPS or any(k < -1 or k > _MAX_FANOUT for k in num_neighbors):
        raise ValueError(f"num_neighbors: at most {_MAX_HOPS} hops of -1 ... {_MAX_FANOUT} neighbours each")
    L = lib()
    local, claim = _neighbor_workspace(csc)
    dev, b, n = seeds.device, int(seeds.numel()), csc.n
    colptr, row = csc.rowptr, csc.col
    nodes, pos_parts, dst_parts = [seeds], [], []
    num_nodes, num_edges = [b], []
    try:
        head = torch.empty(b + 1, dtype=torch.int64, device=dev)      # hop 0's offsets, then the seed status
        # an empty tensor has no data pointer, and the entry points reject NULL: calls with nothing to do are skipped
        if b > 0:
            check(L.dggb_neighbor_seed(p(seeds), i32(b), i32(n), p(local), p(head[b:]), stream()), "neighbor_seed")
        if b > 0 and not num_neighbors and int(head[b]):
            raise ValueError("seeds must be unique node ids in [0, N)")
        frontier = seeds
        for hop, k in enumerate(num_neighbors):
            m = int(frontier.numel())
            if m == 0:
                num_nodes.append(0)
                num_edges.append(0)
                continue
            counts = torch.empty(m, dtype=torch.int64, device=dev)
            check(L.dggb_neighbor_count(p(colptr), i32(n), p(frontier), i32(m), i32(k), i32(int(replace)), p(counts),
                                        stream()), "neighbor_count")
            offsets = head if hop == 0 else torch.empty(m, dtype=torch.int64, device=dev)
            torch.cumsum(counts, 0, out=offsets[:m])
            if hop == 0:
                total, bad = offsets[m - 1:].tolist()                  # one read: the total and the seed status
                if bad:
                    raise ValueError("seeds must be unique node ids in [0, N)")
            else:
                total = int(offsets[m - 1])
            if total > _INT32_MAX:
                raise ValueError(f"hop {hop} would sample {total} edges (more than 2^31 - 1): lower num_neighbors")
            num_edges.append(total)
            if total == 0:
                num_nodes.append(0)
                frontier = frontier[:0]
                continue
            out_pos = torch.empty(total, dtype=torch.int32, device=dev)
            out_dst = torch.empty(total, dtype=torch.int32, device=dev)
            check(L.dggb_neighbor_sample(p(colptr), p(row), p(frontier), i32(m), i32(k), i32(int(replace)), i32(hop),
                                         int(seed) & 0xFFFFFFFFFFFFFFFF, i32(sum(num_nodes[:-1])), p(offsets),
                                         p(local), p(claim), p(out_pos), p(out_dst), stream()), "neighbor_sample")
            flags = torch.empty(total, dtype=torch.int32, device=dev)
            check(L.dggb_neighbor_flag(p(row), p(out_pos), i32(total), p(local), p(claim), p(flags), stream()),
                  "neighbor_flag")
            scan = torch.cumsum(flags, 0, dtype=torch.int32)
            new = int(scan[-1])
            new_nodes = torch.empty(new, dtype=torch.int32, device=dev)
            if new > 0:
                check(L.dggb_neighbor_assign(p(row), p(out_pos), i32(total), p(flags), p(scan), i32(sum(num_nodes)),
                                             p(local), p(new_nodes), stream()), "neighbor_assign")
            nodes.append(new_nodes)
            pos_parts.append(out_pos)
            dst_parts.append(out_dst)
            num_nodes.append(new)
            frontier = new_nodes
        n_id = torch.cat(nodes)
        pos = torch.cat(pos_parts) if pos_parts else torch.empty(0, dtype=torch.int32, device=dev)
        dst = torch.cat(dst_parts) if dst_parts else pos
        e = int(pos.numel())
        edge_index = torch.empty(2, e, dtype=torch.int64, device=dev)
        if e > 0:
            check(L.dggb_neighbor_edges(p(row), p(pos), p(dst), i64(e), p(local), p(edge_index), stream()),
                  "neighbor_edges")
        if b > 0:
            check(L.dggb_neighbor_reset(p(n_id), i32(n_id.numel()), i32(n), p(local), p(claim), stream()),
                  "neighbor_reset")
    except BaseException:
        csc.aux.pop("neighbor_ws", None)       # part of a batch is still registered: the next call starts afresh
        raise
    return n_id, edge_index, pos, num_nodes, num_edges


class NeighborLoader:
    """``for batch in loader``: PyG 2.x ``torch_geometric.loader.NeighborLoader`` over one homogeneous graph, sampled
    on the GPU by ``neighbor_sample``.

    Batches of ``batch_size`` input nodes come from a ``torch.utils.data.DataLoader`` over the input indices, so the
    ``shuffle`` order follows the global CPU generator as in PyG; each batch then draws its 62-bit sampling seed from
    the same generator.  Worker arguments (``num_workers``, ``persistent_workers``, ...) are accepted and ignored.
    A batch is a ``SubgraphBatch`` with the node attributes of the parent sliced by ``n_id`` and its edge attributes by
    ``e_id`` (the caller's edge ids), ``edge_index`` (local ids, row 0 the source), ``n_id``, ``e_id``,
    ``batch_size``, ``num_sampled_nodes`` and ``num_sampled_edges``; its first ``batch_size`` nodes are the batch's
    input nodes, in input order.
    """

    def __init__(self, data, num_neighbors, input_nodes=None, replace=False, directed=True, batch_size=1,
                 shuffle=False, drop_last=False, device=None, **kwargs):
        if not directed:
            raise NotImplementedError("NeighborLoader(directed=False) is not provided")
        if kwargs.get("disjoint"):
            raise NotImplementedError("NeighborLoader(disjoint=True) is not provided")
        if kwargs.get("time_attr") is not None:
            raise NotImplementedError("temporal sampling (time_attr) is not provided")
        if (isinstance(num_neighbors, dict) or isinstance(input_nodes, (tuple, str))
                or hasattr(data, "node_types") or hasattr(data, "edge_types")):
            raise NotImplementedError("heterogeneous graphs are not provided")
        assert data.edge_index is not None
        self.num_neighbors = [int(k) for k in num_neighbors]
        self.replace = bool(replace)
        dev = torch.device(device) if device is not None else (
            data.edge_index.device if data.edge_index.is_cuda else torch.device("cuda"))
        self.device = dev
        self.N = int(getattr(data, "num_nodes", None) or data.x.shape[0])
        if input_nodes is None:
            nodes = torch.arange(self.N)
        else:
            nodes = torch.as_tensor(input_nodes).cpu()
            if nodes.dtype == torch.bool:
                if nodes.shape != (self.N,):
                    raise ValueError(f"input_nodes mask has shape {tuple(nodes.shape)}, expected ({self.N},)")
                nodes = nodes.nonzero().view(-1)
            nodes = nodes.long().view(-1)
        if nodes.numel() and (int(nodes.min()) < 0 or int(nodes.max()) >= self.N):
            raise ValueError(f"input_nodes holds ids outside [0, {self.N})")
        if torch.unique(nodes).numel() != nodes.numel():
            raise ValueError("input_nodes holds repeated nodes")
        self.input_nodes = nodes.to(torch.int32)
        ei = data.edge_index.to(dev)
        self.E = int(ei.shape[1])
        # parent adjacency in CSC order (targets, then sources); perm maps a CSC position to the caller's edge id
        self.perm = torch.argsort(ei[1] * self.N + ei[0], stable=True)
        self.csc = CSRGraph.from_indices(ei.flip(0)[:, self.perm].contiguous(), self.N)
        self._node_attrs, self._edge_attrs, self._other = _split_attrs(data, self.N, self.E, dev)
        self._loader = torch.utils.data.DataLoader(range(int(nodes.numel())), batch_size=batch_size, shuffle=shuffle,
                                                   drop_last=drop_last, collate_fn=self._collate)

    def __len__(self):
        return len(self._loader)

    def __iter__(self):
        return iter(self._loader)

    def _collate(self, index):
        seeds = self.input_nodes[torch.as_tensor(index, dtype=torch.long)].to(self.device)
        seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.long))          # global CPU generator
        n_id, edge_index, pos, num_nodes, num_edges = neighbor_sample(self.csc, seeds, self.num_neighbors, seed,
                                                                      self.replace)
        nl = n_id.long()
        e_id = self.perm[pos.long()]
        batch = SubgraphBatch(num_nodes=int(nl.numel()), edge_index=edge_index, n_id=nl, e_id=e_id,
                              batch_size=int(seeds.numel()), num_sampled_nodes=num_nodes,
                              num_sampled_edges=num_edges)
        for k, v in self._node_attrs.items():
            setattr(batch, k, v[nl])
        for k, v in self._edge_attrs.items():
            setattr(batch, k, v[e_id])
        for k, v in self._other.items():
            setattr(batch, k, v)
        return batch


# ------------------------------------------------------------------------------------------------ graph partitioning
# Constants of the multilevel driver (tests/cluster_ref.py restates it with the same values).
_CMAX_DIV = 1             # cluster weight limit while coarsening: N // (_CMAX_DIV * num_parts), at least 1
_STOP_PER_PART = 2        # coarsen while the graph has more than _STOP_PER_PART * num_parts nodes
_MIN_SHRINK = (19, 20)    # ... and a level keeps fewer than 19/20 of its nodes
_MAX_LEVELS = 32
_LP_ROUNDS = 5            # label-propagation rounds per coarsening level (two sub-rounds each)
_REFINE_ROUNDS = 4        # refinement rounds per level (two sub-rounds each)
_REBALANCE_ROUNDS = 2     # rounds per level that move nodes out of over-full parts into adjacent parts


class _Level:
    """One level of the hierarchy: symmetric int32 CSR with int32 entry weights ewt and node weights vw."""

    def __init__(self, n, rowptr, col, ewt, vw):
        self.n, self.rowptr, self.vw = n, rowptr, vw
        self.nnz = int(col.numel())
        # an empty tensor has no data pointer and the entry points reject NULL: a one-entry stand-in (never read,
        # every row is empty)
        self.col = col if self.nnz else torch.zeros(1, dtype=torch.int32, device=rowptr.device)
        self.ewt = ewt if self.nnz else torch.ones(1, dtype=torch.int32, device=rowptr.device)


def _cap(n, k):
    return (103 * n + 100 * k - 1) // (100 * k)


def _symmetrize(edge_index, n, dev):
    """-> _Level 0: both directions of every edge, self loops dropped, duplicates merged, unit weights."""
    ei = edge_index.to(dev, torch.int64)
    u, v = torch.cat([ei[0], ei[1]]), torch.cat([ei[1], ei[0]])
    keep = u != v
    key = torch.unique(u[keep] * n + v[keep])                   # sorted
    g = CSRGraph.from_indices(torch.stack([key // n, key % n]), n)
    ones = torch.ones(n, dtype=torch.int32, device=dev)
    return _Level(n, g.rowptr, g.col, torch.ones(g.nnz, dtype=torch.int32, device=dev), ones)


def _weights(lab, vw, nlabels, with_anchor=True):
    dev = lab.device
    lw = torch.empty(nlabels, dtype=torch.int32, device=dev)
    anchor = torch.empty(nlabels, dtype=torch.int32, device=dev) if with_anchor else None
    check(lib().dggb_partition_weights(p(lab), p(vw), i32(lab.numel()), i32(nlabels), p(lw), p(anchor), stream()),
          "partition_weights")
    return lw, anchor


def _propose(g, lab, lw, anchor, limit, parity, mode):
    key = torch.empty(g.n, dtype=torch.int64, device=lab.device)
    check(lib().dggb_partition_propose(p(g.rowptr), p(g.col), p(g.ewt), p(g.vw), p(lab), i32(g.n), p(lw), p(anchor),
                                       i32(limit), i32(parity), i32(mode), p(key), stream()), "partition_propose")
    return torch.sort(key, stable=True)                          # ties: node id ascending


def _lp_rounds(g, lab, nlabels, limit, rounds, mode):
    for _ in range(rounds):
        for parity in (0, 1):
            lw, anchor = _weights(lab, g.vw, nlabels, with_anchor=mode != 0)
            keys, order = _propose(g, lab, lw, anchor, limit, parity, mode)
            cum = torch.cumsum(g.vw[order], 0, dtype=torch.int64)
            check(lib().dggb_partition_admit(p(keys), p(order), p(cum), i32(g.n), p(lw), i32(limit), p(lab), stream()),
                  "partition_admit")
    return lab


def _project(map_, idx):
    out = torch.empty(idx.numel(), dtype=torch.int32, device=idx.device)
    check(lib().dggb_partition_project(p(map_), p(idx), i32(idx.numel()), p(out), stream()), "partition_project")
    return out


def _contract(g, cluster, nc):
    """-> the coarse _Level: one node per cluster, the entries between clusters merged with summed weights."""
    L, dev = lib(), cluster.device
    rowptr = torch.zeros(nc + 1, dtype=torch.int32, device=dev)
    cvw = _weights(cluster, g.vw, nc, with_anchor=False)[0]
    cnnz = 0
    if g.nnz:
        keys = torch.empty(g.nnz, dtype=torch.int64, device=dev)
        check(L.dggb_partition_contract_keys(p(g.rowptr), p(g.col), i32(g.n), p(cluster), i32(nc), p(keys), stream()),
              "partition_contract_keys")
        keys, idx = torch.sort(keys)
        heads = torch.empty(g.nnz, dtype=torch.int32, device=dev)
        check(L.dggb_partition_contract_heads(p(keys), i64(g.nnz), p(heads), stream()), "partition_contract_heads")
        scan = torch.cumsum(heads, 0, dtype=torch.int32)
        cnnz = int(scan[-1])
    ccol = torch.empty(cnnz, dtype=torch.int32, device=dev)
    cwt = torch.empty(cnnz, dtype=torch.int32, device=dev)
    if cnnz:
        crow = torch.empty(cnnz, dtype=torch.int64, device=dev)
        check(L.dggb_partition_contract_fill(p(keys), p(idx), p(g.ewt), i64(g.nnz), p(scan), i32(nc), i32(cnnz),
                                             p(crow), p(ccol), p(cwt), stream()), "partition_contract_fill")
        check(L.dggb_coo_rows_to_rowptr(p(crow), i64(cnnz), i32(nc), p(rowptr), stream()), "coo_rows_to_rowptr")
    return _Level(nc, rowptr, ccol, cwt, cvw)


def _initial(g, k):
    """BFS order of the coarsest level cut into k chunks of equal weight."""
    L, dev = lib(), g.rowptr.device
    order = torch.empty(g.n, dtype=torch.int32, device=dev)
    pos = torch.empty(g.n, dtype=torch.int32, device=dev)
    claim = torch.empty(g.n, dtype=torch.int32, device=dev)
    check(L.dggb_partition_bfs(p(g.rowptr), p(g.col), i32(g.n), p(order), p(pos), p(claim), stream()), "partition_bfs")
    w = g.vw[order.long()].long()
    prefix = torch.cumsum(w, 0) - w
    total = int(prefix[-1] + w[-1])
    part = torch.empty(g.n, dtype=torch.int32, device=dev)
    check(L.dggb_partition_chunk(p(order), p(prefix), i32(g.n), i64(total), i32(k), p(part), stream()),
          "partition_chunk")
    return part


def _refine(g, part, k, cap):
    part = _lp_rounds(g, part, k, cap, _REBALANCE_ROUNDS, 3)
    return _lp_rounds(g, part, k, cap, _REFINE_ROUNDS, 1)


def _rebalance(g, part, k, cap):
    """Finest level (unit weights): the over-full parts hand their least-loss nodes to the parts with room."""
    lw, anchor = _weights(part, g.vw, k)
    if int(lw.max()) <= cap:
        return part
    keys, order = _propose(g, part, lw, anchor, cap, 0, 2)
    excess = (lw.long() - cap).clamp_(min=0)
    ex_prefix = torch.cumsum(excess, 0) - excess
    room_cum = torch.cumsum((cap - lw.long()).clamp_(min=0), 0)
    check(lib().dggb_partition_rebalance(p(keys), p(order), i32(g.n), p(lw), p(ex_prefix), p(room_cum), i32(k),
                                         i32(cap), p(part), stream()), "partition_rebalance")
    return _refine(g, part, k, cap)


def _partition_parts(edge_index, n, k, dev):
    """-> (part int32 [n] on dev, number of coarse levels).  The phases and their order are the contract of
    ``dggb_partition_*`` in include/dggb.h; tests/cluster_ref.py restates this driver."""
    if k == 1:
        return torch.zeros(n, dtype=torch.int32, device=dev), 0
    cap = _cap(n, k)
    cmax = max(1, n // (_CMAX_DIV * k))
    g = _symmetrize(edge_index, n, dev)
    levels = []
    while g.n > _STOP_PER_PART * k and len(levels) < _MAX_LEVELS:
        lab = _lp_rounds(g, torch.arange(g.n, dtype=torch.int32, device=dev), g.n, cmax, _LP_ROUNDS, 0)
        used = _weights(lab, g.vw, g.n, with_anchor=False)[0] > 0
        cid = torch.cumsum(used, 0, dtype=torch.int32) - 1
        nc = int(cid[-1]) + 1
        if nc * _MIN_SHRINK[1] > g.n * _MIN_SHRINK[0]:
            break
        cluster = _project(cid, lab)
        levels.append((g, cluster))
        g = _contract(g, cluster, nc)
    part = _refine(g, _initial(g, k), k, cap)
    for fine, cluster in reversed(levels):
        g = fine
        part = _refine(g, _project(part, cluster), k, cap)
    return _rebalance(g, part, k, cap), len(levels)


def _edge_input(graph_or_edge_index, num_nodes):
    if isinstance(graph_or_edge_index, CSRGraph):
        g = graph_or_edge_index
        return g.coo_indices(), g.n
    ei = torch.as_tensor(graph_or_edge_index)
    if ei.dim() != 2 or ei.shape[0] != 2:
        raise ValueError(f"edge_index must be [2, E], got {tuple(ei.shape)}")
    ei = ei.long()
    if num_nodes is None:
        num_nodes = int(ei.max()) + 1 if ei.numel() else 0
    if ei.numel() and (int(ei.min()) < 0 or int(ei.max()) >= num_nodes):
        raise ValueError(f"edge_index holds ids outside [0, {num_nodes})")
    return ei, int(num_nodes)


def partition(graph_or_edge_index, num_parts, num_nodes=None, device=None):
    """Deterministic multilevel k-way partition on the GPU -> (perm int64 [N], partptr int64 [num_parts + 1]).

    The graph is taken undirected (both directions of every edge, self loops dropped, duplicate pairs merged, unit
    node and edge weights), as METIS is given it by torch_sparse.  Every part is non-empty and holds at most
    ``ceil(1.03 N / num_parts)`` nodes; ``perm`` lists the nodes by (part, id) -- the stable form of torch_sparse's
    ``cluster.sort()`` -- and part i is ``perm[partptr[i]:partptr[i+1]]``.  ``num_parts == 1`` is the identity.
    The partitions are not METIS's; the same graph and ``num_parts`` give the same result on every run.
    ``graph_or_edge_index``: a CSRGraph or an int [2, E] edge list (``num_nodes`` defaults to its largest id + 1).
    """
    ei, n = _edge_input(graph_or_edge_index, num_nodes)
    k = int(num_parts)
    if n < 1:
        raise ValueError("partition: the graph has no nodes")
    if not 1 <= k <= n:
        raise ValueError(f"num_parts must be in [1, {n}], got {k}")
    dev = torch.device(device) if device is not None else (ei.device if ei.is_cuda else torch.device("cuda"))
    part, _ = _partition_parts(ei, n, k, dev)
    perm = torch.argsort(part, stable=True)
    partptr = torch.zeros(k + 1, dtype=torch.int64, device=dev)
    torch.cumsum(torch.bincount(part, minlength=k), 0, out=partptr[1:])
    return perm, partptr


def _structure_hash(edge_index, n):
    import hashlib

    h = hashlib.sha256(f"{n}:{int(edge_index.shape[1])}:".encode())
    h.update(edge_index.detach().to("cpu", torch.int64).contiguous().numpy().tobytes())
    return h.hexdigest()


class ClusterData:
    """PyG 2.1 ``torch_geometric.loader.ClusterData`` over one homogeneous graph, partitioned on the GPU by
    ``partition`` (not METIS: the parts differ from PyG's, see the module docstring).

    ``perm`` / ``partptr`` (int64, on the device): part i holds the permuted nodes ``partptr[i] ... partptr[i+1]-1``,
    i.e. the original nodes ``perm[partptr[i]:partptr[i+1]]``.  ``data`` holds the node attributes permuted by
    ``perm``, the edge attributes in the order of the permuted CSR (``data._csr``; ``data.e_id`` maps each CSR entry
    to the caller's edge id; duplicate edges stay separate entries, in edge-id order) and ``edge_index`` of the permuted
    graph.  ``recursive`` is accepted and changes nothing: PyG selects METIS's recursive bisection with it, and this
    partitioner has one (direct k-way) scheme.  With ``save_dir`` the partition is cached in
    ``save_dir/dggb_partition_{num_parts}.pt`` together with a hash of the edge structure; a file written for another
    graph is recomputed and overwritten.  ``log`` prints one line when the partition is computed.
    """

    def __init__(self, data, num_parts, recursive=False, save_dir=None, log=True, device=None):
        import os

        assert data.edge_index is not None
        dev = torch.device(device) if device is not None else (
            data.edge_index.device if data.edge_index.is_cuda else torch.device("cuda"))
        self.device, self.num_parts, self.recursive = dev, int(num_parts), bool(recursive)
        n = int(getattr(data, "num_nodes", None) or data.x.shape[0])
        ei = data.edge_index.to(dev).long()
        self.N, self.E = n, int(ei.shape[1])
        perm = partptr = None
        path = os.path.join(save_dir, f"dggb_partition_{self.num_parts}.pt") if save_dir else None
        digest = _structure_hash(ei, n) if path else None
        if path and os.path.isfile(path):
            saved = torch.load(path, map_location="cpu")
            if isinstance(saved, dict) and saved.get("structure") == digest and saved.get("num_parts") == num_parts:
                perm, partptr = saved["perm"].to(dev), saved["partptr"].to(dev)
        if perm is None:
            perm, partptr = partition(ei, self.num_parts, num_nodes=n, device=dev)
            if log:
                print(f"ClusterData: {n} nodes in {self.num_parts} parts (device partitioner)")
            if path:
                os.makedirs(save_dir, exist_ok=True)
                torch.save(dict(structure=digest, num_parts=self.num_parts, perm=perm.cpu(), partptr=partptr.cpu()),
                           path)
        self.perm, self.partptr = perm, partptr
        self._partptr_host = partptr.cpu().tolist()
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(n, device=dev)
        row, col = inv[ei[0]], inv[ei[1]]
        self.e_id = torch.argsort(row * n + col, stable=True)          # permuted CSR position -> caller's edge id
        self.graph = CSRGraph.from_indices(torch.stack([row[self.e_id], col[self.e_id]]), n)
        node_attrs, edge_attrs, other = _split_attrs(data, n, self.E, dev)
        self._node_attrs = {k: v[perm] for k, v in node_attrs.items()}
        self._edge_attrs = edge_attrs                                    # by the caller's edge id
        self._other = other
        self.data = SubgraphBatch(num_nodes=n, edge_index=self.graph.coo_indices(), e_id=self.e_id, **self._node_attrs,
                                  **{k: v[self.e_id] for k, v in edge_attrs.items()}, **other)
        self.data._csr = self.graph

    def __len__(self):
        return self.num_parts

    def __getitem__(self, idx):
        return self._batch([int(idx) % self.num_parts if int(idx) < 0 else int(idx)])

    def _batch(self, parts):
        """SubgraphBatch of the drawn parts, in draw order: PyG 2.1's narrow / index_select collate."""
        if any(not 0 <= q < self.num_parts for q in parts):
            raise IndexError(f"part index out of range [0, {self.num_parts})")
        L, dev, pp = lib(), self.device, self._partptr_host
        start = [pp[q] for q in parts]
        end = [pp[q + 1] for q in parts]
        base, m = [], 0
        for s, e in zip(start, end):
            base.append(m)
            m += e - s
        node_idx = torch.cat([torch.arange(s, e, dtype=torch.int32) for s, e in zip(start, end)]).to(dev)
        meta = torch.tensor([start, end, base], dtype=torch.int32).to(dev)
        nb = len(parts)
        counts = torch.empty(m, dtype=torch.int32, device=dev)
        check(L.dggb_cluster_batch_count(p(self.graph.rowptr), p(self.graph.col), p(meta[0]), p(meta[1]), i32(nb),
                                         p(node_idx), i32(m), p(counts), stream()), "cluster_batch_count")
        sub_rowptr = torch.zeros(m + 1, dtype=torch.int32, device=dev)
        torch.cumsum(counts, 0, out=sub_rowptr[1:])
        nnz = int(sub_rowptr[-1])
        sub_col = torch.empty(nnz, dtype=torch.int32, device=dev)
        sub_eid = torch.empty(nnz, dtype=torch.int32, device=dev)
        if nnz:
            check(L.dggb_cluster_batch_fill(p(self.graph.rowptr), p(self.graph.col), p(meta[0]), p(meta[1]),
                                            p(meta[2]), i32(nb), p(node_idx), i32(m), p(sub_rowptr), p(sub_col),
                                            p(sub_eid), stream()), "cluster_batch_fill")
        sub = CSRGraph(m, sub_rowptr, sub_col)
        nl = node_idx.long()
        e_id = self.e_id[sub_eid.long()]
        batch = SubgraphBatch(num_nodes=m, edge_index=sub.coo_indices())
        for k, v in self._node_attrs.items():
            setattr(batch, k, v[nl])
        for k, v in self._edge_attrs.items():
            setattr(batch, k, v[e_id])
        for k, v in self._other.items():
            setattr(batch, k, v)
        batch._csr = sub           # consumers inside this package skip the edge list -> CSR conversion
        return batch


class ClusterLoader:
    """PyG 2.1 ``torch_geometric.loader.ClusterLoader``: ``for batch in loader`` yields the sub-graph induced by
    ``batch_size`` parts of a ``ClusterData`` at a time.  The parts come from a ``torch.utils.data.DataLoader`` over
    the part indices, so the ``shuffle`` order follows the global CPU generator as in PyG.  A batch's nodes are the
    drawn parts' nodes in draw order; its ``edge_index`` (local ids) is row-major with each row's columns ascending;
    node attributes are sliced by those nodes and edge attributes by the caller's edge ids.  Worker arguments
    (``num_workers``, ...) are accepted and ignored."""

    def __init__(self, cluster_data, batch_size=1, shuffle=False, drop_last=False, **kwargs):
        self.cluster_data = cluster_data
        self._loader = torch.utils.data.DataLoader(range(len(cluster_data)), batch_size=batch_size, shuffle=shuffle,
                                                   drop_last=drop_last, collate_fn=self._collate)

    def __len__(self):
        return len(self._loader)

    def __iter__(self):
        return iter(self._loader)

    def _collate(self, index):
        return self.cluster_data._batch([int(i) for i in index])
