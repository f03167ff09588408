"""Graphs the partitioner tests share: the real Cora / Citeseer adjacencies, a planted-partition SBM, a grid, and a
Pubmed-shape power-law graph; and the edge-cut yardsticks (recursive Kernighan-Lin bisection, random balanced parts)."""
import os

import numpy as np

from tests import cluster_ref as R

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "real_cora_citeseer.npz")
REAL = {"cora": "cora_gcn_dgg", "citeseer": "citeseer_gcnii_dgg64"}


def real(name):
    """-> (edge_index int64 [2, E] with its self loops, N) of the real adjacency."""
    z = np.load(GOLDEN)
    key = REAL[name]
    return z[f"/{key}/adj_idx"].astype(np.int64), int(z[f"/{key}/labels"].shape[0])


def sbm(n=4096, blocks=16, p_in=0.05, p_out=0.0005, seed=0):
    """-> (edge_index, N, planted part per node): ids shuffled so that the blocks are not id ranges."""
    rng = np.random.default_rng(seed)
    blk = np.arange(n) // (n // blocks)
    iu, ju = np.triu_indices(n, 1)
    keep = rng.random(len(iu)) < np.where(blk[iu] == blk[ju], p_in, p_out)
    shuffle = rng.permutation(n)
    planted = np.empty(n, dtype=np.int64)
    planted[shuffle] = blk
    return np.stack([shuffle[iu[keep]], shuffle[ju[keep]]]), n, planted


def sbm_sparse(n, blocks, deg_in, deg_out, seed=0):
    """Planted partition at sizes where the dense construction does not fit: about deg_in / deg_out edges per node."""
    rng = np.random.default_rng(seed)
    size = n // blocks
    m_in, m_out = n * deg_in // 2, n * deg_out // 2
    u = rng.integers(0, n, m_in)
    v = (u // size) * size + rng.integers(0, size, m_in)
    v = np.minimum(v, n - 1)
    a, b = rng.integers(0, n, m_out), rng.integers(0, n, m_out)
    shuffle = rng.permutation(n)
    return np.stack([shuffle[np.concatenate([u, a])], shuffle[np.concatenate([v, b])]]), n


def grid(side=64):
    g = np.arange(side * side).reshape(side, side)
    return np.concatenate([np.stack([g[:, :-1].ravel(), g[:, 1:].ravel()]),
                           np.stack([g[:-1].ravel(), g[1:].ravel()])], 1), side * side


def kl_cut(edge_index, n, k):
    """Edge cut of networkx's recursive kernighan_lin_bisection (seed 0) into k = 2^j parts."""
    import networkx as nx

    rowptr, col = R.symmetrize(edge_index, n)
    G = nx.Graph()
    G.add_nodes_from(range(n))
    G.add_edges_from(zip(np.repeat(np.arange(n), np.diff(rowptr)).tolist(), col.tolist()))
    parts = [set(range(n))]
    while len(parts) < k:
        parts = [s for q in parts for s in nx.algorithms.community.kernighan_lin_bisection(G.subgraph(q), seed=0)]
    part = np.empty(n, dtype=np.int64)
    for i, q in enumerate(parts):
        part[list(q)] = i
    return R.edge_cut(edge_index, n, part)[0]


def random_cut(edge_index, n, k, seed=0):
    part = np.random.default_rng(seed).permutation(np.arange(n) % k)
    return R.edge_cut(edge_index, n, part)[0]
