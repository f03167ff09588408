"""Host restatement of the k-hop neighbour sampling contract in include/dggb.h (dggb_neighbor_*), as the sequential
loop torch_sparse's neighbor_sample runs, driven by the same Philox stream as the kernels (tests/philox_ref.py)."""
import numpy as np
import torch

from tests.philox_ref import philox4x32_7


def draws(m, hop, k, seed):
    """x[t, i] for slots t < m and draws i < k: lane (i & 3) of philox(counter = (t, (hop << 24) | (i >> 2)), seed)."""
    nb = (k + 3) // 4
    c0 = torch.arange(m, dtype=torch.int64).repeat_interleave(nb)
    c1 = (hop << 24) | torch.arange(nb, dtype=torch.int64).repeat(m)
    outs = philox4x32_7(c0, c1, seed)
    return torch.stack(outs, 1).reshape(m, nb * 4)[:, :k].numpy()


def neighbor_sample_ref(colptr, row, seeds, num_neighbors, seed, replace=False):
    """colptr / row: int numpy CSC (entries of target v = its in-neighbours, sorted by source).
    -> (n_id, edge_index [2, E] (local source, local target), CSC positions, num_sampled_nodes, num_sampled_edges)."""
    colptr = [int(c) for c in colptr]
    row = [int(r) for r in row]
    n_id = [int(s) for s in seeds]
    local = {s: i for i, s in enumerate(n_id)}
    assert len(local) == len(n_id), "seeds must be unique"
    frontier, base = list(n_id), 0
    src, dst, pos = [], [], []
    num_nodes, num_edges = [len(n_id)], []
    for hop, k in enumerate(num_neighbors):
        x = draws(len(frontier), hop, k, seed) if k > 0 and frontier else None
        new, e0 = [], len(pos)
        for t, v in enumerate(frontier):
            beg, d = colptr[v], colptr[v + 1] - colptr[v]
            if d == 0 or k == 0:
                continue
            if k < 0 or (not replace and k >= d):
                picks = range(d)
            elif replace:
                picks = [(int(x[t, i]) * d) >> 32 for i in range(k)]
            else:                                    # Floyd
                chosen = set()
                for i in range(k):
                    j = d - k + i
                    r = (int(x[t, i]) * (j + 1)) >> 32
                    chosen.add(j if r in chosen else r)
                picks = sorted(chosen)
            for q in picks:
                p = beg + q
                u = row[p]
                if u not in local:
                    local[u] = len(n_id)
                    n_id.append(u)
                    new.append(u)
                src.append(local[u])
                dst.append(base + t)
                pos.append(p)
        num_edges.append(len(pos) - e0)
        num_nodes.append(len(new))
        base = len(n_id) - len(new)
        frontier = new
    edge_index = np.array([src, dst], dtype=np.int64).reshape(2, -1)
    return (np.array(n_id, dtype=np.int64), edge_index, np.array(pos, dtype=np.int64), num_nodes, num_edges)
