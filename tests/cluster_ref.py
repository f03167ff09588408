"""NumPy restatement of the multilevel k-way partitioner in include/dggb.h (dggb_partition_*) and of the driver in
dgg_b200.samplers.partition: the same phases in the same order, with the same integer arithmetic and tie-breaking,
vectorised per round.  The GPU result is pinned bit for bit against it (tests/test_gpu_cluster.py)."""
import numpy as np

NONE = np.iinfo(np.int64).max          # key of a node that proposes nothing
BIG = 0x7F7F7F7F                       # anchor of a label nobody holds (cudaMemset 0x7f)

# the driver's constants (dgg_b200.samplers)
CMAX_DIV = 1             # cluster weight limit while coarsening: N // (CMAX_DIV * num_parts), at least 1
STOP_PER_PART = 2        # coarsen while the graph has more than STOP_PER_PART * num_parts nodes
MIN_SHRINK = (19, 20)    # ... and a level keeps fewer than 19/20 of its nodes
MAX_LEVELS = 32
LP_ROUNDS = 5            # label-propagation rounds per coarsening level (two sub-rounds each)
REFINE_ROUNDS = 4        # refinement rounds per level (two sub-rounds each)
REBALANCE_ROUNDS = 2     # rounds per level that move nodes out of over-full parts into adjacent parts


def fmix32(x):
    """MurmurHash3's 32-bit finaliser (a bijection of uint32)."""
    x = np.asarray(x, dtype=np.int64).astype(np.uint32)
    x = x ^ (x >> np.uint32(16))
    x = x * np.uint32(0x85EBCA6B)
    x = x ^ (x >> np.uint32(13))
    x = x * np.uint32(0xC2B2AE35)
    x = x ^ (x >> np.uint32(16))
    return x.astype(np.int64)


def cap_of(n, k):
    return (103 * n + 100 * k - 1) // (100 * k)


def symmetrize(edge_index, n):
    """-> (rowptr, col) int64: both directions of every edge, self loops dropped, duplicates merged, rows sorted."""
    ei = np.asarray(edge_index, dtype=np.int64).reshape(2, -1)
    u, v = np.concatenate([ei[0], ei[1]]), np.concatenate([ei[1], ei[0]])
    keep = u != v
    key = np.unique(u[keep] * n + v[keep])
    row, col = key // n, key % n
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(row, minlength=n))]).astype(np.int64)
    return rowptr, col


# ------------------------------------------------------------------------------------------------------ phases
def weights(lab, vw, nlabels):
    """-> (lw [nlabels] = summed node weight per label, anchor [nlabels] = smallest node holding it, else BIG)."""
    lw = np.bincount(lab, weights=vw, minlength=nlabels).astype(np.int64)
    anchor = np.full(nlabels, BIG, dtype=np.int64)
    np.minimum.at(anchor, lab, np.arange(len(lab), dtype=np.int64))
    return lw, anchor


def propose(rowptr, col, ewt, vw, lab, lw, anchor, limit, parity, mode):
    """-> key [n] int64.  Every active node finds the adjacent label L != own with lw[L] + vw[v] <= limit and the
    largest (conn(L), fmix32(L)), conn = summed weight of the node's entries into L, and gain = conn(L) - conn(own).
      mode 0 (cluster):   active when fmix32(v) & 1 == parity; proposes L when gain > 0.
      mode 1 (refine):    as mode 0, and v is not the anchor of its part (no part is left empty).
      mode 3 (unload):    as mode 1, and lw[own] > limit; proposes L whatever the gain.
    A proposal is key = L << 32 | (2^31 - 1 - gain) (low word unsigned), else NONE.
      mode 2 (evict):     every non-anchor node with lw[own] > limit: key = own << 32 | (2^31 - 1 - gain), gain taken
                          with conn(L) = 0 when there is no L."""
    n = len(rowptr) - 1
    nl = len(lw)
    v = np.arange(n, dtype=np.int64)
    src = np.repeat(v, np.diff(rowptr))
    L = lab[col]
    own = lab
    if mode == 2:
        active = (lw[own] > limit) & (anchor[own] != v)
    else:
        active = (fmix32(v) & 1) == parity
        if mode != 0:
            active &= anchor[own] != v
        if mode == 3:
            active &= lw[own] > limit
    same = L == own[src]
    own_conn = np.bincount(src[same], weights=ewt[same], minlength=n).astype(np.int64)
    cand = ~same & (lw[L] + vw[src] <= limit) & active[src]
    key_sl = src[cand] * nl + L[cand]
    uniq, inv = np.unique(key_sl, return_inverse=True)
    conn = np.bincount(inv, weights=ewt[cand], minlength=len(uniq)).astype(np.int64)
    us, ul = uniq // nl, uniq % nl
    o = np.lexsort((-fmix32(ul), -conn, us))
    us, ul, conn = us[o], ul[o], conn[o]
    first = np.ones(len(us), dtype=bool)
    first[1:] = us[1:] != us[:-1]
    best_conn = np.zeros(n, dtype=np.int64)
    best_l = np.full(n, -1, dtype=np.int64)
    best_conn[us[first]] = conn[first]
    best_l[us[first]] = ul[first]
    key = np.full(n, NONE, dtype=np.int64)
    gain = best_conn - own_conn
    if mode == 2:
        key[active] = (own[active] << 32) | (0x7FFFFFFF - gain[active])
    else:
        m = active & (best_l >= 0) & ((gain > 0) | (mode == 3))
        key[m] = (best_l[m] << 32) | (0x7FFFFFFF - gain[m])
    return key


def sort_keys(key):
    order = np.argsort(key, kind="stable")
    return key[order], order


def segment_sums(ks, order, vw):
    """inclusive prefix of vw over each run of equal key >> 32 in the sorted keys."""
    cum = np.cumsum(vw[order])
    t = ks >> 32
    s = np.searchsorted(ks, t << 32, side="left")
    return t, s, cum - np.where(s > 0, cum[np.maximum(s - 1, 0)], 0)


def admit(ks, order, vw, lw, limit, lab):
    """Proposals per target in key order (gain descending, then node id) while lw[target] + admitted <= limit."""
    t, _, seg = segment_sums(ks, order, vw)
    valid = ks != NONE
    ok = valid & (lw[np.where(valid, t, 0)] + seg <= limit)
    lab = lab.copy()
    lab[order[ok]] = t[ok]
    return lab


def rebalance(ks, order, lw, cap, part):
    """Unit node weights.  The first max(0, lw[p] - cap) proposals of each over-full part p (least cut lost first)
    take the free places of the parts below cap, in part order."""
    k = len(lw)
    excess = np.maximum(lw - cap, 0)
    ex_prefix = np.concatenate([[0], np.cumsum(excess)[:-1]])
    room_cum = np.cumsum(np.maximum(cap - lw, 0))
    valid = ks != NONE
    p = np.where(valid, ks >> 32, 0)
    s = np.searchsorted(ks, p << 32, side="left")
    r = np.arange(len(ks)) - s
    go = valid & (r < excess[p])
    j = ex_prefix[p[go]] + r[go]
    part = part.copy()
    part[order[go]] = np.searchsorted(room_cum, j, side="right")
    assert k > 0
    return part


def contract(rowptr, col, ewt, vw, cluster, nc):
    """-> coarse (rowptr, col, ewt, vw): every pair of clusters joined by an entry, weights summed, rows sorted."""
    n = len(rowptr) - 1
    src = np.repeat(np.arange(n, dtype=np.int64), np.diff(rowptr))
    cu, cw = cluster[src], cluster[col]
    keep = cu != cw
    uniq, inv = np.unique(cu[keep] * nc + cw[keep], return_inverse=True)
    cwt = np.bincount(inv, weights=ewt[keep], minlength=len(uniq)).astype(np.int64)
    crow, ccol = uniq // nc, uniq % nc
    crowptr = np.concatenate([[0], np.cumsum(np.bincount(crow, minlength=nc))]).astype(np.int64)
    cvw = np.bincount(cluster, weights=vw, minlength=nc).astype(np.int64)
    return crowptr, ccol, cwt, cvw


def bfs_order(rowptr, col):
    """Level-synchronous BFS: a frontier node's new neighbours follow it ordered by (parent position, id); a new
    search starts from the smallest unvisited id."""
    n = len(rowptr) - 1
    pos = np.full(n, -1, dtype=np.int64)
    order = np.empty(n, dtype=np.int64)
    tail = cursor = 0
    while tail < n:
        while pos[cursor] >= 0:
            cursor += 1
        order[tail], pos[cursor] = cursor, tail
        head, tail = tail, tail + 1
        while head < tail:
            f = order[head:tail]
            deg = rowptr[f + 1] - rowptr[f]
            par = np.repeat(np.arange(head, tail), deg)
            idx = np.repeat(rowptr[f] - np.cumsum(np.concatenate([[0], deg[:-1]])), deg) + np.arange(deg.sum())
            u = col[idx]
            new = pos[u] < 0
            par, u = par[new], u[new]
            claim = np.full(n, np.iinfo(np.int64).max)
            np.minimum.at(claim, u, par)
            win = claim[u] == par
            par, u = par[win], u[win]
            o = np.lexsort((u, par))
            u = u[o]
            head = tail
            order[tail:tail + len(u)] = u
            pos[u] = np.arange(tail, tail + len(u))
            tail += len(u)
    return order


def chunk(order, vw, k):
    """part of order position i = min(k - 1, P_i * k // W), P_i the weight before it."""
    w = vw[order]
    prefix = np.cumsum(w) - w
    part = np.empty(len(order), dtype=np.int64)
    part[order] = np.minimum(k - 1, prefix * k // int(w.sum()))
    return part


# ------------------------------------------------------------------------------------------------------ driver
def lp_rounds(g, lab, nlabels, limit, rounds, mode):
    rowptr, col, ewt, vw = g
    for r in range(rounds):
        for parity in (0, 1):
            lw, anchor = weights(lab, vw, nlabels)
            ks, order = sort_keys(propose(rowptr, col, ewt, vw, lab, lw, anchor, limit, parity, mode))
            lab = admit(ks, order, vw, lw, limit, lab)
    return lab


def refine(g, part, k, cap):
    part = lp_rounds(g, part, k, cap, REBALANCE_ROUNDS, 3)
    return lp_rounds(g, part, k, cap, REFINE_ROUNDS, 1)


def partition_levels(edge_index, n, k):
    """-> (part [n], number of coarse levels)."""
    if not 1 <= k <= n:
        raise ValueError(f"num_parts must be in [1, {n}]")
    if k == 1:
        return np.zeros(n, dtype=np.int64), 0
    cap = cap_of(n, k)
    cmax = max(1, n // (CMAX_DIV * k))
    rowptr, col = symmetrize(edge_index, n)
    g = (rowptr, col, np.ones(len(col), dtype=np.int64), np.ones(n, dtype=np.int64))
    levels = []
    while len(g[0]) - 1 > STOP_PER_PART * k and len(levels) < MAX_LEVELS:
        nl = len(g[0]) - 1
        lab = lp_rounds(g, np.arange(nl, dtype=np.int64), nl, cmax, LP_ROUNDS, 0)
        used = weights(lab, g[3], nl)[0] > 0
        cid = np.cumsum(used) - 1
        nc = int(used.sum())
        if nc * MIN_SHRINK[1] > nl * MIN_SHRINK[0]:
            break
        levels.append((g, cid[lab]))
        g = contract(*g, cid[lab], nc)
    part = refine(g, chunk(bfs_order(g[0], g[1]), g[3], k), k, cap)
    for fine, cluster in reversed(levels):
        g = fine
        part = refine(g, part[cluster], k, cap)
    lw, anchor = weights(part, g[3], k)
    if lw.max() > cap:
        ks, order = sort_keys(propose(*g, part, lw, anchor, cap, 0, 2))
        part = rebalance(ks, order, lw, cap, part)
        part = lp_rounds(g, part, k, cap, REFINE_ROUNDS, 1)
    return part, len(levels)


def partition(edge_index, n, k):
    """-> (perm [n], partptr [k + 1]) int64: nodes ordered by (part, id)."""
    part, _ = partition_levels(edge_index, n, k)
    perm = np.argsort(part, kind="stable")
    partptr = np.concatenate([[0], np.cumsum(np.bincount(part, minlength=k))])
    return perm.astype(np.int64), partptr.astype(np.int64)


def edge_cut(edge_index, n, part):
    """undirected pairs (loops dropped, duplicates merged) whose ends are in different parts, and their number."""
    rowptr, col = symmetrize(edge_index, n)
    row = np.repeat(np.arange(n), np.diff(rowptr))
    up = row < col
    return int((part[row[up]] != part[col[up]]).sum()), int(up.sum())
