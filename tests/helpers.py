import json

import numpy as np
import torch


def save_golden_npz(path, tree):
    """Nested dicts of tensors (dense or sparse COO), numbers, strings and None -> one compressed .npz that loads
    without pickle.  Integer tensors are stored in the narrowest dtype that holds their values (the file stays small);
    ``load_golden_npz`` restores every tensor with its original dtype, bit for bit."""
    arrays = {}

    def enc(key, v):
        if isinstance(v, torch.Tensor):
            if v.is_sparse:
                v = v.coalesce()
                return {"sparse": list(v.shape), "indices": enc(key + ".indices", v.indices()),
                        "values": enc(key + ".values", v.values())}
            a = v.detach().cpu().numpy()
            if a.dtype.kind in "iu" and a.size:
                a = a.astype(np.result_type(np.min_scalar_type(a.min()), np.min_scalar_type(a.max())))
            arrays[key] = a
            return {"tensor": key, "dtype": str(v.dtype).split(".")[1]}
        if isinstance(v, dict):
            return {"dict": {k: enc(f"{key}/{k}", x) for k, x in v.items()}}
        return {"value": v}

    meta = enc("", tree)
    np.savez_compressed(path, __meta__=np.array(json.dumps(meta)), **arrays)


def load_golden_npz(path):
    with np.load(path, allow_pickle=False) as f:
        def dec(m):
            if "sparse" in m:
                return torch.sparse_coo_tensor(dec(m["indices"]), dec(m["values"]), m["sparse"]).coalesce()
            if "tensor" in m:
                return torch.from_numpy(f[m["tensor"]]).to(getattr(torch, m["dtype"]))
            if "dict" in m:
                return {k: dec(x) for k, x in m["dict"].items()}
            return m["value"]

        return dec(json.loads(str(f["__meta__"])))


def random_graph(n, avg_deg, seed, self_loops=True, hubs=0, hub_deg=0, device="cpu"):
    """Symmetric random graph (+ optional high-degree hub rows) as coalesced COO indices/values."""
    g = torch.Generator().manual_seed(seed)
    m = n * avg_deg // 2
    src = torch.randint(0, n, (m,), generator=g)
    dst = torch.randint(0, n, (m,), generator=g)
    if hubs:
        hs = torch.randint(0, n, (hubs,), generator=g).repeat_interleave(hub_deg)
        hd = torch.randint(0, n, (hubs * hub_deg,), generator=g)
        src, dst = torch.cat([src, hs]), torch.cat([dst, hd])
    keep = src != dst
    src, dst = src[keep], dst[keep]
    i, j = torch.cat([src, dst]), torch.cat([dst, src])
    if self_loops:
        loops = torch.arange(n)
        i, j = torch.cat([i, loops]), torch.cat([j, loops])
    a = torch.sparse_coo_tensor(torch.stack([i, j]), torch.ones(i.numel()), (n, n)).coalesce()
    idx = a.indices().clone()
    val = torch.ones(idx.shape[1])
    return idx.to(device), val.to(device)


def coo(idx, val, n):
    return torch.sparse_coo_tensor(idx, val, (n, n)).coalesce()


def tie_free_rows(dense_scores, idx, rel_gap=1e-5):
    """Rows whose on-edge scores are pairwise separated by > rel_gap (rank parity is asserted there)."""
    n = dense_scores.shape[0]
    ok = torch.ones(n, dtype=torch.bool)
    srt = torch.sort(dense_scores, dim=-1, descending=True).values
    gap = (srt[:, :-1] - srt[:, 1:]).abs()
    both_pos = (srt[:, :-1] > 0) & (srt[:, 1:] > 0)
    bad = (both_pos & (gap <= rel_gap * srt[:, :-1].abs())).any(-1)
    return ~bad


def in_row_order(idx, score):
    """Permutation that lists the entries row by row, each row by score descending (ties: lower column first) --
    the order a stable descending sort of the dense row leaves the support in (zeros sort last)."""
    col_order = torch.argsort(idx[1], stable=True)
    by_score = torch.argsort(score[col_order].double(), descending=True, stable=True)
    perm = col_order[by_score]
    return perm[torch.argsort(idx[0][perm], stable=True)]


def sparse_ranks(idx, score, n):
    """0-based descending rank of every stored entry inside its row (== its position in the dense stable sort)."""
    perm = in_row_order(idx, score)
    rows = idx[0][perm]
    counts = torch.bincount(idx[0], minlength=n)
    start = torch.cumsum(counts, 0) - counts
    rank = torch.empty(idx.shape[1], dtype=torch.long)
    rank[perm] = torch.arange(idx.shape[1]) - start[rows]
    return rank


def tie_free_rows_sparse(idx, score, n, rel_gap=1e-5):
    """Rows whose stored scores are pairwise separated by > rel_gap (relative): ranks computed in a different fp32
    summation order are guaranteed identical there.  O(E log E), no dense N x N (Pubmed / Reddit shapes)."""
    perm = in_row_order(idx, score)
    rows, s = idx[0][perm], score[perm]
    same = rows[1:] == rows[:-1]
    close = (s[:-1] - s[1:]).abs() <= rel_gap * s[:-1].abs()
    ok = torch.ones(n, dtype=torch.bool)
    ok[rows[1:][same & close]] = False
    return ok


def assert_grad_close(got, want, rtol=2e-3, atol_rel=2e-5, what=""):
    """Gradient comparison with the absolute tolerance tied to the tensor's own scale (sums of ~1e5 atomically
    accumulated terms: the error floor is relative to the largest entry, not to each entry)."""
    atol = atol_rel * float(want.abs().max()) + 1e-12
    torch.testing.assert_close(got, want, rtol=rtol, atol=atol, msg=lambda m: f"{what}: {m}")


def near_tie_entries(idx, score, n, rel_gap=1e-5):
    """Stored entries whose score is within rel_gap (relative) of the next / previous one in their row's sorted
    order.  Only THOSE entries can swap ranks under a different fp32 summation order (adjacent swap: every other
    entry of the row keeps its rank), so leaving them out of the loss makes values and gradients comparable for
    everything else -- including the rest of a 1500-entry hub row that almost surely contains some near-tie."""
    perm = in_row_order(idx, score)
    rows, s = idx[0][perm], score[perm]
    same = rows[1:] == rows[:-1]
    close = same & ((s[:-1] - s[1:]).abs() <= rel_gap * s[:-1].abs())
    bad_sorted = torch.zeros(idx.shape[1], dtype=torch.bool)
    bad_sorted[:-1] |= close
    bad_sorted[1:] |= close
    bad = torch.zeros(idx.shape[1], dtype=torch.bool)
    bad[perm] = bad_sorted
    return bad
