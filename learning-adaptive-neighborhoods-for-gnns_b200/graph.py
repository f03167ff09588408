"""Device-resident int32 CSR view of a (coalesced) torch sparse COO adjacency.

The reference keeps adjacencies as torch COO tensors and densifies them at every use
(model.py:1274, 567; dgm.py:1788).  Here the COO tensor stays the public currency (callers do
``.to_dense()`` / ``.coalesce().indices()`` on what DGG returns) but carries a CSR handle so no
consumer inside this package ever densifies or re-sorts it.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, i32, i64, lib, p, stream


class CSRGraph:
    """rowptr int32 [n+1], col int32 [nnz]; rows sorted by column (coalesced COO order)."""

    __slots__ = ("n", "nnz", "rowptr", "col", "indices", "_loops", "_erow", "_max_row_nnz", "aux")

    def __init__(self, n, rowptr, col, indices=None):
        self.n = int(n)
        self.nnz = int(col.numel())
        self.rowptr = rowptr
        self.col = col
        self.indices = indices  # int64 [2, nnz] (built lazily for COO export)
        self._loops = None
        self._erow = None
        self._max_row_nnz = None
        self.aux = {}   # per-structure caches of the consumers (e.g. GAT edge-list plans), alive as long as the graph

    @property
    def erow(self) -> torch.Tensor:
        """int32 [nnz] row index of every entry (built once per structure)."""
        if self._erow is None:
            self._erow = torch.empty(self.nnz, dtype=torch.int32, device=self.col.device)
            if self.nnz > 0:   # no entries: nothing to write (and an empty tensor has no data pointer to pass)
                check(lib().dggb_csr_expand_rows(p(self.rowptr), i32(self.n), p(self._erow), stream()),
                      "csr_expand_rows")
        return self._erow

    @property
    def max_row_nnz(self) -> int:
        """Longest row (one device->host read per structure; -1 while a CUDA graph is being captured and the
        value is not cached yet, which selects the two-launch kernels)."""
        if self._max_row_nnz is None:
            if self.nnz == 0:
                self._max_row_nnz = 0
            elif self.rowptr.is_cuda and torch.cuda.is_current_stream_capturing():
                return -1
            else:
                self._max_row_nnz = int((self.rowptr[1:] - self.rowptr[:-1]).max().item())
        return self._max_row_nnz

    # ------------------------------------------------------------------ construction
    @staticmethod
    def from_indices(indices: torch.Tensor, n: int) -> "CSRGraph":
        """indices: int64 [2, nnz] of a COALESCED COO (row-major sorted)."""
        assert indices.is_cuda and indices.dtype == torch.int64 and indices.dim() == 2
        indices = indices.contiguous()
        nnz = indices.shape[1]
        rowptr = torch.empty(n + 1, dtype=torch.int32, device=indices.device)
        col = torch.empty(nnz, dtype=torch.int32, device=indices.device)
        L = lib()
        check(L.dggb_coo_rows_to_rowptr(p(indices[0]), i64(nnz), i32(n), p(rowptr), stream()), "coo_rows_to_rowptr")
        check(L.dggb_cast_i64_i32(p(indices[1]), p(col), i64(nnz), stream()), "cast_i64_i32")
        return CSRGraph(n, rowptr, col, indices)

    @staticmethod
    def from_coo(adj: torch.Tensor):
        """-> (CSRGraph, values).  Reuses the handle attached by a previous call / by DGG."""
        h = getattr(adj, "_dgg_csr", None)
        if h is not None:
            v = getattr(adj, "_dgg_vals", None)
            if v is None:
                v = adj.values() if adj.is_coalesced() else adj._values()   # values(): keeps the autograd history
            return h, (v if v.dtype == torch.float32 else v.to(torch.float32))
        assert adj.is_sparse and adj.dim() == 2 and adj.shape[0] == adj.shape[1]
        if not adj.is_coalesced():
            adj = adj.coalesce()
        g = CSRGraph.from_indices(adj._indices(), adj.shape[0])
        vals = adj.values().to(torch.float32)            # differentiable view of a coalesced tensor's values
        try:
            adj._dgg_csr = g
        except Exception:
            pass
        return g, vals

    # ------------------------------------------------------------------ A + I
    def with_self_loops(self, vals: torch.Tensor):
        """(A + I) as (CSRGraph, values): existing diagonal entries get +1, missing ones are
        inserted -- the sparse equivalent of (A.to_dense() + eye).to_sparse().coalesce()
        (model.py:1381-1392).  The structure is cached; only values are recomputed."""
        L = lib()
        dev = vals.device
        if self._loops is None:
            out_rowptr = torch.empty(self.n + 1, dtype=torch.int32, device=dev)
            check(L.dggb_add_self_loops_count(p(self.rowptr), p(self.col), i32(self.n), p(out_rowptr), stream()),
                  "add_self_loops_count")
            nnz_out = int(out_rowptr[-1].item())  # one host sync per graph structure
            out_col = torch.empty(nnz_out, dtype=torch.int32, device=dev)
            self._loops = CSRGraph(self.n, out_rowptr, out_col)
        g = self._loops
        if not vals.is_cuda:
            raise RuntimeError("dgg_b200 ops need CUDA tensors (no CPU fallback)")
        vals = vals.contiguous() if vals.dtype == torch.float32 else vals.to(torch.float32).contiguous()
        out_val = torch.empty(g.nnz, dtype=torch.float32, device=dev)
        check(L.dggb_add_self_loops_fill(p(self.rowptr), p(self.col), p(vals), i32(self.n),
                                         p(g.rowptr), p(g.col), p(out_val), stream()), "add_self_loops_fill")
        return g, out_val

    def diag_mask(self) -> torch.Tensor:
        """bool [nnz]: entries on the diagonal."""
        return self.erow == self.col

    # ------------------------------------------------------------------ export
    def coo_indices(self) -> torch.Tensor:
        if self.indices is None:
            counts = (self.rowptr[1:] - self.rowptr[:-1]).to(torch.int64)
            rows = torch.repeat_interleave(torch.arange(self.n, device=self.col.device), counts,
                                           output_size=self.nnz)
            self.indices = torch.stack([rows, self.col.to(torch.int64)])
        return self.indices

    def to_coo(self, vals: torch.Tensor) -> torch.Tensor:
        """A real coalesced torch.sparse_coo_tensor (what the reference returns, dgm.py:1815) carrying
        the CSR handle and the autograd-tracked values."""
        out = torch.sparse_coo_tensor(self.coo_indices(), vals, (self.n, self.n), is_coalesced=True)
        out._dgg_csr = self
        out._dgg_vals = vals
        return out
