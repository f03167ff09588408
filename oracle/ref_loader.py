"""TEST INFRASTRUCTURE ONLY -- loader for the *unmodified* reference modules.

Imports ``dgm`` / ``model`` from the reference checkout that ``DGG_REFERENCE_ROOT``
names (read-only; it is not part of this repository) through three shims and no source
edits (SURVEY.md section 8c / Appendix C):

  1. a stub ``torch_geometric`` registered in ``sys.modules`` (model.py:9-11 and
     utils.py:19-24 import it; it is not installed and not installable here);
  2. ``torch.Tensor.cuda`` neutralised so the hard-coded ``.cuda()`` calls
     (dgm.py:1220, 1226, 1390, 1410, 1798, 1951) are no-ops on a CPU box;
  3. Gumbel injection helpers (dgm.py:1149-1151, 1218-1226; legacy dgm.py:14).

Only ``tests/golden/make_golden.py``, the ``-m "not gpu"`` oracle-pinning tests
(skipped when the reference is absent) and ``bench.py --impl reference`` in this
container may use it.  Nothing in the product path imports this file.
"""
from __future__ import annotations

import argparse
import importlib
import os
import sys
import types

import torch

REFERENCE_ROOT = os.environ.get("DGG_REFERENCE_ROOT", "")


def reference_available() -> bool:
    """True when ``DGG_REFERENCE_ROOT`` names a reference checkout; a name that points anywhere else is an error."""
    if not REFERENCE_ROOT:
        return False
    if not os.path.isfile(os.path.join(REFERENCE_ROOT, "dgm.py")):
        raise FileNotFoundError(f"DGG_REFERENCE_ROOT={REFERENCE_ROOT!r} is not a reference checkout (no dgm.py)")
    return True


# --------------------------------------------------------------------------- #
# stub torch_geometric
# --------------------------------------------------------------------------- #
class _DenseGraphConvStub(torch.nn.Module):
    """PyG 2.1.0 ``DenseGraphConv`` semantics (SURVEY.md a20; source not in repo).

    out = lin_rel(aggr(adj @ x)) + lin_root(x); aggr="mean" divides by
    ``adj.sum(-1, keepdim=True).clamp(min=1)``; inputs are promoted to a batch
    dimension so the result is ``[1, N, F_out]``.  lin_rel has a bias, lin_root
    has none.  Restated from the published PyG 2.1.0 documentation -- parity at
    this boundary is unpinned by the reference's own tests.
    """

    def __init__(self, in_channels, out_channels, aggr="add", bias=True):
        super().__init__()
        assert aggr in ("add", "mean", "max")
        self.aggr = aggr
        self.lin_rel = torch.nn.Linear(in_channels, out_channels, bias=bias)
        self.lin_root = torch.nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, adj, mask=None):
        x = x.unsqueeze(0) if x.dim() == 2 else x
        adj = adj.unsqueeze(0) if adj.dim() == 2 else adj
        out = torch.matmul(adj, x)
        if self.aggr == "mean":
            out = out / adj.sum(dim=-1, keepdim=True).clamp_(min=1)
        out = self.lin_rel(out) + self.lin_root(x)
        return out


def _remove_self_loops(edge_index, edge_attr=None):
    keep = edge_index[0] != edge_index[1]
    return edge_index[:, keep], (None if edge_attr is None else edge_attr[keep])


def _add_self_loops(edge_index, edge_attr=None, fill_value=None, num_nodes=None):
    n = int(edge_index.max()) + 1 if num_nodes is None else num_nodes
    loops = torch.arange(n, dtype=edge_index.dtype, device=edge_index.device)
    return torch.cat([edge_index, torch.stack([loops, loops])], dim=1), edge_attr


def _placeholder(name):
    def _raise(*a, **k):
        raise RuntimeError(f"torch_geometric stub: {name} is a placeholder")

    return _raise


def install_pyg_stub() -> None:
    if "torch_geometric" in sys.modules and not getattr(
        sys.modules["torch_geometric"], "__dgg_stub__", False
    ):
        return  # a real PyG is present: prefer it
    root = types.ModuleType("torch_geometric")
    root.__dgg_stub__ = True
    subs = {}
    for sub in ("nn", "utils", "datasets", "loader", "data", "transforms"):
        m = types.ModuleType(f"torch_geometric.{sub}")
        setattr(root, sub, m)
        subs[sub] = m
        sys.modules[f"torch_geometric.{sub}"] = m
    subs["nn"].DenseGraphConv = _DenseGraphConvStub
    subs["nn"].SAGEConv = _placeholder("SAGEConv")
    subs["nn"].GraphConv = _placeholder("GraphConv")
    subs["utils"].remove_self_loops = _remove_self_loops
    subs["utils"].add_self_loops = _add_self_loops
    subs["utils"].degree = _placeholder("degree")
    subs["utils"].to_networkx = _placeholder("to_networkx")
    subs["utils"].to_scipy_sparse_matrix = _placeholder("to_scipy_sparse_matrix")
    subs["datasets"].KarateClub = _placeholder("KarateClub")
    subs["datasets"].AttributedGraphDataset = _placeholder("AttributedGraphDataset")
    subs["data"].Data = _placeholder("Data")
    sys.modules["torch_geometric"] = root


_ORIG_CUDA = torch.Tensor.cuda


def neutralise_cuda() -> None:
    torch.Tensor.cuda = lambda self, *a, **k: self


def restore_cuda() -> None:
    torch.Tensor.cuda = _ORIG_CUDA


def load_reference(names=("dgm", "model")):
    """Return the reference modules under private names (``_ref_dgm`` ...) so the
    repo's own drop-in ``dgm`` / ``model`` stay importable next to them."""
    if not reference_available():
        raise FileNotFoundError("no reference checkout: set DGG_REFERENCE_ROOT")
    install_pyg_stub()
    neutralise_cuda()
    out = {}
    saved = {n: sys.modules.pop(n, None) for n in ("dgm", "model", "utils")}
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for n in ("dgm", "utils", "model"):
                if n in names or (n == "utils" and "model" in names):
                    out[n] = importlib.import_module(n)
            if "utils" in out and not hasattr(out["utils"].np, "float"):
                out["utils"].np.float = float      # numpy >= 1.24 removed np.float (utils.py:99)
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for n in ("dgm", "model", "utils"):
            mod = sys.modules.pop(n, None)
            if mod is not None:
                sys.modules[f"_ref_{n}"] = mod
            if saved[n] is not None:
                sys.modules[n] = saved[n]
    return out


# --------------------------------------------------------------------------- #
# args + noise injection
# --------------------------------------------------------------------------- #
def default_args(**over) -> argparse.Namespace:
    """The DGG-relevant attribute surface (SURVEY.md Appendix B) with the
    train_small_graphs.py defaults (train_small_graphs.py:78-207)."""
    d = dict(
        extra_edge_dim=0, extra_k_dim=1, dgg_hard=False, deg_mean=3.899,
        deg_std=5.288, dgg_mode_edge_net="u-v-dist", dgg_mode_k_net="x",
        dgg_mode_k_select="k_times_edge_prob", debug_step=3,
        perturb_edge_prob=False, symmetric_noise=True, stochastic_k=False,
        dgg_adj_input="input_adj", n_dgg_layers=2, dgm_dim=128, dgm_temp=10,
        pre_normalize_adj=False,
    )
    d.update(over)
    return argparse.Namespace(**d)


EXTRA_EDGE_DIM = {"u-v-dist": 0, "edge_conv": 0, "A_uv": 0, "u-v-A_uv": 1,
                  "u-v-deg": 2, "u-v-deg-dist": 3}


class FixedGumbel:
    """Replacement for ``module.gumbel`` whose ``sample(shape)`` returns a fixed
    tensor (call sites dgm.py:1220 ``sample([n_triu])`` and 1226
    ``sample([1,N,N])``)."""

    def __init__(self, tensor):
        self.tensor = tensor

    def sample(self, shape):
        shape = tuple(int(s) for s in shape)
        assert tuple(self.tensor.shape) == shape, (self.tensor.shape, shape)
        return self.tensor.clone()
