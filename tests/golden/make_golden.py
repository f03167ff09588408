"""Generate the known-answer fixtures under tests/golden/ by running the
UNMODIFIED reference modules (the checkout ``DGG_REFERENCE_ROOT`` names) through oracle/ref_loader.py:

    DGG_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py

The reference has no tests or golden vectors of its own (SURVEY.md section 4);
these fixtures are what pins oracle/dgg_oracle.py and, through it, the CUDA path.
Each case stores: inputs, the reference ``state_dict``, injected noise, dense
outputs, and gradients of ``loss = sum(out * wt) [+ sum(x_enc * wt2)]``.
"""
from __future__ import annotations

import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402

warnings.filterwarnings("ignore")


def make_graph(n, avg_deg, seed, self_loops=True, weighted=False):
    """Random directed-symmetric graph as coalesced COO (idx int64 [2,E], val)."""
    g = torch.Generator().manual_seed(seed)
    m = n * avg_deg // 2
    src = torch.randint(0, n, (m,), generator=g)
    dst = torch.randint(0, n, (m,), generator=g)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    i = torch.cat([src, dst])
    j = torch.cat([dst, src])
    if self_loops:
        loops = torch.arange(n)
        i, j = torch.cat([i, loops]), torch.cat([j, loops])
    a = torch.sparse_coo_tensor(torch.stack([i, j]), torch.ones(i.numel()), (n, n)).coalesce()
    val = torch.ones_like(a.values())
    if weighted:
        val = 0.5 + torch.rand(val.shape, generator=g)
    return a.indices().clone(), val


def grads_of(loss, tensors):
    gs = torch.autograd.grad(loss, tensors, allow_unused=True)
    return [None if g is None else g.detach().clone() for g in gs]


def gumbel(shape, seed, scale):
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(shape, generator=g).clamp_(1e-10, 1 - 1e-7)
    return scale * -torch.log(-torch.log(u))


def main():
    ref = ref_loader.load_reference()
    rdgm, rmodel = ref["dgm"], ref["model"]
    out = {"cases": {}}
    n, f, h = 48, 24, 16
    idx, val = make_graph(n, 6, seed=1)
    gx = torch.Generator().manual_seed(2)
    x = torch.rand(n, f, generator=gx)
    x = x / x.sum(-1, keepdim=True)
    wt = torch.randn(n, n, generator=gx)
    wt2 = torch.randn(n, h, generator=gx)
    out["graph"] = dict(n=n, f=f, h=h, idx=idx, val=val, x=x, wt=wt, wt2=wt2)

    def adj_of(v=None):
        return torch.sparse_coo_tensor(idx, val if v is None else v, (n, n)).coalesce()

    # ---- class DGG (dgm.py:1730-1815) ------------------------------------
    torch.manual_seed(42)
    m = rdgm.DGG(in_dim=f, latent_dim=h, args=ref_loader.default_args())
    # make the node encoder less degenerate than default init on tiny inputs
    with torch.no_grad():
        m.node_encoder[0].weight.mul_(8.0)
        m.degree_decoder[0].weight.fill_(0.9)
        m.degree_decoder[0].bias.fill_(0.4)
    xg = x.clone().requires_grad_(True)
    sp, xe = m(xg, adj_of())
    dense = sp.to_dense()
    loss = (dense * wt).sum() + (xe * wt2).sum()
    params = list(m.parameters())
    g = grads_of(loss, params + [xg])
    out["cases"]["dgg"] = dict(
        state=m.state_dict(), out=dense.detach(), x_enc=xe.detach(),
        grads={k: gg for (k, _), gg in zip(m.named_parameters(), g[:-1])}, gx=g[-1],
    )

    # ---- DGG_Ablations (dgm.py:1876-1968) --------------------------------
    torch.manual_seed(43)
    m = rdgm.DGG_Ablations(in_dim=f, latent_dim=h, args=ref_loader.default_args())
    with torch.no_grad():
        m.node_encoder[0].weight.mul_(8.0)
    for tag, hard_k in (("ablation_soft", None), ("ablation_hard3", 3)):
        torch.manual_seed(7)
        noise = torch.rand(idx.shape[1]) * 2 - 1   # the draw dgm.py:1933 will make
        torch.manual_seed(7)
        sp, xe = m(x, adj_of(), k=hard_k)
        dense = sp.to_dense()
        loss = (dense * wt).sum()
        ps = [q for q in m.parameters()]
        g = grads_of(loss, ps)
        out["cases"][tag] = dict(
            state=m.state_dict(), noise=noise, hard_k=hard_k, out=dense.detach(),
            grads={k: gg for (k, _), gg in zip(m.named_parameters(), g)},
        )

    # ---- DGG_LearnableK_debug (dgm.py:1077-1727) -------------------------
    idx_w, val_w = idx, make_graph(n, 6, seed=1, weighted=True)[1]
    lk_cases = [
        # (tag, edge_mode, k_mode, select_mode, perturb, symmetric, weighted)
        ("lk_dist_x", "u-v-dist", "x", "k_times_edge_prob", False, True, False),
        ("lk_deg_x", "u-v-deg", "x", "k_times_edge_prob", False, True, False),
        ("lk_auv_inputdeg", "u-v-A_uv", "input_deg", "k_times_edge_prob", False, True, True),
        ("lk_degdist_lnd", "u-v-deg-dist", "learn_normalized_degree", "k_times_edge_prob", False, True, False),
        ("lk_edgeconv_gcn", "edge_conv", "gcn-x-deg", "k_times_edge_prob", False, True, False),
        ("lk_Auv_x", "A_uv", "x", "k_times_edge_prob", False, True, True),
        ("lk_dist_x_cdf", "u-v-dist", "pass", "edge_p-cdf", False, True, False),
        ("lk_dist_x_konly", "u-v-dist", "x", "k_only", False, True, False),
        ("lk_dist_x_pert_sym", "u-v-dist", "x", "k_times_edge_prob", True, True, False),
        ("lk_deg_x_pert_asym", "u-v-deg", "x", "k_times_edge_prob", True, False, False),
    ]
    for tag, em, km, sm, pert, sym, weighted in lk_cases:
        args = ref_loader.default_args(
            dgg_mode_edge_net=em, dgg_mode_k_net=km, dgg_mode_k_select=sm,
            perturb_edge_prob=pert, symmetric_noise=sym,
            extra_edge_dim=ref_loader.EXTRA_EDGE_DIM[em],
        )
        torch.manual_seed(44)
        m = rdgm.DGG_LearnableK_debug(in_dim=f, latent_dim=h, args=args)
        with torch.no_grad():
            m.node_encode_for_edges[0].weight.mul_(8.0)
            m.node_encode_for_k[0].weight.mul_(8.0)
        m.eval()
        noise = None
        if pert:
            if sym:
                noise = gumbel((n * (n - 1) // 2,), 99, 0.3)
            else:
                noise = gumbel((1, n, n), 99, 0.3)
            m.gumbel = ref_loader.FixedGumbel(noise)
        v = val_w if weighted else val
        xg = x.clone().requires_grad_(True)
        sp = m(xg, adj_of(v))
        dense = sp.to_dense()
        loss = (dense * wt).sum()
        named = [(k, q) for k, q in m.named_parameters()]
        g = grads_of(loss, [q for _, q in named] + [xg])
        out["cases"][tag] = dict(
            state={k: t for k, t in m.state_dict().items()}, args=vars(args), val=v,
            noise=noise, out=dense.detach(), nnz=int(sp._nnz()),
            grads={k: gg for (k, _), gg in zip(named, g[:-1])}, gx=g[-1],
        )

    # ---- legacy all-pairs metric (dgm.py:185-351) ------------------------
    import types

    na = 40
    xa = torch.randn(1, na, f, generator=gx)
    G = gumbel((na, na), 5, 1.0)
    orig = rdgm.gumbel_sample
    rdgm.gumbel_sample = lambda logits, temp, sl: orig(logits, G)     # dgm.py:295 arity shim
    m = rdgm.DGG_LearnableK_SDD(in_dim=f, latent_dim=h, dist_fn="metric")
    m.k_net.args = types.SimpleNamespace(stochastic_k=False)          # dgm.py:2053
    with torch.no_grad():
        m.t.fill_(6.0)
        m.k_net.k_project.bias.fill_(3.0)
    wta = torch.randn(na, na, generator=gx)
    adj, k = m(xa, temp=1.0, noise=True)
    loss = (adj[0] * wta).sum()
    named = [(kk, q) for kk, q in m.named_parameters() if q.requires_grad]
    g = grads_of(loss, [q for _, q in named])
    out["cases"]["allpairs_metric"] = dict(
        state=m.state_dict(), x=xa[0], G=G, wt=wta, out=adj[0].detach(), k=k[0].detach(),
        grads={kk: gg for (kk, _), gg in zip(named, g)},
    )
    adj_e, _ = m(xa, temp=10.0, noise=False)
    out["cases"]["allpairs_metric"]["out_eval_t10"] = adj_e[0].detach()
    rdgm.gumbel_sample = orig

    # ---- model-level (model.py) in eval mode ------------------------------
    nclass = 5
    idx_ns, val_ns = make_graph(n, 6, seed=1, self_loops=False)
    out["graph_noself"] = dict(idx=idx_ns, val=val_ns)
    wl = torch.randn(n, nclass, generator=gx)
    out["graph"]["wl"] = wl
    out["graph"]["nclass"] = nclass

    def run_model(tag, cls, args, call, scale_names=()):
        torch.manual_seed(45)
        mm = cls(nfeat=f, nlayers=4, nhidden=h, nclass=nclass, dropout=0.0,
                 lamda=0.5, alpha=0.1, variant=False, args=args)
        with torch.no_grad():
            for kk, q in mm.named_parameters():
                if any(s in kk for s in scale_names):
                    q.mul_(8.0)
        mm.eval()
        res = call(mm)
        logp = res[0] if isinstance(res, tuple) else res
        loss = (logp * wl).sum()
        named = [(kk, q) for kk, q in mm.named_parameters()]
        g = grads_of(loss, [q for _, q in named])
        out["cases"][tag] = dict(
            state=mm.state_dict(), args=vars(args), logp=logp.detach(),
            adj=(res[1].to_dense().detach() if isinstance(res, tuple) and res[1] is not None else None),
            grads={kk: gg for (kk, _), gg in zip(named, g)},
        )

    a_ns = torch.sparse_coo_tensor(idx_ns, val_ns, (n, n)).coalesce()
    args00 = ref_loader.default_args(extra_edge_dim=0)
    run_model("model_gcn_dgg_00", rmodel.GCN_DGG_00, args00,
              lambda mm: mm(x, a_ns), scale_names=("node_encoder",))
    run_model("model_sage_dgg_00", rmodel.SAGE_DGG_00, args00,
              lambda mm: mm(x, a_ns), scale_names=("node_encoder",))
    run_model("model_gat_dgg_00", rmodel.GAT_DGG_00, args00,
              lambda mm: mm(x, a_ns, edge_index=idx_ns), scale_names=("node_encoder",))
    args_lk = ref_loader.default_args(dgg_mode_edge_net="u-v-dist", extra_edge_dim=0)
    run_model("model_gcn_dgg", rmodel.GCN_DGG, args_lk,
              lambda mm: mm(x, a_ns), scale_names=("node_encode_for",))
    run_model("model_gcnii_dgg", rmodel.GCNII_DGG, args_lk,
              lambda mm: mm(x, a_ns), scale_names=("node_encode_for",))
    run_model("model_sage_dgg", rmodel.SAGE_DGG, args_lk,
              lambda mm: mm(x, a_ns), scale_names=("node_encode_for",))

    path = os.path.join(HERE, "dgg_golden.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB;", len(out["cases"]), "cases")


if __name__ == "__main__":
    main()
