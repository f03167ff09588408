"""Known-answer fixtures on the reference's own datasets (BASELINE.json configs[0], configs[1]) produced by
the UNMODIFIED reference modules:

  * Cora      GCN_DGG   (train_small_graphs.py defaults: u-v-deg / x / k_times_edge_prob, extra_edge_dim=2),
                        perturb_edge_prob=True with the symmetric Gumbel(0,0.3) noise INJECTED (seeded);
  * Citeseer  GCNII_DGG 64 layers, n_dgg_layers=2 (edge net u-v-dist).

Weights are not stored: the drop-in modules consume the global RNG exactly like the reference, so
``torch.manual_seed(seed)`` + construction reproduces them bit-for-bit (checked here).  Stored: sparse
features, edges, labels/train mask, log-probs, learned adjacency, selected gradients.  Build container only.
"""
from __future__ import annotations

import os
import sys
import warnings

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402
from tests.helpers import save_golden_npz  # noqa: E402

warnings.filterwarnings("ignore")
KEEP_GRADS = 8   # gradients of the first / last few parameters are stored, plus the norm of all of them


def gumbel(shape, seed, scale):
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(shape, generator=g).clamp_(1e-10, 1 - 1e-7)
    return scale * -torch.log(-torch.log(u))


def load(ref, name):
    cwd = os.getcwd()
    os.chdir(ref_loader.REFERENCE_ROOT)
    try:
        adj, feats, labels, idx_train, _, _ = ref["utils"].load_citation(name, ref_loader.REFERENCE_ROOT)
    finally:
        os.chdir(cwd)
    return adj.coalesce(), feats, labels, idx_train


def run(ref, tag, data, cls, kw, args, seed, noise_seed=None):
    import model as mine

    adj, x, labels, idx_train = data
    n = x.shape[0]
    torch.manual_seed(seed)
    m = getattr(ref["model"], cls)(**kw, args=args)
    torch.manual_seed(seed)
    m2 = getattr(mine, cls)(**kw, args=args)
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2), (k1, k2)
    m.eval()
    if noise_seed is not None:
        for d in m.dggs:
            d.gumbel = ref_loader.FixedGumbel(gumbel((n * (n - 1) // 2,), noise_seed, 0.3))
    res = m(x, adj)
    logp = res[0] if isinstance(res, tuple) else res
    loss = F.nll_loss(logp[idx_train], labels[idx_train])
    named = list(m.named_parameters())
    grads = torch.autograd.grad(loss, [p for _, p in named], allow_unused=True)
    gd = {k: (None if g is None else g.detach()) for (k, _), g in zip(named, grads)}
    small = {k: g for k, g in gd.items() if g is not None and g.numel() <= 70000}
    keep = dict(list(small.items())[:KEEP_GRADS] + list(small.items())[-KEEP_GRADS:])
    out = dict(
        n=n, f=x.shape[1], x_sparse=x.to_sparse().coalesce(), adj_idx=adj.indices(), adj_val=adj.values(),
        labels=labels, idx_train=idx_train, cls=cls, kw=kw, args=vars(args), seed=seed, noise_seed=noise_seed,
        logp=logp.detach(), loss=float(loss), grads=keep,
        grad_norms={k: (None if g is None else float(g.norm())) for k, g in gd.items()},
        state_checksum=float(sum(v.double().abs().sum() for v in m.state_dict().values())),
    )
    if isinstance(res, tuple) and res[1] is not None:
        a = res[1].coalesce()
        out["out_adj_idx"], out["out_adj_val"] = a.indices(), a.values().detach()
    print(tag, "loss", float(loss), "logp", tuple(logp.shape),
          "adj nnz", None if "out_adj_idx" not in out else out["out_adj_idx"].shape[1])
    return out


def main():
    ref = ref_loader.load_reference(("dgm", "model", "utils"))
    fx = {}
    cora = load(ref, "cora")
    a0 = ref_loader.default_args(dgg_mode_edge_net="u-v-deg", extra_edge_dim=2, perturb_edge_prob=True,
                                 symmetric_noise=True)
    fx["cora_gcn_dgg"] = run(ref, "cora_gcn_dgg", cora, "GCN_DGG",
                             dict(nfeat=cora[1].shape[1], nlayers=2, nhidden=64, nclass=7, dropout=0.5, lamda=0.5,
                                  alpha=0.1, variant=False), a0, seed=42, noise_seed=1234)
    cs = load(ref, "citeseer")
    a1 = ref_loader.default_args(dgg_mode_edge_net="u-v-dist", extra_edge_dim=0, n_dgg_layers=2)
    fx["citeseer_gcnii_dgg64"] = run(ref, "citeseer_gcnii_dgg64", cs, "GCNII_DGG",
                                     dict(nfeat=cs[1].shape[1], nlayers=64, nhidden=64, nclass=6, dropout=0.6,
                                          lamda=0.5, alpha=0.1, variant=False), a1, seed=42)
    path = os.path.join(HERE, "real_cora_citeseer.npz")
    save_golden_npz(path, fx)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
