"""CPU: checkpoints in the reference's format round-trip through the drop-in modules, and a ``state_dict`` produced by
the REFERENCE's own classes loads into them key for key: live where a reference checkout exists, otherwise from the
reference state_dicts stored in tests/golden/dgg_golden.pt."""
import argparse
import os

import pytest
import torch

import dgg_b200
import model as models


def _args(**kw):
    d = dict(extra_edge_dim=2, extra_k_dim=1, dgg_hard=False, deg_mean=3.899, deg_std=5.288,
             dgg_mode_edge_net="u-v-deg", dgg_mode_k_net="x", dgg_mode_k_select="k_times_edge_prob", debug_step=3,
             perturb_edge_prob=False, symmetric_noise=True, stochastic_k=False, dgg_adj_input="input_adj",
             n_dgg_layers=2)
    d.update(kw)
    return argparse.Namespace(**d)


def _build(name, args):
    return models.__dict__[name](nfeat=20, nlayers=4, nhidden=16, nclass=3, dropout=0.5, lamda=0.5, alpha=0.1,
                                 variant=False, args=args)


@pytest.mark.parametrize("name", ["GCN_DGG", "GCN_DGG_00", "GCNII_DGG", "SAGE_DGG_00", "GAT_DGG_00", "GCN", "GCNII",
                                  "SAGE", "GAT"])
def test_checkpoint_round_trip(tmp_path, name):
    args = _args(extra_edge_dim=2 if name in ("GCN_DGG", "GCNII_DGG") else 0)
    torch.manual_seed(0)
    a = _build(name, args)
    opt = torch.optim.Adam(a.parameters(), lr=0.01)
    fn = str(tmp_path / "ck.pt")
    dgg_b200.checkpoint.save_checkpoint(fn, args, 7, a, opt)
    torch.manual_seed(1)
    b = _build(name, args)
    assert dgg_b200.checkpoint.load_checkpoint(fn, b) == 7
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)
    torch.save(a.state_dict(), fn)                       # the upstream scripts' bare state_dict
    assert dgg_b200.checkpoint.load_checkpoint(fn, b) is None


# state_dicts of the reference's own classes stored by tests/golden/make_golden.py (tests/golden/dgg_golden.pt)
GOLDEN_STATE = {"GCN_DGG": "model_gcn_dgg", "GCN_DGG_00": "model_gcn_dgg_00", "GCNII_DGG": "model_gcnii_dgg",
                "SAGE_DGG": "model_sage_dgg", "SAGE_DGG_00": "model_sage_dgg_00", "GAT_DGG_00": "model_gat_dgg_00"}


@pytest.mark.parametrize("name", ["GCN_DGG", "GCN_DGG_00", "GCNII_DGG", "SAGE_DGG", "SAGE_DGG_00", "GAT_DGG_00", "GCN",
                                  "GCNII", "SAGE", "GAT"])
def test_reference_state_dict_loads(golden, name):
    from oracle import ref_loader

    if not ref_loader.reference_available():
        if name not in GOLDEN_STATE:
            pytest.skip(f"no stored reference state_dict of {name}: needs a reference checkout (DGG_REFERENCE_ROOT)")
        g, c = golden["graph"], golden["cases"][GOLDEN_STATE[name]]
        ours = models.__dict__[name](nfeat=g["f"], nlayers=4, nhidden=g["h"], nclass=g["nclass"], dropout=0.0,
                                     lamda=0.5, alpha=0.1, variant=False, args=argparse.Namespace(**c["args"]))
        ours.load_state_dict(c["state"], strict=True)
        assert {k: v.shape for k, v in ours.state_dict().items()} == {k: v.shape for k, v in c["state"].items()}
        return
    ref = ref_loader.load_reference(("dgm", "model"))["model"]
    args = _args(extra_edge_dim=2 if name in ("GCN_DGG", "GCNII_DGG", "SAGE_DGG") else 0)
    torch.manual_seed(0)
    theirs = ref.__dict__[name](nfeat=20, nlayers=4, nhidden=16, nclass=3, dropout=0.5, lamda=0.5, alpha=0.1,
                                variant=False, args=args)
    ours = _build(name, args)
    ours.load_state_dict(theirs.state_dict(), strict=True)
    assert sorted(ours.state_dict().keys()) == sorted(theirs.state_dict().keys())
