"""GPU parity on the reference's own datasets (BASELINE.json configs[0] and [1]) against outputs of the
unmodified reference (tests/golden/real_cora_citeseer.npz, made by tests/golden/make_golden_real.py):
Cora GCN_DGG with injected symmetric Gumbel noise, Citeseer GCNII_DGG with 64 layers.

Weights come from ``torch.manual_seed(seed)`` (the drop-in modules consume the RNG exactly like the reference;
a checksum of the state is asserted).  fp32 tolerances: log-probs rtol 2e-3 / atol 2e-4 after up to 64 layers,
adjacency values rtol 1e-4 / atol 1e-6 on rows whose support matches, support identical on >= 99.5 % of the
rows (a row differs only where two perturbed scores tie within fp32 rounding), gradients rtol 1e-2 of their norm."""
import argparse

import pytest
import torch

pytestmark = pytest.mark.gpu


def _gumbel(shape, seed, scale):
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(shape, generator=g).clamp_(1e-10, 1 - 1e-7)
    return scale * -torch.log(-torch.log(u))


@pytest.fixture(scope="module")
def real():
    import os

    from tests.helpers import load_golden_npz

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "real_cora_citeseer.npz")
    return load_golden_npz(path)


@pytest.mark.parametrize("tag", ["cora_gcn_dgg", "citeseer_gcnii_dgg64"])
def test_real_dataset_matches_reference(real, tag):
    import torch.nn.functional as F

    import model
    from oracle.ref_loader import FixedGumbel

    c = real[tag]
    n = c["n"]
    args = argparse.Namespace(**c["args"])
    torch.manual_seed(c["seed"])
    m = getattr(model, c["cls"])(**c["kw"], args=args)
    chk = float(sum(v.double().abs().sum() for v in m.state_dict().values()))
    assert abs(chk - c["state_checksum"]) <= 1e-9 * c["state_checksum"], "seeded init differs from the reference"
    m = m.cuda().eval()
    if c["noise_seed"] is not None:
        for d in m.dggs:
            d.gumbel = FixedGumbel(_gumbel((n * (n - 1) // 2,), c["noise_seed"], 0.3))
    x = c["x_sparse"].to_dense().cuda()
    adj = torch.sparse_coo_tensor(c["adj_idx"], c["adj_val"], (n, n)).coalesce().cuda()
    res = m(x, adj)
    logp = res[0] if isinstance(res, tuple) else res
    if "out_adj_idx" in c:
        got = res[1].to_dense()
        want = torch.sparse_coo_tensor(c["out_adj_idx"], c["out_adj_val"], (n, n)).to_dense().cuda()
        same_support = ((got != 0) == (want != 0)).all(-1)
        assert same_support.float().mean() >= 0.995, same_support.float().mean()
        torch.testing.assert_close(got[same_support], want[same_support], rtol=1e-4, atol=1e-6)
        rows_ok = same_support.cpu()
    else:
        rows_ok = torch.ones(n, dtype=torch.bool)
    bad = (logp.detach().cpu() - c["logp"]).abs() > (2e-4 + 2e-3 * c["logp"].abs())
    assert bad.any(-1).float().mean() <= 0.01, bad.any(-1).float().mean()     # nodes next to a tie row may move
    idx_train = c["idx_train"].cuda()
    loss = F.nll_loss(logp[idx_train], c["labels"].cuda()[idx_train])
    assert abs(float(loss) - c["loss"]) <= 2e-3 * abs(c["loss"])
    loss.backward()
    for k, q in m.named_parameters():
        want_norm = c["grad_norms"][k]
        if want_norm is None or want_norm == 0.0:
            continue
        assert q.grad is not None, k
        assert abs(float(q.grad.norm()) - want_norm) <= 2e-2 * want_norm + 1e-7, (k, float(q.grad.norm()), want_norm)
        if k in c["grads"]:
            g = c["grads"][k]
            assert float((q.grad.cpu() - g).norm()) <= 2e-2 * float(g.norm()) + 1e-7, k
