"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the DGG hot path.

A dense, functional restatement (torch CPU fp32, autograd for gradients) of the
reference algorithm, one function per row of SURVEY.md section 8(a).  Every
function cites the reference file:line it follows.  It is deliberately the
*naive* O(N^2) dense algorithm -- the thing the CUDA path must agree with, not
something to ship: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.

Pinning status: the reference ships no tests or golden vectors (SURVEY.md
section 4), so the oracle is pinned against *outputs of the reference modules
themselves*, run in the build container through ``oracle/ref_loader.py``:
``tests/golden/make_golden.py`` stores those outputs as fixtures and
``tests/test_oracle_pinned.py`` checks every function here against them (and,
when ``DGG_REFERENCE_ROOT`` names a reference checkout, against the live reference modules).
The one third-party piece, PyG 2.1.0 ``DenseGraphConv`` (model.py:128-129), has
no source in the reference tree: ``sage_dense_mean`` restates its published
semantics -- parity unpinned at that boundary.

Parameters are passed as a dict keyed by the reference ``state_dict`` names
(e.g. ``node_encoder.0.weight``) so fixtures and product modules share weights.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

LRELU = 0.01  # nn.LeakyReLU() default slope, used everywhere in dgm.py


def _lin(x, p, name):
    return F.linear(x, p[name + ".weight"], p.get(name + ".bias"))


def dense_from_edges(idx, val, n):
    """torch.sparse.FloatTensor(idx, val, [n,n]).to_dense() (dgm.py:1787-1788):
    duplicates accumulate."""
    out = torch.zeros(n, n, dtype=val.dtype)
    return out.index_put((idx[0], idx[1]), val, accumulate=True)


def rank_desc(dense):
    """Row-wise descending sort -> (sorted values, column order) (dgm.py:1796,
    1404).  ``stable=True`` pins the tie order to "lower column first"; the
    reference's order among exact ties is unspecified."""
    return torch.sort(dense, dim=-1, descending=True, stable=True)


def first_k_tanh(n, k):
    """1 - 0.5 * (1 + tanh(t - k)), t = 0..n-1 (dgm.py:1410-1414, 1798-1803)."""
    t = torch.arange(n).reshape(1, n)
    return 1 - 0.5 * (1 + torch.tanh((t - k) / 1))


def unsort(sorted_vals, order):
    """clone().scatter_(-1, order, sorted_vals) (dgm.py:1810, 1420)."""
    return torch.zeros_like(sorted_vals).scatter(-1, order, sorted_vals)


# --------------------------------------------------------------------------- #
# a4 / a5 : class DGG and DGG_Ablations
# --------------------------------------------------------------------------- #
def dgg_forward(x, idx, n, p, ablation_noise=None, hard_k=None):
    """``DGG.forward`` (dgm.py:1758-1815); with ``ablation_noise`` (a tensor of
    E uniform(-1,1) draws, dgm.py:1933-1935) / ``hard_k`` (dgm.py:1943-1945) it
    is ``DGG_Ablations.forward`` (dgm.py:1904-1968).

    Returns dict(out=[n,n] dense adjacency, x_enc=[n,h], R=[E], k=[n,1])."""
    xe = F.leaky_relu(_lin(x, p, "node_encoder.0"), LRELU)          # 1778
    diff = xe[idx[0]] - xe[idx[1]]                                   # 1781-1783
    feat = F.leaky_relu(_lin(diff, p, "edge_encoder.0"), LRELU)      # 1784
    r = torch.sigmoid(feat.sum(-1))                                  # 1785-1786
    if ablation_noise is not None:
        r = torch.sigmoid(r + ablation_noise)                        # 1933-1935
    dense = dense_from_edges(idx, r, n)                              # 1787-1788
    srt, order = rank_desc(dense)                                    # 1796
    if hard_k is not None:
        srt = srt.clone()
        srt[:, hard_k:] = 0                                          # 1943-1945
        k = None
        weighted = srt
    else:
        k = F.leaky_relu(_lin(dense.sum(-1, keepdim=True), p,
                              "degree_decoder.0"), LRELU)            # 1791-1792
        weighted = srt * (first_k_tanh(n, k) + 1.0)                  # 1798-1807
    out = unsort(weighted, order)                                    # 1810
    return dict(out=out, x_enc=xe, R=r, k=k)


# --------------------------------------------------------------------------- #
# a6-a11, a14 : DGG_LearnableK_debug
# --------------------------------------------------------------------------- #
def k_encoder(x, p, prefix="k_net"):
    """``LearnableKEncoder.forward`` deterministic branch (dgm.py:2058-2063)."""
    return _lin(_lin(x, p, prefix + ".k_mu"), p, prefix + ".k_project")


def edge_prob_net(x, idx, val, n, p, mode):
    """``edge_prob_net`` (dgm.py:1596-1727) -> per-edge probability [E]."""
    u_i, v_i = idx[0], idx[1]
    if mode == "A_uv":                                               # 1720-1725
        return torch.sigmoid(_lin(val.unsqueeze(-1), p, "adj_project").flatten())
    xe = F.leaky_relu(_lin(x, p, "node_encode_for_edges.0"), LRELU)  # 1609
    u, v = xe[u_i], xe[v_i]
    if mode == "u-v-dist":                                           # 1618-1623
        return torch.exp(-0.05 * torch.linalg.vector_norm(u - v, dim=-1, ord=2))
    if mode == "edge_conv":                                          # 1710-1715
        f = _lin(v - u, p, "edge_conv_theta") + _lin(u, p, "edge_conv_phi")
        return torch.sigmoid(_lin(f, p, "edge_conv_encode").flatten())
    deg = dense_from_edges(idx, val, n).sum(-1, keepdim=True)        # 1653 (raw degree)
    if mode == "u-v-A_uv":                                           # 1635-1640
        feat = torch.cat([u, v, val.unsqueeze(-1)], -1)
    elif mode == "u-v-deg":                                          # 1657-1662
        feat = torch.cat([u, v, deg[u_i], deg[v_i]], -1)
    elif mode == "u-v-deg-dist":                                     # 1684-1694
        d = torch.exp(-1.0 * torch.linalg.vector_norm(u - v, dim=-1, ord=2))
        feat = torch.cat([u, v, deg[u_i], deg[v_i], d.unsqueeze(-1)], -1)
    else:
        raise Exception("mode not found")                            # 1727
    h = F.leaky_relu(_lin(feat, p, "edge_encode.0"), LRELU)
    return torch.sigmoid(_lin(h, p, "edge_encode.2").flatten())      # 1665-1666


def normalize_adj(a):
    """A_ij / (sqrt(s_i) sqrt(s_j)), s = ROW sums on both sides
    (model.py:1215-1218, dgm.py:1172-1175)."""
    s = a.sum(-1) ** -0.5
    return s.unsqueeze(-1) * a * s.unsqueeze(0)


def k_estimate_net(x, idx, val, n, p, mode, deg_mean=3.899, deg_std=5.288):
    """``k_estimate_net`` (dgm.py:1472-1586) -> k [n,1] (>= 1) or None."""
    if mode == "pass":
        return None
    a = dense_from_edges(idx, val, n)
    deg = a.sum(-1, keepdim=True)
    if mode == "learn_normalized_degree":                            # 1492-1507
        mu, sd = deg.mean(), deg.std()
        z = k_encoder(_lin((deg - mu) / sd, p, "input_degree_project"), p)
        return F.relu(z * sd + mu) + 1.0
    if mode == "input_deg":                                          # 1509-1526
        z = k_encoder(_lin((deg - deg_mean) / (deg_std + 1e-5), p,
                           "input_degree_project"), p)
        return F.relu(z * deg_std + deg_mean) + 1.0
    xe = F.leaky_relu(_lin(x, p, "node_encode_for_k.0"), LRELU)      # 1532 / 1566
    if mode == "gcn-x-deg":                                          # 1535-1540
        xe = torch.relu(normalize_adj(a) @ xe @ p["k_W"])
    elif mode != "x":
        raise Exception("k mode not found")
    mu, sd = deg.mean(), deg.std()
    feats = torch.cat([xe, (deg - mu) / (sd + 1e-5)], -1)            # 1568-1573
    z = k_encoder(F.leaky_relu(_lin(feats, p, "k_embed.0"), LRELU), p)
    return F.relu(z * sd + mu) + 1.0                                 # 1580-1584


def symmetric_noise(g_triu, n):
    """Noise layout of dgm.py:1218-1223: n(n-1)/2 draws on triu_indices(n,n,1),
    mirrored, zero diagonal."""
    g = torch.zeros(n, n, dtype=g_triu.dtype)
    i, j = torch.triu_indices(n, n, 1)
    g[i, j] = g_triu
    g[j, i] = g_triu
    return g


def select_top_k(pert, k, mode, p=None):
    """``select_top_k`` (dgm.py:1352-1435).  pert: dense [n,n]; k: [n,1]."""
    n = pert.shape[-1]
    srt, order = rank_desc(pert)
    if mode == "edge_p-cdf":                                         # 1368-1401
        return pert  # scatter of the *unweighted* sorted values == identity
    fk = first_k_tanh(n, k)
    if mode == "k_times_edge_prob":                                  # 1402-1421
        return unsort(srt * fk, order)
    if mode == "k_only":                                             # 1423-1435
        return unsort(fk.expand_as(srt).contiguous(), order)
    raise Exception("select mode not found")


def learnable_k_forward(x, idx, val, n, p, edge_mode="u-v-dist", k_mode="x",
                        select_mode="k_times_edge_prob", noise=None,
                        deg_mean=3.899, deg_std=5.288):
    """``DGG_LearnableK_debug.forward`` soft path, debug_step=3
    (dgm.py:1178-1298).  ``noise``: None (perturb_edge_prob=False) or a dense
    [n,n] Gumbel(0,0.3) tensor G (already mirrored if symmetric).

    Returns dict(out=[n,n] dense (to_sparse() of it drops exact zeros), P, k)."""
    pe = edge_prob_net(x, idx, val, n, p, edge_mode)
    dense_p = dense_from_edges(idx, pe, n)
    if noise is not None:
        pert = torch.exp(torch.log(dense_p + 1e-8) + noise)          # 1213-1229
    else:
        pert = dense_p
    k = k_estimate_net(x, idx, val, n, p, k_mode, deg_mean, deg_std)
    out = select_top_k(pert, k, select_mode, p)
    return dict(out=out, P=pe, k=k, pert=pert)


# --------------------------------------------------------------------------- #
# a15 : legacy all-pairs metric DGG (the north-star "N x N pairwise" formula)
# --------------------------------------------------------------------------- #
def allpairs_metric_forward(x, p, noise, temp=1.0, k_bias=1.0, hs_start=2.0,
                            hs_end=-5.0, k_input="raw"):
    """``DGG_LearnableK_SDD.forward(dist_fn="metric")`` for one graph
    (dgm.py:259-341).  noise: dense [n,n] G (training) or None (eval softmax).

    Returns dict(out=[n,n], k=[n,1], y=[n,n] perturbed log-probs)."""
    z = torch.softmax(F.leaky_relu(_lin(x, p, "input_project.0"), LRELU), -1)  # 217-221, 271
    dist = torch.cdist(z.unsqueeze(0), z.unsqueeze(0), p=2).squeeze(0)          # 275
    log_p = torch.log(torch.exp(-p["t"] * dist))                                # 276, 290
    y = log_p + noise if noise is not None else torch.softmax(log_p / temp, -1)  # 292-298 (+ dgm.py:28)
    srt, order = rank_desc(y)                                                   # 301
    k = k_encoder(x if k_input == "raw" else z, p) + k_bias                     # 304-312
    n = x.shape[0]
    interval = hs_start - hs_end
    support = hs_start - interval * torch.arange(n, dtype=torch.float32)        # 315-320
    fk = torch.sigmoid(support.reshape(1, n) + (k - 1) * interval)              # 321-326
    out = unsort(srt * fk, order)                                               # 329-332
    return dict(out=out, k=k, y=y, z=z)


# --------------------------------------------------------------------------- #
# a13, a17-a20 : normalisation and the aggregation layers
# --------------------------------------------------------------------------- #
def gcn_conv(x, adj, w):
    """``GCNConv.forward`` relu((A x) W) (model.py:594-598)."""
    return torch.relu((adj @ x) @ w)


def gcnii_conv(x, adj, h0, w, lamda, alpha, layer, variant=False, residual=False):
    """``DenseGraphConvolution.forward`` (model.py:65-77)."""
    theta = math.log(lamda / layer + 1)
    hi = adj @ x
    if variant:
        support = torch.cat([hi, h0], 1)
        r = (1 - alpha) * hi + alpha * h0
    else:
        support = (1 - alpha) * hi + alpha * h0
        r = support
    out = theta * (support @ w) + (1 - theta) * r
    return out + x if residual else out


def gat_conv_dgg(x, edge_list, adj_dense, w, a, bias, alpha=0.2):
    """``GATConv_DGG.forward`` in eval mode (model.py:556-577): non-edge logits
    are -1e20 * A_ij (== -0.0 where A_ij is 0), i.e. a dense softmax."""
    h = x @ w
    e = F.leaky_relu(torch.cat([h[edge_list[0]], h[edge_list[1]]], 1) @ a, alpha)
    n = h.shape[0]
    att = torch.full((n, n), -1e20).index_put((edge_list[0], edge_list[1]), e[:, 0])
    att = torch.softmax(att * adj_dense, dim=1)
    out = att @ h
    return out + bias if bias is not None else out


def sage_dense_mean(x, adj, w_rel, b_rel, w_root):
    """PyG 2.1.0 ``DenseGraphConv(aggr="mean")`` (model.py:128-129; source not
    in the reference tree -- restated from its published semantics)."""
    agg = (adj @ x) / adj.sum(-1, keepdim=True).clamp(min=1)
    return F.linear(agg, w_rel, b_rel) + F.linear(x, w_root)


def add_self_loops_dense(idx, val, n):
    """(A.to_dense() + I) (model.py:1249-1251)."""
    return dense_from_edges(idx, val, n) + torch.eye(n)


# --------------------------------------------------------------------------- #
# a21 : model forwards (eval mode / dropout off)
# --------------------------------------------------------------------------- #
def gcn_dgg_00_forward(x, idx, val, n, p):
    """``GCN_DGG_00.forward`` (model.py:1368-1428), eval mode.
    p holds ``dggs.0.*``, ``conv1.W``, ``conv2.W``."""
    a = add_self_loops_dense(idx, val, n)
    sp = a.to_sparse().coalesce()
    d = dgg_forward(x, sp.indices(), n, {k[7:]: v for k, v in p.items() if k.startswith("dggs.0.")})
    na = normalize_adj(d["out"])
    xe = d["x_enc"]
    h = gcn_conv(xe + xe, na, p["conv1.W"])                          # 1405-1407
    h = gcn_conv(h + xe, na, p["conv2.W"])
    return dict(logp=F.log_softmax(h, -1), adj=d["out"], x_enc=xe)
