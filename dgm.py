"""Drop-in replacement for the reference ``dgm.py`` (Differentiable Graph Generator), B200-native.

Same class names, constructor/forward signatures, parameter names (``state_dict`` compatible) and
``args`` attribute surface as the reference (SURVEY.md 8b, Appendix B), but nothing here ever builds
a dense N x N matrix: adjacencies stay CSR-resident and every hot op is a hand-written sm_100a kernel
behind the C-ABI in include/dggb.h (bound in dgg_b200/functional.py).  CUDA tensors only.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

import dgg_b200
from dgg_b200 import CSRGraph
from dgg_b200 import functional as K


def sample_gumbel_from_uniform(shape, eps=1e-20):
    """Gumbel(0,1) from uniform draws; same recipe as reference dgm.py:6-11."""
    u = torch.rand(shape, device="cuda" if torch.cuda.is_available() else "cpu")
    return -torch.log(-torch.log(u + eps) + eps)


def gumbel_sample(logits, noise_sample):
    """Reference dgm.py:14-29: the self-loop mask is computed there but never applied, so the
    contract is plain ``logits + noise_sample`` (SURVEY 2.3)."""
    assert logits.shape == noise_sample.shape
    return logits + noise_sample


class _EdgeRankerBase(nn.Module):
    """Shared body of ``DGG`` (dgm.py:1730-1815) and ``DGG_Ablations`` (dgm.py:1876-1968)."""

    def __init__(self, in_dim=32, latent_dim=64, args=None):
        super().__init__()
        self.args = args
        self.node_encoder = nn.Sequential(nn.Linear(in_dim, latent_dim), nn.LeakyReLU())
        self.edge_encoder = nn.Sequential(
            nn.Linear(latent_dim + self.args.extra_edge_dim, latent_dim), nn.LeakyReLU())
        self.degree_decoder = nn.Sequential(nn.Linear(1, 1, bias=True), nn.LeakyReLU())
        self.var_grads = {"edge_p": [], "first_k": [], "out_adj": []}

    def _rank_edges(self, x, adj, noise=None, hard_k=-1):
        assert x.ndim == 2
        assert len(adj.shape) == 2
        graph, _ = CSRGraph.from_coo(adj)
        enc, lin = self.node_encoder[0], self.edge_encoder[0]
        # Linear is linear: We (x_u - x_v) + be == y_u - y_v + be with y = x_enc We^T, so the per-edge
        # E x h x h GEMM of dgm.py:1783-1784 becomes one N x h x h GEMM plus a gather.
        x_enc, y = K.encode_project(x, enc.weight, enc.bias, lin.weight,
                                    self.node_encoder[1].negative_slope)                       # dgm.py:1778, 1784
        dd = self.degree_decoder[0]
        out_vals, k, R, rank = K.dgg_edge(y, lin.bias, dd.weight, dd.bias, graph, noise, hard_k)
        self.last_k, self.last_rank = k.detach(), rank
        return graph, out_vals, x_enc


class DGG(_EdgeRankerBase):
    """Differentiable graph generator, edge-restricted ranker (reference dgm.py:1730-1815).

    forward(x [N,F], adj sparse COO [N,N]) -> (sparse COO [N,N] with the support of ``adj``, x_enc [N,h]).
    ``noise`` is accepted and ignored exactly like the reference (dgm.py:1758)."""

    def forward(self, x, adj, noise=True, writer=None, epoch=None):
        graph, out_vals, x_enc = self._rank_edges(x, adj)
        return graph.to_coo(out_vals), x_enc


class DGG_Ablations(_EdgeRankerBase):
    """Reference dgm.py:1876-1968: uniform(-1,1) score noise + optional hard integer k."""

    def forward(self, x, adj, k=None, writer=None, epoch=None):
        graph, _ = CSRGraph.from_coo(adj)
        noise = torch.rand(graph.nnz, device=x.device) * 2 - 1          # dgm.py:1933
        if k is None:
            graph, out_vals, x_enc = self._rank_edges(x, adj, noise=noise)
            return graph.to_coo(out_vals), x_enc
        graph, out_vals, x_enc = self._rank_edges(x, adj, noise=noise, hard_k=int(k))
        # srt[:, k:] = 0 then to_sparse(): entries ranked >= k are dropped from the support (1943-1945)
        keep = (out_vals != 0).nonzero().flatten()
        idx = graph.coo_indices()[:, keep]
        return torch.sparse_coo_tensor(idx, out_vals[keep], (graph.n, graph.n), is_coalesced=True), x_enc


class LearnableKEncoder(nn.Module):
    """Reference dgm.py:2029-2063: k = k_project(k_mu(x)), or a reparameterised latent sample when
    ``args.stochastic_k`` and training."""

    def __init__(self, in_dim, latent_dim, learn_k_bias=False, args=None):
        super().__init__()
        self.learn_k_bias = learn_k_bias
        self.k_mu = nn.Linear(in_dim, latent_dim)
        self.k_logvar = nn.Linear(in_dim, latent_dim)
        self.k_project = nn.Linear(latent_dim, 1)
        self.args = args

    def latent_sample(self, mu, logvar):
        if self.training:
            std = logvar.mul(0.5).exp_()
            return torch.empty_like(std).normal_().mul(std).add_(mu)
        return mu

    @staticmethod
    def _lin(layer, x):
        # x is [N, small]: the weight gradient dpre^T x reduces over the N nodes into a tiny output, which the library
        # GEMM leaves on a handful of CTAs (Citeseer shape: 70 us for the [16, N] x [N, 32] product, 7 % of the
        # GCNII_DGG-64 step over its three layers); tall_linear sends it through the split-K kernel
        return K.tall_linear(x, layer.weight, layer.bias) if x.is_cuda else layer(x)

    def forward(self, x):
        if self.args.stochastic_k:
            latent_k = self.latent_sample(self._lin(self.k_mu, x), self._lin(self.k_logvar, x))
        else:
            latent_k = self._lin(self.k_mu, x)
        return self._lin(self.k_project, latent_k)


class DGG_LearnableK_SDD(nn.Module):
    """All-pairs DGG (reference dgm.py:185-351, ``dist_fn="metric"``), the north star's
    "N x N pairwise score + Gumbel + soft top-k" path, without ever forming N x N:

        z = softmax(LeakyReLU(x W + b));  y_ij = -t |z_i - z_j| + G_ij;  r = descending rank in row i;
        k_i = k_net(x_i) + k_bias;        adj_ij = y_ij * sigmoid(hs_start - interval r + (k_i - 1) interval)

    The first-k sigmoid is exactly 0 in fp32 for r > k + 11.96 (default hs_start / hs_end), so only the top
    ceil(k_max + k_window) entries per row can be non-zero: they are selected by a fused tcgen05 GEMM + streaming
    top-K kernel (more than 64 per row: several passes, see ``_select``).
    forward(x [B,N,F] or [N,F], temp, noise) -> (sparse COO adjacency [N,N] (list if B > 1), k [B,N,1]).
    ``noise``: True -> Gumbel(0,1) noise (sampled on device, or the tensor set via ``set_noise``);
    False -> softmax(log_p / temp) scores (evaluation branch, dgm.py:298)."""

    KC_MAX = 64          # entries per row one selector pass can return (allpairs kernel limit)
    SIGMOID_ZERO = 88.73  # torch.sigmoid(-x) == 0.0 in fp32 for x > 88.73 (SURVEY 7.3)

    def __init__(self, in_dim=32, latent_dim=64, k_bias=1.0, hard=False, self_loops_noise=False, dist_fn="metric",
                 k_net_input="raw", hs_start=2, hs_end=-5, n_agents=None, learn_k_bias=None, args=None):
        super().__init__()
        torch.manual_seed(0)                                  # reference side effect (dgm.py:207)
        if dist_fn != "metric":
            raise NotImplementedError("only dist_fn='metric' is supported (the 'mlp' branch is log_p == 0)")
        if hard:
            raise NotImplementedError("hard=True: the reference's straight-through branch (dgm.py:344-346) builds "
                                      "dense N x N tensors; only the soft adjacency is provided")
        self.in_dim, self.latent_dim = in_dim, latent_dim
        self.hard, self.self_loops_noise = hard, self_loops_noise
        self.dist_fn, self.k_net_input = dist_fn, k_net_input
        self.input_project = nn.Sequential(nn.Linear(in_dim, latent_dim), nn.LeakyReLU(), nn.Softmax(dim=-1))
        self.t = nn.Parameter(torch.ones(1))
        self.register_buffer("interval", torch.tensor(hs_start - hs_end))
        self.register_buffer("k_bias", torch.tensor(k_bias))
        self.register_buffer("hs_start", torch.tensor(hs_start))
        self.register_buffer("hs_end", torch.tensor(hs_end))
        # first_k = sigmoid(hs_start - interval * (r - (k - 1))) is exactly 0 once r - (k - 1) exceeds this
        # (12.96 for the default hs_start = 2, hs_end = -5); 0.64 ranks of safety margin
        self.k_window = (float(hs_start) + self.SIGMOID_ZERO) / float(hs_start - hs_end) - 1.0 + 0.64
        import argparse
        kargs = args if args is not None else argparse.Namespace(stochastic_k=False)
        self.k_net = LearnableKEncoder(in_dim=in_dim if k_net_input == "raw" else latent_dim,
                                       latent_dim=latent_dim, args=kargs)
        self._noise = None
        self.precision = 3
        # Per-row window sizing without a device->host sync on every forward: the number of entries a row can need,
        # ceil(k_max + k_window), is copied to pinned host memory asynchronously and read by the NEXT forward
        # (k drifts slowly during training); the selector runs with the bucket 16 / 32 / 64 [/ multiples of 64 in
        # several passes] that covers the last observed need with 25 % headroom.  A step whose rows needed more
        # than it was given is reported by ``overflowed()`` / raised at the next forward.  ``exact_kc = True``
        # restores the synchronous, always-exact sizing.
        self.exact_kc = False
        self._need_host = None
        self._need_event = None
        self._kc_last = None

    def set_noise(self, G):
        """Inject the Gumbel tensor [N,N] used by the next forward (parity tests; the reference's
        injection point is ``gumbel_sample``, dgm.py:14)."""
        self._noise = G

    # ------------------------------------------------------------------ window sizing
    @staticmethod
    def _bucket(need):
        for b in (16, 32, 64):
            if need <= b:
                return b
        return 64 * int(math.ceil(need / 64.0))

    def overflowed(self):
        """True if the previous forward's rows needed more entries than the selector was run with (synchronises)."""
        if self._need_event is None:
            return False
        self._need_event.synchronize()
        return int(self._need_host.item()) > self._kc_last

    def _pick_kc(self, k, n):
        # (never more than the n columns a row has: kc == n already selects every one of them)
        need_dev = torch.ceil(k.detach().max() + self.k_window).clamp(min=1.0, max=float(n))
        capturing = k.is_cuda and torch.cuda.is_current_stream_capturing()
        if self.exact_kc and not capturing:
            need = int(need_dev.item())
            kc = self._bucket(need)
        else:
            if self._need_event is None:
                if capturing:
                    raise RuntimeError("DGG_LearnableK_SDD: run one eager forward before capturing a CUDA graph")
                need = int(need_dev.item())                     # first call: one sync to initialise the hint
                kc = self._bucket(int(math.ceil(need * 1.25)))
            else:
                if not capturing:
                    self._need_event.synchronize()              # completed long ago: the previous step's copy
                last_need = int(self._need_host.item())
                if last_need > self._kc_last and not capturing:
                    kc_was = self._kc_last
                    self._kc_last = self._bucket(int(math.ceil(last_need * 1.25)))
                    raise dgg_b200.DggbError(
                        "DGG_LearnableK_SDD: K overflow (DGGB_ERR_K_OVERFLOW) in the previous forward: a row needed "
                        "%d entries, the selector ran with %d; the window has been enlarged, re-run the step "
                        "(or set exact_kc=True)" % (last_need, kc_was))
                kc = self._bucket(int(math.ceil(last_need * 1.25)))
            if not capturing:
                if self._need_host is None:
                    self._need_host = torch.zeros(1, dtype=torch.float32).pin_memory()
                    self._need_event = torch.cuda.Event()
                self._need_host.copy_(need_dev.reshape(1), non_blocking=True)
                self._need_event.record()
        kc = min(kc, n)
        self._kc_last = kc
        return kc

    def _select(self, z, kc, **kw):
        """Top-kc of every row, sorted descending; kc > KC_MAX runs ceil(kc / 64) selector passes, each one
        restricted to the entries that sort strictly after the last one the previous pass returned (the
        two-pass fallback of SURVEY 7.3 generalised to any k)."""
        if kc <= self.KC_MAX:
            return K.allpairs_topk(z, self.t, kc=kc, precision=self.precision, **kw)
        outs, after = [], None
        for p0 in range(0, kc, self.KC_MAX):
            kp = min(self.KC_MAX, kc - p0)
            res = K.allpairs_topk(z, self.t, kc=kp, precision=self.precision, after=after, **kw)
            outs.append(res)
            after = (res[1][:, -1].detach().contiguous(), res[0][:, -1].contiguous())
        idx = torch.cat([o[0] for o in outs], dim=1)
        y = torch.cat([o[1] for o in outs], dim=1)
        if len(outs[0]) == 3:
            return idx, y, outs[0][2]
        return idx, y

    def _one(self, x, temp, noise):
        n = x.shape[0]
        z = self.input_project(x)
        k = self.k_net(x if self.k_net_input == "raw" else z) + self.k_bias          # [N,1]
        kc = self._pick_kc(k, n)
        if noise:
            if self._noise is not None:
                idx, y = self._select(z, kc, noise=self._noise)
            else:   # Gumbel(0,1) generated inside the kernel (counter-based): no N x N noise tensor
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
                idx, y = self._select(z, kc, seed=seed, noise_scale=1.0)
        else:
            # evaluation branch (dgm.py:298): edge_prob = softmax(log_p / temp) over ALL columns.  The ordering is
            # that of log_p; the normaliser sum_j exp(log_p_ij / temp) is accumulated by the same streaming pass.
            # Forward only (inference): the normaliser's gradient would touch all N^2 pairs.
            idx, logp, zsum = self._select(z, kc, inv_temp=1.0 / float(temp))
            y = (torch.exp(logp / float(temp)) / zsum.unsqueeze(-1)).detach()
        r = torch.arange(kc, device=x.device, dtype=torch.float32).reshape(1, kc)
        first_k = torch.sigmoid(self.hs_start - self.interval * r + (k - 1) * self.interval)   # dgm.py:315-326
        vals = y * first_k
        rows = torch.arange(n, device=x.device).reshape(n, 1).expand(n, kc)
        keep = idx >= 0
        adj = torch.sparse_coo_tensor(torch.stack([rows[keep], idx[keep].long()]), vals[keep], (n, n))
        return adj, k

    def forward(self, x, temp, noise=True):
        if x.dim() == 2:
            adj, k = self._one(x, temp, noise)
            return adj, k.unsqueeze(0)
        outs = [self._one(xb, temp, noise) for xb in x]
        adjs = [a for a, _ in outs]
        return (adjs[0] if len(adjs) == 1 else adjs), torch.stack([k for _, k in outs])


class DGG_LearnableK_debug(nn.Module):
    """Reference dgm.py:1077-1727, CSR-resident.  Same parameters (every sub-module of the reference
    exists, used or not, so ``state_dict`` round-trips), same ``args`` surface, same modes:

    edge net (dgm.py:1596-1727): u-v-dist, u-v-A_uv, u-v-deg, u-v-deg-dist, edge_conv, A_uv
    k net    (dgm.py:1472-1586): pass, learn_normalized_degree, input_deg, gcn-x-deg, x
    select   (dgm.py:1352-1435): k_times_edge_prob, k_only, edge_p-cdf (identity on the edge probabilities)

    The dense [N,N] scatter / sort / un-sort of the reference is replaced by in-row ranking on the CSR
    support (off-support entries are exact zeros that sort last).  Entries whose soft first-k weight
    saturates to exactly 0 stay in the returned support as explicit zeros (``to_dense()`` and all
    gradients are identical to the reference, which drops them in ``to_sparse()``).
    ``perturb_edge_prob=True`` (Gumbel noise on all N^2 entries) is evaluated exactly on the union of each
    row's edges and its best off-support entries (see ``_perturb``).
    ``k_only`` spills a row's window past its degree into its first non-edge columns (``_k_only_spill``).
    Not covered: ``dgg_hard`` (SURVEY 2.3: buggy scatter in the reference) -- it raises."""

    TANH_WINDOW = 8.47   # 1 - 0.5 (1 + tanh(z)) == 0.0 in fp32 for z >= 8.4616 (SURVEY A.2)

    def __init__(self, in_dim=32, latent_dim=64, args=None):
        super().__init__()
        self.in_dim, self.latent_dim = in_dim, latent_dim
        self.extra_edge_dim = args.extra_edge_dim
        self.extra_k_dim = args.extra_k_dim
        self.hard = args.dgg_hard
        self.deg_mean, self.deg_std = args.deg_mean, args.deg_std
        self.node_encode_for_edges = nn.Sequential(nn.Linear(in_dim, latent_dim), nn.LeakyReLU())
        self.edge_encode = nn.Sequential(
            nn.Linear(latent_dim * 2 + self.extra_edge_dim, latent_dim), nn.LeakyReLU(), nn.Linear(latent_dim, 1))
        self.t = nn.Parameter(torch.tensor(-0.1))
        self.edge_conv_phi = nn.Linear(latent_dim, latent_dim // 2)
        self.edge_conv_theta = nn.Linear(latent_dim, latent_dim // 2)
        self.edge_conv_encode = nn.Linear(latent_dim // 2, 1)
        self.edge_prob_net_mode = args.dgg_mode_edge_net
        self.input_degree_decode = nn.Linear(3, 1, bias=True)
        self.combine_input_degree = nn.Sequential(nn.Linear(latent_dim + 3, latent_dim), nn.LeakyReLU())
        self.adj_project = nn.Linear(1, 1)
        self.k_net_mode = args.dgg_mode_k_net
        self.signal_project = nn.Linear(256, 1, bias=True)
        self.input_degree_project = nn.Linear(1, 3, bias=True)
        self.node_encode_for_k = nn.Sequential(nn.Linear(in_dim, latent_dim), nn.LeakyReLU())
        self.k_embed = nn.Sequential(nn.Linear(latent_dim + self.extra_k_dim, latent_dim // 2), nn.LeakyReLU())
        self.k_W = nn.Parameter(torch.rand(latent_dim, latent_dim, requires_grad=True))
        if self.k_net_mode in ("input_deg", "learn_normalized_degree"):
            self.k_net = LearnableKEncoder(in_dim=3, latent_dim=latent_dim // 4, args=args)
        else:
            self.k_net = LearnableKEncoder(in_dim=latent_dim // 2, latent_dim=latent_dim // 4, args=args)
        self.k_select_mode = args.dgg_mode_k_select
        self.gumbel = torch.distributions.Gumbel(loc=torch.tensor(0.0), scale=torch.tensor(0.3))
        self.var_grads = {"edge_p": [], "first_k": [], "out_adj": []}
        self.args = args

    def hook(self, grad):
        return grad

    def normalize_adj(self, A_hat):
        if A_hat.is_sparse:
            g, v = CSRGraph.from_coo(A_hat)
            return g.to_coo(K.sym_normalize(v, g))
        row_sum = A_hat.sum(-1) ** -0.5
        return row_sum.unsqueeze(-1) * A_hat * row_sum.unsqueeze(0)

    # ------------------------------------------------------------------ forward
    def forward(self, x, in_adj, noise=True, writer=None, epoch=None):
        assert x.ndim == 2
        assert len(in_adj.shape) == 2
        graph, vals = CSRGraph.from_coo(in_adj)
        n = x.shape[-2]
        edge_p = self.edge_prob_net(graph, vals, x, mode=self.edge_prob_net_mode)         # [E]
        if self.args.debug_step == 0:
            return self.return_hard_or_soft(graph, edge_p)
        # k does not depend on the (perturbed) edge probabilities in any mode (dgm.py:1472-1586)
        k = self.k_estimate_net(n, graph, vals, x, edge_p, mode=self.k_net_mode)           # [N,1] or None
        pert = edge_p
        if self.args.perturb_edge_prob:
            if self.args.debug_step == 1 or self.k_select_mode not in ("k_times_edge_prob", "k_only"):
                raise NotImplementedError("perturb_edge_prob is covered for debug_step=3 with k_times_edge_prob / "
                                          "k_only")
            graph, vals, pert = self._perturb(graph, vals, edge_p, k, n)
        elif self.args.debug_step == 1:
            return self.return_hard_or_soft(graph, pert)
        out = self.select_top_k(graph, k, pert, mode=self.k_select_mode, writer=writer, epoch=epoch)
        if self.k_select_mode == "k_only" and not self.args.perturb_edge_prob:
            graph, vals, out = self._k_only_spill(graph, vals, out, k, n)
        if writer is not None:
            self.get_adj_diff_stats(graph, vals, out, k, writer=writer, epoch=epoch)
        # (detached: a module attribute that carries a grad_fn would keep the whole step's autograd graph -- and the
        # AccumulateGrad nodes of the stream it ran on -- alive into the next step, which breaks CUDA-graph capture)
        self.last_k = None if k is None else k.detach()
        return self.return_hard_or_soft(graph, out)

    # ------------------------------------------------------------------ Gumbel perturbation (dgm.py:1211-1229)
    def _sample_noise(self, n, device):
        """Dense [N,N] Gumbel(0, 0.3) noise laid out exactly like the reference: symmetric = n(n-1)/2 draws
        on triu_indices(n,n,1) mirrored, zero diagonal (1216-1223); asymmetric = one [1,N,N] draw (1226).
        ``self.gumbel`` stays the injection point (tests replace it with a fixed-tensor sampler)."""
        if self.args.symmetric_noise:
            G = torch.zeros(n, n, device=device)
            i, j = torch.triu_indices(n, n, 1, device=device)
            g = self.gumbel.sample([len(i)]).to(device)
            G[i, j] = g
            G[j, i] = g
            return G
        return self.gumbel.sample([1, n, n]).to(device).squeeze(0)

    def _perturb(self, graph, vals, edge_p, k, n):
        """pert = exp(log(P + 1e-8) + G) on ALL N^2 entries: off-support ones become 1e-8 e^G and are ranked
        by G (SURVEY A.2).  Only entries ranked inside the soft first-k window (r < k_i + 8.47) can be
        non-zero, so per row the union of its edges and its W = ceil(k_max + 8.47) + 1 best non-edges (by G) is
        exact: any excluded non-edge is out-ranked by W included ones.  The best non-edges come from the
        streaming top-K selector (all-pairs kernel with t = 0 and the edge positions masked to -inf)."""
        if k is None:
            raise TypeError("unsupported operand type(s) for -: 'Tensor' and 'NoneType'")     # dgm.py:1413
        dev = edge_p.device
        G = self._sample_noise(n, dev)
        idx = graph.coo_indices()
        g_edge = G[idx[0], idx[1]]
        pert_edge = torch.exp(torch.log(edge_p + 1e-8) + g_edge)                               # 1213-1229
        w = min(int(math.ceil(float(k.detach().max()) + self.TANH_WINDOW)) + 1, n)   # output size is data-dependent
        G[idx[0], idx[1]] = float("-inf")          # mask the edge positions in place (restored below): one N x N
        zero = torch.zeros(n, 32, device=dev)
        tz = torch.zeros(1, device=dev)
        sel, after = [], None
        for p0 in range(0, w, 64):                  # > 64 best non-edges per row: continuation passes
            si, sg = K.allpairs_topk(zero, tz, G, min(64, w - p0), 1, after=after)
            sel.append((si, sg))
            after = (sg[:, -1].contiguous(), si[:, -1].contiguous())
        sel_idx, sel_g = torch.cat([a for a, _ in sel], 1), torch.cat([b for _, b in sel], 1)
        G[idx[0], idx[1]] = g_edge
        keep = torch.isfinite(sel_g) & (sel_idx >= 0)
        rows = torch.arange(n, device=dev).reshape(n, 1).expand(n, w)[keep]
        cols = sel_idx[keep].long()
        pert_non = torch.exp(torch.log(torch.full_like(sel_g[keep], 1e-8)) + sel_g[keep])
        # union structure, coalesced order (row-major, columns ascending)
        key = torch.cat([idx[0] * n + idx[1], rows * n + cols])
        order = torch.argsort(key)
        key = key[order]
        u_idx = torch.stack([key // n, key % n])
        u_graph = CSRGraph.from_indices(u_idx, n)
        u_pert = torch.cat([pert_edge, pert_non])[order]
        u_vals = torch.cat([vals, torch.zeros_like(pert_non)])[order]
        return u_graph, u_vals, u_pert

    def return_hard_or_soft(self, graph, edge_vals, idxs=None, k=None, threshold=0.8):
        if self.hard:
            raise NotImplementedError("dgg_hard: the reference's hard branch scatters un-sorted values through "
                                      "sorted indices (SURVEY 2.3); it is fenced off, not reproduced")
        return graph.to_coo(edge_vals)

    def get_adj_diff_stats(self, graph, in_vals, out_vals, k=None, writer=None, epoch=None):
        """TensorBoard stats of dgm.py:1313-1350 on the stored entries (the reference builds ~8 dense N x N
        temporaries for them on every forward, even with writer=None).  ``graph`` is the structure of the OUTPUT
        (the union of the input edges and whatever off-support entries the perturbed / k_only modes added, where
        ``in_vals`` is 0): on-edge = in_adj > 0, off-edge = in_adj == 0 (1321-1328); an entry that is stored in
        neither matrix has difference 0 and is dropped by the reference's ``diff != 0`` filter as well."""
        diff = (in_vals - out_vals).detach()
        on, off = diff[in_vals > 0], diff[in_vals == 0]
        diff, off = on[on != 0], off[off != 0]
        if self.training and writer is not None:
            writer.add_scalar("train_stats/on_edge_mean", diff.mean(), epoch)
            writer.add_scalar("train_stats/on_edge_std", diff.std(), epoch)
            writer.add_scalar("train_stats/off_edge_mean", off.mean(), epoch)     # NaN when nothing is stored off
            writer.add_scalar("train_stats/off_edge_std", off.std(), epoch)       # the support, like the reference
            deg = K.row_sum(in_vals.detach(), graph)
            writer.add_scalar("train_stats/in_deg_mean", deg.mean(), epoch)
            if k is not None:
                writer.add_scalar("train_stats/k_diff_mean", (k.detach().flatten() - deg).mean(), epoch)
                writer.add_scalar("train_stats/k_mean", k.detach().mean(), epoch)

    # ------------------------------------------------------------------ top-k selector (dgm.py:1352-1435)
    def select_top_k(self, graph, k, pert_edge_p, mode="k_times_edge_prob", writer=None, epoch=None):
        if mode == "edge_p-cdf":
            # the reference scatters the *unweighted* sorted values back (dgm.py:1400): identity
            return pert_edge_p
        if mode in ("k_times_edge_prob", "k_only"):
            if k is None:
                raise TypeError("unsupported operand type(s) for -: 'Tensor' and 'NoneType'")  # dgm.py:1413, 1430
            if writer is not None and mode == "k_times_edge_prob":
                rs = K.row_sum(pert_edge_p.detach(), graph)                                    # dgm.py:1406-1408
                writer.add_scalar("values/edge_p_std", rs.std(), epoch)
                writer.add_scalar("values/edge_p_mean", rs.mean(), epoch)
            return K.row_firstk(pert_edge_p, k.reshape(-1), graph, k_only=(mode == "k_only"))
        raise NotImplementedError("dgg_mode_k_select=%r is not covered (see class docstring)" % (mode,))

    def _k_only_spill(self, graph, vals, out, k, n):
        """``k_only`` (dgm.py:1423-1435) gives every column of the dense row the weight fk(rank - k_i), not only the
        edges: a row whose window ceil(k_i + 8.47) is longer than its degree spills into its non-edges, which are
        exact zeros and therefore rank after all edges in the order the sort leaves them -- ascending column index
        for a stable sort (what the oracle pins; the reference's order among exact ties is unspecified).  Returns
        the union structure (edges + spilled columns, coalesced) with the input values (0 off the support) and
        the output values; gradients reach k through both parts."""
        kf = k.reshape(-1)
        deg = (graph.rowptr[1:] - graph.rowptr[:-1]).to(torch.int64)
        win = torch.ceil(kf.detach() + self.TANH_WINDOW).clamp(min=0, max=n).to(torch.int64)
        m = (win - deg).clamp(min=0)
        m = torch.minimum(m, n - deg)                             # non-edges a row can spill into
        if int(m.sum()) == 0:
            return graph, vals, out
        # the first m_i non-edges of row i lie among its first m_i + deg_i columns
        span = torch.where(m > 0, m + deg, torch.zeros_like(m))
        rows = torch.repeat_interleave(torch.arange(n, device=out.device), span)
        start = torch.cumsum(span, 0) - span
        cols = torch.arange(rows.numel(), device=out.device) - start[rows]
        eidx = graph.coo_indices()
        ekey = eidx[0] * n + eidx[1]
        ckey = rows * n + cols
        pos = torch.searchsorted(ekey, ckey).clamp(max=ekey.numel() - 1)
        non_edge = ekey[pos] != ckey
        order = torch.cumsum(non_edge.to(torch.int64), 0) - 1      # running count of non-edges ...
        first = torch.zeros(n, dtype=torch.int64, device=out.device)
        first[span > 0] = (order - non_edge.to(torch.int64) + 1)[start[span > 0]]
        order = order - first[rows]                               # ... restarted at every row
        keep = non_edge & (order < m[rows])
        rows, cols, order = rows[keep], cols[keep], order[keep]
        r = (deg[rows] + order).to(torch.float32)
        spill = 1 - 0.5 * (1 + torch.tanh(r - kf[rows]))          # dgm.py:1427-1431
        key = torch.cat([ekey, rows * n + cols])
        perm = torch.argsort(key)
        key = key[perm]
        u_graph = CSRGraph.from_indices(torch.stack([key // n, key % n]), n)
        u_out = torch.cat([out, spill])[perm]
        u_vals = torch.cat([vals, torch.zeros_like(spill)])[perm]
        return u_graph, u_vals, u_out

    # ------------------------------------------------------------------ degree estimator (dgm.py:1472-1586)
    def k_estimate_net(self, N, graph, vals, x, edge_p, mode="calculate"):
        if mode == "pass":
            return None
        in_deg = K.row_sum(vals, graph).reshape(-1, 1)                                     # [N,1]
        if mode == "learn_normalized_degree":
            mu, var = in_deg.mean(), in_deg.std()
            d = self.k_net(self.input_degree_project((in_deg - mu) / var))
            return F.relu(d * var + mu) + 1.0
        if mode == "input_deg":
            mu, var = self.deg_mean, self.deg_std
            d = self.k_net(self.input_degree_project((in_deg - mu) / (var + 1e-5)))
            return F.relu(d * var + mu) + 1.0
        if mode in ("gcn-x-deg", "x"):
            enc = self.node_encode_for_k
            xe = K.encoder_linear(x, enc[0].weight, enc[0].bias, enc[1].negative_slope)   # tensor cores, x padded once
            if mode == "gcn-x-deg":
                nv = K.sym_normalize(vals, graph)
                fused = K.spmm_gemm(nv, xe, self.k_W, graph, relu=True)                    # relu((A x) k_W), one launch
                xe = fused if fused is not None else torch.relu(K.spmm(nv, xe, graph) @ self.k_W)
            mu, var = in_deg.mean(), in_deg.std()
            # k_embed = Linear(h + 1, h / 2) + LeakyReLU on [x_e || normalised degree]: three zero columns make the
            # width a multiple of four (16-byte rows for the tensor-core forward and the split-K weight gradient)
            pad = (-(xe.shape[1] + 1)) % 4
            feats = torch.cat([xe, (in_deg - mu) / (var + 1e-5)] + ([xe.new_zeros(N, pad)] if pad else []), dim=-1)
            emb = self.k_embed[0]
            d = self.k_net(K.tall_linear(feats, F.pad(emb.weight, (0, pad)), emb.bias, self.k_embed[1].negative_slope))
            return F.relu(d * var + mu) + 1.0
        if mode == "calculate":
            return (in_deg / N) * 2 - 1
        raise Exception("mode not found")

    # ------------------------------------------------------------------ edge probabilities (dgm.py:1596-1727)
    def edge_prob_net(self, graph, vals, x, mode=None):
        """Per-edge probabilities [E] in CSR order.  The E x (2h + M) concat / gather / Linear / LeakyReLU / Linear /
        sigmoid chain of the reference becomes: node encoder (tensor cores), ONE tall GEMM for the per-node halves
        of the first Linear, one fused per-edge kernel (``K.edge_mlp``; see include/dggb.h for the algebra)."""
        if mode == "A_uv":
            return torch.sigmoid(self.adj_project(vals.unsqueeze(-1)).flatten())
        if mode not in ("u-v-dist", "u-v-A_uv", "u-v-deg", "u-v-deg-dist", "edge_conv"):
            raise Exception("mode not found")
        enc = self.node_encode_for_edges
        xe = K.encoder_linear(x, enc[0].weight, enc[0].bias, enc[1].negative_slope)      # dgm.py:1609
        h = xe.shape[1]
        if h % 4 != 0 or vals.requires_grad:
            return self._edge_prob_net_eager(graph, vals, xe, mode)
        if mode == "u-v-dist":
            return K.edge_dist_score(xe, graph, 0.05)                                      # dgm.py:1618-1623
        if mode == "edge_conv":                                                            # dgm.py:1703-1719
            wt, wp = self.edge_conv_theta, self.edge_conv_phi
            p_uv = K.tall_linear(xe, torch.cat([wp.weight - wt.weight, wt.weight], dim=0))
            return K.edge_mlp(p_uv, None, wt.bias + wp.bias, self.edge_conv_encode.weight,
                              self.edge_conv_encode.bias, graph, flags=0, slope=1.0)
        l1, act, l2 = self.edge_encode[0], self.edge_encode[1], self.edge_encode[2]
        p_uv = K.tall_linear(xe, torch.cat([l1.weight[:, :h], l1.weight[:, h:2 * h]], dim=0))
        wx = l1.weight[:, 2 * h:]
        if mode == "u-v-A_uv":
            return K.edge_mlp(p_uv, wx, l1.bias, l2.weight, l2.bias, graph, edge_val=vals, flags=K.EX_VAL,
                              slope=act.negative_slope)
        deg = K.row_sum(vals, graph)                                                       # raw degrees (1653)
        if mode == "u-v-deg":
            return K.edge_mlp(p_uv, wx, l1.bias, l2.weight, l2.bias, graph, deg=deg, flags=K.EX_DEG,
                              slope=act.negative_slope)
        return K.edge_mlp(p_uv, wx, l1.bias, l2.weight, l2.bias, graph, deg=deg, xe=xe, flags=K.EX_DEG | K.EX_DIST,
                          slope=act.negative_slope, dist_scale=1.0)                       # u-v-deg-dist (1671-1702)

    def _edge_prob_net_eager(self, graph, vals, xe, mode):
        """The same formulas as plain tensor ops: hidden widths that are not a multiple of 4, and input adjacencies
        whose VALUES carry gradients (``dgg_adj_input != "input_adj"``: the fused kernels treat the input graph
        as a constant)."""
        idx = graph.coo_indices()
        u, v = xe[idx[0]], xe[idx[1]]
        if mode == "u-v-dist":
            return torch.exp(-0.05 * torch.linalg.vector_norm(u - v, dim=-1, ord=2))
        if mode == "edge_conv":
            feat = self.edge_conv_theta(v - u) + self.edge_conv_phi(u)
            return torch.sigmoid(self.edge_conv_encode(feat).flatten())
        if mode == "u-v-A_uv":
            feat = torch.cat([u, v, vals.unsqueeze(-1)], dim=-1)
        else:
            deg = K.row_sum(vals, graph).reshape(-1, 1)                                    # raw degrees (1653)
            extra = [deg[idx[0]], deg[idx[1]]]
            if mode == "u-v-deg-dist":
                extra.append(torch.exp(-1.0 * torch.linalg.vector_norm(u - v, dim=-1, ord=2)).unsqueeze(-1))
            feat = torch.cat([u, v] + extra, dim=-1)
        return torch.sigmoid(self.edge_encode(feat).flatten())
