"""BUDDY (Chamberlain et al., "Graph Neural Networks for Link Prediction with Subgraph Sketching", ICLR 2023): the pair predictor
over subgraph-sketch features, on this package's kernels.

    sf     = ops.sketch_features(sk, u, v)                        [B, k² + 2k]: A(d1, d2), B_u(d), B_v(d) for d ≤ k = hops
    s      = Drop(ReLU(BN(W_l sf + b_l)))                          BUDDY's label_lin_layer, bn_labels
    xʰ     = Âʰ X,  h = 0 .. k                                     optional node features X [N, F], Â = D^-1/2 (A + I) D^-1/2
                                                                    over the encoder graph (GCN normalisation, nothing learned)
    f      = Drop(ReLU(W_f [x⁰_u ⊙ x⁰_v | … | xᵏ_u ⊙ xᵏ_v] + b_f))   node_feat_dim > 0 only
    logit  = w_o · [s | f] + b_o

BN is BatchNorm1d. In training it normalises with the batch's mean and biased variance, which is GraphNorm with mean_scale fixed
at 1 (F2.graphnorm_act, with ReLU and dropout fused); the (mean, inv_std) it returns update running_mean / running_var as torch
does (momentum 0.1, unbiased variance). In eval it applies the running statistics (ops.graphnorm_apply). BUDDY's RA, degree and
learnable-embedding inputs are not built, and the node features enter as SIGN-style propagated hops rather than through a learned
per-node layer.

Parameters and buffers (torch shapes, so a float64 restatement loads the same state_dict; D = k² + 2k):
    label_lin_layer.{weight [D, D], bias [D]}
    bn_labels.{weight, bias, running_mean, running_var [D], num_batches_tracked}
    lin_feat.{weight [hidden, (k + 1) F], bias [hidden]}         node_feat_dim = F > 0 only; column block h reads xʰ_u ⊙ xʰ_v
    lin.{weight [1, D (+ hidden)], bias [1]}

Widths are padded to multiples of 4 inside the forward (zero rows and columns add nothing); every product is F2.linear, every bias
+ ReLU + dropout F2.bias_act, the endpoint products F2.batch_pair_init and the propagation F2.gcn_aggregate. Dropout masks are
hashes of (seed, site, element), so a seed gives the same bits every time.
"""
from __future__ import annotations

import torch
from torch import nn

from TwoWL.model.ncn import _site_seed
from TwoWL.model.seal import _al, _pad_cols, _pad_rows
from twowl_b200 import functional as F2
from twowl_b200 import graph as G
from twowl_b200 import ops


def _up4(n: int) -> int:
    return (n + 3) // 4 * 4


class BUDDY(nn.Module):
    def __init__(self, hops: int = 2, dropout: float = 0.5, node_feat_dim: int = 0, hidden: int = 32):
        super().__init__()
        if not 1 <= hops <= ops.SKETCH_MAX_HOPS:
            raise ValueError(f"BUDDY: hops = {hops} outside [1, {ops.SKETCH_MAX_HOPS}]")
        if hidden % 4 or hidden < 4:
            raise ValueError(f"BUDDY: hidden must be a positive multiple of 4, got {hidden}")
        self.hops, self.dropout, self.hidden, self.node_feat_dim = int(hops), float(dropout), int(hidden), int(node_feat_dim)
        self.dim = self.hops * self.hops + 2 * self.hops
        self.label_lin_layer = nn.Linear(self.dim, self.dim)
        self.bn_labels = nn.BatchNorm1d(self.dim)
        if self.node_feat_dim:
            self.lin_feat = nn.Linear((self.hops + 1) * self.node_feat_dim, hidden)
        self.lin = nn.Linear(self.dim + (hidden if self.node_feat_dim else 0), 1)
        self.sketch_args = dict(num_perm=128, hll_p=8, seed=0)   # the ops.link_sketches settings scores are read with (train.buddy_fit)

    def _p(self) -> float:
        return self.dropout if (self.training and self.dropout > 0.0) else 0.0

    @torch.no_grad()
    def propagate(self, node_feat: torch.Tensor, edge_index) -> list:
        """[X, ÂX, …, ÂᵏX] (fp32 [N, F padded to a multiple of 4] each) over edge_index (int64 [2, E], e.g. a sample_block
        result): the feature branch's input."""
        if node_feat.shape[1] != self.node_feat_dim or not self.node_feat_dim:
            raise ValueError(f"BUDDY: node_feat must be [N, {self.node_feat_dim}] (the model's node_feat_dim)")
        N = node_feat.shape[0]
        g = G.node_graph(edge_index, N)
        x = F2._pad4(node_feat.float())
        zero = x.new_zeros(x.shape[1])
        xs = [x]
        for _ in range(self.hops):
            x = F2.gcn_aggregate(x, zero, g.dinv, g.ptr, g.col, g.plan, g.tptr, g.tcol, g.tplan, None, 0, 0, g.emask, g.temask)
            xs.append(x)
        return xs

    def _bn_train(self, z: torch.Tensor, gamma, beta, p: float, seed: int) -> torch.Tensor:
        bn = self.bn_labels
        C, B = z.shape[1], z.shape[0]
        if B < 2:
            raise ValueError("BUDDY: training-mode BatchNorm needs more than one pair per batch")
        out, stats = F2.graphnorm_act(z, gamma, beta, z.new_ones(C), None, bn.eps, p, seed, True)
        if bn.track_running_stats:
            with torch.no_grad():
                mean, inv_std = stats[:self.dim].double(), stats[C:C + self.dim].double()
                var = (1.0 / (inv_std * inv_std) - bn.eps) * (B / (B - 1))
                bn.running_mean.mul_(1 - bn.momentum).add_((bn.momentum * mean).to(bn.running_mean.dtype))
                bn.running_var.mul_(1 - bn.momentum).add_((bn.momentum * var).to(bn.running_var.dtype))
                bn.num_batches_tracked.add_(1)
        return out

    def _bn_eval(self, z: torch.Tensor, gamma, beta) -> torch.Tensor:
        bn, C = self.bn_labels, z.shape[1]
        mean = _pad_rows(bn.running_mean.float(), C)
        inv_std = _pad_rows((bn.running_var.double() + bn.eps).rsqrt().float(), C)
        return ops.graphnorm_apply(z.contiguous(), torch.cat((mean, inv_std)), gamma.detach().contiguous(), beta.detach().contiguous(),
                                   z.new_ones(C), 0.0, 0, True)

    def forward(self, sf: torch.Tensor, pairs: torch.Tensor = None, xs: list = None, seed: int = 0) -> torch.Tensor:
        """Logits fp32 [B, 1] of B pairs from their sketch features sf (fp32 [B, k² + 2k], ops.sketch_features); with node features,
        also the pairs (int64 [B, 2]) and xs = propagate(node_feat, edge_index). seed draws the dropout masks when training. Eval
        mode (running statistics) computes no gradient."""
        if (xs is None) != (self.node_feat_dim == 0):
            raise ValueError("BUDDY: pass pairs and xs = propagate(...) exactly when the model was built with node_feat_dim > 0")
        if sf.dim() != 2 or sf.shape[1] != self.dim:
            raise ValueError(f"BUDDY: sf must be [B, {self.dim}] (ops.sketch_features with hops = {self.hops})")
        B, D4 = sf.shape[0], _up4(self.dim)
        p = self._p()
        sd = (lambda site: _site_seed(seed, site) if p > 0.0 else 0)
        lw = self.label_lin_layer.weight
        z = F2.linear(F2._pad4(sf), _al(_pad_cols(_pad_rows(lw, D4), D4)))
        z = F2.bias_act(z, _pad_rows(self.label_lin_layer.bias, D4), B, 1, False, 0.0, 0)
        gamma, beta = _al(_pad_rows(self.bn_labels.weight, D4)), _al(_pad_rows(self.bn_labels.bias, D4))
        s = self._bn_train(z, gamma, beta, p, sd(0)) if self.training else self._bn_eval(z, gamma, beta)
        wo = self.lin.weight
        parts, wparts = [s], [_pad_cols(wo[:, :self.dim], D4)]
        if self.node_feat_dim:
            F4 = xs[0].shape[1]
            h = torch.cat([F2.batch_pair_init(x, pairs) for x in xs], dim=1)
            wf = self.lin_feat.weight.reshape(self.hidden, self.hops + 1, self.node_feat_dim)
            wf = _pad_cols(wf.reshape(-1, self.node_feat_dim), F4).reshape(self.hidden, (self.hops + 1) * F4)
            parts.append(F2.bias_act(F2.linear(h, _al(wf)), self.lin_feat.bias, B, 1, True, p, sd(1)))
            wparts.append(wo[:, self.dim:])
        x = torch.cat(parts, dim=1) if len(parts) > 1 else s
        out = F2.bias_act(F2.linear(x, _pad_rows(torch.cat(wparts, dim=1), 4)), _pad_rows(self.lin.bias, 4), B, 1, False, 0.0, 0)
        return out[:, :1]
