"""NCN, Neural Common Neighbor (Wang, Yang & Zhang, ICLR 2024), and its ablation without the common-neighbour term (the plain
GCN + MLP-decoder link predictor), on this package's kernels.

    h⁰    = Emb(min(x, max_x))                                 x: each node's degree (TwoWL's input, F2.embedding), or
          = node_feat padded to a multiple of 4 columns          node_feat [N, F] when given (as DGCNN pads it)
    hˡ    = GCNConv(hˡ⁻¹)                                      l = 1 .. num_layers, PyG semantics (add_remaining_self_loops,
                                                                symmetric normalisation, bias); ReLU + dropout after every
                                                                layer but the last; h = h^num_layers
    x_ij  = h_i ⊙ h_j                                          for a query pair (i, j)
    x_cn  = Σ_{w ∈ CN(i, j)} h_w                                CN over the adjacency the caller chose (ops.common_neighbors)
    r_ij  = Drop(ReLU(W_ij x_ij + b_ij))
    r_cn  = Drop(ReLU(W_cn x_cn + b_cn))
    z     = Drop(ReLU(W_h [r_ij | r_cn] + b_h))
    logit = w_o · z + b_o

NCN's predictor is MLP_ij(x_ij) + β · MLP_cn(x_cn), then an output MLP. Here the last linear maps of the two branch MLPs and their
sum are one Linear over the concatenation [r_ij | r_cn] (W_h [r_ij | r_cn] = W_h,ij r_ij + W_h,cn r_cn), and the learnable β is
absorbed into W_h's r_cn columns. With cn=False the r_cn branch is gone and z = Drop(ReLU(W_h r_ij + b_h)): the GCN + MLP-decoder
baseline.

Parameters (torch shapes, so a float64 restatement loads the same state_dict):
    emb.weight [max_x + 1, hidden]                             without node_feat
    convs.{l}.lin.weight [hidden, in], convs.{l}.bias [hidden]   in = hidden, or F for the first layer with node_feat
    lin_ij.{weight [hidden, hidden], bias}
    lin_cn.{weight [hidden, hidden], bias}                     cn=True only
    lin_h.{weight [hidden, 2 hidden] (hidden with cn=False), bias}
    lin_o.{weight [1, hidden], bias [1]}

Every product is F2.linear (tcgen05 split-tf32), every bias + ReLU + dropout F2.bias_act, the aggregation F2.gcn_aggregate, the
pair terms F2.pair_init and F2.cn_aggregate; their backward passes are the package's kernels too. Dropout masks are hashes of
(seed, site, element), so a seed gives the same bits every time.
"""
from __future__ import annotations

import torch
from torch import nn

from TwoWL.model.model import GCNConv
from TwoWL.model.seal import _al, _pad_cols, _pad_rows
from twowl_b200 import functional as F2
from twowl_b200 import graph as G
from twowl_b200 import ops


def _site_seed(seed: int, site: int) -> int:
    """The dropout seed of one dropout site: distinct sites of one step draw independent masks."""
    return (int(seed) * 64 + site) % (2 ** 62)


class NCN(nn.Module):
    def __init__(self, max_x: int, hidden: int = 64, num_layers: int = 2, dropout: float = 0.3, cn: bool = True,
                 node_feat_dim: int = 0):
        super().__init__()
        if hidden % 4 or hidden < 4:
            raise ValueError(f"NCN: hidden must be a positive multiple of 4, got {hidden}")
        if num_layers < 1 or max_x < 0:
            raise ValueError(f"NCN: needs num_layers >= 1 and max_x >= 0 (got {num_layers}, {max_x})")
        self.max_x, self.hidden, self.dropout, self.cn = int(max_x), hidden, float(dropout), bool(cn)
        self.node_feat_dim = int(node_feat_dim)
        if self.node_feat_dim == 0:
            self.emb = nn.Embedding(self.max_x + 1, hidden)
        in0 = self.node_feat_dim or hidden
        self.convs = nn.ModuleList([GCNConv(in0 if i == 0 else hidden, hidden) for i in range(num_layers)])
        self.lin_ij = nn.Linear(hidden, hidden)
        if self.cn:
            self.lin_cn = nn.Linear(hidden, hidden)
        self.lin_h = nn.Linear(2 * hidden if self.cn else hidden, hidden)
        self.lin_o = nn.Linear(hidden, 1)

    def _p(self) -> float:
        return self.dropout if (self.training and self.dropout > 0.0) else 0.0

    def encode(self, x: torch.Tensor, edge_index, node_feat: torch.Tensor = None, seed: int = 0) -> torch.Tensor:
        """Node embeddings h fp32 [N, hidden]. x: int64 [N] degrees (read without node_feat); edge_index: int64 [2, E], e.g. a
        sample_block result."""
        if (node_feat is None) != (self.node_feat_dim == 0):
            raise ValueError("NCN: pass node_feat exactly when the model was built with node_feat_dim > 0")
        p = self._p()
        if node_feat is None:
            t = F2.embedding(self.emb.weight, x.reshape(-1).to(torch.int64).clamp(0, self.max_x))
            N = t.shape[0]
        else:
            N = node_feat.shape[0]
        g = G.node_graph(edge_index, N)
        last = len(self.convs) - 1
        for i, conv in enumerate(self.convs):
            if i == 0 and node_feat is not None:
                xin = F2._pad4(node_feat)
                z = F2.linear(xin, _pad_cols(conv.lin.weight, xin.shape[1]))
            else:
                z = F2.linear(t, _al(conv.lin.weight))
            if i == last:
                t = F2.gcn_aggregate(z, _al(conv.bias), g.dinv, g.ptr, g.col, g.plan, g.tptr, g.tcol, g.tplan, None, 0, 0, g.emask,
                                     g.temask)
            else:   # the bias joins ReLU + dropout in one pass
                a = F2.gcn_aggregate(z, z.new_zeros(self.hidden), g.dinv, g.ptr, g.col, g.plan, g.tptr, g.tcol, g.tplan, None, 0, 0,
                                     g.emask, g.temask)
                t = F2.bias_act(a, conv.bias, N, 1, True, p, _site_seed(seed, i) if p > 0.0 else 0)
        return t

    def predict(self, h: torch.Tensor, pairs: torch.Tensor, cn=None, seed: int = 0) -> torch.Tensor:
        """Logits fp32 [B, 1] of the pairs (int64 [B, 2]) from node embeddings h (encode). cn: their ops.CommonNeighbors (cn=True)."""
        B = pairs.shape[0]
        p = self._p()
        sd = (lambda site: _site_seed(seed, site) if p > 0.0 else 0)
        L = len(self.convs)
        r = F2.bias_act(F2.linear(F2.batch_pair_init(h, pairs), _al(self.lin_ij.weight)), self.lin_ij.bias, B, 1, True, p, sd(L))
        if self.cn:
            if cn is None or cn.num_pairs != B:
                raise ValueError("NCN: cn must be the ops.CommonNeighbors of the batch's pairs")
            rc = F2.bias_act(F2.linear(F2.cn_aggregate(h, cn), _al(self.lin_cn.weight)), self.lin_cn.bias, B, 1, True, p, sd(L + 1))
            r = torch.cat((r, rc), dim=1)
        z = F2.bias_act(F2.linear(r, _al(self.lin_h.weight)), self.lin_h.bias, B, 1, True, p, sd(L + 2))
        out = F2.bias_act(F2.linear(z, _pad_rows(self.lin_o.weight, 4)), _pad_rows(self.lin_o.bias, 4), B, 1, False, 0.0, 0)
        return out[:, :1]

    def forward(self, x: torch.Tensor, edge_index, pairs: torch.Tensor, cn=None, node_feat: torch.Tensor = None,
                seed: int = 0) -> torch.Tensor:
        """Logits fp32 [B, 1]: encode over edge_index, then predict the pairs with their common neighbours cn (ops.common_neighbors,
        over whichever adjacency the caller masked). seed draws the dropout masks when training."""
        return self.predict(self.encode(x, edge_index, node_feat, seed), pairs, cn, seed)
