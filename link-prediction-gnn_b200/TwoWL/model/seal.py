"""SEAL's DGCNN (Zhang & Chen 2018), as PyTorch Geometric's examples/seal_link_pred.py builds it, on this package's kernels.

    GCNConv(max_z + 1 + F, hidden) -> (num_layers - 1) x GCNConv(hidden, hidden) -> GCNConv(hidden, 1), each followed by tanh;
    the tanh outputs concatenated (D = hidden * num_layers + 1 channels), SortPooling to k rows per subgraph;
    Conv1d(1, 16, D, D), ReLU, MaxPool1d(2, 2); Conv1d(16, 32, 5), ReLU; flatten channel-major;
    Linear(dense_dim, 128), ReLU, Dropout(dropout), Linear(128, 1).

The input of a node is [one_hot(z, max_z + 1) | node_feat[node]] (node_feat optional, e.g. node2vec embeddings). Parameters keep
torch's shapes and PyG's names (convs.i.lin.weight, convs.i.bias, conv1.weight [16, 1, D], conv2.weight [32, 16, 5],
mlp.lins.{0,1}.{weight,bias}), so a float64 restatement built from torch.nn.Conv1d and PyG's GCNConv loads the same state_dict.

How the arithmetic maps onto kernels:
  * the first layer's product with one_hot(z) is a column gather of its weight (twowl::seal_input), its weight gradient a
    segmented sum over the nodes grouped by label;
  * Conv1d(1, 16, D, D) is a linear map of the [B k, D] SortPooling rows; Conv1d(16, 32, 5) a linear map of im2col windows;
    the convolution outputs stay position-major ([B, L, C]), so the first Linear reads its weight with the columns permuted
    to that order;
  * widths the tensor kernels do not take (the 1-channel GCNConv, the concatenated D, the 1-output Linear) are zero-padded to a
    multiple of 4; the padding carries zeros forward and zero gradients back.

Labels above max_z are clipped to max_z. PyG sizes max_z over every split before training; here it comes from the training
subgraphs (train.seal_fit), and an evaluation subgraph may hold a larger label.
"""
from __future__ import annotations

import math

import torch
from torch import nn

from TwoWL.model.model import GCNConv
from twowl_b200 import functional as F2
from twowl_b200 import graph as G
from twowl_b200 import ops


def sort_pool_k(sizes: torch.Tensor, ratio: float = 0.6) -> int:
    """PyG's SortPooling k from the training subgraphs' node counts: max(10, the ceil(ratio n)-th smallest)."""
    s = torch.sort(sizes.reshape(-1).cpu()).values
    if s.numel() == 0:
        return 10
    return max(10, int(s[int(math.ceil(ratio * s.numel())) - 1]))


def _al(t: torch.Tensor) -> torch.Tensor:
    """t itself, or a copy when its storage is not 16-byte aligned (a parameter inside an optimiser's flat buffer): the vectorised
    kernels read 16-byte rows. Gradients flow back through the copy."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _pad_rows(w: torch.Tensor, rows: int) -> torch.Tensor:
    return w if w.shape[0] == rows else torch.cat((w, w.new_zeros((rows - w.shape[0],) + tuple(w.shape[1:]))))


def _pad_cols(w: torch.Tensor, cols: int) -> torch.Tensor:
    return w if w.shape[1] == cols else torch.cat((w, w.new_zeros((w.shape[0], cols - w.shape[1]))), dim=1)


class _MLP(nn.Module):
    """The parameter layout of PyG's MLP([dense_dim, 128, 1], norm=None): lins.0, lins.1."""

    def __init__(self, dims):
        super().__init__()
        self.lins = nn.ModuleList([nn.Linear(a, b) for a, b in zip(dims[:-1], dims[1:])])


class DGCNN(nn.Module):
    def __init__(self, max_z: int, k: int, hidden: int = 32, num_layers: int = 3, node_feat_dim: int = 0, dropout: float = 0.5):
        super().__init__()
        if hidden % 4 or hidden < 4:
            raise ValueError(f"DGCNN: hidden must be a positive multiple of 4, got {hidden}")
        if num_layers < 1 or k < 10 or max_z < 1:
            raise ValueError(f"DGCNN: needs num_layers >= 1, k >= 10 and max_z >= 1 (got {num_layers}, {k}, {max_z})")
        self.max_z, self.k, self.hidden, self.node_feat_dim, self.dropout = int(max_z), int(k), hidden, int(node_feat_dim), dropout
        self.convs = nn.ModuleList([GCNConv(self.max_z + 1 + self.node_feat_dim, hidden)] +
                                   [GCNConv(hidden, hidden) for _ in range(num_layers - 1)] + [GCNConv(hidden, 1)])
        self.D = hidden * num_layers + 1
        self.Dp = self.D + 3                  # a multiple of 4: the last GCNConv runs 4 wide, its 3 padding columns stay zero
        self.conv1 = nn.Conv1d(1, 16, self.D, self.D)
        self.conv2 = nn.Conv1d(16, 32, 5, 1)
        self.L1 = self.k // 2                 # after MaxPool1d(2, 2)
        self.L2 = self.L1 - 4                 # after conv2
        self.mlp = _MLP([32 * self.L2, 128, 1])

    def forward(self, sub: ops.SealBatch, node_feat: torch.Tensor = None, seed: int = 0) -> torch.Tensor:
        """Logits fp32 [B, 1] of the batch's subgraphs (ops.seal_subgraphs). node_feat [N, F] is read at the subgraphs' nodes.
        seed draws the dropout mask when training (the same seed gives the same bits)."""
        if (node_feat is None) != (self.node_feat_dim == 0):
            raise ValueError("DGCNN: pass node_feat exactly when the model was built with node_feat_dim > 0")
        n, B = sub.nodes.numel(), sub.num_graphs
        ei = sub.edge_index
        g = G.node_graph(ei, n)
        z = sub.z.to(torch.int64).clamp_(0, self.max_z)
        feat = None
        if node_feat is not None:     # gathered 4 wide (the row kernels' width), the padding columns cut off again
            F = node_feat.shape[1]
            feat = ops.gather_rows(F2._pad4(node_feat), sub.nodes)[:, :F]
        hs = []
        for i, conv in enumerate(self.convs):
            last = i == len(self.convs) - 1
            if i == 0:
                zl = F2.seal_input(conv.lin.weight, z, feat)
            else:
                zl = F2.linear(t, _pad_rows(conv.lin.weight, 4) if last else _al(conv.lin.weight))
            bias = _pad_rows(conv.bias, 4) if last else _al(conv.bias)
            h = F2.gcn_aggregate(zl, bias, g.dinv, g.ptr, g.col, g.plan, g.tptr, g.tcol, g.tplan, None, 0, 0, g.emask, g.temask)
            hs.append(h)
            if not last:
                t = F2.seal_tanh(h)
        offs = [self.hidden * i for i in range(len(hs))]
        X = F2.seal_tanh_concat(hs, offs, self.Dp)
        S, _ = F2.sort_pool(X, sub.node_ptr, self.k, self.D - 1)
        y1 = F2.linear(S.reshape(B * self.k, self.Dp), _pad_cols(self.conv1.weight.reshape(16, self.D), self.Dp))
        p1 = F2.bias_act(y1, self.conv1.bias, B, 2, True, 0.0, 0)                      # [B L1, 16]
        y2 = F2.linear(F2.im2col(p1, B, 5), _al(self.conv2.weight.reshape(32, 16 * 5)))    # [B L2, 32]
        f = F2.bias_act(y2, self.conv2.bias, B, 1, True, 0.0, 0).reshape(B, self.L2 * 32)
        lin0, lin1 = self.mlp.lins
        w0 = _al(lin0.weight.reshape(128, 32, self.L2).transpose(1, 2).reshape(128, self.L2 * 32))   # channel- to position-major
        p = self.dropout if (self.training and self.dropout > 0.0) else 0.0
        h = F2.bias_act(F2.linear(f, w0), lin0.bias, B, 1, True, p, int(seed) if p > 0.0 else 0)
        out = F2.bias_act(F2.linear(h, _pad_rows(lin1.weight, 4)), _pad_rows(lin1.bias, 4), B, 1, False, 0.0, 0)
        return out[:, :1]
