"""Drop-in for the reference's TwoWL/operators/datasets.py (dataset, BaseGraph, load_dataset, load,
do_edge_split - datasets.py:9-206). Tensor layouts are the reference's: ``edge_indexs[s]`` int64 [2,E_s]
doubled edges, ``pos1s[s]`` int64 [R_s,2] = [edges ; prediction pairs], ``ys[s]`` fp32 [P_s,1],
``ei2s[s]`` the wedge index of split s. preprocess / setPosDegreeFeature run on the CUDA operators of
TwoWL.utils; the graph tensors must therefore be on a CUDA device before preprocess() (``bg.to(device)``).
"""
from __future__ import annotations

import os

import torch

from TwoWL.utils import *  # noqa: F401,F403
from TwoWL.utils import degree, double, get_ei2, get_ei2_implicit, random_split_edges

PATH_CSV_EDGES = os.environ.get("TWOWL_CSV_EDGES", "raw_data/fb-pages-food/fb-pages-food.csv")  # constant.py:7


class dataset:
    def __init__(self, x, na, ei, ea, pos1, y, ei2):
        self.x = x
        self.na = na
        self.ei = ei
        self.ea = ea
        self.pos1 = pos1
        self.y = y
        self.ei2 = ei2


class BaseGraph:
    def __init__(self, x, node_attr, edge_pos, edge_neg, num_pos, num_neg, pattern):
        self.x = x
        self.node_attr = node_attr
        self.edge_pos = edge_pos
        self.edge_neg = edge_neg
        self.num_pos = num_pos
        self.num_neg = num_neg
        self.num_nodes = x.shape[0]
        self.max_x = None
        self.pattern = pattern
        # extension: '2wl_l' materialises ei2 like the reference; '2wl_l_implicit' keeps WedgeIndex objects
        self.implicit = pattern == "2wl_l_implicit"

    def toString(self):
        return (f"BaseGraph object:\n - x: {self.x}\n - node_attr: {self.node_attr}\n - edge_pos: {self.edge_pos}\n"
                f" - edge_neg: {self.edge_neg}\n - num_pos: {self.num_pos}\n - num_neg: {self.num_neg}\n"
                f" - num_nodes: {self.num_nodes}\n - max_x: {self.max_x}\n - pattern: {self.pattern}")

    def preprocess(self):
        """datasets.py:44-101."""
        npos = [int(v) for v in self.num_pos]
        nneg = [int(v) for v in self.num_neg]
        ep, en = self.edge_pos, self.edge_neg
        self.edge_indexs = [ep[:, :npos[0]], ep[:, :npos[0]], ep[:, :npos[0] + npos[1]]]
        self.edge_attrs = [torch.ones_like(self.edge_indexs[i][0], dtype=torch.float) for i in range(3)]
        pos_edges = [ep[:, :npos[0]], ep[:, npos[0]:npos[0] + npos[1]], ep[:, ep.shape[1] - npos[2]:]]
        neg_edges = [en[:, :nneg[0]], en[:, nneg[0]:nneg[0] + nneg[1]], en[:, en.shape[1] - nneg[2]:]]
        pred_edges = [neg_edges[0]] + [torch.cat((pos_edges[i], neg_edges[i]), dim=1) for i in range(1, 3)]
        self.pos1s = [torch.cat((self.edge_indexs[i].t(), pred_edges[i].t()), dim=0) for i in range(3)]
        dev = ep.device
        self.ys = [torch.zeros((neg_edges[0].shape[1], 1), device=dev)] + [
            torch.cat((torch.ones((pos_edges[i].shape[1], 1), dtype=torch.float, device=dev),
                       torch.zeros((neg_edges[i].shape[1], 1), dtype=torch.float, device=dev)))
            for i in range(1, 3)]
        if self.pattern in ("2wl_l", "2wl_l_implicit"):
            build = get_ei2_implicit if self.implicit else get_ei2
            self.ei2s = [build(self.num_nodes, self.edge_indexs[i], pred_edges[i]) for i in range(3)]
        else:
            self.ei2s = [None for _ in range(3)]

    def split(self, split: int):
        return (self.x[split], self.node_attr, self.edge_indexs[split], self.edge_attrs[split], self.pos1s[split],
                self.ys[split], self.ei2s[split])

    def setPosDegreeFeature(self):
        """datasets.py:107-114 - train/val use the train graph's degree, test uses the val graph's."""
        self.x = ([degree(self.edge_indexs[0], self.num_nodes) for _ in range(0, 2)]
                  + [degree(self.edge_indexs[1], self.num_nodes) for _ in range(2, 3)])
        self.max_x = max([torch.max(_).item() for _ in self.x])

    def to(self, device):
        self.x = self.x.to(device)
        self.edge_pos = self.edge_pos.to(device)
        self.edge_neg = self.edge_neg.to(device)
        return self


def ranking_dataset(bg: BaseGraph, split: int, num_neg: int, seed=0, pattern=None):
    """An evaluation table for ranking metrics (extension: OGB's ogbl-citation2 protocol, filtered): split s's P undirected
    positive pairs (u, v) - the even columns of its doubled positive block, as preprocess slices it - each followed in the table by
    num_neg negatives (u, w) drawn by ops.sample_tail_negatives, w uniform over the nodes that are neither u nor a positive
    partner of u in ANY split (bg.edge_pos). On the conventions of preprocess / split(s): x = bg.x[s] (setPosDegreeFeature must have
    run), ei = bg.edge_indexs[s], pos1 = [ei.T ; double([positives ; negatives in row-major order]).T], y = 1 for the 2P positive
    rows and 0 for the 2 P num_neg negative rows, ei2 the wedge index of that table (`pattern` as BaseGraph's, default bg.pattern).
    The returned dataset carries rank_k = num_neg; TwoWL.model.train.test_ranking reads its logits as [P positives | P x num_neg]
    negatives. split must be 1 (validation) or 2 (test): the training split's positives are edges of its own graph."""
    from twowl_b200 import ops
    s, k = int(split), int(num_neg)
    if s not in (1, 2):
        raise ValueError(f"ranking_dataset: split must be 1 (validation) or 2 (test), got {split}")
    if k < 1:
        raise ValueError(f"ranking_dataset: num_neg must be >= 1, got {num_neg}")
    if not hasattr(bg, "edge_indexs") or not isinstance(bg.x, (list, tuple)):
        raise ValueError("ranking_dataset: run bg.preprocess() and bg.setPosDegreeFeature() first")
    npos = [int(v) for v in bg.num_pos]
    ep = bg.edge_pos
    block = ep[:, npos[0]:npos[0] + npos[1]] if s == 1 else ep[:, ep.shape[1] - npos[2]:]
    pos = block[:, 0::2]                                            # (u, v) once per undirected pair
    u = pos[0].contiguous()
    w = ops.sample_tail_negatives(ep[0], ep[1], bg.num_nodes, u, k, seed=seed)
    neg = torch.stack((u.repeat_interleave(k), w.reshape(-1)))
    dev = ep.device
    y = torch.cat((torch.ones((2 * pos.shape[1], 1), dtype=torch.float, device=dev),
                   torch.zeros((2 * neg.shape[1], 1), dtype=torch.float, device=dev)))
    ds = _eval_table(bg, s, torch.cat((pos, neg), dim=1), y, pattern)
    ds.rank_k = k
    return ds


def _eval_table(bg: BaseGraph, s: int, pairs, y, pattern):
    """The evaluation dataset of split s's graph with the prediction pairs `pairs` ([2, P], one column per undirected pair):
    x = bg.x[s], ei = bg.edge_indexs[s], pos1 = [ei.T ; double(pairs).T], labels y ([2P, 1]), ei2 the wedge index of that
    table for `pattern` (default bg.pattern)."""
    pred = double(pairs)
    ei = bg.edge_indexs[s]
    pos1 = torch.cat((ei.t(), pred.t()), dim=0)
    pattern = bg.pattern if pattern is None else pattern
    if pattern in ("2wl_l", "2wl_l_implicit"):
        ei2 = (get_ei2_implicit if pattern == "2wl_l_implicit" else get_ei2)(bg.num_nodes, ei, pred)
    else:
        ei2 = None
    return dataset(bg.x[s], bg.node_attr, ei, bg.edge_attrs[s], pos1, y, ei2)


def candidate_dataset(bg: BaseGraph, split: int, src, ids, pattern=None):
    """An evaluation table of recommended links (extension: the re-ranking half of link recommendation): the prediction pairs
    are the valid (src[i], ids[i, j]) of TwoWL.model.train.recommend (ids >= 0), in row-major order, each doubled as preprocess
    doubles them, on split s's graph and conventions (x = bg.x[s], ei = bg.edge_indexs[s], ei2 for `pattern`, default
    bg.pattern) - the layout ranking_dataset builds. y is all zeros: there are no labels. The dataset carries cand_ids (ids) and
    cand_mask ([Q, k] bool, the valid entries); TwoWL.model.train.rerank scores it. split may be 0, 1 or 2."""
    s = int(split)
    if s not in (0, 1, 2):
        raise ValueError(f"candidate_dataset: split must be 0, 1 or 2, got {split}")
    if not hasattr(bg, "edge_indexs") or not isinstance(bg.x, (list, tuple)):
        raise ValueError("candidate_dataset: run bg.preprocess() and bg.setPosDegreeFeature() first")
    src = src.reshape(-1).to(torch.int64)
    if ids.dim() != 2 or ids.shape[0] != src.numel():
        raise ValueError(f"candidate_dataset: ids must be [Q, k] with Q = {src.numel()} sources, got {tuple(ids.shape)}")
    mask = ids >= 0
    pairs = torch.stack((src.unsqueeze(1).expand_as(ids)[mask], ids[mask]))
    y = torch.zeros((2 * pairs.shape[1], 1), dtype=torch.float, device=ids.device)
    ds = _eval_table(bg, s, pairs, y, pattern)
    ds.cand_ids, ds.cand_mask = ids, mask
    return ds


class _Data:
    """Stand-in for torch_geometric.data.Data(edge_index=...) as used by load() (datasets.py:165)."""

    def __init__(self, edge_index):
        self.edge_index = edge_index
        self.edge_attr = None
        self.num_nodes = int(edge_index.max().item()) + 1


def negative_sampling(edge_index, num_nodes: int, num_neg_samples: int):
    """Uniform directed non-edges (u,v), not in edge_index, distinct - the contract of PyG's negative_sampling as called at
    datasets.py:176-197 (which passes the graph with its self loops added, so no self loop is ever drawn) - from the seeded
    hash-set sampler kernel (csrc/sampler.cu, twowl_nonedge_sample)."""
    from twowl_b200 import ops
    r, c = ops.sample_non_edges(edge_index[0].to(torch.int64), edge_index[1].to(torch.int64), num_nodes, num_neg_samples,
                                undirected=False)
    return torch.stack((r, c))


def do_edge_split(data, val_ratio=0.05, test_ratio=0.1, neg_pool_max=False):
    """datasets.py:171-206."""
    data = random_split_edges(data, val_ratio, test_ratio)
    loops = torch.arange(data.num_nodes, device=data.train_pos_edge_index.device)
    edge_index = torch.cat((data.train_pos_edge_index, torch.stack((loops, loops))), dim=1)  # add_self_loops
    data.train_neg_edge_index = negative_sampling(edge_index, data.num_nodes, data.train_pos_edge_index.shape[1])
    data.val_neg_edge_index = negative_sampling(torch.cat((edge_index, data.val_pos_edge_index), dim=-1),
                                                data.num_nodes, data.val_pos_edge_index.shape[1])
    data.test_neg_edge_index = negative_sampling(
        torch.cat((edge_index, data.val_pos_edge_index, data.test_pos_edge_index), dim=-1),
        data.num_nodes, data.test_pos_edge_index.shape[1])
    split_edge = {"train": {}, "valid": {}, "test": {}}
    split_edge["train"]["edge"] = data.train_pos_edge_index
    split_edge["train"]["edge_neg"] = data.train_neg_edge_index
    split_edge["valid"]["edge"] = data.val_pos_edge_index
    split_edge["valid"]["edge_neg"] = data.val_neg_edge_index
    split_edge["test"]["edge"] = data.test_pos_edge_index
    split_edge["test"]["edge_neg"] = data.test_neg_edge_index
    return split_edge


def load(args, device="cuda"):
    """datasets.py:154-168 - edge list (the reference's CSV; also .npy / raw binary, operators/synthetic.load_edge_list)
    -> split dict."""
    from TwoWL.operators.synthetic import load_edge_list
    edge_index = load_edge_list(args.get("csv", PATH_CSV_EDGES), device)
    return do_edge_split(_Data(edge_index), args["val_ratio"], args["test_ratio"], False)


def load_dataset(pattern, trn_ratio=0.8, val_ratio=0.05, test_ratio=0.1, csv=None, device="cuda"):
    """datasets.py:123-151."""
    args = {"data_name": "fb-pages-food", "train_name": None, "test_name": None, "val_ratio": val_ratio,
            "test_ratio": test_ratio, "max_train_num": 1000000000}
    if csv is not None:
        args["csv"] = csv
    return graph_from_split(load(args, device), pattern)


def graph_from_split(split_edge, pattern="2wl_l"):
    """The second half of load_dataset (datasets.py:133-151), reusable for synthetic graphs."""
    train_pos, train_neg = double(split_edge["train"]["edge"]), double(split_edge["train"]["edge_neg"])
    val_pos, val_neg = double(split_edge["valid"]["edge"]), double(split_edge["valid"]["edge_neg"])
    test_pos, test_neg = double(split_edge["test"]["edge"]), double(split_edge["test"]["edge_neg"])
    edge_pos = torch.cat((train_pos, val_pos, test_pos), dim=-1)
    edge_neg = torch.cat((train_neg, val_neg, test_neg), dim=-1)
    num_pos = torch.tensor([train_pos.shape[1], val_pos.shape[1], test_pos.shape[1]])
    num_neg = torch.tensor([train_neg.shape[1], val_neg.shape[1], test_neg.shape[1]])
    n_node = int(max(torch.max(edge_pos), torch.max(edge_neg)).item()) + 1
    x = torch.zeros((n_node, 0), device=edge_pos.device)
    return BaseGraph(x, None, edge_pos, edge_neg, num_pos, num_neg, pattern)
