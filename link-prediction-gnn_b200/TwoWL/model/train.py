"""Drop-in for the reference's TwoWL/model/train.py (SURVEY 8(f) row f2): ``train``, ``test``, ``train_routine`` with the
same signatures, return values and record-file formats, minus the Streamlit / matplotlib imports the reference pulls in
through ``from assets.theme import *`` (train.py:8).

What changes underneath:
  * ROC-AUC is computed on the device (``ops.auc``: radix sort + tie-aware rank sum) instead of
    ``pred.sigmoid().cpu().numpy()`` + sklearn every step (train.py:41-43, :61-66); ``train`` makes ONE host read per step
    (loss and score together) where the reference makes two.
  * the loss is ``twowl::bce_with_logits`` (forward + gradient in one kernel pass) and the optimiser may be
    ``twowl_b200.optim.FusedAdam`` (one kernel over a flat parameter buffer; any torch optimizer works as well).
  * ``test`` computes the ROC curve points only when asked (``curve=True``, the default, keeps the reference's
    ``(auc, fpr, tpr)`` return value); ``train_routine`` asks for them only where the reference uses them.
"""
import json
import os
import time

import torch
import torch.nn.functional as F

from TwoWL.utils import sample_block, double
from twowl_b200 import functional as F2
from twowl_b200 import ops

PATH_SAVE_TEST_AUC = "records_auc/"   # constant.py:8 of the reference


class _BatchCursor:
    """The reference's module-level batch state (train.py:12-23): one permutation of the positive and of the negative undirected
    pairs per pass over the data, cut into consecutive slices of pos_bs / neg_bs ids. Redrawn whenever train() is called with
    i == 0 - which train_routine does every epoch (train.py:87)."""

    def __init__(self):
        self.pos_bs = self.neg_bs = 0
        self.perm_pos = self.perm_neg = None

    def reset(self, dataset, batch_size):
        n_edges = dataset.ei.shape[1]
        dev = dataset.x.device
        self.pos_bs = self.neg_bs = batch_size // 2
        self.perm_pos = torch.randperm(n_edges // 2, device=dev)
        self.perm_neg = torch.randperm((dataset.pos1.shape[0] - n_edges) // 2, device=dev)

    def take(self, dataset, i):
        """-> (blocked edge ids = the positive pairs' two directions, readout rows [positives | negatives], labels)."""
        und_pos = self.perm_pos[i * self.pos_bs:(i + 1) * self.pos_bs]
        und_neg = self.perm_neg[i * self.neg_bs:(i + 1) * self.neg_bs]
        rows_pos = double(und_pos, for_index=True)
        rows_neg = double(und_neg, for_index=True) + dataset.ei.shape[1]
        labels = torch.cat((torch.ones(und_pos.numel(), device=und_pos.device),
                            torch.zeros(und_neg.numel(), device=und_pos.device))).unsqueeze(-1)
        return rows_pos, torch.cat((rows_pos, rows_neg)), labels

    def advance(self, i):
        i += 1
        return 0 if (i + 1) * self.pos_bs > self.perm_pos.shape[0] else i


_cursor = _BatchCursor()


def train(mod, opt, dataset, batch_size, i, step=None):
    """train.py:11-47: one batch = batch_size/2 positive + batch_size/2 negative undirected target links, their edges
    blocked from the graph (sample_block), forward, BCE-with-logits, backward, optimizer step.
    -> (loss: float, train AUC: float, next batch index: int).
    step: an optional twowl_b200.graphed.GraphedTrainStep for this dataset / batch size - edge blocking, forward, loss and
    backward are then ONE replayed CUDA graph (the small graphs are launch-bound otherwise)."""
    mod.train()
    if i == 0:
        _cursor.reset(dataset, batch_size)
    blocked, rows, y = _cursor.take(dataset, i)

    opt.zero_grad()
    if step is None:
        ei_new, x_new, ei2_new = sample_block(blocked, dataset.x.shape[0], dataset.ei, dataset.ei2)
        pred = mod(x_new, ei_new, dataset.pos1, rows, ei2_new)
        loss = F2.bce_with_logits(pred, y)      # F.binary_cross_entropy_with_logits + its gradient in one pass (train.py:37)
        loss.backward()
    else:
        loss = step(blocked, rows, y)
        pred = step.logits
    if step is None or getattr(step, "optimizer", None) is None:     # a captured step may contain the optimiser's update
        opt.step()

    with torch.no_grad():
        # ONE host read for loss and score; the AUC ranks the probabilities like the reference does (train.py:41-43)
        both = torch.cat((loss.detach().double().reshape(1), ops.auc(pred.sigmoid(), y)[:1])).cpu()
    return float(both[0]), float(both[1]), _cursor.advance(i)


@torch.no_grad()
def test(mod, dataset, test=False, curve=True):
    """train.py:50-68: full-graph inference, every prediction pair is a target; AUC over one label per undirected pair.
    -> (auc, fpr, tpr); fpr / tpr are None with curve=False (no device->host copy of the scores then)."""
    mod.eval()
    n_edges = dataset.ei.shape[1]
    targets = n_edges + torch.arange(dataset.y.shape[0], device=dataset.x.device)
    prob = mod(dataset.x, dataset.ei, dataset.pos1, targets, dataset.ei2, True).sigmoid()
    labels = dataset.y.reshape(-1)[0::2][: prob.shape[0]]     # the reference's interleaved True/False mask (train.py:62-64)
    score = float(ops.auc(prob, labels)[0].item())
    if not curve:
        return score, None, None
    from sklearn.metrics import roc_curve
    fpr, tpr, _ = roc_curve(labels.cpu().numpy(), prob.cpu().numpy().reshape(-1))
    return score, fpr, tpr


@torch.no_grad()
def test_ranking(mod, dataset, ks=(20, 50, 100)):
    """Ranking evaluation of a link predictor (extension: the OGB link-prediction protocols) -> dict of floats. One full-graph
    forward exactly like test(), every prediction pair a target, then on the device:
      * a table from TwoWL.operators.datasets.ranking_dataset (it has `rank_k`): logits [P positives | P x rank_k negatives, row
        i = positive i's negatives] -> {"mrr": ..., "hits@k": ...} (ops.rank_metrics, OGB's _eval_mrr / ogbl-citation2);
      * any other dataset, e.g. a val / test split with its shared negatives: labels y[0::2] as in test() ->
        {"hits@K": ...} (ops.hits_at_k, OGB's _eval_hits / ogbl-collab).
    The LOGITS are ranked, not sigmoid(logits): in fp32 the sigmoid rounds every logit above about 17 to 1.0, which would create
    ties the model did not produce and change the ranks. One device->host copy for the whole dict."""
    mod.eval()
    n_edges = dataset.ei.shape[1]
    targets = n_edges + torch.arange(dataset.y.shape[0], device=dataset.x.device)
    logits = mod(dataset.x, dataset.ei, dataset.pos1, targets, dataset.ei2, True)
    return rank_scores(logits, dataset, ks)


@torch.no_grad()
def rank_scores(scores, dataset, ks=(20, 50, 100)):
    """The ranking half of test_ranking for any score of the dataset's prediction pairs - one per undirected pair, in the order
    of test(): a model's logits, or a heuristic of heuristic_scores(dataset). Same dict and protocols as test_ranking."""
    logits = scores.reshape(-1)
    ks = [int(k) for k in ks]
    k = getattr(dataset, "rank_k", None)
    if k is not None:
        P = logits.numel() // (1 + int(k))
        assert P * (1 + int(k)) == logits.numel(), "rank_scores: the scores do not have the [P | P x rank_k] layout"
        vals = ops.rank_metrics(logits[:P], logits[P:].reshape(P, int(k)), ks).cpu()
        return {"mrr": float(vals[0]), **{f"hits@{kk}": float(v) for kk, v in zip(ks, vals[1:1 + len(ks)].tolist())}}
    labels = dataset.y.reshape(-1)[0::2][: logits.shape[0]]
    vals = ops.hits_at_k(logits, labels, ks).cpu()
    return {f"hits@{kk}": float(v) for kk, v in zip(ks, vals[:len(ks)].tolist())}


@torch.no_grad()
def heuristic_scores(dataset):
    """Neighbourhood link-prediction heuristics of the dataset's prediction pairs (extension: the baselines OGB's leaderboards
    list) -> {"cn", "jaccard", "aa", "ra"}: fp32 [P] each, one score per undirected pair pos1[E::2] in the order of test() /
    test_ranking(), P = y.shape[0] // 2. The graph is the split's message-passing graph dataset.ei read as undirected and
    simple (twowl_b200.graph.simple_adjacency, built once per edge tensor); scores are computed on the device
    (ops.link_heuristics). rank_scores(heuristic_scores(ds)["aa"], ds) then ranks a heuristic like a model."""
    from twowl_b200 import graph
    n_edges = dataset.ei.shape[1]
    ptr, adj = graph.simple_adjacency(dataset.ei, dataset.x.shape[0])
    pairs = dataset.pos1[n_edges::2][: dataset.y.shape[0] // 2]
    scores = ops.link_heuristics(ptr, adj, pairs[:, 0], pairs[:, 1])
    return dict(zip(ops.HEURISTICS, scores.unbind(0)))


@torch.no_grad()
def global_heuristic_scores(dataset, by="katz", **params):
    """A global link-prediction heuristic of the dataset's prediction pairs (extension: the path-based baselines of SEAL's table)
    -> fp32 [P]: truncated Katz (by="katz") or personalized PageRank (by="ppr") of each undirected pair pos1[E::2], rooted at its
    first endpoint, in the order of test() / test_ranking(), over the split's graph read exactly as heuristic_scores reads it.
    params (steps, damping, max_cols) go to ops.global_heuristics. rank_scores(global_heuristic_scores(ds, "ppr"), ds) ranks it
    like a model."""
    from twowl_b200 import graph
    n_edges = dataset.ei.shape[1]
    ptr, adj = graph.simple_adjacency(dataset.ei, dataset.x.shape[0])
    pairs = dataset.pos1[n_edges::2][: dataset.y.shape[0] // 2]
    return ops.global_heuristics(ptr, adj, pairs[:, 0], pairs[:, 1], by=by, **params)


@torch.no_grad()
def node2vec_embedding(dataset, **params):
    """node2vec embeddings (extension: the reference's learned baseline, SURVEY rows 7-8) -> (emb fp32 [N, dim], losses float64
    [epochs]), trained on the device by ops.node2vec over the split's graph read exactly as heuristic_scores reads it. params (dim,
    walk_length, walks_per_node, window, neg, p, q, epochs, batch_walks, lr, seed) go to ops.node2vec."""
    from twowl_b200 import graph
    ptr, adj = graph.simple_adjacency(dataset.ei, dataset.x.shape[0])
    return ops.node2vec(ptr, adj, **params)


@torch.no_grad()
def embedding_scores(dataset, emb):
    """The link score e_u . e_v of an embedding table (node2vec_embedding) for each prediction pair pos1[E::2], in the order of
    test() -> fp32 [P] (ops.embedding_dot). rank_scores(embedding_scores(ds, emb), ds) and ops.auc(scores, ds.y[0::2]) rank it
    like a model."""
    n_edges = dataset.ei.shape[1]
    pairs = dataset.pos1[n_edges::2][: dataset.y.shape[0] // 2]
    return ops.embedding_dot(emb, pairs[:, 0], pairs[:, 1])


@torch.no_grad()
def recommend_global(dataset, src, k=100, by="ppr", **params):
    """Link recommendation beyond two hops -> (ids int64 [Q, k], scores fp32 [Q, k]): each source's top-k non-neighbours by
    personalized PageRank (by="ppr") or truncated Katz (by="katz") over the split's graph, as recommend() reads it
    (ops.recommend_global; -1 / NaN pad a row with fewer candidates). The ids feed
    TwoWL.operators.datasets.candidate_dataset and rerank() as recommend()'s do."""
    from twowl_b200 import graph
    ptr, adj = graph.simple_adjacency(dataset.ei, dataset.x.shape[0])
    return ops.recommend_global(ptr, adj, src, k, by=by, **params)


@torch.no_grad()
def recommend(dataset, src, k=100, by="aa"):
    """Link recommendation (extension: the retrieval half of a re-ranking pipeline) -> (ids int64 [Q, k], scores fp32 [4, Q, k]):
    each source's top-k two-hop non-neighbours by the heuristic `by`, over the split's message-passing graph dataset.ei read as
    undirected and simple, exactly as heuristic_scores reads it (ops.recommend_links; -1 / NaN pad a row with fewer candidates).
    TwoWL.operators.datasets.candidate_dataset turns the result into a table that rerank() scores with the model."""
    from twowl_b200 import graph
    ptr, adj = graph.simple_adjacency(dataset.ei, dataset.x.shape[0])
    return ops.recommend_links(ptr, adj, src, k, by)


@torch.no_grad()
def rerank(mod, dataset):
    """Re-rank a candidate table of TwoWL.operators.datasets.candidate_dataset with the model -> (ids int64 [Q, k], logits fp32
    [Q, k]). One full-graph forward exactly like test(), every prediction pair a target; each row is then ordered by logit
    descending, ties keeping the heuristic's order, with the padding (-1) last at -inf.
    The logits depend on the whole candidate table, not only on the pair: GraphNorm's statistics run over all pair rows of the
    table (SURVEY §3.4), just as test()'s scores depend on the split. Score one table per set of sources you compare."""
    mod.eval()
    n_edges = dataset.ei.shape[1]
    targets = n_edges + torch.arange(dataset.y.shape[0], device=dataset.x.device)
    return rerank_scores(mod(dataset.x, dataset.ei, dataset.pos1, targets, dataset.ei2, True), dataset)


@torch.no_grad()
def rerank_scores(scores, dataset):
    """The table-sorting half of rerank() for any score of a candidate table's pairs (one per candidate, in the order of test(),
    e.g. ncn_scores(mod, dataset)) -> (ids int64 [Q, k], scores fp32 [Q, k]): each row ordered by score descending, ties keeping the
    heuristic's order, with the padding (-1) last at -inf."""
    logits = scores.reshape(-1)
    mask = dataset.cand_mask
    table = torch.full(mask.shape, float("-inf"), dtype=logits.dtype, device=logits.device)
    table[mask] = logits
    order = torch.sort(table, dim=1, descending=True, stable=True).indices
    return dataset.cand_ids.gather(1, order), table.gather(1, order)


def _record_run(record_dir, dsname, tst_score, seconds, fpr, tpr):
    """train.py:108-134: append 'AUC:<auc>   Time:<s>   ' to the dataset's record file; when this run's (unrounded) score is not
    below any recorded (rounded) one, keep its ROC curve in fpr.json / tpr.json in the working directory."""
    os.makedirs(record_dir, exist_ok=True)
    path = os.path.join(record_dir, f"{dsname}_auc_record_twowl.txt")
    with open(path, "a") as f:
        f.write(f"AUC:{round(tst_score, 4)}   Time:{round(seconds, 4)}   \n")
    with open(path) as f:
        recorded = [float(ln.split()[0].split(":")[1]) for ln in (raw.strip() for raw in f) if ln]
    if fpr is not None and recorded and tst_score >= max(recorded):
        for name, curve in (("fpr.json", fpr), ("tpr.json", tpr)):
            with open(name, "w") as f:
                json.dump(curve.tolist(), f)


def train_routine(dsname, mod, opt, trn_ds, val_ds, tst_ds, epoch, verbose=True, record_dir=PATH_SAVE_TEST_AUC, cuda_graph=False):
    """train.py:71-135: one batch per epoch (the reference resets train_idx every epoch, train.py:87), validation every
    epoch, test on every validation improvement, early stop after 800 epochs without one; appends
    'AUC:<auc>   Time:<s>   ' to <record_dir><dsname>_auc_record_twowl.txt and keeps fpr.json / tpr.json of the best run.
    One deliberate deviation: the reference's `fpr, tpr` are overwritten by every epoch's VALIDATION call (train.py:91), so its
    fpr.json / tpr.json hold the last epoch's validation curve (SURVEY 4: the checked-in files have 1/96 steps); here the
    validation call skips the curve (no device->host copy of the scores per epoch) and the files hold the TEST curve of the
    best validation epoch - the curve the recorded AUC belongs to."""
    say = print if verbose else (lambda *a, **k: None)
    for ds in (trn_ds, val_ds, tst_ds):
        ds.pos1 = ds.pos1.to(torch.long)
    batch_size = val_ds.y.shape[0]
    say(f"batch size{batch_size}")
    step = None
    if cuda_graph:   # the training step as one replayed CUDA graph (dropout included: device-resident seeds)
        from twowl_b200.graphed import GraphedTrainStep
        half = batch_size // 2
        from twowl_b200.optim import FusedAdam
        step = GraphedTrainStep(mod, trn_ds.x.shape[0], trn_ds.ei, trn_ds.pos1, trn_ds.ei2, n_block=2 * half, n_links=2 * half,
                                optimizer=opt if isinstance(opt, FusedAdam) else None)

    patience = 800                       # epochs without a validation improvement before giving up (train.py:83)
    best_val = tst_score = 0
    since_best = 0
    fpr = tpr = None
    started = finished = 0.0
    for ep in range(epoch):
        started = time.time()
        loss, trn_score, _ = train(mod, opt, trn_ds, batch_size, 0, step)
        finished = time.time()
        val_score = test(mod, val_ds, curve=False)[0]
        line = f"epoch: {ep:03d}, trn: time {finished - started:.2f} s, loss {loss:.4f}, trn {trn_score:.4f}, val {val_score:.4f} "
        since_best += 1
        if val_score > best_val:
            best_val, since_best = val_score, 0
            if verbose:
                started = time.time()
                tst_score, fpr, tpr = test(mod, tst_ds, True)
                finished = time.time()
            line += f"tst {tst_score:.4f}"
        say(line)
        if since_best > patience:
            break
    say(f"end test {tst_score:.3f}")
    if verbose and record_dir is not None:
        _record_run(record_dir, dsname, tst_score, finished - started, fpr, tpr)
    return best_val


def _seal_graph(dataset):
    from twowl_b200 import graph
    return graph.simple_adjacency(dataset.ei, dataset.x.shape[0])


def _link_targets(dataset):
    """The training targets of SEAL and NCN: the undirected pairs of ei (pos1[:E:2], label 1) and the negatives pos1[E::2] (label 0)."""
    n_edges = dataset.ei.shape[1]
    pos, neg = dataset.pos1[:n_edges:2], dataset.pos1[n_edges::2]
    y = torch.cat((torch.ones(pos.shape[0], device=pos.device), torch.zeros(neg.shape[0], device=pos.device)))
    return torch.cat((pos, neg)).to(torch.long), y


def seal_fit(trn_ds, epochs, batch_size, lr=1e-4, hops=1, max_nodes_per_hop=0, seed=0, node_feat=None, hidden=32, num_layers=3,
             dropout=0.5):
    """Train SEAL's DGCNN (TwoWL.model.seal) on a training split (extension: the reference's SEAL baseline, SURVEY row 6)
    -> (model, losses float64 [steps]). Targets: every undirected pair of trn_ds.ei and the negatives pos1[E::2]; each batch of
    batch_size targets (a seeded permutation per epoch) gets its enclosing subgraphs extracted on the fly over the split's graph
    (ops.seal_subgraphs, hops / max_nodes_per_hop), then forward, BCE-with-logits, backward and a FusedAdam step (lr). SortPooling's
    k and max_z come from the training subgraphs (PyG's 60% rule, seal.sort_pool_k). node_feat [N, F] is optional per-node input.
    The same seed gives the same losses and weights bit for bit."""
    from TwoWL.model.seal import DGCNN, sort_pool_k
    from twowl_b200.optim import FusedAdam
    ptr, adj = _seal_graph(trn_ds)
    pairs, y = _link_targets(trn_ds)
    T = pairs.shape[0]
    sub_kw = dict(hops=hops, max_nodes_per_hop=max_nodes_per_hop, seed=seed)
    sizes = ops.seal_subgraph_sizes(ptr, adj, pairs[:, 0], pairs[:, 1], **sub_kw)
    max_z = 1
    for q in range(0, T, 4096):
        sub = ops.seal_subgraphs(ptr, adj, pairs[q:q + 4096, 0], pairs[q:q + 4096, 1], index_base=q, **sub_kw)
        max_z = max(max_z, int(sub.z.max()) if sub.z.numel() else 1)
    with torch.random.fork_rng(devices=[pairs.device]):
        torch.manual_seed(seed)
        mod = DGCNN(max_z, sort_pool_k(sizes), hidden, num_layers, 0 if node_feat is None else node_feat.shape[1], dropout)
    mod = mod.to(pairs.device).train()
    opt = FusedAdam(mod.parameters(), lr=lr)
    gen = torch.Generator(device="cpu")
    gen.manual_seed(seed)
    losses = []
    step = 0
    for _ in range(epochs):
        perm = torch.randperm(T, generator=gen).to(pairs.device)
        for b in range(0, T, batch_size):
            ids = perm[b:b + batch_size]
            # a capped layer's sample keys on the target's position in this epoch's order: a fresh sample per epoch
            sub = ops.seal_subgraphs(ptr, adj, pairs[ids, 0], pairs[ids, 1], index_base=b, **sub_kw)
            opt.zero_grad()
            loss = F2.bce_with_logits(mod(sub, node_feat, seed=(seed * 1000003 + step) % (2 ** 62)), y[ids].unsqueeze(-1))
            loss.backward()
            opt.step()
            losses.append(loss.detach().double().reshape(1))
            step += 1
    mod.eval()
    return mod, (torch.cat(losses).cpu() if losses else torch.zeros(0, dtype=torch.float64))


@torch.no_grad()
def seal_scores(mod, dataset, hops=1, max_nodes_per_hop=0, seed=0, node_feat=None, batch_size=1024):
    """SEAL logits of the dataset's prediction pairs pos1[E::2] -> fp32 [P], in the order of test(): each pair's enclosing subgraph
    over the split's graph (ops.seal_subgraphs, index_base = the pair's index), scored by the DGCNN in eval mode.
    rank_scores(seal_scores(mod, ds), ds) and ops.auc(scores, ds.y[0::2]) rank it like any other score."""
    mod.eval()
    ptr, adj = _seal_graph(dataset)
    n_edges = dataset.ei.shape[1]
    pairs = dataset.pos1[n_edges::2][: dataset.y.shape[0] // 2].to(torch.long)
    out = []
    for q in range(0, pairs.shape[0], batch_size):
        sub = ops.seal_subgraphs(ptr, adj, pairs[q:q + batch_size, 0], pairs[q:q + batch_size, 1], hops=hops,
                                 max_nodes_per_hop=max_nodes_per_hop, seed=seed, index_base=q)
        out.append(mod(sub, node_feat).reshape(-1))
    return torch.cat(out) if out else torch.zeros(0, device=pairs.device)


def ncn_fit(trn_ds, epochs, batch_size, lr=1e-3, hidden=64, num_layers=2, dropout=0.3, cn=True, node_feat=None, seed=0):
    """Train NCN (TwoWL.model.ncn; cn=False: the GCN + MLP-decoder baseline) on a training split (extension: the message-passing
    link predictors of the OGB leaderboards) -> (model, losses float64 [steps]). Targets: every undirected pair of trn_ds.ei
    (label 1) and the negatives pos1[E::2] (label 0), as seal_fit takes them, in a seeded permutation per epoch. Per batch of
    batch_size targets, NCN's protocol: the batch's positive edges are removed from the encoder's graph (sample_block, which also
    gives the degree input) and from the adjacency the common neighbours are read from (ops.adjacency_pair_mask passed to
    ops.common_neighbors); then the full-graph encoder, the predictor on the batch, BCE-with-logits, backward and a FusedAdam step
    (lr). Degrees are clipped to the split's maximum. node_feat [N, F] replaces the degree input. The same seed gives the same
    losses and weights bit for bit."""
    from TwoWL.model.ncn import NCN
    from twowl_b200 import graph
    from twowl_b200.optim import FusedAdam
    N = trn_ds.x.shape[0]
    ptr, adj = graph.simple_adjacency(trn_ds.ei, N)
    pairs, y = _link_targets(trn_ds)
    T, n_pos = pairs.shape[0], trn_ds.ei.shape[1] // 2
    max_x = int(trn_ds.x.max()) if N else 0
    with torch.random.fork_rng(devices=[pairs.device]):
        torch.manual_seed(seed)
        mod = NCN(max_x, hidden, num_layers, dropout, cn, 0 if node_feat is None else node_feat.shape[1])
    mod = mod.to(pairs.device).train()
    opt = FusedAdam(mod.parameters(), lr=lr)
    gen = torch.Generator(device="cpu")
    gen.manual_seed(seed)
    losses = []
    step = 0
    for _ in range(epochs):
        perm = torch.randperm(T, generator=gen).to(pairs.device)
        for b in range(0, T, batch_size):
            ids = perm[b:b + batch_size]
            bp = pairs[ids]
            pos = ids[ids < n_pos]                     # target k < n_pos is the undirected edge (ei[:, 2k], ei[:, 2k + 1])
            ei_new, x_new, _ = sample_block(double(pos, for_index=True), N, trn_ds.ei, None)
            cn_lists = None
            if cn:
                cn_lists = ops.common_neighbors(ptr, adj, bp[:, 0], bp[:, 1],
                                                ops.adjacency_pair_mask(ptr, adj, pairs[pos, 0], pairs[pos, 1]))
            opt.zero_grad()
            logits = mod(x_new, ei_new, bp, cn_lists, node_feat, seed=(seed * 1000003 + step) % (2 ** 62))
            loss = F2.bce_with_logits(logits, y[ids].unsqueeze(-1))
            loss.backward()
            opt.step()
            losses.append(loss.detach().double().reshape(1))
            step += 1
    mod.eval()
    return mod, (torch.cat(losses).cpu() if losses else torch.zeros(0, dtype=torch.float64))


@torch.no_grad()
def ncn_scores(mod, dataset, node_feat=None, batch_size=65536):
    """NCN logits of the dataset's prediction pairs pos1[E::2] -> fp32 [P], in the order of test(): one encoder pass over dataset.ei
    with nothing removed, then the predictor over batches of pairs with their common neighbours in the split's simple graph
    (graph.simple_adjacency). A pair's logit depends on that pair alone, so the result does not depend on batch_size, bit for bit.
    rank_scores(ncn_scores(mod, ds), ds), ops.auc(scores, ds.y[0::2]) and rerank_scores rank it like any other score."""
    from twowl_b200 import graph
    mod.eval()
    N = dataset.x.shape[0]
    ptr, adj = graph.simple_adjacency(dataset.ei, N)
    n_edges = dataset.ei.shape[1]
    pairs = dataset.pos1[n_edges::2][: dataset.y.shape[0] // 2].to(torch.long)
    h = mod.encode(dataset.x, dataset.ei, node_feat)
    out = []
    for q in range(0, pairs.shape[0], batch_size):
        bp = pairs[q:q + batch_size]
        cn_lists = ops.common_neighbors(ptr, adj, bp[:, 0], bp[:, 1]) if mod.cn else None
        out.append(mod.predict(h, bp, cn_lists).reshape(-1))
    return torch.cat(out) if out else torch.zeros(0, device=pairs.device)


def _buddy_batch_features(ptr, adj, pairs, ids, n_pos, hops, sketch_args):
    """buddy_fit's structure features of the targets pairs[ids] -> (fp32 [B, hops² + 2 hops], the positive target ids): the
    split's simple adjacency (ptr, adj) is sketched with the batch's positive edges masked out, then the pairs are read."""
    pos = ids[ids < n_pos]                             # target k < n_pos is the undirected edge (ei[:, 2k], ei[:, 2k + 1])
    mask = ops.adjacency_pair_mask(ptr, adj, pairs[pos, 0], pairs[pos, 1])
    sk = ops.link_sketches(ptr, adj, hops, entry_mask=mask, **sketch_args)
    return ops.sketch_features(sk, pairs[ids, 0], pairs[ids, 1]), pos


def buddy_fit(trn_ds, epochs, batch_size, lr=1e-3, hops=2, num_perm=128, hll_p=8, dropout=0.5, hidden=32, node_feat=None, seed=0):
    """Train BUDDY (TwoWL.model.buddy; extension: the subgraph-sketching link predictors of the OGB leaderboards) on a training
    split -> (model, losses float64 [steps]). Targets and their order are ncn_fit's: every undirected pair of trn_ds.ei (label 1)
    and the negatives pos1[E::2] (label 0), in a seeded permutation per epoch. Per batch of batch_size targets, NCN's protocol: the
    batch's positive edges are deleted before its features are made, so no target link is seen. The split's simple adjacency is
    sketched with those edges masked out (ops.adjacency_pair_mask, ops.link_sketches with hops / num_perm / hll_p, sketch seed
    `seed`) and the batch's ops.sketch_features read from it; with node_feat [N, F] the propagation runs over sample_block's graph.
    Then forward, BCE-with-logits, backward and a FusedAdam step (lr). A trailing batch of one target is skipped (training-mode
    BatchNorm needs two). The same seed gives the same losses and weights bit for bit."""
    from TwoWL.model.buddy import BUDDY
    from twowl_b200 import graph
    from twowl_b200.optim import FusedAdam
    N = trn_ds.x.shape[0]
    ptr, adj = graph.simple_adjacency(trn_ds.ei, N)
    pairs, y = _link_targets(trn_ds)
    T, n_pos = pairs.shape[0], trn_ds.ei.shape[1] // 2
    with torch.random.fork_rng(devices=[pairs.device]):
        torch.manual_seed(seed)
        mod = BUDDY(hops, dropout, 0 if node_feat is None else node_feat.shape[1], hidden)
    mod.sketch_args = dict(num_perm=num_perm, hll_p=hll_p, seed=seed)
    mod = mod.to(pairs.device).train()
    opt = FusedAdam(mod.parameters(), lr=lr)
    gen = torch.Generator(device="cpu")
    gen.manual_seed(seed)
    losses = []
    step = 0
    for _ in range(epochs):
        perm = torch.randperm(T, generator=gen).to(pairs.device)
        for b in range(0, T, batch_size):
            ids = perm[b:b + batch_size]
            if ids.numel() < 2:
                continue
            bp = pairs[ids]
            sf, pos = _buddy_batch_features(ptr, adj, pairs, ids, n_pos, hops, mod.sketch_args)
            xs = None
            if node_feat is not None:
                ei_new, _, _ = sample_block(double(pos, for_index=True), N, trn_ds.ei, None)
                xs = mod.propagate(node_feat, ei_new)
            opt.zero_grad()
            logits = mod(sf, bp, xs, seed=(seed * 1000003 + step) % (2 ** 62))
            loss = F2.bce_with_logits(logits, y[ids].unsqueeze(-1))
            loss.backward()
            opt.step()
            losses.append(loss.detach().double().reshape(1))
            step += 1
    mod.eval()
    return mod, (torch.cat(losses).cpu() if losses else torch.zeros(0, dtype=torch.float64))


@torch.no_grad()
def buddy_scores(mod, dataset, node_feat=None, batch_size=65536):
    """BUDDY logits of the dataset's prediction pairs pos1[E::2] -> fp32 [P], in the order of test(): the split's simple graph is
    sketched once with nothing removed (the num_perm / hll_p / seed buddy_fit trained with), the propagation of node_feat runs over
    dataset.ei, and the model scores batches of pairs in eval mode. A pair's logit depends on that pair alone, so the result does
    not depend on batch_size, bit for bit. rank_scores(buddy_scores(mod, ds), ds), ops.auc(scores, ds.y[0::2]) and rerank_scores
    rank it like any other score."""
    from twowl_b200 import graph
    mod.eval()
    N = dataset.x.shape[0]
    ptr, adj = graph.simple_adjacency(dataset.ei, N)
    n_edges = dataset.ei.shape[1]
    pairs = dataset.pos1[n_edges::2][: dataset.y.shape[0] // 2].to(torch.long)
    sk = ops.link_sketches(ptr, adj, mod.hops, **mod.sketch_args)
    xs = mod.propagate(node_feat, dataset.ei) if node_feat is not None else None
    out = []
    for q in range(0, pairs.shape[0], batch_size):
        bp = pairs[q:q + batch_size]
        out.append(mod(ops.sketch_features(sk, bp[:, 0], bp[:, 1]), bp, xs).reshape(-1))
    return torch.cat(out) if out else torch.zeros(0, device=pairs.device)
