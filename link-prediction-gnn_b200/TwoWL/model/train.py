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
    logits = mod(dataset.x, dataset.ei, dataset.pos1, targets, dataset.ei2, True).reshape(-1)
    ks = [int(k) for k in ks]
    k = getattr(dataset, "rank_k", None)
    if k is not None:
        P = logits.numel() // (1 + int(k))
        assert P * (1 + int(k)) == logits.numel(), "test_ranking: the logits do not have the [P | P x rank_k] layout"
        vals = ops.rank_metrics(logits[:P], logits[P:].reshape(P, int(k)), ks).cpu()
        return {"mrr": float(vals[0]), **{f"hits@{kk}": float(v) for kk, v in zip(ks, vals[1:1 + len(ks)].tolist())}}
    labels = dataset.y.reshape(-1)[0::2][: logits.shape[0]]
    vals = ops.hits_at_k(logits, labels, ks).cpu()
    return {f"hits@{kk}": float(v) for kk, v in zip(ks, vals[:len(ks)].tolist())}


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
