"""Evaluation metrics computed where the probabilities live.

The reference's evaluation loop (/root/reference/src/utils.py:298-325) copies every batch's probabilities to the
host (`.data.cpu().numpy()`, :305) and hands Python lists to sklearn. Once a forward pass is a ~50 us graph replay
that per-batch device->host sync is the whole cost of a validation epoch, so the batches stay on the device and the
metrics are computed there (one sort + a few reductions), with ONE small device->host copy of the results.

AUC is the Mann-Whitney statistic with average ranks for tied scores, which is what sklearn.metrics.roc_auc_score
computes (trapezoidal ROC); F1 / recall / precision use sklearn's zero_division=0 convention.
"""
from __future__ import annotations

import torch

__all__ = ["binary_metrics", "device_metrics"]


def binary_metrics(prob1: torch.Tensor, pred: torch.Tensor, labels: torch.Tensor) -> dict:
    """prob1: P(class 1) per node, pred: predicted class (0/1), labels: true class (0/1); any device.
    Returns python floats: auc, f1 (positive class), f1_macro, recall, precision, recall_macro, precision_macro,
    accuracy, gmean."""
    y = labels.reshape(-1).to(torch.int64)
    p = pred.reshape(-1).to(torch.int64)
    s = prob1.reshape(-1).to(torch.float64)
    n = y.numel()
    # ---- AUC: rank-sum with average ranks over ties
    s_sorted, order = torch.sort(s)
    _, inv, counts = torch.unique_consecutive(s_sorted, return_inverse=True, return_counts=True)
    cum = counts.cumsum(0).to(torch.float64)
    avg_rank = (2.0 * cum - counts.to(torch.float64) + 1.0) * 0.5          # mean of ranks start+1 .. cum (1-based)
    ranks = avg_rank[inv]
    y_sorted = y[order]
    n_pos = y.sum().to(torch.float64)
    n_neg = float(n) - n_pos
    auc = (ranks[y_sorted == 1].sum() - n_pos * (n_pos + 1.0) * 0.5) / (n_pos * n_neg)
    # ---- confusion counts
    tp = ((p == 1) & (y == 1)).sum().to(torch.float64)
    tn = ((p == 0) & (y == 0)).sum().to(torch.float64)
    fp = ((p == 1) & (y == 0)).sum().to(torch.float64)
    fn = ((p == 0) & (y == 1)).sum().to(torch.float64)

    def div(a, b):
        return torch.where(b > 0, a / b.clamp_min(1.0), torch.zeros_like(a))

    prec1, rec1 = div(tp, tp + fp), div(tp, tp + fn)
    prec0, rec0 = div(tn, tn + fn), div(tn, tn + fp)
    f1_1 = div(2 * prec1 * rec1, prec1 + rec1)
    f1_0 = div(2 * prec0 * rec0, prec0 + rec0)
    out = torch.stack([auc, f1_1, 0.5 * (f1_0 + f1_1), rec1, prec1, 0.5 * (rec0 + rec1), 0.5 * (prec0 + prec1),
                       (tp + tn) / float(max(n, 1)), torch.sqrt(rec1 * rec0)]).cpu().tolist()
    keys = ["auc", "f1", "f1_macro", "recall", "precision", "recall_macro", "precision_macro", "accuracy", "gmean"]
    return dict(zip(keys, out))


def device_metrics(prob_2n: torch.Tensor, labels: torch.Tensor) -> dict:
    """``binary_metrics`` of pred = (prob[1] > prob[0]) computed by one kernel chain (``pcg_binary_metrics``: sort,
    counts, best threshold) plus one device->host copy. prob_2n: planar [2, n] fp32 CUDA tensor (row 1 = P(class 1));
    labels: 0 / 1 per node. Returns python floats: the keys of ``binary_metrics`` plus best_f1_macro / best_threshold
    (the distinct value t of prob[1] whose cut "positive iff prob[1] >= t" has the largest macro-F1, ties to the larger
    t), n_pos, n_neg and the confusion counts tp, fp, tn, fn."""
    from . import _lib

    if prob_2n.dim() != 2 or prob_2n.shape[0] != 2 or not prob_2n.is_cuda:
        raise ValueError(f"device_metrics: prob must be a [2, n] CUDA tensor, got {tuple(prob_2n.shape)}")
    n = int(prob_2n.shape[1])
    if n == 0:
        raise ValueError("device_metrics: no nodes")
    prob = prob_2n.to(torch.float32).contiguous()
    y = torch.as_tensor(labels, device=prob.device).reshape(-1)
    if y.numel() != n:
        raise ValueError(f"device_metrics: {y.numel()} labels for {n} nodes")
    if bool(((y != 0) & (y != 1)).any()):
        raise ValueError("device_metrics: labels must be 0 or 1")
    y = y.to(torch.int32).contiguous()
    L = _lib.lib()
    ws = torch.empty(int(L.pcg_binary_metrics_workspace_bytes(n)), dtype=torch.uint8, device=prob.device)
    out = torch.empty(_lib.METRICS_WORDS, dtype=torch.float64, device=prob.device)
    _lib.check(L.pcg_binary_metrics(prob.data_ptr(), y.data_ptr(), n, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                    _lib.stream_ptr()), "pcg_binary_metrics")
    return dict(zip(_lib.METRICS_KEYS, out.cpu().tolist()))
