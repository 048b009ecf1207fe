"""Evaluation metrics computed where the probabilities live.

The reference's evaluation loop (/root/reference/src/utils.py:298-325) copies every batch's probabilities to the
host (`.data.cpu().numpy()`, :305) and hands Python lists to sklearn. Once a forward pass is a ~50 us graph replay
that per-batch device->host sync is the whole cost of a validation epoch, so the batches stay on the device and the
metrics are computed there (one sort + a few reductions), with ONE small device->host copy of the results.

AUC is the Mann-Whitney statistic with average ranks for tied scores, which is what sklearn.metrics.roc_auc_score
computes (trapezoidal ROC); F1 / recall / precision use sklearn's zero_division=0 convention.
"""
from __future__ import annotations

import operator

import numpy as np
import torch

__all__ = ["binary_metrics", "device_metrics", "device_curve", "device_operating_points"]


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


def _checked_inputs(prob_2n, labels, what):
    """(n, prob fp32 [2, n], labels int32 [n]) on the probabilities' device, after the checks of the device metrics."""
    if prob_2n.dim() != 2 or prob_2n.shape[0] != 2 or not prob_2n.is_cuda:
        raise ValueError(f"{what}: prob must be a [2, n] CUDA tensor, got {tuple(prob_2n.shape)}")
    n = int(prob_2n.shape[1])
    if n == 0:
        raise ValueError(f"{what}: no nodes")
    prob = prob_2n.to(torch.float32).contiguous()
    y = torch.as_tensor(labels, device=prob.device).reshape(-1)
    if y.numel() != n:
        raise ValueError(f"{what}: {y.numel()} labels for {n} nodes")
    if bool(((y != 0) & (y != 1)).any()):
        raise ValueError(f"{what}: labels must be 0 or 1")
    return n, prob, y.to(torch.int32).contiguous()


def _run_metrics(prob_2n, labels, what, checked=None):
    """pcg_binary_metrics on a fresh workspace: (n, workspace, out) on the probabilities' device."""
    from . import _lib

    n, prob, y = checked or _checked_inputs(prob_2n, labels, what)
    L = _lib.lib()
    ws = torch.empty(int(L.pcg_binary_metrics_workspace_bytes(n)), dtype=torch.uint8, device=prob.device)
    out = torch.empty(_lib.METRICS_WORDS, dtype=torch.float64, device=prob.device)
    _lib.check(L.pcg_binary_metrics(prob.data_ptr(), y.data_ptr(), n, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                    _lib.stream_ptr()), "pcg_binary_metrics")
    return n, ws, out


def device_metrics(prob_2n: torch.Tensor, labels: torch.Tensor) -> dict:
    """``binary_metrics`` of pred = (prob[1] > prob[0]) computed by one kernel chain (``pcg_binary_metrics``: sort,
    counts, best threshold) plus one device->host copy. prob_2n: planar [2, n] fp32 CUDA tensor (row 1 = P(class 1));
    labels: 0 / 1 per node. Returns python floats: the keys of ``binary_metrics`` plus best_f1_macro / best_threshold
    (the distinct value t of prob[1] whose cut "positive iff prob[1] >= t" has the largest macro-F1, ties to the larger
    t), n_pos, n_neg, the confusion counts tp, fp, tn, fn, and the ranking metrics: ap (sklearn's
    average_precision_score), recall_at_k (K = n_pos, ties counted by their expected share; also Precision@K) and
    best_gmean / best_gmean_threshold (the cut with the largest sqrt(TPR * TNR), ties to the larger t). ap and
    recall_at_k are NaN without positives. Definitions: include/pcgnn_b200.h."""
    from . import _lib

    _, _, out = _run_metrics(prob_2n, labels, "device_metrics")
    return dict(zip(_lib.METRICS_KEYS, out.cpu().tolist()))


def _curve_buffers(n: int, device):
    """(thr fp32 [n], tp int64 [n], fp int64 [n], count int64 [1]): the outputs of ``pcg_binary_curve``."""
    return (torch.empty(n, dtype=torch.float32, device=device), torch.empty(n, dtype=torch.int64, device=device),
            torch.empty(n, dtype=torch.int64, device=device), torch.empty(1, dtype=torch.int64, device=device))


def _read_curve(ws: torch.Tensor, n: int, bufs) -> tuple:
    """``pcg_binary_curve`` over a workspace the last ``pcg_binary_metrics`` on the current stream filled, then one
    8-byte read of G: views [:G] of the buffers."""
    from . import _lib

    thr, tp, fp, count = bufs
    _lib.check(_lib.lib().pcg_binary_curve(ws.data_ptr(), ws.numel(), n, thr.data_ptr(), tp.data_ptr(), fp.data_ptr(),
                                           count.data_ptr(), _lib.stream_ptr()), "pcg_binary_curve")
    G = int(count.item())
    return thr[:G], tp[:G], fp[:G]


def device_curve(prob_2n: torch.Tensor, labels: torch.Tensor) -> tuple:
    """ROC / PR curve of prob[1] against 0 / 1 labels: (thresholds fp32 [G], tp int64 [G], fp int64 [G]) as device
    tensors, one entry per distinct value t of prob[1] in ascending order with the counts of the cut "positive iff
    prob[1] >= t". TPR = tp / n_pos, FPR = fp / n_neg, precision = tp / (tp + fp): sklearn's roc_curve
    (drop_intermediate=False) and precision_recall_curve in reverse order, without their sentinel point.
    ``pcg_binary_metrics`` (sort) then ``pcg_binary_curve`` (no further sort) and one 8-byte read of G."""
    n, ws, _ = _run_metrics(prob_2n, labels, "device_curve")
    return _read_curve(ws, n, _curve_buffers(n, prob_2n.device))


def _point_requests(n: int, top_k=(), fpr=(), max_fpr=()) -> tuple:
    """The request arrays of ``pcg_binary_points`` for a set of n nodes: (kind int32 [m], arg float64 [m]) numpy
    arrays, the top_k requests first, then fpr, then max_fpr, each in the caller's order. Raises ValueError for a K
    that is not an integer in [1, n], an fpr outside [0, 1], a max_fpr outside (0, 1] (NaN included), or no
    request at all."""
    from . import _lib

    kind, arg = [], []
    for k in top_k:
        try:
            K = operator.index(k)
        except TypeError:
            raise ValueError(f"top_k: K must be an integer (a budget of q * n alerts is ceil(q * n)), got {k!r}") from None
        if not 1 <= K <= n:
            raise ValueError(f"top_k: K={K} outside [1, n={n}]")
        kind.append(_lib.POINT_TOP_K)
        arg.append(float(K))
    for kd, name, fs, lo_open in ((_lib.POINT_TPR_AT_FPR, "fpr", fpr, False), (_lib.POINT_PAUC, "max_fpr", max_fpr, True)):
        for f in fs:
            f = float(f)
            if not ((0.0 < f if lo_open else 0.0 <= f) and f <= 1.0):
                raise ValueError(f"{name}: {f} outside {'(0' if lo_open else '[0'}, 1]")
            kind.append(kd)
            arg.append(f)
    if not kind:
        raise ValueError("no operating-point requests (top_k, fpr and max_fpr are all empty)")
    if len(kind) > _lib.POINTS_MAX:
        raise ValueError(f"{len(kind)} operating-point requests, at most {_lib.POINTS_MAX}")
    return np.asarray(kind, dtype=np.int32), np.asarray(arg, dtype=np.float64)


def _points_dict(words, kind, arg) -> dict:
    """``pcg_binary_points``' output words [m * PCG_POINT_WORDS] (host) as python floats per request, grouped by kind
    in request order: {"top_k": [{k, recall, precision, threshold, tp, fp}], "tpr_at_fpr": [{max_fpr, tpr, fpr,
    threshold, tp, fp}], "pauc": [{max_fpr, pauc, area}]}."""
    from . import _lib

    w = np.asarray(words, dtype=np.float64).reshape(len(kind), _lib.POINT_WORDS).tolist()
    out = {"top_k": [], "tpr_at_fpr": [], "pauc": []}
    for kd, a, (v0, v1, thr, tp, fp) in zip(kind.tolist(), arg.tolist(), w):
        if kd == _lib.POINT_TOP_K:
            out["top_k"].append(dict(k=int(a), recall=v0, precision=v1, threshold=thr, tp=tp, fp=fp))
        elif kd == _lib.POINT_TPR_AT_FPR:
            out["tpr_at_fpr"].append(dict(max_fpr=a, tpr=v0, fpr=v1, threshold=thr, tp=tp, fp=fp))
        else:
            out["pauc"].append(dict(max_fpr=a, pauc=v0, area=v1))
    return out


def device_operating_points(prob_2n: torch.Tensor, labels: torch.Tensor, top_k=(), fpr=(), max_fpr=()) -> dict:
    """Metrics at operating points the caller chooses, for prob[1] against 0 / 1 labels (definitions:
    include/pcgnn_b200.h, pcg_binary_points):

    * ``top_k``: review budgets K (integers, 1 <= K <= n): Recall@K and Precision@K of the K highest scores, with the
      scores tied with the K-th counted by their expected share (as ``recall_at_k``), the K-th highest score as
      ``threshold`` and the expected tp / fp among the K;
    * ``fpr``: false-alarm ceilings f in [0, 1]: the largest TPR over the cuts "positive iff prob[1] >= t" with
      FP <= f * n_neg, the FPR it reaches, its threshold t and its integer tp / fp (nothing flagged: t = inf);
    * ``max_fpr``: f in (0, 1]: sklearn's ``roc_auc_score(max_fpr=f)`` (``pauc``, standardised; f = 1 gives the AUC)
      and the unstandardised area under the ROC curve up to FPR = f (``area``).

    Rates are NaN where a class they divide by is absent. ``pcg_binary_metrics`` (the sort), ``pcg_binary_points``
    and one device->host copy; requests are checked on the host (ValueError). Returns python floats, each list in
    request order: {"top_k": [{k, recall, precision, threshold, tp, fp}], "tpr_at_fpr": [{max_fpr, tpr, fpr,
    threshold, tp, fp}], "pauc": [{max_fpr, pauc, area}]}."""
    from . import _lib

    checked = _checked_inputs(prob_2n, labels, "device_operating_points")
    kind, arg = _point_requests(checked[0], top_k, fpr, max_fpr)
    n, ws, _ = _run_metrics(prob_2n, labels, "device_operating_points", checked)
    L, m, dev = _lib.lib(), len(kind), ws.device
    kind_d, arg_d = torch.from_numpy(kind).to(dev), torch.from_numpy(arg).to(dev)
    pws = torch.empty(int(L.pcg_binary_points_workspace_bytes(n, m)), dtype=torch.uint8, device=dev)
    out = torch.empty(m * _lib.POINT_WORDS, dtype=torch.float64, device=dev)
    _lib.check(L.pcg_binary_points(ws.data_ptr(), ws.numel(), n, kind_d.data_ptr(), arg_d.data_ptr(), m, out.data_ptr(),
                                   pws.data_ptr(), pws.numel(), _lib.stream_ptr()), "pcg_binary_points")
    return _points_dict(out.cpu().numpy(), kind, arg)
