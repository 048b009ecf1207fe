"""The ranking words of pcg_binary_metrics (ap, recall_at_k, best_gmean, best_gmean_threshold) and pcg_binary_curve
(metrics.device_curve, GraphedEvalPass.curve) against sklearn and a numpy float64 brute force written from the
definitions in include/pcgnn_b200.h; directly and through the evaluation pass (PC-GNN on C2, GraphSAGE on C4)."""
import warnings

import numpy as np
import pytest
import torch

from test_gpu_eval_pass import _model, _same

RANK_KEYS = ("ap", "recall_at_k", "best_gmean", "best_gmean_threshold")


def _reference(p1, y):
    """Brute force over the tie groups of p1 (ascending, stable): thresholds and integer TP / FP of every group cut,
    recall_at_k and the best G-mean cut (ties to the larger threshold), in float64 with the kernel's operation order."""
    p1 = np.asarray(p1, dtype=np.float32)
    y = np.asarray(y).astype(np.int64)
    order = np.argsort(p1, kind="stable")
    s, ys = p1[order].astype(np.float64), y[order]
    n, P = len(s), int(y.sum())
    N = n - P
    pre = np.concatenate([[0], np.cumsum(ys)])
    starts = np.flatnonzero(np.concatenate([[True], s[1:] != s[:-1]]))
    ends = np.append(starts[1:], n)
    tp = P - pre[starts]
    fp = (n - starts) - tp
    rk = float("nan")
    if P > 0:
        c = n - P
        g = int(np.searchsorted(starts, c, side="right")) - 1
        lo, hi = int(starts[g]), int(ends[g])
        tpk = float(P - pre[hi]) + float(pre[hi] - pre[lo]) * float(hi - c) / float(hi - lo)
        rk = tpk / P
    tpr = tp / P if P > 0 else np.zeros(len(starts))
    tnr = (N - fp) / N if N > 0 else np.zeros(len(starts))
    gm = np.sqrt(tpr * tnr)
    at = len(gm) - 1 - int(np.argmax(gm[::-1]))
    return dict(thr=s[starts], tp=tp, fp=fp, recall_at_k=rk, best_gmean=float(gm[at]),
                best_gmean_threshold=float(s[starts[at]]), P=P, N=N, top=int(ys[n - P:].sum()) if P else 0)


def _inputs(n, kind):
    rng = np.random.default_rng(1000 + n)
    p1, p0 = rng.random(n).astype(np.float32), rng.random(n).astype(np.float32)
    y = (rng.random(n) < 0.12).astype(np.int64)
    if n > 1:
        y[0], y[1] = 1, 0
    if kind == "quantised":
        p1 = (np.round(p1 * 20) / 20).astype(np.float32)     # 21 values: groups span chunks of 2048 positions
    if kind == "one_class":
        y[:] = 0
    if kind == "all_positive":
        y[:] = 1
    return p1, p0, y


def _check_rank(m, p1, y):
    """m's ranking words against sklearn and the brute force; returns the brute force."""
    from sklearn.metrics import average_precision_score

    assert m.keys() >= set(RANK_KEYS)
    ref = _reference(p1, y)
    if ref["P"] == 0:
        assert np.isnan(m["ap"]) and np.isnan(m["recall_at_k"])
    else:
        want = average_precision_score(y, p1.astype(np.float64))
        assert abs(m["ap"] - want) <= 1e-12 * abs(want), (m["ap"], want)
        assert m["recall_at_k"] == ref["recall_at_k"]
    assert m["best_gmean"] == ref["best_gmean"] and m["best_gmean_threshold"] == ref["best_gmean_threshold"]
    return ref


def _check_curve(curve, p1, y, ref):
    from sklearn.metrics import precision_recall_curve, roc_curve

    thr, tp, fp = (t.cpu().numpy() for t in curve)
    assert thr.dtype == np.float32 and tp.dtype == np.int64 and fp.dtype == np.int64
    assert np.array_equal(thr.astype(np.float64), ref["thr"])
    assert np.array_equal(tp, ref["tp"]) and np.array_equal(fp, ref["fp"])
    s = p1.astype(np.float64)
    P, N = ref["P"], ref["N"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                                  # one class only: sklearn warns, tpr or fpr NaN
        fpr, tpr, rthr = roc_curve(y, s, drop_intermediate=False)
    fpr, tpr, rthr = fpr[1:][::-1], tpr[1:][::-1], rthr[1:][::-1]      # ascending, without the sentinel
    assert np.array_equal(rthr, thr.astype(np.float64))
    if P > 0:
        assert np.array_equal(np.rint(tpr * P).astype(np.int64), tp)
    if N > 0:
        assert np.array_equal(np.rint(fpr * N).astype(np.int64), fp)
    if P > 0:
        prec, rec, pthr = precision_recall_curve(y, s, drop_intermediate=False)
        assert np.array_equal(pthr, thr.astype(np.float64))
        assert np.array_equal(prec[:-1], tp / (tp + fp).astype(np.float64))
        assert np.array_equal(rec[:-1], tp / float(P))


def test_reference_agrees_with_sklearn_and_a_literal_count():
    """CPU: the cumulative brute force against sklearn's curve and the literal top-P count / every cut from scratch."""
    from sklearn.metrics import roc_curve

    rng = np.random.default_rng(9)
    for n in (1, 2, 40, 700):
        for q in (None, 7):
            p1 = rng.random(n).astype(np.float32)
            if q:
                p1 = (np.round(p1 * q) / q).astype(np.float32)
            y = (rng.random(n) < 0.3).astype(np.int64)
            ref = _reference(p1, y)
            for g, t in enumerate(ref["thr"]):
                cut = p1 >= np.float32(t)
                assert ref["tp"][g] == int((cut & (y == 1)).sum()) and ref["fp"][g] == int((cut & (y == 0)).sum())
            if 0 < ref["P"] < n:
                fpr, tpr, _ = roc_curve(y, p1.astype(np.float64), drop_intermediate=False)
                assert np.array_equal(np.rint(tpr[1:][::-1] * ref["P"]).astype(np.int64), ref["tp"])
            if ref["P"] and len(np.unique(p1)) == n:
                assert ref["recall_at_k"] == ref["top"] / ref["P"]
            if ref["P"] and q:
                # the expected count over random orders of the ties, by sampling tie orders
                acc = 0.0
                for _ in range(400):
                    o = np.lexsort((rng.random(n), p1))
                    acc += y[o][n - ref["P"]:].sum()
                assert abs(acc / 400 / ref["P"] - ref["recall_at_k"]) <= 0.1


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 8192, 8193, 100_000, 3_000_000])
@pytest.mark.parametrize("kind", ["random", "quantised", "one_class", "all_positive"])
def test_rank_metrics_and_curve_against_sklearn_and_brute_force(n, kind):
    from pcgnn_b200.metrics import device_curve, device_metrics

    p1, p0, y = _inputs(n, kind)
    prob = torch.from_numpy(np.stack([p0, p1])).cuda()
    yt = torch.from_numpy(y).cuda()
    m = device_metrics(prob, yt)
    assert _same(m, device_metrics(prob, yt))                             # bit-identical reruns
    ref = _check_rank(m, p1, y)
    if ref["P"] and len(np.unique(p1)) == n:
        assert m["recall_at_k"] == ref["top"] / ref["P"]
    curve = device_curve(prob, yt)
    _check_curve(curve, p1, y, ref)
    again = device_curve(prob, yt)
    assert all(torch.equal(a, b) for a, b in zip(curve, again))


@pytest.mark.gpu
def test_c2_pass_rank_keys_and_curve_match_sklearn():
    from pcgnn_b200.runtime import GraphedEvalPass

    d, _, model = _model("yelp", seed=72)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    ev = GraphedEvalPass(model, nodes, labels, 1024)
    m = ev.run()
    p1 = ev.probs()[:, 1].cpu().numpy()
    ref = _check_rank(m, p1, labels)
    _check_curve(ev.curve(), p1, labels, ref)
    assert ev.captures == 1 and _same(m, ev.run())


@pytest.mark.gpu
def test_c4_graphsage_rank_keys_and_curve_on_log_probabilities():
    from test_gpu_eval_pass_baselines import _build

    from pcgnn_b200.metrics import device_curve
    from pcgnn_b200.runtime import GraphedEvalPass
    from pcgnn_b200.synth import make_graph

    d = make_graph("amazon", seed=72)
    model, _, _ = _build("sage", d.feat, d.homo, E=64, seed=72)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    ev = GraphedEvalPass(model, nodes, labels, 1024)
    m = ev.run()
    lp = ev.probs()[:, 1].cpu().numpy()          # log-probabilities: the ranking is that of the probabilities
    assert (lp <= 0).all()
    ref = _check_rank(m, lp, labels)
    curve = ev.curve()
    _check_curve(curve, lp, labels, ref)
    fresh = device_curve(ev.probs().t().contiguous(), torch.from_numpy(labels).cuda())
    assert all(torch.equal(a, b) for a, b in zip(curve, fresh))


@pytest.mark.gpu
def test_curve_after_interleaved_training_steps_matches_a_fresh_device_curve():
    from pcgnn_b200.metrics import device_curve
    from pcgnn_b200.parallel import FusedAdam, GradAllReduce
    from pcgnn_b200.runtime import GraphedEvalPass, GraphedTrainStep

    d, _, model = _model(seed=75)
    rng = np.random.default_rng(75)
    B, n_steps = 128, 4
    batches = [rng.choice(d.idx_train, B) for _ in range(n_steps)]
    nodes = np.arange(d.feat.shape[0])
    y = torch.from_numpy(d.labels[nodes]).cuda()
    reducer = GradAllReduce(model.parameters()).attach()
    opt = FusedAdam(reducer, lr=0.01, weight_decay=1e-3)
    eng = model.inter1.engine()
    eng.set_features(model.inter1.features.weight)
    cap = GraphedTrainStep.plan(eng, batches, model.inter1.thresholds, 0.5)
    step = GraphedTrainStep(model, opt, B, cap, reducer=reducer, warmup_batch=(batches[0], d.labels[batches[0]]))
    step.load_plan([(b, d.labels[b]) for b in batches])
    ev = GraphedEvalPass(model, nodes, d.labels[nodes], 1024)
    prev = None
    for _ in range(2):
        ev.run()
        probs = ev.probs().t().clone()
        for _ in range(n_steps):
            step.run_planned()
        curve = [t.clone() for t in ev.curve()]              # the run's workspace, read after the training steps
        fresh = device_curve(probs, y)
        assert all(torch.equal(a, b) for a, b in zip(curve, fresh))
        if prev is not None:
            assert not torch.equal(prev, probs)                 # the second run scored the trained weights
        prev = probs
    assert not step.overflowed()
