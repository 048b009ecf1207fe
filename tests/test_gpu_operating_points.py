"""Caller-chosen operating points (pcg_binary_points: Recall / Precision at K, TPR at FPR <= f, standardised partial
AUC) against a numpy float64 brute force written from the definitions in include/pcgnn_b200.h and against sklearn;
directly (metrics.device_operating_points, the C ABI) and through the evaluation pass (PC-GNN on C2, GraphSAGE on C4)."""
import itertools
import math
import warnings

import numpy as np
import pytest
import torch

FPRS = (0.0, 1e-3, 0.01, 0.5, 1.0)
MAX_FPRS = (1e-3, 0.01, 0.1, 1.0)
NAN5 = [math.nan] * 5


def _groups(p1):
    """Sorted scores (float32, ascending, stable) and the tie groups' [lo, hi) bounds."""
    s = np.sort(np.asarray(p1, dtype=np.float32), kind="stable")
    lo = np.flatnonzero(np.concatenate([[True], s[1:] != s[:-1]]))
    return s, lo, np.append(lo[1:], len(s))


def _top_k(p1, y, K):
    """Top K from masks: the positives strictly above the K-th highest score t plus the positives tied with t by the
    share of the tie's slots above the cut, in the kernel's operation order."""
    p1 = np.asarray(p1, dtype=np.float32)
    pos = np.asarray(y) != 0
    n, P = len(p1), int(pos.sum())
    t = np.sort(p1, kind="stable")[n - K]
    above, tied = p1 > t, p1 == t
    tp = float(int((pos & above).sum())) + float(int((pos & tied).sum())) * float(K - int(above.sum())) / float(
        int(tied.sum()))
    return [tp / P if P else math.nan, tp / float(K), float(t), tp, float(K) - tp]


def _cuts(p1, y):
    """Every group cut "positive iff p1 >= t", by descending t: (t, TP, FP) as arrays."""
    s, lo, _ = _groups(p1)
    ys = np.asarray(y)[np.argsort(np.asarray(p1, dtype=np.float32), kind="stable")] != 0
    pre = np.concatenate([[0], np.cumsum(ys)])
    P, n = int(ys.sum()), len(s)
    tp = P - pre[lo]
    fp = (n - lo) - tp
    return s[lo][::-1].astype(np.float64), tp[::-1], fp[::-1]


def _tpr_at_fpr(cuts, P, N, f):
    if P == 0 or N == 0:
        return NAN5
    t, tp, fp = cuts
    ok = np.flatnonzero(fp.astype(np.float64) <= f * float(N))
    if ok.size == 0:
        return [0.0, 0.0, math.inf, 0.0, 0.0]
    i = ok[-1]                                        # the lowest qualifying threshold: the largest TP
    return [tp[i] / P, fp[i] / N, float(t[i]), float(tp[i]), float(fp[i])]


def _pauc(cuts, P, N, f):
    """Trapezoids over the ROC points (0, 0), (FP / N, TP / P) by descending threshold, clipped at FPR = f."""
    if P == 0 or N == 0:
        return NAN5
    _, tp, fp = cuts
    x, yv = np.concatenate([[0.0], fp / N]), np.concatenate([[0.0], tp / P])
    x0, x1, y0, y1 = x[:-1], x[1:], yv[:-1], yv[1:]
    keep = x0 < f
    x0, x1, y0, y1 = x0[keep], x1[keep], y0[keep], y1[keep]
    cut = x1 > f
    xe = np.where(cut, f, x1)
    ye = np.where(cut, y0 + (y1 - y0) * (f - x0) / np.where(cut, x1 - x0, 1.0), y1)
    A = float(np.sum((xe - x0) * (ye + y0))) * 0.5
    lo_area = 0.5 * f * f
    return [0.5 * (1.0 + (A - lo_area) / (f - lo_area)), A, math.nan, math.nan, math.nan]


def _brute(p1, y, top_k, fpr, max_fpr):
    """The expected result of device_operating_points, as {kind: [[5 words], ...]} in request order."""
    pos = np.asarray(y) != 0
    P, N = int(pos.sum()), int((~pos).sum())
    cuts = _cuts(p1, y)
    return {"top_k": [_top_k(p1, y, K) for K in top_k], "tpr_at_fpr": [_tpr_at_fpr(cuts, P, N, f) for f in fpr],
            "pauc": [_pauc(cuts, P, N, f) for f in max_fpr]}


def _words(res):
    """device_operating_points' dict as {kind: [[5 words], ...]} (the layout of the header)."""
    return {"top_k": [[d["recall"], d["precision"], d["threshold"], d["tp"], d["fp"]] for d in res["top_k"]],
            "tpr_at_fpr": [[d["tpr"], d["fpr"], d["threshold"], d["tp"], d["fp"]] for d in res["tpr_at_fpr"]],
            "pauc": [[d["pauc"], d["area"], math.nan, math.nan, math.nan] for d in res["pauc"]]}


def _equal(a, b, pauc_tol=0.0):
    """Same NaNs; every word equal, pAUC words within pauc_tol."""
    for kind in ("top_k", "tpr_at_fpr", "pauc"):
        assert len(a[kind]) == len(b[kind]), kind
        for wa, wb in zip(a[kind], b[kind]):
            wa, wb = np.asarray(wa, dtype=np.float64), np.asarray(wb, dtype=np.float64)
            assert np.array_equal(np.isnan(wa), np.isnan(wb)), (kind, wa, wb)
            tol = pauc_tol * (kind == "pauc")
            with np.errstate(invalid="ignore"):
                ok = (wa == wb) | (np.abs(wa - wb) <= tol)
            assert np.all(ok[~np.isnan(wa)]), (kind, wa, wb)


def _ks(p1, y):
    """K = 1, P, n and K's whose K-th highest score sits inside a tie group (the largest group and the one at the
    middle position), so that the cut splits the group."""
    s, lo, hi = _groups(p1)
    n, P = len(s), int(np.asarray(y).sum())
    ks = [1, n] + ([P] if P else [])
    big = np.flatnonzero(hi - lo >= 3)
    if big.size:
        mid = int(np.searchsorted(lo, n // 2, side="right")) - 1
        for g in {int(big[np.argmax((hi - lo)[big])]), mid if hi[mid] - lo[mid] >= 3 else int(big[0])}:
            ks.append(n - (int(lo[g]) + 1))           # c = n - K = lo + 1: inside the group
    return ks


def test_brute_force_agrees_with_sklearn_and_every_tie_order():
    """CPU: the brute force's pAUC against roc_auc_score(max_fpr), TPR at FPR against a scan of roc_curve's cuts, and
    the top-K counts against the average over every ordering of the tied group at the cut."""
    from sklearn.metrics import roc_auc_score, roc_curve

    rng = np.random.default_rng(11)
    for n in (2, 9, 60, 700):
        for q in (None, 5):
            p1 = rng.random(n).astype(np.float32)
            if q:
                p1 = (np.round(p1 * q) / q).astype(np.float32)
            y = (rng.random(n) < 0.3).astype(np.int64)
            y[0], y[1] = 1, 0
            P, N = int(y.sum()), n - int(y.sum())
            ref = _brute(p1, y, [], FPRS, MAX_FPRS)
            for f, w in zip(MAX_FPRS, ref["pauc"]):
                want = roc_auc_score(y, p1.astype(np.float64), max_fpr=f)
                assert abs(w[0] - want) <= 1e-12, (n, q, f, w[0], want)
            fpr, tpr, thr = roc_curve(y, p1.astype(np.float64), drop_intermediate=False)
            fps, tps = np.rint(fpr * N), np.rint(tpr * P)
            for f, w in zip(FPRS, ref["tpr_at_fpr"]):
                i = np.flatnonzero(fps <= f * N)[-1]  # roc_curve's first point is (0, 0) at threshold inf
                assert w == [tps[i] / P, fps[i] / N, float(thr[i]), tps[i], fps[i]], (n, q, f)
    # every ordering of the tied group at the cut
    for trial in range(30):
        n = int(rng.integers(3, 12))
        p1 = rng.integers(0, 3, n).astype(np.float32)
        y = (rng.random(n) < 0.5).astype(np.int64)
        for K in range(1, n + 1):
            t = np.sort(p1)[n - K]
            above, tied = p1 > t, p1 == t
            slots = K - int(above.sum())
            labels = y[tied]
            if len(labels) > 7:
                continue
            orders = list(itertools.permutations(labels))
            tp = int(y[above].sum()) + sum(sum(o[:slots]) for o in orders) / len(orders)
            got = _top_k(p1, y, K)
            assert abs(got[3] - tp) <= 1e-12 and got[2] == float(t), (trial, K)
            assert abs(got[1] - tp / K) <= 1e-12
            if y.sum():
                assert abs(got[0] - tp / y.sum()) <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 8192, 8193, 100_000, 3_000_000])
@pytest.mark.parametrize("kind", ["random", "quantised", "one_class", "all_positive"])
def test_operating_points_against_brute_force_and_sklearn(n, kind):
    from sklearn.metrics import roc_auc_score
    from test_gpu_eval_pass import _same
    from test_gpu_rank_metrics import _inputs

    from pcgnn_b200.metrics import device_metrics, device_operating_points

    p1, p0, y = _inputs(n, kind)
    prob = torch.from_numpy(np.stack([p0, p1])).cuda()
    yt = torch.from_numpy(y).cuda()
    ks = _ks(p1, y)
    res = device_operating_points(prob, yt, top_k=ks, fpr=FPRS, max_fpr=MAX_FPRS)
    assert [d["k"] for d in res["top_k"]] == ks and [d["max_fpr"] for d in res["pauc"]] == list(MAX_FPRS)
    got = _words(res)
    _equal(got, _brute(p1, y, ks, FPRS, MAX_FPRS), pauc_tol=1e-12)
    again = _words(device_operating_points(prob, yt, top_k=ks, fpr=FPRS, max_fpr=MAX_FPRS))
    _equal(got, again)                                                   # bit-identical reruns
    m = device_metrics(prob, yt)
    P, N = int(y.sum()), n - int(y.sum())
    if P:
        k_eq_p = got["top_k"][ks.index(P)][0]
        assert np.float64(k_eq_p).tobytes() == np.float64(m["recall_at_k"]).tobytes()
    if P and N:
        assert abs(got["pauc"][-1][0] - m["auc"]) <= 1e-12               # max_fpr = 1 is the AUC
        for f, w in zip(MAX_FPRS, got["pauc"]):
            want = roc_auc_score(y, p1.astype(np.float64), max_fpr=f)
            assert abs(w[0] - want) <= 1e-12, (f, w[0], want)
    assert _same(m, device_metrics(prob, yt))


@pytest.mark.gpu
def test_abi_out_of_range_requests_write_nan_and_bad_calls_are_refused():
    """Requests the host checks of device_operating_points would refuse, written straight into the device arrays:
    each writes PCG_POINT_WORDS NaN while the valid requests around them are answered. Malformed calls fail on the
    host before any launch."""
    from pcgnn_b200 import _lib
    from pcgnn_b200.metrics import _run_metrics

    n = 5000
    rng = np.random.default_rng(5)
    prob = torch.from_numpy(rng.random((2, n), dtype=np.float32)).cuda()
    y = (rng.random(n) < 0.2).astype(np.int64)
    _, ws, _ = _run_metrics(prob, torch.from_numpy(y).cuda(), "test")
    kind = [0, 0, 0, 0, 0, 1, 1, 1, 2, 2, 2, 3, -1, 0, 1, 2]
    arg = [0.0, n + 1.0, 2.5, math.nan, -math.inf, -0.1, 1.5, math.nan, 0.0, 1.5, math.nan, 0.5, 1.0, 10.0, 0.1, 0.1]
    m = len(kind)
    kd = torch.tensor(kind, dtype=torch.int32, device="cuda")
    ad = torch.tensor(arg, dtype=torch.float64, device="cuda")
    L = _lib.lib()
    pws = torch.empty(int(L.pcg_binary_points_workspace_bytes(n, m)), dtype=torch.uint8, device="cuda")
    out = torch.zeros(m * _lib.POINT_WORDS, dtype=torch.float64, device="cuda")

    def call(m_=m, out_=out.data_ptr(), ws_bytes=pws.numel(), kind_=kd.data_ptr()):
        return L.pcg_binary_points(ws.data_ptr(), ws.numel(), n, kind_, ad.data_ptr(), m_, out_, pws.data_ptr(),
                                   ws_bytes, _lib.stream_ptr())

    _lib.check(call(), "pcg_binary_points")
    w = out.cpu().numpy().reshape(m, _lib.POINT_WORDS)
    assert np.isnan(w[:13]).all()
    ref = _brute(prob[1].cpu().numpy(), y, [10], [0.1], [0.1])
    _equal({"top_k": [w[13].tolist()], "tpr_at_fpr": [w[14].tolist()], "pauc": [w[15].tolist()]}, ref, pauc_tol=1e-12)
    for bad in (dict(m_=0), dict(m_=_lib.POINTS_MAX + 1), dict(out_=None), dict(kind_=None), dict(ws_bytes=8)):
        assert call(**bad) != 0, bad
    assert L.pcg_binary_points_workspace_bytes(n, 0) == 0


def _same_points(a, b):
    from test_gpu_eval_pass import _same

    return a.keys() == b.keys() and all(len(a[k]) == len(b[k]) and all(_same(x, z) for x, z in zip(a[k], b[k]))
                                        for k in a)


def _check_pass(model, nodes, labels):
    """A pass with requests against one without (words 0-20 bit-identical), its operating points against
    device_operating_points of its own probabilities, and new request values without a new recording."""
    from test_gpu_eval_pass import _same

    from pcgnn_b200 import _lib
    from pcgnn_b200.metrics import device_operating_points
    from pcgnn_b200.runtime import GraphedEvalPass

    n, P = len(nodes), int(np.sum(labels))
    ops = dict(top_k=[1, P, 100, n], fpr=[0.0, 0.01, 0.1], max_fpr=[0.01, 0.1, 1.0])
    plain = GraphedEvalPass(model, nodes, labels, 1024)
    ev = GraphedEvalPass(model, nodes, labels, 1024, operating_points=ops)
    m0, m1 = plain.run(), ev.run()
    assert "operating_points" not in m0
    assert _same(m0, {k: m1[k] for k in _lib.METRICS_KEYS})
    yt = torch.from_numpy(np.asarray(labels)).cuda()
    assert _same_points(m1["operating_points"], device_operating_points(ev.probs().t(), yt, **ops))
    assert m1["operating_points"]["top_k"][1]["recall"] == m1["recall_at_k"]
    assert abs(m1["operating_points"]["pauc"][-1]["pauc"] - m1["auc"]) <= 1e-12
    new = dict(top_k=[2, P // 2 + 1, 500, n - 1], fpr=[0.001, 0.05, 1.0], max_fpr=[0.001, 0.3, 0.5])
    ev.set_operating_points(**new)
    m2 = ev.run()
    assert ev.captures == 1
    assert _same(m0, {k: m2[k] for k in _lib.METRICS_KEYS})
    assert [d["k"] for d in m2["operating_points"]["top_k"]] == new["top_k"]
    assert _same_points(m2["operating_points"], device_operating_points(ev.probs().t(), yt, **new))
    with pytest.raises(ValueError):
        ev.set_operating_points(top_k=[1], fpr=[0.1], max_fpr=[0.1])
    with pytest.raises(ValueError):
        ev.set_operating_points(top_k=[0, 1, 2, 3], fpr=[0.1, 0.2, 0.3], max_fpr=[0.1, 0.2, 0.3])
    with pytest.raises(_lib.PcgError):
        plain.set_operating_points(top_k=[1])
    with pytest.raises(ValueError):
        GraphedEvalPass(model, nodes, labels, 1024, operating_points=dict(top_k=[n + 1]))
    return m2, ev


@pytest.mark.gpu
def test_c2_pass_operating_points():
    from test_gpu_eval_pass import _model

    d, _, model = _model("yelp", seed=72)
    nodes = np.asarray(d.idx_rest)
    _check_pass(model, nodes, d.labels[nodes])


@pytest.mark.gpu
def test_c4_graphsage_operating_points_on_log_probabilities():
    from test_gpu_eval_pass_baselines import _build

    from pcgnn_b200.synth import make_graph

    d = make_graph("amazon", seed=72)
    model, _, _ = _build("sage", d.feat, d.homo, E=64, seed=72)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    m, ev = _check_pass(model, nodes, labels)
    lp = ev.probs()[:, 1].cpu().numpy()
    assert (lp <= 0).all()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = _brute(lp, labels, [d_["k"] for d_ in m["operating_points"]["top_k"]],
                     [d_["max_fpr"] for d_ in m["operating_points"]["tpr_at_fpr"]],
                     [d_["max_fpr"] for d_ in m["operating_points"]["pauc"]])
    _equal(_words(m["operating_points"]), ref, pauc_tol=1e-12)           # thresholds are log-probabilities
