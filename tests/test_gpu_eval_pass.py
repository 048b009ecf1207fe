"""GPU: runtime.GraphedEvalPass (a whole node set scored by replays of one recorded batch graph, metrics computed on the
device by pcg_binary_metrics) against the reference-facing path (model.to_prob, utils.test, metrics.binary_metrics),
sklearn and a numpy brute force; and the guarantee that evaluating between epochs leaves a recorded training run alone."""
import numpy as np
import pytest
import torch

from helpers import build_cuda_pcgnn, random_params

pytestmark = pytest.mark.gpu

BASE_KEYS = ("auc", "f1", "f1_macro", "recall", "precision", "recall_macro", "precision_macro", "accuracy", "gmean")
# metrics.binary_metrics divides F1's 2PR by (P + R).clamp_min(1.0), which understates F1 whenever P + R < 1; the
# kernel computes sklearn's F1, so those two keys are checked against sklearn and every other key against binary_metrics
F1_KEYS = ("f1", "f1_macro")


def _model(spec="tiny_amz", seed=71, E=64, **kw):
    from pcgnn_b200.synth import make_graph

    d = make_graph(spec, seed=seed, dup_feature_frac=0.1 if spec == "tiny_amz" else 0.0)
    rng = np.random.default_rng(seed)
    params = random_params(rng, d.feat.shape[1], E, d.graph.n_rel)
    return d, params, build_cuda_pcgnn(d.feat, d.graph, sorted(d.train_pos), params, **kw)


def _to_prob_batches(model, nodes, labels, B):
    """model.to_prob (no grad: the cached infer graph) on the pass's padded entries, rows of the real nodes only, and
    on the unpadded last batch."""
    from pcgnn_b200.runtime import pack_eval_plan

    plan = pack_eval_plan(nodes, B)
    n = len(nodes)
    padded, last = [], None
    with torch.no_grad():
        for e, ids in enumerate(plan):
            k = min(B, n - e * B)
            p = model.to_prob(ids.tolist(), np.zeros(B, np.int64), train_flag=False)[0]
            padded.append(p[:k])
        s = (len(plan) - 1) * B
        last = model.to_prob(list(nodes[s:]), labels[s:], train_flag=False)[0]
    return torch.cat(padded), last


def _check_probs(got, want):
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-7), float((got - want).abs().max())
    clear = (want[:, 1] - want[:, 0]).abs() > 1e-5
    assert torch.equal(got.argmax(1)[clear], want.argmax(1)[clear])


def _same(a: dict, b: dict):
    return a.keys() == b.keys() and all(np.array_equal(np.float64(a[k]), np.float64(b[k]), equal_nan=True) for k in a)


def test_probabilities_match_to_prob_on_padded_and_unpadded_batches():
    from pcgnn_b200.runtime import GraphedEvalPass

    d, _, model = _model()
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    B = 128
    assert len(nodes) % B != 0
    ev = GraphedEvalPass(model, nodes, labels, B)
    m = ev.run()
    got = ev.probs()
    assert got.shape == (len(nodes), 2)
    padded, last = _to_prob_batches(model, nodes, labels, B)
    _check_probs(got, padded)
    _check_probs(got[(ev.n_entries - 1) * B:], last)
    assert m["n_pos"] + m["n_neg"] == len(nodes) and m["n_pos"] == int(labels.sum())
    assert ev.captures == 1 and _same(m, ev.run()) and ev.captures == 1


def test_c2_validation_set_matches_to_prob_binary_metrics_and_utils_test():
    from sklearn.metrics import f1_score

    from pcgnn_b200.metrics import binary_metrics
    from pcgnn_b200.runtime import GraphedEvalPass
    from pcgnn_b200.utils import test as utils_test

    d, _, model = _model("yelp", seed=72)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    B = 1024
    ev = GraphedEvalPass(model, nodes, labels, B)
    assert ev.n_entries == 27 and len(nodes) == 27572
    m = ev.run()
    got = ev.probs().clone()
    padded, last = _to_prob_batches(model, nodes, labels, B)
    _check_probs(got, padded)
    _check_probs(got[(ev.n_entries - 1) * B:], last)
    # the pass's metrics are binary_metrics of its own probabilities
    y = torch.from_numpy(labels).cuda()
    ref = binary_metrics(got[:, 1], got.argmax(1), y)
    assert abs(m["auc"] - ref["auc"]) <= 1e-12 * abs(ref["auc"])
    for k in BASE_KEYS[1:]:
        if k not in F1_KEYS:
            assert abs(m[k] - ref[k]) <= 1e-12 * max(abs(ref[k]), 1e-300), k
    pred, yy = got[:, 1] > got[:, 0], y == 1
    assert m["tp"] == int((pred & yy).sum()) and m["fp"] == int((pred & ~yy).sum())
    assert m["tn"] == int((~pred & ~yy).sum()) and m["fn"] == int((~pred & yy).sum())
    yd, pd = labels, pred.long().cpu().numpy()
    assert abs(m["f1"] - f1_score(yd, pd, zero_division=0)) <= 1e-12
    assert abs(m["f1_macro"] - f1_score(yd, pd, average="macro", zero_division=0)) <= 1e-12
    # ... and agree with utils.test within what the near-tied nodes can move
    auc, recall, f1_macro, precision = utils_test(list(nodes), labels, model, B, print_line=False)
    ties = int(((got[:, 1] - got[:, 0]).abs() <= 1e-5).sum())
    tol = 1e-9 + 4.0 * ties / max(1.0, min(m["n_pos"], m["tp"] + m["fp"]))
    assert abs(auc - m["auc"]) <= 1e-4
    assert abs(recall - m["recall"]) <= tol and abs(precision - m["precision"]) <= tol
    assert abs(f1_macro - ref["f1_macro"]) <= tol            # utils.test reports binary_metrics' F1
    assert _same(m, ev.run())


def _best_threshold_numpy(p1, y):
    """Every distinct value t of p1 as a cut (positive iff p1 >= t), sklearn's macro-F1 (zero_division=0)."""
    order = np.argsort(p1, kind="stable")
    s, ys = p1[order].astype(np.float64), y[order].astype(np.int64)
    n, P = len(s), int(y.sum())
    N = n - P
    before = np.concatenate([[0], np.cumsum(ys)])
    starts = np.flatnonzero(np.concatenate([[True], s[1:] != s[:-1]]))
    best, at = -1.0, -1
    for j in starts:
        tp = float(P - before[j])
        fp = float(n - j) - tp
        fn, tn = float(P) - tp, float(N) - fp
        f = _macro(tp, fp, tn, fn)
        if f >= best:
            best, at = f, j
    return best, float(s[at])


def _macro(tp, fp, tn, fn):
    def r(a, b):
        return a / b if b > 0 else 0.0

    p1, r1, p0, r0 = r(tp, tp + fp), r(tp, tp + fn), r(tn, tn + fn), r(tn, tn + fp)
    return 0.5 * (r(2.0 * p1 * r1, p1 + r1) + r(2.0 * p0 * r0, p0 + r0))


@pytest.mark.parametrize("n", [1, 7, 8192, 8193, 100_000])
@pytest.mark.parametrize("kind", ["random", "quantised", "one_class"])
def test_metrics_kernel_against_binary_metrics_sklearn_and_brute_force(n, kind):
    from sklearn.metrics import f1_score, precision_score, recall_score, roc_auc_score

    from pcgnn_b200.metrics import binary_metrics, device_metrics

    rng = np.random.default_rng(n)
    p1, p0 = rng.random(n).astype(np.float32), rng.random(n).astype(np.float32)
    y = (rng.random(n) < 0.15).astype(np.int64)
    if n > 1:
        y[0], y[1] = 1, 0
    if kind == "quantised":
        p1, p0 = np.round(p1 * 20) / 20, np.round(p0 * 20) / 20     # heavy ties, also between p1 and p0
    if kind == "one_class":
        y[:] = 0
    prob = torch.from_numpy(np.stack([p0, p1]).astype(np.float32)).cuda()
    m = device_metrics(prob, torch.from_numpy(y).cuda())
    assert _same(m, device_metrics(prob, torch.from_numpy(y).cuda()))           # bit-identical reruns
    pred = (prob[1] > prob[0]).long()
    ref = binary_metrics(prob[1], pred, torch.from_numpy(y).cuda())
    for k in BASE_KEYS:
        if k in F1_KEYS:
            continue
        if np.isnan(ref[k]):
            assert np.isnan(m[k]), k
        else:
            assert abs(m[k] - ref[k]) <= 1e-12 * max(abs(ref[k]), 1e-300), (k, m[k], ref[k])
    p1d, yd, pd = prob[1].cpu().numpy().astype(np.float64), y, pred.cpu().numpy()
    if 0 < yd.sum() < n:
        assert abs(m["auc"] - roc_auc_score(yd, p1d)) <= 1e-12
    else:
        assert np.isnan(m["auc"])
    assert abs(m["f1_macro"] - f1_score(yd, pd, average="macro", labels=[0, 1], zero_division=0)) <= 1e-12
    assert abs(m["f1"] - f1_score(yd, pd, zero_division=0)) <= 1e-12
    assert abs(m["precision"] - precision_score(yd, pd, zero_division=0)) <= 1e-12
    assert abs(m["recall"] - recall_score(yd, pd, zero_division=0)) <= 1e-12
    best, t = _best_threshold_numpy(prob[1].cpu().numpy(), yd)
    assert m["best_f1_macro"] == best and m["best_threshold"] == t
    assert m["n_pos"] == yd.sum() and m["n_neg"] == n - yd.sum()


def test_metrics_kernel_best_threshold_small_brute_force():
    """The cumulative form of the brute force above against the literal one (every cut evaluated from scratch)."""
    from pcgnn_b200.metrics import device_metrics

    rng = np.random.default_rng(5)
    for n in (2, 30, 500):
        p1 = np.round(rng.random(n) * 13) / 13
        y = (rng.random(n) < 0.3).astype(np.int64)
        best, at = -1.0, None
        for t in np.unique(p1.astype(np.float32)):
            pr = p1.astype(np.float32) >= t
            f = _macro(float((pr & (y == 1)).sum()), float((pr & (y == 0)).sum()), float((~pr & (y == 0)).sum()),
                       float((~pr & (y == 1)).sum()))
            if f >= best:
                best, at = f, float(t)
        prob = torch.from_numpy(np.stack([1 - p1, p1]).astype(np.float32)).cuda()
        m = device_metrics(prob, torch.from_numpy(y).cuda())
        assert m["best_f1_macro"] == best and m["best_threshold"] == at


def test_evaluation_between_epochs_leaves_training_bit_identical():
    from pcgnn_b200.parallel import FusedAdam, GradAllReduce
    from pcgnn_b200.runtime import GraphedEvalPass, GraphedTrainStep

    d, params, _ = _model(seed=73)
    rng = np.random.default_rng(73)
    B, n_steps, epochs = 128, 4, 3
    batches = [rng.choice(d.idx_train, B) for _ in range(n_steps)]
    nodes = np.arange(d.feat.shape[0])
    runs = []
    for with_eval in (False, True):
        model = build_cuda_pcgnn(d.feat, d.graph, sorted(d.train_pos), params)
        evals = []
        if with_eval:
            ev = GraphedEvalPass(model, nodes, d.labels[nodes], 1024)
            evals.append((ev.run(), ev.probs().clone()))          # recorded on the parameters' original storage
        reducer = GradAllReduce(model.parameters()).attach()
        opt = FusedAdam(reducer, lr=0.01, weight_decay=1e-3)      # moves every parameter into its flat buffer
        eng = model.inter1.engine()
        eng.set_features(model.inter1.features.weight)
        cap = GraphedTrainStep.plan(eng, batches, model.inter1.thresholds, 0.5)
        step = GraphedTrainStep(model, opt, B, cap, reducer=reducer, warmup_batch=(batches[0], d.labels[batches[0]]))
        step.load_plan([(b, d.labels[b]) for b in batches])
        losses = []
        for _ in range(epochs):
            for _ in range(n_steps):
                step.run_planned()
            losses.append(step.plan_losses().clone())
            if with_eval:
                evals.append((ev.run(), ev.probs().clone()))
        assert not step.overflowed()
        weights = torch.cat([p.detach().reshape(-1) for p in model.parameters() if p.requires_grad]).cpu()
        runs.append((torch.stack(losses).cpu(), weights))
        if with_eval:
            assert ev.captures == 2                               # the storage move re-recorded once
            assert not torch.equal(evals[0][1], evals[1][1])      # replays read the trained weights
            assert not torch.equal(evals[1][1], evals[2][1])
            fresh = GraphedEvalPass(model, nodes, d.labels[nodes], 1024)
            assert _same(fresh.run(), evals[-1][0]) and torch.equal(fresh.probs(), evals[-1][1])
    assert torch.equal(runs[0][0], runs[1][0])
    assert torch.equal(runs[0][1], runs[1][1])


def test_refusals():
    from pcgnn_b200 import _lib
    from pcgnn_b200.runtime import GraphedEvalPass

    d, params, model = _model(seed=74)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    # too few slots: the overflow words of the batches make run() raise, and nothing else is disturbed
    want = GraphedEvalPass(model, nodes, labels, 128)
    m = want.run()
    tiny = GraphedEvalPass(model, nodes, labels, 128, cap_slots=1)
    with pytest.raises(_lib.PcgError, match="cap_slots"):
        tiny.run()
    assert _same(want.run(), m)
    with pytest.raises(ValueError, match="at least one node"):
        GraphedEvalPass(model, [], [], 128)
    with pytest.raises(ValueError, match="0 or 1"):
        GraphedEvalPass(model, nodes, labels * 2, 128)
    # shapes the fused kernels do not cover, a trainable feature table, a row partition
    d96, _, m96 = _model(seed=74, E=96)
    with pytest.raises(_lib.PcgError, match="pcg_tile_supported"):
        GraphedEvalPass(m96, nodes, labels, 128)
    _, _, trainable = _model(seed=74, trainable_features=True)
    with pytest.raises(_lib.PcgError, match="trainable"):
        GraphedEvalPass(trainable, nodes, labels, 128)
    part = build_cuda_pcgnn(d.feat, d.graph.row_partition(0, d.feat.shape[0] // 2), sorted(d.train_pos), params)
    with pytest.raises(_lib.PcgError, match="partitioned"):
        GraphedEvalPass(part, nodes, labels, 128)
    with pytest.raises(_lib.PcgError, match="PCALayer"):
        GraphedEvalPass(model.inter1, nodes, labels, 128)
