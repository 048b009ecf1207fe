"""GPU: runtime.GraphedEvalPass on the GCN / GraphSAGE baselines (select-all, aggregate, pcg_encoder_fwd and
pcg_eval_head in one recorded batch graph) against the modules' own to_prob, the oracle port, utils.test,
metrics.binary_metrics, sklearn and a numpy brute force; its independence of the batching; weights changing under it;
and its refusals."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import rel_err
from oracle import port
from test_gpu_eval_pass import _best_threshold_numpy, _same

pytestmark = pytest.mark.gpu

KINDS = ("gcn", "sage", "sage_self", "sage_agg_self")
BASE_KEYS = ("auc", "recall", "precision", "recall_macro", "precision_macro", "accuracy", "gmean")


def _graph_with_missing_self_loops(homo):
    """The union graph with the self loop of every other node removed (where the row keeps other entries), so that
    the aggregators' union with the target itself adds an id for half of the nodes."""
    from pcgnn_b200.graph import RelGraph

    n, ip, ix = homo.n_nodes, homo.indptr, homo.indices
    row = np.repeat(np.arange(n), np.diff(ip))
    deg = np.diff(ip)
    keep = ~((ix == row) & (row % 2 == 0) & (deg[row] > 1))
    counts = np.bincount(row[keep], minlength=n)
    return RelGraph(n, [np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)], [ix[keep].astype(np.int32)])


def _build(kind, feat, graph, E=64, seed=0, trainable=False, n_classes=2):
    """(model, enc_w, head_w): GCN(GCNEncoder(GCNAggregator)); GraphSage as the reference builds it
    (model_handler.py:97-98: MeanAggregator, Encoder(gcn=True)), with the self concat (Encoder(gcn=False)), or with
    MeanAggregator(gcn=True)."""
    import torch.nn as nn

    from pcgnn_b200 import graphsage as gs

    rng = np.random.default_rng(seed)
    F_ = feat.shape[1]
    features = nn.Embedding(*feat.shape)
    features.weight = nn.Parameter(torch.from_numpy(np.ascontiguousarray(feat)), requires_grad=trainable)
    features = features.cuda()
    if kind == "gcn":
        enc = gs.GCNEncoder(features, F_, E, graph, gs.GCNAggregator(features, cuda=True), cuda=True)
        model = gs.GCN(n_classes, enc)
    else:
        agg = gs.MeanAggregator(features, cuda=True, gcn=kind == "sage_agg_self")
        enc = gs.Encoder(features, F_, E, graph, agg, gcn=kind != "sage_self", cuda=True)
        model = gs.GraphSage(n_classes, enc)
    enc_w = port.xavier(rng, E, enc.weight.shape[1])
    head = port.xavier(rng, n_classes, E)
    with torch.no_grad():
        enc.weight.copy_(torch.from_numpy(enc_w))
        model.weight.copy_(torch.from_numpy(head))
    return model.cuda(), enc_w, head


class _PortSAGEWithSelf(port.PortSAGE):
    """MeanAggregator(gcn=True): the mean over the row united with the target itself (graphsage.py:78-79)."""

    def encode(self, nodes):
        picked = [set(self.graph.row(0, v).tolist()) | {v} for v in nodes]
        return F.relu(self.enc_w.mm(port._dense_mask_agg(self.feat, picked, "mean").t()))


def _port_probs(kind, feat, graph, enc_w, head, nodes):
    if kind == "gcn":
        pm = port.PortGCN(feat, graph, enc_w, head)
    elif kind == "sage_agg_self":
        pm = _PortSAGEWithSelf(feat, graph, enc_w, head)
    else:
        pm = port.PortSAGE(feat, graph, enc_w, head, concat_self=kind == "sage_self")
    with torch.no_grad():
        logits = pm.forward([int(v) for v in nodes])
    return torch.sigmoid(logits) if kind == "gcn" else F.log_softmax(logits, dim=1)


def _to_prob(model, nodes, B):
    """model.to_prob over the batches utils.test makes (no padding), concatenated."""
    nodes = [int(v) for v in nodes]
    with torch.no_grad():
        return torch.cat([model.to_prob(nodes[s:s + B]) for s in range(0, len(nodes), B)])


def _check(got, want, kind):
    atol = 1e-7 if kind == "gcn" else 1e-6            # GraphSage: log-probabilities
    assert torch.allclose(got, want, rtol=1e-5, atol=atol), float((got - want).abs().max())
    clear = (want[:, 1] - want[:, 0]).abs() > 1e-5
    assert torch.equal(got.argmax(1)[clear], want.argmax(1)[clear])


def _tiny(seed=81):
    from pcgnn_b200.synth import make_graph

    d = make_graph("tiny_amz", seed=seed)
    return d, _graph_with_missing_self_loops(d.homo)


@pytest.mark.parametrize("kind", KINDS)
def test_probabilities_match_to_prob_and_the_port(kind):
    from pcgnn_b200.runtime import GraphedEvalPass

    d, graph = _tiny()
    model, enc_w, head = _build(kind, d.feat, graph)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    B = 128
    assert len(nodes) % B != 0
    ev = GraphedEvalPass(model, nodes, labels, B)
    m = ev.run()
    got = ev.probs().clone()
    assert got.shape == (len(nodes), 2)
    _check(got, _to_prob(model, nodes, B), kind)
    assert rel_err(got.cpu().numpy(), _port_probs(kind, d.feat, graph, enc_w, head, nodes).numpy()) <= 1e-5
    assert m["n_pos"] == int(labels.sum()) and m["n_neg"] == len(nodes) - int(labels.sum())
    assert ev.captures == 1 and _same(m, ev.run()) and torch.equal(ev.probs(), got) and ev.captures == 1


@pytest.mark.parametrize("kind", KINDS)
def test_probabilities_do_not_depend_on_the_batching(kind):
    """Every row's arithmetic is the target's own (its slots in order, fixed encoder and head chains): the same node
    gives the same bits at any batch size, at any position, with any padding, and repeated."""
    from pcgnn_b200.runtime import GraphedEvalPass

    d, graph = _tiny()
    model, _, _ = _build(kind, d.feat, graph)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    B = 128
    ev = GraphedEvalPass(model, nodes, labels, B)
    ev.run()
    full = ev.probs().clone()
    one = GraphedEvalPass(model, nodes, labels, len(nodes))   # one entry, no padding
    one.run()
    assert torch.equal(one.probs(), full)
    rng = np.random.default_rng(3)
    rep = rng.choice(len(nodes), 300)
    rep[:3] = rep[3]
    for pick in (np.arange(1), np.arange(B), np.arange(B + 1), rep):
        sub = GraphedEvalPass(model, nodes[pick], labels[pick], B)
        m = sub.run()
        assert torch.equal(sub.probs(), full[torch.from_numpy(pick).cuda()]), len(pick)
        assert m["n_pos"] == int(labels[pick].sum())


@pytest.mark.parametrize("kind", ["gcn", "sage"])
def test_c4_metrics_match_binary_metrics_sklearn_utils_test_and_brute_force(kind):
    from sklearn.metrics import f1_score

    from pcgnn_b200.metrics import binary_metrics
    from pcgnn_b200.runtime import GraphedEvalPass
    from pcgnn_b200.synth import make_graph
    from pcgnn_b200.utils import test as utils_test

    d = make_graph("amazon", seed=72)
    model, _, _ = _build(kind, d.feat, d.homo, E=64, seed=72)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    B = 1024
    ev = GraphedEvalPass(model, nodes, labels, B)
    assert ev.n_entries == 6 and len(nodes) == 5184
    m = ev.run()
    got = ev.probs().clone()
    _check(got, _to_prob(model, nodes, B), kind)
    # the pass's metrics are binary_metrics of its own probabilities (log-probabilities for GraphSage)
    y = torch.from_numpy(labels).cuda()
    ref = binary_metrics(got[:, 1], got.argmax(1), y)
    for k in BASE_KEYS:
        assert abs(m[k] - ref[k]) <= 1e-12 * max(abs(ref[k]), 1e-300), k
    pred, yy = got[:, 1] > got[:, 0], y == 1
    assert m["tp"] == int((pred & yy).sum()) and m["fp"] == int((pred & ~yy).sum())
    assert m["tn"] == int((~pred & ~yy).sum()) and m["fn"] == int((~pred & yy).sum())
    pd = pred.long().cpu().numpy()
    assert abs(m["f1"] - f1_score(labels, pd, zero_division=0)) <= 1e-12
    assert abs(m["f1_macro"] - f1_score(labels, pd, average="macro", zero_division=0)) <= 1e-12
    best, t = _best_threshold_numpy(got[:, 1].cpu().numpy(), labels)
    assert m["best_f1_macro"] == best and m["best_threshold"] == t
    auc, _, _, _ = utils_test(list(nodes), labels, model, B, print_line=False)
    assert abs(auc - m["auc"]) <= 1e-4
    assert _same(m, ev.run())


def test_weight_updates_rebinding_and_module_state():
    """An in-place optimizer step is read by the next run() without a new recording; binding the aggregator to another
    graph re-records; the aggregator's own per-call state is what it was before."""
    from pcgnn_b200.runtime import GraphedEvalPass
    from pcgnn_b200.synth import make_graph

    d, graph = _tiny()
    model, _, _ = _build("gcn", d.feat, graph)
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    agg = model.enc.aggregator
    with torch.no_grad():
        model.to_prob(nodes[:50].tolist())
    before = {k: getattr(agg, k) for k in ("cap_slots_hint", "last_selection", "last_agg", "last_targets")}
    ev = GraphedEvalPass(model, nodes, labels, 128)
    ev.run()
    first = ev.probs().clone()
    for k, v in before.items():
        assert getattr(agg, k) is v, k
    opt = torch.optim.Adam(model.parameters(), lr=0.05)
    model.loss(nodes[:128].tolist(), torch.from_numpy(labels[:128]).cuda()).backward()
    opt.step()
    ev.run()
    assert ev.captures == 1 and not torch.equal(ev.probs(), first)
    _check(ev.probs(), _to_prob(model, nodes, 128), "gcn")
    other = make_graph("tiny_amz", seed=82).homo
    agg.bind_graph(other)
    model.enc.adj_lists = other
    ev.run()
    assert ev.captures == 2
    _check(ev.probs(), _to_prob(model, nodes, 128), "gcn")


def test_gcn_training_run_with_evaluations_between_epochs():
    """FusedAdam moves the parameters into its flat buffer (the pass re-records once); a GCN epoch plan run with
    evaluations between its epochs gives the same losses and weights, bit for bit, as the same run without them."""
    from pcgnn_b200.parallel import FusedAdam, GradAllReduce
    from pcgnn_b200.runtime import GraphedEvalPass, GraphedTrainStep

    d, graph = _tiny(seed=83)
    rng = np.random.default_rng(83)
    B, n_steps, epochs = 128, 4, 3
    batches = [rng.choice(d.idx_train, B) for _ in range(n_steps)]
    nodes = np.arange(d.feat.shape[0])
    runs = []
    for with_eval in (False, True):
        model, _, _ = _build("gcn", d.feat, graph, seed=83)
        agg = model.enc.aggregator
        evals = []
        if with_eval:
            ev = GraphedEvalPass(model, nodes, d.labels[nodes], 256)
            evals.append((ev.run(), ev.probs().clone()))
        reducer = GradAllReduce(model.parameters()).attach()
        opt = FusedAdam(reducer, lr=0.01, weight_decay=1e-3)
        agg._get_engine().set_features(agg.features.weight)
        cap = max(agg.slots_bound(b) for b in batches)
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
        assert agg.cap_slots_hint == cap
        weights = torch.cat([p.detach().reshape(-1) for p in model.parameters() if p.requires_grad]).cpu()
        runs.append((torch.stack(losses).cpu(), weights))
        if with_eval:
            assert ev.captures == 2
            assert not torch.equal(evals[0][1], evals[1][1]) and not torch.equal(evals[1][1], evals[2][1])
            fresh = GraphedEvalPass(model, nodes, d.labels[nodes], 256)
            assert _same(fresh.run(), evals[-1][0]) and torch.equal(fresh.probs(), evals[-1][1])
    assert torch.equal(runs[0][0], runs[1][0])
    assert torch.equal(runs[0][1], runs[1][1])


def test_overflow_and_refusals():
    from pcgnn_b200 import _lib
    from pcgnn_b200.runtime import GraphedEvalPass

    d, graph = _tiny()
    nodes = np.asarray(d.idx_rest)
    labels = d.labels[nodes]
    model, _, _ = _build("sage", d.feat, graph)
    want = GraphedEvalPass(model, nodes, labels, 128)
    m = want.run()
    tiny = GraphedEvalPass(model, nodes, labels, 128, cap_slots=100)
    with pytest.raises(_lib.PcgError, match=r"cap_slots=100 .*first: entry 0"):
        tiny.run()
    assert _same(want.run(), m)
    for kind, kw, match in (("sage", dict(trainable=True), "trainable"),
                            ("sage_self", dict(E=1024), "pcg_encoder_fwd"),
                            ("gcn", dict(n_classes=3), "two-class")):
        bad, _, _ = _build(kind, d.feat, graph, **kw)
        with pytest.raises(_lib.PcgError, match=match):
            GraphedEvalPass(bad, nodes, labels, 128)
    half = d.feat.shape[0] // 2
    part, _, _ = _build("gcn", d.feat, graph.row_partition(0, half))
    inside = nodes[nodes < half]
    with pytest.raises(_lib.PcgError, match="partitioned"):
        GraphedEvalPass(part, inside, d.labels[inside], 128)
    with pytest.raises(_lib.PcgError, match="GCN over GCNEncoder"):
        GraphedEvalPass(model.enc, nodes, labels, 128)
