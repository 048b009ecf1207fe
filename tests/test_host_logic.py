"""CPU: host-side logic of the product (graph formats, synthetic data, capacity sizing, sampler weights,
the import shim). No kernels are called."""
import importlib
import random
import sys

import numpy as np
import pytest

from oracle import c_oracle, ref_harness as H
from pcgnn_b200 import _lib
from pcgnn_b200.graph import RelGraph, adj_lists_from_csr, csr_from_edges
from pcgnn_b200.synth import make_graph


def test_csr_matches_sparse_to_adjlist_rules():
    """Self loop on every node, both directions, duplicates merged, rows sorted (utils.py:233-239)."""
    n = 7
    src, dst = [0, 0, 3, 3, 5], [1, 1, 4, 0, 5]
    ip, ix = csr_from_edges(n, src, dst)
    adj = adj_lists_from_csr(ip, ix)
    assert adj[0] == {0, 1, 3} and adj[1] == {0, 1} and adj[3] == {0, 3, 4} and adj[6] == {6}
    for v in range(n):
        row = ix[ip[v]:ip[v + 1]]
        assert np.all(np.diff(row) > 0)


def test_from_adj_lists_roundtrip_with_numpy_integer_members():
    d = make_graph("tiny", seed=1)
    adj = d.graph.to_adj_lists()
    adj = [{np.int64(k): {np.int32(x) for x in v} for k, v in a.items()} for a in adj]
    g2 = RelGraph.from_adj_lists(adj, d.graph.n_nodes)
    assert np.array_equal(g2.indptr, d.graph.indptr) and np.array_equal(g2.indices, d.graph.indices)
    u = d.graph.union()
    for v in (0, 5, 77):
        want = set().union(*[set(d.graph.row(r, v).tolist()) for r in range(3)])
        assert set(u.row(0, v).tolist()) == want


def test_synthetic_shapes_follow_the_spec():
    d = make_graph("tiny_amz", seed=2)
    assert d.feat.shape == (900, 25) and d.graph.n_rel == 3
    assert d.labels[:100].sum() == 0 and min(d.idx_train) >= 100          # unlabeled prefix excluded
    assert np.allclose(d.feat.sum(1), d.feat.sum(1))                         # finite
    assert abs(len(d.idx_train) / 800 - 0.4) < 0.02
    assert set(d.train_pos) == {v for v, y in zip(d.idx_train, d.y_train) if y == 1}
    assert all(int(d.graph.degrees(r).min()) >= 1 for r in range(3))        # self loops


def test_pick_weights_and_replay_equal_random_choices():
    from pcgnn_b200.utils import pick_weights
    from oracle import port

    d = make_graph("tiny", seed=4)
    w = pick_weights(d.idx_train, d.y_train, d.homo)
    homo = d.homo.to_adj_lists()[0]
    y = d.y_train
    lf = (y.sum() - len(y)) * y + len(y)
    assert np.array_equal(w, np.array([len(homo[v]) for v in d.idx_train]) / lf)
    random.seed(11)
    want = random.choices(d.idx_train, weights=w, k=200)
    random.seed(11)
    u = [random.random() for _ in range(200)]
    assert port.pick_step_replay(d.idx_train, w, u) == want


def _oracle_slots(graph, score, nodes, pool, train):
    sp, _ = c_oracle.choose(graph, score, nodes, np.ones(len(nodes), bool), pool=pool, train=train)
    return int(((np.diff(sp) + _lib.SLOT - 1) // _lib.SLOT).sum())


def test_slots_bound_is_an_upper_bound_of_the_oracle_sizes():
    d = make_graph("tiny", seed=5, dup_feature_frac=0.2)
    rng = np.random.default_rng(0)
    nodes = rng.choice(d.idx_train, 100)
    score = rng.normal(size=d.feat.shape[0]).astype(np.float32)
    pool = sorted(d.train_pos)
    need = _oracle_slots(d.graph, score, nodes, pool, True)
    total = int(d.graph.choose_slot_demand([0.5] * 3, 0.5, len(pool), True)[nodes].sum())
    assert total >= need


def test_choose_slot_demand_is_the_oracle_demand_in_eval_mode():
    """Unique targets, rows of several slots: in eval mode an item fills exactly the slots of its k kept ids. Train mode
    reserves k + o slots per item before the union with the pool, so there the demand is only a bound."""
    d = make_graph("amazon", seed=72)
    rng = np.random.default_rng(0)
    nodes = rng.choice(np.unique(d.idx_train), 256, replace=False)
    score = rng.normal(size=d.feat.shape[0]).astype(np.float32)
    pool = sorted(d.train_pos)
    for train in (False, True):
        demand = d.graph.choose_slot_demand([0.5] * 3, 0.5, len(pool), train)
        got, need = int(demand[nodes].sum()), _oracle_slots(d.graph, score, nodes, pool, train)
        assert (got >= need) if train else (got == need), (train, got, need)
        assert d.graph.choose_slot_demand([0.5] * 3, 0.5, len(pool), train) is demand        # memoised


def test_select_all_slot_demand_is_whole_rows_in_slots():
    """Per node, each relation's row in 64-id slots, and one slot for an empty row (it may take the target itself)."""
    deg = ([0, 1, 63, 64, 65, 128, 129, 0], [0, 0, 1, 64, 0, 200, 1, 65])
    ips = [np.concatenate([[0], np.cumsum(dr)]) for dr in deg]
    g = RelGraph(8, ips, [np.zeros(ip[-1], dtype=np.int32) for ip in ips])
    assert g.select_all_slot_demand().tolist() == [1 + 1, 1 + 1, 1 + 1, 1 + 1, 2 + 1, 2 + 4, 3 + 1, 1 + 2]


def test_shim_routes_reference_imports_to_this_package():
    import pcgnn_b200.shim as shim
    from pcgnn_b200 import layers, utils

    try:
        shim.install(reference_root=H.REF_ROOT if H.available() else None)
        assert importlib.import_module("src.layers") is layers
        assert importlib.import_module("src.utils").pick_step is utils.pick_step
        gs = importlib.import_module("src.graphsage")
        for name in ("nn", "Variable", "torch", "F", "init", "random", "GCN", "GraphSage", "MeanAggregator",
                     "Encoder", "GCNAggregator", "GCNEncoder"):
            assert hasattr(gs, name), name                  # model_handler.py gets these via `import *`
        mod = importlib.import_module("src.model")
        assert hasattr(mod, "PCALayer")
        if H.available():
            assert mod.__file__.startswith(H.REF_ROOT)      # the reference's own model.py, unchanged
    finally:
        shim.uninstall()


@pytest.mark.skipif(not H.available(), reason="reference tree not present")
def test_reference_model_handler_imports_through_the_shim():
    """`from src.model_handler import ModelHandler` resolves every hot-path name to this package."""
    import pcgnn_b200.shim as shim
    from pcgnn_b200 import layers

    if H.REF_ROOT not in sys.path:
        sys.path.insert(0, H.REF_ROOT)
    try:
        shim.install(reference_root=H.REF_ROOT)
        mh = importlib.import_module("src.model_handler")
        assert mh.InterAgg3 is layers.InterAgg3 and mh.IntraAgg is layers.IntraAgg
        assert mh.pick_step.__module__.endswith("utils") and "pcgnn" in mh.pick_step.__module__
        assert mh.PCALayer.__module__ == "src.model"
    finally:
        shim.uninstall()


def test_big_graph_generator_is_partition_independent():
    """C5 generator: any rank can make any row range; labels, split, pool and features agree everywhere."""
    import torch
    from pcgnn_b200.synth_big import BigSpec, make_partition

    mk = lambda rows, rank, world: make_partition(BigSpec(nodes_per_rank=rows, feat_dim=4, rel_mean_deg=(2.0, 5.0, 9.0),
                                                          max_degree=5000, seed=3), rank, world, "cpu")
    full = mk(6000, 0, 1)
    ipf, ixf = full.graph.device("cpu")
    parts = [mk(2000, r, 3) for r in range(3)]
    for part in parts:
        assert torch.equal(part.train_pos, full.train_pos) and torch.equal(part.labels, full.labels)
        assert torch.equal(part.feat, full.feat)
        ip, ix = part.graph.device("cpu")
        lo, n = part.row_lo, part.graph.n_nodes
        for r in range(3):
            a = ixf[ipf[r * 6000 + lo]:ipf[r * 6000 + lo + n]]
            b = ix[ip[r * n]:ip[(r + 1) * n]]
            assert torch.equal(a, b)
        nodes, lab = part.sample_batches(1, 512, seed=1)[0]
        assert int(nodes.min()) >= lo and int(nodes.max()) < lo + n
        assert 0.35 < float(lab.float().mean()) < 0.65          # label-balanced like pick_step
    rows = ixf[ipf[5]:ipf[6]]
    assert 5 in rows.tolist() and bool((rows[1:] > rows[:-1]).all())   # self loop, ascending ids


def test_pos_neg_split_keeps_order_and_matches_the_reference():
    """utils.pos_neg_split (utils.py:256-271): ids with label 1 / the rest, both in `nodes` order."""
    from pcgnn_b200.utils import pos_neg_split

    rng = np.random.default_rng(0)
    nodes = rng.permutation(500)[:300].tolist()
    labels = (rng.random(300) < 0.2).astype(np.int64)
    pos, neg = pos_neg_split(nodes, labels)
    assert pos == [n for n, y in zip(nodes, labels) if y == 1]
    assert neg == [n for n, y in zip(nodes, labels) if y != 1]
    assert sorted(pos + neg) == sorted(nodes)
    assert pos_neg_split([], []) == ([], [])
    if H.available():
        ref_utils = H.load(canonical=False).utils
        rpos, rneg = ref_utils.pos_neg_split(list(nodes), labels)
        assert list(rpos) == pos and list(rneg) == neg


def test_from_scipy_applies_self_loops_and_symmetrisation():
    """RelGraph.from_scipy == sparse_to_adjlist's dict of sets (utils.py:226-254): identity added, both
    directions, rows ascending; directed input, duplicate entries and explicit zeros included."""
    import scipy.sparse as sp

    rng = np.random.default_rng(1)
    n = 60
    mats = []
    for nnz in (80, 400):
        r, c = rng.integers(0, n, nnz), rng.integers(0, n, nnz)
        mats.append(sp.csc_matrix((np.ones(nnz), (r, c)), shape=(n, n)))      # directed, with duplicates
    g = RelGraph.from_scipy(mats)
    assert g.n_rel == 2 and g.n_nodes == n
    for r, m in enumerate(mats):
        dense = (m.toarray() != 0)
        want = dense | dense.T | np.eye(n, dtype=bool)
        for v in range(n):
            row = g.row(r, v)
            assert np.array_equal(row, np.nonzero(want[v])[0])
    one = RelGraph.from_scipy(mats[0])
    assert one.n_rel == 1 and np.array_equal(one.indices, g.relation(0)[1])
    if H.available():
        ref_utils = H.load(canonical=False).utils
        adj = ref_utils.sparse_to_adjlist_for_train(mats[1])
        for v in range(n):
            assert set(int(x) for x in adj[v]) == set(g.row(1, v).tolist())


def test_bench_deals_every_target_once_and_balances_row_length():
    """bench.deal: the ranks' shards partition the global batch, have equal sizes and near-equal neighbour counts."""
    import bench

    rng = np.random.default_rng(0)
    weight = (rng.pareto(1.2, 5000) * 20 + 1).astype(np.int64)          # power-law row lengths
    nodes = rng.integers(0, 5000, 1024)
    labels = rng.integers(0, 2, 1024)
    for world in (2, 4, 8):
        parts = [bench.deal(nodes, labels, weight, r, world) for r in range(world)]
        assert sorted(np.concatenate([p[0] for p in parts]).tolist()) == sorted(nodes.tolist())
        assert all(len(p[0]) == 1024 // world for p in parts)
        loads = np.array([weight[p[0]].sum() for p in parts], dtype=np.float64)
        contiguous = np.array([weight[nodes[r * (1024 // world):(r + 1) * (1024 // world)]].sum() for r in range(world)])
        assert loads.max() / loads.mean() <= contiguous.max() / contiguous.mean() + 1e-9
        assert loads.max() - loads.min() <= weight[nodes].max()           # greedy dealing: off by at most one target
        for (n, l) in parts:                                             # labels stay attached to their nodes
            idx = [np.nonzero(nodes == v)[0] for v in n]
            assert all(l[j] in labels[i] for j, i in enumerate(idx))


def test_device_metrics_equal_sklearn():
    """metrics.binary_metrics (the device-side replacement of the sklearn calls in utils.test, utils.py:316-325)."""
    import torch
    from sklearn.metrics import f1_score, precision_score, recall_score, roc_auc_score

    from pcgnn_b200.metrics import binary_metrics

    rng = np.random.default_rng(0)
    for n, quant in ((500, None), (2000, 20), (64, 3)):
        y = (rng.random(n) < 0.2).astype(np.int64)
        s = np.clip(rng.normal(0.3 + 0.25 * y, 0.2), 0, 1)
        if quant:
            s = np.round(s * quant) / quant                  # many tied scores
        pred = (s > 0.5).astype(np.int64)
        m = binary_metrics(torch.from_numpy(s), torch.from_numpy(pred), torch.from_numpy(y))
        assert abs(m["auc"] - roc_auc_score(y, s)) < 1e-12
        assert abs(m["f1"] - f1_score(y, pred, zero_division=0)) < 1e-12
        assert abs(m["f1_macro"] - f1_score(y, pred, average="macro", zero_division=0)) < 1e-12
        assert abs(m["recall"] - recall_score(y, pred, zero_division=0)) < 1e-12
        assert abs(m["precision"] - precision_score(y, pred, zero_division=0)) < 1e-12
        assert abs(m["recall_macro"] - recall_score(y, pred, average="macro", zero_division=0)) < 1e-12
        assert abs(m["precision_macro"] - precision_score(y, pred, average="macro", zero_division=0)) < 1e-12
        assert abs(m["accuracy"] - (pred == y).mean()) < 1e-12
    # degenerate: nothing predicted positive -> zero_division=0 convention
    y = np.array([0, 1, 0, 1]); pred = np.zeros(4, dtype=np.int64); s = np.array([.1, .2, .3, .4])
    m = binary_metrics(torch.from_numpy(s), torch.from_numpy(pred), torch.from_numpy(y))
    assert m["f1"] == 0.0 and m["precision"] == 0.0 and m["recall"] == 0.0
    assert abs(m["auc"] - roc_auc_score(y, s)) < 1e-12


def test_fastloop_routes_on_cpu():
    """fastloop (host logic only, no kernels): the loss subclass keeps its autograd node; backward() without arguments
    stores the recorded gradients only while enabled; every other use, and every optimizer the hook does not recognise,
    goes through torch's own code."""
    import torch

    from pcgnn_b200 import fastloop

    def make():
        ws = [torch.nn.Parameter(torch.ones(3)), torch.nn.Parameter(torch.ones(2, 2))]
        loss = ws[0].sum() * 2 + ws[1].sum() * 3
        flat = torch.arange(8.0)
        return ws, fastloop.wrap(loss, flat, [(0, 3, (3,)), (4, 4, (2, 2))], ws), flat

    assert not fastloop.enabled()
    ws, loss, _ = make()
    assert isinstance(loss, fastloop.StepLoss) and loss.grad_fn is not None and float(loss.item()) == 18.0
    loss.backward()                                              # not enabled: autograd
    assert torch.equal(ws[0].grad, torch.full((3,), 2.0)) and torch.equal(ws[1].grad, torch.full((2, 2), 3.0))

    fastloop.enable()
    try:
        fastloop.enable()                                        # idempotent
        ws, loss, flat = make()
        loss.backward()                                          # enabled: the recorded gradients, no engine
        assert torch.equal(ws[0].grad, torch.tensor([0.0, 1.0, 2.0]))
        assert torch.equal(ws[1].grad, torch.tensor([[4.0, 5.0], [6.0, 7.0]]))
        flat.add_(100.0)                                         # the static buffer is rewritten by the next replay ...
        assert torch.equal(ws[0].grad, torch.tensor([0.0, 1.0, 2.0]))        # ... the handed-out gradients are a copy
        # an optimizer the hook does not take over: torch's own step consumes those gradients
        opt = torch.optim.SGD(ws, lr=1.0)
        opt.step()
        assert torch.equal(ws[0].detach(), torch.tensor([1.0, 0.0, -1.0])) and "_pcg_flat" not in opt.__dict__
        ws, loss, _ = make()
        opt = torch.optim.Adam(ws, lr=0.1, amsgrad=True)         # Adam variant outside the kernel's formula: left alone
        loss.backward()
        opt.step()
        assert "_pcg_flat" not in opt.__dict__ and len(opt.state) == 2
        # second backward on the same loss accumulates like autograd; explicit gradient / scaled loss: torch's route
        ws, loss, _ = make()
        loss.backward(retain_graph=True)
        loss.backward()
        assert torch.equal(ws[0].grad, torch.tensor([0.0, 2.0, 4.0]))
        ws, loss, _ = make()
        loss.backward(torch.tensor(2.0))
        assert torch.equal(ws[0].grad, torch.full((3,), 4.0))
        ws, loss, _ = make()
        (loss * 0.5).backward()
        assert torch.equal(ws[1].grad, torch.full((2, 2), 1.5))
    finally:
        fastloop.disable()
    assert not fastloop.enabled()
