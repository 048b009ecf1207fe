"""CPU: the evaluation plan of the GCN / GraphSAGE baselines (padding with the set's lowest-degree node, because
pcg_select_all aggregates every padding row's whole neighbour row) and which baseline builds runtime.GraphedEvalPass
takes."""
import numpy as np
import pytest

from pcgnn_b200.runtime import pack_eval_plan


def _indptr(degrees):
    return np.concatenate([[0], np.cumsum(degrees)]).astype(np.int64)


@pytest.mark.parametrize("n,B", [(1, 4), (3, 4), (5, 2), (9, 4), (5184, 1024)])
def test_baseline_plan_pads_with_the_sets_lowest_degree_node(n, B):
    rng = np.random.default_rng(n)
    N = 10 * n
    deg = rng.integers(2, 500, N)
    nodes = rng.permutation(N)[:n]
    deg[nodes[n // 2]] = 1                                   # the set's unique shortest row, in the middle of the set
    plan = pack_eval_plan(nodes.tolist(), B, _indptr(deg))
    k = -(-n // B)
    assert plan.dtype == np.int32 and plan.shape == (k, B)
    flat = plan.reshape(-1)
    assert np.array_equal(flat[:n], nodes)
    assert (flat[n:] == nodes[n // 2]).all()


def test_ties_go_to_the_first_such_node_in_the_given_order():
    deg = np.array([5, 1, 7, 1, 3])
    plan = pack_eval_plan([4, 3, 0, 1], 3, _indptr(deg))
    assert plan.reshape(-1).tolist() == [4, 3, 0, 1, 3, 3]


def test_full_entries_need_no_padding():
    nodes = np.arange(16)[::-1]
    assert np.array_equal(pack_eval_plan(nodes, 4, _indptr(np.arange(1, 17))), pack_eval_plan(nodes, 4))


def test_ids_outside_the_graph_raise():
    with pytest.raises(ValueError, match="not a row"):
        pack_eval_plan([0, 1, 5], 2, _indptr([1, 1, 1, 1, 1]))


def test_c4_last_entry_slot_demand():
    """C4 (amazon union graph, idx_rest, B = 1024): the last entry holds 64 nodes and 960 padding rows. Every padding
    row costs the slots of its node's whole row, so the set's shortest row (306 entries) keeps that entry at about half
    the slots of a full one; the entry's first id as the padding made it cost as much as a full entry."""
    from pcgnn_b200.synth import make_graph

    d = make_graph("amazon", seed=72)
    ip = d.homo.indptr
    nodes = np.asarray(d.idx_rest)
    B = 1024
    slots = lambda ids: int(d.homo.select_all_slot_demand()[ids].sum())

    plan = pack_eval_plan(nodes, B, ip)
    assert plan.shape == (6, B) and len(nodes) == 5184
    pad = plan[-1, -1]
    assert ip[pad + 1] - ip[pad] == (ip[nodes + 1] - ip[nodes]).min()
    assert slots(plan[-1]) == slots(nodes[5 * B:]) + (6 * B - len(nodes)) * slots(np.array([pad]))
    full = max(slots(e) for e in plan[:-1])
    assert slots(plan[-1]) < 0.5 * full <= slots(pack_eval_plan(nodes, B)[-1])


def test_which_baseline_builds_the_pass_takes():
    import torch
    import torch.nn as nn

    from pcgnn_b200 import _lib
    from pcgnn_b200 import graphsage as gs
    from pcgnn_b200.graph import RelGraph
    from pcgnn_b200.runtime import _baseline_parts

    g = RelGraph(3, [np.array([0, 1, 2, 3])], [np.array([0, 1, 2], dtype=np.int32)])
    features = nn.Embedding(3, 4)
    features.weight = nn.Parameter(torch.zeros(3, 4), requires_grad=False)

    def sage(agg_self, enc_gcn):
        agg = gs.MeanAggregator(features, gcn=agg_self)
        return gs.GraphSage(2, gs.Encoder(features, 4, 8, g, agg, gcn=enc_gcn)), agg

    gcn_agg = gs.GCNAggregator(features)
    gcn = gs.GCN(2, gs.GCNEncoder(features, 4, 8, g, gcn_agg))
    assert _baseline_parts(gcn) == (gcn_agg, True, False, 0)
    for agg_self in (False, True):
        for enc_gcn in (True, False):
            model, agg = sage(agg_self, enc_gcn)
            assert _baseline_parts(model) == (agg, agg_self, not enc_gcn, 1)
    mixed = gs.GCN(2, gs.Encoder(features, 4, 8, g, gs.MeanAggregator(features), gcn=True))
    for other in (mixed, gcn.enc, gcn_agg, nn.Linear(2, 2)):
        with pytest.raises(_lib.PcgError, match="GCN over GCNEncoder"):
            _baseline_parts(other)
