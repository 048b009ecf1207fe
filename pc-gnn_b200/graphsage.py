"""GraphSAGE / GCN baselines on the same aggregation kernels — same surface as
/root/reference/src/graphsage.py (MeanAggregator :42-96, Encoder :99-150, GraphSage :16-39,
GCNAggregator :181-232, GCNEncoder :234-275, GCN :154-178).

The reference's ``model_handler.py`` does ``from src.graphsage import *`` and picks up ``nn``,
``Variable``, ``torch``, ``F``, ``init`` and ``random`` through it (model_handler.py:13, 85, 150),
so this module re-exports those names too (no ``__all__`` on purpose).

The aggregators take the whole neighbour row of every target (∪ self for GCN), i.e. the select-all
mode of the kernels: no copy of the id lists, the aggregation warps read the CSR directly. Graph
input: ``adj_lists`` may be the reference's dict-of-sets (converted once) or a ``RelGraph``.
"""
import random

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Variable
from torch.nn import init

from . import _lib
from .engine import Engine
from .graph import RelGraph
from .layers import _AggregateFn, _feature_table


class _EncoderFn(torch.autograd.Function):
    """relu(W @ X^T) -> [E,B] with X = aggregated rows (or [self | aggregate]) as one kernel per direction
    (``pcg_encoder_fwd`` / ``_bwd``); frozen feature table (model_handler.py:85-86). Reference: graphsage.py:145-149,
    :274."""

    @staticmethod
    def forward(ctx, engine, agg, targets, weight):
        weight = weight.contiguous()
        out = engine.encoder_fwd(agg, weight, targets)
        ctx.engine, ctx.targets, ctx.w_ptr = engine, targets, weight.data_ptr()
        ctx.save_for_backward(agg, out)
        return out

    @staticmethod
    def backward(ctx, d_out):
        agg, out = ctx.saved_tensors
        eng = ctx.engine
        sink = eng.grad_sink.get(ctx.w_ptr) if eng.grad_sink is not None else None
        d_w = eng.encoder_bwd(agg, out, d_out, ctx.targets, sink)
        return None, None, None, (None if sink is not None else d_w)


def _encoder_fits(enc, eng) -> bool:
    """Whether pcg_encoder_fwd / _bwd take this encoder: the weight and a tile of targets fit in shared memory."""
    return (enc.weight.shape[1] * (eng.ldf + 33) + enc.weight.numel()) * 4 <= 190 * 1024


def _encode(enc, nodes, with_self):
    """Shared forward of Encoder / GCNEncoder: aggregate, then the encoder kernel when the feature table is frozen
    (the reference's setup) or the torch ops when it trains."""
    agg_mod = enc.aggregator
    neigh_feats = agg_mod.forward(nodes, _Rows(len(nodes)))
    eng = agg_mod._engine
    table = getattr(enc.features, "weight", None)
    native = (eng is not None and isinstance(table, torch.Tensor) and not table.requires_grad and neigh_feats.is_cuda
              and agg_mod.last_targets is not None and neigh_feats.shape[0] > 0 and neigh_feats.shape[1] == eng.F
              and _encoder_fits(enc, eng))
    if native:
        full = agg_mod.last_agg          # [B, ldf] as the kernel wrote it (row stride ldf)
        return _EncoderFn.apply(eng, full, agg_mod.last_targets if with_self else None, enc.weight)
    if with_self:
        dev = neigh_feats.device
        index = nodes.to(dev) if isinstance(nodes, torch.Tensor) else torch.as_tensor(
            np.asarray([int(v) for v in nodes]), device=dev, dtype=torch.long)
        combined = torch.cat((enc.features(index.long()), neigh_feats), dim=1)
    else:
        combined = neigh_feats
    return F.relu(enc.weight.mm(combined.t()))


class _Rows:
    """Stand-in for the list of neighbour sets the reference builds per batch
    (`[self.adj_lists[int(node)] for node in nodes]`, graphsage.py:133, 267): the kernels read the
    rows from the CSR, so nothing is materialised."""

    def __init__(self, n):
        self._n = n

    def __len__(self):
        return self._n


class _RowAggregator(nn.Module):
    """Shared machinery: normalised sum over whole CSR rows of a single-relation graph."""

    _norm = _lib.NORM_MEAN

    def _setup(self, features, cuda):
        self.features = features
        self.cuda = cuda
        self._graph = None
        self._graph_src = None
        self._engine = None
        self.cap_slots_hint = None      # fixed slot capacity (CUDA-graph use); else sized from the host ids
        self.last_selection = None
        self.last_agg = self.last_targets = None    # the padded aggregate / device ids of the last call (encoder kernels)

    def bind_graph(self, adj_lists):
        """Give the aggregator the graph its rows come from (the encoders call this once)."""
        if adj_lists is not self._graph_src:
            self._graph_src = adj_lists
            self._graph = adj_lists if isinstance(adj_lists, RelGraph) else None
            self._engine = None

    def _device(self):
        w = getattr(self.features, "weight", None)
        return w.device if isinstance(w, torch.Tensor) else torch.device("cuda", torch.cuda.current_device())

    def _get_engine(self):
        dev = self._device()
        if self._engine is None or self._engine.device != dev:
            if self._graph is None:
                self._graph = RelGraph.from_adj_lists([self._graph_src])
            self._engine = Engine(self._graph, dev)
        return self._engine

    def _run(self, eng, targets, cap, add_self, n_table=None):
        table = _feature_table(self.features, eng.N if n_table is None else n_table, eng.device)
        eng.set_features(table)
        sel = eng.select_all(targets, add_self, cap, self._norm)
        self.last_selection = sel
        agg = _AggregateFn.apply(table, eng, sel, table.shape[1]) if table.requires_grad else eng.aggregate(sel)
        self.last_agg, self.last_targets = agg, (targets if n_table is None else None)
        return agg[:, :table.shape[1]]

    def _aggregate(self, nodes, to_neighs, add_self):
        if self._graph_src is None or not isinstance(to_neighs, _Rows):
            return self._aggregate_lists(nodes, to_neighs, add_self)
        eng = self._get_engine()
        targets, host = eng.upload_targets(nodes)
        if self.cap_slots_hint is not None:
            cap = int(self.cap_slots_hint)
        else:
            cap = self.slots_bound(targets.cpu().numpy() if host is None else host)
        return self._run(eng, targets, cap, add_self)

    def slots_bound(self, nodes) -> int:
        """Slot capacity that covers a batch of node ids (the graph's per-node select-all demand, summed)."""
        return int(self._get_engine().graph.select_all_slot_demand()[np.asarray(nodes, dtype=np.int64)].sum())

    def _aggregate_lists(self, nodes, to_neighs, add_self):
        """Explicit neighbour sets (stand-alone aggregator use, or sub-sampled rows): a one-off graph
        whose row i is the i-th set, so duplicate targets keep their own rows."""
        rows = {}
        for i, s in enumerate(to_neighs):
            s = set(int(x) for x in s)
            if add_self:
                s.add(int(nodes[i]))       # graphsage.py:79 / :210
            rows[i] = s
        n_ids = 1 + max((max(s) for s in rows.values() if s), default=0)
        eng = Engine(RelGraph.from_adj_lists([rows], max(n_ids, len(rows))), self._device())
        eng.strict_rows = False            # graph rows are batch positions, not node ids
        targets = torch.arange(len(rows), dtype=torch.int32, device=eng.device)
        cap = int(eng.graph.select_all_slot_demand()[:len(rows)].sum())
        return self._run(eng, targets, cap, False, n_table=n_ids)


class MeanAggregator(_RowAggregator):
    """Mean of the neighbours' rows (graphsage.py:42-96). With gcn=True the target joins its own
    neighbourhood (:78-79)."""

    def __init__(self, features, cuda=False, gcn=False):
        super().__init__()
        self._setup(features, cuda)
        self.gcn = gcn

    def forward(self, nodes, to_neighs, num_sample=None):
        if num_sample is not None:
            # graphsage.py:70-75: sub-sample rows longer than num_sample with Python's `random`
            # (never enabled by the reference's Encoder, :133).
            if isinstance(to_neighs, _Rows):
                g = self._get_engine().graph
                to_neighs = [set(g.row(0, int(n)).tolist()) for n in nodes]
            to_neighs = [set(random.sample(sorted(tn), num_sample)) if len(tn) >= num_sample else set(tn)
                         for tn in to_neighs]
            return self._aggregate_lists(nodes, to_neighs, self.gcn)
        return self._aggregate(nodes, to_neighs, self.gcn)


class GCNAggregator(_RowAggregator):
    """Neighbours ∪ {self}, divided by sqrt(count) (graphsage.py:181-232)."""

    _norm = _lib.NORM_RSQRT

    def __init__(self, features, cuda=False):
        super().__init__()
        self._setup(features, cuda)

    def forward(self, nodes, to_neighs):
        return self._aggregate(nodes, to_neighs, True)


class Encoder(nn.Module):
    """GraphSAGE encoder (graphsage.py:99-150): relu(W @ [self | mean(neigh)]^T), or without the
    self half when gcn=True."""

    def __init__(self, features, feature_dim, embed_dim, adj_lists, aggregator, num_sample=10, base_model=None,
                 gcn=False, cuda=False, feature_transform=False):
        super().__init__()
        self.features = features
        self.feat_dim = feature_dim
        self.adj_lists = adj_lists
        self.aggregator = aggregator
        if base_model is not None:
            self.base_model = base_model
        self.gcn = gcn
        self.embed_dim = embed_dim
        self.cuda = cuda
        self.aggregator.cuda = cuda
        self.aggregator.bind_graph(adj_lists)
        self.weight = nn.Parameter(torch.FloatTensor(embed_dim, self.feat_dim if self.gcn else 2 * self.feat_dim))
        init.xavier_uniform_(self.weight)

    def forward(self, nodes):
        return _encode(self, nodes, with_self=not self.gcn)


class GCNEncoder(nn.Module):
    """GCN encoder (graphsage.py:234-275): relu(W[E,F] @ agg^T)."""

    def __init__(self, features, feature_dim, embed_dim, adj_lists, aggregator, base_model=None, cuda=False,
                 feature_transform=False):
        super().__init__()
        self.features = features
        self.feat_dim = feature_dim
        self.adj_lists = adj_lists
        self.aggregator = aggregator
        if base_model is not None:
            self.base_model = base_model
        self.embed_dim = embed_dim
        self.cuda = cuda
        self.aggregator.cuda = cuda
        self.aggregator.bind_graph(adj_lists)
        self.weight = nn.Parameter(torch.FloatTensor(embed_dim, self.feat_dim))
        init.xavier_uniform_(self.weight)

    def forward(self, nodes):
        return _encode(self, nodes, with_self=False)


class _Head(nn.Module):
    def __init__(self, num_classes, enc):
        super().__init__()
        self.enc = enc
        self.xent = nn.CrossEntropyLoss()
        self.weight = nn.Parameter(torch.FloatTensor(num_classes, enc.embed_dim))
        init.xavier_uniform_(self.weight)

    def forward(self, nodes):
        embeds = self.enc(nodes)
        return self.weight.mm(embeds).t()

    def loss(self, nodes, labels):
        embeds = self.enc(nodes)
        eng = getattr(self.enc.aggregator, "_engine", None)
        if (eng is not None and embeds.is_cuda and self.weight.shape[0] == 2 and embeds.shape[1] > 0
                and isinstance(self.xent, nn.CrossEntropyLoss) and isinstance(embeds.grad_fn, _EncoderFn._backward_cls)):
            # head + cross-entropy as one kernel per direction (pcg_head_loss_*, lambda = 0: no label-similarity term)
            from .layers import HeadLossFn, _as_device_labels

            lab = _as_device_labels(labels, embeds.device)
            center = torch.zeros((embeds.shape[1], 2), dtype=torch.float32, device=embeds.device)
            loss, _ = HeadLossFn.apply(eng, embeds, self.weight, center, lab, 0.0)
            return loss
        return self.xent(self.weight.mm(embeds).t(), labels.squeeze())


class GraphSage(_Head):
    """graphsage.py:16-39. (The reference's to_prob uses log_softmax(dim=2) on a 2-D tensor and
    raises; dim=1 is used here.)"""

    def to_prob(self, nodes, *unused, **unused_kw):
        return F.log_softmax(self.forward(nodes), dim=1)


class GCN(_Head):
    """graphsage.py:154-178."""

    def to_prob(self, nodes, *unused, **unused_kw):
        return torch.sigmoid(self.forward(nodes))
