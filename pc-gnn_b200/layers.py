"""PC-GNN layers on the B200-native kernels — same public surface as /root/reference/src/layers.py.

  InterAgg1 / InterAgg3 / InterAgg5 (features, feature_dim, embed_dim, train_pos, adj_lists, intraggs,
                                     inter='GNN', cuda=True)       reference: layers.py:417, :161, :16
      .forward(nodes, labels, train_flag=True) -> (combined [E,B], center_scores [B,2])  (:207-291)
  IntraAgg(features, feat_dim, embed_dim, train_pos, rho, cuda=False)                    (:539-560)
      .forward(nodes, batch_labels, to_neighs_list, batch_scores, neigh_scores, pos_scores,
               sample_list, train_flag) -> (to_feats [B,E], samp_scores)                 (:562-630)
  choose_step_neighs(...), choose_step_test(...)                                         (:633-738)

Parameter names, shapes and state_dict keys are the reference's, so its ``model.py`` /
``model_handler.py`` (and checkpoints) work unchanged. What differs is where the work happens: the
neighbour lookup, label-aware filter, oversampling, set union and mean aggregation are CUDA kernels
over an HBM-resident CSR (``engine.Engine``); nothing is computed on the host and there is no CPU
path (constructing on a machine without the built extension / a GPU raises at first use).

Tie rule (the reference's is implementation-defined, SURVEY.md F6): equal distances are ordered by
neighbour id, pool ties by position in ``train_pos``.
"""
from __future__ import annotations

from itertools import chain

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn import init

from . import _lib
from .engine import Engine
from .graph import RelGraph, item_slots

__all__ = ["InterAgg1", "InterAgg3", "InterAgg5", "InterAgg", "IntraAgg", "choose_step_neighs",
           "choose_step_test", "HeadLossFn", "TrainStepFn"]


# ------------------------------------------------------------------------------------------------
class _AggregateFn(torch.autograd.Function):
    """agg = engine.aggregate(selection); differentiable w.r.t. the feature table only when that
    table is trainable (the reference freezes it, model_handler.py:85-86)."""

    @staticmethod
    def forward(ctx, table, engine, sel, feat_dim):
        feat = engine.set_features(table)
        ctx.engine, ctx.sel, ctx.feat_dim, ctx.shape = engine, sel, feat_dim, tuple(feat.shape)
        return engine.aggregate(sel, feat)

    @staticmethod
    def backward(ctx, d_agg):
        g = torch.zeros(ctx.shape, dtype=torch.float32, device=d_agg.device)
        ctx.engine.aggregate_bwd(ctx.sel, d_agg, g)
        return g[:, :ctx.feat_dim], None, None, None


class _DenseFn(torch.autograd.Function):
    """combined [E,B] = relu(cat(self, relu(cat(self, agg_r) @ W_r) ...) @ W).t() as ONE kernel (``pcg_dense_fwd``),
    with the weight gradients as the backward (``pcg_dense_bwd``). Used when the feature table is frozen, which
    is the reference's configuration (model_handler.py:85-86); reference math: layers.py:616-629, 273-289."""

    @staticmethod
    def forward(ctx, engine, targets, agg, agg_rep, feat_dim, w_inter, *w_intra):
        w_intra = [w.contiguous() for w in w_intra]
        w_inter = w_inter.contiguous()
        out, cat = engine.dense_fwd(targets, agg, w_intra, w_inter, feat_dim, agg_rep)
        ctx.engine, ctx.feat_dim, ctx.n_rel, ctx.agg_rep = engine, feat_dim, len(w_intra), agg_rep
        ctx.w_ptrs = [w_inter.data_ptr()] + [w.data_ptr() for w in w_intra]
        ctx.save_for_backward(agg, w_inter, cat, out)
        return out

    @staticmethod
    def backward(ctx, d_out):
        agg, w_inter, cat, out = ctx.saved_tensors
        eng = ctx.engine
        sinks = None
        if eng.grad_sink is not None:          # gradients go straight into the flat buffer (see Engine.grad_sink)
            views = [eng.grad_sink.get(q) for q in ctx.w_ptrs]
            if all(v is not None for v in views):
                sinks = (views[0], views[1:])
        d_intra, d_inter = eng.dense_bwd(agg, w_inter, cat, out, d_out, ctx.feat_dim, ctx.n_rel, ctx.agg_rep, sinks)
        if sinks is not None:
            return (None,) * (6 + ctx.n_rel)
        return (None, None, None, None, None, d_inter, *d_intra)


class _CenterFn(torch.autograd.Function):
    """center_scores [B,2] = label_clf(features[batch]) (layers.py:236-243) as one kernel, with label_clf's
    weight / bias gradients as the backward (the feature table is frozen)."""

    @staticmethod
    def forward(ctx, engine, targets, weight, bias):
        weight = weight.contiguous()
        ctx.engine, ctx.targets = engine, targets
        ctx.w_ptrs = (weight.data_ptr(), bias.data_ptr())
        return engine.center_fwd(targets, weight, bias)

    @staticmethod
    def backward(ctx, d_center):
        eng = ctx.engine
        sinks = None
        if eng.grad_sink is not None:
            views = (eng.grad_sink.get(ctx.w_ptrs[0]), eng.grad_sink.get(ctx.w_ptrs[1]))
            if views[0] is not None and views[1] is not None:
                sinks = views
        d_w, d_b = eng.center_bwd(ctx.targets, d_center, sinks)
        if sinks is not None:
            return None, None, None, None
        return None, None, d_w, d_b


class HeadLossFn(torch.autograd.Function):
    """PCALayer's head and loss (model.py:38, :54-61) as one kernel per direction:
    loss = CE(W @ combined, y) + lambda * CE(center_scores, y)."""

    @staticmethod
    def forward(ctx, engine, combined, weight, center, labels, lam):
        combined, weight, center = combined.contiguous(), weight.contiguous(), center.contiguous()
        loss, logits, p1, q1 = engine.head_loss_fwd(combined, weight, center, labels, lam)
        ctx.engine, ctx.lam = engine, lam
        ctx.w_ptr = weight.data_ptr()
        ctx.save_for_backward(combined, weight, labels, p1, q1)
        ctx.mark_non_differentiable(logits)
        return loss, logits

    @staticmethod
    def backward(ctx, d_loss, _d_logits):
        combined, weight, labels, p1, q1 = ctx.saved_tensors
        eng = ctx.engine
        sink = eng.grad_sink.get(ctx.w_ptr) if eng.grad_sink is not None else None
        d_emb, d_center, d_w = eng.head_loss_bwd(combined, weight, labels, p1, q1, ctx.lam, d_loss, sink)
        return None, d_emb, (None if sink is not None else d_w), d_center, None, None


class _TileFn(torch.autograd.Function):
    """(combined [E,B], center_scores [B,2]) = relation transforms + combine + label_clf head as ONE kernel
    (``pcg_tile_fwd``: activations stay in shared memory, weights stream in by TMA bulk copies); backward =
    the weight gradients (``pcg_dense_bwd``, ``pcg_center_bwd``). Frozen feature table (model_handler.py:85-86);
    reference math: layers.py:616-629, 273-289, 236-243."""

    @staticmethod
    def forward(ctx, engine, targets, agg, agg_rep, feat_dim, need_grad, clf_w, clf_b, w_inter, *w_intra):
        w_intra = [w.contiguous() for w in w_intra]
        w_inter, clf_w = w_inter.contiguous(), clf_w.contiguous()
        out, center, cat = engine.tile_fwd(targets, agg, agg_rep, w_intra, w_inter, clf_w, clf_b, need_grad)
        ctx.engine, ctx.feat_dim, ctx.n_rel, ctx.agg_rep, ctx.targets = engine, feat_dim, len(w_intra), agg_rep, targets
        ctx.w_ptrs = [w_inter.data_ptr()] + [w.data_ptr() for w in w_intra]
        ctx.clf_ptrs = (clf_w.data_ptr(), clf_b.data_ptr())
        if need_grad:
            ctx.save_for_backward(agg, w_inter, cat, out)
        return out, center

    @staticmethod
    def backward(ctx, d_out, d_center):
        agg, w_inter, cat, out = ctx.saved_tensors
        eng = ctx.engine
        n_in = 9 + ctx.n_rel
        grads = [None] * n_in
        if d_center is not None:
            sinks = None
            if eng.grad_sink is not None:
                views = (eng.grad_sink.get(ctx.clf_ptrs[0]), eng.grad_sink.get(ctx.clf_ptrs[1]))
                sinks = views if views[0] is not None and views[1] is not None else None
            d_w, d_b = eng.center_bwd(ctx.targets, d_center, sinks)
            if sinks is None:
                grads[6], grads[7] = d_w, d_b
        if d_out is not None:
            sinks = None
            if eng.grad_sink is not None:
                views = [eng.grad_sink.get(q) for q in ctx.w_ptrs]
                sinks = (views[0], views[1:]) if all(v is not None for v in views) else None
            d_intra, d_inter = eng.dense_bwd(agg, w_inter, cat, out, d_out, ctx.feat_dim, ctx.n_rel, ctx.agg_rep, sinks)
            if sinks is None:
                grads[8] = d_inter
                grads[9:] = list(d_intra)
        return tuple(grads)


class TrainStepFn(torch.autograd.Function):
    """loss = CE(W_head @ combined, y) + lambda * CE(center_scores, y) (model.py:38, :54-61) with everything
    behind the aggregation in ONE pass (``pcg_tile_train``): in a training step dLoss == 1 is known at forward
    time, so the forward launch also produces every weight gradient; backward() only hands them out (scaled by
    the incoming gradient). With ``engine.grad_sink`` set the kernels store the gradients straight into the flat
    gradient buffer and backward() returns nothing."""

    @staticmethod
    def forward(ctx, engine, targets, labels, agg, agg_rep, lam, pdl, w_head, clf_w, clf_b, w_inter, *w_intra):
        params = [w_head, clf_w, clf_b, w_inter, *w_intra]
        cont = [w.contiguous() for w in params]
        sink = engine.grad_sink
        views = [sink.get(w.data_ptr()) for w in params] if sink is not None else None
        if views is not None and all(v is not None for v in views):
            g = views
            ctx.flat = None
            engine.grads_in_sinks = True      # backward() has nothing left to do (runtime.GraphedTrainStep skips it)
        else:
            sizes = [w.numel() for w in params]
            pad = [(n + 3) // 4 * 4 for n in sizes]          # 16-byte aligned starts for the float4 stores
            flat = torch.empty(sum(pad), dtype=torch.float32, device=engine.device)
            g, o = [], 0
            for w, n, q in zip(params, sizes, pad):
                g.append(flat[o:o + n].view_as(w))
                o += q
            ctx.flat, ctx.views = flat, g
        grads = dict(head=g[0], clf_w=g[1], clf_b=g[2], inter=g[3], intra=g[4:])
        loss, out, center, _ = engine.tile_train(targets, labels, agg, agg_rep, cont[4:], cont[3], cont[1], cont[2],
                                                 cont[0], lam, grads, pdl=pdl)
        ctx.n_in = 7 + len(params)
        ctx.mark_non_differentiable(out, center)
        return loss, out, center

    @staticmethod
    def backward(ctx, d_loss, _d_out, _d_center):
        if ctx.flat is None:
            return (None,) * ctx.n_in
        ctx.flat.mul_(d_loss)
        return (None,) * 7 + tuple(ctx.views)


def _feature_table(features, n_nodes, device, ids=None):
    """The [N,F] table behind the reference's `features` callable (an nn.Embedding in
    model_handler.py:85; any id->rows callable is accepted)."""
    if isinstance(features, nn.Embedding):
        return features.weight
    w = getattr(features, "weight", None)
    if isinstance(w, torch.Tensor) and w.dim() == 2 and (n_nodes is None or w.shape[0] >= n_nodes):
        return w
    if n_nodes is None:   # explicit-list call: the largest id mentioned bounds the table
        lists, nodes, pool = ids
        n_nodes = 1 + max(max((int(x) for x in chain.from_iterable(lists)), default=0),
                          max((int(v) for v in nodes), default=0), max((int(p) for p in pool), default=0))
    return features(torch.arange(n_nodes, device=device))


def _as_device_labels(labels, device):
    if labels is None:
        return None
    if not isinstance(labels, torch.Tensor):
        labels = torch.as_tensor(np.asarray(labels))
    return labels.to(device=device, dtype=torch.int64).reshape(-1).contiguous()


class IntraAgg(nn.Module):
    """Intra-relation aggregator (reference: layers.py:539-630). Holds W_r [2F,E]."""

    def __init__(self, features, feat_dim, embed_dim, train_pos, rho, cuda=False):
        super().__init__()
        self.features = features
        self.cuda = cuda
        self.feat_dim = feat_dim
        self.embed_dim = embed_dim
        self.train_pos = train_pos
        self.rho = rho
        self.weight = nn.Parameter(torch.FloatTensor(2 * self.feat_dim, self.embed_dim))
        init.xavier_uniform_(self.weight)
        self._engine = None

    def transform(self, self_feats, agg_feats):
        """relu(cat(self, agg) @ W_r)  (layers.py:625-629)."""
        return F.relu(torch.cat((self_feats, agg_feats), dim=1).mm(self.weight))

    def forward(self, nodes, batch_labels, to_neighs_list, batch_scores, neigh_scores, pos_scores, sample_list,
                train_flag):
        """Reference calling convention with explicit neighbour lists and scores (layers.py:562)."""
        dev = self.weight.device
        if self._engine is None or self._engine.device != dev:
            self._engine = Engine(None, dev)
        eng = self._engine
        sel, dist, meta = _choose_explicit(eng, batch_scores, batch_labels if train_flag else None, neigh_scores,
                                           to_neighs_list, pos_scores if train_flag else None,
                                           self.train_pos if train_flag else None, sample_list, self.rho, train_flag)
        table = _feature_table(self.features, None, dev, ids=(to_neighs_list, nodes, self.train_pos))
        agg = _AggregateFn.apply(table, eng, sel, self.feat_dim)
        idx = torch.as_tensor(np.asarray([int(v) for v in nodes]), device=dev, dtype=torch.long)
        to_feats = self.transform(self.features(idx), agg[:, :self.feat_dim])
        lab = _as_device_labels(batch_labels, dev) if train_flag else None
        return to_feats, _LazyScores(sel, dist, meta, lab, train_flag)


class _LazyScores:
    """`samp_scores` (layers.py:695, 736): list over targets of the distances of the chosen
    neighbours. InterAgg discards it (layers.py:268-270), so it is materialised only on access."""

    def __init__(self, sel, dist, meta, labels, train):
        self._args = (sel, dist, meta, labels, train)
        self._val = None

    def _get(self):
        if self._val is None:
            sel, dist, meta, labels, train = self._args
            lab = labels.cpu().numpy() if labels is not None else None
            self._val = _sets_and_scores(sel, dist, meta, lab, train)[1]
            self._args = None
        return self._val

    def __iter__(self):
        return iter(self._get())

    def __len__(self):
        return len(self._get())

    def __getitem__(self, i):
        return self._get()[i]


def _explicit_csr(neighs_list, neigh_scores, device):
    """Batch-local CSR (row i = neighbour ids of target i, ascending) + per-entry score column 0."""
    lens = np.fromiter((len(x) for x in neighs_list), dtype=np.int64, count=len(neighs_list))
    indptr = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=indptr[1:])
    ids = np.fromiter((int(x) for x in chain.from_iterable(neighs_list)), dtype=np.int64, count=int(indptr[-1]))
    rows = np.repeat(np.arange(len(lens), dtype=np.int64), lens)
    order = np.lexsort((ids, rows))
    flat = torch.cat([torch.as_tensor(s).reshape(-1, 2)[:, 0] for s in neigh_scores]).detach()
    entry_score = flat.to(device=device, dtype=torch.float32)[torch.from_numpy(order).to(device)].contiguous()
    return (torch.from_numpy(indptr).to(device), torch.from_numpy(ids[order].astype(np.int32)).to(device),
            entry_score, lens)


def _choose_explicit(eng, center_scores, center_labels, neigh_scores, neighs_list, minor_scores, minor_list,
                     sample_list, sample_rate, train):
    dev = eng.device
    B = len(neighs_list)
    indptr, indices, entry_score, lens = _explicit_csr(neighs_list, neigh_scores, dev)
    center = torch.as_tensor(center_scores).detach().to(dev, torch.float32).reshape(-1, 2)[:, 0].contiguous()
    k_list = np.asarray([int(k) for k in sample_list], dtype=np.int64)
    k_over = torch.from_numpy(k_list.astype(np.int32)).to(dev)
    sorted_pool = None
    P = 0
    if train and minor_list is not None and len(minor_list):
        pool = torch.as_tensor(np.asarray([int(p) for p in minor_list], dtype=np.int32)).to(dev)
        pool_score = torch.as_tensor(minor_scores).detach().to(dev, torch.float32).reshape(-1, 2)[:, 0].contiguous()
        P = int(pool.shape[0])
        sorted_pool = eng.sort_pool(pool, pool_score)
    oo = np.minimum((k_list * float(sample_rate)).astype(np.int64), P) if train else np.zeros_like(k_list)
    cap = int(item_slots(lens, k_list, sample_rate, P, train).sum()) + 1
    targets = torch.arange(B, dtype=torch.int32, device=dev)
    labels = _as_device_labels(center_labels, dev) if train else None
    sel, dist = eng.choose(targets, labels, train, [0.5], float(sample_rate), cap, entry_score=entry_score,
                           center_score=center, k_override=k_over, sorted_pool=sorted_pool,
                           indptr=indptr, indices=indices, n_nodes=B, n_rel=1,
                           max_degree=int(lens.max()) if B else 0, want_dist=True)
    return sel, dist, (lens, k_list, oo)


def _sets_and_scores(sel, dist, meta, labels_host, train):
    lens, k_list, oo = meta
    base = sel.it_base.cpu().numpy()
    m = sel.it_m.cpu().numpy()
    idx = sel.idx.cpu().numpy()
    dist = dist.cpu().numpy()
    sets, scores = [], []
    for i in range(sel.B):
        d, c = int(lens[i]), int(k_list[i])
        k = c if d > c + 1 else d
        sets.append(set(idx[base[i]:base[i] + m[i]].tolist()))
        seg = dist[base[i]:base[i] + k]
        row = np.sort(seg, kind="stable").tolist() if d > c + 1 else seg.tolist()
        if train and labels_host is not None and labels_host[i] == 1:
            o = int(oo[i])
            row = row + np.sort(dist[base[i] + k:base[i] + k + o], kind="stable").tolist()
        scores.append(row)
    return sets, scores


def choose_step_neighs(center_scores, center_labels, neigh_scores, neighs_list, minor_scores, minor_list, sample_list,
                       sample_rate):
    """Train-mode choose step with the reference's signature and return value (layers.py:633-697):
    (list of sets of kept ids, list of distance lists). The selection runs on the GPU; the host only
    formats the kernel's output into Python sets and ordered distance lists."""
    dev = torch.device("cuda", torch.cuda.current_device())
    eng = Engine(None, dev)
    sel, dist, meta = _choose_explicit(eng, center_scores, center_labels, neigh_scores, neighs_list, minor_scores,
                                       minor_list, sample_list, sample_rate, True)
    lab = _as_device_labels(center_labels, dev).cpu().numpy()
    return _sets_and_scores(sel, dist, meta, lab, True)


def choose_step_test(center_scores, neigh_scores, neighs_list, sample_list):
    """Eval-mode choose step (layers.py:700-738)."""
    dev = torch.device("cuda", torch.cuda.current_device())
    eng = Engine(None, dev)
    sel, dist, meta = _choose_explicit(eng, center_scores, None, neigh_scores, neighs_list, None, None, sample_list,
                                       0.0, False)
    return _sets_and_scores(sel, dist, meta, None, False)


# ------------------------------------------------------------------------------------------------
class InterAgg(nn.Module):
    """Inter-relation aggregator for any number of relations R (reference: three hand-unrolled
    copies InterAgg1 / InterAgg3 / InterAgg5, layers.py:417-535, :161-291, :16-158).

    adj_lists: the reference's ``list[dict[int -> set[int]]]`` (converted to a CSR once, here), or a
    ready ``graph.RelGraph`` (needed when a dict-of-sets is infeasible)."""

    n_relations = None

    def __init__(self, features, feature_dim, embed_dim, train_pos, adj_lists, intraggs, inter='GNN', cuda=True):
        super().__init__()
        R = len(intraggs)
        if self.n_relations is not None and R != self.n_relations:
            raise ValueError(f"{type(self).__name__} takes {self.n_relations} intra-aggregators, got {R}")
        self.features = features
        self.dropout = 0.6
        self.adj_lists = adj_lists
        for r, ia in enumerate(intraggs):
            setattr(self, f"intra_agg{r + 1}", ia)
            ia.cuda = cuda
        self.embed_dim = embed_dim
        self.feat_dim = feature_dim
        self.cuda = cuda
        self.train_pos = train_pos
        self.thresholds = [0.5] * R                      # layers.py:193 (hard-coded filter ratio)
        self.weight = nn.Parameter(torch.FloatTensor(self.embed_dim * R + self.feat_dim, self.embed_dim))
        init.xavier_uniform_(self.weight)
        self.label_clf = nn.Linear(self.feat_dim, 2)     # layers.py:200
        self.weights_log = []
        self.thresholds_log = [self.thresholds]
        self.relation_score_log = []
        self._R = R
        self._graph = adj_lists if isinstance(adj_lists, RelGraph) else None
        self._engine = None
        self.cap_slots_hint = None      # set to a fixed capacity to avoid sizing from host ids
        self.score_override = None      # tests: inject an [N] score table (identical score bits)
        self.center_on_side_stream = False   # runtime.GraphedTrainStep: label_clf head as a parallel graph branch
        self.scores_external = False    # the caller refreshes eng.score itself (runtime.GraphedTrainStep on a
        #                                 partitioned graph: slice kernel -> all-gather -> this forward)
        self.last_selection = None
        self.use_pdl = False            # runtime.GraphedTrainStep: programmatic dependent launch of the fused kernels
        self.graph_cache = True         # record the reference-facing calls into CUDA graphs (stepgraph.StepGraphCache)
        self.stage_in = None            # runtime.GraphedTrainStep (host batches): (src, dst, bytes) of the packed ids / labels in
        #                                 mapped pinned memory; copied by the step's first kernel (Engine.pool_scores / stage)
        self._graphs = None
        self._fused_memo = {}

    # -- plumbing ---------------------------------------------------------------------------
    def intra_aggs(self):
        return [getattr(self, f"intra_agg{r + 1}") for r in range(self._R)]

    def engine(self) -> Engine:
        dev = self.weight.device
        if self._engine is None or self._engine.device != dev:
            if self._graph is None:
                self._graph = RelGraph.from_adj_lists(self.adj_lists)
            if self._graph.n_rel != self._R:
                raise ValueError(f"{self._R} intra-aggregators but {self._graph.n_rel} relations")
            self._engine = Engine(self._graph, dev)
            self._engine.set_pool(self.train_pos)
        return self._engine

    # -- forward ----------------------------------------------------------------------------
    def _select(self, eng, targets, lab, train_flag, cap, *, workspace=None):
        """Score table -> pool sort -> choose (filter + oversample + union) for device-resident ids / labels and a
        given slot capacity (layers.py:216-262, 633-738). Pure kernel launches on the current stream.
        workspace: a choose workspace of the caller's own (see ``Engine.choose``) instead of the engine's."""
        rho = self.intra_agg1.rho
        dev = eng.device
        cur = torch.cuda.current_stream(dev)
        side = eng.side_stream(0)
        own_scores = self.score_override is None and not self.scores_external
        stage, self.stage_in = self.stage_in, None

        if own_scores and eng.P and train_flag:
            # Three branches fork behind the pool-score kernel and meet in front of the selection kernels:
            #   side 0: preparation of the choose step (repeated targets, item sizes, slot prefix sum, tier queues): no scores
            #   side 1: pool sort, from the pool members' scores alone (layers.py:232, :237)
            #   main  : score table of every node, column 0 (layers.py:231, :236) [+ slice exchange on a row partition]
            pool_score = eng.pool_scores(self.label_clf.weight, self.label_clf.bias, stage=stage)
            side1 = eng.side_stream(1)
            side.wait_stream(cur)
            side1.wait_stream(cur)
            with torch.cuda.stream(side):
                sel = eng.choose(targets, lab, train_flag, self.thresholds, rho, cap, phases=1, workspace=workspace)
            with torch.cuda.stream(side1):
                eng.sort_pool_from(pool_score)
            eng.score_table_only(self.label_clf.weight, self.label_clf.bias)
            cur.wait_stream(side)
            cur.wait_stream(side1)
        else:
            if stage is not None:
                eng.stage(*stage)        # also the common node in front of the fork
            else:
                eng.fork_point()
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                sel = eng.choose(targets, lab, train_flag, self.thresholds, rho, cap, phases=1, workspace=workspace)
            if self.score_override is not None:
                eng.score.copy_(self.score_override)
                eng.resort_pool()
            elif self.scores_external:
                eng.resort_pool()
            elif train_flag:
                eng.score_table(self.label_clf.weight, self.label_clf.bias)
            else:       # eval: no oversampling, the pool is not needed (layers.py:700-738)
                eng.score_table_only(self.label_clf.weight, self.label_clf.bias)
            cur.wait_stream(side)
        eng.choose(targets, lab, train_flag, self.thresholds, rho, cap, phases=2, sel=sel, workspace=workspace)
        self.last_selection = sel
        return sel

    def _choose_and_aggregate(self, nodes, labels, train_flag):
        """Upload of the batch's ids / labels, then ``_select``. Returns (engine, feature table, targets int32,
        device labels, selection)."""
        eng = self.engine()
        dev = eng.device
        table = _feature_table(self.features, eng.N_global, dev)
        eng.set_features(table)
        targets, host = eng.upload_targets(nodes)
        rho = self.intra_agg1.rho
        lab = _as_device_labels(labels, dev) if train_flag else None
        if self.cap_slots_hint is not None:
            cap = int(self.cap_slots_hint)
        else:
            cap = eng.slots_bound(targets.cpu().numpy() if host is None else host, self.thresholds, rho, train_flag)
        return eng, table, targets, lab, self._select(eng, targets, lab, train_flag, cap)

    def graphs(self):
        """The CUDA-graph cache behind the reference-facing calls (``stepgraph.StepGraphCache``)."""
        if self._graphs is None:
            from .stepgraph import StepGraphCache

            self._graphs = StepGraphCache(self)
        return self._graphs

    def _frozen_fast_path(self, table, B) -> bool:
        return (not table.requires_grad) and self.embed_dim <= 256 and B > 0 \
            and isinstance(self.label_clf, nn.Linear) and self.label_clf.bias is not None

    def _fused_ok(self, eng, table, B) -> bool:
        """Frozen table + shapes the fused tile kernels cover (remembered per batch size: this sits on the per-call
        path of the reference-facing API, where every microsecond of host time counts)."""
        if not self._frozen_fast_path(table, B):
            return False
        eng.set_features(table)
        key = (B, eng.F, self.embed_dim)
        ok = self._fused_memo.get(key)
        if ok is None:
            ok = self._fused_memo[key] = eng.tile_supported(B, self._R, self.embed_dim)
        return ok

    def train_loss(self, nodes, labels, head_weight, lam):
        """PCALayer.loss for a training step (model.py:47-61) with the whole dense part, both losses and every
        weight gradient in one pass (``TrainStepFn``); None when the shapes / a trainable feature table rule the
        fused kernels out (the caller then composes forward() with torch ops like the reference does)."""
        eng = self.engine()
        table = _feature_table(self.features, eng.N_global, eng.device)
        B = len(nodes) if not isinstance(nodes, torch.Tensor) else int(nodes.shape[0])
        if not self._fused_ok(eng, table, B):
            return None
        if self.graphs().usable(eng, table, B):
            # host ids (the reference's calling convention): upload into static buffers + ONE graph replay
            loss = self.graphs().train_loss(eng, nodes, labels, head_weight, float(lam))
            if loss is not None:
                return loss
        eng, table, targets, lab, sel = self._choose_and_aggregate(nodes, labels, True)
        agg = eng.aggregate(sel, copy_dups=False)     # repeated targets: the dense kernels read it_rep's row
        loss, _, _ = TrainStepFn.apply(eng, targets, lab, agg, sel.it_rep, float(lam), bool(self.use_pdl), head_weight,
                                       self.label_clf.weight, self.label_clf.bias, self.weight,
                                       *[ia.weight for ia in self.intra_aggs()])
        return loss

    def forward(self, nodes, labels, train_flag=True):
        if not torch.is_grad_enabled() or not any(p.requires_grad for p in self.parameters()):
            # no gradients wanted (utils.test -> to_prob): the whole forward is one cached graph replay
            eng = self.engine()
            table = _feature_table(self.features, eng.N_global, eng.device)
            B = len(nodes) if not isinstance(nodes, torch.Tensor) else int(nodes.shape[0])
            if self._fused_ok(eng, table, B) and self.graphs().usable(eng, table, B):
                res = self.graphs().infer(eng, nodes, labels, train_flag)
                if res is not None:
                    return res
        eng, table, targets, lab, sel = self._choose_and_aggregate(nodes, labels, train_flag)
        dev = eng.device
        B = targets.shape[0]
        fused = self._frozen_fast_path(table, B)
        if fused and eng.tile_supported(B, self._R, self.embed_dim):
            # frozen features (the reference's setup): aggregation, then ONE kernel for the dense part
            agg = eng.aggregate(sel, copy_dups=False)
            ws = [self.label_clf.weight, self.label_clf.bias, self.weight] + [ia.weight for ia in self.intra_aggs()]
            need_grad = torch.is_grad_enabled() and any(w.requires_grad for w in ws)
            return _TileFn.apply(eng, targets, agg, sel.it_rep, self.feat_dim, need_grad, *ws)
        side = None
        if fused:   # [B,2] with gradient to label_clf (layers.py:236-243), one kernel
            if self.center_on_side_stream:
                # independent of choose / aggregate / the dense part: run it (and, since autograd replays a node on
                # its forward stream, its backward) on a side stream, next to them; joined below
                cur = torch.cuda.current_stream(dev)
                side = eng.side_stream()
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    center_scores = _CenterFn.apply(eng, targets, self.label_clf.weight, self.label_clf.bias)
            else:
                center_scores = _CenterFn.apply(eng, targets, self.label_clf.weight, self.label_clf.bias)
        else:
            idx = targets.long()
            self_feats = self.features(idx)
            center_scores = self.label_clf(self_feats)
        if fused:
            # shapes the tile kernel does not cover (E not a multiple of 64): aggregation + the GEMM kernels
            agg = eng.aggregate(sel, copy_dups=False)     # repeated targets: the dense kernels read it_rep's row
            combined = _DenseFn.apply(eng, targets, agg, sel.it_rep, self.feat_dim, self.weight,
                                      *[ia.weight for ia in self.intra_aggs()])
            if side is not None:
                torch.cuda.current_stream(dev).wait_stream(side)
            return combined, center_scores
        agg = _AggregateFn.apply(table, eng, sel, self.feat_dim)
        agg = agg.view(self._R, B, -1)[:, :, :self.feat_dim]

        # relation transforms + inter-relation combine: layers.py:625-629, 273-289
        r_feats = [ia.transform(self_feats, agg[r]) for r, ia in enumerate(self.intra_aggs())]
        cat_feats = torch.cat([self_feats] + r_feats, dim=1)
        combined = F.relu(cat_feats.mm(self.weight).t())
        return combined, center_scores


class InterAgg1(InterAgg):
    n_relations = 1


class InterAgg3(InterAgg):
    n_relations = 3


class InterAgg5(InterAgg):
    n_relations = 5
