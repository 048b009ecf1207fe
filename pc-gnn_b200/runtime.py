"""CUDA-graph training step: the whole step (score table, pool sort, choose, aggregate, relation
transforms, combine, head, both losses, backward, Adam) captured once and replayed per batch.

The reference's trainer (/root/reference/src/model_handler.py:128-156) rebuilds Python lists and
launches ~70 small library kernels per batch; once the hot path is a handful of kernels the step is
launch-bound, so the launches are recorded into a graph and only the batch's ids/labels are copied
into static device buffers before each replay. Per-batch sizes that depend on the data (how many
neighbours survive the filter) stay on the device: the kernels write counts into a status block and
work inside a fixed-capacity slot buffer sized from the epoch's batches (``plan``).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .metrics import _point_requests, _points_dict

__all__ = ["GraphedTrainStep", "GraphedEvalPass", "pack_eval_plan"]


class GraphedTrainStep:
    """model: pcgnn_b200.model.PCALayer (hot path: the InterAgg at ``model.inter1``) or graphsage.GCN / GraphSage
    (hot path: ``model.enc.aggregator``); optimizer must be capturable (e.g. Adam(capturable=True, fused=True))."""

    def __init__(self, model, optimizer, batch_size: int, cap_slots: int, reducer=None, world: int = 1,
                 warmup_batch=None, use_pdl: bool = True):
        """optimizer: a capturable torch optimizer (gradient mean over ranks by NCCL between two graphs), or a
        ``parallel.FusedAdam`` (gradient exchange over peer memory + Adam inside the one step graph)."""
        from .engine import PinnedStaging
        from .parallel import FusedAdam

        self.use_pdl = bool(use_pdl)
        self.fused = isinstance(optimizer, FusedAdam)
        self.model, self.opt, self.B = model, optimizer, int(batch_size)
        self.reducer, self.world = reducer, world
        # the module that sizes the per-step slot buffer: InterAgg for PC-GNN, the row aggregator for GCN / SAGE
        self._sizer = model.inter1 if hasattr(model, "inter1") else model.enc.aggregator
        dev = next(p for p in model.parameters() if p.requires_grad).device
        self.dev = dev
        self._sizer.cap_slots_hint = int(cap_slots)
        self.cap_slots = int(cap_slots)
        if hasattr(model, "inter1") and model.inter1.engine().score_group is not None:
            model.inter1.scores_external = True
        if hasattr(model, "inter1"):
            model.inter1.center_on_side_stream = True
        # ids and labels of a step share ONE static device buffer ([B int64 labels | B int32 ids]) so that a host batch
        # is one pinned staging copy + one H2D; the pinned buffers form a ring guarded by events: back-to-back run()
        # calls never rewrite a buffer whose copy is still queued behind the previous replay
        self._packed = torch.zeros(3 * self.B, dtype=torch.int32, device=dev)
        self.labels = self._packed[:2 * self.B].view(torch.int64)
        self.nodes = self._packed[2 * self.B:]
        self._pin = PinnedStaging(3 * self.B, torch.int32)
        self._pin_loss = torch.zeros(1, dtype=torch.float32, pin_memory=True)
        self._loss_event = torch.cuda.Event()
        self.loss = None
        # host batches (fused optimizer): a second recording of the step whose FIRST kernel also fetches the packed batch
        # out of one pinned buffer at a fixed address (mapped host memory) and which ends with a 4-byte store of the
        # loss into a pinned word, so that a host batch costs one graph launch and one event wait (no copy calls around it)
        self._pin_in = torch.zeros(3 * self.B, dtype=torch.int32, pin_memory=True)
        self._pin_in_np = self._pin_in.numpy()
        self._pin_loss_np = self._pin_loss.numpy()
        self._host_done = torch.cuda.Event()
        self._host_pending = False
        self.g_host = None
        self.loss_host = None
        # epoch plan (load_plan / run_planned): every batch of an epoch in HBM, a device cursor, a third recording that
        # fetches entry `cursor` and stores its loss into losses[cursor]
        self._plan = None               # int32 [n_steps, 3B]
        self._plan_losses = None        # fp32 [n_steps]
        self._cursor = torch.zeros(1, dtype=torch.int32, device=dev)
        self.g_plan = None
        if reducer is not None:
            # the captured graph writes the gradients through the parameters' .grad tensors: they must BE the views
            # of the reducer's flat buffer (otherwise the graph keeps accumulating into tensors nobody zeroes)
            for p_, v_ in zip(reducer.params, reducer.views):
                if p_.grad is None or p_.grad.data_ptr() != v_.data_ptr():
                    reducer.attach()
                    break
        # row-partitioned graph: the score slices are exchanged by an eager all-gather BETWEEN two graphs
        # (slice kernel | all-gather | everything else), so no collective is captured
        eng = model.inter1.engine() if hasattr(model, "inter1") else None
        self._xeng = eng if (eng is not None and eng.score_group is not None) else None
        self.g_pre = None
        if warmup_batch is not None:
            self.nodes.copy_(torch.as_tensor(np.asarray(warmup_batch[0], dtype=np.int32)))
            self.labels.copy_(torch.as_tensor(np.asarray(warmup_batch[1], dtype=np.int64)))
        self._capture()

    # -- one eager step on the static buffers (also what gets captured) -------------------------
    def _score_pre(self):
        inter = self.model.inter1
        self._xeng.set_features(inter.features.weight)
        self._xeng.score_local(inter.label_clf.weight, inter.label_clf.bias)

    def _stage_in(self):
        """(recorded) the packed batch out of the pinned buffer, by a KERNEL reading the mapped host memory: PC-GNN
        models hand the copy to ``InterAgg._select``, where it rides on the step's first kernel (the pool scores,
        which need no ids); other models get a copy kernel in front. No memcpy node: the recording stays a graph of
        kernels (with copy nodes in it the branches of the step were measured to start several microseconds apart)."""
        nbytes = self._packed.numel() * 4
        if self._plan is not None and self._staging_plan:
            job = (self._plan.data_ptr(), self._packed.data_ptr(), nbytes, self._cursor.data_ptr(), self._plan.shape[0],
                   nbytes)
        else:
            job = (_lib.host_device_ptr(self._pin_in), self._packed.data_ptr(), nbytes)
        inter = getattr(self.model, "inter1", None)
        if inter is not None and hasattr(inter, "stage_in"):
            inter.stage_in = job
        elif len(job) > 3:
            _lib.check(_lib.lib().pcg_stage_indexed(job[0], job[1], job[2], job[3], job[4], job[5], 0, 0,
                                                    _lib.stream_ptr()), "pcg_stage_indexed")
        else:
            _lib.check(_lib.lib().pcg_stage(job[0], job[1], job[2], _lib.stream_ptr()), "pcg_stage")

    def _fwd_bwd(self, host_io: bool = False):
        if self._xeng is not None and not torch.cuda.is_current_stream_capturing():
            self._score_pre()                      # eager warm-up steps: slice, exchange, then the forward
            self._xeng.score_exchange()
        if host_io:
            self._stage_in()
        if self.fused:
            pass                                   # the fused step leaves the gradients zeroed
        elif self.reducer is not None:
            self.reducer.zero()
        else:
            self.opt.zero_grad(set_to_none=False)
        eng = self.model.inter1.engine() if (self.fused and hasattr(self.model, "inter1")) else None
        if eng is not None:
            # every parameter has exactly one producer kernel and the buffer is zero: let the kernels store the
            # gradients in place (no AccumulateGrad adds in the graph)
            eng.grad_sink = {p.data_ptr(): v for p, v in zip(self.reducer.params, self.reducer.views)}
        try:
            if eng is not None:
                eng.grads_in_sinks = False
            loss = self.model.loss(self.nodes, self.labels)
            if eng is None or not eng.grads_in_sinks:    # fused pass: the forward launch stored every gradient
                loss.backward()
        finally:
            if eng is not None:
                eng.grad_sink = None
            inter = getattr(self.model, "inter1", None)
            if host_io and getattr(inter, "stage_in", None) is not None:
                inter.stage_in = None
                raise RuntimeError("the staged batch copy was not consumed by the forward pass")
        return loss.detach()

    def _capture(self):
        # programmatic dependent launch for the kernels recorded below (see include/pcgnn_b200.h: pcg_set_pdl).
        # Measured on C2 (profiles/README.md): the fused dense kernel and the exchange + Adam kernel gain from starting
        # under the tail of the kernel in front (mask 2 | 8: 91.2 -> 87.8 us per replay); the cluster-launched
        # weight-gradient kernel and the pool sort lose (mask 4: +10 us), so they keep full dependencies.
        import os

        mask = int(os.environ.get("PCG_PDL_MASK", "10")) if self.use_pdl else 0
        prev = _lib.lib().pcg_set_pdl(mask)
        try:
            self._capture_graphs()
        finally:
            _lib.lib().pcg_set_pdl(prev)

    def _capture_graphs(self):
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):       # warm-up on a side stream (allocator, lazy inits, cuBLAS handles)
            for _ in range(3):
                if self.reducer is None:
                    for p in self.model.parameters():
                        if p.requires_grad and p.grad is None:
                            p.grad = torch.zeros_like(p)
                self._fwd_bwd()
                if self.fused:
                    self.reducer.zero()
                # no optimizer step during warm-up: parameters stay as the caller initialised them
            if self.fused:
                torch.cuda.current_stream(self.dev).wait_stream(s)
        if self.fused:
            torch.cuda.synchronize(self.dev)
            if self._xeng is not None:
                self.g_pre = torch.cuda.CUDAGraph()
                with _lib.capture(self.g_pre):
                    self._score_pre()
            self.g_fb = torch.cuda.CUDAGraph()
            with _lib.capture(self.g_fb):
                self.loss = self._fwd_bwd()
                self.opt.step()                    # gradient mean over the ranks + Adam, one kernel
            self.g_opt = None
            return
        with torch.cuda.stream(s):
            # Create the optimizer state OUTSIDE the graph: torch builds it lazily in the first step(), and a
            # captured lazy init would re-zero the moments on every replay. Step once, then undo it.
            params = [p for g in self.opt.param_groups for p in g["params"] if p.requires_grad]
            backup = [p.detach().clone() for p in params]
            had_state = len(self.opt.state) > 0
            saved = None
            if had_state:
                saved = {k: {n: (v.clone() if isinstance(v, torch.Tensor) else v) for n, v in st.items()}
                         for k, st in self.opt.state.items()}
            self.opt.step()
            with torch.no_grad():
                for p, b in zip(params, backup):
                    p.copy_(b)
                for k, st in self.opt.state.items():
                    for n, v in st.items():
                        if isinstance(v, torch.Tensor):
                            v.copy_(saved[k][n]) if had_state else v.zero_()
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        if self._xeng is not None:
            self.g_pre = torch.cuda.CUDAGraph()
            with _lib.capture(self.g_pre):
                self._score_pre()
        self.g_fb = torch.cuda.CUDAGraph()
        with _lib.capture(self.g_fb):
            self.loss = self._fwd_bwd()
        self.g_opt = torch.cuda.CUDAGraph()
        with _lib.capture(self.g_opt):
            self.opt.step()

    _staging_plan = False

    def _capture_host_graph(self, plan: bool = False):
        """Fused optimizer only: the step with its batch fetch and its loss store recorded as kernels of the graph.
        plan: the batch comes from entry `cursor` of the device-resident epoch plan, the loss goes into losses[cursor]
        and the cursor advances."""
        import os

        torch.cuda.synchronize(self.dev)
        mask = int(os.environ.get("PCG_PDL_MASK", "10")) if self.use_pdl else 0
        prev = _lib.lib().pcg_set_pdl(mask)
        self._staging_plan = plan
        try:
            if not plan:
                self._pin_in.copy_(self._packed)       # whatever batch is resident: replays before run() stay meaningful
            g = torch.cuda.CUDAGraph()
            with _lib.capture(g):
                cur = torch.cuda.current_stream(self.dev)
                loss = self._fwd_bwd(host_io=True)
                # the loss leaves (a 4-byte store into the mapped pinned word) next to the exchange + Adam kernel
                side = torch.cuda.Stream(device=self.dev) if not hasattr(self.model, "inter1") \
                    else self.model.inter1.engine().side_stream(2)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    if plan:
                        _lib.check(_lib.lib().pcg_stage_indexed(loss.data_ptr(), self._plan_losses.data_ptr(), 4,
                                                                self._cursor.data_ptr(), self._plan.shape[0], 0, 4, 1,
                                                                _lib.stream_ptr()), "pcg_stage_indexed")
                    else:
                        _lib.check(_lib.lib().pcg_stage(loss.data_ptr(), _lib.host_device_ptr(self._pin_loss), 4,
                                                        _lib.stream_ptr()), "pcg_stage")
                self.opt.step()
                cur.wait_stream(side)
            if plan:
                self.g_plan = g
            else:
                self.g_host, self.loss_host = g, loss
        finally:
            self._staging_plan = False
            _lib.lib().pcg_set_pdl(prev)

    def _replay(self, host: bool = False, plan: bool = False):
        if self.g_pre is not None:
            self.g_pre.replay()
            self._xeng.score_exchange()
        if plan:
            self.g_plan.replay()
            return None
        if host:
            self.g_host.replay()
            return self.loss_host
        self.g_fb.replay()
        if self.fused:
            return self.loss
        if self.world > 1 and self.reducer is not None:
            self.reducer()                       # one NCCL all-reduce of the flat gradient
            self.reducer.flat.div_(self.world)
        self.g_opt.replay()
        return self.loss

    # -- public --------------------------------------------------------------------------------
    def run_device(self, nodes_dev: torch.Tensor, labels_dev: torch.Tensor):
        """Batch already in HBM (int32 ids, int64 labels). Returns the (device) loss tensor."""
        if nodes_dev.dtype == torch.int32 and labels_dev.dtype == torch.int64 and labels_dev.is_contiguous():
            # both copies in ONE multi-tensor kernel (labels seen as int32 pairs)
            B = self.B
            torch._foreach_copy_([self._packed[:2 * B], self._packed[2 * B:]],
                                 [labels_dev.view(torch.int32).reshape(-1), nodes_dev.reshape(-1)], non_blocking=True)
        else:
            self.nodes.copy_(nodes_dev, non_blocking=True)
            self.labels.copy_(labels_dev, non_blocking=True)
        return self._replay()

    def run(self, nodes, labels):
        """Batch on the host (numpy arrays, or lists, of ids and labels): one pinned staging copy + one H2D + replay.
        Returns the (device) loss tensor."""
        B = self.B
        if self.fused:
            # one graph launch: the step's kernels read the batch from / write the loss to pinned host memory themselves.
            # The pinned input buffer is free again once the previous replay has finished.
            if self.g_host is None:
                self._capture_host_graph()
            if self._host_pending:
                self._host_done.synchronize()
            pin = self._pin_in_np
            pin[:2 * B].view(np.int64)[:] = labels
            pin[2 * B:] = nodes
            loss = self._replay(host=True)
            self._host_done.record(torch.cuda.current_stream(self.dev))
            self._host_pending = True
            return loss
        host = np.empty(3 * B, dtype=np.int32)
        host[:2 * B].view(np.int64)[:] = labels
        host[2 * B:] = nodes
        self._pin.upload(host, self._packed)
        return self._replay()

    def run_item(self, nodes, labels) -> float:
        """``run`` + the loss as a Python float (device->host through a pinned word; cheaper than ``.item()``'s
        pageable copy). Fused optimizer: the D2H copy is the last node of the recorded step, so this is one graph
        launch and one event wait."""
        loss = self.run(nodes, labels)
        if self.fused:
            self._host_done.synchronize()
            self._host_pending = False
            return float(self._pin_loss_np[0])
        self._pin_loss.copy_(loss.reshape(1), non_blocking=True)
        self._loss_event.record(torch.cuda.current_stream(self.dev))
        self._loss_event.synchronize()
        return float(self._pin_loss[0])

    # -- epoch plan: the batch loop of model_handler.py:128-150 with the epoch's batches resident in HBM --------------
    def load_plan(self, batches):
        """Upload a whole epoch: ``batches`` = sequence of (ids, labels), each exactly ``batch_size`` long. One packed
        host array, one H2D; afterwards ``run_planned()`` replays the step for the next entry (wrapping around) without
        the host touching a batch: the recorded step fetches entry ``cursor`` itself, stores its loss into
        ``plan_losses()[cursor]`` and advances the cursor on the device. Fused optimizer only."""
        if not self.fused:
            raise RuntimeError("epoch plans need the fused optimizer (parallel.FusedAdam)")
        B, n = self.B, len(batches)
        if n == 0:
            raise ValueError("load_plan: no batches")
        host = np.empty((n, 3 * B), dtype=np.int32)
        for i, (ids, labels) in enumerate(batches):
            if len(ids) != B or len(labels) != B:
                raise ValueError(f"load_plan: batch {i} has {len(ids)} ids / {len(labels)} labels, the recorded step takes "
                                 f"exactly {B} (run a partial last batch through model.loss)")
            host[i, :2 * B].view(np.int64)[:] = labels
            host[i, 2 * B:] = ids
        plan = torch.from_numpy(host).to(self.dev)
        if self._plan is not None and self._plan.shape == plan.shape:
            self._plan.copy_(plan)                     # same addresses: the recording stays valid
        else:
            self._plan = plan
            self._plan_losses = torch.zeros(n, dtype=torch.float32, device=self.dev)
            self.g_plan = None
        self._cursor.zero_()
        if self.g_plan is None:
            self._capture_host_graph(plan=True)
        return n

    def run_planned(self):
        """One step on the next entry of the plan: a graph replay, nothing else."""
        if self.g_plan is None:
            raise RuntimeError("run_planned: call load_plan(batches) first")
        self._replay(plan=True)

    def plan_losses(self) -> torch.Tensor:
        """Device tensor of the planned steps' losses (entry i = the most recent step on plan entry i)."""
        return self._plan_losses

    def overflowed(self) -> bool:
        """True if ANY replay since the last call needed more slots than the captured capacity (its results were
        incomplete: re-plan with a larger capacity). PC-GNN models: a workspace word every choose call ORs its flag
        into (``Engine.overflow_since_reset``); GCN / SAGE: the last replay's status block. Syncs."""
        if hasattr(self.model, "inter1"):
            return self.model.inter1.engine().overflow_since_reset()
        sel = self._sizer.last_selection
        return bool(sel is not None and sel.overflowed())

    @staticmethod
    def plan(engine, batches, thresholds, rho) -> int:
        """Slot capacity covering every batch of an epoch plan (the largest ``Engine.slots_bound`` of a batch)."""
        return max(engine.slots_bound(n, thresholds, rho, True) for n in batches)


# -- evaluation: the test loop of utils.py:298-333 over a whole node set, recorded ------------------------------------
def pack_eval_plan(nodes, batch_size: int, indptr=None) -> np.ndarray:
    """A node set as an int32 [n_entries, batch_size] plan in the given order. The last entry is padded with copies of
    its own first id: pcg_choose folds repeated targets onto their first occurrence (``it_rep``), so the padding adds
    no choose or aggregate work, and the rows it produces are never written out.

    indptr: CSR row offsets of a one-relation graph (the GCN / GraphSAGE baselines). pcg_select_all does not fold
    repeated targets, so every padding row aggregates its node's whole row; with indptr the padding repeats the set's
    node with the shortest row (the first such node in the given order) instead."""
    B = int(batch_size)
    if B <= 0:
        raise ValueError(f"batch_size must be positive, got {batch_size}")
    ids = np.asarray(nodes, dtype=np.int64).reshape(-1)
    n = ids.shape[0]
    if n == 0:
        raise ValueError("an evaluation pass needs at least one node")
    if ids.min() < 0 or ids.max() > np.iinfo(np.int32).max:
        raise ValueError("node ids must lie in [0, 2^31)")
    n_entries = -(-n // B)
    plan = np.empty((n_entries, B), dtype=np.int32)
    flat = plan.reshape(-1)
    flat[:n] = ids
    if indptr is None:
        flat[n:] = ids[(n_entries - 1) * B]
    else:
        ip = np.asarray(indptr, dtype=np.int64)
        if ids.max() >= ip.shape[0] - 1:
            raise ValueError(f"node id {int(ids.max())} is not a row of the graph ({ip.shape[0] - 1} rows)")
        flat[n:] = ids[np.argmin(ip[ids + 1] - ip[ids])]
    return plan


def _baseline_parts(model):
    """(aggregator, add_self, with_self, head mode) of graphsage.GCN over GCNEncoder(GCNAggregator) or GraphSage over
    Encoder(MeanAggregator); None for PCALayer over an InterAgg; PcgError for anything else."""
    from .graphsage import GCN, Encoder, GCNAggregator, GCNEncoder, GraphSage, MeanAggregator
    from .layers import InterAgg
    from .model import PCALayer

    if isinstance(model, PCALayer) and isinstance(getattr(model, "inter1", None), InterAgg):
        return None
    enc = getattr(model, "enc", None)
    agg = getattr(enc, "aggregator", None)
    if isinstance(model, GCN) and isinstance(enc, GCNEncoder) and isinstance(agg, GCNAggregator):
        return agg, True, False, 0
    if isinstance(model, GraphSage) and isinstance(enc, Encoder) and isinstance(agg, MeanAggregator):
        return agg, bool(agg.gcn), not enc.gcn, 1
    raise _lib.PcgError("GraphedEvalPass runs PCALayer over an InterAgg, GCN over GCNEncoder(GCNAggregator) or "
                        f"GraphSage over Encoder(MeanAggregator), not {type(model).__name__}")


class GraphedEvalPass:
    """Scores a whole node set (validation, test, all nodes) with PCALayer, graphsage.GCN or graphsage.GraphSage and
    computes its metrics on the device: ``run()`` is n_entries replays of one recorded batch graph, one replay of a
    metrics graph and one host wait.

    The ids are uploaded once as a plan of ``batch_size``-wide entries. PCALayer's batch graph fetches entry ``cursor``
    (``InterAgg.stage_in``), runs the eval-mode selection (score table, choose) with a choose workspace of its own,
    the aggregation, the fused dense kernel and the head + sigmoid (``pcg_eval_head``). The baselines' batch graph
    fetches the entry (``pcg_stage_indexed``), selects the targets' whole rows (``pcg_select_all``, with the target
    itself where the aggregator adds it), aggregates them with the aggregator's norm, runs ``pcg_encoder_fwd`` (with
    the self rows for ``Encoder(gcn=False)``) and the head + to_prob's sigmoid (GCN) or log-softmax (GraphSage); their
    plans are padded with the set's lowest-degree node (``pack_eval_plan``'s indptr). Either writes a planar [2, n]
    buffer, then advances the cursor with a copy of the batch's overflow word into a per-entry array. The metrics graph
    runs ``pcg_binary_metrics`` (with ``operating_points``, then ``pcg_binary_points``) and copies the result block and
    the overflow words to pinned memory.

    ``operating_points``: None, or a dict with any of the lists ``top_k``, ``fpr`` and ``max_fpr`` of
    ``metrics.device_operating_points``; ``run()`` then also returns them under ``"operating_points"``. The requests
    live in device memory read by the recorded graph, so ``set_operating_points`` changes their values without
    re-recording.

    Replays read the current parameter values, so in-place updates (optimizer steps) need nothing; a parameter or the
    feature table moving to new storage, new thresholds (PCALayer) or another engine (an aggregator bound to another
    graph) re-record on the next ``run()``. The modules' own state (``last_selection``, ``cap_slots_hint``, ...) is
    left alone. There is no torch fallback: models, tables, graphs and shapes the recorded path does not cover raise
    ``PcgError``."""

    def __init__(self, model, nodes, labels, batch_size: int, cap_slots: int | None = None, operating_points=None):
        self._homo = _baseline_parts(model)
        eng = model.inter1.engine() if self._homo is None else self._homo[0]._get_engine()
        plan = pack_eval_plan(nodes, batch_size, None if self._homo is None else eng.graph.indptr[:eng.N + 1])
        y = np.asarray(labels).reshape(-1)
        n = int(np.asarray(nodes).reshape(-1).shape[0])
        if y.shape[0] != n:
            raise ValueError(f"{y.shape[0]} labels for {n} nodes")
        if not np.isin(y, (0, 1)).all():
            raise ValueError("labels must be 0 or 1")
        self.model, self.B, self.n = model, int(batch_size), n
        self.n_entries = int(plan.shape[0])
        self._state()                                  # refusals before any allocation
        self._pt_host = None if operating_points is None else _point_requests(n, **operating_points)
        m = 0 if self._pt_host is None else len(self._pt_host[0])
        dev = eng.device
        L = _lib.lib()
        self._plan_host = plan
        self._plan = torch.from_numpy(plan).to(dev)
        self._labels = torch.from_numpy(y.astype(np.int32)).to(dev)
        self._nodes = torch.empty(self.B, dtype=torch.int32, device=dev)
        self._cursor = torch.zeros(1, dtype=torch.int32, device=dev)
        self._prob = torch.empty((2, n), dtype=torch.float32, device=dev)
        # [metrics (doubles) | operating points (doubles) | overflow word of every entry]: one block, one copy to the host
        W, self._ovf_at = _lib.METRICS_WORDS, 2 * (_lib.METRICS_WORDS + m * _lib.POINT_WORDS)
        self._res = torch.zeros(self._ovf_at + self.n_entries, dtype=torch.int32, device=dev)
        self._out = self._res[:2 * W].view(torch.float64)
        self._pts = self._res[2 * W:self._ovf_at].view(torch.float64)
        self._ovf = self._res[self._ovf_at:]
        if m:
            self._pt_kind = torch.from_numpy(self._pt_host[0]).to(dev)
            self._pt_arg = torch.from_numpy(self._pt_host[1]).to(dev)
            self._pt_ws = torch.empty(int(L.pcg_binary_points_workspace_bytes(n, m)), dtype=torch.uint8, device=dev)
        self._pin = torch.zeros(self._res.numel(), dtype=torch.int32, pin_memory=True)
        self._pin_np = self._pin.numpy()
        self._mws = torch.empty(int(L.pcg_binary_metrics_workspace_bytes(n)), dtype=torch.uint8, device=dev)
        self._cap_arg = cap_slots
        if self._homo is None:
            inter = model.inter1
            # the pass's own choose workspace, sized for its batch and initialised once: the engine's shared one is
            # reallocated when a larger batch comes along, which recorded graphs must never see
            ws_bytes = int(L.pcg_choose_workspace_bytes(self.B, eng.R, eng.max_degree, eng.N))
            self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _lib.check(L.pcg_choose_workspace_init(self._ws.data_ptr(), ws_bytes, eng.N, _lib.stream_ptr()),
                       "pcg_choose_workspace_init")
            if cap_slots is None:
                cap_slots = max(eng.slots_bound(e, inter.thresholds, inter.intra_agg1.rho, False) for e in plan)
            self.cap_slots = int(cap_slots)
        else:
            self.cap_slots = self._baseline_capacity()
        self._done = torch.cuda.Event()
        self._key = None
        self._curve = None                             # pcg_binary_curve's outputs, allocated by the first curve()
        self._ran = False
        self.g_batch = self.g_metrics = None
        self.captures = 0

    def _baseline_capacity(self) -> int:
        """The caller's capacity, else exactly the largest per-entry slot demand on the aggregator's current graph."""
        if self._cap_arg is not None:
            return int(self._cap_arg)
        return max(self._homo[0].slots_bound(e) for e in self._plan_host)

    def _params(self):
        if self._homo is not None:
            return [self.model.weight, self.model.enc.weight]
        inter = self.model.inter1
        return [self.model.weight, inter.label_clf.weight, inter.label_clf.bias, inter.weight] + \
            [ia.weight for ia in inter.intra_aggs()]

    @staticmethod
    def _check_params(params, eng):
        if any(not p.is_contiguous() or p.dtype != torch.float32 or p.device != eng.device for p in params):
            raise _lib.PcgError("GraphedEvalPass: parameters must be contiguous fp32 tensors on the engine's device")

    def _state(self):
        """What the recording bakes in (parameter and feature-table addresses, thresholds / engine), after the
        refusals."""
        import torch.nn as nn

        from .layers import _feature_table

        if self._homo is not None:
            return self._state_baseline()
        inter = self.model.inter1
        eng = inter.engine()
        table = _feature_table(inter.features, eng.N_global, eng.device)
        if table.requires_grad:
            raise _lib.PcgError("GraphedEvalPass: the feature table is trainable (the recorded path has no gradient to it)")
        if eng.graph.partitioned or eng.score_group is not None or eng._bcast is not None or inter.scores_external:
            raise _lib.PcgError("GraphedEvalPass: row-partitioned graphs and exchanged score tables are not supported")
        if self.model.weight.shape[0] != 2 or not isinstance(inter.label_clf, nn.Linear) or inter.label_clf.bias is None:
            raise _lib.PcgError("GraphedEvalPass: needs a two-class head and label_clf = nn.Linear with a bias")
        params = self._params()
        self._check_params(params, eng)
        eng.set_features(table)
        E = int(inter.weight.shape[1])
        if not eng.tile_supported(self.B, eng.R, E):
            raise _lib.PcgError(f"GraphedEvalPass: pcg_tile_supported rejects B={self.B} R={eng.R} F={eng.F} E={E}")
        return tuple(p.data_ptr() for p in params) + (eng.feat.data_ptr(),), tuple(float(t) for t in inter.thresholds)

    def _state_baseline(self):
        from .graphsage import _encoder_fits
        from .layers import _feature_table

        agg, _, with_self, _ = self._homo
        enc = self.model.enc
        eng = agg._get_engine()
        table = _feature_table(agg.features, eng.N, eng.device)
        if table.requires_grad:
            raise _lib.PcgError("GraphedEvalPass: the feature table is trainable (the recorded path has no gradient to it)")
        if eng.graph.partitioned or eng.R != 1:
            raise _lib.PcgError("GraphedEvalPass: the baselines need an unpartitioned one-relation graph (row-partitioned "
                                f"or multi-relation graphs are not supported; this one has {eng.R} relations)")
        if self.model.weight.shape[0] != 2:
            raise _lib.PcgError("GraphedEvalPass: needs a two-class head")
        params = self._params()
        self._check_params(params, eng)
        eng.set_features(table)
        E, f_in = int(enc.weight.shape[0]), eng.F * (2 if with_self else 1)
        if enc.weight.shape[1] != f_in or self.model.weight.shape[1] != E or not _encoder_fits(enc, eng):
            raise _lib.PcgError(f"GraphedEvalPass: pcg_encoder_fwd does not take an encoder weight of shape "
                                f"{tuple(enc.weight.shape)} (F={eng.F}, head {tuple(self.model.weight.shape)})")
        return tuple(p.data_ptr() for p in params) + (eng.feat.data_ptr(),), eng

    def _record(self):
        from .stepgraph import StepGraphCache

        if self._homo is not None:
            return self._record_baseline()
        inter = self.model.inter1
        eng = inter.engine()
        p = [q.detach() for q in self._params()]
        head, w_inter, w_intra = p[0], p[3], p[4:]
        B, nb = self.B, self.n_entries
        cur = self._cursor.data_ptr()

        def batch():
            inter.stage_in = (self._plan.data_ptr(), self._nodes.data_ptr(), B * 4, cur, nb, B * 4)
            sel = inter._select(eng, self._nodes, None, False, self.cap_slots, workspace=self._ws)
            agg = eng.aggregate(sel, copy_dups=False)
            out, _, _ = eng.tile_fwd(self._nodes, agg, sel.it_rep, w_intra, w_inter, None, None, False)
            self._head_and_overflow(out, head, 0, sel)
            return sel

        last = inter.last_selection
        try:
            self.g_batch, _ = StepGraphCache._capture(batch, eng.device)
            self.g_metrics, _ = StepGraphCache._capture(self._metrics, eng.device)
        finally:
            inter.stage_in = None
            inter.last_selection = last
        self.captures += 1

    def _record_baseline(self):
        from .stepgraph import StepGraphCache

        agg, add_self, with_self, mode = self._homo
        eng = agg._get_engine()
        head, w_enc = [q.detach() for q in self._params()]
        B, nb = self.B, self.n_entries
        self.cap_slots = self._baseline_capacity()

        def batch():
            eng.stage(self._plan.data_ptr(), self._nodes.data_ptr(), B * 4, self._cursor.data_ptr(), nb, B * 4)
            sel = eng.select_all(self._nodes, add_self, self.cap_slots, agg._norm)
            emb = eng.encoder_fwd(eng.aggregate(sel), w_enc, self._nodes if with_self else None)
            self._head_and_overflow(emb, head, mode, sel)
            return sel

        self.g_batch, _ = StepGraphCache._capture(batch, eng.device)
        self.g_metrics, _ = StepGraphCache._capture(self._metrics, eng.device)
        self.captures += 1

    def _head_and_overflow(self, emb, head, mode, sel):
        """(recorded) pcg_eval_head into the entry's rows of the probability buffer, then the batch's overflow word into
        the entry's slot of the overflow array, advancing the cursor."""
        L = _lib.lib()
        cur, nb = self._cursor.data_ptr(), self.n_entries
        _lib.check(L.pcg_eval_head(emb.data_ptr(), int(emb.shape[0]), self.B, head.data_ptr(), mode, self.n, cur, nb,
                                   self._prob.data_ptr(), _lib.stream_ptr()), "pcg_eval_head")
        _lib.check(L.pcg_stage_indexed(sel.status[_lib.ST_OVERFLOW:].data_ptr(), self._ovf.data_ptr(), 4, cur, nb, 0, 4, 1,
                                       _lib.stream_ptr()), "pcg_stage_indexed")

    def _metrics(self):
        L = _lib.lib()
        _lib.check(L.pcg_binary_metrics(self._prob.data_ptr(), self._labels.data_ptr(), self.n, self._out.data_ptr(),
                                        self._mws.data_ptr(), self._mws.numel(), _lib.stream_ptr()), "pcg_binary_metrics")
        if self._pt_host is not None:
            _lib.check(L.pcg_binary_points(self._mws.data_ptr(), self._mws.numel(), self.n, self._pt_kind.data_ptr(),
                                           self._pt_arg.data_ptr(), len(self._pt_host[0]), self._pts.data_ptr(),
                                           self._pt_ws.data_ptr(), self._pt_ws.numel(), _lib.stream_ptr()),
                       "pcg_binary_points")
        _lib.check(L.pcg_stage(self._res.data_ptr(), _lib.host_device_ptr(self._pin), self._res.numel() * 4,
                               _lib.stream_ptr()), "pcg_stage")

    def run(self) -> dict:
        """Scores every node and returns the metrics as python floats: the keys of ``metrics.binary_metrics`` (pred =
        prob[1] > prob[0], as utils.test) plus best_f1_macro, best_threshold, n_pos, n_neg, tp / fp / tn / fn, ap,
        recall_at_k, best_gmean and best_gmean_threshold (``metrics.device_metrics``).
        The metrics are computed on ``probs()`` as they are: for GraphSage, log-probabilities, so ``best_threshold``
        and ``best_gmean_threshold`` are log-probabilities there (pred, AUC and the ranking keys ap, recall_at_k,
        best_f1_macro and best_gmean need no conversion: log is monotone).
        A pass built with ``operating_points`` adds the key ``"operating_points"`` (``metrics.device_operating_points``'
        result for the current requests, computed in the same metrics graph); for GraphSage its thresholds are
        log-probabilities too, its counts and rates need no conversion.
        Raises PcgError when a batch needed more slots than ``cap_slots`` (its scores would be incomplete)."""
        key = self._state()
        if key != self._key:
            self.g_batch = self.g_metrics = None
            self._record()
            self._key = key
        self._cursor.zero_()
        for _ in range(self.n_entries):
            self.g_batch.replay()
        self.g_metrics.replay()
        self._ran = True
        self._done.record(torch.cuda.current_stream(self._prob.device))
        self._done.synchronize()
        W = _lib.METRICS_WORDS
        bad = np.flatnonzero(self._pin_np[self._ovf_at:])
        if bad.size:
            raise _lib.PcgError(f"GraphedEvalPass: {bad.size} of {self.n_entries} batches needed more than cap_slots="
                                f"{self.cap_slots} slots (first: entry {int(bad[0])}); build the pass with a larger capacity")
        res = dict(zip(_lib.METRICS_KEYS, self._pin_np[:2 * W].view(np.float64).tolist()))
        if self._pt_host is not None:
            res["operating_points"] = _points_dict(self._pin_np[2 * W:self._ovf_at].view(np.float64), *self._pt_host)
        return res

    def set_operating_points(self, top_k=(), fpr=(), max_fpr=()):
        """New values for the requests of a pass built with ``operating_points``, the same number of each kind (the
        recorded graph reads them from device memory: no re-recording). Used from the next ``run()`` on."""
        if self._pt_host is None:
            raise _lib.PcgError("GraphedEvalPass.set_operating_points: the pass was built without operating_points")
        kind, arg = _point_requests(self.n, top_k, fpr, max_fpr)
        if not np.array_equal(kind, self._pt_host[0]):
            raise ValueError("GraphedEvalPass.set_operating_points: needs as many top_k, fpr and max_fpr requests as the "
                             "pass was built with (build a new pass for other counts)")
        self._pt_arg.copy_(torch.from_numpy(arg))
        self._pt_host = (kind, arg)

    def curve(self) -> tuple:
        """ROC / PR curve of the last ``run()`` (``metrics.device_curve`` of ``probs()``): (thresholds fp32 [G],
        tp int64 [G], fp int64 [G]) on the device, ascending thresholds. One eager launch over the metrics workspace
        the run left and one 8-byte read of G; the tensors are views of buffers of the pass that the next ``curve()``
        overwrites. For GraphSage the thresholds are log-probabilities (the counts are those of the probabilities)."""
        from .metrics import _curve_buffers, _read_curve

        if not self._ran:
            raise _lib.PcgError("GraphedEvalPass.curve: run() first (the curve is read from the last run's metrics)")
        if self._curve is None:
            self._curve = _curve_buffers(self.n, self._prob.device)
        return _read_curve(self._mws, self.n, self._curve)

    def probs(self) -> torch.Tensor:
        """[n, 2] view of the last run's to_prob output (PCALayer: its first output), in the caller's node order:
        probabilities for PCALayer and GCN, log-probabilities for GraphSage."""
        return self._prob.t()
