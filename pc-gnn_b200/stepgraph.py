"""CUDA-graph cache behind the reference-facing calls.

The reference's trainer calls ``model.loss(batch_nodes: list, labels)`` / ``model.to_prob(...)`` once per batch
(/root/reference/src/model_handler.py:142-156, utils.py:298-312). On this package's kernels such a call is ~9
launches whose host-side cost (argument marshalling, allocator, Python) exceeds their GPU time, so ``InterAgg``
records them ONCE per (batch size, mode) into a CUDA graph and afterwards only uploads the batch's ids / labels
into static buffers and replays: the caller's loop stays exactly the reference's, nothing to opt into.

What a cached graph bakes in, and how each is kept honest:
  * parameter / feature-table addresses  -> compared on every call, a change re-records the graph
  * the slot capacity of the selection    -> the batch's training-mode ``Engine.slots_bound`` (it covers eval mode too)
                                             on every call; a batch that needs more re-records with a larger capacity
  * lambda, rho, thresholds               -> part of the cache key
Training graphs hold the whole step behind the upload (score table, pool sort, choose, aggregate, the fused dense
/ loss / gradient kernels); the returned loss carries an autograd node whose backward hands out the gradients the
replay computed (scaled by the incoming gradient), so ``loss.backward(); optimizer.step()`` work unchanged.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, fastloop
from .engine import PinnedStaging

__all__ = ["StepGraphCache"]

MAX_GRAPHS = 8        # per InterAgg: (batch size, mode) combinations kept


class _ReplayLossFn(torch.autograd.Function):
    """loss of a replayed training graph; backward = the gradients that replay stored, times the incoming one."""

    @staticmethod
    def forward(ctx, loss_static, flat_static, views, *params):
        ctx.flat, ctx.views, ctx.n = flat_static, views, len(params)
        return loss_static.clone()

    @staticmethod
    def backward(ctx, d_loss):
        scaled = ctx.flat * d_loss          # fresh tensor: the static buffer is rewritten by the next replay
        return (None, None, None, *[scaled[off:off + n].view(shape) for off, n, shape in ctx.views])


class _Slot:
    def __init__(self, key, ptrs, cap):
        self.key, self.ptrs, self.cap = key, ptrs, cap
        self.graph = None
        self.nodes = self.labels = None
        self.out = None


class StepGraphCache:
    def __init__(self, inter):
        self.inter = inter
        self.slots = {}
        self.stage_nodes = None
        self.stage_labels = None
        self.replays = 0
        self.captures = 0

    def _ids(self, nodes):
        if isinstance(nodes, torch.Tensor):
            return None if nodes.is_cuda else nodes.numpy().astype(np.int32, copy=False)
        return np.asarray(nodes, dtype=np.int32)

    # ------------------------------------------------------------------ applicability
    def usable(self, eng, table, B) -> bool:
        inter = self.inter
        return (inter.graph_cache and B > 0 and not torch.cuda.is_current_stream_capturing()
                and inter.score_override is None and not inter.scores_external and inter.cap_slots_hint is None
                and eng.score_group is None and eng._bcast is None and not eng.graph.partitioned
                and eng.grad_sink is None and not table.requires_grad)

    def _slot(self, eng, key, ptrs, host, build):
        need = eng.slots_bound(host, self.inter.thresholds, self.inter.intra_agg1.rho, True)
        slot = self.slots.get(key)
        if slot is not None and (slot.ptrs != ptrs or slot.cap < need):
            del self.slots[key]
            slot = None
        if slot is None:
            if len(self.slots) >= MAX_GRAPHS:
                self.slots.pop(next(iter(self.slots)))
            slot = _Slot(key, ptrs, max(int(need * 1.5) + 16, 64))
            build(slot)
            self.slots[key] = slot
            self.captures += 1
        return slot

    def _upload(self, slot, host_ids, nodes, labels, dev):
        B = slot.nodes.shape[0]
        if self.stage_nodes is None or self.stage_nodes.n < B:
            self.stage_nodes = PinnedStaging(max(B, 1024), torch.int32)
            self.stage_labels = PinnedStaging(max(B, 1024), torch.int64)
        if host_ids is not None:
            self.stage_nodes.upload(host_ids, slot.nodes)
        else:
            slot.nodes.copy_(nodes, non_blocking=True)
        if labels is not None and slot.labels is not None:
            if isinstance(labels, torch.Tensor):
                slot.labels.copy_(labels.reshape(-1), non_blocking=True)
            else:
                self.stage_labels.upload(np.asarray(labels, dtype=np.int64).reshape(-1), slot.labels)

    @staticmethod
    def _capture(fn, dev):
        """Two eager runs on a side stream (allocator, lazy attribute setup), then the recording."""
        lib = _lib.lib()
        prev = lib.pcg_set_pdl(2)             # programmatic dependent launch of the fused dense kernel (see pcg_set_pdl)
        try:
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s):
                for _ in range(2):
                    fn()
            torch.cuda.current_stream(dev).wait_stream(s)
            g = torch.cuda.CUDAGraph()
            with _lib.capture(g):
                out = fn()
        finally:
            lib.pcg_set_pdl(prev)
        return g, out

    # ------------------------------------------------------------------ training step
    def train_loss(self, eng, nodes, labels, head_weight, lam):
        """loss tensor (with autograd) of one training batch through a cached graph, or None when the ids live on
        the device (then there is nothing to upload: the caller uses the eager path or runtime.GraphedTrainStep)."""
        inter = self.inter
        host = self._ids(nodes)
        if host is None:
            return None
        B = host.shape[0]
        params = [head_weight, inter.label_clf.weight, inter.label_clf.bias, inter.weight] + \
                 [ia.weight for ia in inter.intra_aggs()]
        ptrs = tuple(p.data_ptr() for p in params) + (eng.feat.data_ptr(),)
        key = ("train", B, float(lam), float(inter.intra_agg1.rho), tuple(float(t) for t in inter.thresholds))
        dev = eng.device

        def build(slot):
            slot.nodes = torch.zeros(B, dtype=torch.int32, device=dev)
            slot.labels = torch.zeros(B, dtype=torch.int64, device=dev)
            slot.nodes.copy_(torch.from_numpy(host))               # a real batch for the warm-up runs
            sizes = [p.numel() for p in params]
            pad = [(n + 3) // 4 * 4 for n in sizes]
            slot.flat = torch.zeros(sum(pad), dtype=torch.float32, device=dev)
            slot.views, g, o = [], [], 0
            for p, n, q in zip(params, sizes, pad):
                slot.views.append((o, n, tuple(p.shape)))
                g.append(slot.flat[o:o + n].view_as(p))
                o += q
            grads = dict(head=g[0], clf_w=g[1], clf_b=g[2], inter=g[3], intra=g[4:])
            cont = [p.detach() for p in params]

            def fn():
                sel = inter._select(eng, slot.nodes, slot.labels, True, slot.cap)
                agg = eng.aggregate(sel, copy_dups=False)
                loss, out, center, _ = eng.tile_train(slot.nodes, slot.labels, agg, sel.it_rep, cont[4:], cont[3], cont[1],
                                                      cont[2], cont[0], lam, grads, pdl=inter.use_pdl)
                return loss, sel

            slot.graph, (slot.out, slot.sel) = self._capture(fn, dev)

        slot = self._slot(eng, key, ptrs, host, build)
        self._upload(slot, host, nodes, labels, dev)
        slot.graph.replay()
        self.replays += 1
        inter.last_selection = slot.sel
        loss = _ReplayLossFn.apply(slot.out, slot.flat, slot.views, *params)
        if fastloop.enabled():
            return fastloop.wrap(loss, slot.flat, slot.views, params)
        return loss

    # ------------------------------------------------------------------ forward without gradients (to_prob / eval)
    def infer(self, eng, nodes, labels, train_flag):
        """(combined [E,B], center [B,2]) of a no-grad forward through a cached graph, or None (device ids)."""
        inter = self.inter
        host = self._ids(nodes)
        if host is None:
            return None
        B = host.shape[0]
        params = [inter.label_clf.weight, inter.label_clf.bias, inter.weight] + [ia.weight for ia in inter.intra_aggs()]
        ptrs = tuple(p.data_ptr() for p in params) + (eng.feat.data_ptr(),)
        key = ("infer", B, bool(train_flag), float(inter.intra_agg1.rho), tuple(float(t) for t in inter.thresholds))
        dev = eng.device

        def build(slot):
            slot.nodes = torch.zeros(B, dtype=torch.int32, device=dev)
            slot.labels = torch.zeros(B, dtype=torch.int64, device=dev) if train_flag else None
            slot.nodes.copy_(torch.from_numpy(host))
            cont = [p.detach() for p in params]

            def fn():
                sel = inter._select(eng, slot.nodes, slot.labels, bool(train_flag), slot.cap)
                agg = eng.aggregate(sel, copy_dups=False)
                out, center, _ = eng.tile_fwd(slot.nodes, agg, sel.it_rep, cont[3:], cont[2], cont[0], cont[1], False)
                return (out, center), sel

            slot.graph, (slot.out, slot.sel) = self._capture(fn, dev)

        slot = self._slot(eng, key, ptrs, host, build)
        self._upload(slot, host, nodes, labels if train_flag else None, dev)
        slot.graph.replay()
        self.replays += 1
        inter.last_selection = slot.sel
        out, center = slot.out
        return out.clone(), center.clone()
