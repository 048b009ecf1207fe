"""Device-side runtime of the pick-and-choose path: owns the HBM-resident graph, the padded feature
table, the score table and the per-step scratch, and issues the C-ABI calls (``_lib``).

One engine per (graph, device). Everything is asynchronous on torch's current CUDA stream; the only
host<->device traffic per step is the upload of the target ids (and labels if they arrive on the
host), which the reference's ``forward(nodes: list, labels)`` signature makes unavoidable.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .graph import RelGraph

__all__ = ["Engine", "Selection", "PinnedStaging", "padded_ld"]


def padded_ld(feat_dim: int) -> int:
    """Row stride (floats) of the device feature table: one 128-byte line for F <= 32, else the next
    multiple of 4 (16-byte vector loads)."""
    return 32 if feat_dim <= 32 else (feat_dim + 3) // 4 * 4


class PinnedStaging:
    """Pinned host staging for small per-step uploads (target ids, labels): a ring of buffers, each guarded by an
    event recorded behind its host-to-device copy, so that the host never rewrites a buffer whose copy is still
    queued (back-to-back steps without a sync in between would otherwise train on the NEXT batch's ids)."""

    def __init__(self, n: int, dtype, depth: int = 3):
        self.n, self.dtype = int(n), dtype
        self.bufs = [torch.empty(self.n, dtype=dtype, pin_memory=True) for _ in range(depth)]
        self.events = [None] * depth
        self.i = 0

    def upload(self, host_array, dst: torch.Tensor):
        """dst[:len] <- host_array (numpy) through the next free pinned buffer, asynchronously."""
        k = len(host_array)
        i = self.i
        self.i = (i + 1) % len(self.bufs)
        if self.events[i] is not None:
            self.events[i].synchronize()          # the copy that last used this buffer has finished
        self.bufs[i].numpy()[:k] = host_array
        dst[:k].copy_(self.bufs[i][:k], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dst.device))
        self.events[i] = ev
        return dst[:k]


class Selection:
    """Result of a choose / select-all call: per item w = r*B + i an id list inside ``idx``."""

    __slots__ = ("B", "R", "idx", "slot_item", "it_slot0", "it_m", "it_base", "it_extra", "it_done", "it_rep",
                 "status", "cap_slots", "norm", "_blob")

    def lists(self):
        """Host copy: list over items of sorted id arrays (tests / compat API only: syncs)."""
        m, base = self.item_sizes()
        idx = self.idx.cpu().numpy()
        extra = self.it_extra.cpu().numpy() if self.it_extra is not None else None
        out = []
        for w in range(self.B * self.R):
            ids = idx[base[w]:base[w] + m[w]]
            if extra is not None and extra[w] >= 0:
                ids = np.append(ids, extra[w])
            out.append(np.sort(ids))
        return out

    def item_sizes(self):
        """Host copies of (m, base) per item. Only representative items carry sizes on the device
        (``it_rep``: repeated targets share the list of their first occurrence); resolved here."""
        m = self.it_m.cpu().numpy()
        base = self.it_base.cpu().numpy()
        if self.it_rep is not None:
            rep = self.it_rep.cpu().numpy()
            m, base = m[rep], base[rep]
        return m, base

    def overflowed(self) -> bool:
        return bool(self.status[_lib.ST_OVERFLOW].item())


class Engine:
    def __init__(self, graph: RelGraph | None, device=None):
        if not torch.cuda.is_available():
            raise _lib.PcgError("pcgnn_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.lib()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise _lib.PcgError(f"pcgnn_b200 runs on CUDA devices only (got {self.device})")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if self.device.index != torch.cuda.current_device():
            # the C ABI launches on the CURRENT device and keeps per-process side streams (one process drives one
            # GPU, like every multi-GPU run of this package): refuse instead of launching on the wrong device
            raise _lib.PcgError(f"engine for {self.device} but the current device is cuda:{torch.cuda.current_device()}: "
                                "call torch.cuda.set_device() first (one process per GPU)")
        self.graph = graph
        self.row_lo = 0
        if graph is not None:
            # N: rows held here; N_global: nodes of the whole graph (ids, features, scores and the pool are global)
            self.N, self.R = graph.n_nodes, graph.n_rel
            self.row_lo, self.N_global = graph.row_lo, graph.n_global
            if self.R > _lib.MAX_REL:
                raise ValueError(f"at most {_lib.MAX_REL} relations are supported")
            self.indptr, self.indices = graph.device(self.device)
            deg = np.diff(graph.indptr)
            self.max_degree = int(deg.max()) if deg.size else 0
        else:   # explicit-list use only (IntraAgg.forward / choose_step_* compat calls)
            self.N = self.N_global = self.R = self.max_degree = 0
            self.indptr = self.indices = None
        self.strict_rows = True     # feature table must have exactly one row per graph node
        self._feat_key = None
        self._feat_src = None
        self.feat = None            # [N, ldf] fp32, zero padded
        self.F = self.ldf = 0
        self.score = None           # [N]
        self.pool = None            # int32 [P]
        self.sorted_pool = None     # (ps_score, ps_pos, ps_id, workspace)
        self.pool_pos_of = None     # int32 [N]: node id -> pool position or -1
        self.entry_pool_pos = None  # int32 [nnz]: the same per CSR entry (coalesced reads in the kernels)
        self.P = 0
        self._pin = None
        self._ws = None
        self._ws_nodes = None
        self.score_group = None     # torch.distributed group over which the score slices are all-gathered (C5)
        # {parameter data_ptr: gradient view}: while set (runtime.GraphedTrainStep with a flat, pre-zeroed gradient
        # buffer), the backward kernels write a parameter's gradient straight into its view and autograd gets
        # None for it, which removes the AccumulateGrad add kernels from the step
        self.grad_sink = None
        self.grads_in_sinks = False  # set by layers.TrainStepFn when its forward stored the gradients into the sinks
        self._bcast = None          # (PeerRegion, epoch tensor): scores are broadcast into every rank's table (C5)

    # ------------------------------------------------------------------ resident tables
    def set_features(self, weight: torch.Tensor):
        """Padded device copy of the [N,F] feature table (re-made only when the source changes)."""
        # cache on the IDENTITY of the source tensor (kept alive here) + its version counter: a table built by a
        # `features` callable is a fresh tensor on every call (possibly at a recycled address) and is re-padded
        key = (weight._version, tuple(weight.shape), weight.device)
        if self._feat_src is weight and key == self._feat_key:
            return self.feat
        self._feat_src = weight
        w = weight.detach()
        if self.graph is not None and self.strict_rows and w.shape[0] != self.N_global:
            raise ValueError(f"feature table has {w.shape[0]} rows, graph has {self.N_global} nodes")
        F_ = w.shape[1]
        ld = padded_ld(F_)
        if ld == F_ and w.is_contiguous() and w.dtype == torch.float32 and w.device == self.device \
                and w.data_ptr() % 16 == 0:
            feat = w
        else:
            feat = torch.zeros((w.shape[0], ld), dtype=torch.float32, device=self.device)
            feat[:, :F_] = w.to(self.device, torch.float32)
        self.feat, self.F, self.ldf = feat, F_, ld
        self._feat_key = key
        if self.score is None and self.graph is not None:
            self.score = torch.empty(self.N_global, dtype=torch.float32, device=self.device)
        return feat

    def set_pool(self, train_pos):
        """Train-positive pool (order preserved: ties are broken by pool position, src/layers.py:687-690).
        A list / array of global node ids, or an int32 device tensor (C5: ~4e5 ids made on the GPU)."""
        if isinstance(train_pos, torch.Tensor):
            self.pool = train_pos.to(self.device, torch.int32).contiguous()
        else:
            self.pool = torch.from_numpy(np.asarray(list(train_pos), dtype=np.int32)).to(self.device)
        self.P = int(self.pool.shape[0])
        self.sorted_pool = self._alloc_sorted_pool(self.P)
        self.pool_pos_of = None
        self.entry_pool_pos = None
        if self.graph is not None:
            self.pool_pos_of = torch.empty(self.N_global, dtype=torch.int32, device=self.device)
            rc = self.lib.pcg_pool_positions(self.pool.data_ptr(), self.P, self.N_global, self.pool_pos_of.data_ptr(),
                                             _lib.stream_ptr())
            _lib.check(rc, "pcg_pool_positions")
            if self.P <= _lib.KB_MAX_POOL:      # larger pools use the row-position test, not the per-item bitmap
                self.entry_pool_pos = torch.empty(max(self.indices.shape[0], 1), dtype=torch.int32, device=self.device)
                rc = self.lib.pcg_entry_pool_positions(self.indices.data_ptr(), self.indices.shape[0],
                                                       self.pool_pos_of.data_ptr(), self.entry_pool_pos.data_ptr(),
                                                       _lib.stream_ptr())
                _lib.check(rc, "pcg_entry_pool_positions")

    def _alloc_sorted_pool(self, P):
        n = max(P, 1)
        dev = self.device
        ws = torch.empty(int(self.lib.pcg_sort_pool_workspace_bytes(P)), dtype=torch.uint8, device=dev)
        return (torch.empty(n, dtype=torch.float32, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                torch.empty(n, dtype=torch.int32, device=dev), ws)

    def sort_pool(self, pool, pool_score):
        """Score-sorted view of an explicit pool (``pcg_sort_pool``): (ps_score, ps_pos, ps_id)."""
        P = int(pool.shape[0])
        ps, pp, pi, ws = self._alloc_sorted_pool(P)
        rc = self.lib.pcg_sort_pool(pool_score.data_ptr(), pool.data_ptr(), P, ps.data_ptr(), pp.data_ptr(),
                                    pi.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
        _lib.check(rc, "pcg_sort_pool")
        return ps, pp, pi

    def score_table(self, clf_weight: torch.Tensor, clf_bias: torch.Tensor):
        """score[v] = <feat[v], clf_weight[0]> + clf_bias[0] for all nodes, then the pool sorted by it.

        Row-partitioned graph with ``score_group`` set (C5): every rank scores only the nodes whose rows it
        holds and the slices are all-gathered (the halo exchange of the partitioned path: neighbours' scores
        outside the rank's node range come from their owners), then the pool is sorted from the full table."""
        w = clf_weight.detach()
        b = clf_bias.detach()
        if not w.is_contiguous():
            w = w.contiguous()
        ps, pp, pi, ws = self.sorted_pool if self.pool is not None else (None, None, None, None)
        if self._bcast is not None:
            region, epoch = self._bcast
            lo = self.row_lo
            rc = self.lib.pcg_score_bcast(self.feat.data_ptr() + lo * self.ldf * 4, self.N, self.F, self.ldf,
                                          w.data_ptr(), b.data_ptr(), lo, self.N_global, region.regions, region.rank,
                                          region.world, epoch.data_ptr(), _lib.stream_ptr())
            _lib.check(rc, "pcg_score_bcast")
            self.resort_pool()
            return self.score
        if self.score_group is not None:
            self.score_local(w, b)
            self.score_exchange()
            self.resort_pool()
            return self.score
        rc = self.lib.pcg_score_table(self.feat.data_ptr(), self.N_global, self.F, self.ldf, w.data_ptr(), b.data_ptr(),
                                      self.score.data_ptr(), _lib.ptr(self.pool), self.P, _lib.ptr(ps), _lib.ptr(pp),
                                      _lib.ptr(pi), _lib.ptr(ws), 0 if ws is None else ws.numel(), _lib.stream_ptr())
        _lib.check(rc, "pcg_score_table")
        return self.score

    def stage(self, src_ptr: int, dst_ptr: int, nbytes: int, cursor_ptr: int = 0, count: int = 0, src_stride: int = 0):
        """Copy by a kernel (``pcg_stage``): either side may be page-locked host memory (device address from
        ``host_device_ptr``); keeps a recorded step free of memcpy nodes. With a device cursor word the source is entry
        ``*cursor % count`` of a plan (``pcg_stage_indexed``)."""
        if cursor_ptr:
            _lib.check(self.lib.pcg_stage_indexed(src_ptr, dst_ptr, int(nbytes), cursor_ptr, int(count), int(src_stride), 0,
                                                  0, _lib.stream_ptr()), "pcg_stage_indexed")
        else:
            _lib.check(self.lib.pcg_stage(src_ptr, dst_ptr, int(nbytes), _lib.stream_ptr()), "pcg_stage")

    def pool_scores(self, clf_weight: torch.Tensor, clf_bias: torch.Tensor, stage=None):
        """Scores of the pool members only (``pcg_pool_scores``; bit-identical to the table's values): the pool sort
        can then run next to the score-table kernel / the score exchange instead of behind it.
        stage = (src_ptr, dst_ptr, nbytes[, cursor_ptr, count, src_stride]): that copy rides on extra CTAs of the kernel
        (``pcg_pool_scores_stage``); with a cursor the source is entry ``*cursor % count`` of an epoch plan."""
        if not self.P:
            if stage is not None:
                self.stage(*stage)
            return None
        if getattr(self, "_pool_score", None) is None or self._pool_score.shape[0] != self.P:
            self._pool_score = torch.empty(self.P, dtype=torch.float32, device=self.device)
        w = clf_weight.detach()
        w = w if w.is_contiguous() else w.contiguous()
        if stage is not None:
            rc = self.lib.pcg_pool_scores_stage(self.feat.data_ptr(), self.F, self.ldf, w.data_ptr(),
                                                clf_bias.detach().data_ptr(), self.pool.data_ptr(), self.P,
                                                self._pool_score.data_ptr(), stage[0], stage[1], int(stage[2]),
                                                stage[3] if len(stage) > 3 else None, int(stage[4]) if len(stage) > 3 else 0,
                                                int(stage[5]) if len(stage) > 3 else 0, _lib.stream_ptr())
        else:
            rc = self.lib.pcg_pool_scores(self.feat.data_ptr(), self.F, self.ldf, w.data_ptr(),
                                          clf_bias.detach().data_ptr(), self.pool.data_ptr(), self.P,
                                          self._pool_score.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_pool_scores")
        return self._pool_score

    def sort_pool_from(self, pool_score: torch.Tensor):
        """Sort the resident pool by the given per-position scores into the engine's sorted-pool arrays."""
        ps, pp, pi, ws = self.sorted_pool
        rc = self.lib.pcg_sort_pool(pool_score.data_ptr(), self.pool.data_ptr(), self.P, ps.data_ptr(), pp.data_ptr(),
                                    pi.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
        _lib.check(rc, "pcg_sort_pool")

    def score_table_only(self, clf_weight: torch.Tensor, clf_bias: torch.Tensor):
        """The score table without the pool sort (the caller sorts the pool from ``pool_scores`` on another stream).
        Row partitions exchange their slices as ``score_table`` does."""
        w = clf_weight.detach()
        w = w if w.is_contiguous() else w.contiguous()
        b = clf_bias.detach()
        if self._bcast is not None:
            region, epoch = self._bcast
            lo = self.row_lo
            rc = self.lib.pcg_score_bcast(self.feat.data_ptr() + lo * self.ldf * 4, self.N, self.F, self.ldf,
                                          w.data_ptr(), b.data_ptr(), lo, self.N_global, region.regions, region.rank,
                                          region.world, epoch.data_ptr(), _lib.stream_ptr())
            _lib.check(rc, "pcg_score_bcast")
            return self.score
        if self.score_group is not None:
            self.score_local(w, b)
            self.score_exchange()
            return self.score
        rc = self.lib.pcg_score_table(self.feat.data_ptr(), self.N_global, self.F, self.ldf, w.data_ptr(), b.data_ptr(),
                                      self.score.data_ptr(), None, 0, None, None, None, None, 0, _lib.stream_ptr())
        _lib.check(rc, "pcg_score_table")
        return self.score

    def enable_score_broadcast(self, group=None):
        """Row-partitioned graph, several ranks: keep the score table in memory that every peer has mapped, so that
        ``score_table`` becomes slice kernel + stores into all peers' tables + arrival wait (``pcg_score_bcast``),
        capturable in the step graph. For training steps (see the write-after-read note in csrc/pcg_comm.cu)."""
        from .parallel import PeerRegion

        region = PeerRegion(int(self.lib.pcg_score_region_bytes(self.N_global)), group)
        if region.world == 1:
            return
        if region.world * self.N != self.N_global:
            raise ValueError("score broadcast needs equal row ranges (n_global == world * rows per rank)")

        class _Mem:      # __cuda_array_interface__ view of the region's table
            def __init__(self, ptr, n):
                self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}

        self._score_mem = _Mem(region.own, self.N_global)
        self.score = torch.as_tensor(self._score_mem, device=self.device)
        self._bcast = (region, torch.zeros(1, dtype=torch.int32, device=self.device))
        self.score_group = None

    def score_local(self, w: torch.Tensor, b: torch.Tensor):
        """Partitioned graph: scores of the nodes whose rows live here, written into their slice of the table."""
        lo = self.row_lo
        rc = self.lib.pcg_score_table(self.feat.data_ptr() + lo * self.ldf * 4, self.N, self.F, self.ldf,
                                      w.detach().data_ptr(), b.detach().data_ptr(), self.score.data_ptr() + lo * 4,
                                      None, 0, None, None, None, None, 0, _lib.stream_ptr())
        _lib.check(rc, "pcg_score_table")

    def score_exchange(self):
        """All-gather of the score slices over ``score_group`` (the halo exchange of the partitioned path)."""
        import torch.distributed as dist

        world = dist.get_world_size(self.score_group)
        if world * self.N != self.N_global:
            raise ValueError("score exchange needs equal row ranges (n_global == world * rows per rank)")
        dist.all_gather_into_tensor(self.score, self.score[self.row_lo:self.row_lo + self.N], group=self.score_group)

    def resort_pool(self):
        """Re-sort the resident pool after ``self.score`` was written by someone else (tests inject a table)."""
        if self.P:
            ps, pp, pi, ws = self.sorted_pool
            gathered = self.score[self.pool.long()].contiguous()
            rc = self.lib.pcg_sort_pool(gathered.data_ptr(), self.pool.data_ptr(), self.P, ps.data_ptr(), pp.data_ptr(),
                                        pi.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
            _lib.check(rc, "pcg_sort_pool")

    # ------------------------------------------------------------------ per-step inputs
    def upload_targets(self, nodes):
        """int32 device tensor of the batch's node ids (+ the host copy, for capacity sizing)."""
        if isinstance(nodes, torch.Tensor):
            if nodes.is_cuda:
                return nodes.to(torch.int32), None
            host = nodes.numpy().astype(np.int32, copy=False)
        else:
            host = np.asarray(nodes, dtype=np.int32)
        B = host.shape[0]
        if self._pin is None or self._pin.n < B:
            self._pin = PinnedStaging(max(B, 1024), torch.int32)
        dst = torch.empty(B, dtype=torch.int32, device=self.device)
        return self._pin.upload(host, dst), host

    def slots_bound(self, host_targets, thresh, rho, train) -> int:
        """Upper bound of the slots a batch needs: the graph's per-node choose demand summed over the host ids (every
        target counted as positive when training, since labels may live on the device)."""
        demand = self.graph.choose_slot_demand(thresh, rho, self.P, train)
        return max(int(demand[np.asarray(host_targets, dtype=np.int64) - self.row_lo].sum()), 1)

    # ------------------------------------------------------------------ kernels
    def _new_selection(self, B, R, cap_slots, with_sel_idx, with_extra):
        W = B * R
        dev = self.device
        # one allocation, carved into typed views (int64 part first for alignment)
        n64 = W
        n32 = (cap_slots * _lib.SLOT if with_sel_idx else 0) + cap_slots + 4 * W + (W if with_extra else 0) \
            + _lib.STATUS_WORDS
        blob = torch.empty(n64 * 2 + n32, dtype=torch.int32, device=dev)
        s = Selection()
        s._blob = blob
        s.B, s.R, s.cap_slots = B, R, cap_slots
        s.it_base = blob[:n64 * 2].view(torch.int64)
        o = n64 * 2

        def take(n):
            nonlocal o
            v = blob[o:o + n]
            o += n
            return v

        s.idx = take(cap_slots * _lib.SLOT) if with_sel_idx else self.indices
        s.slot_item = take(cap_slots)
        s.it_slot0 = take(W)
        s.it_m = take(W)
        s.it_done = take(W)
        s.it_extra = take(W) if with_extra else None
        s.it_rep = take(W) if with_sel_idx else None
        s.status = take(_lib.STATUS_WORDS)
        s.norm = _lib.NORM_MEAN
        return s

    def choose(self, targets, labels, train: bool, thresh, rho: float, cap_slots: int, *,
               entry_score=None, center_score=None, k_override=None, sorted_pool=None,
               indptr=None, indices=None, n_nodes=None, n_rel=None, max_degree=None,
               want_dist: bool = False, phases: int = 3, sel: Selection | None = None, workspace=None):
        """Top-k filter + oversample for every (relation, target) item (``pcg_choose``).

        Default: the engine's resident graph, score table and pool. The keyword overrides carry the
        explicit-list calling convention of IntraAgg.forward / choose_step_* (src/layers.py:562, 633).
        Returns the Selection (and the distance buffer when want_dist).
        phases=1 runs only the score-independent preparation (callers put it on a side stream next to
        ``score_table``), phases=2 the selection on the Selection a phases=1 call returned.
        workspace: a caller-owned uint8 device buffer of at least ``pcg_choose_workspace_bytes`` bytes, initialised
        by ``pcg_choose_workspace_init`` for this node count, used instead of the engine's shared one (which grows, and
        so moves, with the batch size: a recorded graph that must outlive other calls brings its own)."""
        B = int(targets.shape[0])
        R = self.R if n_rel is None else n_rel
        s = sel if sel is not None else self._new_selection(B, R, cap_slots, True, False)
        maxdeg = self.max_degree if max_degree is None else max_degree
        nn_ = self.N if n_nodes is None else n_nodes
        ws_bytes = self.lib.pcg_choose_workspace_bytes(B, R, maxdeg, nn_)
        if workspace is not None:
            if workspace.numel() < ws_bytes:
                raise _lib.PcgError(f"choose workspace has {workspace.numel()} bytes, this call needs {ws_bytes}")
            ws = workspace
        elif self._ws is None or self._ws.numel() < ws_bytes or self._ws_nodes != nn_:
            # the head of the workspace is the per-node "first occurrence" table, which the kernels expect
            # (and leave) all-0x7f: initialise it whenever the buffer or the node count behind it changes
            if self._ws is None or self._ws.numel() < ws_bytes:
                self._ws = torch.empty(int(ws_bytes), dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.pcg_choose_workspace_init(self._ws.data_ptr(), self._ws.numel(), nn_, _lib.stream_ptr()),
                       "pcg_choose_workspace_init")
            self._ws_nodes = nn_
        if workspace is None:
            ws = self._ws
        th = (C.c_double * R)(*[float(x) for x in thresh])
        use_table = entry_score is None
        if sorted_pool is None and self.sorted_pool is not None and use_table:
            sorted_pool = self.sorted_pool[:3]
        ps, pp, pi = sorted_pool if sorted_pool is not None else (None, None, None)
        P = (self.P if use_table else int(ps.shape[0])) if ps is not None else 0
        dist = torch.empty(cap_slots * _lib.SLOT, dtype=torch.float32, device=self.device) if want_dist else None
        rc = self.lib.pcg_choose(
            (self.indptr if indptr is None else indptr).data_ptr(),
            (self.indices if indices is None else indices).data_ptr(),
            self.N if n_nodes is None else n_nodes, self.row_lo if n_nodes is None else 0, R,
            (self.score.data_ptr() if self.score is not None else None) if use_table else None, _lib.ptr(entry_score),
            _lib.ptr(center_score),
            targets.data_ptr(), _lib.ptr(labels) if train else None, B, th, _lib.ptr(k_override), float(rho),
            _lib.ptr(ps), _lib.ptr(pp), _lib.ptr(pi), _lib.ptr(self.entry_pool_pos) if use_table else None, P,
            int(bool(train)), maxdeg, s.idx.data_ptr(), _lib.ptr(dist),
            cap_slots, s.slot_item.data_ptr(), s.it_slot0.data_ptr(), s.it_m.data_ptr(), s.it_base.data_ptr(),
            s.it_done.data_ptr(), s.it_rep.data_ptr(), ws.data_ptr(), int(ws_bytes), s.status.data_ptr(),
            int(phases), _lib.stream_ptr())
        _lib.check(rc, "pcg_choose")
        return (s, dist) if want_dist else s

    def overflow_since_reset(self) -> bool:
        """True if ANY choose call since the last query ran out of slots (or met a target whose row this partition
        does not hold): the kernels OR their flag into a workspace word that, unlike a call's status block, survives
        later calls and CUDA-graph replays. Reads and clears it. Syncs."""
        if self._ws is None:
            return False
        off = int(self.lib.pcg_choose_sticky_offset(self._ws_nodes))
        word = self._ws[off:off + 4].view(torch.int32)
        hit = bool(word.item())
        if hit:
            word.zero_()
        return hit

    def select_all(self, targets, add_self: bool, cap_slots: int, norm: int) -> Selection:
        """GraphSAGE / GCN selection: whole rows (∪ self), no copy (``pcg_select_all``)."""
        if self.graph is not None and self.graph.partitioned:
            raise NotImplementedError("select-all runs on unpartitioned graphs only")
        B = int(targets.shape[0])
        s = self._new_selection(B, self.R, cap_slots, False, True)
        s.norm = norm
        rc = self.lib.pcg_select_all(self.indptr.data_ptr(), self.indices.data_ptr(), self.N, self.R,
                                     targets.data_ptr(), B, int(bool(add_self)), cap_slots, s.slot_item.data_ptr(),
                                     s.it_slot0.data_ptr(), s.it_m.data_ptr(), s.it_base.data_ptr(),
                                     s.it_extra.data_ptr(), s.it_done.data_ptr(), s.status.data_ptr(),
                                     _lib.stream_ptr())
        _lib.check(rc, "pcg_select_all")
        return s

    def aggregate(self, sel: Selection, feat=None, copy_dups: bool = True) -> torch.Tensor:
        """agg [R*B, ldf] = normalised sum of the selected rows (``pcg_aggregate``). copy_dups=False leaves the
        rows of repeated targets unwritten: the consumer must read row ``sel.it_rep[w]`` (dense_fwd / dense_bwd do)."""
        feat = self.feat if feat is None else feat
        ldf = feat.shape[1]
        W = sel.B * sel.R
        agg = torch.empty((W, ldf), dtype=torch.float32, device=self.device)
        partial = torch.empty((sel.cap_slots, ldf), dtype=torch.float32, device=self.device)
        rc = self.lib.pcg_aggregate(feat.data_ptr(), ldf, sel.idx.data_ptr(), sel.slot_item.data_ptr(),
                                    sel.it_slot0.data_ptr(), sel.it_m.data_ptr(), sel.it_base.data_ptr(),
                                    _lib.ptr(sel.it_extra), _lib.ptr(sel.it_rep), int(copy_dups), W, sel.cap_slots,
                                    sel.status.data_ptr(), sel.norm, partial.data_ptr(), sel.it_done.data_ptr(),
                                    agg.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_aggregate")
        return agg

    def aggregate_bwd(self, sel: Selection, d_agg: torch.Tensor, feat_grad: torch.Tensor):
        """feat_grad[j] += d_agg[w] * norm for every selected j (``pcg_aggregate_bwd``)."""
        ldf = feat_grad.shape[1]
        W = sel.B * sel.R
        d_agg = d_agg.contiguous()
        if sel.it_rep is not None:      # duplicates' gradients flow through their representative's list
            folded = torch.zeros_like(d_agg)
            folded.index_add_(0, sel.it_rep.long(), d_agg)
            d_agg = folded
        rc = self.lib.pcg_aggregate_bwd(d_agg.data_ptr(), ldf, sel.idx.data_ptr(), sel.slot_item.data_ptr(),
                                        sel.it_slot0.data_ptr(), sel.it_m.data_ptr(), sel.it_base.data_ptr(),
                                        _lib.ptr(sel.it_extra), W, sel.cap_slots, sel.status.data_ptr(), sel.norm,
                                        feat_grad.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_aggregate_bwd")
        return feat_grad

    # ------------------------------------------------------------------ fused dense part
    def dense_fwd(self, targets, agg, w_intra, w_inter, feat_dim, agg_rep=None):
        """(combined [E,B], cat [B, F+R*E]) = relation transforms + inter-relation combine (``pcg_dense_fwd``)."""
        B = int(targets.shape[0])
        R = len(w_intra)
        E = int(w_inter.shape[1])
        K2 = feat_dim + R * E
        cat = torch.empty((B, K2), dtype=torch.float32, device=self.device)
        out = torch.empty((E, B), dtype=torch.float32, device=self.device)
        ptrs = (C.c_void_p * R)(*[w.data_ptr() for w in w_intra])
        rc = self.lib.pcg_dense_fwd(self.feat.data_ptr(), self.ldf, feat_dim, targets.data_ptr(), B, R, E,
                                    agg.data_ptr(), _lib.ptr(agg_rep), ptrs, w_inter.data_ptr(), cat.data_ptr(), out.data_ptr(),
                                    _lib.stream_ptr())
        _lib.check(rc, "pcg_dense_fwd")
        return out, cat

    # ------------------------------------------------------------------ fused dense part (csrc/pcg_tile.cu)
    def tile_supported(self, B: int, R: int, E: int) -> bool:
        return B > 0 and bool(self.lib.pcg_tile_supported(int(B), int(R), int(self.F), int(E)))

    def tile_fwd(self, targets, agg, agg_rep, w_intra, w_inter, w_clf, b_clf, keep_cat: bool):
        """(combined [E,B], center [B,2] or None, cat [B,F+R*E] or None): relation transforms + combine + label_clf
        head as ONE kernel (``pcg_tile_fwd``); cat is kept only for the autograd backward (``dense_bwd``)."""
        B, R, E = int(targets.shape[0]), len(w_intra), int(w_inter.shape[1])
        dev = self.device
        out = torch.empty((E, B), dtype=torch.float32, device=dev)
        center = torch.empty((B, 2), dtype=torch.float32, device=dev) if w_clf is not None else None
        cat = torch.empty((B, self.F + R * E), dtype=torch.float32, device=dev) if keep_cat else None
        ptrs = (C.c_void_p * R)(*[w.data_ptr() for w in w_intra])
        rc = self.lib.pcg_tile_fwd(self.feat.data_ptr(), self.ldf, self.F, targets.data_ptr(), B, R, E, agg.data_ptr(),
                                   agg.shape[1], _lib.ptr(agg_rep), ptrs, w_inter.data_ptr(), _lib.ptr(w_clf),
                                   _lib.ptr(b_clf), int(bool(keep_cat)), out.data_ptr(), _lib.ptr(center),
                                   _lib.ptr(cat), _lib.stream_ptr())
        _lib.check(rc, "pcg_tile_fwd")
        return out, center, cat

    def tile_train(self, targets, labels, agg, agg_rep, w_intra, w_inter, w_clf, b_clf, w_head, lam, grads,
                   want_logits=False, pdl=False):
        """One fused training pass behind the aggregation (``pcg_tile_train``): loss and ALL weight gradients.
        grads = dict(inter=, intra=[...], clf_w=, clf_b=, head=) of contiguous fp32 tensors that are overwritten.
        Returns (loss 0-d, combined [E,B], center [B,2], logits [B,2] or None)."""
        B, R, E = int(targets.shape[0]), len(w_intra), int(w_inter.shape[1])
        dev = self.device
        buf = torch.empty(E * B + 2 * B + (2 * B if want_logits else 0) + 1, dtype=torch.float32, device=dev)
        out = buf[:E * B].view(E, B)
        center = buf[E * B:E * B + 2 * B].view(B, 2)
        logits = buf[E * B + 2 * B:E * B + 4 * B].view(B, 2) if want_logits else None
        loss = buf[-1:]
        scratch = torch.empty(int(self.lib.pcg_tile_scratch_floats(B, R, self.F, E)), dtype=torch.float32, device=dev)
        ptrs = (C.c_void_p * R)(*[w.data_ptr() for w in w_intra])
        gptrs = (C.c_void_p * R)(*[g.data_ptr() for g in grads["intra"]])
        rc = self.lib.pcg_tile_train(self.feat.data_ptr(), self.ldf, self.F, targets.data_ptr(), B, R, E, agg.data_ptr(),
                                     agg.shape[1], _lib.ptr(agg_rep), ptrs, w_inter.data_ptr(), w_clf.data_ptr(),
                                     b_clf.data_ptr(), w_head.data_ptr(), labels.data_ptr(), float(lam), out.data_ptr(),
                                     center.data_ptr(), _lib.ptr(logits), loss.data_ptr(), gptrs,
                                     grads["inter"].data_ptr(), grads["clf_w"].data_ptr(), grads["clf_b"].data_ptr(),
                                     grads["head"].data_ptr(), scratch.data_ptr(), int(bool(pdl)), _lib.stream_ptr())
        _lib.check(rc, "pcg_tile_train")
        return loss.view(()), out, center, logits

    def fork_point(self):
        """A (4-byte memset) node in front of a stream fork. Inside a captured CUDA graph two ROOT branches start
        several microseconds apart (measured: the second root kernel began 5 us after the first one had ended),
        while branches that fork behind a common predecessor start together."""
        if getattr(self, "_fork_word", None) is None:
            self._fork_word = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._fork_word.zero_()

    def side_stream(self, which: int = 0):
        if getattr(self, "_sides", None) is None:
            self._sides = {}
        if which not in self._sides:
            # high priority: the side branches are short kernels that must get SM slots next to the main branch
            self._sides[which] = torch.cuda.Stream(device=self.device, priority=-1)
        return self._sides[which]

    def sink_of(self, param):
        """Gradient view registered for this parameter tensor, or None."""
        return None if self.grad_sink is None else self.grad_sink.get(param.data_ptr())

    def dense_bwd(self, agg, w_inter, cat, out, d_out, feat_dim, n_rel, agg_rep=None, sinks=None):
        """Weight gradients of the fused dense part (``pcg_dense_bwd``): (list of dW_r [2F,E], dW [F+R*E,E]).
        sinks = (d_inter_view, [d_intra_views]) writes them in place instead of into fresh buffers."""
        B = int(cat.shape[0])
        E = int(w_inter.shape[1])
        K2 = feat_dim + n_rel * E
        n = int(self.lib.pcg_dense_bwd_scratch_floats(B, n_rel, feat_dim, E))
        scratch = torch.empty(n, dtype=torch.float32, device=self.device)
        # one buffer for all gradients: [dW (K2*E) | dW_1 (2F*E) | ... ]
        if sinks is not None:
            d_inter, d_intra = sinks
        else:
            flat = torch.empty(K2 * E + n_rel * 2 * feat_dim * E, dtype=torch.float32, device=self.device)
            d_inter = flat[:K2 * E].view(K2, E)
            d_intra = [flat[K2 * E + r * 2 * feat_dim * E: K2 * E + (r + 1) * 2 * feat_dim * E].view(2 * feat_dim, E)
                       for r in range(n_rel)]
        ptrs = (C.c_void_p * n_rel)(*[g.data_ptr() for g in d_intra])
        d_out = d_out.contiguous()
        rc = self.lib.pcg_dense_bwd(agg.shape[1], feat_dim, B, n_rel, E, agg.data_ptr(), _lib.ptr(agg_rep), w_inter.data_ptr(),
                                    cat.data_ptr(), out.data_ptr(), d_out.data_ptr(), ptrs, d_inter.data_ptr(),
                                    scratch.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_dense_bwd")
        return d_intra, d_inter

    # ------------------------------------------------------------------ GraphSAGE / GCN encoder (csrc/pcg_homo.cu)
    def encoder_fwd(self, agg, w, targets=None):
        """out [E,B] = relu(W @ X^T), X = agg rows or [feat[targets] | agg] (``pcg_encoder_fwd``)."""
        B, E = int(agg.shape[0]), int(w.shape[0])
        out = torch.empty((E, B), dtype=torch.float32, device=self.device)
        rc = self.lib.pcg_encoder_fwd(agg.data_ptr(), agg.stride(0), self.feat.data_ptr() if targets is not None else None,
                                      self.ldf, _lib.ptr(targets), self.F, w.data_ptr(), B, E, out.data_ptr(),
                                      _lib.stream_ptr())
        _lib.check(rc, "pcg_encoder_fwd")
        return out

    def encoder_bwd(self, agg, out, d_out, targets=None, sink=None):
        """d_w [E, F or 2F] of the encoder (``pcg_encoder_bwd``)."""
        B, E = int(agg.shape[0]), int(out.shape[0])
        f_in = self.F * (2 if targets is not None else 1)
        d_w = sink if sink is not None else torch.empty((E, f_in), dtype=torch.float32, device=self.device)
        scratch = torch.empty(int(self.lib.pcg_encoder_scratch_floats(B, f_in, E)), dtype=torch.float32, device=self.device)
        rc = self.lib.pcg_encoder_bwd(agg.data_ptr(), agg.stride(0), self.feat.data_ptr() if targets is not None else None,
                                      self.ldf, _lib.ptr(targets), self.F, B, E, out.data_ptr(), d_out.contiguous().data_ptr(),
                                      d_w.data_ptr(), scratch.data_ptr(), self._tickets()[3:].data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_encoder_bwd")
        return d_w

    # ------------------------------------------------------------------ heads
    def _tickets(self):
        if getattr(self, "_ticket_buf", None) is None:
            self._ticket_buf = torch.zeros(8, dtype=torch.int32, device=self.device)
        return self._ticket_buf

    def center_fwd(self, targets, w, b):
        """center [B,2] = label_clf on the targets' own features (``pcg_center_fwd``)."""
        B = int(targets.shape[0])
        out = torch.empty((B, 2), dtype=torch.float32, device=self.device)
        rc = self.lib.pcg_center_fwd(self.feat.data_ptr(), self.ldf, self.F, targets.data_ptr(), B, w.data_ptr(),
                                     b.data_ptr(), out.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_center_fwd")
        return out

    def center_bwd(self, targets, d_center, sinks=None):
        B = int(targets.shape[0])
        if sinks is not None:
            d_w, d_b = sinks
        else:
            flat = torch.empty(2 * self.F + 2, dtype=torch.float32, device=self.device)
            d_w, d_b = flat[:2 * self.F].view(2, self.F), flat[2 * self.F:]
        scratch = torch.empty(int(self.lib.pcg_head_scratch_floats(B, self.F, 1)), dtype=torch.float32,
                              device=self.device)
        d_center = d_center.contiguous()
        rc = self.lib.pcg_center_bwd(self.feat.data_ptr(), self.ldf, self.F, targets.data_ptr(), B, d_center.data_ptr(),
                                     d_w.data_ptr(), d_b.data_ptr(), scratch.data_ptr(),
                                     self._tickets()[0:].data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_center_bwd")
        return d_w, d_b

    def head_loss_fwd(self, emb, w, center, labels, lam):
        E, B = int(emb.shape[0]), int(emb.shape[1])
        buf = torch.empty(4 * B + 1, dtype=torch.float32, device=self.device)
        logits, p1, q1, loss = buf[:2 * B].view(B, 2), buf[2 * B:3 * B], buf[3 * B:4 * B], buf[4 * B:]
        scratch = torch.empty(int(self.lib.pcg_head_scratch_floats(B, 1, E)), dtype=torch.float32, device=self.device)
        rc = self.lib.pcg_head_loss_fwd(emb.data_ptr(), E, B, w.data_ptr(), center.data_ptr(), labels.data_ptr(),
                                        float(lam), logits.data_ptr(), p1.data_ptr(), q1.data_ptr(), loss.data_ptr(),
                                        scratch.data_ptr(), self._tickets()[1:].data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_head_loss_fwd")
        return loss.view(()), logits, p1, q1

    def head_loss_bwd(self, emb, w, labels, p1, q1, lam, d_loss, sink=None):
        E, B = int(emb.shape[0]), int(emb.shape[1])
        d_emb = torch.empty((E, B), dtype=torch.float32, device=self.device)
        d_center = torch.empty((B, 2), dtype=torch.float32, device=self.device)
        d_w = sink if sink is not None else torch.empty((2, E), dtype=torch.float32, device=self.device)
        scratch = torch.empty(int(self.lib.pcg_head_scratch_floats(B, 1, E)), dtype=torch.float32, device=self.device)
        d_loss = d_loss.contiguous()
        rc = self.lib.pcg_head_loss_bwd(emb.data_ptr(), E, B, w.data_ptr(), labels.data_ptr(), p1.data_ptr(),
                                        q1.data_ptr(), float(lam), d_loss.data_ptr(), d_emb.data_ptr(),
                                        d_center.data_ptr(), d_w.data_ptr(), scratch.data_ptr(),
                                        self._tickets()[2:].data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "pcg_head_loss_bwd")
        return d_emb, d_center, d_w
