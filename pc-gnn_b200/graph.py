"""HBM-resident multi-relation CSR graph.

The reference keeps every relation as a ``defaultdict(set)`` built by
``sparse_to_adjlist`` (/root/reference/src/utils.py:226-254: self loop on every
node, every edge stored in both directions) and walks it with Python set
operations once per target per step (/root/reference/src/layers.py:216-227).
Here the R relations are stacked into ONE CSR whose row ``r * N + v`` is the
neighbour list of node ``v`` under relation ``r``, ids ascending, so a kernel
work item ``(target, relation)`` is a single row lookup.

Layout (all contiguous, device copies made once):
  indptr   int64  [R*N + 1]   row offsets into ``indices``
  indices  int32  [nnz]       neighbour ids, ascending inside a row
"""
from __future__ import annotations

import numpy as np

from ._lib import SLOT

__all__ = ["RelGraph", "csr_from_edges", "adj_lists_from_csr", "item_slots"]


def item_slots(d, c, rho, P, train):
    """Slots the choose kernel gives items with row lengths ``d`` and kept counts ``c`` (int64 arrays): k kept ids, plus
    the oversampled pool members when training, in whole slots. Mirrors ``item_counts()`` in csrc/pcg_common.cuh, with
    every target counted as positive."""
    k = np.where(d > c + 1, c, d)
    o = np.minimum((c * float(rho)).astype(np.int64), P) if train else 0
    return (k + o + SLOT - 1) // SLOT


def csr_from_edges(n_nodes: int, src, dst, *, symmetric: bool = True, self_loops: bool = True):
    """(indptr int64 [N+1], indices int32 [nnz]) from an edge list.

    Mirrors what ``sparse_to_adjlist`` produces (utils.py:233 adds the identity,
    :238-239 inserts both directions), with duplicate edges merged the way a
    ``set`` merges them and every row sorted by neighbour id.
    """
    src = np.asarray(src, dtype=np.int64).ravel()
    dst = np.asarray(dst, dtype=np.int64).ravel()
    parts_s, parts_d = [src], [dst]
    if symmetric:
        parts_s.append(dst)
        parts_d.append(src)
    if self_loops:
        ar = np.arange(n_nodes, dtype=np.int64)
        parts_s.append(ar)
        parts_d.append(ar)
    s = np.concatenate(parts_s)
    d = np.concatenate(parts_d)
    if s.size and (s.min() < 0 or d.min() < 0 or s.max() >= n_nodes or d.max() >= n_nodes):
        raise ValueError("edge endpoint outside [0, n_nodes)")
    key = s * np.int64(n_nodes) + d
    key.sort(kind="stable")            # radix path; np.unique's hash path is ~10x slower here
    if key.size:
        key = key[np.concatenate(([True], key[1:] != key[:-1]))]
    rows = key // n_nodes
    indices = (key - rows * n_nodes).astype(np.int32)
    indptr = np.zeros(n_nodes + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=n_nodes), out=indptr[1:])
    return indptr, indices


def adj_lists_from_csr(indptr, indices, rows=None):
    """dict[int -> set[int]] view of (some rows of) one relation, the shape the
    reference's layers index with ``adj_list[int(node)]`` (layers.py:219)."""
    from collections import defaultdict

    out = defaultdict(set)
    it = range(len(indptr) - 1) if rows is None else rows
    for v in it:
        v = int(v)
        out[v] = set(indices[indptr[v]:indptr[v + 1]].tolist())
    return out


class RelGraph:
    """R stacked relations over N nodes (host numpy + lazily made device copy).

    A ROW PARTITION of a larger graph (config C5: CSR rows split by node range over the GPUs) is the same
    object with ``row_lo`` / ``n_global`` set: it holds the rows of nodes [row_lo, row_lo + n_nodes) of a graph
    with ``n_global`` nodes; neighbour ids stay global."""

    def __init__(self, n_nodes: int, indptr_list, indices_list, row_lo: int = 0, n_global: int | None = None):
        self.n_nodes = int(n_nodes)
        self.row_lo = int(row_lo)
        self.n_global = int(n_global) if n_global is not None else self.n_nodes + self.row_lo
        if self.row_lo < 0 or self.row_lo + self.n_nodes > self.n_global:
            raise ValueError("row range outside the global graph")
        self.n_rel = len(indptr_list)
        if self.n_rel == 0:
            raise ValueError("at least one relation is required")
        offs = [0]
        for ip, ix in zip(indptr_list, indices_list):
            ip = np.asarray(ip)
            if ip.shape[0] != self.n_nodes + 1:
                raise ValueError("indptr must have n_nodes + 1 entries")
            if int(ip[-1]) != len(ix):
                raise ValueError("indptr[-1] must equal len(indices)")
            offs.append(offs[-1] + len(ix))
        self.rel_offsets = np.asarray(offs, dtype=np.int64)
        indptr = np.empty(self.n_rel * self.n_nodes + 1, dtype=np.int64)
        for r, ip in enumerate(indptr_list):
            indptr[r * self.n_nodes:(r + 1) * self.n_nodes] = np.asarray(ip[:-1], dtype=np.int64) + offs[r]
        indptr[-1] = offs[-1]
        self.indptr = indptr
        self.indices = (np.concatenate([np.asarray(ix, dtype=np.int32) for ix in indices_list])
                        if offs[-1] else np.zeros(0, dtype=np.int32))
        self._dev = {}

    # ---- constructors -------------------------------------------------
    @classmethod
    def from_adj_lists(cls, adj_lists, n_nodes: int | None = None):
        """From the reference's ``list[dict[int -> set[int]]]`` (keys and members
        may be numpy integer scalars, utils.py:236-239). Rows are sorted by id."""
        if isinstance(adj_lists, dict):
            adj_lists = [adj_lists]
        if n_nodes is None:
            n_nodes = 0
            for adj in adj_lists:
                for k, vs in adj.items():
                    n_nodes = max(n_nodes, int(k) + 1)
                    if len(vs):
                        n_nodes = max(n_nodes, int(max(vs)) + 1)
        ips, ixs = [], []
        for adj in adj_lists:
            deg = np.zeros(n_nodes, dtype=np.int64)
            for k, vs in adj.items():
                deg[int(k)] = len(vs)
            ip = np.zeros(n_nodes + 1, dtype=np.int64)
            np.cumsum(deg, out=ip[1:])
            ix = np.empty(int(ip[-1]), dtype=np.int32)
            for k, vs in adj.items():
                k = int(k)
                if deg[k]:
                    row = np.fromiter((int(x) for x in vs), dtype=np.int32, count=int(deg[k]))
                    row.sort()
                    ix[ip[k]:ip[k + 1]] = row
            ips.append(ip)
            ixs.append(ix)
        return cls(n_nodes, ips, ixs)

    @classmethod
    def from_scipy(cls, mats):
        """From scipy sparse adjacency matrices, applying the same self-loop +
        symmetrisation rule as ``sparse_to_adjlist_for_train`` (utils.py:244-254)."""
        if not isinstance(mats, (list, tuple)):
            mats = [mats]
        n = mats[0].shape[0]
        ips, ixs = [], []
        for m in mats:
            coo = m.tocoo()
            ip, ix = csr_from_edges(n, coo.row, coo.col)
            ips.append(ip)
            ixs.append(ix)
        return cls(n, ips, ixs)

    # ---- views ---------------------------------------------------------
    def relation(self, r: int):
        """(indptr [N+1] rebased to 0, indices) of relation r."""
        n = self.n_nodes
        lo = self.rel_offsets[r]
        ip = self.indptr[r * n:(r + 1) * n + 1] - lo
        return ip, self.indices[lo:self.rel_offsets[r + 1]]

    def row(self, r: int, v: int):
        """Neighbour ids of GLOBAL node v under relation r (v must lie in this partition)."""
        lv = v - self.row_lo
        b = self.indptr[r * self.n_nodes + lv]
        e = self.indptr[r * self.n_nodes + lv + 1]
        return self.indices[b:e]

    @property
    def partitioned(self) -> bool:
        return self.row_lo != 0 or self.n_global != self.n_nodes

    def row_partition(self, lo: int, hi: int):
        """The rows [lo, hi) of this (unpartitioned) graph as a partition object (copies)."""
        if self.partitioned:
            raise ValueError("already a partition")
        ips, ixs = [], []
        for r in range(self.n_rel):
            ip, ix = self.relation(r)
            ips.append(ip[lo:hi + 1] - ip[lo])
            ixs.append(ix[ip[lo]:ip[hi]])
        return RelGraph(hi - lo, ips, ixs, row_lo=lo, n_global=self.n_nodes)

    @classmethod
    def from_device_csr(cls, n_rows: int, n_rel: int, indptr, indices, row_lo: int = 0, n_global: int | None = None):
        """Wrap a stacked CSR that already lives on a device (torch tensors: indptr int64 [R*n_rows + 1],
        indices int32 [nnz]) without a host copy of the indices (C5: ~10^9 entries generated on the GPU)."""
        g = cls.__new__(cls)
        g.n_nodes, g.n_rel = int(n_rows), int(n_rel)
        g.row_lo = int(row_lo)
        g.n_global = int(n_global) if n_global is not None else g.n_nodes + g.row_lo
        g.indptr = indptr.cpu().numpy()
        g.indices = None                      # device only
        g.rel_offsets = g.indptr[::g.n_nodes][:g.n_rel + 1].copy() if g.n_nodes else np.zeros(n_rel + 1, np.int64)
        g._dev = {_device_key(indices.device): (indptr, indices)}
        return g

    def degrees(self, r: int):
        n = self.n_nodes
        return np.diff(self.indptr[r * n:(r + 1) * n + 1])

    # ---- slot demand: per-node tables behind the host's slot capacities ----
    def choose_slot_demand(self, thresholds, rho, P, train):
        """Read-only int64 [n_nodes]: the slots the choose kernel can give a target, summed over relations, with
        ``c = ceil(d * thresholds[r])`` (``item_slots``). A batch's capacity is the sum over its targets."""
        thr = tuple(float(t) for t in thresholds)
        return self._slot_demand((thr, float(rho), int(P), bool(train)),
                                 lambda r, d: item_slots(d, np.ceil(d * thr[r]).astype(np.int64), rho, P, train))

    def select_all_slot_demand(self):
        """Read-only int64 [n_nodes]: the slots the select-all kernel can give a target, summed over relations: each row
        in whole slots, and one slot for an empty row (it may still take the target itself)."""
        return self._slot_demand(None, lambda r, d: np.maximum((d + SLOT - 1) // SLOT, 1))

    def _slot_demand(self, key, per_relation):
        memo = self.__dict__.setdefault("_slot_demand_memo", {})     # lazily: from_device_csr skips __init__
        if key not in memo:
            memo[key] = sum(per_relation(r, self.degrees(r)) for r in range(self.n_rel))
            memo[key].flags.writeable = False
        return memo[key]

    def union(self):
        """Single-relation graph whose rows are the union over relations — the
        ``homo`` graph the reference hands to pick_step / GCN / SAGE
        (model_handler.py:63-64,130)."""
        n = self.n_nodes
        rows = np.repeat(np.tile(np.arange(n, dtype=np.int64), self.n_rel),
                         np.diff(self.indptr))
        ip, ix = csr_from_edges(n, rows, self.indices, symmetric=False, self_loops=False)
        return RelGraph(n, [ip], [ix])

    def to_adj_lists(self, rows=None):
        return [adj_lists_from_csr(*self.relation(r), rows=rows) for r in range(self.n_rel)]

    @property
    def nnz(self):
        return int(self.indices.shape[0])

    def device(self, device):
        """(indptr, indices) torch tensors on ``device`` (cached)."""
        import torch

        key = _device_key(device)
        if key not in self._dev:
            if self.indices is None:
                raise ValueError(f"this graph lives on {list(self._dev)} only")
            self._dev[key] = (torch.from_numpy(self.indptr).to(device),
                              torch.from_numpy(self.indices).to(device))
        return self._dev[key]


def _device_key(device) -> str:
    import torch

    d = torch.device(device)
    if d.type == "cuda" and d.index is None:
        d = torch.device("cuda", torch.cuda.current_device())
    return str(d)
