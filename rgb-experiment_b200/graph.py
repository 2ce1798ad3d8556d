"""Device-resident graph objects built by the integer CUDA kernels, and their cache.

PyG keeps graphs in COO and re-runs ``gcn_norm`` (self-loop concat + degree scatter + two
gathers) on every forward of every layer, three times per epoch (SURVEY.md 3.1).  Here the edge
list is edited and sorted ONCE into a CSR over targets (forward aggregation) and, lazily, a CSR
over sources (backward), cached on the identity of the ``edge_index`` tensor that reaches the
layers (stable across epochs, SURVEY.md Appendix B10).
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import weakref
from collections import OrderedDict
from typing import Optional

import torch

from . import _lib
from ._lib import GraphStruct, check, lib, ptr, stream_of

LOOP_NONE, LOOP_ADD, LOOP_ADD_REMAINING, LOOP_REMOVE_THEN_ADD = 0, 1, 2, 3
NORM_INV_SQRT, NORM_INV_MEAN, NORM_COUNT = 0, 1, 2

DEFAULT_CHUNK = 1024        # rows with more edges than this are split ...
DEFAULT_LONG_CHUNK = 4096   # ... into CTA work items of this many edges
# Small graphs (fewer rows than one wave of row groups keeps busy): a hop is a few microseconds of work and its
# latency is the LONGEST row's chain of dependent gathers (~0.4 us per 8-edge step: the Cora-shaped hub of 251 edges
# alone takes 25 of the hop's 31 us), not launch overhead -- so rows are split much earlier.  Measured, Cora-shaped
# APPNP K=10 F=7: 307 us with chunk 1024, 184 us with 64/512, 162 us with 32/256 (profiles/r02_small_graph_latency.txt).
SMALL_GRAPH_ROWS = 148 * 4 * 32
SMALL_CHUNK, SMALL_LONG_CHUNK = 32, 256


def default_chunks(n_rows: int):
    return (SMALL_CHUNK, SMALL_LONG_CHUNK) if n_rows < SMALL_GRAPH_ROWS else (DEFAULT_CHUNK, DEFAULT_LONG_CHUNK)
HOT_L2_BYTES = 64 << 20     # L2 budget for the hot (most gathered) feature rows; 0 turns the tagging off
DEFAULT_WINDOW = -1         # row schedule: -1 = global degree sort (fastest on B200, profiles/r01_sweep_v2.txt),
                            # w > 0 = degree-sorted inside windows of w rows, 0 = natural order
# Locality groups (csrc/cluster.cu): on graphs whose feature matrix will not fit L2 the rows are scheduled community
# by community -- (group rank, -degree) -- so that the rows in flight gather from one L2-resident slice.
CLUSTER = os.environ.get("RGBMP_CLUSTER", "auto")      # auto | 0 | 1
CLUSTER_MIN_NODES = 200_000     # auto: below this every realistic feature matrix is L2-resident anyway
CLUSTER_MIN_DEGREE = 4.0        # auto: mean degree below which a community's slice is not re-used enough to matter
CLUSTER_SEEDS = 512             # 256 / 1024 / 4096 seeds gave the same hop time (2.86 / 2.84 / 2.85 ms); fewer seeds chain faster on the host
CLUSTER_TAUS = (0.3, 0.15, 0.05, 0.0, 0.0)   # the fifth round labels the last few hundred nodes; a sixth changed none
CLUSTER_CONN_STRIDE = 4         # the connectivity matrix only orders the groups: every 4th row is sample enough
CLUSTER_MIN_INTRA = 0.25        # share of edges inside a group below which the graph has no community structure to use
                                # (a uniform random graph still reaches ~0.15: every node shares a group with the neighbour it copied)
cluster_stats = {"built": 0, "used": 0, "last": None}


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


class CSR:
    """One orientation of the graph: rowptr int64 [n_rows+1], col int32 [nnz], eid int32 [nnz]
    (position in the edited edge list), plus the long-row work lists and the ctypes descriptor."""

    def __init__(self, key: torch.Tensor, other: torch.Tensor, n_rows: int, n_cols: int,
                 chunk: Optional[int] = None, long_chunk: Optional[int] = None, window: Optional[int] = None,
                 groups=None, finish: bool = True, named: bool = False):
        L = lib()
        dev = key.device
        st = stream_of(dev)
        nnz = key.numel()
        self.n_rows, self.n_cols, self.nnz, self.device = n_rows, n_cols, nnz, dev
        self.rowptr = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
        self.col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        self.eid = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        wsb = L.rgbmp_csr_build_workspace_bytes(nnz, n_rows)
        ws = _ws(wsb, dev)
        check(L.rgbmp_csr_build(ptr(key), ptr(other), nnz, n_rows, ptr(self.rowptr), ptr(self.col), ptr(self.eid),
                                ptr(ws), ws.numel(), dev.index, st), "csr_build")
        self.col, self.eid = self.col[:nnz], self.eid[:nnz]
        if finish:
            self._finish(chunk, long_chunk, window, groups, named=named)

    @classmethod
    def from_arrays(cls, rowptr: torch.Tensor, col: torch.Tensor, n_cols: int, chunk: Optional[int] = None,
                    long_chunk: Optional[int] = None, window: Optional[int] = None) -> "CSR":
        """Wrap a CSR that exists already (row-generated graphs, synth.rowgen_block): rowptr int64
        [n_rows+1], col int32 [nnz] on the device.  No edge ids (eid is None)."""
        _lib.require_cuda(rowptr, "rowptr")
        if rowptr.dtype != torch.int64 or col.dtype != torch.int32:
            raise RuntimeError("CSR.from_arrays needs int64 rowptr and int32 col")
        self = cls.__new__(cls)
        self.n_rows, self.n_cols, self.nnz, self.device = rowptr.numel() - 1, int(n_cols), col.numel(), rowptr.device
        if self.nnz >= (1 << 31):
            raise RuntimeError("nnz >= 2^31 in one partition: use more row blocks")
        self.rowptr, self.col, self.eid = rowptr.contiguous(), col.contiguous(), None
        self._finish(chunk, long_chunk, window)
        return self

    def degree_order(self) -> torch.Tensor:
        """int32 [n_rows]: rows by degree, longest first (stable) -- the default schedule and the seed ranking."""
        L = lib()
        order = torch.empty(self.n_rows, dtype=torch.int32, device=self.device)
        ws = _ws(L.rgbmp_row_order_workspace_bytes(self.n_rows), self.device)
        check(L.rgbmp_row_order(ptr(self.rowptr), self.n_rows, self.n_rows, ptr(order), ptr(ws), ws.numel(),
                                self.device.index, stream_of(self.device)), "row_order")
        return order

    def _finish(self, chunk: int, long_chunk: int, window: Optional[int], groups=None, deg_order=None,
                named: bool = False):
        """Row schedule, long-row work lists, descriptor.  groups = (group int32 [n_rows], n_groups): schedule by
        (group, -degree) and list the long rows in that order too (locality groups, see Graph).  named: the rows are
        already numbered in that schedule (Graph.named_fwd) -- identity schedule, long rows in id order, and like
        any locality-grouped schedule no hot tags."""
        L = lib()
        dev, n_rows, nnz = self.device, self.n_rows, self.nnz
        st = stream_of(dev)
        dc, dl = default_chunks(n_rows)
        self.chunk, self.long_chunk = int(dc if chunk is None else chunk), int(dl if long_chunk is None else long_chunk)
        self.n_long = self.n_items = 0
        self.long_rows = self.long_item_ptr = self.item_long = self.item_start = None
        self.row_order = None
        self.clustered = groups is not None or named
        window = DEFAULT_WINDOW if window is None else int(window)
        if window < 0:
            window = n_rows
        if n_rows > 1 and nnz > 0 and not named:
            if groups is not None:
                grp, n_groups = groups
                self.row_order = torch.empty(n_rows, dtype=torch.int32, device=dev)
                ws = _ws(L.rgbmp_row_order_workspace_bytes(n_rows), dev)
                check(L.rgbmp_row_order_grouped(ptr(self.rowptr), n_rows, n_rows, ptr(grp), int(n_groups), ptr(self.row_order),
                                                ptr(ws), ws.numel(), dev.index, st), "row_order_grouped")
            elif window >= n_rows and deg_order is not None:
                self.row_order = deg_order
            elif window > 0:
                self.row_order = torch.empty(n_rows, dtype=torch.int32, device=dev)
                ws = _ws(L.rgbmp_row_order_workspace_bytes(n_rows), dev)
                check(L.rgbmp_row_order(ptr(self.rowptr), n_rows, window, ptr(self.row_order), ptr(ws), ws.numel(),
                                        dev.index, st), "row_order")
        self._split_long_rows(self.row_order if self.clustered else None)
        self._norm = {}
        self._tagged = {}
        self.struct = self._make_struct(self.col, 0)
        self.ref = C.byref(self.struct)

    def _make_struct(self, col: torch.Tensor, tagged: int) -> GraphStruct:
        return GraphStruct(self.n_rows, self.n_cols, self.nnz, ptr(self.rowptr), ptr(col), self.chunk, self.long_chunk,
                           self.n_long, self.n_items, ptr(self.long_rows), ptr(self.long_item_ptr),
                           ptr(self.item_long), ptr(self.item_start), ptr(self.row_order), tagged)

    def col_freq(self) -> torch.Tensor:
        """int32 [n_cols]: how often each column (feature row) is gathered by one pass over this CSR."""
        v = self._norm.get("freq")
        if v is None:
            v = torch.empty(max(self.n_cols, 1), dtype=torch.int32, device=self.device)
            check(lib().rgbmp_col_freq(ptr(self.col), self.nnz, self.n_cols, ptr(v), self.device.index,
                                       stream_of(self.device)), "col_freq")
            self._norm["freq"] = v
        return v

    def hot_ref(self, row_bytes: int):
        """Descriptor whose column ids carry the hot tag (bit 31) for feature rows of `row_bytes`
        bytes, or the plain descriptor when the whole feature matrix fits the L2 budget anyway.
        The hot set = the most frequently gathered rows that fit HOT_L2_BYTES; built once per
        row size class and cached."""
        if HOT_L2_BYTES <= 0 or self.nnz == 0 or self.n_cols * row_bytes <= HOT_L2_BYTES or self.clustered:
            return self.ref        # a locality-grouped schedule keeps its own working set in L2: pinning the global hubs costs it room
        k_hot = max(1, HOT_L2_BYTES // max(row_bytes, 1))
        hit = self._tagged.get(k_hot)
        if hit is None:
            freq = self.col_freq()[: self.n_cols]
            # threshold = frequency of the k_hot-th most popular column (ties above the budget stay cold)
            thresh = int(torch.kthvalue(freq, self.n_cols - k_hot + 1).values.item()) + 1
            tagged = torch.empty(self.nnz, dtype=torch.int32, device=self.device)
            check(lib().rgbmp_col_tag(ptr(self.col), self.nnz, ptr(freq), thresh, ptr(tagged), self.device.index,
                                      stream_of(self.device)), "col_tag")
            st = self._make_struct(tagged, 1)
            hit = (tagged, st, C.byref(st))
            self._tagged[k_hot] = hit
        return hit[2]

    def _split_long_rows(self, order=None):
        L = lib()
        dev, st = self.device, stream_of(self.device)
        if self.n_rows == 0 or self.nnz == 0:
            return
        counts = torch.empty(2, dtype=torch.int64, device=dev)
        check(L.rgbmp_longrow_count(ptr(self.rowptr), self.n_rows, self.chunk, self.long_chunk, ptr(counts),
                                    dev.index, st), "longrow_count")
        n_long, n_items = (int(v) for v in counts.tolist())       # one sync at build time
        if n_long == 0:
            return
        self.n_long, self.n_items = n_long, n_items
        self.long_rows = torch.empty(n_long, dtype=torch.int32, device=dev)
        self.long_item_ptr = torch.empty(n_long + 1, dtype=torch.int32, device=dev)
        self.item_long = torch.empty(n_items, dtype=torch.int32, device=dev)
        self.item_start = torch.empty(n_items, dtype=torch.int64, device=dev)
        ws = _ws(L.rgbmp_longrow_fill_workspace_bytes(self.n_rows), dev)
        check(L.rgbmp_longrow_fill_ordered(ptr(self.rowptr), self.n_rows, self.chunk, self.long_chunk, ptr(order), n_long,
                                           n_items, ptr(self.long_rows), ptr(self.long_item_ptr), ptr(self.item_long),
                                           ptr(self.item_start), ptr(ws), ws.numel(), dev.index, st), "longrow_fill")

    def norm(self, mode: int) -> torch.Tensor:
        """Per-row vector from the degree: deg^-1/2 | 1/max(deg,1) | max(deg,1)."""
        v = self._norm.get(mode)
        if v is None:
            v = torch.empty(self.n_rows, dtype=torch.float32, device=self.device)
            check(lib().rgbmp_degree_norm(ptr(self.rowptr), self.n_rows, mode, ptr(v), self.device.index,
                                          stream_of(self.device)), "degree_norm")
            self._norm[mode] = v
        return v

    def degree(self) -> torch.Tensor:
        return self.rowptr[1:] - self.rowptr[:-1]

    def spmm_workspace(self, F: int) -> Optional[torch.Tensor]:
        if self.n_items == 0:
            return None
        return _ws(self.n_items * ((F + 3) // 4 * 4) * 4 + 256, self.device)


def chain_groups(W) -> "tuple":
    """Linear order of the groups in which strongly connected ones are adjacent: greedy chain on the connectivity
    normalised by the groups' volumes, W[a,b] / (vol_a * vol_b), with an exponentially decayed affinity to the
    recently placed groups.  Host-side (numpy) over an S x S matrix, S <= 4096.  Returns (rank int64 [S], share of
    the edges that stay inside a group)."""
    import numpy as np
    W = np.asarray(W, dtype=np.float64)
    S = W.shape[0]
    W = W + W.T                                     # symmetrise: in- and out-edges pull alike
    tot = W.sum()
    intra = float(np.trace(W) / tot) if tot > 0 else 0.0
    vol = W.sum(1) + 1e-9
    Wn = W / vol[:, None] / vol[None, :]
    np.fill_diagonal(Wn, 0.0)
    rank = np.zeros(S, dtype=np.int64)
    aff = np.zeros(S)
    cur = int(np.argmax(vol))
    for pos in range(S):                            # in-place vector ops only: ~5 us per step
        rank[cur] = pos
        aff *= 0.5
        aff += Wn[cur]
        aff[cur] = -np.inf                          # placed groups can never win again (-inf survives decay and adds)
        cur = int(aff.argmax())
    return rank, intra


def locality_groups(csr: "CSR", deg_order: torch.Tensor):
    """(group int32 [N], n_groups) for the row schedule, or None when clustering is off / not worth it / finds no
    community structure.  Seeded leaves-first label propagation on the device (rgbmp_cluster_lpa), group-to-group
    connectivity on the device, chaining of the S groups on the host.  One small D2H (S*S*4 bytes) per graph."""
    mode = CLUSTER
    N, nnz = csr.n_rows, csr.nnz
    if mode == "0" or csr.n_rows != csr.n_cols:
        return None
    if mode != "1" and (N < CLUSTER_MIN_NODES or nnz < CLUSTER_MIN_DEGREE * N):
        return None
    L = lib()
    dev = csr.device
    st = stream_of(dev)
    S = int(min(CLUSTER_SEEDS, N))
    plain = GraphStruct(csr.n_rows, csr.n_cols, csr.nnz, ptr(csr.rowptr), ptr(csr.col), 0, 0, 0, 0, None, None, None, None,
                        None, 0)
    import time
    trace = os.environ.get("RGBMP_CLUSTER_TRACE")
    if trace:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
    label = torch.empty(N, dtype=torch.int32, device=dev)
    ws = _ws(L.rgbmp_cluster_workspace_bytes(N), dev)
    taus = (C.c_float * len(CLUSTER_TAUS))(*CLUSTER_TAUS)
    check(L.rgbmp_cluster_lpa(C.byref(plain), ptr(deg_order), S, len(CLUSTER_TAUS), taus, ptr(label), ptr(ws), ws.numel(),
                              dev.index, st), "cluster_lpa")
    if trace:
        torch.cuda.synchronize()
        t1 = time.perf_counter()
    W = torch.empty((S, S), dtype=torch.int32, device=dev)
    check(L.rgbmp_cluster_connectivity(C.byref(plain), ptr(label), S, int(CLUSTER_CONN_STRIDE), ptr(W), dev.index, st),
          "cluster_connectivity")
    Wh = W.cpu().numpy().astype("int64") & 0xFFFFFFFF
    if trace:
        t2 = time.perf_counter()
    rank, intra = chain_groups(Wh)
    if trace:
        print(f"[rgbmp cluster] lpa {1e3 * (t1 - t0):.2f} ms, connectivity + D2H {1e3 * (t2 - t1):.2f} ms, "
              f"host chain {1e3 * (time.perf_counter() - t2):.2f} ms, intra {intra:.3f}", flush=True)
    cluster_stats["built"] += 1
    cluster_stats["last"] = {"groups": S, "intra_group_edge_share": round(intra, 4)}
    if mode != "1" and intra < CLUSTER_MIN_INTRA:
        return None
    cluster_stats["used"] += 1
    group = torch.from_numpy(rank).to(device=dev, dtype=torch.int32)[label.long()].contiguous()
    return group, S


class Graph:
    """Edited edge list + forward CSR (+ lazy transpose CSR, normalisation vectors, edge weights)."""

    def __init__(self, edge_index: torch.Tensor, num_nodes: int, loop_mode: int = LOOP_NONE,
                 chunk: Optional[int] = None, long_chunk: Optional[int] = None, window: Optional[int] = None):
        _lib.require_cuda(edge_index, "edge_index")
        if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise RuntimeError("edge_index must be an int64 tensor of shape [2, E]")
        L = lib()
        dev = edge_index.device
        st = stream_of(dev)
        ei = edge_index if edge_index.is_contiguous() else edge_index.contiguous()
        E, N = ei.size(1), int(num_nodes)
        self.N, self.E_in, self.loop_mode, self.device = N, E, loop_mode, dev
        self._chunk, self._long_chunk, self._window = chunk, long_chunk, window
        e_src = torch.empty(max(E + N, 1), dtype=torch.int32, device=dev)
        e_dst = torch.empty(max(E + N, 1), dtype=torch.int32, device=dev)
        nnz_dev = torch.empty(1, dtype=torch.int64, device=dev)
        ws = _ws(L.rgbmp_edge_edit_workspace_bytes(E, N), dev)
        check(L.rgbmp_edge_edit(ptr(ei[0]) if E else None, ptr(ei[1]) if E else None, E, N, loop_mode, ptr(e_src),
                                ptr(e_dst), ptr(nnz_dev), ptr(ws), ws.numel(), dev.index, st), "edge_edit")
        nnz = int(nnz_dev.item())                                  # the one sync of the build
        if nnz < 0:
            raise RuntimeError(f"edge_index contains node ids outside [0, {N})")
        self.nnz = nnz
        self.e_src, self.e_dst = e_src[:nnz], e_dst[:nnz]          # edited list: kept edges, then loops
        self.fwd = CSR(self.e_dst, self.e_src, N, N, chunk, long_chunk, window, finish=False)   # rows = targets i, col = sources j
        deg_order = self.fwd.degree_order() if (N > 1 and nnz > 0 and (window is None or window < 0)) else None
        self.groups = locality_groups(self.fwd, deg_order) if deg_order is not None else None
        self.fwd._finish(chunk, long_chunk, window, self.groups, deg_order)
        self._bwd: Optional[CSR] = None
        self._named: Optional[CSR] = None
        self._lock = threading.Lock()
        self._vals = {}
        self._perm_memo = {}

    # transpose CSR: rows = sources j, col = targets i (built on first backward)
    @property
    def bwd(self) -> CSR:
        if self._bwd is None:
            with self._lock:
                if self._bwd is None:
                    self._bwd = CSR(self.e_src, self.e_dst, self.N, self.N, self._chunk, self._long_chunk, self._window,
                                    groups=self.groups)     # the groups are a property of the NODES: same for both orientations
        return self._bwd

    @property
    def named_fwd(self) -> Optional[CSR]:
        """The forward CSR under the node naming pos = inverse(fwd.row_order), or None when the graph has no
        locality-grouped schedule.  Row i of it is node fwd.row_order[i]; its schedule is the identity, so a K-hop call
        on it reads and writes the iterate, the teleport term and the output rows in order and every group's feature
        rows form one contiguous slice.  Built from the same edited edge list by the same stable sort, every row keeps
        its edges in the same order: sums, long-row splits and results are bit-identical to those on fwd.  No edge
        ids (eid is None): only the K-hop paths use it."""
        if self._named is None and self.groups is not None and self.fwd.row_order is not None:
            with self._lock:
                if self._named is None:
                    order = self.fwd.row_order.long()
                    pos = torch.empty(self.N, dtype=torch.int32, device=self.device)
                    pos[order] = torch.arange(self.N, dtype=torch.int32, device=self.device)
                    csr = CSR(pos.index_select(0, self.e_dst), pos.index_select(0, self.e_src), self.N, self.N,
                              self.fwd.chunk, self.fwd.long_chunk, named=True)
                    csr.eid = None
                    self._named = csr
        return self._named

    def dinv(self) -> torch.Tensor:
        """deg_in^-1/2 with inf -> 0 (gcn_norm, dagnn.py:27-30; unit edge weights)."""
        return self.fwd.norm(NORM_INV_SQRT)

    def gcn_val(self, transpose: bool = False) -> torch.Tensor:
        """Per-edge symmetric weights dinv[src]*1*dinv[dst] in the CSR order of the chosen orientation."""
        key = ("gcn", transpose)
        v = self._vals.get(key)
        if v is None:
            csr = self.bwd if transpose else self.fwd
            d = self.dinv()
            v = torch.empty(max(self.nnz, 1), dtype=torch.float32, device=self.device)
            check(lib().rgbmp_gcn_edge_weight(ptr(csr.rowptr), ptr(csr.col), csr.n_rows, ptr(d), ptr(d), ptr(v),
                                              self.device.index, stream_of(self.device)), "gcn_edge_weight")
            v = v[:self.nnz]
            self._vals[key] = v
        return v

    def tpos(self) -> torch.Tensor:
        """int32 [nnz]: forward-CSR position of every transpose-CSR entry."""
        v = self._vals.get("tpos")
        if v is None:
            inv = torch.empty(self.nnz, dtype=torch.int32, device=self.device)
            inv[self.fwd.eid.long()] = torch.arange(self.nnz, dtype=torch.int32, device=self.device)
            v = inv[self.bwd.eid.long()].contiguous()
            self._vals["tpos"] = v
        return v

    def fwd_to_bwd(self, csr_vals: torch.Tensor) -> torch.Tensor:
        """[nnz(,H)] values in forward-CSR order -> transpose-CSR order."""
        return csr_vals[self.tpos().long()].contiguous()

    def undirected_csr(self, symmetrize: bool = True):
        """(rowptr int64 [N+1], col int32 [n_u]): the unique (src, dst) pairs of the edited edge list -- with
        `symmetrize` every reversed pair as well (to_undirected) -- as a CSR over src with each row's columns sorted,
        the set SuperGAT's negative sampler rejects candidates against.  Built once (rgbmp_coalesce, then a lower_bound
        row pointer) and held like the transpose CSR, instead of a 2 nnz coalesce on every training forward."""
        key = ("undirected", bool(symmetrize))
        v = self._vals.get(key)
        if v is None:
            from .shim.utils import _coalesce_cuda
            pairs = _coalesce_cuda(torch.stack([self.e_src, self.e_dst]).to(torch.int64), self.N, bool(symmetrize))
            nodes = torch.arange(self.N + 1, dtype=torch.int64, device=self.device)
            rowptr = torch.searchsorted(pairs[0].contiguous(), nodes)
            v = (rowptr, pairs[1].to(torch.int32))
            self._vals[key] = v
        return v

    def edge_index(self) -> torch.Tensor:
        """The edited edge list as an int64 [2, nnz] tensor (what PyG's loop utilities return)."""
        v = self._vals.get("edge_index")
        if v is None:
            v = torch.stack([self.e_src, self.e_dst]).to(torch.int64)
            self._vals["edge_index"] = v
        return v

    def to_csr_order(self, edge_vals: torch.Tensor, transpose: bool = False) -> torch.Tensor:
        """edge-ordered [nnz] or [nnz,H] float32 -> CSR order of the chosen orientation.  The last permuted
        tensor of each orientation is remembered on the identity (weakref + _version) of its source: DAGNN's Prop
        passes the SAME `norm` to all K hops of a forward (dagnn.py:41-46), so K-1 of K permutations are hits."""
        last = self._perm_memo.get(transpose)
        if last is not None and last[0]() is edge_vals and last[1] == edge_vals._version and \
                not (edge_vals.requires_grad and torch.is_grad_enabled()):
            return last[2]
        csr = self.bwd if transpose else self.fwd
        ev = edge_vals.detach().contiguous().to(torch.float32)
        H = 1 if ev.dim() == 1 else ev.size(1)
        out = torch.empty_like(ev)
        check(lib().rgbmp_edge_permute(ptr(ev), ptr(csr.eid), self.nnz, H, 0, ptr(out), self.device.index,
                                       stream_of(self.device)), "edge_permute")
        try:
            self._perm_memo[transpose] = (weakref.ref(edge_vals), edge_vals._version, out)
        except TypeError:
            pass
        return out

    def to_edge_order(self, csr_vals: torch.Tensor, transpose: bool = False) -> torch.Tensor:
        _lib.require_f32(csr_vals, "to_edge_order")
        csr = self.bwd if transpose else self.fwd
        cv = csr_vals.contiguous()
        H = 1 if cv.dim() == 1 else cv.size(1)
        out = torch.empty_like(cv)
        check(lib().rgbmp_edge_permute(ptr(cv), ptr(csr.eid), self.nnz, H, 1, ptr(out), self.device.index,
                                       stream_of(self.device)), "edge_permute")
        return out


# --------------------------------------------------------------------------------------------
# cache keyed on the identity of the edge_index tensor that reaches the layers
#
# An entry lives exactly as long as the edge_index TENSOR it was built from: a weakref callback drops
# it when that tensor dies (so the allocator can never hand its address to a different edge list that
# would alias the key), nothing here keeps the caller's tensor alive, and the total is capped in BYTES
# (RGBMP_GRAPH_CACHE_MB, default 32768: a products-sized Graph with both orientations, weights and hot
# tags is ~5 GB).  On a CUDA out-of-memory error the caches are emptied and the call is retried once
# (`oom_retry`) -- the reference's sweeps treat any RuntimeError as "model too big"
# (examples/all_dataset_baseline.py:65-66), so memory pinned by earlier datasets must not cause one.
# --------------------------------------------------------------------------------------------
_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()      # key -> (Graph, weakref to the keyed tensor, nbytes)
_CACHE_LOCK = threading.RLock()
_CACHE_MAX = 16
_CACHE_MAX_BYTES = int(float(os.environ.get("RGBMP_GRAPH_CACHE_MB", "32768")) * (1 << 20))
stats = {"hits": 0, "builds": 0, "evicted": 0, "oom_retries": 0}


def _graph_key(edge_index: torch.Tensor, num_nodes: int, loop_mode: int, reverse: bool) -> tuple:
    return (edge_index.data_ptr(), edge_index._version, tuple(edge_index.shape), tuple(edge_index.stride()),
            int(num_nodes), int(loop_mode), str(edge_index.device), bool(reverse))


def _drop(key) -> None:
    with _CACHE_LOCK:
        _CACHE.pop(key, None)


def cache_bytes() -> int:
    with _CACHE_LOCK:
        return sum(v[2] for v in _CACHE.values())


def _build_nbytes(g: "Graph") -> int:
    """Bytes a freshly built Graph holds, plus what its lazily built parts will add (transpose CSR, weights in
    both orientations, one hot-tagged column copy each, the renamed forward CSR of a locality-grouped graph): the cap
    is about what an entry may grow to."""
    nnz, n = g.nnz, g.N
    named = 8 * (n + 1) + 4 * nnz + 4 * n if g.groups is not None else 0
    return 2 * 4 * nnz + 2 * (8 * (n + 1) + 8 * nnz + 4 * n) + 2 * 4 * nnz + 2 * 4 * nnz + named


def oom_retry(fn):
    """Run fn(); on a CUDA OOM drop every cached graph and memoised result, return the blocks to the driver
    and try once more."""
    try:
        return fn()
    except torch.cuda.OutOfMemoryError:
        stats["oom_retries"] += 1
        clear_cache()
        from . import memo
        memo.clear()
        from .shim import utils as _u
        _u.clear_memo()
        torch.cuda.empty_cache()
        return fn()


def get_graph(edge_index: torch.Tensor, num_nodes: int, loop_mode: int, reverse: bool = False) -> Graph:
    """Cached Graph of `edge_index` (reverse=True: of edge_index.flip(0), keyed on the ORIGINAL tensor so that
    callers which need the reversed orientation -- PTA, SURVEY B7 -- do not mint a new cache key per call)."""
    key = _graph_key(edge_index, num_nodes, loop_mode, reverse)
    with _CACHE_LOCK:
        hit = _CACHE.get(key)
        if hit is not None and hit[1]() is edge_index:
            _CACHE.move_to_end(key)
            stats["hits"] += 1
            return hit[0]
    src = edge_index.flip(0).contiguous() if reverse else edge_index
    g = oom_retry(lambda: Graph(src, num_nodes, loop_mode))
    del src
    nbytes = _build_nbytes(g)
    with _CACHE_LOCK:
        _CACHE[key] = (g, weakref.ref(edge_index, lambda _r, k=key: _drop(k)), nbytes)
        _CACHE.move_to_end(key)
        stats["builds"] += 1
        while len(_CACHE) > 1 and (len(_CACHE) > _CACHE_MAX or sum(v[2] for v in _CACHE.values()) > _CACHE_MAX_BYTES):
            _CACHE.popitem(last=False)
            stats["evicted"] += 1
    return g


def clear_cache():
    with _CACHE_LOCK:
        _CACHE.clear()
