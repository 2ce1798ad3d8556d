"""1-D node-row partition of the propagation across the GPUs of one NVSwitch box (SURVEY.md 8e).

Rank p owns the output rows [p*R, (p+1)*R) with R = ceil(N / P), the CSR rows of that block (global
column ids) and the matching rows of every feature matrix.  One exchange step per hop: an
all-gather of the iterate's rows (NCCL over NVLink 5 through ``torch.distributed``), after which
each rank runs the SAME fused SpMM kernel on its row block.  The host logic (row ranges, edge
bucketing, the exchange) is plain torch and runs under gloo on CPU for the world_size-2 tests;
only ``build_local_csr`` / ``PartitionedAPPNP`` touch the CUDA library.
"""
from __future__ import annotations

import os
from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist


def rows_per_rank(N: int, world: int) -> int:
    return (N + world - 1) // world


def row_range(N: int, rank: int, world: int) -> Tuple[int, int]:
    R = rows_per_rank(N, world)
    lo = min(N, rank * R)
    return lo, min(N, lo + R)


class Grid:
    """Process grid of a K-hop propagation: `Pr` row groups x `Pf` feature groups (world = Pr * Pf).

    K-hop propagation acts on every feature column independently, so the feature axis can be
    split with NO communication; only ranks that share a feature slice (a "row group" of Pr ranks)
    exchange iterate rows.  Against the pure row partition (Pf = 1) a grid divides the per-hop
    NVLink volume of every GPU by Pf -- (Pr-1)/Pr * N * F/Pf elements instead of (P-1)/P * N * F --
    at the same gather bytes per GPU (P/Pf times fewer rows... of F/Pf-wide features over Pf times more edges).
    rank = rp * Pf + fp."""

    def __init__(self, rank: int, world: int, feature_groups: int = 1):
        if world % feature_groups != 0:
            raise RuntimeError(f"feature_groups={feature_groups} does not divide world={world}")
        self.rank, self.world, self.Pf, self.Pr = rank, world, feature_groups, world // feature_groups
        self.rp, self.fp = rank // feature_groups, rank % feature_groups
        self.row_group = None          # torch.distributed group of the ranks sharing my feature slice
        self.col_group = None          # ... of the ranks sharing my row block (they hold the other slices)
        if world > 1 and feature_groups > 1:
            for f in range(feature_groups):   # every rank creates every group, in the same order
                g = dist.new_group([r * feature_groups + f for r in range(self.Pr)])
                if f == self.fp:
                    self.row_group = g
            for r in range(self.Pr):
                g = dist.new_group([r * feature_groups + f for f in range(feature_groups)])
                if r == self.rp:
                    self.col_group = g

    def warm_up(self, device) -> None:
        """One tiny collective on every group this rank belongs to: NCCL builds a sub-communicator lazily, at the
        first collective (seconds on an 8-GPU box) -- pay it here, not inside a timed graph build or step."""
        t = torch.zeros(1, device=device)
        for g in (None, self.row_group, self.col_group):
            if g is not None or self.world > 1:
                dist.all_reduce(t, group=g)
                # NCCL also connects lazily per ALGORITHM: the build's first all-gather (ring) after an all-reduce
                # (tree / NVLS) paid another 2-4 s on 4 and 8 GPUs (round-2 bench lines) -- run one of each kind
                n = dist.get_world_size(group=g)
                full = torch.zeros(n, device=device)
                dist.all_gather_into_tensor(full, t, group=g)
                objs = [None] * n
                dist.all_gather_object(objs, 0, group=g)
        torch.cuda.synchronize(device)
        if self.world > 1:
            dist.barrier()

    def feature_slice(self, F: int, align: int = 4, fp: Optional[int] = None):
        """[lo, hi) of the feature columns of feature group `fp` (default: mine).  Slices start on
        `align`-element boundaries (16-byte vectors) and the vector units are spread evenly."""
        fp = self.fp if fp is None else fp
        units = (F + align - 1) // align
        base, rem = divmod(units, self.Pf)
        if base == 0:
            raise RuntimeError(f"feature_groups={self.Pf} exceeds the {units} {align}-element vectors of F={F}")
        lo_u = fp * base + min(fp, rem)
        hi_u = lo_u + base + (1 if fp < rem else 0)
        return min(F, lo_u * align), min(F, hi_u * align)


def auto_feature_groups(world: int, F: int) -> int:
    """Feature groups of the default grid.  The per-hop NVLink volume of a GPU shrinks with Pf while
    rows get narrower (F/Pf).  Measured (profiles/r01_multigpu.txt): products-shaped APPNP F=47 --
    4 GPUs 4x1 87.1 / 2x2 89.8 GTEPS, 8 GPUs 8x1 102 / 4x2 147 / 2x4 113; papers100M-shaped bf16
    F=128 -- 4 GPUs 4x1 71 / 2x2 59 ms per hop."""
    if world >= 4 and world % 2 == 0 and F >= 32:
        return 2
    return 1


def community_naming(group: torch.Tensor, N: int):
    """Rename the nodes so that equal-sized row blocks are runs of whole locality groups: new id = position in
    (group rank, old id) order.  Returns (perm, inv) int64 [N]: perm[new] = old, inv[old] = new.  Plain torch: the same
    answer on every rank from the same `group`, on any device."""
    ids = torch.arange(N, dtype=torch.int64, device=group.device)
    perm = torch.argsort(group.to(torch.int64) * N + ids)             # keys are unique: no tie order to worry about
    inv = torch.empty_like(perm)
    inv[perm] = ids
    return perm, inv


def block_keeps_groups(R: int, row_bytes: Optional[int]) -> bool:
    """Schedule of a row block (tools/emulate_rank.py, profiles/r02_emulated_rank.txt): blocks whose result is ~90 MB and more
    keep the locality-grouped schedule, with long rows split at 256 edges (a (group, -degree) order leaves long rows in the
    last wave: 2x1 block 1.52 ms with chunk 1024, 1.42 with 256; 4x1 0.77 vs 0.84 without groups); smaller blocks run the
    plain degree schedule faster (4x2: 0.425 vs 0.453 ms, 8x1: 0.374 vs 0.399, 8x2: 0.215 vs 0.234).  row_bytes unknown:
    a million rows decide."""
    return (R * row_bytes >= 90e6) if row_bytes else (R >= 1_000_000)


def local_edges(e_src: torch.Tensor, e_dst: torch.Tensor, lo: int, hi: int):
    """Edges whose TARGET falls in [lo, hi), order preserved: (local target id, global source id).
    Because the filter keeps the relative order, the stable CSR of the bucket equals the matching
    row block of the global stable CSR."""
    m = (e_dst >= lo) & (e_dst < hi)
    return (e_dst[m] - lo).to(torch.int32), e_src[m].to(torch.int32)


def all_gather_rows(local: torch.Tensor, full: torch.Tensor, group=None):
    """full[p*R:(p+1)*R] = rank p's `local` ([R, ld], same shape on every rank)."""
    dist.all_gather_into_tensor(full, local, group=group)
    return full


def check_post_step(R: int, clamp=None, reset=None) -> None:
    """Shapes of label propagation's post-step on a row block of R rows: clamp = (lo, hi); reset = (mask [R],
    values [R, >= F]) -- rows of THIS block, in its naming."""
    if clamp is not None and len(clamp) != 2:
        raise RuntimeError("clamp takes (lo, hi)")
    if reset is not None:
        mask, vals = reset
        if mask.dim() != 1 or mask.size(0) != R or vals.dim() != 2 or vals.size(0) != R:
            raise RuntimeError(f"reset takes (mask [{R}], values [{R}, F]) rows of this block; got "
                               f"{tuple(mask.shape)} / {tuple(vals.shape)}")


class PartitionedPropagator:
    """Device-agnostic K-hop driver: z <- post(a * A_hat z + b * z0) on a row partition.

    spmm(x_full [P*R, ld], z0_local, a, b[, clamp=, reset=]) -> next local iterate [R, ld] is injected: the CUDA
    kernel in production, the CPU oracle in the gloo tests.  The label-propagation post-step (clamp, then the reset
    rows) belongs to the same hop, so it goes to `spmm` with it; `spmm` is called without those keywords when the run
    has no post-step (APPNP / SGC)."""

    def __init__(self, N: int, rank: int, world: int, spmm: Callable, group=None):
        self.N, self.rank, self.world, self.group = N, rank, world, group
        self.R = rows_per_rank(N, world)
        self.lo, self.hi = row_range(N, rank, world)
        self.spmm = spmm

    def run(self, z0_local: torch.Tensor, K: int, a: float, b: float,
            full: Optional[torch.Tensor] = None, clamp=None, reset=None) -> torch.Tensor:
        R, ld = z0_local.shape
        assert R == self.R, "every rank passes ceil(N/P) rows (pad the last block)"
        check_post_step(R, clamp, reset)
        post = {k: v for k, v in (("clamp", clamp), ("reset", reset)) if v is not None}
        if full is None:
            full = torch.empty((R * self.world, ld), dtype=z0_local.dtype, device=z0_local.device)
        cur = z0_local
        for _ in range(K):
            if self.world > 1:
                all_gather_rows(cur, full, self.group)
                src = full
            else:
                src = cur
            cur = self.spmm(src, z0_local, a, b, **post)
        return cur


# ------------------------------------------------------------------------------------------------
# CUDA side
# ------------------------------------------------------------------------------------------------
class LocalBlock:
    """This rank's CSR row block + normalisation, built by the integer kernels."""

    def __init__(self, edge_index: torch.Tensor, N: int, loop_mode: int, rank: int, world: int, group=None,
                 transpose_of: Optional["LocalBlock"] = None, relabel: bool = False, row_bytes: Optional[int] = None):
        """transpose_of: build the block of the TRANSPOSED graph (rows = sources in my range, columns =
        targets) for the backward pass; it reuses the forward block's D^-1/2 (the backward of
        D^-1/2 A D^-1/2 is D^-1/2 A^T D^-1/2 with the same degree vector, also on directed graphs).

        relabel: rename the nodes so that a row block is a run of whole locality groups (communities) instead of a
        run of ids: new id = position in (group rank, old id) order.  A rank then gathers mostly from its own
        communities' slice of the iterate (tools/emulate_rank.py --by-community: the row block's hop 7-15 % faster on the
        products-shaped graph).  The propagation is the same operator on the renamed graph: row i of every [N, F] operand
        and result is node `perm[i]` of the caller's numbering (`perm` new -> old, `inv` old -> new; None when the
        graph has no community structure to use).  A transposed block takes its forward block's naming.
        row_bytes: bytes of one row of the feature slice this block will propagate (F_local * element size), if known:
        decides between the locality-grouped and the plain degree schedule of the block (below)."""
        from . import _lib
        from ._lib import check, lib, ptr, stream_of
        from .graph import CSR, NORM_INV_SQRT, _ws
        L = lib()
        dev = edge_index.device
        E = edge_index.size(1)
        ei = edge_index.contiguous()
        e_src = torch.empty(max(E + N, 1), dtype=torch.int32, device=dev)
        e_dst = torch.empty(max(E + N, 1), dtype=torch.int32, device=dev)
        nnz_dev = torch.empty(1, dtype=torch.int64, device=dev)
        ws = _ws(L.rgbmp_edge_edit_workspace_bytes(E, N), dev)
        check(L.rgbmp_edge_edit(ptr(ei[0]), ptr(ei[1]), E, N, loop_mode, ptr(e_src), ptr(e_dst), ptr(nnz_dev),
                                ptr(ws), ws.numel(), dev.index, stream_of(dev)), "edge_edit")
        nnz = int(nnz_dev.item())
        if nnz < 0:
            raise RuntimeError("edge_index contains node ids outside [0, N)")
        self.nnz_global = nnz
        self.N, self.rank, self.world = N, rank, world
        self.R = rows_per_rank(N, world)
        self.lo, self.hi = row_range(N, rank, world)
        e_src, e_dst = e_src[:nnz], e_dst[:nnz]
        # locality groups of the row schedule (graph.locality_groups): a property of the NODES of the whole graph, so
        # every rank derives them from the (replicated) edge list and gets the same answer without communication;
        # the transposed block reuses the forward block's
        from .graph import locality_groups
        self.perm = self.inv = None
        if transpose_of is not None:
            self.groups, self.perm, self.inv = transpose_of.groups, transpose_of.perm, transpose_of.inv
        else:
            whole = CSR(e_dst, e_src, N, N, finish=False)
            self.groups = locality_groups(whole, whole.degree_order()) if N > 1 and nnz > 0 else None
            del whole
            if relabel and self.groups is not None:
                grp, n_groups = self.groups
                self.perm, self.inv = community_naming(grp, N)                    # new id -> old id, old id -> new id
                self.groups = (grp[self.perm].contiguous(), n_groups)            # group of every node under its new name
        if self.inv is not None:
            e_src = self.inv[e_src.long()].to(torch.int32)
            e_dst = self.inv[e_dst.long()].to(torch.int32)
        if transpose_of is None:
            key, other = local_edges(e_src, e_dst, self.lo, self.hi)
        else:                                   # bucket by SOURCE: row = local source id, col = global target id
            key, other = local_edges(e_dst, e_src, self.lo, self.hi)
        del e_src, e_dst
        local_groups = None
        if self.groups is not None and block_keeps_groups(self.R, row_bytes):
            grp, n_groups = self.groups
            mine = torch.zeros(self.R, dtype=torch.int32, device=dev)
            mine[: self.hi - self.lo] = grp[self.lo:self.hi]
            local_groups = (mine, n_groups)
        ck = (256, 2048) if local_groups is not None else (None, None)
        self.csr = CSR(key, other, self.R, self.R * world, chunk=ck[0], long_chunk=ck[1], groups=local_groups)
        self._norms(group, transpose_of)

    @classmethod
    def from_rowgen(cls, n_nodes: int, n_edges: int, rank: int, world: int, group=None, device=None, **gen_kw):
        """Row block of a row-generated graph (synth.rowgen_block): the CSR exists by construction --
        no edge list, no sort -- and each rank generates only its own rows (config C5)."""
        from . import synth
        from .graph import CSR
        self = cls.__new__(cls)
        self.N, self.rank, self.world = n_nodes, rank, world
        self.R = rows_per_rank(n_nodes, world)
        self.lo, self.hi = row_range(n_nodes, rank, world)
        self.groups = self.perm = self.inv = None
        rowptr, col = synth.rowgen_block(n_nodes, n_edges, self.lo, self.hi, device=device, **gen_kw)
        if self.hi - self.lo < self.R:             # pad the last block with empty rows
            rowptr = torch.cat([rowptr, rowptr[-1:].expand(self.R - (self.hi - self.lo))])
        self.csr = CSR.from_arrays(rowptr, col, self.R * world)
        t = torch.tensor([self.csr.nnz], dtype=torch.int64, device=device)
        if world > 1:
            dist.all_reduce(t, group=group)
        self.nnz_global = int(t.item())
        self._norms(group)
        return self

    def _norms(self, group, transpose_of=None):
        from ._lib import check, lib, ptr, stream_of
        from .graph import NORM_INV_SQRT
        L, dev, world = lib(), self.csr.device, self.world
        self.nnz_local = self.csr.nnz
        if transpose_of is not None:
            self.dinv_local, self.dinv_full = transpose_of.dinv_local, transpose_of.dinv_full
        else:
            self.dinv_local = self.csr.norm(NORM_INV_SQRT)                  # in-degrees of my rows are complete
            self.dinv_full = torch.empty(self.R * world, dtype=torch.float32, device=dev)
            if world > 1:
                dist.all_gather_into_tensor(self.dinv_full, self.dinv_local, group=group)
            else:
                self.dinv_full.copy_(self.dinv_local)
        self.val = torch.empty(max(self.nnz_local, 1), dtype=torch.float32, device=dev)
        check(L.rgbmp_gcn_edge_weight(ptr(self.csr.rowptr), ptr(self.csr.col), self.R, ptr(self.dinv_local),
                                      ptr(self.dinv_full), ptr(self.val), dev.index, stream_of(dev)),
              "gcn_edge_weight")


class PeerBuffers:
    """`n_buf` device buffers of [rows, ld] elements per rank, each mapped into every other rank of
    the box through CUDA IPC (rgbmp_peer_alloc / rgbmp_peer_open), so that a kernel on rank p can
    store straight into rank q's copy over NVLink.  ptrs[b][q] = address (in THIS process) of rank
    q's buffer b; local[b] = this rank's buffer b as a torch tensor."""

    def __init__(self, rows: int, ld: int, dtype, device, rank: int, world: int, group=None, n_buf: int = 2):
        import ctypes as C
        from ._lib import check, lib
        L = lib()
        self.device, self.rank, self.world, self._open, self._own = device, rank, world, [], []
        esz = torch.empty((), dtype=dtype).element_size()
        nbytes = rows * ld * esz
        handles = []
        for _ in range(n_buf):
            p, h = C.c_void_p(), (C.c_ubyte * 64)()
            check(L.rgbmp_peer_alloc(nbytes, C.byref(p), h, device.index), "peer_alloc")
            self._own.append(p.value)
            handles.append(bytes(h))
        gathered = [None] * world
        dist.all_gather_object(gathered, handles, group=group)
        self.ptrs = []
        for b in range(n_buf):
            row = []
            for q in range(world):
                if q == rank:
                    row.append(self._own[b])
                else:
                    p = C.c_void_p()
                    hb = (C.c_ubyte * 64).from_buffer_copy(gathered[q][b])
                    check(L.rgbmp_peer_open(hb, C.byref(p), device.index), "peer_open")
                    self._open.append(p.value)
                    row.append(p.value)
            self.ptrs.append(row)
        self.local = [_wrap(p, nbytes, device).view(dtype).view(rows, ld) for p in self._own]

    def close(self):
        from ._lib import lib
        L = lib()
        torch.cuda.synchronize(self.device)
        for p in self._open:
            L.rgbmp_peer_close(p, self.device.index)
        self._open = []
        self.local = []
        for p in self._own:
            L.rgbmp_peer_free(p, self.device.index)
        self._own = []


class _RawCuda:
    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _wrap(ptr: int, nbytes: int, device) -> torch.Tensor:
    return torch.as_tensor(_RawCuda(ptr, nbytes), device=device)


class PartitionedAPPNP:
    """APPNP / LP-style K-hop propagation over a LocalBlock.

    mode="push" (default on a multi-GPU box): ONE fused kernel per hop -- the SpMM's epilogue
    stores every finished row of the new iterate into ALL ranks' copies of the full iterate over
    NVLink (peer-mapped buffers, ping/pong), so the all-gather overlaps the aggregation row by row;
    a 4-byte NCCL all-reduce orders the hops.  The normalisation is folded into row scalings (the
    buffers hold D^-1/2 z, no per-edge weight stream) and the last hop stays local.
    mode="allgather": the baseline -- NCCL all_gather_into_tensor of the iterate rows, then the SpMM."""

    def __init__(self, block: LocalBlock, F: int, group=None, mode: str = "push", dtype=torch.float32,
                 ld: Optional[int] = None):
        from . import _lib, ops
        _lib.dtype_code(torch.empty(0, dtype=dtype))        # float32 / bfloat16 only: anything else raises here
        self.block, self.F, self.group, self.dtype = block, F, group, dtype
        self.ld = ops.padded_width(F, dtype) if ld is None else int(ld)
        if self.ld < ops.padded_width(F, dtype) or self.ld % ops.padded_width(1, dtype) != 0:
            raise RuntimeError(f"ld={self.ld} is not a vector-aligned width >= F={F}")
        dev = block.csr.device
        R, P = block.R, block.world
        self.mode = mode if P > 1 else "allgather"
        self.launches_per_hop = 1 + (2 if block.csr.n_items > 0 else 0)
        if self.mode == "push":
            self.peers = PeerBuffers(R * P, self.ld, dtype, dev, block.rank, P, group, n_buf=2)
            self.tick = torch.zeros(1, dtype=torch.int32, device=dev)
            self.out = torch.zeros((R, self.ld), dtype=dtype, device=dev)
            for t in self.peers.local:
                t.zero_()
            return
        self.full = torch.empty((R * P, self.ld), dtype=dtype, device=dev)
        self.ping = torch.zeros((R, self.ld), dtype=dtype, device=dev)
        self.pong = torch.zeros((R, self.ld), dtype=dtype, device=dev)
        self._flip = False

        def spmm(x_full, z0_local, a, b, clamp=None, reset=None):
            out = self.pong if self._flip else self.ping
            self._flip = not self._flip
            tele = dict(b=b, T=z0_local, ldt=z0_local.stride(0)) if b != 0.0 else {}
            post = {} if reset is None else ops.reset_rows(*reset, F)     # run() converted the rows: no copy here
            ep = ops.make_epilogue(a=a, clamp=clamp, **tele, **post)
            ops.spmm_raw(block.csr, x_full[:, :F], block.val, ep=ep, keep=(z0_local,), out=out[:, :F])
            return out

        self.driver = PartitionedPropagator(block.N, block.rank, block.world, spmm, group)
        self.launches_per_hop = 1 + (2 if block.csr.n_items > 0 else 0)

    def run(self, z0_local: torch.Tensor, K: int, alpha: float = 0.0, *, teleport=None, clamp=None,
            reset=None) -> torch.Tensor:
        """z0_local: [R, ld] (padded rows beyond N are zero).  Returns this rank's rows of z_K.
        alpha = 0 is the plain K-hop GCN propagation A_hat^K z0 (no teleport read).

        Label propagation (ops.label_propagation on a LOOP_NONE block) through the same hops:
          teleport=(a, b): z <- a * A_hat z + b * z0 in place of (1 - alpha, alpha); LP's is (alpha, 1 - alpha);
          clamp=(lo, hi): every new iterate is clamped after the teleport;
          reset=(mask [R], values [R, >= F]): then the masked rows of every new iterate take their `values` (read as
          float32, RESET_AFTER_CLAMP).  Rows are this block's."""
        from . import _lib
        if z0_local.dtype != self.dtype:
            _lib.dtype_code(z0_local)
            raise RuntimeError(f"z0_local is {z0_local.dtype}; this propagation was built for {self.dtype}")
        a, b = (1.0 - alpha, alpha) if teleport is None else (float(teleport[0]), float(teleport[1]))
        from . import ops
        check_post_step(self.block.R, clamp, reset)
        post = {} if reset is None else ops.reset_rows(*reset, self.F)    # once per run
        if self.mode != "push":
            if reset is not None:
                reset = (post["reset_mask"], post["reset_val"])
            return self.driver.run(z0_local, K, a, b, self.full, clamp=clamp, reset=reset)
        blk, F, R = self.block, self.F, self.block.R
        full = self.peers.local
        d = blk.dinv_local
        # folded normalisation: the peer buffers hold u_k = D^-1/2 z_k (what the hop gathers, no per-edge
        # weight stream); the epilogue rebuilds z_{k+1} = post(a * d_i * sum_j u_k[j] + b * z0_i) and pushes d_i * z_{k+1}
        u0 = ops.row_scale(z0_local, d)
        dist.all_gather_into_tensor(full[0], u0, group=self.group)                # iterate 0 everywhere
        # timing-only switches for attributing the hop time (results are WRONG with either of them set)
        dbg_self_only = os.environ.get("RGBMP_DEBUG_PUSH") == "self"
        dbg_no_tick = os.environ.get("RGBMP_DEBUG_TICK") == "0"
        tele = dict(b=b, T=z0_local, ldt=z0_local.stride(0)) if b != 0.0 else {}
        for k in range(K):
            src, nxt, last = full[k & 1], (k + 1) & 1, k == K - 1
            if last:                       # the result stays local and unscaled: no push, no tick
                ep = ops.make_epilogue(row_scale=d, a=a, clamp=clamp, **tele, **post)
                ops.spmm_raw(blk.csr, src[:, :F], None, ep=ep, keep=(z0_local, d), out=self.out[:, :F])
                break
            peers = [self.peers.ptrs[nxt][blk.rank]] if dbg_self_only else self.peers.ptrs[nxt]
            ep = ops.make_epilogue(row_scale=d, a=a, out2_scale=d, peers=peers, peer_row0=blk.rank * R,
                                   ld_peer=self.ld, clamp=clamp, **tele, **post)
            ops.spmm_raw(blk.csr, src[:, :F], None, ep=ep, keep=(z0_local, d), store_local=False)
            if not dbg_no_tick:
                dist.all_reduce(self.tick, group=self.group)     # orders the hops: every push has landed
        return self.out

    def close(self):
        if self.mode == "push":
            self.peers.close()


# ------------------------------------------------------------------------------------------------
# autograd over the partitioned propagation (distributed training epochs)
# ------------------------------------------------------------------------------------------------
class _DistKHop(torch.autograd.Function):
    """z = M z0 on this rank's rows / feature slice; the map is linear, so the backward is the same
    K-hop recursion on the transposed row block (SURVEY.md A8: nothing but the graph is saved)."""

    @staticmethod
    def forward(ctx, z0_local, fwd_run, bwd_run):
        ctx.bwd_run = bwd_run
        return fwd_run(z0_local.contiguous()).clone()

    @staticmethod
    def backward(ctx, dz):
        return ctx.bwd_run(dz.contiguous()).clone(), None, None


class _GatherSlices(torch.autograd.Function):
    """[R, ld_slice] feature slices of the ranks that share a row block -> [R, F]; backward = own slice."""

    @staticmethod
    def forward(ctx, z_slice, grid: "Grid", F: int, col_group):
        ctx.grid, ctx.F, ctx.ld = grid, F, z_slice.size(1)
        if grid.Pf == 1:
            return z_slice[:, :F]
        parts = torch.empty((grid.Pf * z_slice.size(0), z_slice.size(1)), dtype=z_slice.dtype, device=z_slice.device)
        dist.all_gather_into_tensor(parts, z_slice.contiguous(), group=col_group)
        parts = parts.view(grid.Pf, z_slice.size(0), z_slice.size(1))
        out = torch.empty((z_slice.size(0), F), dtype=z_slice.dtype, device=z_slice.device)
        for f in range(grid.Pf):
            a, b = grid.feature_slice(F, fp=f)
            out[:, a:b] = parts[f, :, : b - a]
        return out

    @staticmethod
    def backward(ctx, dout):
        grid, F = ctx.grid, ctx.F
        a, b = grid.feature_slice(F)
        d = torch.zeros((dout.size(0), ctx.ld), dtype=dout.dtype, device=dout.device)
        d[:, : b - a] = dout[:, a:b]
        return d, None, None, None


class DistAPPNP(torch.nn.Module):
    """APPNP(K, alpha) over a process grid, differentiable: forward(h [R, F] rows of my row block) ->
    [R, F] propagated rows.  Forward and backward each run the fused-push K-hop on their own row
    block (forward CSR / transposed CSR); feature slices are re-assembled with one all-gather among
    the Pf ranks of a row block.  `make_runner(block, F_slice)` builds the K-hop executor -- the CUDA
    PartitionedAPPNP in production, a CPU stand-in in the gloo tests."""

    def __init__(self, grid: "Grid", F: int, K: int, alpha: float, fwd_runner, bwd_runner, col_group=None, align: int = 4):
        super().__init__()
        self.grid, self.F, self.K, self.alpha = grid, F, K, alpha
        self.fwd_runner, self.bwd_runner, self.col_group = fwd_runner, bwd_runner, col_group
        self.ld = self.slice_ld(grid, F, align)
        from . import memo as _memo_cfg
        self.eval_memo, self._memo, self.memo_hits = _memo_cfg.enabled(), None, 0

    @staticmethod
    def slice_ld(grid: "Grid", F: int, align: int = 4) -> int:
        """Common leading dimension of every rank's feature-slice buffers (widest slice, vector aligned)."""
        w = max(b - a for a, b in (grid.feature_slice(F, align, fp=f) for f in range(grid.Pf)))
        return (w + align - 1) // align * align

    def forward(self, h: torch.Tensor) -> torch.Tensor:
        if torch.is_grad_enabled() or not self.eval_memo:
            return self._propagate(h)
        # SURVEY 8f f2: the caller's two eval forwards per epoch are identical -- reuse the first result when EVERY
        # rank sees bit-identical input rows again (the decision is all-reduced: a rank must never skip a collective
        # that its peers enter)
        memo = self._memo
        same = memo is not None and memo[0].shape == h.shape and torch.equal(memo[0], h)
        flag = torch.tensor([1 if same else 0], dtype=torch.int32, device=h.device)
        if self.grid.world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            self.memo_hits += 1
            return memo[1].clone()
        out = self._propagate(h)
        self._memo = (h.detach().clone(), out.detach().clone())
        return out

    def _propagate(self, h: torch.Tensor) -> torch.Tensor:
        a, b = self.grid.feature_slice(self.F)
        z0 = torch.zeros((h.size(0), self.ld), dtype=h.dtype, device=h.device)
        z0[:, : b - a] = h[:, a:b]
        z = _DistKHop.apply(z0, lambda t: self.fwd_runner(t, self.K, self.alpha),
                            lambda t: self.bwd_runner(t, self.K, self.alpha))
        return _GatherSlices.apply(z, self.grid, self.F, self.col_group)


class DistCorrectAndSmooth:
    """Correct & Smooth (shim.nn.CorrectAndSmooth, SURVEY A15) over a process grid: `correct` / `smooth` take this rank's
    [R, F] rows in the block's naming (R = ceil(N / Pr); rows >= N of the last block are padding) and return [R, F] rows.

    Both label propagations run through `runner(z0 [R, ld], K, *, teleport=(a, b), clamp=, reset=) -> [R, ld]` on this
    rank's feature slice `grid.feature_slice(F)` -- PartitionedAPPNP.run on a LOOP_NONE block built with
    ld = DistCorrectAndSmooth.slice_ld(grid, F, dtype) in production, a CPU stand-in in the gloo tests.  What the
    reference computes over the whole graph is reduced over the grid:
      * sigma = sum |error[mask]| / numel and the mean row sum of y_soft (checked to be 1, as the reference does):
        float64 partial sums of the real rows, taken once per row (by the ranks of feature group 0, which hold the
        same full-width rows as the rest of their row block) and all-reduced over every rank, then rounded once --
        so sigma does not depend on the grid;
      * the per-row L1 norm of the smoothed error: taken over the full row after the feature slices are assembled
        (one all-gather among the Pf ranks of a row block, which the [R, F] result needs anyway);
      * fixed-scale correction resets this rank's rows of the training mask to its rows of the error.
    Padded rows count nowhere and keep scale 1, so they never turn into NaN.  float32 / bfloat16 only."""

    def __init__(self, num_correction_layers, correction_alpha, num_smoothing_layers, smoothing_alpha,
                 autoscale=True, scale=1.0, *, grid: "Grid", N: int, runner, col_group=None):
        self.num_correction_layers, self.correction_alpha = int(num_correction_layers), float(correction_alpha)
        self.num_smoothing_layers, self.smoothing_alpha = int(num_smoothing_layers), float(smoothing_alpha)
        self.autoscale, self.scale = autoscale, scale
        self.grid, self.N, self.runner = grid, N, runner
        self.col_group = grid.col_group if col_group is None else col_group
        self.R = rows_per_rank(N, grid.Pr)
        lo, hi = row_range(N, grid.rp, grid.Pr)
        self.n_real = hi - lo                     # rows of this block that are nodes; the rest is padding

    @staticmethod
    def slice_ld(grid: "Grid", F: int, dtype=torch.float32) -> int:
        """Leading dimension of the [R, ld] slice buffers the runners take: the widest slice, 16-byte vectors."""
        v = 8 if dtype == torch.bfloat16 else 4
        return (DistAPPNP.slice_ld(grid, F) + v - 1) // v * v

    def _check(self, y_soft: torch.Tensor):
        if y_soft.dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError(f"DistCorrectAndSmooth takes float32 / bfloat16 rows (got {y_soft.dtype})")
        if y_soft.dim() != 2 or y_soft.size(0) != self.R:
            raise RuntimeError(f"y_soft must be this block's [{self.R}, F] rows (got {tuple(y_soft.shape)})")

    def _one_hot(self, y_true: torch.Tensor, y_soft: torch.Tensor) -> torch.Tensor:
        if y_true.dtype == torch.long:
            return torch.nn.functional.one_hot(y_true.view(-1), y_soft.size(-1)).to(y_soft.dtype)
        return y_true

    def _propagate(self, y: torch.Tensor, K: int, alpha: float, clamp=None, reset_mask=None) -> torch.Tensor:
        """Label propagation of the [R, F] rows `y` (res = (1 - alpha) * y; K x {y = alpha * A_hat y + res; post}),
        reset rows taking their values from `y`; returns the assembled [R, F] rows."""
        if K == 0:
            return y
        F = y.size(1)
        a, b = self.grid.feature_slice(F)
        z0 = torch.zeros((y.size(0), self.slice_ld(self.grid, F, y.dtype)), dtype=y.dtype, device=y.device)
        z0[:, : b - a] = y[:, a:b]
        reset = None if reset_mask is None else (reset_mask, z0)
        z = self.runner(z0, K, teleport=(alpha, 1.0 - alpha), clamp=clamp, reset=reset)
        # the runner's result lives in its own buffers, which its next run overwrites
        return _GatherSlices.apply(z, self.grid, F, self.col_group).clone()

    @torch.no_grad()
    def correct(self, y_soft: torch.Tensor, y_true: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        self._check(y_soft)
        R, n = self.R, self.n_real
        y_true = self._one_hot(y_true, y_soft)
        error = torch.zeros_like(y_soft)
        error[mask] = y_true - y_soft[mask]
        if mask.dtype == torch.bool:
            numel, bad = mask.sum(), mask[n:].sum()
        else:
            numel, bad = mask.numel(), (mask >= n).sum()
        stats = torch.zeros(5, dtype=torch.float64, device=y_soft.device)
        if self.grid.fp == 0:                      # every rank of a row block holds the same rows: count them once
            stats[0] = y_soft[:n].sum(dtype=torch.float64)
            stats[1] = n
            stats[2] = error[mask].abs().sum(dtype=torch.float64)
            stats[3] = numel
            stats[4] = bad
        if self.grid.world > 1:
            dist.all_reduce(stats)
        ysum, nodes, abs_err, numel, bad = stats.tolist()
        if bad:
            raise RuntimeError(f"the training mask selects {int(bad)} padded rows (>= N in the last block)")
        assert abs(ysum / nodes - 1.0) < 1e-2
        if self.autoscale:
            smoothed = self._propagate(error, self.num_correction_layers, self.correction_alpha, clamp=(-1.0, 1.0))
            sigma = torch.tensor(abs_err / numel if numel else float("nan"), dtype=y_soft.dtype, device=y_soft.device)
            scale = sigma / smoothed.abs().sum(dim=1, keepdim=True)
            scale[scale.isinf() | (scale > 1000)] = 1.0
            scale[n:] = 1.0
            return y_soft + scale * smoothed
        rmask = mask if mask.dtype == torch.bool else torch.zeros(
            R, dtype=torch.bool, device=y_soft.device).index_fill_(0, mask, True)
        smoothed = self._propagate(error, self.num_correction_layers, self.correction_alpha, reset_mask=rmask)
        return y_soft + self.scale * smoothed

    @torch.no_grad()
    def smooth(self, y_soft: torch.Tensor, y_true: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        self._check(y_soft)
        y_soft = y_soft.clone()
        y_soft[mask] = self._one_hot(y_true, y_soft)
        return self._propagate(y_soft, self.num_smoothing_layers, self.smoothing_alpha, clamp=(0.0, 1.0))
