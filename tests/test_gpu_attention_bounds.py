"""The fused attention family (csrc/att.cu: GAT, SuperGAT MX and SD, FAConv; forward and backward) against fp64, with an
element-wise error bound per output, at the split geometry that ships on graphs of SMALL_GRAPH_ROWS rows or more
(chunk 1024 / long_chunk 4096: the unsplit 33..1024-edge rows, work items of up to 4096 edges cut into Q = 256 / G
sub-ranges) as well as at the small-graph geometry (32 / 256).

Graphs.  The "degree ladder" (ladder_edges) has 24,000 nodes, so a default build splits at 1024 / 4096, random
background edges of mean degree 8, dedicated target rows whose in-degree after LOOP_REMOVE_THEN_ADD is each value of
LADDER, and dedicated source rows with the same out-degrees (the transpose CSR the backward walks).  The same edge list
is also built with chunk 32 / long_chunk 256, and `hub` / `medium` of helpers.CASES run at their own (small)
geometry.  test_ladder_geometry asserts that each build is the split it is meant to be.  References are computed from
the oracle's edited edge list (oracle.pyg_restated), never from the kernel's CSR; gradients come from fp64 autograd.
The fp64 arithmetic runs on the device; its own error (about deg * 2^-53) is far below every term here and is not
counted.

The bound.  As bound() in test_gpu_bf16.py: unit roundoff times a counted number of roundings, times the fp64
magnitude twin of the quantity (the same expression with every term in absolute value), to first order in u (the
neglected terms are below k^2 u^2 with k < 5000, i.e. under 2e-4 of the bound itself).  gamma(m) = m u / (1 - m u)
is Higham's bound for a sum in which a term passes m roundings.

  Logits, log2 domain.  The kernels take a_src / a_dst (a_l / a_r) times float(log2 e) -- two roundings each --,
  add them (one), and apply the float slope to negative values (the rounded constant and the product: two).  The
  error rho_ij of the logit t_ij therefore is, with a = a_src[j] + a_dst[i], A = |a_src[j]| + |a_dst[i]| and
  c = slope or 1 by the branch,
     GAT  rho = c log2e (2u A + u |a|) + [a < 0] 2u |t|
     MX   rho = c log2e (sig (2u A + u |a|) + |a| sig (r_sig + u)) + [raw < 0] 2u |t|, where sig = sigmoid(<x_i,x_j>)
          comes from rcp(1 + ex2(-d log2e)):  r_sig = (1 - sig)(gamma(C) D + 2u |d| + EX2) + u + RCP, d = <x_i, x_j>,
          D = <|x_i|, |x_j|> (the C-term dot product: per lane two chains of four FMAs and their sum, then log2(LPH)
          shuffle additions, so C is replaced by 5 + log2(LPH) -- dot_depth), 2u |d| the argument's two roundings;
     SD   rho = c log2e ls (gamma(C) D + 4u |d|) + [d < 0] 2u |t|: ls = float(1/sqrt(C)), ls * float(log2e) and the
          product with the dot product are four roundings.
  A logit error rho turns into a relative error ln2 * rho of that edge's exponential.

  Forward weight of edge (i, j), relative error
     eps_ij = ln2 (rho_ij + 2u |t_ij - m_i|) + EX2 (1 + R_ij + M_ij) + u (R_ij + M_ij + 1):
  the subtraction t - m and the subtractions of every later rescale or merge factor together are at most
  2u |t - m| (they telescope to the row maximum m); one ex2 for the term itself, one per rescale of the running
  accumulator after the term was added (R_ij: the kernel tests for a new maximum once per step of U = 2 edges, so a
  term sees at most the steps left in its sub-range) and one per merge (M_ij: 2 for a split row, the group merge in the
  work-item kernel and the item merge in the combine kernel); the rescale products, and the product with the mask
  value, round once each.  ex2.approx.ftz flushes results below 2^-126 to zero (as does a rescale factor that
  small, whose terms are then below 2^-126 too): each weight may also lose TINY = 2^-126 absolutely (s >= 1, the
  maximum's term is 1), so the error of alpha_ij is alpha_ij eps_ij + TINY.  The normalisation s -> 1/(s + 1e-16) -> acc * inv rounds three times, and s is a sum of
  the same depth as acc.  Per output element
     B_out = sum_j |mask| |x_j| (alpha eps_ij + TINY) + S_i (Ebar_i + 2 gamma(m_i) + gamma(3)),
     S_i = sum_j alpha_ij |mask_ij| |x_j|  (the output twin),  Ebar_i = sum_j (alpha_ij eps_ij + TINY) (the denominator's),
  m_i the summation depth of the split the kernel ran: deg for an unsplit row, ceil(min(deg, long_chunk) / Q) + Q +
  items for a split row (a group's sub-range, the group merge over Q partials, the item merge).  The training forward's
  second aggregate P_i = sum alpha l' mask x_j and q_i = sum alpha l' take the same bound with the extra rounding of
  alpha * slope on negative logits (2u).

  Backward.  The kernels rebuild alpha_ij = ex2(t - m') * inv from the forward's statistics: m' = (m ln2) log2e is
  the forward's maximum after four roundings (|m|-proportional: ln2 4u |m|), inv carries the forward sum's error
  (Ebar_i + gamma(m_i)) and two roundings, the product one more:
     eps_b = ln2 (rho + 4u |m_i| + u |t - m_i|) + EX2 + Ebar_i + gamma(m_i) + gamma(3),  and again + TINY absolutely.
  S_i = <dout_i, out_i> is formed from the forward's fp32 out, so dS_i = <|dout_i|, B_out_i> + gamma(C) <|dout|, |out|>.
  The softmax backward alpha (mask dalpha - S_i) l' has the twin alpha (|mask dalpha| + |S_i|) l'; its error is that
  twin times eps_b + 3u (+ 2u for the slope) plus alpha l' (|mask| gamma(dot_depth) <|dout_i|, |x_j|> + dS_i).
  Every gradient is then a sum over one CSR row of the pass that forms it (the transpose CSR for dX / da_src / da_l,
  the forward CSR for MX / SD's dXf and da_r, with the plain-sum depth of that split) of per-edge terms: bound = sum
  of the terms' errors + gamma(depth) * sum of their twins.  MX's dlogit = draw (u ln2) sig (1 - sig) and SD's draw * ls add the
  errors of their factors; da_dst = <dout, P> - S q and FAConv's da_r = <dout, Q> (formed in the prep kernel) add
  the cancellation s2 - S q: u |s2| + 2u |S q|.

  FAConv: w = tanhf(a_l + a_r) * dinv_j * dinv_i * mask.  tanhf within TANH, its argument's rounding through
  (1 - t^2), dinv = 1/sqrt(deg) in IEEE arithmetic (two roundings each), three products: |t| 7u + TANH |t| +
  (1 - t^2) u |a| per weight, then the sum over the row.

  Constants.  u = 2^-24 (fp32, round to nearest).  EX2 and RCP: the PTX ISA documents ex2.approx.ftz.f32 to 2 ulp and
  rcp.approx.ftz.f32 to 1 ulp across the full range; relative to the value that is at most 2^-22 and 2^-23.  An
  exhaustive sweep on a B200 over every float argument the kernels use (ex2 on [-127, 64] with a normal result,
  rcp on [2^-125, 2^125]; NVIDIA B200, 1000 W power limit) measured a relative error of at most 2^-22.71 for ex2
  (2.06 ulp of the correctly rounded float at worst) and 2^-23.28 for rcp (0.98 ulp): within EX2 and RCP.  TANH = 2^-22: tanhf is accurate to 2 ulp (CUDA C++ Programming Guide, mathematical
  functions, single precision).

  The kink.  leaky_relu has no derivative at 0.  Score scalars are drawn on a grid that keeps a_src + a_dst
  (a_l + a_r) at least 2^-11 from 0 (on_grid) -- far above any logit error here --, and SD's features carry one sign
  per (node, head) with magnitudes >= 0.2 (sd_features), so no logit lies within its error bound of the kink and the
  kernel takes the branch the reference takes on every edge.

Rejection (test_bound_rejects_wrong_answers): the same bound rejects a reference with one edge removed from the last
work item of the 4097-edge row, with one head's logits taken from its neighbour in a two-tile shape, and with one work
item of a split row merged against its own maximum instead of the row's.  In the randn regime the forward bound stays
below CEIL of the output twin, so it is not vacuous.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import CASES
from oracle import pyg_restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24          # unit roundoff of fp32
EX2 = 2.0 ** -22        # ex2.approx.ftz.f32: 2 ulp (PTX ISA), confirmed by a sweep on a B200 (module docstring)
RCP = 2.0 ** -23        # rcp.approx.ftz.f32: 1 ulp (PTX ISA), confirmed likewise
TINY = 2.0 ** -126      # .ftz: ex2 returns 0 for results below the smallest normal float, an absolute loss per weight
TANH = 2.0 ** -22       # tanhf: 2 ulp (CUDA C++ Programming Guide, single-precision mathematical functions)
LOG2E = 1.0 / math.log(2.0)
LN2 = math.log(2.0)
SLOPE = 0.2
CEIL = 2.0 ** -11       # randn regime: max bound / S of a forward; the rescale count of 1024-edge unsplit rows dominates
LADDER = (1, 2, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 4095, 4096, 4097, 8192, 12289, 40000)
N_LADDER = 24_000       # above SMALL_GRAPH_ROWS (18,944): a default build splits at 1024 / 4096
GRAPH_SEED = 20261018   # bench.py's GRAPH_SEED: the Reddit-shaped graph the reddit_gat workload times


def P():
    import rgb_experiment_b200 as P_
    return P_


def gamma(m):
    return m * U / (1 - m * U)


def att_G(H, Cp):
    """Lanes per row group of att_shape (csrc/att.cu) for H heads of Cp (padded) channels."""
    width = Cp if H == 1 else min(128 // Cp, H) * Cp
    g = 4
    while g < (width + 7) // 8:
        g <<= 1
    return g


def dot_depth(H, Cp):
    """Roundings a product passes in the kernels' per-head dot products: two chains of four FMAs per lane, their sum,
    then log2(LPH) shuffle additions over the lanes of the head (head_sum)."""
    lph = att_G(H, Cp) if H == 1 else Cp // 8
    return 5 + int(math.log2(lph))


def head_pad(H, C):
    if H == 1:
        return C
    c = 8
    while c < C:
        c <<= 1
    return c


def seg_sum(v, idx, n):
    return torch.zeros((n,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device).index_add_(0, idx, v)


def seg_max(v, idx, n):
    out = torch.full((n,) + tuple(v.shape[1:]), -math.inf, dtype=v.dtype, device=v.device)
    return out.scatter_reduce_(0, idx.view(-1, *([1] * (v.dim() - 1))).expand_as(v), v, "amax", include_self=True)


def assert_within(y, ref, bnd, what):
    err = (y.detach().double() - ref).abs()
    bad = err > bnd
    if bool(bad.any()):
        r = (err / bnd.clamp_min(1e-300))[bad]
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.numel()} elements beyond the bound "
                             f"(worst x{float(r.max()):.3g})")


def rejected(y, ref, bnd):
    return bool(((y.detach().double() - ref).abs() > bnd).any())


# ------------------------------------------------------------------------------------------------------------------
# graphs and their split geometry
# ------------------------------------------------------------------------------------------------------------------
def ladder_edges(seed=0):
    """(edge_index [2, E] without self loops, n, in-ladder targets, out-ladder sources, pivots).  Target T_k receives
    LADDER[k] - 1 edges (the loop makes LADDER[k]): first from its pivot P_k -- P_k has no other out-edge, so its score
    decides the first in-edge of T_k alone --, then from plain nodes.  Source S_k sends LADDER[k] - 1 edges to plain
    nodes.  T_k has no out-edge but its loop, which the edited list appends last: its last in-edge in CSR order."""
    gen = torch.Generator().manual_seed(seed)
    K, n = len(LADDER), N_LADDER
    plain0 = 3 * K

    def plain(k):
        return plain0 + torch.randint(n - plain0, (k,), generator=gen)

    src, dst = [], []
    for k, d in enumerate(LADDER):
        if d >= 2:
            src += [torch.tensor([2 * K + k]), plain(d - 2)]
            dst.append(torch.full((d - 1,), k))
    for k, d in enumerate(LADDER):
        src.append(torch.full((d - 1,), K + k))
        dst.append(plain(d - 1))
    bs, bd = plain(8 * n), plain(8 * n)
    keep = bs != bd
    src.append(bs[keep])
    dst.append(bd[keep])
    ei = torch.stack([torch.cat(src), torch.cat(dst)]).long()
    return ei, n, torch.arange(K), torch.arange(K, 2 * K), torch.arange(2 * K, 3 * K)


def geom(key, n, chunk, long_chunk, G):
    """Per edge of the edited list, in the CSR of rows `key` (stable: a row's edges keep their edited-list order):
    R = rescales the running maximum can apply after the edge was added, M = merges (0 or 2); per row: depth = the
    summation depth of the split the kernel ran."""
    E = key.numel()
    dev = key.device
    order = torch.argsort(key, stable=True)
    deg = torch.bincount(key, minlength=n)
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    rowptr[1:] = torch.cumsum(deg, 0)
    pos = torch.empty(E, dtype=torch.int64, device=dev)
    pos[order] = torch.arange(E, device=dev) - rowptr[key[order]]
    ln = deg[key]
    Q = 256 // G
    split = ln > chunk
    base = torch.where(split, pos // long_chunk * long_chunk, torch.zeros_like(pos))
    ilen = torch.where(split, torch.clamp(ln - base, max=long_chunk), ln)
    per = torch.where(split, (ilen + Q - 1) // Q, ilen)
    q = (pos - base) // per
    slen = torch.minimum(per, ilen - q * per)
    spos = pos - base - q * per
    R_ = (slen + 1) // 2 - 1 - spos // 2
    items = (deg + long_chunk - 1) // long_chunk
    depth = torch.where(deg > chunk, (torch.clamp(deg, max=long_chunk) + Q - 1) // Q + Q + items, deg)
    return {"R": R_.double(), "M": 2.0 * split.double(), "depth": depth.double(), "order": order, "pos": pos,
            "deg": deg, "item": torch.where(split, pos // long_chunk, -torch.ones_like(pos))}


class Setup:
    """One graph at one split geometry: the GPU Graph (both orientations), the oracle's edited edge list on the
    device and the per-edge geometry of each orientation for a lane-group width G."""

    def __init__(self, ei, n, **kw):
        self.n, self.kw = n, kw
        self.ei = ei.to(DEV)
        self.ed = R.edit_loops(ei, n, R.LOOP_REMOVE_THEN_ADD).to(DEV)
        self.g = P().Graph(self.ei, n, P().LOOP_REMOVE_THEN_ADD, **kw)
        self._gfa = None
        self._geo = {}

    def gfa(self):
        """FAConv aggregates the LOOP_ADD_REMAINING list: the same list when the input has no self loops."""
        if self._gfa is None:
            assert torch.equal(R.edit_loops(self.ei.cpu(), self.n, R.LOOP_ADD_REMAINING), self.ed.cpu())
            self._gfa = P().Graph(self.ei, self.n, P().LOOP_ADD_REMAINING, **self.kw)
        return self._gfa

    def geom(self, orient, G):
        k = (orient, G)
        if k not in self._geo:
            csr = getattr(self.g, orient)
            self._geo[k] = geom(self.ed[1] if orient == "fwd" else self.ed[0], self.n, csr.chunk, csr.long_chunk, G)
        return self._geo[k]


_SETUPS = {}


def setup(name):
    if name not in _SETUPS:
        if name.startswith("ladder"):
            ei, n, *_ = ladder_edges()
            kw = {} if name == "ladder/1024" else dict(chunk=32, long_chunk=256)
            _SETUPS[name] = Setup(ei, n, **kw)
        else:
            ei, n = CASES[name]()
            _SETUPS[name] = Setup(ei, n)
    return _SETUPS[name]


@pytest.fixture(scope="module", autouse=True)
def _free_setups():
    yield
    _SETUPS.clear()
    torch.cuda.empty_cache()


def test_ladder_geometry():
    """The builds are the splits the bounds assume: default chunking of a 24,000-node graph is 1024 / 4096; the
    ladder's degrees are exact; the CSR keeps the edited-list order within a row; unsplit rows of 33..1024 edges,
    split rows in both orientations, a row of at least 3 work items; work items start at multiples of long_chunk."""
    ei, n, T, S, _ = ladder_edges()
    for name, (chunk, lc) in (("ladder/1024", (1024, 4096)), ("ladder/32", (32, 256))):
        st = setup(name)
        g, ed = st.g, st.ed
        assert torch.equal(torch.bincount(ed[1], minlength=n)[T.to(DEV)].cpu(), torch.tensor(LADDER))
        assert torch.equal(torch.bincount(ed[0], minlength=n)[S.to(DEV)].cpu(), torch.tensor(LADDER))
        assert 200_000 < ed.size(1) < 600_000
        for orient, key, other in (("fwd", ed[1], ed[0]), ("bwd", ed[0], ed[1])):
            csr = getattr(g, orient)
            assert (csr.chunk, csr.long_chunk) == (chunk, lc), orient
            gm = st.geom(orient, 8)
            assert torch.equal(csr.col.long(), other[gm["order"]]), orient
            deg = gm["deg"]
            assert csr.n_long > 0 and int((deg > chunk).sum()) == csr.n_long, orient
            ni = csr.long_item_ptr.long()
            assert int((ni[1:] - ni[:-1]).max()) >= 3, orient
            starts = csr.item_start - csr.rowptr[csr.long_rows.long()[csr.item_long.long()]]
            assert bool((starts % lc == 0).all()), orient
        if chunk == 1024:
            deg = st.geom("fwd", 8)["deg"]
            assert int(((deg >= 33) & (deg <= 1024)).sum()) >= 6
    assert setup("hub").g.fwd.n_long > 0 and setup("medium").g.fwd.n_long > 0


# ------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------
def on_grid(v):
    """Values k / 1024 + 2^-12: any sum of two of them is at least 2^-11 from 0 (and so is 8 times it); exact in fp32."""
    return torch.floor(v * 1024) / 1024 + 2.0 ** -12


def scores(n, H, regime, gen):
    """(a_nbr, a_own) [n, H] for a logit regime.  late / early act on the ladder's rows: T_k's loop (its last in-edge)
    or its pivot edge (its first) gets the row's largest logit; early puts the others ~130 log2-units below, where
    ex2 flushes them to zero."""
    K = len(LADDER)
    a_n, a_o = on_grid(torch.randn(n, H, generator=gen)), on_grid(torch.randn(n, H, generator=gen))
    if regime == "peaked":
        a_n, a_o = a_n * 8, a_o * 8
    elif regime == "ties":
        a_n = torch.full((n, H), 2.0 ** -12)
    elif regime == "late":
        a_n[:K] = 12 + 2.0 ** -12
    elif regime == "early":
        a_n[2 * K:3 * K] = 90 + 2.0 ** -12
    return a_n, a_o


def sd_features(n, H, C, gen, scale=1.0):
    """One sign per (node, head), magnitudes 0.2 + 0.5 |randn|: |<x_i, x_j>| >= 0.04 C, never near the kink."""
    sign = torch.where(torch.rand(n, H, 1, generator=gen) < 0.5, -1.0, 1.0)
    return sign * (0.2 + 0.5 * torch.randn(n, H, C, generator=gen).abs()) * scale


# ------------------------------------------------------------------------------------------------------------------
# fp64 references and bounds
# ------------------------------------------------------------------------------------------------------------------
def slope_or_one(neg):
    """leaky_relu' in fp64 (a torch.where on Python scalars would give the float32 0.2)"""
    return 1.0 - (1.0 - SLOPE) * neg.double()


class Logits:
    """Exact log2-domain logits t [E, H] of a softmax score, their error bound rho, leaky_relu' factor lp, negative mask."""

    def __init__(self, t, rho, neg):
        self.t, self.rho, self.neg = t, rho, neg
        self.lp = slope_or_one(neg)


def gat_logits(a_n, a_o, src, dst):
    a = a_n[src] + a_o[dst]
    A = a_n[src].abs() + a_o[dst].abs()
    neg = a < 0
    c = slope_or_one(neg)
    t = LOG2E * c * a
    return Logits(t, c * LOG2E * (2 * U * A + U * a.abs()) + neg * 2 * U * t.abs(), neg)


def sig_rel(sig, d, D, Cd):
    return (1 - sig) * (gamma(Cd) * D + 2 * U * d.abs() + EX2) + U + RCP


def mx_logits(a_n, a_o, x3, src, dst, Cd):
    a = a_n[src] + a_o[dst]
    A = a_n[src].abs() + a_o[dst].abs()
    d = (x3[dst] * x3[src]).sum(-1)
    D = (x3[dst].abs() * x3[src].abs()).sum(-1)
    sig = torch.sigmoid(d)
    rs = sig_rel(sig, d, D, Cd)
    raw = a * sig
    neg = raw < 0
    c = slope_or_one(neg)
    t = LOG2E * c * raw
    rho = c * LOG2E * (sig * (2 * U * A + U * a.abs()) + a.abs() * sig * (rs + U)) + neg * 2 * U * t.abs()
    L = Logits(t, rho, neg)
    L.a, L.A, L.sig, L.rs = a, A, sig, rs
    return L


def sd_logits(x3, src, dst, C, Cd):
    ls = 1.0 / math.sqrt(C)
    d = (x3[dst] * x3[src]).sum(-1)
    D = (x3[dst].abs() * x3[src].abs()).sum(-1)
    neg = d < 0
    c = slope_or_one(neg)
    t = LOG2E * c * ls * d
    L = Logits(t, c * LOG2E * ls * (gamma(Cd) * D + 4 * U * d.abs()) + neg * 2 * U * t.abs(), neg)
    L.ls = ls
    return L


def softmax_forward(L, x3, mu, src, dst, n, gm, drop=None, item_shift=None):
    """fp64 forward of a softmax score from the edge list, with its bound.  drop: bool [E] edges left out of the
    reference; item_shift: (bool [E], [E, H]) log2 factors applied to chosen edges' exponentials (tests of the
    bound's power to reject)."""
    t = L.t
    H = t.size(1)
    m = seg_max(t if drop is None else t.masked_fill(drop.view(-1, 1), -math.inf), dst, n)
    p = torch.exp2(t - m[dst])
    if drop is not None:
        p = p.masked_fill(drop.view(-1, 1), 0.0)
    if item_shift is not None:
        p = torch.where(item_shift[0].view(-1, 1), p * torch.exp2(item_shift[1]), p)
    s = seg_sum(p, dst, n)
    alpha = p / s[dst]
    eps = (LN2 * (L.rho + 2 * U * (t - m[dst]).abs()) + (EX2 * (1 + gm["R"] + gm["M"]) + U * (gm["R"] + gm["M"] + 1)).view(-1, 1))
    mu_ = torch.ones_like(alpha) if mu is None else mu
    w = alpha * mu_
    ae = alpha * eps + TINY                                  # absolute error of a weight, flushed results included
    ax = x3[src].abs()
    out = seg_sum(w.unsqueeze(-1) * x3[src], dst, n)
    S = seg_sum(w.abs().unsqueeze(-1) * ax, dst, n)
    Ebar = seg_sum(ae, dst, n)
    norm = (Ebar + (2 * gamma(gm["depth"]) + gamma(3)).view(-1, 1)).unsqueeze(-1)
    B = seg_sum((mu_.abs() * ae).unsqueeze(-1) * ax, dst, n) + S * norm
    r = {"alpha": alpha, "m": m, "eps": eps, "Ebar": Ebar, "out": out, "S": S, "B": B, "w": w, "norm": norm}
    # training forward: P = sum alpha l' mask x_j and q = sum alpha l' (alpha * slope rounds twice more)
    ae2 = (alpha * (eps + L.neg * 2 * U) + TINY) * L.lp
    w2 = w * L.lp
    r["out2"] = seg_sum(w2.unsqueeze(-1) * x3[src], dst, n)
    r["B2"] = seg_sum((mu_.abs() * ae2).unsqueeze(-1) * ax, dst, n) + seg_sum(w2.abs().unsqueeze(-1) * ax, dst, n) * norm
    r["q"] = seg_sum(alpha * L.lp, dst, n)
    r["Bq"] = seg_sum(ae2, dst, n) + r["q"] * norm.squeeze(-1)
    return r


def softmax_backward_common(L, fw, x3, mu, d3, src, dst, n, gmF, Cp, Cd):
    """Per-edge pieces of every softmax backward: eps_b, the softmax-backward value, twin and error per edge."""
    out3 = fw["out"]
    S = (d3 * out3).sum(-1)
    dS = (d3.abs() * fw["B"]).sum(-1) + gamma(Cp) * (d3.abs() * out3.abs()).sum(-1)
    m = fw["m"]
    eb = (LN2 * (L.rho + 4 * U * m[dst].abs() + U * (L.t - m[dst]).abs()) + EX2 + fw["Ebar"][dst]
          + gamma(gmF["depth"]).view(-1, 1)[dst] + gamma(3))
    alpha = fw["alpha"]
    mu_ = torch.ones_like(alpha) if mu is None else mu
    dd = (d3[dst] * x3[src]).sum(-1)
    D = (d3[dst].abs() * x3[src].abs()).sum(-1)
    ae = alpha * eb + TINY                                   # absolute error of the rebuilt alpha
    mag = ((mu_ * dd).abs() + S[dst].abs()) * L.lp
    tw = alpha * mag
    err = ae * mag + tw * (3 * U + L.neg * 2 * U) + alpha * L.lp * (mu_.abs() * gamma(Cd) * D + dS[dst])
    return {"S": S, "dS": dS, "eb": eb, "ae": ae, "mu": mu_, "tw": tw, "err": err}


def row_bound(err, twin, idx, n, depth):
    """sum over a CSR row of per-edge errors + gamma(depth) * sum of the per-edge twins"""
    g = gamma(depth).view(-1, *([1] * (twin.dim() - 1)))
    return seg_sum(err, idx, n) + g * seg_sum(twin, idx, n)


def ceiling_ok(B, S):
    live = S > 0
    return float((B[live] / S[live]).max())


# ------------------------------------------------------------------------------------------------------------------
# GAT
# ------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 7), (1, 41), (1, 128), (8, 8), (16, 8), (2, 16), (5, 32), (2, 128), (3, 100), (8, 10)]
GAT_CASES = ([("ladder/1024", H, C, "randn", False) for H, C in SHAPES]
             + [("ladder/1024", H, C, r, False) for H, C in ((8, 8), (1, 41)) for r in ("peaked", "ties", "late", "early")]
             + [("ladder/1024", 8, 8, "randn", True), ("ladder/1024", 2, 128, "randn", True)]
             + [("ladder/32", H, C, "randn", False) for H, C in SHAPES]
             + [("ladder/32", 16, 8, "late", True)]
             + [(c, H, C, "randn", False) for c in ("hub", "medium") for H, C in ((8, 8), (1, 41), (5, 32))])


def gat_case(name, H, C, regime, masked, seed=0):
    """(kernel results, fp64 references, bounds) of one GAT forward + backward."""
    p = P()
    st = setup(name)
    n, src, dst = st.n, st.ed[0], st.ed[1]
    E = src.numel()
    gen = torch.Generator().manual_seed(seed + 1000 * H + C)
    x = torch.randn(n, H, C, generator=gen)
    a_n, a_o = scores(n, H, regime, gen)
    dout = torch.randn(n, H * C, generator=gen)
    keep = (torch.rand(E, H, generator=gen) > 0.3).float() / 0.7 if masked else None
    kd = None if keep is None else keep.to(DEV)
    xg, sg, dg = (t.to(DEV).clone().requires_grad_(True) for t in (x.view(n, H * C), a_n, a_o))
    out = p.ops.gat(xg, sg, dg, st.g, H, C, SLOPE, kd)
    out.backward(dout.to(DEV))
    with torch.no_grad():
        out_eval = p.ops.gat(xg.detach(), sg.detach(), dg.detach(), st.g, H, C, SLOPE, kd)
    # fp64 reference from the edited edge list (autograd for the gradients)
    xo, so, do_ = (t.detach().to(DEV, torch.float64).requires_grad_(True) for t in (x, a_n, a_o))
    mu = None if keep is None else keep.to(DEV).double()
    alpha = R.softmax(F.leaky_relu(so[src] + do_[dst], SLOPE), dst, num_nodes=n)
    ref = R.scatter_add(xo[src] * (alpha if mu is None else alpha * mu).unsqueeze(-1), dst, dim=0, dim_size=n)
    d64 = dout.to(DEV).double()
    ref.reshape(n, H * C).backward(d64)
    # bounds
    Cp = head_pad(H, C)
    G = att_G(H, Cp)
    gmF, gmT = st.geom("fwd", G), st.geom("bwd", G)
    x3 = xo.detach()
    L = gat_logits(so.detach(), do_.detach(), src, dst)
    fw = softmax_forward(L, x3, mu, src, dst, n, gmF)
    assert torch.allclose(fw["out"], ref.detach(), rtol=1e-12, atol=1e-12)
    d3 = d64.view(n, H, C)
    bc = softmax_backward_common(L, fw, x3, mu, d3, src, dst, n, gmF, Cp, dot_depth(H, Cp))
    V = fw["alpha"] * bc["mu"].abs()
    adout = d3.abs()[dst]
    B_dx = row_bound(((bc["ae"] + U * fw["alpha"]) * bc["mu"].abs()).unsqueeze(-1) * adout, V.unsqueeze(-1) * adout, src, n, gmT["depth"])
    B_da_src = row_bound(bc["err"], bc["tw"], src, n, gmT["depth"])
    s2 = (d3 * fw["out2"]).sum(-1)
    Sq = bc["S"] * fw["q"]
    B_da_dst = ((d3.abs() * fw["B2"]).sum(-1) + gamma(Cp) * (d3.abs() * fw["out2"].abs()).sum(-1)
                + bc["dS"] * fw["q"].abs() + bc["S"].abs() * fw["Bq"] + U * (s2.abs() + 2 * Sq.abs()))
    return {
        "fw": fw, "ref": ref.detach().reshape(n, H * C), "B": fw["B"].reshape(n, H * C), "S": fw["S"].reshape(n, H * C),
        "got": [(out, "out"), (out_eval, "eval out"), (xg.grad, "dX"), (sg.grad, "da_src"), (dg.grad, "da_dst")],
        "want": [(ref.detach().reshape(n, H * C), fw["B"].reshape(n, H * C)), (ref.detach().reshape(n, H * C), fw["B"].reshape(n, H * C)),
                 (xo.grad.reshape(n, H * C), B_dx.reshape(n, H * C)), (so.grad, B_da_src), (do_.grad, B_da_dst)],
        "L": L, "x3": x3, "mu": mu, "gmF": gmF, "out": out,
    }


def check_case(r, what):
    for (y, name), (ref, B) in zip(r["got"], r["want"]):
        assert_within(y, ref, B, f"{what}: {name}")


@pytest.mark.parametrize("name,H,C,regime,masked", GAT_CASES)
def test_gat_bounds(name, H, C, regime, masked):
    r = gat_case(name, H, C, regime, masked)
    check_case(r, f"GAT {name} {H}x{C} {regime} masked={masked}")
    if regime == "randn":
        share = ceiling_ok(r["B"], r["S"])
        assert share <= CEIL, f"bound / S = {share:.3g} > {CEIL:.3g}"


# ------------------------------------------------------------------------------------------------------------------
# SuperGAT MX
# ------------------------------------------------------------------------------------------------------------------
MX_CASES = ([("ladder/1024", H, C, "randn", False) for H, C in ((8, 8), (16, 8), (1, 41), (1, 128), (5, 32), (2, 128), (3, 100))]
            + [("ladder/1024", 8, 8, "peaked", False), ("ladder/1024", 8, 8, "randn", True)]
            + [("ladder/32", H, C, "randn", False) for H, C in ((8, 8), (1, 7), (2, 16))]
            + [("medium", 8, 10, "randn", False)])


def logit_backward(L, fw, bc, x3, d3, src, dst, n, gmF, gmT, dlog_f, dlog_err, das_f=None, das_err=None):
    """dX of a score that reads <x_i, x_j> (MX, SD): the transpose pass sums alpha mask dout_i + dlogit x_i over a source's
    out-edges and adds the forward pass's sum of dlogit x_j over its in-edges (one more rounding)."""
    dl, dle = dlog_f, dlog_err
    V = fw["alpha"] * bc["mu"].abs()
    adT = d3.abs()[dst]
    axi, axj = x3.abs()[dst], x3.abs()[src]
    twT = V.unsqueeze(-1) * adT + dl.unsqueeze(-1) * axi
    erT = ((bc["ae"] + U * fw["alpha"]) * bc["mu"].abs()).unsqueeze(-1) * adT + dle.unsqueeze(-1) * axi
    twF = dl.unsqueeze(-1) * axj
    erF = dle.unsqueeze(-1) * axj
    T_ = row_bound(erT, twT, src, n, gmT["depth"])
    F_ = row_bound(erF, twF, dst, n, gmF["depth"])
    return T_ + F_ + U * (seg_sum(twT, src, n) + seg_sum(twF, dst, n))


def mx_case(name, H, C, regime, masked, seed=0):
    p = P()
    st = setup(name)
    n, src, dst = st.n, st.ed[0], st.ed[1]
    E = src.numel()
    gen = torch.Generator().manual_seed(seed + 100 * H + C)
    x = torch.randn(n, H, C, generator=gen) * 0.7
    a_n, a_o = scores(n, H, regime, gen)
    dout = torch.randn(n, H * C, generator=gen)
    keep = (torch.rand(E, H, generator=gen) > 0.3).float() / 0.7 if masked else None
    kd = None if keep is None else keep.to(DEV)
    xg, lg, rg = (t.to(DEV).clone().requires_grad_(True) for t in (x.view(n, H * C), a_n, a_o))
    out = p.ops.supergat_mx(xg, lg, rg, st.g, H, C, SLOPE, kd)
    out.backward(dout.to(DEV))
    with torch.no_grad():
        out_eval = p.ops.supergat_mx(xg.detach(), lg.detach(), rg.detach(), st.g, H, C, SLOPE, kd)
    xo, lo, ro = (t.detach().to(DEV, torch.float64).requires_grad_(True) for t in (x, a_n, a_o))
    mu = None if keep is None else keep.to(DEV).double()
    logit = (xo[dst] * xo[src]).sum(-1)              # R.supergat_mx_alpha with the score scalars given per node
    e = F.leaky_relu((lo[src] + ro[dst]) * logit.sigmoid(), SLOPE)
    alpha = R.softmax(e, dst, num_nodes=n)
    ref = R.scatter_add(xo[src] * (alpha if mu is None else alpha * mu).unsqueeze(-1), dst, dim=0, dim_size=n)
    d64 = dout.to(DEV).double()
    ref.reshape(n, H * C).backward(d64)
    Cp = head_pad(H, C)
    G = att_G(H, Cp)
    gmF, gmT = st.geom("fwd", G), st.geom("bwd", G)
    x3 = xo.detach()
    L = mx_logits(lo.detach(), ro.detach(), x3, src, dst, dot_depth(H, Cp))
    fw = softmax_forward(L, x3, mu, src, dst, n, gmF)
    assert torch.allclose(fw["out"], ref.detach(), rtol=1e-12, atol=1e-12)
    d3 = d64.view(n, H, C)
    bc = softmax_backward_common(L, fw, x3, mu, d3, src, dst, n, gmF, Cp, dot_depth(H, Cp))
    sig, a, rs = L.sig, L.a, L.rs
    g1 = sig * (1 - sig)
    # dlogit = draw * (uu ln2) * sig * (1 - sig): uu = a log2e (3 roundings on A), ln2 (constant and product), sig,
    # 1 - sig (sig's error and the subtraction), three products
    ua = 2 * U * L.A + U * a.abs() + 2 * U * a.abs()
    dl = bc["tw"] * a.abs() * g1
    dle = bc["err"] * a.abs() * g1 + bc["tw"] * (ua * g1 + a.abs() * g1 * rs + a.abs() * sig * (sig * rs + U * (1 - sig))
                                                 + 3 * U * a.abs() * g1)
    B_dx = logit_backward(L, fw, bc, x3, d3, src, dst, n, gmF, gmT, dl, dle)
    das_tw = bc["tw"] * sig
    das_err = bc["err"] * sig + bc["tw"] * sig * rs
    B_dl = row_bound(das_err, das_tw, src, n, gmT["depth"])
    B_dr = row_bound(das_err, das_tw, dst, n, gmF["depth"])
    refo = ref.detach().reshape(n, H * C)
    return {
        "fw": fw, "B": fw["B"].reshape(n, H * C), "S": fw["S"].reshape(n, H * C),
        "got": [(out, "out"), (out_eval, "eval out"), (xg.grad, "dX"), (lg.grad, "da_l"), (rg.grad, "da_r")],
        "want": [(refo, fw["B"].reshape(n, H * C)), (refo, fw["B"].reshape(n, H * C)),
                 (xo.grad.reshape(n, H * C), B_dx.reshape(n, H * C)), (lo.grad, B_dl), (ro.grad, B_dr)],
    }


@pytest.mark.parametrize("name,H,C,regime,masked", MX_CASES)
def test_supergat_mx_bounds(name, H, C, regime, masked):
    r = mx_case(name, H, C, regime, masked)
    check_case(r, f"MX {name} {H}x{C} {regime} masked={masked}")
    if regime == "randn":
        share = ceiling_ok(r["B"], r["S"])
        assert share <= CEIL, f"bound / S = {share:.3g} > {CEIL:.3g}"


# ------------------------------------------------------------------------------------------------------------------
# SuperGAT SD
# ------------------------------------------------------------------------------------------------------------------
SD_CASES = ([("ladder/1024", H, C, "randn", False) for H, C in ((8, 8), (16, 8), (1, 41), (1, 128), (5, 32), (2, 128), (8, 10))]
            + [("ladder/1024", 8, 8, "peaked", False), ("ladder/1024", 3, 100, "randn", True)]
            + [("ladder/32", H, C, "randn", False) for H, C in ((8, 8), (1, 7))]
            + [("hub", 2, 16, "randn", False)])


def sd_oracle(x64, ed, n, H, Cc, slope=SLOPE, keep=None):
    """SD attention + aggregate in fp64 from the edited edge list (test_gpu_supergat_sd.sd_oracle, given the edited
    list): x64 [n, H, C], keep [E, H] in edge order."""
    e = F.leaky_relu((x64[ed[1]] * x64[ed[0]]).sum(-1) / math.sqrt(Cc), slope)
    alpha = R.softmax(e, ed[1], num_nodes=n)
    if keep is not None:
        alpha = alpha * keep
    return R.scatter_add(x64[ed[0]] * alpha.unsqueeze(-1), ed[1], dim=0, dim_size=n).reshape(n, H * Cc)


def sd_case(name, H, C, regime, masked, seed=0):
    p = P()
    st = setup(name)
    n, src, dst = st.n, st.ed[0], st.ed[1]
    E = src.numel()
    gen = torch.Generator().manual_seed(seed + 10 * H + C)
    x = sd_features(n, H, C, gen, math.sqrt(8.0) if regime == "peaked" else 1.0)
    dout = torch.randn(n, H * C, generator=gen)
    keep = (torch.rand(E, H, generator=gen) > 0.3).float() / 0.7 if masked else None
    kd = None if keep is None else keep.to(DEV)
    xg = x.view(n, H * C).to(DEV).clone().requires_grad_(True)
    out = p.ops.supergat_sd(xg, st.g, H, C, SLOPE, kd)
    out.backward(dout.to(DEV))
    with torch.no_grad():
        out_eval = p.ops.supergat_sd(xg.detach(), st.g, H, C, SLOPE, kd)
    xo = x.detach().to(DEV, torch.float64).requires_grad_(True)
    mu = None if keep is None else keep.to(DEV).double()
    ref = sd_oracle(xo, st.ed, n, H, C, keep=mu)
    d64 = dout.to(DEV).double()
    ref.backward(d64)
    Cp = head_pad(H, C)
    G = att_G(H, Cp)
    gmF, gmT = st.geom("fwd", G), st.geom("bwd", G)
    x3 = xo.detach()
    L = sd_logits(x3, src, dst, C, dot_depth(H, Cp))
    fw = softmax_forward(L, x3, mu, src, dst, n, gmF)
    assert torch.allclose(fw["out"].reshape(n, H * C), ref.detach(), rtol=1e-12, atol=1e-12)
    d3 = d64.view(n, H, C)
    bc = softmax_backward_common(L, fw, x3, mu, d3, src, dst, n, gmF, Cp, dot_depth(H, Cp))
    dl = bc["tw"] * L.ls                                     # dlogit = draw * ls: ls rounded, one product
    dle = (bc["err"] + bc["tw"] * 2 * U) * L.ls
    B_dx = logit_backward(L, fw, bc, x3, d3, src, dst, n, gmF, gmT, dl, dle)
    refo = ref.detach()
    return {
        "fw": fw, "B": fw["B"].reshape(n, H * C), "S": fw["S"].reshape(n, H * C),
        "got": [(out, "out"), (out_eval, "eval out"), (xg.grad, "dX")],
        "want": [(refo, fw["B"].reshape(n, H * C)), (refo, fw["B"].reshape(n, H * C)), (xo.grad.reshape(n, H * C), B_dx.reshape(n, H * C))],
    }


@pytest.mark.parametrize("name,H,C,regime,masked", SD_CASES)
def test_supergat_sd_bounds(name, H, C, regime, masked):
    r = sd_case(name, H, C, regime, masked)
    check_case(r, f"SD {name} {H}x{C} {regime} masked={masked}")
    if regime == "randn":
        share = ceiling_ok(r["B"], r["S"])
        assert share <= CEIL, f"bound / S = {share:.3g} > {CEIL:.3g}"


# ------------------------------------------------------------------------------------------------------------------
# FAConv
# ------------------------------------------------------------------------------------------------------------------
FA_CASES = ([("ladder/1024", C, False) for C in (7, 64, 100, 128)] + [("ladder/1024", 64, True)]
            + [("ladder/32", C, False) for C in (7, 128)])


@pytest.mark.parametrize("name,C,masked", FA_CASES)
def test_faconv_bounds(name, C, masked):
    p = P()
    st = setup(name)
    g = st.gfa()
    n, src, dst = st.n, st.ed[0], st.ed[1]
    E = src.numel()
    gen = torch.Generator().manual_seed(C)
    x = torch.randn(n, C, generator=gen)
    a_l, a_r = torch.randn(n, 1, generator=gen), torch.randn(n, 1, generator=gen)
    dout = torch.randn(n, C, generator=gen)
    keep = (torch.rand(E, generator=gen) > 0.5).float() / 0.5 if masked else None
    kd = None if keep is None else keep.to(DEV)
    xg, lg, rg = (t.to(DEV).clone().requires_grad_(True) for t in (x, a_l, a_r))
    out = p.ops.faconv(xg, lg, rg, g, kd)
    out.backward(dout.to(DEV))
    with torch.no_grad():
        out_eval = p.ops.faconv(xg.detach(), lg.detach(), rg.detach(), g, kd)
    xo, lo, ro = (t.detach().to(DEV, torch.float64).requires_grad_(True) for t in (x, a_l, a_r))
    mu = None if keep is None else keep.to(DEV).double()
    ref = R.faconv_aggregate(xo, torch.zeros_like(xo), lo, ro, st.ei, 0.0, mu)
    d64 = dout.to(DEV).double()
    ref.backward(d64)
    G = att_G(1, C)
    gmF, gmT = st.geom("fwd", G), st.geom("bwd", G)
    deg = gmF["deg"].double()
    dinv = torch.where(deg > 0, deg.rsqrt(), torch.zeros_like(deg))
    dd = dinv[src] * dinv[dst]
    mu_ = torch.ones(E, dtype=torch.float64, device=DEV) if mu is None else mu
    a = lo.detach().view(-1)[src] + ro.detach().view(-1)[dst]
    t = torch.tanh(a)
    dt = (1 - t * t) * U * a.abs() + TANH * t.abs()          # tanhf of the rounded sum
    one_m = 1 - t * t
    d1m = 2 * t.abs() * dt + U * t * t + U * one_m            # 1 - t*t: t's error, the product, the subtraction
    w, we = t * dd * mu_, dd * mu_.abs() * (dt + 7 * U * t.abs())     # dinv twice (2 roundings each), 3 products
    w2, w2e = one_m * dd * mu_, dd * mu_.abs() * (d1m + 7 * U * one_m)
    x3 = xo.detach()
    ax = x3.abs()[src]
    B = row_bound(we.view(-1, 1) * ax, w.abs().view(-1, 1) * ax, dst, n, gmF["depth"])
    out2 = seg_sum(w2.view(-1, 1) * x3[src], dst, n)
    B2 = row_bound(w2e.view(-1, 1) * ax, w2.abs().view(-1, 1) * ax, dst, n, gmF["depth"])
    adT = d64.abs()[dst]
    B_dx = row_bound(we.view(-1, 1) * adT, w.abs().view(-1, 1) * adT, src, n, gmT["depth"])
    dot = (d64[dst] * x3[src]).sum(-1)
    D = (d64.abs()[dst] * x3.abs()[src]).sum(-1)
    tw = dd * mu_.abs() * one_m * dot.abs()
    er = dd * mu_.abs() * (one_m * (gamma(dot_depth(1, C)) * D + 7 * U * dot.abs()) + dot.abs() * d1m)
    B_dl = row_bound(er, tw, src, n, gmT["depth"])
    B_dr = (d64.abs() * B2).sum(-1) + gamma(C) * (d64.abs() * out2.abs()).sum(-1)
    what = f"FAConv {name} C={C} masked={masked}"
    for y, want, bnd, nm in ((out, ref.detach(), B, "out"), (out_eval, ref.detach(), B, "eval out"), (xg.grad, xo.grad, B_dx, "dX"),
                             (lg.grad.view(-1), lo.grad.view(-1), B_dl, "da_l"), (rg.grad.view(-1), ro.grad.view(-1), B_dr, "da_r")):
        assert_within(y, want, bnd, f"{what}: {nm}")
    share = ceiling_ok(B, seg_sum(w.abs().view(-1, 1) * ax, dst, n))
    assert share <= CEIL, f"bound / S = {share:.3g} > {CEIL:.3g}"


# ------------------------------------------------------------------------------------------------------------------
# the bound rejects wrong answers
# ------------------------------------------------------------------------------------------------------------------
def test_bound_rejects_wrong_answers():
    """Changed references, computed the same way, each with its own bound; the kernel's output is left as it is."""
    st = setup("ladder/1024")
    n, src, dst = st.n, st.ed[0], st.ed[1]
    K = len(LADDER)
    # 1. one edge of the last work item of the 4097-edge row left out (its loop: the item holds that edge alone)
    H, C = 8, 8
    r = gat_case("ladder/1024", H, C, "randn", False)
    y = r["out"].detach().view(n, H, C)
    fw0 = r["fw"]
    assert_within(y, fw0["out"], fw0["B"], "unchanged reference")
    row = LADDER.index(4097)
    gm = r["gmF"]
    last = (dst == row) & (gm["pos"] == 4096)
    assert int(last.sum()) == 1 and int(gm["item"][last]) == 1
    fw = softmax_forward(r["L"], r["x3"], None, src, dst, n, gm, drop=last)
    assert rejected(y[row], fw["out"][row], fw["B"][row]), "an edge removed from the last work item passes"
    # 3. one work item of the 12289-edge row merged against its own maximum (factor 2^(M - m_item) left out)
    row = LADDER.index(12289)
    inrow = dst == row
    t = r["L"].t
    sub = [seg_max(t[inrow & (gm["item"] == k)], torch.zeros(int((inrow & (gm["item"] == k)).sum()), dtype=torch.long, device=DEV), 1)[0]
           for k in range(4)]
    M = torch.stack(sub).max(0).values
    k = int(torch.stack([(M - s).min() for s in sub]).argmax())
    sel = inrow & (gm["item"] == k)
    fw = softmax_forward(r["L"], r["x3"], None, src, dst, n, gm, item_shift=(sel, (M - sub[k]).expand(src.numel(), H)))
    assert rejected(y[row], fw["out"][row], fw["B"][row]), "an item merged against its own maximum passes"
    # 2. one head's logits taken from its neighbour in a two-tile shape (5 heads of 32: tiles of 4 + 1)
    H, C = 5, 32
    r = gat_case("ladder/1024", H, C, "randn", False)
    y = r["out"].detach().view(n, H, C)
    L = r["L"]
    t2 = L.t.clone()
    t2[:, 4] = L.t[:, 3]
    L2 = type(L)(t2, L.rho, L.neg)
    fw = softmax_forward(L2, r["x3"], None, src, dst, n, r["gmF"])
    rows = torch.arange(3 * K, n, device=DEV)
    assert rejected(y[rows, 4], fw["out"][rows, 4], fw["B"][rows, 4]), "head 4 with head 3's logits passes"


# ------------------------------------------------------------------------------------------------------------------
# the bench's own graph: the Reddit-shaped graph and build of bench.py --workload reddit_gat
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def reddit():
    p = P()
    import rgb_experiment_b200.synth as S
    sg = S.make_named("reddit", seed=GRAPH_SEED, device=DEV, features=False)
    n = sg.num_nodes
    g = p.get_graph(sg.edge_index, n, p.LOOP_REMOVE_THEN_ADD)
    ed = R.edit_loops(sg.edge_index, n, R.LOOP_REMOVE_THEN_ADD)
    assert ed.size(1) == g.nnz
    deg = torch.bincount(ed[1], minlength=n)
    gen = torch.Generator(device=DEV).manual_seed(5)
    picks = [torch.argsort(deg, descending=True, stable=True)[:64]]
    for lo, hi in ((33, 64), (65, 256), (257, 1024), (1025, 4096)):
        band = torch.nonzero((deg >= lo) & (deg <= hi)).view(-1)
        assert band.numel() >= 64, (lo, hi)
        picks.append(band[torch.randperm(band.numel(), generator=gen, device=DEV)[:64]])
    picks.append(torch.randperm(n, generator=gen, device=DEV)[:512])
    rows = torch.unique(torch.cat(picks))
    keep = torch.zeros(n, dtype=torch.bool, device=DEV)
    keep[rows] = True
    sub = ed[:, keep[ed[1]]]                                 # the rows' in-edges, in edited-list order
    yield {"sg": sg, "g": g, "n": n, "rows": rows, "sub": sub, "clustered": g.fwd.clustered}
    del sg, g, ed, sub
    torch.cuda.empty_cache()


@pytest.mark.parametrize("op,H,C,scale", [("gat", 8, 8, 1.0), ("gat", 8, 8, 3.0), ("gat", 1, 41, 1.0), ("mx", 8, 8, 1.0)])
def test_reddit_rows_forward(reddit, op, H, C, scale):
    """The bench layer's forward on sampled target rows -- the 64 longest, 64 from each degree band 33-64, 65-256,
    257-1024, 1025-4096, 512 at random -- against fp64 from the rows' in-edges, with whatever schedule the build picked
    (fwd.clustered is recorded in the failure message)."""
    p = P()
    n, rows, sub, g = reddit["n"], reddit["rows"], reddit["sub"], reddit["g"]
    gen = torch.Generator(device=DEV).manual_seed(H * 100 + C)
    x = torch.randn(n, H * C, device=DEV, generator=gen) * (0.7 if op == "mx" else 1.0)
    a_n = torch.randn(n, H, device=DEV, generator=gen) * scale
    a_o = torch.randn(n, H, device=DEV, generator=gen) * scale
    with torch.no_grad():
        fn = p.ops.gat if op == "gat" else p.ops.supergat_mx
        out = fn(x, a_n, a_o, g, H, C, SLOPE).view(n, H, C)
    src, dst = sub[0], sub[1]
    Cp = head_pad(H, C)
    gm = geom(dst, n, g.fwd.chunk, g.fwd.long_chunk, att_G(H, Cp))
    x3 = x.double().view(n, H, C)
    if op == "gat":
        L = gat_logits(a_n.double(), a_o.double(), src, dst)
        e = F.leaky_relu(a_n.double()[src] + a_o.double()[dst], SLOPE)
    else:
        L = mx_logits(a_n.double(), a_o.double(), x3, src, dst, dot_depth(H, Cp))
        e = F.leaky_relu((a_n.double()[src] + a_o.double()[dst]) * (x3[dst] * x3[src]).sum(-1).sigmoid(), SLOPE)
    fw = softmax_forward(L, x3, None, src, dst, n, gm)
    alpha = R.softmax(e, dst, num_nodes=n)
    ref = R.scatter_add(x3[src] * alpha.unsqueeze(-1), dst, dim=0, dim_size=n)
    assert torch.allclose(fw["out"][rows], ref[rows], rtol=1e-12, atol=1e-12)
    assert_within(out[rows], ref[rows], fw["B"][rows], f"reddit {op} {H}x{C} x{scale} clustered={reddit['clustered']}")
    assert int((gm["deg"][rows] > g.fwd.chunk).sum()) >= 64 and g.fwd.n_items > 0


# ------------------------------------------------------------------------------------------------------------------
# schedule and dropout at the 1024 / 4096 geometry
# ------------------------------------------------------------------------------------------------------------------
def _all_ops(p, g, gfa, n, **kw):
    """name -> callable(inputs) for the four ops at one shape each, dropout keyword arguments kw(name, H)."""
    return {
        "gat": (lambda x, a, b, k: p.ops.gat(x, a, b, g, 8, 8, SLOPE, **k), 8, 64),
        "mx": (lambda x, a, b, k: p.ops.supergat_mx(x, a, b, g, 8, 8, SLOPE, **k), 8, 64),
        "sd": (lambda x, a, b, k: p.ops.supergat_sd(x, g, 5, 32, SLOPE, **k), 5, 160),
        "fa": (lambda x, a, b, k: p.ops.faconv(x, a, b, gfa, **k), 1, 100),
    }


def _run(fn, ins, dout, k):
    ins = [t.clone().requires_grad_(True) for t in ins]
    out = fn(*ins, k)
    out.backward(dout)
    return [out.detach()] + [t.grad for t in ins if t.grad is not None]


def _inputs(n, H, F_, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    return ([torch.randn(n, F_, device=DEV, generator=gen) * 0.7, torch.randn(n, H, device=DEV, generator=gen),
             torch.randn(n, H, device=DEV, generator=gen)], torch.randn(n, F_, device=DEV, generator=gen))


def test_grouped_schedule_equals_degree_schedule(monkeypatch):
    """The locality-grouped row schedule (graph.CLUSTER = "1") against the degree schedule on the ladder: all four ops,
    forward and every gradient, bit for bit (a row's arithmetic does not depend on when it runs)."""
    p = P()
    import rgb_experiment_b200.graph as G_
    st = setup("ladder/1024")
    assert not st.g.fwd.clustered
    monkeypatch.setattr(G_, "CLUSTER", "1")
    gc = p.Graph(st.ei, st.n, p.LOOP_REMOVE_THEN_ADD)
    gcfa = p.Graph(st.ei, st.n, p.LOOP_ADD_REMAINING)
    assert gc.fwd.clustered and gc.bwd.clustered and gc.fwd.n_items == st.g.fwd.n_items
    plain, grouped = _all_ops(p, st.g, st.gfa(), st.n), _all_ops(p, gc, gcfa, st.n)
    for name, (fn, H, F_) in plain.items():
        ins, dout = _inputs(st.n, H, F_, len(name))
        if name == "fa":
            ins = [ins[0], ins[1][:, :1], ins[2][:, :1]]
        a = _run(fn, ins, dout, {})
        b = _run(grouped[name][0], ins, dout, {})
        assert len(a) == len(b) >= 2
        for i, (u, v) in enumerate(zip(a, b)):
            assert torch.equal(u, v), (name, i, float((u - v).abs().max()))


def test_fused_dropout_equals_explicit_mask_at_large_geometry():
    """Fused attention dropout (mask regenerated in the kernels from a seed) against the explicit mask of the same seed,
    on the ladder at 1024 / 4096: all four ops, output and every gradient, bit for bit."""
    p = P()
    ops = p.ops
    st = setup("ladder/1024")
    for name, (fn, H, F_) in _all_ops(p, st.g, st.gfa(), st.n).items():
        ins, dout = _inputs(st.n, H, F_, 7 + len(name))
        if name == "fa":
            ins = [ins[0], ins[1][:, :1], ins[2][:, :1]]
        s = 31 + F_
        fused = _run(fn, ins, dout, dict(dropout_p=0.3, generator=torch.Generator(device=DEV).manual_seed(s)))
        mask = ops.dropout_mask(st.g, H, 0.3, ops.dropout_seed(DEV, torch.Generator(device=DEV).manual_seed(s)))
        explicit = _run(fn, ins, dout, dict(drop_edge=mask.view(-1) if name == "fa" else mask))
        for i, (u, v) in enumerate(zip(fused, explicit)):
            assert torch.equal(u, v), (name, i, float((u - v).abs().max()))
