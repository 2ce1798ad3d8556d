"""bf16 storage with fp32 accumulation: SpMM launch shapes, epilogues, K-hop families, autograd and C&S against a
plain fp64 reference, elementwise; plus the dtype contract of every public op (correct, or RuntimeError -- never a
misread).

The reference is the oracle's edited edge list and gcn_norm weights (oracle.pyg_restated) summed in fp64 on the
bf16 inputs, which are exact in fp64.  Every bound is derived from the unit roundoffs (bound() and khop_ref() say
where each term comes from); none is scaled by a safety factor.

One metamorphic relation ties the two instantiations together: for a fixed launch shape the bf16 kernel does the same
fp32 arithmetic in the same order as the fp32 kernel on x.float(), and only the final store rounds differently, so
    spmm_bf16(x) == spmm_f32(x.float()).to(bfloat16)        bit for bit, split rows included.
"""
import math

import pytest
import torch

from helpers import CASES
from oracle import pyg_restated as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BF = torch.bfloat16
U16 = 2.0 ** -8        # unit roundoff of bf16 (8 significant bits, round to nearest even)
U32 = 2.0 ** -24       # unit roundoff of fp32
SHAPES = [(G, V, U) for G in (1, 2, 4, 8, 16, 32) for V in (1, 2) for U in (2, 4, 8, 18, 20)]
REL = (16, 1, 4)       # launch shape of the cross-dtype comparisons that do not sweep shapes
# fp32 roundings on the path of one term besides the row's additions (the m of gamma_m):
NORM_W = 5             # gcn weight fl(fl(1/fl(sqrt(deg_j))) * fl(1/fl(sqrt(deg_i)))): two per factor, one for the product
FOLD = 6               # folded D^-1/2: d_j (2) and the pre-scale product (1), d_i (2) and the row-scale product (1)
TELE = 3               # a * v, b * T and their sum
CEIL = 2.0 ** -4       # a K-hop budget (K <= 10) must stay below this share of ||ref||_inf to mean anything


def P():
    import rgb_experiment_b200 as P_
    return P_


def tune(G, V, U):
    return G | (V << 8) | (U << 16)


def gamma(m):
    m = m.double()
    return m * U32 / (1 - m * U32)


def bound(ref, S, m, rounded=None):
    """Elementwise bound on |y - ref| for ONE SpMM plus its epilogue, fp32 arithmetic and a bf16 store:
      * U16 * |ref|              the round-to-nearest store of the fp32 result y32 into bf16, |bf16(y32) - y32| <= 2^-8 |y32|;
      * (1 + U16) * gamma_m * S  the fp32 arithmetic before the store (|y32 - ref| <= gamma_m * S, Higham Thm 3.1 / 4.2
                                 with m roundings on every term's path; the factor 1 + U16 is the store rounding of that
                                 error itself).  S = |a| |rs| sum |w| |x| + |b| |T| is the sum of the terms' magnitudes,
                                 m = row degree + the fp32 roundings of the weights / epilogue (NORM_W, FOLD, TELE, ...),
                                 + 256 + work items for a split row (one partial per group of the CTA, G >= 1, then one
                                 per work item in the combine kernel);
      * U16 * rounded            one more bf16 rounding of an intermediate that storage rounds (e.g. the pre-scaled copy
                                 D^-1/2 x the next hop gathers), `rounded` = the magnitude that intermediate enters with."""
    b = U16 * ref.abs() + (1 + U16) * gamma(m).view(-1, 1) * S
    if rounded is not None:
        b = b + U16 * rounded
    return b


def assert_within(y, ref, bnd, what):
    err = (y.detach().double().cpu() - ref).abs()
    bad = err > bnd
    if bool(bad.any()):
        r = (err / bnd.clamp_min(1e-300))[bad]
        raise AssertionError(f"{what}: {int(bad.sum())} of {err.numel()} elements beyond the bound (worst x{float(r.max()):.3g})")


class Op:
    """W in fp64 from the oracle's edited edge list: W[i, j] = sum of the weights of the edges j -> i (all >= 0, so
    |W| = W).  deg / deg_t = products the kernel accumulates per row of the forward / transposed CSR."""

    def __init__(self, ei, n, mode, weight):
        if weight == "gcn":
            ed, w = R.gcn_norm(ei, None, n, add_self_loops=(mode == R.LOOP_ADD_REMAINING), dtype=torch.float64)
        else:
            ed = R.edit_loops(ei, n, mode)
            w = torch.ones(ed.size(1), dtype=torch.float64)
        src, dst = ed[0], ed[1]
        self.n = n
        self.A = torch.sparse_coo_tensor(torch.stack([dst, src]), w, (n, n)).coalesce()
        self.At = torch.sparse_coo_tensor(torch.stack([src, dst]), w, (n, n)).coalesce()
        self.deg = torch.bincount(dst, minlength=n).double()
        self.deg_t = torch.bincount(src, minlength=n).double()

    def __call__(self, x, t=False):
        return torch.sparse.mm(self.At if t else self.A, x)


def m_of(csr, deg, ops):
    """m of bound() per row of `csr` (the GPU CSR the call ran on: its chunking decides which rows were split)."""
    m = deg + ops
    if csr.n_items > 0:
        split = deg > csr.chunk
        m = m + torch.where(split, 256 + torch.ceil(deg / csr.long_chunk), torch.zeros_like(deg))
    return m


_GRAPHS = {}


def setup(case, mode, **kw):
    """(GPU Graph, fp64 unit-weight Op, fp64 gcn Op) of a test case, built once per module."""
    key = (case, mode, tuple(sorted(kw.items())))
    if key not in _GRAPHS:
        ei, n = CASES[case]()
        _GRAPHS[key] = (P().Graph(ei.to(DEV), n, mode, **kw), Op(ei, n, mode, "ones"),
                        Op(ei, n, mode, "gcn") if mode in (R.LOOP_NONE, R.LOOP_ADD_REMAINING) else None, ei, n)
    return _GRAPHS[key]


def feats(n, F, seed, scale=1.0, positive=False):
    """bf16 features.  positive: the K-hop families carry rows of one sign (class scores, label distributions); with
    signs mixed, the terms gathered at a hub cancel and |W| |z| outgrows |W z| hop after hop."""
    x = torch.randn(n, F, generator=torch.Generator().manual_seed(seed)) * scale
    return (x.abs() if positive else x).to(BF)


def cross_dtype(p, csr, x, val=None, tune_word=0, **epkw):
    """(bf16 result, fp32 kernel on x.float() rounded to bf16) for one spmm_raw call; bf16 operands of the epilogue
    (T, acc_in) are passed as float copies to the fp32 call, reset values are fp32 in both."""
    def run(dt):
        kw = {}
        keep = []
        for k, v in epkw.items():
            if k in ("T", "acc_in") and v is not None:
                v, ld = p.ops.as_rows(v.to(dt))
                kw["ldt" if k == "T" else "ld_acc"] = ld
            kw[k] = v
            keep.append(v)
        ep = p.ops.make_epilogue(**kw) if kw else None
        return p.ops.spmm_raw(csr, x.to(dt), val, ep=ep, keep=keep, tune=tune_word)
    return run(BF), run(torch.float32).to(BF)


# ------------------------------------------------------------------------------------------------------------------
# SpMM
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("F", [8, 47, 128])
@pytest.mark.parametrize("weighted", [False, True])
def test_every_launch_shape_bf16(weighted, F):
    """Every instantiated (G, V, U), weighted and unweighted, on `medium` (it has split rows): within the bound,
    bit-identical to the fp32 instantiation rounded to bf16, and unsplit rows identical across shapes."""
    p = P()
    g, op1, opg, _, n = setup("medium", R.LOOP_ADD_REMAINING)
    x = feats(n, F, F)
    op, val, ops = (opg, g.gcn_val(False), NORM_W) if weighted else (op1, None, 0)
    x64 = x.double()
    ref = op(x64)
    bnd = bound(ref, op(x64.abs()), m_of(g.fwd, op.deg, ops))
    short = (g.fwd.degree() <= g.fwd.chunk)
    assert int((~short).sum()) > 0
    xd = x.to(DEV)
    first = None
    for G, V, U in SHAPES:
        yb, yf = cross_dtype(p, g.fwd, xd, val, tune(G, V, U))
        assert yb.dtype == BF
        assert_within(yb, ref, bnd, f"G{G} V{V} U{U}")
        assert torch.equal(yb, yf), (G, V, U)
        if first is None:
            first = yb
        assert torch.equal(yb[short], first[short]), (G, V, U)


@pytest.mark.parametrize("F", [1, 8, 9, 24, 40, 47, 64, 72, 128, 136, 256, 264, 520])
@pytest.mark.parametrize("case", list(CASES) + ["hub/1024", "medium/1024"])
def test_default_shape_across_widths_bf16(case, F):
    """The heuristic launch shape at widths across every choose_shape threshold and the blockIdx.y tiling, on every
    case, and with the large-graph split geometry (chunk 1024, long_chunk 4096).  Unsplit rows do not depend on the
    shape, so they also equal the fp32 run (whose default shape differs) rounded to bf16."""
    p = P()
    name, kw = (case.split("/")[0], dict(chunk=1024, long_chunk=4096)) if "/" in case else (case, {})
    g, _, opg, _, n = setup(name, R.LOOP_ADD_REMAINING, **kw)
    x = feats(n, F, 100 + F)
    y = p.ops.propagate(x.to(DEV), g, "gcn")
    assert y.dtype == BF and y.shape == (n, F)
    x64 = x.double()
    ref = opg(x64)
    assert_within(y, ref, bound(ref, opg(x64.abs()), m_of(g.fwd, opg.deg, NORM_W)), case)
    short = (g.fwd.degree() <= g.fwd.chunk) if g.fwd.n_items > 0 else torch.ones(n, dtype=torch.bool, device=DEV)
    y32 = p.ops.propagate(x.to(DEV).float(), g, "gcn").to(BF)
    assert torch.equal(y[short], y32[short])


def _epilogue_cases(p, g, op1, n, F):
    """name -> (spmm_raw epilogue kwargs, fp64 reference function of the raw row sum s, S, extra roundings)."""
    d = g.dinv()
    d64 = d.double().cpu().view(-1, 1)
    cnt = g.fwd.norm(p.graph.NORM_COUNT)
    c64 = cnt.double().cpu().view(-1, 1)
    T = feats(n, F, 7)
    A = feats(n, F, 8)
    rv = feats(n, F, 9, 0.5)
    mask = torch.zeros(n, dtype=torch.bool)
    mask[::3] = True
    T64, A64, rv64 = T.double(), A.double(), rv.double()
    mk = lambda v, lo=-math.inf, hi=math.inf: v.clamp(lo, hi)  # noqa: E731
    tele = dict(row_scale=d, a=0.9, b=0.1, T=T.to(DEV))
    m8 = mask.to(torch.uint8).to(DEV)
    rvd = rv.float().to(DEV)
    return {
        "mean": (dict(row_scale=cnt, row_div=True), lambda s: s / c64, lambda s: s / c64, 1),
        "row_scale": (dict(row_scale=d), lambda s: d64 * s, lambda s: d64 * s, FOLD // 2),
        "teleport": (tele, lambda s: 0.9 * d64 * s + 0.1 * T64, lambda s: 0.9 * d64 * s + 0.1 * T64.abs(), FOLD // 2 + TELE),
        "clamp": (dict(tele, clamp=(-0.25, 0.25)), lambda s: mk(0.9 * d64 * s + 0.1 * T64, -0.25, 0.25),
                  lambda s: 0.9 * d64 * s + 0.1 * T64.abs(), FOLD // 2 + TELE),
        "reset_before_teleport": (dict(tele, reset_mask=m8, reset_val=rvd, ld_reset=F, reset_when=1),
                                  lambda s: 0.9 * torch.where(mask.view(-1, 1), rv64, d64 * s) + 0.1 * T64,
                                  lambda s: 0.9 * torch.where(mask.view(-1, 1), rv64.abs(), d64 * s) + 0.1 * T64.abs(),
                                  FOLD // 2 + TELE),
        "reset_after_clamp": (dict(tele, clamp=(-0.25, 0.25), reset_mask=m8, reset_val=rvd, ld_reset=F, reset_when=2),
                              lambda s: torch.where(mask.view(-1, 1), rv64, mk(0.9 * d64 * s + 0.1 * T64, -0.25, 0.25)),
                              lambda s: 0.9 * d64 * s + 0.1 * T64.abs(), FOLD // 2 + TELE),
        "acc_in": (dict(acc_in=A.to(DEV), row_scale=d), lambda s: d64 * (A64 + s), lambda s: d64 * (A64.abs() + s),
                   FOLD // 2 + 1),
    }


@pytest.mark.parametrize("F", [47, 264])
def test_epilogues_bf16(F):
    """Every epilogue variant in bf16 on `medium` (split rows go through the combine kernel's epilogue): within the
    bound and bit-identical to the fp32 instantiation rounded to bf16.  Reset rows are passed as fp32 (the header
    contract) in both calls."""
    p = P()
    g, op1, _, _, n = setup("medium", R.LOOP_ADD_REMAINING)
    x = feats(n, F, F + 1)
    x64 = x.double()
    s, sa = op1(x64), op1(x64.abs())
    m_base = m_of(g.fwd, op1.deg, 0)
    for name, (kw, f_ref, f_S, ops) in _epilogue_cases(p, g, op1, n, F).items():
        yb, yf = cross_dtype(p, g.fwd, x.to(DEV), None, tune(*REL), **kw)
        ref = f_ref(s)
        assert_within(yb, ref, bound(ref, f_S(sa), m_base + ops), name)
        assert torch.equal(yb, yf), name
    # gcn weights (per-edge FMA) and the scatter-mean through the public op, default shape
    y = p.ops.propagate(x.to(DEV), g, "mean")
    c64 = g.fwd.norm(p.graph.NORM_COUNT).double().cpu().view(-1, 1)
    assert_within(y, s / c64, bound(s / c64, sa / c64, m_base + 1), "propagate mean")


def test_skip_empty_leaves_rows_without_edges_untouched_bf16():
    p = P()
    g, op1, _, _, n = setup("isolated", R.LOOP_NONE)
    F = 24
    x = feats(n, F, 3)
    empty = (g.fwd.degree() == 0).cpu()
    assert int(empty.sum()) >= 60
    out = torch.full((n, F), 7.0, dtype=BF, device=DEV)
    p.ops.spmm_raw(g.fwd, x.to(DEV), None, ep=p.ops.make_epilogue(skip_empty=True), out=out)
    out = out.cpu()
    assert bool((out[empty] == 7.0).all())
    ref = op1(x.double())
    assert_within(out[~empty], ref[~empty], bound(ref, op1(x.double().abs()), m_of(g.fwd, op1.deg, 0))[~empty], "skip_empty")


@pytest.mark.parametrize("F", [47, 264])
def test_peer_push_bf16_equals_fp32_push_rounded(F):
    """Fused all-gather into three local copies, as 16-byte stores and as bulk copies: every pushed bf16 row is the
    fp32 push of the same call rounded once (the pre-scale multiplies the fp32 value, then the store rounds), and it
    is within the bound of d_i * ref_i."""
    p = P()
    L = p._lib.lib()
    g, op1, _, _, n = setup("medium", R.LOOP_ADD_REMAINING)
    d = g.dinv()
    d64 = d.double().cpu().view(-1, 1)
    x = feats(n, F, 5)
    T = feats(n, F, 6)
    row0, tail = 3, 2

    def push(dt):
        xb, ldx = p.ops.as_rows(x.to(DEV).to(dt))
        tb, ldt = p.ops.as_rows(T.to(DEV).to(dt))
        ld = p.ops.padded_width(F, dt)
        bufs = [torch.full((row0 + n + tail, ld), float("nan"), dtype=dt, device=DEV) for _ in range(3)]
        ep = p.ops.make_epilogue(row_scale=d, a=0.9, b=0.1, T=tb, ldt=ldt, out2_scale=d,
                                 peers=[b.data_ptr() for b in bufs], peer_row0=row0, ld_peer=ld)
        assert p.ops.spmm_raw(g.fwd, xb, None, ep=ep, keep=(xb, tb, d, bufs), store_local=False, tune=tune(*REL)) is None
        torch.cuda.synchronize()
        return [b[row0:row0 + n, :F] for b in bufs]

    s, sa = op1(x.double()), op1(x.double().abs())
    ref = d64 * (0.9 * d64 * s + 0.1 * T.double())
    bnd = bound(ref, d64 * (0.9 * d64 * sa + 0.1 * T.double().abs()), m_of(g.fwd, op1.deg, FOLD + TELE))
    old = L.rgbmp_set_push_bulk(0)
    try:
        for bulk in (0, 1):
            L.rgbmp_set_push_bulk(bulk)
            got, want = push(BF), push(torch.float32)
            for a, b in zip(got, want):
                assert torch.equal(a, b.to(BF)), bulk
                assert_within(a, ref, bnd, f"peer push bulk={bulk}")
    finally:
        L.rgbmp_set_push_bulk(old)


def test_row_scale_kernel_bf16():
    p = P()
    n, F = 3000, 47
    x = feats(n, F, 11)
    sc = torch.rand(n, generator=torch.Generator().manual_seed(12)) + 0.5
    for divide in (False, True):
        y = p.ops.row_scale(x.to(DEV), sc.to(DEV), divide)
        y32 = p.ops.row_scale(x.to(DEV).float(), sc.to(DEV), divide)
        assert torch.equal(y, y32.to(BF))
        s64 = sc.double().view(-1, 1)
        ref = x.double() / s64 if divide else x.double() * s64
        assert_within(y, ref, bound(ref, ref.abs(), torch.ones(n)), f"divide={divide}")


def test_unaligned_views_hot_tag_and_locality_schedule_bf16(monkeypatch):
    """Non-contiguous / not 16-byte aligned bf16 views go through the as_rows copy and give the same bits as the
    contiguous input; a forced hot tag and a forced locality-grouped schedule change no bit either."""
    p = P()
    import rgb_experiment_b200.graph as G_
    ei, n = CASES["medium"]()
    F = 47
    g = p.Graph(ei.to(DEV), n, p.LOOP_ADD_REMAINING)
    val = g.gcn_val(False)
    big = feats(n, 61, 13).to(DEV)
    x = big[:, 3:3 + F]                                    # row stride 61, offset 6 bytes
    assert x.data_ptr() % 16 != 0 and not x.is_contiguous()
    plain = p.ops.spmm_raw(g.fwd, x.contiguous(), val, hot=False)
    assert torch.equal(p.ops.spmm_raw(g.fwd, x, val), plain)
    xt = x.t().contiguous().t()                            # column-major view
    assert xt.stride(1) != 1
    assert torch.equal(p.ops.spmm_raw(g.fwd, xt, val), plain)
    _, _, opg, _, _ = setup("medium", R.LOOP_ADD_REMAINING)
    ref = opg(x.double().cpu())
    assert_within(plain, ref, bound(ref, opg(x.double().cpu().abs()), m_of(g.fwd, opg.deg, NORM_W)), "plain")
    monkeypatch.setattr(G_, "HOT_L2_BYTES", 4096)
    tagged = p.ops.spmm_raw(g.fwd, x, val, hot=True)
    assert len(g.fwd._tagged) == 1
    assert torch.equal(tagged, plain)
    monkeypatch.setattr(G_, "HOT_L2_BYTES", 0)
    monkeypatch.setattr(G_, "CLUSTER", "1")
    gc = p.Graph(ei.to(DEV), n, p.LOOP_ADD_REMAINING)
    assert gc.fwd.clustered
    assert torch.equal(p.ops.spmm_raw(gc.fwd, x, gc.gcn_val(False)), plain)


# ------------------------------------------------------------------------------------------------------------------
# K hops
# ------------------------------------------------------------------------------------------------------------------
def khop_ref(op, csr, x0, K, a, b, T, ops, *, t=False, folded=False, clamp=None, reset=None):
    """fp64 reference of K hops z <- post(a * W z + b * T) and an elementwise error budget E carried next to it:
        E_{k+1} = |a| W E_k + r_{k+1},
    r = bound() of one hop taken at the computed input (|z~_k| <= |ref_k| + E_k), its store term taken at
    |ref_{k+1}| + |a| W E_k; folded hops add the bf16 rounding of the pre-scaled copy they gather (U16 * |a| W |z~_k|,
    also the first hop's row_scale of x0).  Clamp is 1-Lipschitz, and where the whole interval ref +- E lies beyond a
    clamp limit both values clamp to it (error: the fp32 limit, U32 |limit|, and the store).  Reset rows hold the bf16
    reset values exactly."""
    deg = op.deg_t if t else op.deg
    m = m_of(csr, deg, ops)
    ref, E = x0.clone(), torch.zeros_like(x0)
    for _ in range(K):
        new = a * op(ref, t) + (b * T if T is not None else 0.0)
        mag = abs(a) * op(ref.abs() + E, t)
        prop = abs(a) * op(E, t)
        S = mag + (abs(b) * T.abs() if T is not None else 0.0)
        pre = prop + gamma(m).view(-1, 1) * S + (U16 * mag if folded else 0.0)    # |y32 - ref| before clamp and store
        if clamp is not None:
            lo, hi = clamp
            sat = (new - pre >= hi) | (new + pre <= lo)
            new = new.clamp(lo, hi)
            pre = torch.where(sat, U32 * new.abs(), pre)
        E = pre + U16 * (new.abs() + pre)
        if reset is not None:
            mask, rv = reset
            new[mask] = rv[mask]
            E[mask] = 0.0
        ref = new
    return ref, E


def assert_budget(y, ref, E, what, ceiling=CEIL):
    assert_within(y, ref, E, what)
    share = float(E.abs().max() / ref.abs().max())
    assert share <= ceiling, f"{what}: budget {share:.3g} of ||ref|| exceeds {ceiling:.3g}"


@pytest.mark.parametrize("case", ["loops_dups", "hub", "medium"])
@pytest.mark.parametrize("fold", [True, False])
@pytest.mark.parametrize("K", [1, 2, 10])
def test_appnp_bf16(case, fold, K):
    """Every bf16 K-hop runs the K-launch driver (the one-cluster kernel is fp32-only)."""
    p = P()
    g, _, opg, _, n = setup(case, R.LOOP_ADD_REMAINING)
    x = feats(n, 47, K, positive=True)
    z = p.ops.appnp(x.to(DEV), g, K, 0.1, fold)
    assert z.dtype == BF
    x64 = x.double()
    ref, E = khop_ref(opg, g.fwd, x64, K, 0.9, 0.1, x64, (FOLD if fold else NORM_W) + TELE, folded=fold)
    assert_budget(z, ref, E, f"appnp K={K} fold={fold}")
    assert torch.allclose(ref, R.appnp_propagate(x64, CASES[case]()[0], K, 0.1), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("fold", [True, False])
def test_gcn_power_bf16(fold):
    p = P()
    g, _, opg, ei, n = setup("medium", R.LOOP_ADD_REMAINING)
    x = feats(n, 40, 21, positive=True)
    y = p.ops.gcn_power(x.to(DEV), g, 3, fold)
    ref, E = khop_ref(opg, g.fwd, x.double(), 3, 1.0, 0.0, None, FOLD if fold else NORM_W, folded=fold)
    assert_budget(y, ref, E, f"gcn_power fold={fold}")


@pytest.mark.parametrize("fold", [True, False])
@pytest.mark.parametrize("post", ["clamp", "reset"])
def test_label_propagation_bf16(post, fold):
    """reset: the reset rows are distinct bf16 values; they reach the epilogue as fp32 rows (a bf16 buffer read as
    float would run past its end and put garbage in every reset row)."""
    p = P()
    g, _, opg, _, n = setup("medium", R.LOOP_NONE)
    F, K, alpha = 10, 10, 0.8
    x = feats(n, F, 31, 0.5, positive=True)
    rv = feats(n, F, 32, 0.5)
    mask = torch.zeros(n, dtype=torch.bool)
    mask[::4] = True
    x64 = x.double()
    if post == "clamp":
        y = p.ops.label_propagation(g, x.to(DEV), K, alpha, clamp=(-0.3, 0.3), fold=fold)
        ref, E = khop_ref(opg, g.fwd, x64, K, alpha, 1 - alpha, x64, (FOLD if fold else NORM_W) + TELE, folded=fold,
                          clamp=(-0.3, 0.3))
    else:
        y = p.ops.label_propagation(g, x.to(DEV), K, alpha, reset_mask=mask.to(DEV), reset_val=rv.to(DEV), fold=fold)
        ref, E = khop_ref(opg, g.fwd, x64, K, alpha, 1 - alpha, x64, (FOLD if fold else NORM_W) + TELE, folded=fold,
                          reset=(mask, rv.double()))
        assert torch.equal(y.cpu()[mask], rv[mask])
    assert_budget(y, ref, E, f"label_propagation {post} fold={fold}")


@pytest.mark.parametrize("case", ["loops_dups", "medium"])
def test_dagnn_hops_bf16_each_hop_from_the_stored_previous_hop(case):
    """Each stored hop against ONE fp64 hop of the GPU's own stored previous hop: the single-call bound, K times."""
    p = P()
    g, _, opg, _, n = setup(case, R.LOOP_ADD_REMAINING)
    x = feats(n, 9, 41)
    S = p.ops.dagnn_hops(x.to(DEV), g, 4)
    assert S.shape == (n, 5, 9) and S.dtype == BF
    Sh = S.double().cpu()
    assert torch.equal(Sh[:, 0], x.double())
    m = m_of(g.fwd, opg.deg, NORM_W)
    for k in range(1, 5):
        prev = Sh[:, k - 1]
        ref = opg(prev)
        assert_within(Sh[:, k], ref, bound(ref, opg(prev.abs()), m), f"hop {k}")


@pytest.mark.parametrize("alpha", [0.0, 0.1])
@pytest.mark.parametrize("K", [2, 10])
def test_partitioned_appnp_bf16_world_size_1(alpha, K):
    p = P()
    import rgb_experiment_b200.partition as PT
    _, _, opg, ei, n = setup("medium", R.LOOP_ADD_REMAINING)
    F = 24
    blk = PT.LocalBlock(ei.to(DEV), n, p.LOOP_ADD_REMAINING, 0, 1)
    prop = PT.PartitionedAPPNP(blk, F, dtype=BF)
    x = feats(n, F, 51)
    z0 = torch.zeros((blk.R, prop.ld), dtype=BF, device=DEV)
    z0[:n, :F] = x.to(DEV)
    out = prop.run(z0, K, alpha)[:n, :F]
    x64 = x.double()
    ref, E = khop_ref(opg, blk.csr, x64, K, 1 - alpha, alpha, x64 if alpha else None, NORM_W + TELE)
    assert_budget(out, ref, E, f"PartitionedAPPNP alpha={alpha} K={K}")


# ------------------------------------------------------------------------------------------------------------------
# autograd
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,mode", [("sum", R.LOOP_NONE), ("mean", R.LOOP_REMOVE_THEN_ADD), ("gcn", R.LOOP_ADD_REMAINING)])
def test_propagate_backward_bf16(kind, mode):
    """dx = W^T dy on the transposed CSR; mean first divides dy by the count in bf16 (one more rounding)."""
    p = P()
    g, op1, opg, _, n = setup("medium", mode)
    F = 47
    x, dy = feats(n, F, 61), feats(n, F, 62)
    xg = x.to(DEV).requires_grad_(True)
    p.ops.propagate(xg, g, kind).backward(dy.to(DEV))
    assert xg.grad.dtype == BF
    dy64 = dy.double()
    op = opg if kind == "gcn" else op1
    rounded = None
    if kind == "mean":
        c64 = op1.deg.clamp_min(1).view(-1, 1)
        dy64 = dy64 / c64
        rounded = op1(dy64.abs(), t=True)
    ref = op(dy64, t=True)
    ops = {"sum": 0, "mean": 1, "gcn": NORM_W}[kind]
    assert_within(xg.grad, ref, bound(ref, op(dy64.abs(), t=True), m_of(g.bwd, op.deg_t, ops), rounded), kind)


@pytest.mark.parametrize("fold", [True, False])
def test_appnp_backward_bf16(fold):
    p = P()
    g, _, opg, _, n = setup("medium", R.LOOP_ADD_REMAINING)
    F, K = 47, 5
    x, dz = feats(n, F, 71), feats(n, F, 72, positive=True)
    xg = x.to(DEV).requires_grad_(True)
    p.ops.appnp(xg, g, K, 0.1, fold).backward(dz.to(DEV))
    dz64 = dz.double()
    ref, E = khop_ref(opg, g.bwd, dz64, K, 0.9, 0.1, dz64, (FOLD if fold else NORM_W) + TELE, t=True, folded=fold)
    assert_budget(xg.grad, ref, E, f"appnp backward fold={fold}")


# ------------------------------------------------------------------------------------------------------------------
# Correct and Smooth in bf16 against the oracle layer
# ------------------------------------------------------------------------------------------------------------------
RB = U16 + 2 * U32     # one elementwise bf16 torch op: computed in fp32 (2^-24), then rounded to bf16 (2^-8)
CS_CEIL = CEIL         # 50 hops at alpha 0.8: the budget settles near r / (1 - 0.8), five hops' roundings, not 50


def _cs_data(case):
    ei, n = CASES[case]()
    ei = R.to_undirected(ei, n)
    C = 5
    gen = torch.Generator().manual_seed(3)
    y_soft = torch.softmax(torch.randn(n, C, generator=gen), -1).to(BF)
    y = torch.randint(C, (n,), generator=gen)
    mask = torch.rand(n, generator=gen) < 0.4
    return ei, n, C, y_soft, y, mask


@pytest.mark.parametrize("case", ["loops_dups", "hub"])
@pytest.mark.parametrize("autoscale", [True, False])
def test_correct_and_smooth_bf16(case, autoscale):
    """correct: the error rows y_true - y_soft are formed in bf16 (one rounding: an input perturbation of U16 |e| on
    the masked rows, which autoscale=False also resets to), propagated 50 hops (budget as khop_ref), then combined with
    y_soft by bf16 torch ops, one rounding each.  smooth: exact inputs, 50 clamped hops."""
    p = P()
    from rgb_experiment_b200.shim import nn as PL
    from oracle import layers as OL
    ei, n, C, y_soft, y, mask = _cs_data(case)
    L_, alpha, scale = 50, 0.8, 0.7
    kw = dict(num_correction_layers=L_, correction_alpha=alpha, num_smoothing_layers=L_, smoothing_alpha=alpha,
              autoscale=autoscale, scale=scale)
    o, gl = OL.CorrectAndSmooth(**kw), PL.CorrectAndSmooth(**kw)
    ys64 = y_soft.double()
    c_o = o.correct(ys64.clone(), y[mask], mask, ei)
    c_g = gl.correct(y_soft.to(DEV), y[mask].to(DEV), mask.to(DEV), ei.to(DEV))
    assert c_g.dtype == BF
    g = p.graph.get_graph(ei.to(DEV), n, p.LOOP_NONE)
    op = Op(ei, n, R.LOOP_NONE, "gcn")
    err0 = torch.zeros_like(ys64)
    err0[mask] = torch.nn.functional.one_hot(y[mask], C).double() - ys64[mask]
    e_in = RB * err0.abs()                             # the error rows y_true - y_soft formed by one bf16 torch op
    # K-hop budget from a perturbed start: E_0 = e_in, and the reset rows (autoscale=False) hold the rounded errors
    m = m_of(g.fwd, op.deg, FOLD + TELE)
    ref, E = err0.clone(), e_in.clone()
    for _ in range(L_):
        new = alpha * op(ref) + (1 - alpha) * err0
        if autoscale:
            new = new.clamp(-1.0, 1.0)
        mag = alpha * op(ref.abs() + E)
        prop = alpha * op(E) + (1 - alpha) * e_in      # the teleport term reads the rounded error rows too
        E = prop + bound(new.abs() + prop, mag + (1 - alpha) * (err0.abs() + e_in), m, mag)
        if not autoscale:
            new[mask] = err0[mask]
            E[mask] = e_in[mask]
        ref = new
    assert float(E.max() / ref.abs().max()) <= CS_CEIL
    if autoscale:
        # scale_i = sigma / sum_c |sm_ic|: sigma from the rounded error rows (fp32 sum, bf16 result, bf16 division), the
        # row sum of the smoothed matrix within sum_c E_ic, its fp32 additions and its bf16 result, then a bf16 division
        numel = int(mask.sum())
        sig = err0[mask].abs().sum() / numel
        sig_e = sig * ((1 + U16) * (1 + RB) ** 2 * (1 + float(gamma(torch.tensor(float(err0[mask].numel()))))) - 1)
        rs, rE = ref.abs().sum(1, keepdim=True), E.sum(1, keepdim=True)
        rs_e = rE + float(gamma(torch.tensor(float(C)))) * (rs + rE)
        rs_e = rs_e + RB * (rs + rs_e)
        assert bool((rs - rs_e > 0).all()), "a row sum of the smoothed matrix is not bounded away from 0"
        sc = sig / rs
        lo, hi = (sig - sig_e) / (rs + rs_e) * (1 - RB), (sig + sig_e) / (rs - rs_e) * (1 + RB)
        assert bool((hi <= 1000).all())
        t_ref = sc * ref
        t_e = sc * E + torch.maximum(hi - sc, sc - lo) * (ref.abs() + E)
    else:
        t_ref = scale * ref
        t_e = scale * E + U32 * (t_ref.abs() + scale * E)     # 0.7 enters the bf16 product as the float 0.7f
    t_e = t_e + RB * (t_ref.abs() + t_e)               # the bf16 product
    want = ys64 + t_ref
    assert torch.allclose(want, c_o, rtol=1e-12, atol=1e-12)
    assert_within(c_g, c_o, t_e + RB * (want.abs() + t_e), f"correct autoscale={autoscale}")
    # smooth: exact one-hot / bf16 inputs, clamp (0, 1)
    c_in = c_o.to(BF)
    s_o = o.smooth(c_in.double(), y[mask], mask, ei)
    s_g = gl.smooth(c_in.to(DEV), y[mask].to(DEV), mask.to(DEV), ei.to(DEV))
    y0 = c_in.double().clone()
    y0[mask] = torch.nn.functional.one_hot(y[mask], C).double()
    ref, E = khop_ref(op, g.fwd, y0, L_, alpha, 1 - alpha, y0, FOLD + TELE, folded=True, clamp=(0.0, 1.0))
    assert torch.allclose(ref, s_o, rtol=1e-12, atol=1e-12)
    assert_budget(s_g, s_o, E, "smooth", CS_CEIL)


# ------------------------------------------------------------------------------------------------------------------
# dtype contract: correct, or RuntimeError before any launch -- never a misread
# ------------------------------------------------------------------------------------------------------------------
def _contract_calls(p, g, gr, gn, n):
    """name -> callable(dtype): the op on fixed inputs converted to that dtype."""
    H, Cc = 2, 8
    gen = torch.Generator().manual_seed(91)

    def a(*shape):
        return torch.randn(*shape, generator=gen)
    A2, a1, a2, X, Xr = a(n, H * Cc), a(n, H), a(n, H), a(n, 8), a(n, 8)
    ew, mw, eg = a(g.nnz).abs(), a(g.nnz, 4), a(gn.nnz, H)
    on = lambda t, dt: t.to(DEV, dt)  # noqa: E731
    every = torch.ones(n, dtype=torch.bool, device=DEV)
    return {
        "gat": lambda dt: p.ops.gat(on(A2, dt), on(a1, dt), on(a2, dt), gr, H, Cc),
        "supergat_mx": lambda dt: p.ops.supergat_mx(on(A2, dt), on(a1, dt), on(a2, dt), gr, H, Cc),
        "faconv": lambda dt: p.ops.faconv(on(A2[:, :Cc], dt), on(a1[:, :1], dt), on(a2[:, :1], dt), g),
        "edge_sddmm": lambda dt: p.ops.edge_sddmm(on(A2, dt), on(A2, dt), gn, H, Cc),
        "edge_u_add_v": lambda dt: p.ops.edge_u_add_v(on(a1, dt), on(a2, dt), gn),
        "edge_softmax": lambda dt: p.ops.edge_softmax(on(eg, dt), gn),
        "spmm_heads": lambda dt: p.ops.spmm_heads(on(eg, dt), on(A2, dt), gn, H, Cc),
        "to_edge_order": lambda dt: g.to_edge_order(on(ew, dt)),
        "propagate_weighted_backward": lambda dt: _weighted_backward(p, g, on(X, dt), on(ew, dt)),
        "segment_reduce": lambda dt: p.ops.segment_reduce(on(mw, dt), g),
        "row_scale": lambda dt: p.ops.row_scale(on(X, dt), g.dinv()),
        "propagate": lambda dt: p.ops.propagate(on(X, dt), g, "gcn"),
        "appnp": lambda dt: p.ops.appnp(on(X, dt), g, 3, 0.1),
        "gcn_power": lambda dt: p.ops.gcn_power(on(X, dt), g, 2),
        "dagnn_hops": lambda dt: p.ops.dagnn_hops(on(X, dt), g, 2),
        "label_propagation_reset": lambda dt: p.ops.label_propagation(gn, on(X, dt), 3, 0.8, reset_mask=every,
                                                                      reset_val=on(Xr, dt)),
        "pta_inference": lambda dt: p.ops.pta_inference(on(X, dt), g, 3, 0.1),
    }


def _weighted_backward(p, g, x, w):
    x.requires_grad_(True)
    w.requires_grad_(True)
    p.ops.propagate_weighted(x, w, g).sum().backward()
    return x.grad, w.grad


ATTENTION = {"gat", "supergat_mx", "faconv", "edge_sddmm", "edge_u_add_v", "edge_softmax", "spmm_heads", "to_edge_order"}


def test_dtype_contract_correct_or_runtime_error_never_a_misread():
    """Under guard bands (test_gpu_guard_bands.GuardedAllocator): the fp32-only attention / edge-score kernels refuse
    bf16, fp16 and fp64; the SpMM / K-hop ops take bf16 (checked against fp64 in the tests above, here against the
    fp32 kernels on the same values) and refuse fp16 and fp64; the bf16 weight gradient of propagate_weighted is
    computed from fp32 copies.  Then every shim layer in bf16 / fp16 / fp64: correct (within 2^-5 of the same layer
    in fp32, far from the O(1) error of a misread) or RuntimeError."""
    from test_gpu_guard_bands import GuardedAllocator
    p = P()
    from rgb_experiment_b200.shim import nn as PL
    p.graph.clear_cache()
    p.memo.clear()
    ei, n = CASES["hub"]()
    eid = ei.to(DEV)
    ga = GuardedAllocator()
    ga.install()
    try:
        g = p.Graph(eid, n, p.LOOP_ADD_REMAINING)
        gr = p.Graph(eid, n, p.LOOP_REMOVE_THEN_ADD)
        gn = p.Graph(eid, n, p.LOOP_NONE)
        calls = _contract_calls(p, g, gr, gn, n)
        for name, fn in calls.items():
            for dt in (BF, torch.float16, torch.float64):
                if name in ATTENTION or dt != BF:
                    with pytest.raises(RuntimeError):
                        fn(dt)
                    continue
                got = fn(dt)
                want = fn(torch.float32)
                for a, b in zip(got if isinstance(got, tuple) else (got,), want if isinstance(want, tuple) else (want,)):
                    assert torch.isfinite(a.float()).all(), name
                    err = float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))
                    assert err <= 2.0 ** -5, (name, err)
        torch.cuda.synchronize()
        x = torch.randn(n, 16, generator=torch.Generator().manual_seed(92))
        layers = {
            "GCNConv": lambda: PL.GCNConv(16, 8), "SAGEConv": lambda: PL.SAGEConv(16, 8), "GATConv": lambda: PL.GATConv(16, 8, heads=2),
            "SuperGATConv": lambda: PL.SuperGATConv(16, 8, heads=2), "APPNP": lambda: PL.APPNP(3, 0.1),
            "SGConv": lambda: PL.SGConv(16, 8, K=2), "FAConv": lambda: PL.FAConv(16), "GINConv": lambda: PL.GINConv(torch.nn.Identity()),
            "GatedGraphConv": lambda: PL.GatedGraphConv(16, 2),
        }
        for name, mk in layers.items():
            torch.manual_seed(0)
            ref_layer = mk().to(DEV).eval()
            args = lambda dt: (x.to(DEV, dt), x.to(DEV, dt), eid) if name == "FAConv" else (x.to(DEV, dt), eid)  # noqa: E731
            with torch.no_grad():
                want = ref_layer(*args(torch.float32))
                for dt in (BF, torch.float16, torch.float64):
                    layer = mk().to(DEV).eval()
                    layer.load_state_dict(ref_layer.state_dict())
                    layer = layer.to(dt)
                    try:
                        got = layer(*args(dt))
                    except RuntimeError:
                        continue
                    assert dt == BF and name not in ("GATConv", "SuperGATConv", "FAConv"), (name, dt)
                    err = float((got.double() - want.double()).abs().max() / want.double().abs().max())
                    assert err <= 2.0 ** -5, (name, dt, err)
        torch.cuda.synchronize()
    finally:
        ga.uninstall()
        p.graph.clear_cache()
        p.memo.clear()
    assert len(ga.records) > 50
    assert ga.violations() == 0
