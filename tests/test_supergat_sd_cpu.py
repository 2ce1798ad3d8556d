"""SuperGATConv's SD attention without a GPU: a dense fp64 statement of the paper's equation agrees with the oracle
layer; RGBMP_ATT_SD has the shape rules of MX; the attention entry points reject bad SD arguments before touching a
device, and refuse unknown scores and bad dropout arguments for every score.

  SuperGAT  Kim & Oh 2021, eq. 3 (SD)   e_ij = (Wh_i . Wh_j) / sqrt(C),  alpha = softmax_j(leaky_relu(e_ij))
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from helpers import CASES
from oracle import layers as OL
from test_oracle_dense_forms import counts, leaky, masked_softmax_rows


@pytest.mark.parametrize("case", ["tiny", "loops_dups", "isolated", "hub"])
@pytest.mark.parametrize("H,Cc,concat", [(2, 3, True), (3, 5, False), (1, 7, True)])
def test_sd_dense_equals_oracle_layer(case, H, Cc, concat):
    ei, n = CASES[case]()
    torch.manual_seed(H * 10 + Cc)
    layer = OL.SuperGATConv(6, Cc, heads=H, concat=concat, attention_type="SD").double().eval()
    with torch.no_grad():
        layer.bias.normal_()
    rng = np.random.default_rng(5)
    X = rng.standard_normal((n, 6))
    with torch.no_grad():
        got = layer(torch.from_numpy(X), ei).numpy()
    W = layer.lin.weight.detach().numpy()                   # [H*C, 6]
    Xp = (X @ W.T).reshape(n, H, Cc)
    M = counts(ei, n, drop_loops=True, add_loop="all")     # loops removed, one loop per node added
    out = np.zeros((n, H, Cc))
    for h in range(H):
        x = Xp[:, h, :]
        E = leaky((x @ x.T) / math.sqrt(Cc))                # E[i, j]: target i, source j (symmetric)
        out[:, h, :] = masked_softmax_rows(E, M) @ x
    want = (out.reshape(n, H * Cc) if concat else out.mean(axis=1)) + layer.bias.detach().numpy()
    assert np.allclose(got, want, rtol=0, atol=1e-12)


def L():
    import rgb_experiment_b200 as R
    return R._lib.lib()


def test_sd_supported_shapes_are_mx_shapes():
    lib = L()
    for H in (1, 2, 3, 5, 8, 16, 64):
        for Cc in (1, 4, 7, 8, 10, 16, 32, 41, 47, 64, 100, 128, 129, 130, 256):
            assert lib.rgbmp_att_supported(3, H, Cc) == lib.rgbmp_att_supported(1, H, Cc), (H, Cc)
    assert lib.rgbmp_att_supported(3, 8, 8) == 1 and lib.rgbmp_att_supported(3, 1, 130) == 0
    assert lib.rgbmp_att_supported(4, 8, 8) == 0


# fake device addresses: every rejection below happens before anything is dereferenced or a device is selected
FAKE = 1 << 20


def _graph(n=4, nnz=6, square=True):
    from rgb_experiment_b200._lib import GraphStruct
    return GraphStruct(n, n if square else n + 1, nnz, FAKE, FAKE, 0, 0, 0, 0, None, None, None, None, None, 0)


def _drop(seed=FAKE, eid=FAKE, eid_t=FAKE):
    from rgb_experiment_b200._lib import DropoutStruct
    return DropoutStruct(seed, eid, eid_t, 1 << 31, 2.0)


def _fwd(g=None, X=FAKE, H=8, Cc=8, drop=None, d=None, out=FAKE, rowmax=FAKE, rowsum=FAKE, ws=FAKE, scale=0.35,
         score=3, a=None, dinv=None, out2=None, rowq=None):
    g = _graph() if g is None else g
    return L().rgbmp_att_forward(C.byref(g) if g is not False else None, score, X, 64, a, a, dinv, H, Cc, 0.2, scale,
                                 drop, None if d is None else C.byref(d), out, 64, rowmax, rowsum, out2, 64, rowq, ws,
                                 1 << 30, 0, None)


def _bwd(g=None, gT=None, X=FAKE, H=8, Cc=8, drop=None, tpos=None, d=None, out=FAKE, dout=FAKE, dX=FAKE, dXf=FAKE,
         ws=FAKE, scale=0.35, score=3, a=None, dinv=None, out2=None, rowq=None):
    g = _graph() if g is None else g
    gT = _graph() if gT is None else gT
    return L().rgbmp_att_backward(C.byref(g), C.byref(gT) if gT is not False else None, score, X, 64, a, a, dinv, H, Cc,
                                  0.2, scale, drop, tpos, None if d is None else C.byref(d), FAKE, FAKE, rowq, out, 64,
                                  out2, 64, dout, 64, dX, 64, dXf, 64, a, a, ws, 1 << 30, 0, None)


def _rc(rc, code, fn, msg=b""):
    assert rc == code
    err = L().rgbmp_last_error()
    assert fn.encode() in err and msg in err and b"bad device" not in err, err


def _einval(rc, fn, msg=b""):
    from rgb_experiment_b200._lib import EINVAL
    _rc(rc, EINVAL, fn, msg)


def _erange(rc, fn):
    from rgb_experiment_b200._lib import ERANGE
    _rc(rc, ERANGE, fn, b"unsupported score")


def test_att_forward_sd_argument_errors():
    fn = "rgbmp_att_forward"
    _einval(_fwd(g=False), fn)
    for kw in ({"X": None}, {"out": None}, {"rowmax": None}, {"rowsum": None}, {"ws": None}):
        _einval(_fwd(**kw), fn)
    _einval(_fwd(drop=FAKE, d=_drop()), fn)                 # both dropout forms
    for H, Cc in ((8, 12), (2, 130), (1, 129), (3, 7), (0, 8)):
        _erange(_fwd(H=H, Cc=Cc), fn)
    _einval(_fwd(d=_drop(eid=None)), fn)
    _einval(_fwd(d=_drop(seed=None)), fn)
    _einval(_fwd(g=_graph(square=False)), fn)
    _einval(_fwd(scale=float("nan")), fn)
    _einval(_fwd(out2=FAKE, rowq=FAKE), fn)                # SD has no second aggregate


def test_att_backward_sd_argument_errors():
    fn = "rgbmp_att_backward"
    _einval(_bwd(gT=False), fn)
    for kw in ({"X": None}, {"out": None}, {"dout": None}, {"dX": None}, {"dXf": None}, {"ws": None},
               {"drop": FAKE}):                            # an explicit mask needs tpos
        _einval(_bwd(**kw), fn)
    _einval(_bwd(drop=FAKE, tpos=FAKE, d=_drop()), fn)
    for H, Cc in ((8, 12), (2, 130), (1, 129), (3, 7)):
        _erange(_bwd(H=H, Cc=Cc), fn)
    _einval(_bwd(d=_drop(eid_t=None)), fn)
    _einval(_bwd(d=_drop(eid=None)), fn)
    _einval(_bwd(gT=_graph(n=5)), fn)                       # not the transpose of g
    _einval(_bwd(scale=float("inf")), fn)


# every argument the score reads, so that only the one under test is wrong: GAT / MX / FA read a_nbr, a_own;
# FA is single-head and reads dinv; the GAT / FA backward reads the training-mode forward's out2 (GAT also rowq)
SCORES = {0: dict(H=8, a=FAKE, out2=FAKE, rowq=FAKE), 1: dict(H=8, a=FAKE),
          2: dict(H=1, a=FAKE, dinv=FAKE, out2=FAKE)}


def test_unknown_scores_are_out_of_range():
    for score in (-1, 4):
        _erange(_fwd(score=score, a=FAKE), "rgbmp_att_forward")
        _erange(_bwd(score=score, a=FAKE), "rgbmp_att_backward")


@pytest.mark.parametrize("score", sorted(SCORES))
def test_gat_mx_fa_dropout_argument_errors(score):
    kw = SCORES[score]
    fwd_kw = {k: v for k, v in kw.items() if k not in ("out2", "rowq")}   # inference forward
    fn, both, seed_eid = "rgbmp_att_forward", b"at most one of drop / d", b"dropout needs seed"
    _einval(_fwd(score=score, drop=FAKE, d=_drop(), **fwd_kw), fn, both)
    _einval(_fwd(score=score, d=_drop(seed=None), **fwd_kw), fn, seed_eid)
    _einval(_fwd(score=score, d=_drop(eid=None), **fwd_kw), fn, seed_eid)
    fn = "rgbmp_att_backward"
    _einval(_bwd(score=score, drop=FAKE, tpos=FAKE, d=_drop(), **kw), fn, both)
    _einval(_bwd(score=score, d=_drop(seed=None), **kw), fn, seed_eid)
    _einval(_bwd(score=score, d=_drop(eid_t=None), **kw), fn, seed_eid)
    if score == 1:                                          # MX also runs a pass on the forward CSR
        _einval(_bwd(score=score, d=_drop(eid=None), **kw), fn, seed_eid)
