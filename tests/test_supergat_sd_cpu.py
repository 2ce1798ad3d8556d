"""SuperGATConv's SD attention without a GPU: a dense fp64 statement of the paper's equation agrees with the oracle
layer; RGBMP_ATT_SD has the shape rules of MX; the SD entry points reject bad arguments with RGBMP_EINVAL before
touching a device, and the generic attention entry points keep refusing score 3.

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


def _fwd(g=None, X=FAKE, H=8, Cc=8, drop=None, d=None, out=FAKE, rowmax=FAKE, rowsum=FAKE, ws=FAKE, scale=0.35):
    g = _graph() if g is None else g
    return L().rgbmp_att_sd_forward(C.byref(g) if g is not False else None, X, 64, H, Cc, scale, 0.2, drop,
                                    None if d is None else C.byref(d), out, 64, rowmax, rowsum, ws, 1 << 30, 0, None)


def _bwd(g=None, gT=None, X=FAKE, H=8, Cc=8, drop=None, tpos=None, d=None, out=FAKE, dout=FAKE, dX=FAKE, dXf=FAKE,
         ws=FAKE, scale=0.35):
    g = _graph() if g is None else g
    gT = _graph() if gT is None else gT
    return L().rgbmp_att_sd_backward(C.byref(g), C.byref(gT) if gT is not False else None, X, 64, H, Cc, scale, 0.2,
                                     drop, tpos, None if d is None else C.byref(d), FAKE, FAKE, out, 64, dout, 64,
                                     dX, 64, dXf, 64, ws, 1 << 30, 0, None)


def _einval(rc, fn):
    from rgb_experiment_b200._lib import EINVAL
    assert rc == EINVAL
    assert fn.encode() in L().rgbmp_last_error()


def test_sd_forward_argument_errors():
    fn = "rgbmp_att_sd_forward"
    _einval(_fwd(g=False), fn)
    for kw in ({"X": None}, {"out": None}, {"rowmax": None}, {"rowsum": None}, {"ws": None}):
        _einval(_fwd(**kw), fn)
    _einval(_fwd(drop=FAKE, d=_drop()), fn)                 # both dropout forms
    for H, Cc in ((8, 12), (2, 130), (1, 129), (3, 7), (0, 8)):
        _einval(_fwd(H=H, Cc=Cc), fn)
    _einval(_fwd(d=_drop(eid=None)), fn)
    _einval(_fwd(d=_drop(seed=None)), fn)
    _einval(_fwd(g=_graph(square=False)), fn)
    _einval(_fwd(scale=float("nan")), fn)


def test_sd_backward_argument_errors():
    fn = "rgbmp_att_sd_backward"
    _einval(_bwd(gT=False), fn)
    for kw in ({"X": None}, {"out": None}, {"dout": None}, {"dX": None}, {"dXf": None}, {"ws": None},
               {"drop": FAKE}):                            # an explicit mask needs tpos
        _einval(_bwd(**kw), fn)
    _einval(_bwd(drop=FAKE, tpos=FAKE, d=_drop()), fn)
    for H, Cc in ((8, 12), (2, 130), (1, 129), (3, 7)):
        _einval(_bwd(H=H, Cc=Cc), fn)
    _einval(_bwd(d=_drop(eid_t=None)), fn)
    _einval(_bwd(d=_drop(eid=None)), fn)
    _einval(_bwd(gT=_graph(n=5)), fn)                       # not the transpose of g


def test_generic_entry_points_still_refuse_score_3():
    from rgb_experiment_b200._lib import ERANGE
    lib = L()
    g = _graph()
    rc = lib.rgbmp_att_forward(C.byref(g), 3, FAKE, 64, FAKE, FAKE, None, 8, 8, 0.2, None, FAKE, 64, FAKE, FAKE, None,
                               0, None, FAKE, 1 << 30, 0, None)
    assert rc == ERANGE and b"unsupported score 3" in lib.rgbmp_last_error()
    rc = lib.rgbmp_att_backward(C.byref(g), C.byref(g), 3, FAKE, 64, FAKE, FAKE, None, 8, 8, 0.2, None, None, FAKE,
                                FAKE, None, FAKE, 64, None, 0, FAKE, 64, FAKE, 64, FAKE, 64, FAKE, FAKE, FAKE, 1 << 30,
                                0, None)
    assert rc == ERANGE and b"unsupported score 3" in lib.rgbmp_last_error()
