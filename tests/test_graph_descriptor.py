"""Every entry point that takes an rgbmp_graph_t checks it against the same rules (include/rgbmp.h, next to the
struct), before it selects a device: a descriptor and its rowptr exist, n_cols fits int32, the long-row lists are
complete whenever n_items > 0, and hot-tagged column ids (bit 31 set by rgbmp_col_tag) reach only the SpMM entry
points, whose kernels strip the tag.  Any other kernel would gather X + col * ld with the tag still set.

Runs without a GPU: the addresses are fake and every call also carries one bad argument that the entry point
refuses right after the graph checks, so no call reaches a device.  For a good descriptor that argument is what
the error names, which is how the tagged SpMM calls show that they got past the graph checks.
"""
import ctypes as C

import pytest

FAKE = 1 << 20
N = 4


def L():
    import rgb_experiment_b200 as R
    return R._lib.lib()


def graph(**kw):
    from rgb_experiment_b200._lib import GraphStruct
    g = GraphStruct(N, N, 6, FAKE, FAKE, 0, 0, 0, 0, None, None, None, None, None, 0)
    for k, v in kw.items():
        setattr(g, k, v)
    return g


def sample():
    from rgb_experiment_b200._lib import SgatSampleStruct
    return SgatSampleStruct(FAKE, FAKE, FAKE, 1 << 31)


def _ref(g):
    return None if g is None else C.byref(g)


# entry point -> (graph arguments, call(graphs) with one bad non-graph argument, what that argument's error says)
def _spmm(g):
    return L().rgbmp_spmm(_ref(g["g"]), None, FAKE, 64, FAKE, 64, 16, 7, None, 0, FAKE, 1 << 20, 0, None)


def _khop(g):
    return L().rgbmp_khop(_ref(g["g"]), None, FAKE, 64, FAKE, FAKE, 64, FAKE, 64, None, 0, 0, 16, 7, 2, None, 0, FAKE,
                          1 << 20, 0, None)


def _appnp_host(g):
    return L().rgbmp_appnp_host(_ref(g["g"]), FAKE, FAKE, FAKE, 0, 2, 0.1, FAKE, FAKE, FAKE, FAKE, 64, FAKE, 1 << 20, 0,
                                None)


def _att_forward(g):
    return L().rgbmp_att_forward(_ref(g["g"]), 4, FAKE, 64, FAKE, FAKE, None, 8, 8, 0.2, 0.0, None, None, FAKE, 64,
                                 FAKE, FAKE, None, 64, None, FAKE, 1 << 30, 0, None)


def _att_backward(g):
    return L().rgbmp_att_backward(_ref(g["g"]), _ref(g["gT"]), 4, FAKE, 64, FAKE, FAKE, None, 8, 8, 0.2, 0.0, None, None,
                                  None, FAKE, FAKE, FAKE, FAKE, 64, FAKE, 64, FAKE, 64, FAKE, 64, None, 64, FAKE, FAKE,
                                  FAKE, 1 << 30, 0, None)


def _sgat_loss_forward(g):
    s = sample()
    return L().rgbmp_sgat_loss_forward(_ref(g["g"]), _ref(g["gneg"]), C.byref(s), FAKE, 64, 0, 1.0, FAKE, FAKE, FAKE,
                                       1 << 20, 0, None)


def _sgat_loss_backward(g):
    s = sample()
    return L().rgbmp_sgat_loss_backward(_ref(g["g"]), _ref(g["gT"]), _ref(g["gneg"]), _ref(g["gnegT"]), C.byref(s), FAKE,
                                        64, 0, 1.0, FAKE, FAKE, FAKE, 64, 0, None)


def _cluster_lpa(g):
    taus = (C.c_float * 1)(0.5)
    return L().rgbmp_cluster_lpa(_ref(g["g"]), FAKE, 2, 0, taus, FAKE, FAKE, 1 << 20, 0, None)


ENTRY = {
    "spmm": (("g",), _spmm, b"bad dtype"),
    "khop": (("g",), _khop, b"bad dtype"),
    "appnp_host": (("g",), _appnp_host, b"bad argument"),
    "att_forward": (("g",), _att_forward, b"unsupported score"),
    "att_backward": (("g", "gT"), _att_backward, b"unsupported score"),
    "sddmm": (("g",), lambda g: L().rgbmp_sddmm(_ref(g["g"]), FAKE, 64, FAKE, 64, 0, 8, FAKE, 0, None), b"bad argument"),
    "u_add_v": (("g",), lambda g: L().rgbmp_u_add_v(_ref(g["g"]), FAKE, FAKE, 0, FAKE, 0, None), b"bad argument"),
    "seg_softmax": (("g",), lambda g: L().rgbmp_seg_softmax(_ref(g["g"]), FAKE, 0, FAKE, 0, None), b"bad argument"),
    "seg_softmax_backward": (("g",), lambda g: L().rgbmp_seg_softmax_backward(_ref(g["g"]), FAKE, FAKE, 0, FAKE, 0, None),
                             b"bad argument"),
    "seg_sum": (("g",), lambda g: L().rgbmp_seg_sum(_ref(g["g"]), FAKE, 0, FAKE, 0, None), b"bad argument"),
    "spmm_heads": (("g",), lambda g: L().rgbmp_spmm_heads(_ref(g["g"]), FAKE, FAKE, 64, 0, 8, FAKE, 64, 0, None),
                   b"bad argument"),
    "sgat_loss_forward": (("g", "gneg"), _sgat_loss_forward, b"F = 0 outside"),
    "sgat_loss_backward": (("g", "gT", "gneg", "gnegT"), _sgat_loss_backward, b"F = 0 outside"),
    "cluster_lpa": (("g",), _cluster_lpa, b"bad argument"),
    "cluster_connectivity": (("g",), lambda g: L().rgbmp_cluster_connectivity(_ref(g["g"]), FAKE, 2, 0, FAKE, 0, None),
                             b"bad argument"),
}
TAGS_OK = {"spmm", "khop", "appnp_host"}     # their kernels strip bit 31 before they gather
PARAMS = [(name, arg) for name, (args, _, _) in ENTRY.items() for arg in args]


def _call(name, arg, bad):
    """Call `name` with every graph argument good except `arg`, which is `bad`; return (rc, error text)."""
    args, call, _ = ENTRY[name]
    graphs = {a: graph() for a in args}
    graphs[arg] = bad
    rc = call(graphs)
    err = L().rgbmp_last_error()
    assert f"rgbmp_{name}".encode() in err and b"bad device" not in err, err
    return rc, err


def _refused(name, arg, bad, code, msg):
    rc, err = _call(name, arg, bad)
    assert rc == code and msg in err, (rc, err)


@pytest.mark.parametrize("name,arg", PARAMS)
def test_good_descriptor_passes_the_graph_checks(name, arg):
    rc, err = _call(name, arg, graph())
    assert rc != 0 and ENTRY[name][2] in err, err


@pytest.mark.parametrize("name,arg", PARAMS)
def test_null_descriptor_or_rowptr(name, arg):
    from rgb_experiment_b200._lib import EINVAL
    _refused(name, arg, None, EINVAL, b"bad graph descriptor")
    _refused(name, arg, graph(rowptr=None), EINVAL, b"bad graph descriptor")


@pytest.mark.parametrize("name,arg", PARAMS)
def test_n_cols_must_fit_int32(name, arg):
    from rgb_experiment_b200._lib import ERANGE
    _refused(name, arg, graph(n_cols=1 << 31), ERANGE, b"n_cols exceeds int32")


@pytest.mark.parametrize("name,arg", PARAMS)
def test_incomplete_long_row_lists(name, arg):
    from rgb_experiment_b200._lib import EINVAL
    _refused(name, arg, graph(chunk=32, long_chunk=256, n_long=1, n_items=3), EINVAL, b"incomplete long-row lists")
    lists = dict(long_rows=FAKE, long_item_ptr=FAKE, item_long=FAKE, item_start=FAKE)
    _refused(name, arg, graph(long_chunk=256, n_long=1, n_items=3, **lists), EINVAL, b"incomplete long-row lists")


@pytest.mark.parametrize("name,arg", PARAMS)
def test_hot_tags_only_where_the_kernels_strip_them(name, arg):
    from rgb_experiment_b200._lib import EINVAL
    if name in TAGS_OK:
        rc, err = _call(name, arg, graph(col_tagged=1))
        assert rc != 0 and ENTRY[name][2] in err, err
    else:
        _refused(name, arg, graph(col_tagged=1), EINVAL, b"hot-tagged column ids")
