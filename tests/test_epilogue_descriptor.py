"""rgbmp_spmm and rgbmp_khop check an rgbmp_epilogue_t against the same rules (include/rgbmp.h, next to the struct),
once per call and before they select a device: reset rows come with their mask, values and a leading dimension of at
least F, as does every other row operand that is given; peers are at most RGBMP_MAX_PEERS non-NULL, 16-byte aligned
buffers; row_map does not combine with peers, acc_in or reset rows.  rgbmp_khop stores every hop itself, so it also
refuses Y2, acc_in, skip_empty and peers, and row_map together with `hops`.

Runs without a GPU: the addresses are fake and every call names the invalid device 1 << 20.  A call that passes the
checks therefore stops at `bad device`; one that breaks a rule never gets that far.
"""
import ctypes as C

import pytest

FAKE = 1 << 20
BAD_DEVICE = 1 << 20
N = 4
F = 16


def L():
    import rgb_experiment_b200 as R
    return R._lib.lib()


def graph():
    from rgb_experiment_b200._lib import GraphStruct
    return GraphStruct(N, N, 6, FAKE, FAKE, 0, 0, 0, 0, None, None, None, None, None, 0)


def epilogue(**kw):
    from rgb_experiment_b200._lib import Epilogue
    e = Epilogue()
    e.a = 1.0
    for k, v in kw.items():
        if k == "peers":
            for q, p in enumerate(v):
                e.peer_out[q] = p
            e.n_peers = len(v)
        else:
            setattr(e, k, v)
    return e


def spmm(ep, Y=FAKE):
    g = graph()
    return L().rgbmp_spmm(C.byref(g), None, FAKE, F, Y, F, F, 0, None if ep is None else C.byref(ep), 0, FAKE, 1 << 20,
                          BAD_DEVICE, None)


def khop(ep, hops=None):
    g = graph()
    return L().rgbmp_khop(C.byref(g), None, FAKE, F, FAKE, FAKE, F, FAKE, F, hops, F, N * F, F, 0, 2,
                          None if ep is None else C.byref(ep), 0, FAKE, 1 << 20, BAD_DEVICE, None)


ENTRY = {"spmm": spmm, "khop": khop}
RESET = dict(reset_when=2, reset_mask=FAKE, reset_val=FAKE, ld_reset=F)
PEERS = dict(peers=[FAKE, FAKE + 16], ld_peer=F)

# rule -> (epilogue fields that break it, return code, what the error says); both entry points refuse them
RULES = {
    "reset_when above 2": (dict(RESET, reset_when=3), "EINVAL", b"bad reset_when 3"),
    "reset_when negative": (dict(RESET, reset_when=-1), "EINVAL", b"bad reset_when -1"),
    "reset before teleport without mask": (dict(RESET, reset_when=1, reset_mask=None), "EINVAL", b"reset rows need"),
    "reset after clamp without mask": (dict(RESET, reset_mask=None), "EINVAL", b"reset rows need"),
    "reset without values": (dict(RESET, reset_val=None), "EINVAL", b"reset rows need"),
    "ld_reset below F": (dict(RESET, ld_reset=F - 1), "EINVAL", b"reset rows need"),
    "ldt below F": (dict(T=FAKE, ldt=F - 1, b=0.5), "EINVAL", b"T needs ldt >= F"),
    "Y2 without out2_scale": (dict(Y2=FAKE, ldy2=F), "EINVAL", b"Y2 needs out2_scale"),
    "ldy2 below F": (dict(Y2=FAKE, ldy2=F - 1, out2_scale=FAKE), "EINVAL", b"Y2 needs out2_scale and ldy2 >= F"),
    "ld_acc below F": (dict(acc_in=FAKE, ld_acc=F - 1), "EINVAL", b"acc_in needs ld_acc >= F"),
    "n_peers negative": (dict(n_peers=-1), "EINVAL", b"bad n_peers -1"),
    "n_peers above 8": (dict(n_peers=9), "EINVAL", b"bad n_peers 9"),
    "null peer buffer": (dict(PEERS, peers=[FAKE, None]), "EINVAL", b"null peer buffer 1"),
    "misaligned peer buffer": (dict(PEERS, peers=[FAKE, FAKE + 4]), "EALIGN", b"peer buffer 1 not 16-byte aligned"),
    "ld_peer below F": (dict(PEERS, ld_peer=F - 1), "EINVAL", b"peers need ld_peer >= F"),
    "row_map with peers": (dict(PEERS, row_map=FAKE), "EINVAL", b"row_map does not combine with peers"),
    "row_map with acc_in": (dict(acc_in=FAKE, ld_acc=F, row_map=FAKE), "EINVAL", b"row_map does not combine with peers"),
    "row_map with reset rows": (dict(RESET, row_map=FAKE), "EINVAL", b"row_map does not combine with peers"),
}

# epilogues rgbmp_spmm takes and rgbmp_khop refuses: the K-hop driver owns every hop's stores
KHOP_ONLY = {
    "Y2": dict(Y2=FAKE, ldy2=F, out2_scale=FAKE),
    "acc_in": dict(acc_in=FAKE, ld_acc=F),
    "skip_empty": dict(skip_empty=1),
    "peers": PEERS,
}

WELL_FORMED = {
    "null": None,
    "identity": {},
    "every row operand": dict(row_scale=FAKE, row_div=1, T=FAKE, ldt=F, b=0.5, clamp=1, lo=-1.0, hi=1.0,
                              out2_scale=FAKE, **RESET),
    "reset before teleport": dict(RESET, reset_when=1, ld_reset=F + 4),
    "row_map": dict(row_map=FAKE, row_scale=FAKE, out2_scale=FAKE, T=FAKE, ldt=F),
}


def _call(entry, fields, **kw):
    rc = ENTRY[entry](None if fields is None else epilogue(**fields), **kw)
    err = L().rgbmp_last_error()
    assert f"rgbmp_{entry}".encode() in err, err
    return rc, err


def _refused(entry, fields, code, msg, **kw):
    from rgb_experiment_b200 import _lib
    rc, err = _call(entry, fields, **kw)
    assert rc == getattr(_lib, code) and msg in err and b"bad device" not in err, (rc, err)


def _passes(entry, fields, **kw):
    from rgb_experiment_b200._lib import EINVAL
    rc, err = _call(entry, fields, **kw)
    assert rc == EINVAL and b"bad device" in err, (rc, err)


@pytest.mark.parametrize("entry", ENTRY)
@pytest.mark.parametrize("form", WELL_FORMED)
def test_well_formed_epilogue_passes_the_checks(entry, form):
    _passes(entry, WELL_FORMED[form])


@pytest.mark.parametrize("entry", ENTRY)
@pytest.mark.parametrize("rule", RULES)
def test_every_rule_is_checked_before_the_device(entry, rule):
    fields, code, msg = RULES[rule]
    _refused(entry, fields, code, msg)


@pytest.mark.parametrize("field", KHOP_ONLY)
def test_khop_refuses_the_fields_of_a_single_launch(field):
    _refused("khop", KHOP_ONLY[field], "EINVAL", b"not K-hop epilogue fields")
    _passes("spmm", KHOP_ONLY[field])


def test_khop_refuses_row_map_with_every_hop_kept():
    _refused("khop", dict(row_map=FAKE), "EINVAL", b"row_map does not combine with hops", hops=FAKE)
    _passes("khop", dict(row_map=FAKE))
    _passes("khop", {}, hops=FAKE)


def test_spmm_needs_an_output():
    _refused("spmm", {}, "EINVAL", b"no output", Y=None)
    _refused("spmm", None, "EINVAL", b"no output", Y=None)
    _refused("spmm", dict(out2_scale=FAKE, acc_in=FAKE, ld_acc=F), "EINVAL", b"no output", Y=None)
    _passes("spmm", KHOP_ONLY["Y2"], Y=None)       # the pre-scaled copy alone, or the pushes alone, are an output
    _passes("spmm", KHOP_ONLY["peers"], Y=None)
