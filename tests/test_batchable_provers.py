"""Issue and show in BatchableProof form (afx_issue_batchable, afx_show_batchable and their _device forms; include/aeonflux_b200.h):
zkp's prove_batchable, which runs prove_compact's prover and returns the blinding commitments instead of the challenge.

Checked on the host emulation and, with -m gpu, on the CUDA library:
- parity with the oracle on every golden shape: the Python oracle's prover commitments (recorded from zkp.Prover.prove_compact) and
  the C oracle's verify trace give the expected words; every word that is not a commitment is the compact prover's;
- the output verifies under verify_batchable, verify_batchable_rlc and the Python restatement of zkp's verify_batchable;
- identity commitments (zeroed blindings) are written as 32 zero bytes with status 0 and rejected by the verifiers;
- multi-pass host calls, malformed items, the _device forms and the exact return codes of every precondition;
- the C++ wrapper (tests/cpp/batchable_driver.cpp);
- on the GPU, 65,536-item batches into the random-linear-combination verifiers."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from aeonflux_b200._binding import afx_issuance_out, afx_presentation_batch
from tests.common import GOLDEN_SHAPES, REQ, load_golden, to_batchable, words

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, ARG, SHAPE, NO_SECRET = 0, -1, -5, -6


@pytest.fixture(scope="module")
def emu():
    from aeonflux_b200._binding import Binding
    from tests.test_host_logic import build_hostemu
    return Binding(ctypes.CDLL(build_hostemu()))


@pytest.fixture(scope="module", params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def binding(request, emu):
    if request.param == "emu":
        return emu
    from aeonflux_b200._lib import load
    return load()


def golden_issuer(g):
    return bytes.fromhex(g["sysparams"]), bytes.fromhex(g["issuer_pub"]), bytes.fromhex(g["secret"])


def py_issuer(sp, ip, sk, n):
    from oracle.pyoracle import aeonflux as A, ristretto as R
    return A.Issuer(A.SystemParameters.from_bytes(sp), A.IssuerParameters(R.decompress(ip[:32]), R.decompress(ip[32:])),
                    A.SecretKey(*[int.from_bytes(sk[4 + 32 * i:36 + 32 * i], "little") for i in range(4)],
                                [int.from_bytes(sk[132 + 32 * i:164 + 32 * i], "little") for i in range(n)], R.decompress(sk[-32:])))


def python_prover_commitments(g, monkeypatch):
    """The blinding commitments the Python oracle's provers make for golden item 0 (oracle/pyoracle/synth.py:make_item):
    (the issuance proof's three, the presentation's: main proof first, then each proof of encryption)."""
    from oracle.pyoracle import synth as S, zkp as Z
    calls, orig = [], Z.Prover.prove_compact

    def recording(self, blindings):
        c, resp, cm = orig(self, blindings)
        calls.append(list(cm))
        return c, resp, cm
    monkeypatch.setattr(Z.Prover, "prove_compact", recording)
    S.make_item(S.make_issuer(g["n"]), tuple(g["request"]), tuple(g["hide"]), g["config"].encode(), g["items"][0]["item"])
    return calls[0], [w for cm in calls[1:] for w in cm]


def word_map(kinds):
    """The BatchableProof presentation layout as (source, index): ("w", i) = word i of the compact layout, ("c", j) = commitment j."""
    from oracle.pyoracle import flat as F
    W = F.presentation_num_words(list(kinds))
    nc = F.presentation_num_constraints(list(kinds)) + 5 * sum(k == 3 for k in kinds)
    return F.compact_to_batchable_words(list(kinds), [("w", i) for i in range(W)], [("c", j) for j in range(nc)])


def assert_same_non_commitment_words(kinds, batchable, compact):
    """Every word of the batchable presentations that is not a commitment (responses, points, revealed values) is the compact one."""
    for k, (src, i) in enumerate(word_map(kinds)):
        if src == "w":
            assert (batchable[:, k] == compact[:, i]).all(), (k, i)


def issuance_to_batchable(issu, commitments):
    from tests.test_host_logic import issuance_to_batchable as f
    return f(issu, commitments)


# ---- parity with the oracle ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", GOLDEN_SHAPES)
def test_show_batchable_matches_the_oracle(binding, coracle, monkeypatch, name):
    from aeonflux_b200 import Issuer, PresentationBatch
    from oracle.pyoracle import flat as F
    g = load_golden(name)
    sp, ip, sk = golden_issuer(g)
    e = g["items"][0]
    orc = coracle.Issuer(sp, ip, sk)
    rk = bytes(REQ[k] for k in g["request"])
    kinds, pres, _, showin = orc.synth(rk, g["hide"], g["config"].encode(), 0, 5, want_issuances=False, want_show_inputs=True)
    user = Issuer(sp, ip, None, max_batch=3, _binding=binding)               # showing needs no issuer secret
    fields = np.ascontiguousarray(showin.transpose(1, 0, 2))
    fields[2, 3, 0] ^= 1                                                     # item 3: V no longer decodes (or is another point)
    res, st, dbg = user.show_batch(kinds, fields, debug=True, batchable=True)
    comp, cst, cdbg = user.show_batch(kinds, fields, debug=True)
    got, cgot = res.fields.transpose(1, 0, 2), comp.fields.transpose(1, 0, 2)
    assert res.fields.shape[0] == binding.L.afx_batchable_num_fields(len(kinds), kinds)
    assert (st == cst).all() and not st[[0, 1, 2, 4]].any()
    assert (dbg["commitments"] == cdbg["commitments"]).all()
    if st[3]:
        assert not got[3].any()
    # item 0: the golden compact presentation with the Python oracle prover's commitments in place of the challenges
    _, pcm = python_prover_commitments(g, monkeypatch)
    expect0 = F.compact_to_batchable_words(list(kinds), [bytes.fromhex(w) for w in e["words"]], pcm)
    assert got[0].tobytes() == b"".join(expect0)
    if e["verdict"] == 0:
        assert [c.hex() for c in pcm] == e["commitments"]                    # ... which are the verify trace's
    ok = [0, 1, 2, 4]
    ov, _, tr = orc.verify_presentations(kinds, pres, trace=True)
    if not ov.any():                                                         # the C oracle's trace, on every item
        assert (got[ok] == to_batchable(kinds, pres, tr["commitments"])[ok]).all()
    assert_same_non_commitment_words(kinds, got, cgot)                      # responses: the compact prover's
    iss = Issuer(sp, ip, sk, max_batch=3, _binding=binding)
    vc = iss.verify_batch(comp)
    assert (iss.verify_batchable(res) == vc).all() and list(vc[ok]) == [e["verdict"]] * 4
    vr, fell_back = iss.verify_batchable_rlc(PresentationBatch(kinds, res.fields[:, ok]), bytes(range(32)))
    assert list(vr) == [e["verdict"]] * 4 and fell_back == (2 if e["verdict"] else 0)
    py = py_issuer(sp, ip, sk, g["n"])
    assert F.verify_flat(py, kinds, [got[0, w].tobytes() for w in range(got.shape[1])], batchable=True)[0] == e["verdict"]


@pytest.mark.parametrize("name", GOLDEN_SHAPES)
def test_issue_batchable_matches_the_oracle(binding, coracle, monkeypatch, name):
    from aeonflux_b200 import Issuer, RequestBatch
    from oracle.pyoracle import flat as F
    from tests.common import golden_issue_request
    g = load_golden(name)
    sp, ip, sk = golden_issuer(g)
    n, e = g["n"], g["items"][0]
    ik = bytes(e["issuance_kinds"])
    iss = Issuer(sp, ip, sk, max_batch=3, _binding=binding)
    attrs, rnd = golden_issue_request(g, e)
    res, st, dbg = iss.issue_batch(RequestBatch.from_request(ik, attrs[None], rnd[None]), debug=True, batchable=True)
    iw = words(e["issuance_words"])
    expect = np.concatenate([iw[:n + 3], words(e["issuance_commitments"]), iw[n + 4:]])
    assert st[0] == 0 and res.fields.shape == (2 * n + 11, 1, 32)
    assert res.fields[:, 0].tobytes() == expect.tobytes()
    pcm, _ = python_prover_commitments(g, monkeypatch)
    assert b"".join(pcm) == words(e["issuance_commitments"]).tobytes()      # the Python prover's are the verify trace's
    from oracle.pyoracle import aeonflux as A, ristretto as R
    ipp = A.IssuerParameters(R.decompress(ip[:32]), R.decompress(ip[32:]))
    assert F.verify_issuance_flat(A.SystemParameters.from_bytes(sp), ipp, ik, [w.tobytes() for w in res.fields[:, 0]], batchable=True)[0] == 0
    # fresh randomness against the C oracle, 5 items (two passes), one malformed
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(23)
    Ab = np.repeat(attrs[None], 5, axis=0)
    Rb = rng.integers(0, 256, (5, n + 7, 64), dtype=np.uint8)
    Ab[3, 0] = 0xff
    out, status, _ = orc.issue(ik, Ab, Rb)
    res, st = iss.issue_batch(RequestBatch.from_request(ik, Ab, Rb), batchable=True)
    comp, cst = iss.issue_batch(RequestBatch.from_request(ik, Ab, Rb))
    assert (st == status).all() and (cst == status).all() and list(status) == [0, 0, 0, 1, 0]
    ok = [0, 1, 2, 4]
    compact = np.ascontiguousarray(np.concatenate([Ab, out], axis=1)[ok])
    ov, _, tr = orc.verify_issuances(ik, compact, trace=True)
    assert not ov.any()
    got = res.fields.transpose(1, 0, 2)
    assert (got[ok] == issuance_to_batchable(compact, tr["commitments"])).all()
    assert not got[3, n:].any()                                              # the malformed request: all-zero words
    cgot = comp.fields.transpose(1, 0, 2)
    assert (got[:, :n + 3] == cgot[:, :n + 3]).all() and (got[:, n + 6:] == cgot[:, n + 4:]).all()   # t, U, V and the responses
    assert list(iss.verify_issuance_batchable(res)) == [0, 0, 0, 1, 0]
    user = Issuer(sp, ip, None, max_batch=3, _binding=binding)
    assert list(user.verify_batchable_rlc(res, bytes(32), issuance=True)[0]) == [0, 0, 0, 1, 0]


# ---- identity commitments ------------------------------------------------------------------------------------------------

def test_identity_commitments_are_written_and_rejected(binding, coracle):
    """Zeroed blindings make identity commitments (tests/test_identity_commitments.py).  zkp's prover appends them unchecked:
    the batchable provers write 32 zero bytes with status 0, the compact proof from the same inputs verifies, and verify_batchable
    rejects the item with verdict 1, as the Python restatement of zkp's verify_batchable does."""
    from aeonflux_b200 import Issuer, PresentationBatch, RequestBatch
    from oracle.pyoracle import aeonflux as A, flat as F, ristretto as R
    from tests.test_identity_commitments import show_rng_start, zero_patterns
    n = 4
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, _, issu, showin = orc.synth(b"SSPE", [0, 3], b"batchable-identity", 0, 4, want_show_inputs=True)
    r0 = show_rng_start(kinds)
    pats = zero_patterns((showin.shape[1] - r0) // 2 - 1, 3)
    show = np.stack([showin[j % len(showin)] for j in range(len(pats) + 1)])   # the last item keeps its blindings
    for j, pat in enumerate(pats):
        for b in pat:
            show[j, r0 + 2 * (b + 1):r0 + 2 * (b + 2)] = 0
    user = Issuer(sp, ip, None, max_batch=8, _binding=binding)
    fields = np.ascontiguousarray(show.transpose(1, 0, 2))
    res, st = user.show_batch(kinds, fields, batchable=True)
    comp, cst = user.show_batch(kinds, fields)
    assert not st.any() and not cst.any()
    compact = np.ascontiguousarray(comp.fields.transpose(1, 0, 2))
    ov, _, tr = orc.verify_presentations(kinds, compact, trace=True)
    assert not ov.any()                                                      # the compact proofs verify
    ident = ~tr["commitments"].any(axis=-1)
    assert ident.all(axis=1).any() and (ident.any(axis=1) & ~ident.all(axis=1)).any() and not ident[-1].any()
    got = res.fields.transpose(1, 0, 2)
    assert (got == to_batchable(kinds, compact, tr["commitments"])).all()
    cpos = [k for k, (src, _) in enumerate(word_map(kinds)) if src == "c"]
    assert ((~got[:, cpos].any(axis=-1)) == ident).all()                     # identity commitments: 32 zero bytes
    iss = Issuer(sp, ip, sk, max_batch=8, _binding=binding)
    v = iss.verify_batchable(res)
    assert (v == ident.any(axis=1)).all()
    assert (iss.verify_batchable_rlc(res, bytes(32))[0] == v).all()
    py = py_issuer(sp, ip, sk, n)
    for i in (0, len(pats) // 2, len(pats)):
        assert F.verify_flat(py, kinds, [got[i, w].tobytes() for w in range(got.shape[1])], batchable=True)[0] == v[i]
    # issuances: zeroed issuance blindings
    ik = bytes([0, 0, 2, 2])
    ipats = zero_patterns(n + 5, 2)
    m = len(ipats) + 1
    attrs = np.ascontiguousarray(np.stack([issu[j % len(issu), :n] for j in range(m)]))
    rnd = np.random.default_rng(9).integers(0, 256, (m, n + 7, 64), dtype=np.uint8)
    for j, pat in enumerate(ipats):
        for b in pat:
            rnd[j, 2 + b] = 0
    res, st = iss.issue_batch(RequestBatch.from_request(ik, attrs, rnd), batchable=True)
    comp, cst = iss.issue_batch(RequestBatch.from_request(ik, attrs, rnd))
    assert not st.any() and not cst.any()
    compact = np.ascontiguousarray(comp.fields.transpose(1, 0, 2))
    ov, _, tr = orc.verify_issuances(ik, compact, trace=True)
    assert not ov.any()
    ident = ~tr["commitments"].any(axis=-1)
    assert ident.all(axis=1).any() and (ident.any(axis=1) & ~ident.all(axis=1)).any() and not ident[-1].any()
    got = res.fields.transpose(1, 0, 2)
    assert (got == issuance_to_batchable(compact, tr["commitments"])).all()
    assert ((~got[:, n + 3:n + 6].any(axis=-1)) == ident).all()
    v = user.verify_issuance_batchable(res)
    assert (v == ident.any(axis=1)).all()
    sysp = A.SystemParameters.from_bytes(sp)
    ipp = A.IssuerParameters(R.decompress(ip[:32]), R.decompress(ip[32:]))
    assert [F.verify_issuance_flat(sysp, ipp, ik, [got[i, w].tobytes() for w in range(2 * n + 11)], batchable=True)[0] for i in range(m)] == list(v)


# ---- passes and device forms ------------------------------------------------------------------------------------------------

def test_multi_pass_calls_equal_one_item_at_a_time(binding, coracle):
    """A ragged batch of 19 items over max_batch = 8 (the pipelined path of the host calls) equals the same items proved one
    per call; malformed items in the middle give status 1 and all-zero words and leave their neighbours alone."""
    from aeonflux_b200 import Issuer, PresentationBatch, RequestBatch
    n, count = 4, 19
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, _, issu, showin = orc.synth(b"SSPE", [0, 3], b"batchable-passes", 0, count, want_show_inputs=True)
    fields = np.ascontiguousarray(showin.transpose(1, 0, 2))
    fields[1, 7] = 0xff                                                      # item 7: U does not decode
    fields[0, 11, 31] = 0xff                                                 # item 11: t >= l
    iss = Issuer(sp, ip, sk, max_batch=8, _binding=binding)
    res, st = iss.show_batch(kinds, fields, batchable=True)
    assert list(np.where(st)[0]) == [7, 11]
    assert not res.fields[:, [7, 11]].any()
    for i in range(count):
        one, s1 = iss.show_batch(kinds, fields[:, i:i + 1], batchable=True)
        assert s1[0] == st[i] and (one.fields[:, 0] == res.fields[:, i]).all(), i
    v = iss.verify_batchable(res)
    assert list(np.where(v)[0]) == [7, 11]
    ik = bytes([0, 0, 2, 2])
    attrs = np.ascontiguousarray(issu[:, :n])
    attrs[5, 2] = 0xff                                                       # item 5: a point attribute that does not decode
    rnd = np.random.default_rng(4).integers(0, 256, (count, n + 7, 64), dtype=np.uint8)
    req = RequestBatch.from_request(ik, attrs, rnd)
    ires, ist = iss.issue_batch(req, batchable=True)
    assert list(np.where(ist)[0]) == [5] and not ires.fields[n:, 5].any()
    for i in range(count):
        one, s1 = iss.issue_batch(RequestBatch(ik, req.fields[:, i:i + 1]), batchable=True)
        assert s1[0] == ist[i] and (one.fields[:, 0] == ires.fields[:, i]).all(), i
    assert list(np.where(iss.verify_issuance_batchable(ires))[0]) == [5]


def run_device(binding, emu, fn, fields, n_out):
    """A _device prover call on struct-of-arrays fields [n_in][count][32] -> (out [n_out][count][32], status).  On the host emulation
    device memory is host memory."""
    count = fields.shape[1]
    if binding is emu:
        out, st = np.zeros((n_out, count, 32), np.uint8), np.zeros(count, np.uint8)
        fn(count, np.ascontiguousarray(fields).ctypes.data, out.ctypes.data, st.ctypes.data, 0)
        return out, st
    import torch
    d_in = torch.from_numpy(np.ascontiguousarray(fields)).cuda()
    d_out = torch.empty((n_out, count, 32), dtype=torch.uint8, device="cuda")
    d_st = torch.empty(count, dtype=torch.uint8, device="cuda")
    fn(count, d_in.data_ptr(), d_out.data_ptr(), d_st.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), d_st.cpu().numpy()


def test_device_forms_equal_the_host_forms(binding, emu, coracle):
    from aeonflux_b200 import Issuer, RequestBatch
    n = 4
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, _, issu, showin = orc.synth(b"SSPE", [0, 3], b"batchable-device", 0, 6, want_show_inputs=True)
    fields = np.ascontiguousarray(showin.transpose(1, 0, 2))
    fields[2, 4, 0] ^= 1
    iss = Issuer(sp, ip, sk, max_batch=6, _binding=binding)
    res, st = iss.show_batch(kinds, fields, batchable=True)
    nb = binding.L.afx_batchable_num_fields(n, kinds)
    out, dst = run_device(binding, emu, lambda c, f, o, s, q: iss.show_batch_device(kinds, c, f, o, s, q, batchable=True), fields, nb)
    assert (dst == st).all() and (out == res.fields).all()
    ik = bytes([0, 0, 2, 2])
    rnd = np.random.default_rng(8).integers(0, 256, (6, n + 7, 64), dtype=np.uint8)
    req = RequestBatch.from_request(ik, np.ascontiguousarray(issu[:, :n]), rnd)
    ires, ist = iss.issue_batch(req, batchable=True)
    out, dst = run_device(binding, emu, lambda c, f, o, s, q: iss.issue_batch_device(ik, c, f, o, s, q, batchable=True), req.fields, n + 11)
    assert (dst == ist).all() and (out == ires.fields[n:]).all()


# ---- exact return codes ------------------------------------------------------------------------------------------------------

N, MAX = 4, 4
KINDS = bytes([0, 0, 2, 2])
SHOW_KINDS = bytes([1, 0, 2, 3])
BAD = bytes([0, 0, 2, 9])
DUMMY = ctypes.c_void_p(16)       # a non-null "buffer" that no failing check dereferences
HOST, DEVICE = ("issue_batchable", "show_batchable"), ("issue_batchable_device", "show_batchable_device")


@pytest.fixture(scope="module")
def contexts(emu, coracle):
    sp, ip, sk = (bytes(x) for x in coracle.make_issuer(N))
    L, hs = emu.L, []
    for secret in (sk, None):
        h = ctypes.c_void_p()
        assert L.afx_ctx_create(sp, len(sp), ip, secret, len(secret) if secret else 0, 0, MAX, ctypes.byref(h)) == OK
        hs.append(h)
    yield hs
    for h in hs:
        L.afx_ctx_destroy(h)


def call(L, name, c, kinds="default", count=0, null=False, nf_delta=0, out_delta=0):
    """afx_<name> with (kinds, count) and buffers that are null only where asked."""
    if isinstance(kinds, str):
        kinds = KINDS if name.startswith("issue") else SHOW_KINDS
    buf = None if null else DUMMY
    fn = getattr(L, "afx_" + name)
    n = N if kinds is None else len(kinds)
    if name.endswith("_device"):
        return fn(c, n, kinds, count, buf, buf, buf, None)
    k = kinds or KINDS
    if name.startswith("issue"):
        nf, nout = L.afx_request_num_fields(len(k)), len(k) + 11
    else:
        nf, nout = L.afx_show_num_fields(len(k), k), L.afx_batchable_num_fields(len(k), k)
    fp = None if null else ctypes.cast((ctypes.c_void_p * (nf + 1))(), ctypes.POINTER(ctypes.c_void_p))
    op = None if null else ctypes.cast((ctypes.c_void_p * (nout + 1))(), ctypes.POINTER(ctypes.c_void_p))
    b = afx_presentation_batch(n, kinds, count, fp, nf + nf_delta)
    o = afx_issuance_out(op, nout + out_delta)
    return fn(c, ctypes.byref(b), ctypes.byref(o), buf, None)


@pytest.mark.parametrize("name", HOST + DEVICE)
def test_return_codes(emu, contexts, name):
    L, (ctx, user) = emu.L, contexts
    assert call(L, name, None) == ARG and call(L, name, None, count=1) == ARG
    assert call(L, name, ctx, kinds=None) == ARG
    assert call(L, name, ctx, count=1, null=True) == ARG
    assert call(L, name, ctx, count=0, null=True) == OK
    assert call(L, name, ctx) == OK
    assert call(L, name, ctx, kinds=BAD) == SHAPE
    assert call(L, name, ctx, kinds=bytes([0, 0, 2])) == SHAPE               # an attribute count different from the issuer's
    if name.startswith("issue"):
        assert call(L, name, ctx, kinds=SHOW_KINDS) == SHAPE                 # hidden kinds cannot be issued
        assert call(L, name, user) == NO_SECRET
        assert call(L, name, user, kinds=BAD) == NO_SECRET                   # before the shape is compiled
    else:
        assert call(L, name, user) == OK                                     # showing needs no issuer secret
    if name in HOST:
        for d in (1, -1):
            assert call(L, name, ctx, nf_delta=d) == ARG
            assert call(L, name, ctx, out_delta=d) == ARG
    else:
        assert call(L, name, ctx, count=MAX + 1) == ARG
        assert call(L, name, user, count=MAX + 1) == (NO_SECRET if name.startswith("issue") else ARG)


def test_calls_while_two_submissions_are_outstanding(emu, contexts):
    L, (ctx, _) = emu.L, contexts
    t = [ctypes.c_uint64(), ctypes.c_uint64()]
    for k in range(2):
        assert L.afx_verify_presentations_wire_submit(ctx, N, KINDS, 0, DUMMY, DUMMY, ctypes.byref(t[k])) == OK
    for name in HOST + DEVICE:
        assert call(L, name, ctx) == ARG, name
        assert call(L, name, ctx, kinds=BAD) == ARG, name                     # refused before the shape is compiled
    for k in range(2):
        assert L.afx_wait(ctx, t[k].value) == OK
    for name in HOST + DEVICE:
        assert call(L, name, ctx) == OK, name


def test_linked_and_batchable_together_is_a_shape_error(emu, coracle):
    from aeonflux_b200 import Issuer
    from aeonflux_b200._binding import AfxError
    sp, ip, sk = coracle.make_issuer(N)
    user = Issuer(sp, ip, None, max_batch=MAX, _binding=emu)
    with pytest.raises(AfxError) as e:
        user.show_batch(SHOW_KINDS, np.zeros((emu.L.afx_show_num_fields(N, SHOW_KINDS), 1, 32), np.uint8), linked=True, batchable=True)
    assert e.value.code == SHAPE


# ---- C++ wrapper -------------------------------------------------------------------------------------------------------------

DRIVER = os.path.join(ROOT, "tests", "cpp", "batchable_driver.cpp")


def run_cpp_driver(tmp_path, coracle, lib_dir, lib_name, count, max_batch):
    from tests.test_cpp_host import write_fixture
    fx = tmp_path / "fixture.bin"
    write_fixture(fx, coracle, count)
    exe = str(tmp_path / "batchable_driver")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, DRIVER, "-L" + lib_dir, "-l" + lib_name, "-Wl,-rpath," + lib_dir])
    out = subprocess.run([exe, str(fx), str(max_batch)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout


def test_cpp_wrapper_on_emulation(tmp_path, coracle):
    from tests.test_host_logic import build_hostemu
    so = build_hostemu()
    out = run_cpp_driver(tmp_path, coracle, os.path.dirname(so), "afx_hostemu", 20, 8)
    assert "batchable_driver ok: 20 items" in out and "host-emulation" in out


@pytest.mark.gpu
def test_cpp_wrapper_on_gpu(tmp_path, coracle):
    from aeonflux_b200.build import CSRC
    out = run_cpp_driver(tmp_path, coracle, CSRC, "aeonflux_b200", 1000, 512)
    assert "batchable_driver ok: 1000 items" in out and "cuda sm_100a" in out


# ---- full size on the GPU ----------------------------------------------------------------------------------------------------

def full_size_show_inputs(orc, rk, hide, tag, creds, draws, seed):
    """creds credentials x draws rng draws: draw 0 is the oracle's own rng (its presentations are returned), the rest are random."""
    from tests.test_identity_commitments import show_rng_start
    kinds, pres, issu, showin = orc.synth(rk, hide, tag, 0, creds, want_show_inputs=True)
    r0 = show_rng_start(kinds)
    items = np.tile(showin, (draws, 1, 1))
    items[creds:, r0:] = np.random.default_rng(seed).integers(0, 256, items[creds:, r0:].shape, dtype=np.uint8)
    return kinds, pres, issu, np.ascontiguousarray(items.transpose(1, 0, 2))


@pytest.mark.gpu
def test_readme4_full_size_show_batchable_into_the_rlc_verifier(coracle):
    from aeonflux_b200 import Issuer, PresentationBatch
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    creds, draws = 2048, 32
    kinds, pres, _, fields = full_size_show_inputs(orc, b"SSPE", [0, 3], b"batchable-full", creds, draws, 31)
    N_ = creds * draws
    user = Issuer(sp, ip, None, max_batch=N_)
    res, st = user.show_batch(kinds, fields, batchable=True)
    comp, cst = user.show_batch(kinds, fields)
    assert not st.any() and not cst.any() and res.count == N_
    iss = Issuer(sp, ip, sk, max_batch=N_)
    v, fell_back = iss.verify_batchable_rlc(res, bytes(range(32)))
    assert not v.any() and fell_back == 0
    bad_idx = [7, 30001, N_ - 1]
    bad = res.fields.copy()
    nc = 2 + 2                                                               # README-4: Z, C_x_1 and two C_y constraints
    for i in bad_idx:
        bad[nc, i, 0] ^= 1                                                   # the response z
    v, fell_back = iss.verify_batchable_rlc(PresentationBatch(kinds, bad), bytes(range(32)))
    assert list(np.where(v)[0]) == bad_idx and fell_back == 1
    # a 256-item sample against the oracle: the compact proofs verify there, and its trace gives the commitments
    sample = np.sort(np.random.default_rng(2).choice(N_, 256, replace=False))
    sample[:8] = np.arange(8)                                                # draw 0: the oracle's own presentations
    sample = np.unique(sample)
    compact = np.ascontiguousarray(comp.fields[:, sample].transpose(1, 0, 2))
    assert (compact[sample < creds] == pres[sample[sample < creds]]).all()
    ov, _, tr = orc.verify_presentations(kinds, compact, trace=True)
    assert not ov.any()
    assert (res.fields[:, sample].transpose(1, 0, 2) == to_batchable(kinds, compact, tr["commitments"])).all()


@pytest.mark.gpu
def test_full_size_issue_batchable_into_the_rlc_verifier(coracle):
    from aeonflux_b200 import Issuer, RequestBatch
    n, N_ = 4, 65536
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    _, _, issu = orc.synth(b"SSPE", [], b"batchable-issue-full", 0, 2048)
    ik = bytes([0, 0, 2, 2])
    attrs = np.ascontiguousarray(np.tile(issu[:, :n], (N_ // 2048, 1, 1)))
    rnd = np.random.default_rng(12).integers(0, 256, (N_, n + 7, 64), dtype=np.uint8)
    iss = Issuer(sp, ip, sk, max_batch=N_)
    res, st = iss.issue_batch(RequestBatch.from_request(ik, attrs, rnd), batchable=True)
    assert not st.any()
    user = Issuer(sp, ip, None, max_batch=N_)
    v, fell_back = user.verify_batchable_rlc(res, bytes(32), issuance=True)
    assert not v.any() and fell_back == 0
    sample = np.random.default_rng(3).choice(N_, 256, replace=False)
    out, status, _ = orc.issue(ik, attrs[sample], rnd[sample])
    compact = np.ascontiguousarray(np.concatenate([attrs[sample], out], axis=1))
    ov, _, tr = orc.verify_issuances(ik, compact, trace=True)
    assert not status.any() and not ov.any()
    assert (res.fields[:, sample].transpose(1, 0, 2) == issuance_to_batchable(compact, tr["commitments"])).all()


@pytest.mark.gpu
def test_s16_show_batchable_through_the_exact_verifier(coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(16)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, _, _, fields = full_size_show_inputs(orc, b"SSSSSSPP" + b"E" * 8, [0, 1] + list(range(8, 16)), b"batchable-s16", 1024, 4, 16)
    user = Issuer(sp, ip, None, max_batch=4096)
    res, st = user.show_batch(kinds, fields, batchable=True)
    assert not st.any() and res.count == 4096
    iss = Issuer(sp, ip, sk, max_batch=4096)
    assert not iss.verify_batchable(res).any()
