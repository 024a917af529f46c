"""Recomputed commitments that are the identity.

The verify MSMs compute Q = R/2 of every constraint's commitment R and k_commit_encode encodes 2Q, all of an item's commitments under
one field inversion (engine.cuh:commit_encode_job).  R is the identity exactly when the batch's factor for it is zero, which must
neither poison the item's other encodings nor come out as anything but 32 zero bytes.  An honest prover whose blindings are zero
makes such commitments: the rng words behind a blinding are s || 0^32 with s = 0.  Here the prover zeroes one blinding, every
blinding but one, or all of them, so that identities land in the first, middle and last commitments and in every one; issuances
also get t = 0 or a zero scalar attribute, which makes tU or M_i -- the batch that a BatchableProof issuance encodes before its
transcript -- the identity.  Verdicts, Z, commitments and challenges must equal the oracle's, and encoding all of an item's
commitments under one inversion (AFX_COMMIT_ENCODE_PER=64) or three at a time must give the same bytes as one commitment per
thread, whose inversion does not depend on the other commitments."""
import ctypes

import numpy as np
import pytest

from tests.common import compare_with_oracle_trace

SHAPES = {"readme4": (4, b"SSPE", [0, 3]), "s16": (16, b"SSSSSSPP" + b"E" * 8, [0, 1] + list(range(8, 16)))}
PERS = ("1", "3", "64")


@pytest.fixture(scope="module")
def emu():
    from aeonflux_b200._binding import Binding
    from tests.test_host_logic import build_hostemu
    return Binding(ctypes.CDLL(build_hostemu()))


def zero_patterns(nb, step=1):
    """Subsets of the blindings 0 .. nb-1 to zero: each alone, every one, and every one but one."""
    every = list(range(nb))
    return [[b] for b in range(0, nb, step)] + [every] + [[c for c in every if c != b] for b in range(0, nb, step)]


def show_rng_start(kinds):
    """Index of the first rng word of afx_show's input (include/aeonflux_b200.h): after t, U, V, the attributes and the keypair."""
    q = 3 + sum(3 if k == 3 else 1 for k in kinds)
    return q + (4 if 3 in kinds else 0)


def run_per(monkeypatch, per, fn):
    monkeypatch.setenv("AFX_COMMIT_ENCODE_PER", per)
    try:
        return fn()
    finally:
        monkeypatch.delenv("AFX_COMMIT_ENCODE_PER")


def assert_same_runs(runs):
    """Every encoder batching gives the verdicts and debug dumps of one commitment per thread, byte for byte."""
    v1, d1 = runs[PERS[0]]
    for per in PERS[1:]:
        v, d = runs[per]
        assert (v == v1).all(), per
        for key in d1:
            assert (np.asarray(d[key]) == np.asarray(d1[key])).all(), (per, key)


def assert_identity_coverage(ident):
    """ident [items][commitments]: identities in the first, a middle and the last commitment, in all of them, and beside others."""
    nc = ident.shape[1]
    assert ident[:, 0].any() and ident[:, nc // 2].any() and ident[:, -1].any()
    assert ident.all(axis=1).any()
    assert (ident.any(axis=1) & ~ident.all(axis=1)).any()


@pytest.mark.parametrize("shape", list(SHAPES))
def test_identity_commitments_in_presentations(emu, coracle, monkeypatch, shape):
    from aeonflux_b200 import Issuer, PresentationBatch
    n, rk, hide = SHAPES[shape]
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, _, _, showin = orc.synth(rk, hide, b"identity-" + shape.encode(), 0, 4, want_show_inputs=True)
    r0 = show_rng_start(kinds)
    nb = (showin.shape[1] - r0) // 2 - 1                     # rng pair 0 is z, the rest are blindings
    pats = zero_patterns(nb, 1 if shape == "readme4" else 5)
    show = np.stack([showin[j % len(showin)] for j in range(len(pats))])
    for j, pat in enumerate(pats):
        for b in pat:
            show[j, r0 + 2 * (b + 1):r0 + 2 * (b + 2)] = 0
    user = Issuer(sp, ip, None, max_batch=len(pats), _binding=emu)
    got, st = user.show_wire(kinds, show)
    assert not st.any()
    ov, _, tr = orc.verify_presentations(kinds, got, trace=True)
    assert not ov.any()                                        # identity blinding commitments are valid in a compact proof
    ident = ~tr["commitments"].any(axis=-1)
    assert_identity_coverage(ident)
    iss = Issuer(sp, ip, sk, max_batch=len(pats), _binding=emu)
    runs = {per: run_per(monkeypatch, per, lambda: iss.verify_batch(PresentationBatch.from_items(kinds, got), debug=True)) for per in PERS}
    assert_same_runs(runs)
    v, dbg = runs[PERS[0]]
    compare_with_oracle_trace(v, dbg, ov, tr)
    assert (dbg["commitments"].transpose(1, 0, 2)[:, :tr["commitments"].shape[1]] == tr["commitments"]).all()   # the zero rows too
    # the same items as BatchableProofs: the wire now carries the identity commitments, which verify_batchable rejects
    from tests.common import to_batchable
    bb = PresentationBatch.from_items(kinds, to_batchable(kinds, got, dbg["commitments"].transpose(1, 0, 2)))
    runs = {per: run_per(monkeypatch, per, lambda: iss.verify_batchable(bb, debug=True)) for per in PERS}
    assert_same_runs(runs)
    assert (runs[PERS[0]][0] == ident.any(axis=1)).all()
    iss.close()
    user.close()


def test_identity_commitments_in_issuances(emu, coracle, monkeypatch):
    from aeonflux_b200 import Issuer, PresentationBatch, RequestBatch
    from oracle.pyoracle import aeonflux as A, flat as F, ristretto as R
    from tests.test_host_logic import issuance_to_batchable
    n, rk, hide = SHAPES["readme4"]
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    _, _, issu = orc.synth(rk, hide, b"identity-issuance", 0, 4)
    ik = bytes(0 if c == ord("S") else 2 for c in rk)
    nb = n + 5
    pats = zero_patterns(nb)
    m = len(pats) + 3
    attrs = np.ascontiguousarray(np.stack([issu[j % len(issu), :n] for j in range(m)]))
    rnd = np.random.default_rng(5).integers(0, 256, (m, n + 7, 64), dtype=np.uint8)      # t, U, blinding[n + 5]
    for j, pat in enumerate(pats):
        for b in pat:
            rnd[j, 2 + b] = 0
    rnd[m - 3, 0] = 0                   # t = 0: tU is the identity
    attrs[m - 2, 0] = 0                 # a zero scalar attribute: M_0 is the identity
    attrs[m - 1, :2] = 0                # both scalar attributes zero: M_0 and M_1
    iss = Issuer(sp, ip, sk, max_batch=m, _binding=emu)
    res, st = iss.issue_batch(RequestBatch.from_request(ik, attrs, rnd))
    out, status, _ = orc.issue(ik, attrs, rnd)
    assert not st.any() and not status.any()
    issued = np.ascontiguousarray(res.fields.transpose(1, 0, 2))
    assert (issued[:, n:] == out).all()
    ov, _, tr = orc.verify_issuances(ik, issued, trace=True)
    assert list(ov) == [0] * len(pats) + [1, 1, 1]             # the reference rejects an identity tU or M_i
    assert_identity_coverage(~tr["commitments"][:len(pats)].any(axis=-1))
    runs = {per: run_per(monkeypatch, per, lambda: iss.verify_issuance_batch(PresentationBatch.from_items(ik, issued), debug=True)) for per in PERS}
    assert_same_runs(runs)
    v, dbg = runs[PERS[0]]
    compare_with_oracle_trace(v, dbg, ov, tr)
    ok = ov == 0
    assert (dbg["commitments"].transpose(1, 0, 2)[ok] == tr["commitments"][ok]).all()
    # BatchableProof issuances: tU and the M_i are encoded (one batch) before the transcript derives the challenge
    bi = issuance_to_batchable(issued, dbg["commitments"].transpose(1, 0, 2))
    runs = {per: run_per(monkeypatch, per, lambda: iss.verify_issuance_batchable(PresentationBatch.from_items(ik, bi), debug=True)) for per in PERS}
    assert_same_runs(runs)
    v, dbg = runs[PERS[0]]
    assert (dbg["challenges"][0][ok] == issued[ok, n + 3]).all()   # the derived challenge is the compact proof's
    sysp = A.SystemParameters.from_bytes(sp)
    ipp = A.IssuerParameters(R.decompress(ip[:32]), R.decompress(ip[32:]))
    expect = [F.verify_issuance_flat(sysp, ipp, ik, [bi[i, w].tobytes() for w in range(bi.shape[1])], batchable=True)[0] for i in range(m)]
    assert list(v) == expect
    iss.close()
