"""Every ladder at the extremes of its scalar recoding.

Each scalar multiplication of the engine looks up a table by a recoded digit: signed radix 16 (per-item bases, every prover term,
the aMAC, decrypt), biased radix 4096 or radix 2^16 (the constant terms of the verify MSMs, sc.cuh) and the radix-16 comb
(constant-only jobs).  Random scalars reach the extreme digits -- the last entries of the 2,048- and 32,768-entry tables -- with
probability 2^-12 to 2^-16 per digit, so a batch of a few hundred items never does.  Here the scalars are chosen: one set of
canonical scalars whose recodings hold every extreme digit at every position goes into the challenge and response words of honest
presentations and issuances, into the rng words behind t, z and the blindings, into the symmetric keypair and into the issuer's
secret key, and every output is compared with the oracle byte for byte.  Each check runs on the host emulation and, under -m gpu,
on the CUDA library."""
import ctypes

import numpy as np
import pytest

from tests.common import compare_with_oracle_trace, issuance_scalar_words, presentation_scalar_words

L = 2**252 + 27742317777372353535851937790883648493
P = 2**255 - 19
B12 = sum(2048 << (12 * j) for j in range(21))      # sc_bias4096's bias
B16 = sum(32768 << (16 * j) for j in range(15))     # sc_bias65536's bias


def from_digits(digits, bits):
    return sum(d << (bits * j) for j, d in enumerate(digits))


def alternate(a, b, count, top, bits):
    """The scalar whose `count` low digits alternate a, b, ... and whose top digit is `top`."""
    return from_digits([a if j % 2 == 0 else b for j in range(count)] + [top], bits)


SCALARS = [
    0, 1, 2, L - 1, L - 2, 2**252 - 1, 2**252, (L - 1) // 2,
    int("7" * 62 + "8", 16),              # radix 16: 63 digits -8, top digit 1
    int("7" * 63, 16),                    # radix 16: 63 digits +7
    2**252 - B12,                         # radix 4096: 21 digits -2048 (the last table entry), top digit 1
    2**252 - 1 - B12,                     # radix 4096: 21 digits +2047
    2**240 - B16,                         # radix 2^16: 15 digits -32768 (the last table entry), top digit 1
    2**252 - B16,                         # radix 2^16: 15 digits -32768 and the largest top digit, 2^12
    2**252 - 1 - B16,                     # radix 2^16: 15 digits +32767
    alternate(-8, 0, 63, 1, 4), alternate(0, 7, 63, 0, 4),
    alternate(-2048, 0, 21, 1, 12), alternate(0, 2047, 21, 0, 12),
    alternate(-32768, 0, 15, 2**12, 16), alternate(0, 32767, 15, 0, 16),
]


# ---- the recodings of sc.cuh, restated ------------------------------------------------------------------------------------

def recode16(a):
    """sc_recode16 + sc_digit16: 64 signed digits, packed as nibbles and sign-extended."""
    digits, carry = [], 0
    for i in range(64):
        d = ((a >> (4 * i)) & 15) + carry
        carry = (d + 8) >> 4
        nib = (d - (carry << 4)) & 15
        digits.append(nib - 16 if nib >= 8 else nib)
    return digits


def digits4096(a):
    """sc_bias4096 + sc_digit4096: 21 digits of (a + B12) mod 2^256 minus 2048, then the unbiased top (bits 252..255)."""
    out = (a + B12) % 2**256
    return [((out >> (12 * j)) & 0xfff) - 2048 for j in range(21)] + [out >> 252]


def digits65536(a):
    """sc_bias65536 + sc_digit65536: 15 halfwords of (a + B16) mod 2^256 minus 32768, then the unbiased top halfword."""
    out = (a + B16) % 2**256
    return [((out >> (16 * j)) & 0xffff) - 32768 for j in range(15)] + [out >> 240]


RECODINGS = {"radix 16": (recode16, 4, -8, 7), "radix 4096": (digits4096, 12, -2048, 2047), "radix 2^16": (digits65536, 16, -32768, 32767)}


def test_scalar_set_reaches_every_extreme_digit():
    """Every low digit position of every recoding holds its minimum (the last table entry), its maximum and 0 in some scalar of
    the set, and the set holds the largest top digit any canonical scalar has.  The top digit is floor((a + bias) / radix^top) and
    grows with a, so l - 1 has the largest one."""
    assert all(0 <= s < L for s in SCALARS) and len(set(SCALARS)) == len(SCALARS)
    for name, (recode, bits, lo, hi) in RECODINGS.items():
        table = [recode(s) for s in SCALARS]
        assert all(from_digits(d, bits) == s for d, s in zip(table, SCALARS)), name
        for j in range(len(table[0]) - 1):
            assert {lo, 0, hi} <= {d[j] for d in table}, (name, j)
        top = recode(L - 1)[-1]
        assert max(d[-1] for d in table) == top and 0 in {d[-1] for d in table}, name
    assert recode16(L - 1)[-1] == 1 and digits4096(L - 1)[-1] == 1 and digits65536(L - 1)[-1] == 2**12


# ---- fixtures and helpers ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def emu():
    from aeonflux_b200._binding import Binding
    from tests.test_host_logic import build_hostemu
    return Binding(ctypes.CDLL(build_hostemu()))


def emu_issuers(emu, monkeypatch):
    """Contexts on the host emulation.  wide: build the radix-2^16 constant tables (they fit its 72 MB budget for up to 24
    generators, i.e. up to 6 attributes); otherwise the verify MSMs use the radix-4096 tables, the emulation's default."""
    from aeonflux_b200 import Issuer

    def make(sp, ip, sk, wide=False, max_batch=64):
        if wide:
            monkeypatch.setenv("AFX_HOSTEMU_CTAB16", "1")
        else:
            monkeypatch.delenv("AFX_HOSTEMU_CTAB16", raising=False)
        return Issuer(sp, ip, sk, max_batch=max_batch, _binding=emu)
    return make


def gpu_issuers(monkeypatch):
    """Contexts on the B200.  wide: the library's default table budget (radix-2^16 tables for every issuer here); otherwise budget
    0, the radix-4096 tables."""
    from aeonflux_b200 import Issuer

    def make(sp, ip, sk, wide=True, max_batch=64):
        if wide:
            monkeypatch.delenv("AFX_CTAB16_BUDGET_MB", raising=False)
        else:
            monkeypatch.setenv("AFX_CTAB16_BUDGET_MB", "0")
        return Issuer(sp, ip, sk, device=0, max_batch=max_batch)
    return make


def word(v):
    return np.frombuffer(int(v).to_bytes(32, "little"), np.uint8)


def num(w):
    return int.from_bytes(bytes(w), "little")


# request kinds and hidden indices: README-4, S16 and a 3-attribute shape (hidden scalar, revealed point, hidden plaintext)
SHAPES = {"readme4": (4, b"SSPE", [0, 3]), "s16": (16, b"SSSSSSPP" + b"E" * 8, [0, 1] + list(range(8, 16))), "three": (3, b"SPE", [0, 2])}


def issuance_kinds(rk):
    return bytes(0 if c == ord("S") else 2 for c in rk)


def with_extreme_scalars(items, scalar_words):
    """For every scalar of the set: one copy of an honest item per scalar word with that word replaced by the scalar, and one copy
    with every scalar word replaced.  -> [len(SCALARS) * (len(scalar_words) + 1)][W][32]"""
    out = []
    for j, s in enumerate(SCALARS):
        for k, w in enumerate(list(scalar_words) + [None]):
            it = items[(j + k) % len(items)].copy()
            it[list(scalar_words) if w is None else w] = word(s)
            out.append(it)
    return np.stack(out)


def assert_matches_tiled_trace(v, dbg, ov, tr, reps):
    """compare_with_oracle_trace for a batch that is the oracle's batch repeated `reps` times (vectorised)."""
    assert (v == np.tile(ov, reps)).all()
    eng = {"Z": dbg["Z"], "commitments": dbg["commitments"].transpose(1, 0, 2), "challenges": dbg["challenges"].transpose(1, 0, 2)}
    for key, o in tr.items():
        o = np.tile(o, (reps,) + (1,) * (o.ndim - 1))
        e = eng[key][:, :o.shape[1]] if o.ndim == 3 else eng[key]
        assert ((e == o) | ~o.any(axis=-1, keepdims=True)).all(), key


# ---- 2. verify paths ----------------------------------------------------------------------------------------------------------

def check_verify_paths(make_issuer, coracle, shape, wide, tile_past=0):
    """Presentations and issuances whose scalar words -- challenges, responses, revealed scalars, t -- hold the scalars of the set, one
    word at a time and then all of them:
    the items are rejected, and Z, every commitment and every challenge the oracle computed match byte for byte.  A batch of a few
    hundred items takes the split aMAC ladder (k_ladders_parts); with tile_past, the same batch repeated past that many items takes
    the fused k_ladders launch and must give the same bytes.  The context must hold the wide constant tables iff `wide`."""
    from aeonflux_b200 import PresentationBatch
    n, rk, hide = SHAPES[shape]
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, pres, issu = orc.synth(rk, hide, b"extremes-" + shape.encode(), 0, 8)
    ik = issuance_kinds(rk)
    bad_p = with_extreme_scalars(pres, presentation_scalar_words(kinds))
    bad_i = with_extreme_scalars(issu, issuance_scalar_words(ik))
    reps = tile_past // len(bad_p) + 1 if tile_past else 1
    iss = make_issuer(sp, ip, sk, wide, max_batch=len(bad_p) * reps)
    narrow = make_issuer(sp, ip, sk, False, max_batch=1)
    assert iss.launch_count == narrow.launch_count + int(wide)          # the radix-2^16 table setup ran iff wide
    narrow.close()
    for ks, items, issuance in ((kinds, bad_p, False), (ik, bad_i, True)):
        if issuance:
            ov, _, tr = orc.verify_issuances(ks, items, trace=True)
            run = lambda b: iss.verify_issuance_batch(b, debug=True)      # noqa: E731
        else:
            ov, _, tr = orc.verify_presentations(ks, items, trace=True)
            run = lambda b: iss.verify_batch(b, debug=True)               # noqa: E731
        assert ov.all()
        v, dbg = run(PresentationBatch.from_items(ks, items))
        compare_with_oracle_trace(v, dbg, ov, tr)
        # the oracle got as far as the commitments in every row but some of the first block, scalar 0: there a zero t or scalar
        # attribute of an issuance is the identity point the reference rejects first, and with every word zero a presentation's
        # commitments are identities -- all-zero encodings, which compare_with_oracle_trace skips, so they are checked here
        per = len(items) // len(SCALARS)
        blank = ~tr["commitments"].any(axis=(1, 2))
        assert blank[per - 1] and not blank[per:].any()
        if not issuance:
            assert blank[:per].sum() == 1 and not dbg["commitments"][:, per - 1].any()
        if reps > 1:
            vb, dbgb = run(PresentationBatch.from_items(ks, np.tile(items, (reps, 1, 1))))
            assert_matches_tiled_trace(vb, dbgb, ov, tr, reps)
    assert not iss.verify_batch(PresentationBatch.from_items(kinds, pres)).any()
    assert not iss.verify_issuance_batch(PresentationBatch.from_items(ik, issu)).any()
    iss.close()


EMU_VERIFY = [("readme4", False), ("readme4", True), ("three", False), ("three", True), ("s16", False)]   # S16's wide tables exceed the emulation's budget


@pytest.mark.parametrize("shape,wide", EMU_VERIFY)
def test_verify_paths_on_emulation(emu, coracle, monkeypatch, shape, wide):
    check_verify_paths(emu_issuers(emu, monkeypatch), coracle, shape, wide)


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [True, False])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_verify_paths_on_gpu(coracle, monkeypatch, shape, wide):
    check_verify_paths(gpu_issuers(monkeypatch), coracle, shape, wide, tile_past=8192)


# ---- 3. prover paths ----------------------------------------------------------------------------------------------------------

def show_layout(kinds):
    """Word indices of afx_show's input (include/aeonflux_b200.h): the attribute words, the keypair (or None) and the first rng word."""
    attrs, q = [], 3                                  # t, U, V
    for k in kinds:
        attrs.append(q)
        q += 3 if k == 3 else 1                       # a hidden plaintext is M1, M2, m3
    kp = q if 3 in kinds else None
    return attrs, kp, q + (4 if kp is not None else 0)


def python_show(spy, ipy, kinds, row):
    """AnonymousCredential::show of the Python oracle on one afx_show input row -> the flat presentation words."""
    from oracle.pyoracle import aeonflux as A, flat as F, ristretto as R
    b = [bytes(w) for w in row]
    dec = R.decompress
    attrs, kp_at, r0 = show_layout(kinds)
    shown = []
    for k, q in zip(kinds, attrs):
        if k == 3:
            shown.append(("SP", A.Plaintext(dec(b[q]), dec(b[q + 1]), num(b[q + 2]))))
        elif k == 2:
            shown.append(("PP", dec(b[q])))
        else:
            shown.append(("PS" if k == 0 else "SS", num(b[q])))
    kp = A.SymmetricKeypair(num(b[kp_at]), num(b[kp_at + 1]), num(b[kp_at + 2]), dec(b[kp_at + 3])) if kp_at is not None else None
    sc = [R.sc_from_wide(b[q] + b[q + 1]) for q in range(r0, len(b), 2)]
    h_s, h_p = kinds.count(1), kinds.count(3)
    p = A.presentation_prove(spy, ipy, A.Amac(num(b[0]), dec(b[1]), dec(b[2])), shown, kp, sc[0], sc[1:4 + h_s],
                             [sc[4 + h_s + 6 * e:10 + h_s + 6 * e] for e in range(h_p)])
    return np.frombuffer(b"".join(F.presentation_to_words(p)), np.uint8).reshape(-1, 32)


def check_prover_paths(make_issuer, coracle, shape):
    """Issuer::issue and AnonymousCredential::show with the rng words chosen so that t, z and every blinding are scalars of the set
    (Scalar::random reduces 64 rng bytes, so s || 0^32 draws s); the scalar attributes and the keypair come from the set too, and
    item j uses SCALARS[j] everywhere.  The credentials afx_issue makes are shown.  afx_issue and afx_show (struct-of-arrays and
    item-major) are byte-identical to the oracles, and the presentations verify as the oracle says."""
    from aeonflux_b200 import PresentationBatch, RequestBatch
    from oracle.pyoracle import aeonflux as A, ristretto as R
    n, rk, hide = SHAPES[shape]
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    m = len(SCALARS)
    kinds, _, issu, showin = orc.synth(rk, hide, b"extremes-prover-" + shape.encode(), 0, m, want_show_inputs=True)
    ik = issuance_kinds(rk)
    scalar_attrs = [k for k in range(n) if ik[k] == 0]
    attrs = np.ascontiguousarray(issu[:, :n])
    rnd = np.random.default_rng(12).integers(0, 256, (m, n + 7, 64), dtype=np.uint8)      # t, U, blinding[n + 5]
    for j, s in enumerate(SCALARS):
        attrs[j, scalar_attrs] = word(s)
        rnd[j, :, 32:] = 0
        rnd[j, :, :32] = word(s)
        rnd[j, 1] = np.random.default_rng(j).integers(0, 256, 64, dtype=np.uint8)         # U stays a random point
    iss = make_issuer(sp, ip, sk, max_batch=m)
    res, st = iss.issue_batch(RequestBatch.from_request(ik, attrs, rnd))
    out, status, _ = orc.issue(ik, attrs, rnd)
    assert not status.any() and not st.any()
    issued = np.ascontiguousarray(res.fields.transpose(1, 0, 2))
    assert (issued[:, n:] == out).all(), "afx_issue differs from the oracle"
    assert all(num(out[j, 0]) == s for j, s in enumerate(SCALARS))                       # t is the chosen scalar
    wout, wst = iss.issue_wire(ik, np.ascontiguousarray(RequestBatch.from_request(ik, attrs, rnd).fields.transpose(1, 0, 2)))
    assert not wst.any() and (wout == issued).all()
    oi, _ = orc.verify_issuances(ik, issued)
    assert (iss.verify_issuance_batch(res) == oi).all()
    # show the credentials just issued, with z, the blindings and the keypair from the set
    spy = A.SystemParameters.from_bytes(sp)
    ipy = A.IssuerParameters(R.decompress(ip[:32]), R.decompress(ip[32:]))
    at, kp_at, r0 = show_layout(kinds)
    show = showin.copy()
    show[:, :3] = out[:, :3]                                                             # t, U, V
    for j, s in enumerate(SCALARS):
        for k in scalar_attrs:
            show[j, at[k]] = word(s)
        if kp_at is not None:
            show[j, kp_at:kp_at + 3] = word(s)
            show[j, kp_at + 3] = np.frombuffer((spy.G_a * s + spy.G_a0 * s + spy.G_a1 * s).compress(), np.uint8)
        show[j, r0::2] = word(s)
        show[j, r0 + 1::2] = 0
    user = make_issuer(sp, ip, None, max_batch=m)
    pres, st = user.show_batch(kinds, np.ascontiguousarray(show.transpose(1, 0, 2)))
    assert not st.any()
    got = np.ascontiguousarray(pres.fields.transpose(1, 0, 2))
    for j in range(m):
        assert (got[j] == python_show(spy, ipy, list(kinds), show[j])).all(), ("afx_show differs from the oracle", shape, hex(SCALARS[j]))
    wgot, wst = user.show_wire(kinds, show)
    assert not wst.any() and (wgot == got).all()
    ov, _ = orc.verify_presentations(kinds, got)
    assert (iss.verify_batch(PresentationBatch.from_items(kinds, got)) == ov).all()
    assert list(ov) == [1] + [0] * (m - 1)        # item 0 (t = z = 0) makes C_x_1 and Z the identity, which verification rejects
    iss.close()
    user.close()


@pytest.mark.parametrize("shape", ["readme4", "three"])
def test_prover_paths_on_emulation(emu, coracle, monkeypatch, shape):
    check_prover_paths(emu_issuers(emu, monkeypatch), coracle, shape)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["readme4", "three"])
def test_prover_paths_on_gpu(coracle, monkeypatch, shape):
    check_prover_paths(gpu_issuers(monkeypatch), coracle, shape)


def check_encryption_keypairs(make_issuer, coracle):
    """Keypair::encrypt / Keypair::decrypt with a, a0, a1 from the set -- all three equal, and three consecutive scalars of the set in
    turn: the ciphertexts are the C oracle's and decrypt to the original data and plaintexts."""
    from tests import symoracle
    sp, ip, _ = coracle.make_issuer(4)
    iss = make_issuer(sp, ip, None, max_batch=8)
    data = np.random.default_rng(30).integers(0, 256, (5, 30), dtype=np.uint8)
    data[0] = 0                                                                        # M1 = identity
    pts, st = iss.encode_plaintexts(data)
    assert not st.any()
    m = len(SCALARS)
    for j, s in enumerate(SCALARS):
        for kp in ((s, s, s), (s, SCALARS[(j + 1) % m], SCALARS[(j + 2) % m])):
            kpb = b"".join(int(x).to_bytes(32, "little") for x in kp)
            ct, st = iss.encrypt(kpb, pts)
            oct_, ost, _ = symoracle.encrypt(kpb, pts)
            assert not st.any() and not ost.any()
            assert (ct == oct_).all(), ("afx_encrypt differs from the oracle", [hex(x) for x in kp])
            back, pts2, st = iss.decrypt(kpb, ct, plaintexts=True)
            assert not st.any() and (back == data).all() and (pts2 == pts).all(), [hex(x) for x in kp]
    iss.close()


def test_encryption_keypairs_on_emulation(emu, coracle, monkeypatch):
    check_encryption_keypairs(emu_issuers(emu, monkeypatch), coracle)


@pytest.mark.gpu
def test_encryption_keypairs_on_gpu(coracle, monkeypatch):
    check_encryption_keypairs(gpu_issuers(monkeypatch), coracle)


def check_chosen_secret_key(make_issuer, coracle):
    """README-4 issuers whose x_0, x_1 and y_i are scalars of the set (SecretKey::generate draws them with Scalar::random, which can
    return any canonical scalar), so the aMAC ladder reads its batch-uniform secret digits at their extremes: honest presentations
    verify with the oracle's Z, commitments and challenges, and afx_issue is byte-identical to the oracle."""
    from aeonflux_b200 import PresentationBatch, RequestBatch
    from oracle.pyoracle import aeonflux as A
    n = 4
    sp, _, sk0 = coracle.make_issuer(n)
    spy = A.SystemParameters.from_bytes(sp)
    w, wp = num(sk0[4:36]), num(sk0[36:68])
    ik = bytes([0, 0, 2, 2])
    rng = np.random.default_rng(40)
    for g in range(0, len(SCALARS), n + 2):
        xs = [SCALARS[(g + k) % len(SCALARS)] for k in range(n + 2)]
        key = A.SecretKey(w, wp, xs[0], xs[1], xs[2:], spy.G_w * w)
        ip, sk = A.IssuerParameters.generate(spy, key).to_bytes(), key.to_bytes()
        orc = coracle.Issuer(sp, ip, sk)
        kinds, pres, issu = orc.synth(b"SSPE", [0, 3], b"extremes-key-%d" % g, 0, 6)
        pres[5, 1, 0] ^= 1
        iss = make_issuer(sp, ip, sk, max_batch=8)
        ov, _, tr = orc.verify_presentations(kinds, pres, trace=True)
        assert list(ov) == [0, 0, 0, 0, 0, 1]
        v, dbg = iss.verify_batch(PresentationBatch.from_items(kinds, pres), debug=True)
        compare_with_oracle_trace(v, dbg, ov, tr)
        assert not iss.verify_issuance_batch(PresentationBatch.from_items(ik, issu)).any()
        attrs = np.ascontiguousarray(issu[:, :n])
        rnd = rng.integers(0, 256, (len(attrs), n + 7, 64), dtype=np.uint8)
        res, st = iss.issue_batch(RequestBatch.from_request(ik, attrs, rnd))
        out, status, _ = orc.issue(ik, attrs, rnd)
        assert not st.any() and not status.any() and (res.fields.transpose(1, 0, 2)[:, n:] == out).all(), [hex(x) for x in xs]
        iss.close()


def test_chosen_secret_key_on_emulation(emu, coracle, monkeypatch):
    check_chosen_secret_key(emu_issuers(emu, monkeypatch), coracle)


@pytest.mark.gpu
def test_chosen_secret_key_on_gpu(coracle, monkeypatch):
    check_chosen_secret_key(gpu_issuers(monkeypatch), coracle)


# ---- 4. primitive hooks ---------------------------------------------------------------------------------------------------------

def degenerate_field_inputs():
    """Field elements where the Elligator map's denominator D = (-1 - d*r)(r + d), r = i*t^2, is zero: t = +-sqrt(d*i) and
    +-sqrt(i/d) (both are squares mod p); the 32-byte words t + p and t with bit 255 set (from_bytes drops bit 255); and 0, 1, p - 1,
    p, p + 1, 2^255 - 1, +-i."""
    from oracle.pyoracle import ristretto as R
    d, i = R.D, R.SQRT_M1
    ts = []
    for sq in (d * i % P, i * pow(d, -1, P) % P):
        ok, t = R.sqrt_ratio_i(sq, 1)
        assert ok and t * t % P == sq
        for u in (t, P - t):
            r = i * u * u % P
            assert (P - 1 - d * r) * (r + d) % P == 0
            ts += [u, u + P, u | 2**255]
    return ts + [0, 1, P - 1, P, P + 1, 2**255 - 1, i, P - i, 2**255, 2**255 + 1]


def check_primitive_extremes(iss):
    """The hooks behind the ladders on the set: scalar * point (ops 2 and 10) against the Python oracle for the basepoint, random
    points and the identity; the biased radix-2^16 recoding (op 12) and the radix-4096 one (op 11) recompose to their input; and the
    degenerate field inputs through from_uniform_bytes (op 1) and decompress (op 0)."""
    from oracle.pyoracle import ristretto as R
    rng = np.random.default_rng(50)
    pts = [R.BASEPOINT, R.Point.identity()] + [R.from_uniform_bytes(rng.bytes(64)) for _ in range(3)]
    rows = [(s, p) for s in SCALARS for p in pts]
    inp = np.stack([np.concatenate([word(s), np.frombuffer(p.compress(), np.uint8)]) for s, p in rows])
    exp = np.stack([np.frombuffer((p * s).compress(), np.uint8) for s, p in rows])
    for name in ("scalarmult", "ladder_scalarmult"):
        out, ok = iss.selftest_primitive(name, inp)
        assert ok.all()
        bad = np.nonzero((out != exp).any(axis=1))[0]
        assert len(bad) == 0, (name, hex(rows[bad[0]][0]), rows[bad[0]][1].compress().hex())
    # recodings: the set, 12- and 16-bit field patterns and non-canonical values; op 12's flag says whether the top digit is <= 2^13 + 1
    pat = lambda f, bits: sum(f << (bits * j) for j in range(256 // bits))      # noqa: E731
    cases = SCALARS + [L, 2**253 - 1, 2**253 + 2**241, 2**254, 2**256 - 2**252 - 1, 2**256 - 1]
    cases += [pat(f, 16) % 2**256 for f in (0, 0x7fff, 0x8000, 0x8001, 0xffff)] + [pat(f, 12) % 2**256 for f in (0, 0x7ff, 0x800, 0xfff)]
    cases += [int.from_bytes(rng.bytes(32), "little") % L for _ in range(200)]
    rec_in = np.stack([word(c) for c in cases])
    out, ok = iss.selftest_primitive("recode65536", rec_in)
    assert (out == rec_in).all()
    assert list(ok) == [int(digits65536(c)[-1] <= 2**13 + 1) for c in cases]
    assert ok[:len(SCALARS)].all()
    out, ok = iss.selftest_primitive("recode4096", rec_in)
    assert ok.all() and (out == rec_in).all()
    # degenerate Elligator inputs, in either half of the 64 bytes
    ts = degenerate_field_inputs()
    uni = [(a, b) for a in ts for b in (0, 1, ts[0])] + [(b, a) for a in ts for b in (0, ts[0])]
    inp = np.stack([np.concatenate([word(a % 2**256), word(b % 2**256)]) for a, b in uni])
    out, _ = iss.selftest_primitive("from_uniform", inp)
    for k, row in enumerate(inp):
        assert out[k].tobytes() == R.from_uniform_bytes(row.tobytes()).compress(), ("from_uniform", hex(uni[k][0]), hex(uni[k][1]))
    # decompress: the even one of i and p - i has s^2 = -1, so u2 = 1 + s^2 = 0 and the inverse square root is taken of 0
    even_i = R.SQRT_M1 if R.SQRT_M1 % 2 == 0 else P - R.SQRT_M1
    enc = np.stack([word(v % 2**256) for v in [even_i] + ts])
    out, ok = iss.selftest_primitive("decompress_compress", enc)
    exp_ok = [R.decompress(e.tobytes()) is not None for e in enc]
    assert list(ok) == exp_ok and not ok[0]
    assert (out[ok == 1] == enc[ok == 1]).all()


def test_primitive_extremes_on_emulation(emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, _ = coracle.make_issuer(1)
    check_primitive_extremes(Issuer(sp, ip, None, max_batch=4, _binding=emu))


@pytest.mark.gpu
def test_primitive_extremes_on_gpu(coracle):
    from aeonflux_b200 import Issuer
    sp, ip, _ = coracle.make_issuer(1)
    check_primitive_extremes(Issuer(sp, ip, None, device=0, max_batch=4))
