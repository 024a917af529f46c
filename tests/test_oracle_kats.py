"""Pins the Python oracle to external known-answer tests (SURVEY 8c): Keccak via hashlib's SHA3,
merlin's published transcript + STROBE conformance vectors, RFC 9496 constants and generator
multiples, libsodium 1.0.20 ristretto255 (recorded answers), and the reference's own test verdicts."""
import hashlib
import json
import os

import pytest

from oracle.pyoracle import aeonflux as A, flat as F, merlin as M, ristretto as R, synth as S
from oracle.pyoracle.zkp import domain_sep, get_challenge

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_keccak_matches_sha3():
    for msg in (b"", b"abc", b"x" * 135):
        st = bytearray(200)
        m = bytearray(msg.ljust(136, b"\0"))
        m[len(msg)] ^= 0x06
        m[135] ^= 0x80
        for i in range(136):
            st[i] ^= m[i]
        M.keccak_f1600(st)
        assert bytes(st[:32]) == hashlib.sha3_256(msg).digest()


def test_merlin_kat():
    t = M.Transcript(b"test protocol")
    t.append_message(b"some label", b"some data")
    assert t.challenge_bytes(b"challenge", 32).hex() == "d5a21972d0d5fe320c0d263fac7fffb8145aa640af6e9bca177c03c7efcf0615"


def test_strobe_conformance():
    s = M.Strobe128(b"Conformance Test Protocol")
    s.meta_ad(b"ms", False); s.meta_ad(b"g", True); s.ad(bytes([99] * 1024), False); s.meta_ad(b"prf", False)
    p1 = s.prf(32, False)
    assert p1.hex() == "b48e645ca17c667fd5206ba57a6a228d72d8e1903814d3f17f622996d7cfefb0"
    s.meta_ad(b"key", False); s.key(p1, False); s.meta_ad(b"prf", False)
    assert s.prf(32, False).hex() == "07e45cce8078cee259e3e375bb85d75610e2d1e1201c5f645045a194edd49ff8"


def test_rfc9496_constants():
    assert R.D == 37095705934669439343138083508754565189542113879843219016388785533085940283555
    assert R.SQRT_M1 == 19681161376707505956807079304988542015446066515923890162744021073123829784752
    assert R.INVSQRT_A_MINUS_D == 54469307008909316920995813868745141605393597292927456921205312896311721017578
    assert R.ONE_MINUS_D_SQ == 1159843021668779879193775521855586647937357759715417654439879720876111806838
    assert R.D_MINUS_ONE_SQ == 40440834346308536858101042469323190826248399146238708352240133220865137265952
    assert R.BASEPOINT.compress() == R.BASEPOINT_COMPRESSED
    assert (R.BASEPOINT * 2).compress().hex() == "6a493210f7499cd17fecb510ae0cea23a110e8d5b901f8acadd3095c73a3b919"
    assert (R.BASEPOINT * 0).compress() == bytes(32)
    assert (R.BASEPOINT * R.L).compress() == bytes(32)


def test_rfc9496_appendix_a():
    """RFC 9496 Appendix A in full (tests/golden/rfc9496.json): the 16 generator multiples (A.1), all 29 invalid encodings by
    group (A.2), hash-to-group (A.3) -- Python oracle, and libsodium 1.0.20's answers (tests/golden/sodium.json) beside it."""
    g = json.load(open(os.path.join(GOLD, "rfc9496.json")))
    sod = _sodium()["rfc9496"]
    assert len(g["multiples"]) == 16
    for k, h in enumerate(g["multiples"]):
        assert (R.BASEPOINT * k).compress().hex() == h
        dec = R.decompress(bytes.fromhex(h))
        assert dec is not None and dec.compress().hex() == h
        if k:
            assert sod["multiples_1_to_15"][k - 1] == h
    assert sum(len(v) for v in g["invalid"].values()) == 29
    for group, encs in g["invalid"].items():
        for h, valid in zip(encs, sod["invalid_is_valid_point"][group], strict=True):
            assert R.decompress(bytes.fromhex(h)) is None, (group, h)
            assert not valid, (group, h)
    for e, sodium_out in zip(g["hash_to_group"], sod["hash_to_group"], strict=True):
        assert hashlib.sha512(e["label"].encode()).hexdigest() == e["input"]
        assert R.from_uniform_bytes(bytes.fromhex(e["input"])).compress().hex() == e["output"]
        assert sodium_out == e["output"]


def test_transcript_regression_vector_v1():
    t = M.Transcript(b"2019/1416 anonymous credential")
    domain_sep(t, b"2019/1416 presentation proof")
    t.append_message(b"scvar", b"z")
    t.append_message(b"ptvar", b"I"); t.append_message(b"val", R.BASEPOINT_COMPRESSED)
    t.append_message(b"blindcom", b"Z"); t.append_message(b"val", (R.BASEPOINT * 2).compress())
    assert R.sc_to_bytes(get_challenge(t, b"chal")).hex() == "6a1903a05ed023c17d4242f82dc8fcc25bb331a93bb54ab970eb4c1abc292f0e"


def _sodium():
    """libsodium's outputs on the inputs of these tests, recorded by tests/golden/make_sodium.py."""
    return json.load(open(os.path.join(GOLD, "sodium.json")))


def test_against_libsodium():
    rounds = _sodium()["rounds"]
    rng = A.ShakeRng(b"sodium")
    assert len(rounds) == 60
    for r in rounds:
        b = rng.fill(32)
        assert b.hex() == r["b"]
        assert (R.decompress(b) is not None) == r["b_valid"]
        h = rng.fill(64)
        assert h.hex() == r["h"]
        P = R.from_uniform_bytes(h)
        assert P.compress().hex() == r["from_hash"]
        s = rng.scalar()
        assert R.sc_to_bytes(s).hex() == r["s"]
        assert (P * s).compress().hex() == r["scalarmult"]
        h2 = rng.fill(64)
        assert h2.hex() == r["h2"]
        Q = R.from_uniform_bytes(h2)
        assert (P - Q).compress().hex() == r["sub"]
        assert R.sc_to_bytes(R.sc_from_wide(h)).hex() == r["scalar_reduce"]


def test_golden_prims():
    g = json.load(open(os.path.join(GOLD, "prims.json")))
    for e in g["decompress"]:
        assert (R.decompress(bytes.fromhex(e["in"])) is not None) == e["valid"]
    for e in g["from_uniform"]:
        assert R.from_uniform_bytes(bytes.fromhex(e["in"])).compress().hex() == e["out"]
    for e in g["scalarmult"][:4]:
        assert (R.decompress(bytes.fromhex(e["p"])) * int.from_bytes(bytes.fromhex(e["s"]), "little")).compress().hex() == e["out"]


def test_reference_test_verdicts():
    """Shapes and outcomes of the reference's own tests: presentation.rs:545-584 (accept),
    :618-638 (attribute swapped after issuance => reject), issuance.rs:271-295 (identity plaintext => reject)."""
    iss = S.make_issuer(1)
    it = S.make_item(iss, ("PS",), (), b"t-scalar1", 0)
    iss.verify(it["presentation"])
    # bad_credential_proof_1_scalar_revealed: present a different scalar than the MACed one
    rng = A.ShakeRng(b"t-bad")
    attrs = [("PS", rng.scalar())]
    p = A.presentation_prove(iss.system_parameters, iss.issuer_parameters, it["amac"], attrs, None, rng.scalar(),
                             [rng.scalar() for _ in range(3)], [])
    with pytest.raises(A.VerificationFailure):
        iss.verify(p)
    # issuance_proof_identity_plaintext
    iss6 = S.make_issuer(6)
    rng = A.ShakeRng(b"t-ident")
    pl = A.Plaintext.from_bytes30(bytes(30))
    assert pl.M1.is_identity()
    attrs = [("EP", pl), ("PS", rng.scalar()), ("PS", rng.scalar()), ("PP", rng.point()), ("PP", rng.point()), ("PS", rng.scalar())]
    proof, (amac, _) = iss6.issue(attrs, rng)
    with pytest.raises(A.VerificationFailure):
        A.issuance_verify(proof, iss6.system_parameters, iss6.issuer_parameters, amac, attrs)
    with pytest.raises(A.MacCreationError):
        iss6.issue(attrs[:5], rng)


def test_golden_presentations_python_oracle():
    g = json.load(open(os.path.join(GOLD, "readme4.json")))
    iss = S.make_issuer(4)
    assert iss.system_parameters.to_bytes().hex() == g["sysparams"]
    assert iss.amacs_key.to_bytes().hex() == g["secret"]
    e = g["items"][0]
    words = [bytes.fromhex(w) for w in e["words"]]
    v, tr = F.verify_flat(iss, bytes(e["kinds"]), words)
    assert v == e["verdict"] == 0 and tr["Z"].hex() == e["Z"] and [c.hex() for c in tr["commitments"]] == e["commitments"]
    for c in e["corrupted"][:3]:
        v, tr = F.verify_flat(iss, bytes(e["kinds"]), [bytes.fromhex(w) for w in c["words"]])
        assert v == c["verdict"] == 1


def test_encode_decode_and_encryption_roundtrip():
    """encoding.rs:91-103, symmetric.rs:298-310, encryption.rs:221-244."""
    sp = S.make_issuer(5).system_parameters
    rng = A.ShakeRng(b"t-enc")
    data = rng.fill(30)
    P, ctr = A.encode_to_group(data)
    d2, ctr2 = A.decode_from_group(P)
    assert d2 == data and ctr == ctr2
    kp, _ = A.SymmetricKeypair.generate(sp, rng)
    pt = A.Plaintext.from_bytes30(b"This is a tsunami alert test..")
    pe = A.encryption_prove(sp, pt, 1, kp, rng.scalar(), [rng.scalar() for _ in range(6)])
    dec = kp.decrypt(pe.E1, pe.E2)
    assert dec.M1 == pt.M1 and dec.M2 == pt.M2 and dec.m3 == pt.m3
    A.encryption_verify(pe, sp)
