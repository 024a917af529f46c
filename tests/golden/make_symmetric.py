"""Generates tests/golden/symmetric.json from the Python oracle: Plaintext::from(&[u8; 30]) (encoding.rs:56-70,
symmetric.rs:135-143), Keypair::encrypt and Keypair::decrypt (symmetric.rs:252-261,273-289) on seeded inputs.

    python tests/golden/make_symmetric.py

Holds: 32 seeded data strings, the zero string and the first seeded string whose M1 needs at least 20 candidate encodings, with
their Plaintext words; a keypair a || a0 || a1 and a second one; the ciphertexts under the first; and decrypt results, accepted and
rejected (wrong keypair, another item's E2, E1 and E2 swapped, an undecodable E1).
"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle.pyoracle import aeonflux as A, ristretto as R  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
UNDECODABLE = bytes([3]) + bytes(31)


def decrypt(kp, E1enc, E2enc):
    """-> (data hex, [M1, M2, m3] hex) or None for UndecryptableAttribute / an undecodable word."""
    E1, E2 = R.decompress(E1enc), R.decompress(E2enc)
    if E1 is None or E2 is None:
        return None
    try:
        pt = kp.decrypt(E1, E2)
    except ValueError:
        return None
    return {"data": pt.M1.compress()[1:31].hex(), "plaintext": [pt.M1.compress().hex(), pt.M2.compress().hex(), R.sc_to_bytes(pt.m3).hex()]}


def main():
    rng = A.ShakeRng(b"aeonflux_b200 symmetric golden")
    data = [rng.fill(30) for _ in range(32)] + [bytes(30)]
    while True:                                      # about 1 string in 250 needs 20 candidates or more
        d = rng.fill(30)
        if A.encode_to_group(d)[1] >= 19:            # the counter is the 0-based index of the accepted candidate
            data.append(d)
            break
    kp = A.SymmetricKeypair(rng.scalar(), rng.scalar(), rng.scalar(), None)
    other = A.SymmetricKeypair(rng.scalar(), rng.scalar(), rng.scalar(), None)
    items = []
    for d in data:
        pt = A.Plaintext.from_bytes30(d)
        E1, E2 = kp.encrypt(pt)
        items.append({"data": d.hex(), "candidates": A.encode_to_group(d)[1] + 1,
                      "plaintext": [pt.M1.compress().hex(), pt.M2.compress().hex(), R.sc_to_bytes(pt.m3).hex()],
                      "ciphertext": [E1.compress().hex(), E2.compress().hex()]})
    ct = [[bytes.fromhex(h) for h in it["ciphertext"]] for it in items]
    cases = []
    for i in range(len(items)):
        cases.append({"case": "honest", "keypair": "keypair", "ciphertext": [c.hex() for c in ct[i]]})
    for i in range(4):
        j = (i + 1) % len(items)
        cases.append({"case": "wrong keypair", "keypair": "other", "ciphertext": [c.hex() for c in ct[i]]})
        cases.append({"case": "another item's E2", "keypair": "keypair", "ciphertext": [ct[i][0].hex(), ct[j][1].hex()]})
        cases.append({"case": "E1 and E2 swapped", "keypair": "keypair", "ciphertext": [ct[i][1].hex(), ct[i][0].hex()]})
        cases.append({"case": "undecodable E1", "keypair": "keypair", "ciphertext": [UNDECODABLE.hex(), ct[i][1].hex()]})
    for c in cases:
        k = kp if c["keypair"] == "keypair" else other
        c["result"] = decrypt(k, *(bytes.fromhex(h) for h in c["ciphertext"]))

    def kp_hex(k):
        return (R.sc_to_bytes(k.a) + R.sc_to_bytes(k.a0) + R.sc_to_bytes(k.a1)).hex()
    out = {"keypair": kp_hex(kp), "other": kp_hex(other), "items": items, "decrypt": cases}
    with open(os.path.join(HERE, "symmetric.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
