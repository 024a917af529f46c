"""Generates tests/golden/sodium.json: what libsodium's ristretto255 functions return on the inputs of the libsodium
known-answer tests (tests/test_oracle_kats.py), so that those tests hold the oracle to libsodium on any machine.

    python tests/golden/make_sodium.py /path/to/libsodium.so        (a libsodium >= 1.0.18 built with ristretto255)
"""
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle.pyoracle import aeonflux as A, ristretto as R  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROUNDS = 60


def main(path):
    lib = ctypes.CDLL(path)
    assert lib.sodium_init() >= 0
    lib.sodium_version_string.restype = ctypes.c_char_p
    out = ctypes.create_string_buffer(32)
    rfc = json.load(open(os.path.join(HERE, "rfc9496.json")))
    mult = []
    for k in range(1, len(rfc["multiples"])):
        assert lib.crypto_scalarmult_ristretto255(out, k.to_bytes(32, "little"), R.BASEPOINT_COMPRESSED) == 0
        mult.append(out.raw.hex())
    valid = {g: [bool(lib.crypto_core_ristretto255_is_valid_point(bytes.fromhex(h))) for h in encs] for g, encs in rfc["invalid"].items()}
    h2g = []
    for e in rfc["hash_to_group"]:
        lib.crypto_core_ristretto255_from_hash(out, bytes.fromhex(e["input"]))
        h2g.append(out.raw.hex())
    # the same draws, in the same order, as test_against_libsodium
    rng = A.ShakeRng(b"sodium")
    rounds = []
    for _ in range(ROUNDS):
        r = {"b": rng.fill(32)}
        r["b_valid"] = bool(lib.crypto_core_ristretto255_is_valid_point(r["b"]))
        r["h"] = rng.fill(64)
        lib.crypto_core_ristretto255_from_hash(out, r["h"])
        r["from_hash"] = enc = out.raw
        r["s"] = R.sc_to_bytes(rng.scalar())
        assert lib.crypto_scalarmult_ristretto255(out, r["s"], enc) == 0
        r["scalarmult"] = out.raw
        r["h2"] = rng.fill(64)
        lib.crypto_core_ristretto255_from_hash(out, r["h2"])
        q = out.raw
        lib.crypto_core_ristretto255_sub(out, enc, q)
        r["sub"] = out.raw
        lib.crypto_core_ristretto255_scalar_reduce(out, r["h"])
        r["scalar_reduce"] = out.raw
        rounds.append({k: (v.hex() if isinstance(v, bytes) else v) for k, v in r.items()})
    data = {"source": "libsodium %s: crypto_scalarmult_ristretto255 and crypto_core_ristretto255_{is_valid_point,from_hash,sub,scalar_reduce}"
                      % lib.sodium_version_string().decode(),
            "rfc9496": {"multiples_1_to_15": mult, "invalid_is_valid_point": valid, "hash_to_group": h2g},
            "rounds": rounds}
    json.dump(data, open(os.path.join(HERE, "sodium.json"), "w"), indent=0)
    print("sodium.json:", data["source"], len(rounds), "rounds")


if __name__ == "__main__":
    main(sys.argv[1])
