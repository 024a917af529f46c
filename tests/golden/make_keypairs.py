"""Generates tests/golden/keypairs.json from the Python oracle: Keypair::derive (symmetric.rs:197-215) of seeded master secrets under
the system parameters of both bench issuers (bench_data/issuer4.bin, issuer16.bin).

    python tests/golden/make_keypairs.py

Holds: the master secrets -- all-zero, all-0xff, the bench fixture's (tests/golden/make_bench_fixture.py, whose keypair4.bin and
keypair16.bin it derives) and 30 seeded random ones -- and, per issuer file, the keypair a || a0 || a1 || pk of each.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle.pyoracle import aeonflux as A, ristretto as R  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
BENCH_SECRET = b"aeonflux-b200 bench keypair".ljust(64, b"\0")


def main():
    rng = A.ShakeRng(b"aeonflux_b200 keypair golden")
    secrets = [bytes(64), b"\xff" * 64, BENCH_SECRET] + [rng.fill(64) for _ in range(30)]
    out = {"master_secrets": [s.hex() for s in secrets], "keypairs": {}}
    for name in ("issuer4.bin", "issuer16.bin"):
        sp = A.SystemParameters.from_bytes(bench.load_issuer(name)[0])
        kps = []
        for s in secrets:
            k = A.SymmetricKeypair.derive(s, sp)
            kps.append((R.sc_to_bytes(k.a) + R.sc_to_bytes(k.a0) + R.sc_to_bytes(k.a1) + k.pk.compress()).hex())
        out["keypairs"][name] = kps
    with open(os.path.join(HERE, "keypairs.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
