#!/usr/bin/env python
"""Rates of the batch attribute-encryption calls (Plaintext::from, Keypair::encrypt, Keypair::decrypt, Keypair::derive) on one GPU,
printed as one JSON line:
  - device-resident items/s of afx_encode_plaintexts_device / afx_encrypt_device / afx_decrypt_device / afx_derive_keypairs_device
    (CUDA events, warmed up, inputs of 2^20 items = 30 + 96 + 64 + 64 MB, larger than the L2, are read once per call);
  - end-to-end items/s through the host calls (host buffers in and out, passes of max_batch);
  - the C oracle's rate on all host cores over a prefix of the same inputs;
  - algorithmic IMAD per item from bench.py's cost model and the resulting fraction of the IMAD peak;
  - the GPU's name, power limit and SM clocks, queried in the same run.
    python tools/bench_symmetric.py [--items 1048576] [--steps 5] [--cpu-items 65536]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from bench import ADD, COMPRESS, DBL, DECOMPRESS, ELLIGATOR2, MADD, TABLE  # noqa: E402

# Limb-products per item.  A constant-schedule ladder adds all 64 radix-16 digits: 252 doublings and 64 additions.  Encoding tries
# about 4 candidate encodings on average (the warp waits for its slowest lane, which the model does not count).  Derive is pk on the
# radix-16 comb: 64 mixed adds per generator, no doublings.
LADDER_CT = 252 * DBL + 64 * ADD
MODEL = {
    "encode": 4 * DECOMPRESS + ELLIGATOR2 + COMPRESS,
    "encrypt": 2 * DECOMPRESS + TABLE + 2 * LADDER_CT + ADD + 2 * COMPRESS,
    "decrypt": 2 * DECOMPRESS + 2 * TABLE + 2 * LADDER_CT + ADD + ELLIGATOR2 + 2 * COMPRESS,
    "derive": 3 * 64 * MADD + COMPRESS,
}
MODEL_NOTE = ("field multiplications only: the SHA-512 compressions (one in encode and decrypt, three in derive) are 64-bit logic "
              "work the model does not count")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True)
    name, power, sm, sm_max = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(power), "sm_mhz": float(sm), "sm_max_mhz": float(sm_max)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--cpu-items", type=int, default=65536)
    args = ap.parse_args()
    import torch
    from aeonflux_b200 import Issuer
    from tests import symoracle
    from tests.symoracle import derive as derive_oracle
    if not torch.cuda.is_available():
        raise SystemExit("bench_symmetric.py needs a CUDA device")
    N = args.items
    sp, ip, _ = bench.load_issuer("issuer4.bin")
    kp = open(os.path.join(ROOT, "bench_data", "keypair4.bin"), "rb").read()[:96]
    iss = Issuer(sp, ip, None, device=0, max_batch=N)
    rng = np.random.default_rng(2024)
    data = rng.integers(0, 256, (N, 30), dtype=np.uint8)
    secrets = rng.integers(0, 256, (N, 64), dtype=np.uint8)
    d_data = torch.from_numpy(data).cuda()
    d_ms = torch.from_numpy(secrets).cuda()
    d_kp = torch.empty((4, N, 32), dtype=torch.uint8, device="cuda")
    d_pt = torch.empty((3, N, 32), dtype=torch.uint8, device="cuda")
    d_ct = torch.empty((2, N, 32), dtype=torch.uint8, device="cuda")
    d_back = torch.empty((N, 30), dtype=torch.uint8, device="cuda")
    d_st = torch.empty(N, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    calls = {
        "encode": lambda: iss.encode_plaintexts_device(N, d_data.data_ptr(), d_pt.data_ptr(), d_st.data_ptr(), s),
        "encrypt": lambda: iss.encrypt_device(kp, N, d_pt.data_ptr(), d_ct.data_ptr(), d_st.data_ptr(), s),
        "decrypt": lambda: iss.decrypt_device(kp, N, d_ct.data_ptr(), d_back.data_ptr(), d_st.data_ptr(), None, s),
        "derive": lambda: iss.derive_keypairs_device(N, d_ms.data_ptr(), d_kp.data_ptr(), s),
    }
    info = gpu_info()
    device = {}
    for name, fn in calls.items():
        fn()                                                   # warm-up (and the inputs of the next call)
        torch.cuda.synchronize()
        assert int(d_st.sum()) == 0, name                     # derive has no status: its keypairs are checked below
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(args.steps):
                fn()
            e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        device[name] = {"ms_per_call": round(ms, 3), "items_per_s": round(N / (ms * 1e-3))}
    assert (d_back.cpu().numpy() == data).all()
    info_after = gpu_info()
    e2e = {}
    t0 = time.perf_counter(); pts, st = iss.encode_plaintexts(data); t1 = time.perf_counter()
    cts, st1 = iss.encrypt(kp, pts); t2 = time.perf_counter()
    back, st2 = iss.decrypt(kp, cts); t3 = time.perf_counter()
    kps = iss.derive_keypairs(secrets); t4 = time.perf_counter()
    assert not (st.any() or st1.any() or st2.any()) and (back == data).all()
    assert (kps == d_kp.cpu().numpy().transpose(1, 0, 2).reshape(N, 128)).all()
    for name, dt in (("encode", t1 - t0), ("encrypt", t2 - t1), ("decrypt", t3 - t2), ("derive", t4 - t3)):
        e2e[name] = {"s": round(dt, 3), "items_per_s": round(N / dt)}
    cores = len(os.sched_getaffinity(0))
    M = min(args.cpu_items, N)
    opt, s_enc = symoracle.encode(data[:M], threads=cores)
    oct_, _, s_ecr = symoracle.encrypt(kp, opt, threads=cores)
    odata, _, _, s_dec = symoracle.decrypt(kp, oct_, threads=cores)
    okp, s_der = derive_oracle.derive(sp, ip, secrets[:M], threads=cores)
    assert (opt == pts[:M]).all() and (oct_ == cts[:M]).all() and (odata == data[:M]).all() and (okp == kps[:M]).all()
    cpu = {name: {"items": M, "items_per_s": round(M / sec)}
           for name, sec in (("encode", s_enc), ("encrypt", s_ecr), ("decrypt", s_dec), ("derive", s_der))}
    imad_peak = 148 * 64 * info["sm_max_mhz"] * 1e6
    model = {}
    for name, lp in MODEL.items():
        imad = 2 * lp
        model[name] = {"imad_per_item": int(imad), "fraction_of_imad_peak": round(imad * device[name]["items_per_s"] / imad_peak, 3)}
    print(json.dumps({"items": N, "steps": args.steps, "gpu": info, "gpu_after": info_after, "device_resident": device, "end_to_end": e2e,
                      "cpu_oracle": dict(cpu, cores=cores), "work_model": model, "work_model_note": MODEL_NOTE, "imad_peak_per_s": imad_peak}))
    iss.close()


if __name__ == "__main__":
    main()
