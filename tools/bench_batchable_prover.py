#!/usr/bin/env python
"""The BatchableProof provers against the compact ones on one GPU, printed as one JSON line:
  - show vs show_batchable and issue vs issue_batchable, device-resident (afx_*_device, CUDA events, L2 flushed before each timed
    call, the two forms alternated) and end to end through the host calls (host buffers in and out);
  - the user-to-issuer pipeline show_batchable -> verify_batchable_rlc against show -> verify_batch, end to end;
  - README-4 at 65,536 items and S16 at 16,384 (C-oracle credentials, fresh rng bytes per item), and the GPU's name, power limit
    and SM clocks, queried in the same run.  Every output is checked: statuses 0, every verdict 0, no exact RLC chunk.
    python tools/bench_batchable_prover.py [--steps 5] [--rounds 3]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_symmetric import gpu_info  # noqa: E402

SHAPES = {"readme4": (4, b"SSPE", [0, 3], 2048, 32), "s16": (16, b"SSSSSSPP" + b"E" * 8, [0, 1] + list(range(8, 16)), 1024, 16)}


def show_inputs(orc, rk, hide, creds, draws, seed):
    """creds C-oracle credentials x draws fresh rng draws -> (kinds, show fields [n_in][count][32])."""
    kinds, _, issu, showin = orc.synth(rk, hide, b"bench-batchable", 0, creds, want_show_inputs=True)
    r0 = 3 + sum(3 if k == 3 else 1 for k in kinds) + (4 if 3 in kinds else 0)
    items = np.tile(showin, (draws, 1, 1))
    items[:, r0:] = np.random.default_rng(seed).integers(0, 256, items[:, r0:].shape, dtype=np.uint8)
    return kinds, issu, np.ascontiguousarray(items.transpose(1, 0, 2))


def run_shape(torch, coracle, name, steps, rounds):
    from aeonflux_b200 import Issuer, RequestBatch
    n, rk, hide, creds, draws = SHAPES[name]
    N = creds * draws
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    kinds, issu, fields = show_inputs(orc, rk, hide, creds, draws, 5)
    ik = bytes(0 if c == ord("S") else 2 for c in rk)
    rnd = np.random.default_rng(6).integers(0, 256, (N, n + 7, 64), dtype=np.uint8)
    req = RequestBatch.from_request(ik, np.ascontiguousarray(np.tile(issu[:, :n], (draws, 1, 1))), rnd)
    iss = Issuer(sp, ip, sk, device=0, max_batch=N)
    stream = torch.cuda.current_stream()
    s = stream.cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    d_show, d_req = torch.from_numpy(fields).cuda(), torch.from_numpy(np.ascontiguousarray(req.fields)).cuda()
    d_st = torch.empty(N, dtype=torch.uint8, device="cuda")
    n_out = {"show": iss.num_fields(kinds), "show_batchable": iss._b.L.afx_batchable_num_fields(n, kinds), "issue": n + 9, "issue_batchable": n + 11}
    d_out = {k: torch.empty((w, N, 32), dtype=torch.uint8, device="cuda") for k, w in n_out.items()}
    calls = {
        "show": lambda: iss.show_batch_device(kinds, N, d_show.data_ptr(), d_out["show"].data_ptr(), d_st.data_ptr(), s),
        "show_batchable": lambda: iss.show_batch_device(kinds, N, d_show.data_ptr(), d_out["show_batchable"].data_ptr(), d_st.data_ptr(), s, batchable=True),
        "issue": lambda: iss.issue_batch_device(ik, N, d_req.data_ptr(), d_out["issue"].data_ptr(), d_st.data_ptr(), s),
        "issue_batchable": lambda: iss.issue_batch_device(ik, N, d_req.data_ptr(), d_out["issue_batchable"].data_ptr(), d_st.data_ptr(), s, batchable=True),
    }
    device = {k: [] for k in calls}
    for _ in range(rounds):                                   # the compact and batchable forms alternate
        for k, fn in calls.items():
            device[k].append(bench.time_device(torch, stream, flush, fn, steps))
            assert int(d_st.sum().item()) == 0, k
    dev = {k: {"ms_per_call": [round(x, 3) for x in v], "items_per_s_best": round(N / (min(v) * 1e-3))} for k, v in device.items()}
    e2e, results = {}, {}
    for _ in range(rounds):
        for k in calls:
            t0 = time.perf_counter()
            if k.startswith("show"):
                res, st = iss.show_batch(kinds, fields, batchable=k.endswith("batchable"))
            else:
                res, st = iss.issue_batch(req, batchable=k.endswith("batchable"))
            e2e.setdefault(k, []).append(time.perf_counter() - t0)
            assert not st.any(), k
            results[k] = res
    e2e = {k: {"s": [round(x, 4) for x in v], "items_per_s_best": round(N / min(v))} for k, v in e2e.items()}
    assert (d_out["show_batchable"].cpu().numpy() == results["show_batchable"].fields).all()
    assert (d_out["issue_batchable"].cpu().numpy() == results["issue_batchable"].fields[n:]).all()
    pipe = {"show_then_verify_batch": [], "show_batchable_then_verify_batchable_rlc": []}
    for _ in range(rounds):
        t0 = time.perf_counter()
        res, _ = iss.show_batch(kinds, fields)
        assert not iss.verify_batch(res).any()
        t1 = time.perf_counter()
        res, _ = iss.show_batch(kinds, fields, batchable=True)
        v, exact = iss.verify_batchable_rlc(res, bytes(32))
        assert not v.any() and exact == 0
        t2 = time.perf_counter()
        pipe["show_then_verify_batch"].append(t1 - t0)
        pipe["show_batchable_then_verify_batchable_rlc"].append(t2 - t1)
    pipe = {k: {"s": [round(x, 4) for x in v], "items_per_s_best": round(N / min(v))} for k, v in pipe.items()}
    v, exact = iss.verify_batchable_rlc(results["issue_batchable"], bytes(32), issuance=True)
    assert not v.any() and exact == 0
    iss.close()
    return {"items": N, "device_resident": dev, "end_to_end": e2e, "pipeline_end_to_end": pipe}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    from oracle import coracle
    if not torch.cuda.is_available():
        raise SystemExit("bench_batchable_prover.py needs a CUDA device")
    coracle.build()
    info = gpu_info()
    out = {"gpu": info, "steps": args.steps, "rounds": args.rounds}
    for name in SHAPES:
        out[name] = run_shape(torch, coracle, name, args.steps, args.rounds)
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
