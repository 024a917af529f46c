#!/usr/bin/env python
"""End-to-end rate of verifying presentations of several disclosure patterns of one issuer, printed as one JSON line:
  - records/s of afx_verify_presentations_mixed_wire (the records bucketed by shape on the device);
  - records/s of bucketing the same records on the host (a row gather of 32-byte words into one page-locked buffer per shape) plus
    one afx_verify_presentations_wire call per shape, verdicts scattered back to record order;
  - records/s of afx_stream_push + afx_stream_flush with every shape registered on the one context;
  - the device time of k_bucket_records and k_unbucket_records per call (torch.profiler, in a run of its own after the timings);
  - for reference, records/s of one afx_verify_presentations_wire call over as many records of the README-4 shape alone;
  - the GPU's name, power limit and SM clocks, queried in the same run.
Workloads: `--records` README-4-issuer presentations (distinct, made on the device) in page-locked memory, shuffled at random:
  mix4  the four disclosure patterns of request SSPE in equal parts ([SS,PS,PP,SP], [PS,PS,PP,SP], [SS,SS,PP,SP], [PS,PS,PP,PP]);
  mix2  [SS,PS,PP,SP] and [PS,PS,PP,PP], 50:50.
Every call verifies the whole set (58 MB for mix4, more than the 126 MB L2 holds together with the workspace), max_batch = --records.
    python tools/bench_mixed.py [--records 65536] [--steps 5] [--out result.json]"""
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

PATTERNS = {"mix4": [bytes([1, 0, 2, 3]), bytes([0, 0, 2, 3]), bytes([1, 1, 2, 3]), bytes([0, 0, 2, 2])],
            "mix2": [bytes([1, 0, 2, 3]), bytes([0, 0, 2, 2])]}


def workload(torch, iss, patterns, n, seed):
    """(pools, order, pinned blob, offsets): n distinct presentations, n / len(patterns) per pattern, interleaved at random."""
    from aeonflux_b200.shard import interleave_records
    per = n // len(patterns)
    pools = []
    for k, kinds in enumerate(patterns):
        dev = bench.synthesize_on_device(torch, iss, per, seed + k, torch.cuda.current_stream(), kinds, "keypair4.bin")
        pools.append(np.ascontiguousarray(dev.cpu().numpy().transpose(1, 0, 2)))
        del dev
    order = np.random.default_rng(seed).permutation(np.repeat(np.arange(len(patterns), dtype=np.uint8), per)).astype(np.uint8)
    blob, offsets = interleave_records(pools, order)
    pinned = iss.host_array(blob.shape)
    pinned[:] = blob
    return pools, order, pinned, offsets


def host_bucketed(iss, patterns, pinned, offsets, order, buckets):
    """Host bucketing into the page-locked buckets, one wire call per shape, verdicts back in record order."""
    words = pinned.reshape(-1, 32)
    out = np.empty(len(order), np.uint8)
    for s, kinds in enumerate(patterns):
        pos = np.nonzero(order == s)[0]
        b = buckets[s][:len(pos)]
        nf = b.shape[1]
        np.take(words, ((offsets[pos] // 32).astype(np.int64)[:, None] + np.arange(nf)[None, :]), axis=0, out=b)
        out[pos] = iss.verify_wire(kinds, b)
    return out


def streamed(ms, shape_ids, pinned, offsets, order):
    v = np.empty(len(order), np.uint8)
    ms.push(pinned, offsets, shape_ids[order], v)
    ms.flush()
    return v


def rate(fn, n, steps):
    fn()                                    # warm-up: shapes compiled, workspace and staging allocated
    fn()
    t = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
    return {"records_per_s": n / float(np.median(t)), "ms_median": 1e3 * float(np.median(t)), "ms_min": 1e3 * min(t), "ms_max": 1e3 * max(t)}


def kernel_times(torch, fn, names):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
    res = {}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                res[k] = {"us_per_call": e.device_time_total / 3.0, "launches_per_call": e.count / 3.0}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from aeonflux_b200 import Issuer
    from aeonflux_b200.shard import MixedStream
    if not torch.cuda.is_available():
        raise SystemExit("bench_mixed.py needs a CUDA device")
    N = args.records
    sp, ip, sk = bench.load_issuer("issuer4.bin")
    iss = Issuer(sp, ip, sk, device=0, max_batch=N)
    result = {"gpu": gpu_info(), "records": N, "max_batch": N, "steps": args.steps, "workloads": {}}
    for wi, (name, patterns) in enumerate(PATTERNS.items()):
        pools, order, pinned, offsets = workload(torch, iss, patterns, N, 500 + 10 * wi)
        buckets = [iss.host_array((N, p.shape[1], 32)) for p in pools]
        ms = MixedStream()
        shape_ids = np.array([ms.add_shape(iss, k) for k in patterns], np.uint8)
        mixed = lambda: iss.verify_mixed_wire(patterns, pinned, order)      # noqa: E731
        v = mixed()
        assert not v.any(), "honest presentations rejected"
        assert (host_bucketed(iss, patterns, pinned, offsets, order, buckets) == v).all()
        assert (streamed(ms, shape_ids, pinned, offsets, order) == v).all()
        w = {"patterns": [list(k) for k in patterns], "bytes": int(pinned.size),
             "mixed_wire": rate(mixed, N, args.steps),
             "host_bucketed_wire_per_shape": rate(lambda: host_bucketed(iss, patterns, pinned, offsets, order, buckets), N, args.steps),
             "stream_one_context": rate(lambda: streamed(ms, shape_ids, pinned, offsets, order), N, args.steps)}
        ms.close()
        result["workloads"][name] = w
        del pools, buckets
    # reference: the same number of records of one shape in one wire call
    kinds = PATTERNS["mix4"][0]
    dev = bench.synthesize_on_device(torch, iss, N, 600, torch.cuda.current_stream(), kinds, "keypair4.bin")
    one = iss.host_array((N, iss.num_fields(kinds), 32))
    one[:] = dev.cpu().numpy().transpose(1, 0, 2)
    del dev
    result["single_shape_wire_readme4"] = rate(lambda: iss.verify_wire(kinds, one), N, args.steps)
    # device time of the bucketing kernels (profiler run after every timing)
    pools, order, pinned, offsets = workload(torch, iss, PATTERNS["mix4"], N, 700)
    result["kernels_mix4"] = kernel_times(torch, lambda: iss.verify_mixed_wire(PATTERNS["mix4"], pinned, order),
                                          ["k_bucket_records", "k_unbucket_records"])
    result["gpu_after"] = gpu_info()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
