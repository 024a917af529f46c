#!/usr/bin/env python
"""End-to-end rate of issuing and showing over records of several shapes of one issuer, printed as one JSON line:
  - records/s of afx_issue_mixed_wire / afx_show_mixed_wire (the records bucketed by shape on the device, the outputs put back in
    record order on the device);
  - records/s of bucketing the same records on the host (a row gather of 32-byte words into one page-locked buffer per shape), one
    afx_issue_wire / afx_show_wire call per shape into page-locked outputs, and the outputs scattered back to record order;
  - for reference, records/s of one *_wire call over as many records of the first shape alone;
  - the device time of k_bucket_records and k_unbucket_records per call, and of every kernel of the call together (torch.profiler,
    in a run of its own after the timings);
  - the GPU's name, power limit and SM clocks, queried in the same run.
Workloads, README-4 issuer, `--records` records in page-locked memory (inputs and outputs), shuffled at random, max_batch = --records:
  issue3  requests of three request kind vectors ([0,0,2,2], [0,2,0,2], [2,2,2,2]) in equal parts;
  show4   show inputs of the four disclosure patterns of request SSPE in equal parts ([SS,PS,PP,SP], [PS,PS,PP,SP],
          [SS,SS,PP,SP], [PS,PS,PP,PP]), made on the device from credentials the device issued.
    python tools/bench_mixed_provers.py [--records 65536] [--steps 5] [--out result.json]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_mixed import kernel_times, rate  # noqa: E402
from bench_symmetric import gpu_info  # noqa: E402

REQUEST_KINDS = [bytes([0, 0, 2, 2]), bytes([0, 2, 0, 2]), bytes([2, 2, 2, 2])]
SHOW_PATTERNS = [bytes([1, 0, 2, 3]), bytes([0, 0, 2, 3]), bytes([1, 1, 2, 3]), bytes([0, 0, 2, 2])]


def requests_for(iss, kinds, count, seed):
    """count requests of request kinds `kinds`, item-major [count][3n + 14][32]: random scalar attributes (< 2^252), point attributes
    from the engine's from_uniform_bytes primitive, random rng words."""
    rng = np.random.default_rng(seed)
    n = len(kinds)
    attrs = rng.integers(0, 256, (count, n, 32), dtype=np.uint8)
    attrs[:, :, 31] &= 0x0f
    pts = [i for i, k in enumerate(kinds) if k == 2]
    if pts:
        enc, _ = iss.selftest_primitive("from_uniform", rng.integers(0, 256, (count * len(pts), 64), dtype=np.uint8))
        attrs[:, pts] = enc.reshape(count, len(pts), 32)
    return np.ascontiguousarray(np.concatenate([attrs, rng.integers(0, 256, (count, 2 * (n + 7), 32), dtype=np.uint8)], axis=1))


def show_inputs_on_device(iss, kinds, count, seed, keypair_file="keypair4.bin"):
    """count distinct show inputs of shape `kinds`, item-major [count][afx_show_num_fields][32]: random attributes issued into
    credentials on the device (as bench.synthesize_on_device makes them), one symmetric keypair, random rng words."""
    rng = np.random.default_rng(seed)
    kinds = bytes(kinds)
    n = len(kinds)
    h_s, h_p = sum(k == 1 for k in kinds), sum(k == 3 for k in kinds)
    issue_kinds = bytes(0 if k in (0, 1) else 2 for k in kinds)
    req = requests_for(iss, issue_kinds, count, seed)
    cred, status = iss.issue_wire(issue_kinds, req)
    assert not status.any()
    rows = [cred[:, n:n + 3]]                               # t, U, V
    extra = iss.selftest_primitive("from_uniform", rng.integers(0, 256, (max(h_p, 1) * count, 64), dtype=np.uint8))[0].reshape(count, -1, 32)
    m3 = rng.integers(0, 256, (count, max(h_p, 1), 32), dtype=np.uint8)
    m3[:, :, 31] &= 0x0f
    p = 0
    for i, k in enumerate(kinds):
        if k == 3:      # a plaintext: M1 (the issued point attribute), M2, m3
            rows += [req[:, i:i + 1], extra[:, p:p + 1], m3[:, p:p + 1]]
            p += 1
        else:
            rows.append(req[:, i:i + 1])
    if h_p:
        kp = np.frombuffer(open(os.path.join(ROOT, "bench_data", keypair_file), "rb").read(), np.uint8).reshape(1, 4, 32)
        rows.append(np.broadcast_to(kp, (count, 4, 32)))
    rows.append(rng.integers(0, 256, (count, 2 * (1 + 3 + h_s + 6 * h_p), 32), dtype=np.uint8))
    out = np.ascontiguousarray(np.concatenate(rows, axis=1))
    assert out.shape[1] == iss._b.L.afx_show_num_fields(n, kinds)
    return out


def pinned_copy(iss, a):
    p = iss.host_array(a.shape)
    p[:] = a
    return p


def shuffled(counts, seed):
    return np.random.default_rng(seed).permutation(np.repeat(np.arange(len(counts), dtype=np.uint8), counts)).astype(np.uint8)


def host_bucketed(iss, issue, kinds_list, pinned_in, in_off, order, buckets, outs, out_words, out_off):
    """Host bucketing into page-locked buckets, one wire call per shape into page-locked outputs, outputs and status scattered back
    to record order."""
    words_in, words_out = pinned_in.reshape(-1, 32), out_words.reshape(-1, 32)
    status = np.empty(len(order), np.uint8)
    for s, kinds in enumerate(kinds_list):
        pos = np.nonzero(order == s)[0]
        b, o = buckets[s][:len(pos)], outs[s][:len(pos)]
        np.take(words_in, (in_off[pos] // 32)[:, None] + np.arange(b.shape[1])[None, :], axis=0, out=b)
        _, st = iss.issue_wire(kinds, b, out=o) if issue else iss.show_wire(kinds, b, out=o)
        words_out[(out_off[pos] // 32)[:, None] + np.arange(o.shape[1])[None, :]] = o
        status[pos] = st
    return status


def workload(iss, issue, kinds_list, counts, seed, steps):
    from aeonflux_b200 import _binding as B
    pools = [requests_for(iss, k, c, seed + s) if issue else show_inputs_on_device(iss, k, c, seed + s)
             for s, (k, c) in enumerate(zip(kinds_list, counts))]
    from aeonflux_b200.shard import interleave_records
    order = shuffled(counts, seed)
    blob, in_off = interleave_records(pools, order)
    pinned_in = pinned_copy(iss, blob)
    in_off = in_off.astype(np.int64)
    out_sizes = B.mixed_record_bytes(iss._b, kinds_list, "issuance" if issue else "presentation")
    out_off = B.record_offsets(out_sizes, order)
    out = iss.host_array(int(out_off[-1]))
    out_host = iss.host_array(int(out_off[-1]))
    buckets = [iss.host_array(p.shape) for p in pools]
    outs = [iss.host_array((len(p), int(sz) // 32, 32)) for p, sz in zip(pools, out_sizes)]
    fn = iss.issue_mixed_wire if issue else iss.show_mixed_wire
    mixed = lambda: fn(kinds_list, pinned_in, order, out=out)      # noqa: E731
    hb = lambda: host_bucketed(iss, issue, kinds_list, pinned_in, in_off, order, buckets, outs, out_host, out_off[:-1])   # noqa: E731
    _, st = mixed()
    assert not st.any(), "honest inputs rejected"
    assert (hb() == st).all() and (out_host == out).all(), "the mixed call differs from the per-shape wire calls"
    n = len(order)
    w = {"shapes": [list(k) for k in kinds_list], "counts": list(map(int, counts)), "input_bytes": int(pinned_in.size),
         "output_bytes": int(out.size), "mixed_wire": rate(mixed, n, steps), "host_bucketed_wire_per_shape": rate(hb, n, steps)}
    # reference: one wire call over as many records of the first shape
    one = pinned_copy(iss, np.concatenate([pools[0]] * ((n + len(pools[0]) - 1) // len(pools[0])))[:n])
    one_out = iss.host_array((n, int(out_sizes[0]) // 32, 32))
    wire = (lambda: iss.issue_wire(kinds_list[0], one, out=one_out)) if issue else (lambda: iss.show_wire(kinds_list[0], one, out=one_out))
    w["single_shape_wire"] = rate(wire, n, steps)
    return w, mixed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from aeonflux_b200 import Issuer
    if not torch.cuda.is_available():
        raise SystemExit("bench_mixed_provers.py needs a CUDA device")
    N = args.records
    sp, ip, sk = bench.load_issuer("issuer4.bin")
    iss = Issuer(sp, ip, sk, device=0, max_batch=N)
    result = {"gpu": gpu_info(), "records": N, "max_batch": N, "steps": args.steps, "workloads": {}}
    calls = {}
    for name, issue, kinds_list, seed in (("issue3", True, REQUEST_KINDS, 800), ("show4", False, SHOW_PATTERNS, 900)):
        counts = [N // len(kinds_list) + (1 if s < N % len(kinds_list) else 0) for s in range(len(kinds_list))]
        result["workloads"][name], calls[name] = workload(iss, issue, kinds_list, counts, seed, args.steps)
    # device time per call (profiler runs after every timing)
    for name, fn in calls.items():
        k = kernel_times(torch, fn, ["k_bucket_records", "k_unbucket_records"])
        k["all_kernels_us_per_call"] = all_kernel_time(torch, fn)
        result["workloads"][name]["kernels"] = k
    result["gpu_after"] = gpu_info()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def all_kernel_time(torch, fn):
    """Device time of every kernel of one call (memsets and copies excluded), averaged over three calls."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if "afx::k_" in e.key) / 3.0


if __name__ == "__main__":
    main()
