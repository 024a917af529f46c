#!/usr/bin/env python
"""bench.py -- presentations verified/sec (Issuer::verify, 4 attributes) on N B200s, with the integer-pipe roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one pass of the hot path over one batch of B = 65,536 README-4 presentations per GPU (BASELINE.json configs[1]).
  value   device-resident: every rank verifies its own 65,536 items already in HBM (afx_verify_presentations_device, CUDA events on
          the launching stream, L2 flushed between steps), max over ranks;
  e2e     the product's multi-GPU path on ONE global batch of N x 65,536 items in host memory: ShardedIssuer.verify_wire --
          contiguous slice per rank -> afx_verify_presentations_wire (H2D of the slice, kernels, D2H of the verdicts) -> accept /
          reject bitmap all-gathered (NCCL) -- every rank ends up with all N x 65,536 verdicts, inside the timed region.
secondary (reported beside the headline):
  stream_config5   BASELINE configs[4]: an item-mixed stream of 2^22 presentations (README-4 / S16 50:50, 1 % corrupted), rank r
                   pushing its contiguous slice through afx_stream_* (page-locked double buffers per shape, asynchronous wire
                   submits), bitmap gathered; the CPU port's rate on a sample of the same stream beside it; at every N;
  configs[2], configs[3] (N = 1): Issuer::issue, CredentialIssuance::verify, S16 Issuer::verify with host-buffer e2e, per-kernel
                   fraction of the IMAD peak and a CPU leg; AnonymousCredential::show and the BatchableProof modes.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KINDS_README4 = bytes([1, 0, 2, 3])   # [SecretScalar, PublicScalar, PublicPoint, SecretPoint]  (README.md:44-117, attrs 0 and 3 hidden)
KINDS_S16 = bytes([1, 1, 0, 0, 0, 0, 2, 2] + [3] * 8)
WORDS, WORDS_S16 = 28, 143
L_ORDER = 2**252 + 27742317777372353535851937790883648493

# One config object for BOTH arms (native and --impl reference): the driver compares them.
CONFIG = {"workload": "batch Issuer::verify of 65,536 README-4 presentations [SS,PS,PP,SP] per GPU (BASELINE configs[1])",
          "batch_per_gpu": 65536, "kinds": list(KINDS_README4), "bytes_per_item": WORDS * 32,
          "l2": "GPU arm: 256 MiB flush write between timed steps, and the 1.2 GB workspace of a step exceeds the L2; CPU arm: n/a",
          "input": "GPU arm: 65,536 distinct presentations per GPU, issued and shown on the device from random attributes (afx_issue -> "
                   "afx_show), a sample cross-checked against the CPU oracle; CPU arm: 8,192 distinct presentations from the oracle's prover, "
                   "tiled to the 65,536-item batch (its schedule does not depend on the item)"}

# ---- algorithmic work model (SURVEY 8d): limb-products per field op, 1 limb-product = 2 IMAD issue slots (IMAD.WIDE is half rate,
# measured: profiles/r01_microbench_imad.json) ----------------------------------------------------------------------------------
S_LP, M_LP = 44, 72
DBL, ADD, MADD = 4 * S_LP + 4 * M_LP, 8 * M_LP, 7 * M_LP
DECOMPRESS, COMPRESS = 258 * S_LP + 24 * M_LP, 256 * S_LP + 30 * M_LP
TABLE = DBL + 7 * ADD
ELLIGATOR2 = 2 * (254 * S_LP + 30 * M_LP) + ADD          # RistrettoPoint::from_uniform_bytes: two Elligator maps and one addition
KECCAK_ALU_OPS = 4560                                     # 32-bit logic ops of one Keccak-f[1600] (24 rounds x ~190; DESIGN.md section 4)


def work_model(kinds):
    """Algorithmic limb-products per item and per stage for a presentation shape (minimal schedule of SURVEY 8d)."""
    n = len(kinds)
    r_s, h_s = sum(k == 0 for k in kinds), sum(k == 1 for k in kinds)
    r_p, h_p = sum(k == 2 for k in kinds), sum(k == 3 for k in kinds)
    n_dec = 3 + n + r_p + 7 * h_p
    n_msm = 2 + h_s + r_s + r_p + 5 * h_p
    var_terms = 1 + 2 + h_s + r_s + r_p + h_p * (1 + 2 + 2 + 3 + 1)
    con_terms = 1 + 2 + 2 * h_s + r_s + r_p + h_p * (3 + 1 + 0 + 1 + 2)
    points = n_dec * DECOMPRESS + (var_terms - 1) * TABLE + 2 * h_p * COMPRESS
    amac = 252 * DBL + (2 + n) * (7 + 64) * ADD + r_s * 64 * MADD + (r_s + r_p + 2) * ADD + COMPRESS + TABLE
    msm = n_msm * 253 * DBL + var_terms * (253 / 6) * ADD + con_terms * (253 / 9) * MADD + n_msm * COMPRESS
    total = points + amac + msm
    return {"points": points, "amac": amac, "msm": msm, "total": total}


def issuance_verify_model(n_s, n_p):
    """CredentialIssuance::verify, n = n_s scalar + n_p point attributes (SURVEY 8d's issuance rows, same costs): decompress U, V and
    the point attributes; tU = t*U (variable base); M_i = m_i*G_m[i] (constant base) for the scalar attributes; three MSMs with
    3, n + 4 and n + 4 terms (constant bases: 3 + (n + 4) + 1, variable: U, tU, M_i x n, V); compress tU, the scalar M_i and the three
    commitments."""
    n = n_s + n_p
    var, con = 3 + n, 3 + (n + 4) + 1
    points = (2 + n_p) * DECOMPRESS + var * TABLE
    ladders = (253 * DBL + (253 / 6) * ADD + COMPRESS) + n_s * ((253 / 9) * MADD + COMPRESS) \
        + 3 * 253 * DBL + var * (253 / 6) * ADD + con * (253 / 9) * MADD + 3 * COMPRESS
    return {"points": points, "msm": ladders, "total": points + ladders}


def issue_model(n_s, n_p):
    """Issuer::issue = Amac::tag + ProofOfIssuance::prove with every scalar secret (constant schedule, radix-16 digits, no digit skipped:
    64 additions per term): U by two Elligator maps; M_i = m_i*G_m[i] on the comb (64 madd); V = W + (x0 + x1 t)*U + sum y_i*M_i with the
    scalar-attribute terms folded onto G_m[i]; tU; the three blinding commitments (C_W: 2 constant terms, I: 3 + n constant terms -- comb, no
    doublings; V: U, tU and the point attributes variable, G_w and the scalar attributes' G_m[i] constant); compress U, V, tU, the scalar
    M_i and the three commitments."""
    n = n_s + n_p
    points = n_p * DECOMPRESS + ELLIGATOR2 + COMPRESS + (2 + n_p) * TABLE
    ladders = n_s * 64 * MADD \
        + 252 * DBL + (1 + n_p) * 64 * ADD + n_s * 64 * MADD + ADD \
        + 252 * DBL + 64 * ADD \
        + (2 + 3 + n) * 64 * MADD + 252 * DBL + (2 + n_p) * 64 * ADD + (1 + n_s) * 64 * MADD \
        + (2 + n_s + 3) * COMPRESS
    return {"points": points, "msm": ladders, "total": points + ladders}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md).  Started before the warm-up (nvidia-smi needs a moment to
    come up, longer on an 8-GPU box) and polled every 25 ms; rows are time-stamped on arrival and summary() only uses those
    that arrived inside the marked timed windows."""

    def __init__(self, index):
        self.index, self.rows, self.proc, self.windows = index, [], None, []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.rows.append((time.time(), line)) for line in self.proc.stdout], daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def window(self):
        sampler = self

        class _W:
            def __enter__(self):
                self.t0 = time.time()

            def __exit__(self, *a):
                sampler.windows.append((self.t0, time.time()))
        return _W()

    def stop(self):
        if self.proc:
            time.sleep(0.05)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if not any(a <= ts <= b + 0.03 for a, b in self.windows):
                continue
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"], "samples": 0, "rows_total": len(self.rows)}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "windows": "device-resident and end-to-end timed regions"}


def load_issuer(name):
    blob = open(os.path.join(ROOT, "bench_data", name), "rb").read()
    n = int.from_bytes(blob[:4], "little")
    a = 32 * (9 + 2 * n) + 4 if n >= 3 else 32 * (12 + n) + 4
    return blob[:a], blob[a:a + 64], blob[a + 64:]


def load_fixture(batch):
    pres = np.fromfile(os.path.join(ROOT, "bench_data", "readme4_1024.bin"), np.uint8).reshape(-1, WORDS, 32)
    sp, ip, sk = load_issuer("issuer4.bin")
    reps = (batch + len(pres) - 1) // len(pres)
    items = np.tile(pres, (reps, 1, 1))[:batch]
    return sp, ip, sk, items


def synthesize_on_device(torch, issuer, B, seed, stream, kinds=KINDS_README4, keypair_file="keypair4.bin"):
    """B DISTINCT honest presentations of shape `kinds` made on the GPU itself: random attributes (points through the engine's
    from_uniform_bytes primitive) -> Issuer::issue (credentials) -> AnonymousCredential::show with the hidden kinds hidden (fresh z
    and blindings per item, one symmetric keypair).  Returns the device-resident struct-of-arrays batch [n_fields][B][32].
    (Needs no CPU oracle; a sample is cross-checked against it afterwards.)"""
    rng = np.random.default_rng(seed)
    s = stream.cuda_stream
    kinds = bytes(kinds)
    n = len(kinds)
    h_s, h_p = sum(k == 1 for k in kinds), sum(k == 3 for k in kinds)

    def rand_words(k):
        return torch.from_numpy(rng.integers(0, 256, (k, B, 32), dtype=np.uint8)).cuda()

    def rand_scalars(k):
        w = rng.integers(0, 256, (k, B, 32), dtype=np.uint8); w[:, :, 31] &= 0x0f       # < 2^252 < l
        return torch.from_numpy(w).cuda()

    n_pts = sum(k == 2 for k in kinds) + 2 * h_p
    pts_host, _ = issuer.selftest_primitive("from_uniform", rng.integers(0, 256, (max(n_pts, 1) * B, 64), dtype=np.uint8))
    pts = torch.from_numpy(pts_host.reshape(max(n_pts, 1), B, 32)).cuda()
    sc = rand_scalars(sum(k in (0, 1) for k in kinds) + h_p)                            # scalar attributes, then one m3 per plaintext
    status = torch.empty(B, dtype=torch.uint8, device="cuda")
    attr, show_attr, pi, si = [], [], 0, 0
    m3_base = sum(k in (0, 1) for k in kinds)
    hp_seen = 0
    for k in kinds:
        if k in (0, 1):
            attr.append(sc[si]); show_attr.append(sc[si:si + 1]); si += 1
        elif k == 2:
            attr.append(pts[pi]); show_attr.append(pts[pi:pi + 1]); pi += 1
        else:    # a plaintext (M1, M2, m3): it enters the aMAC through M1 (amacs.rs:241)
            attr.append(pts[pi]); show_attr.append(torch.stack([pts[pi], pts[pi + 1], sc[m3_base + hp_seen]])); pi += 2; hp_seen += 1
    issue_kinds = bytes(0 if k in (0, 1) else 2 for k in kinds)
    req = torch.cat([torch.stack(attr), rand_words(2 * (n + 7))])
    cred = torch.empty((n + 9, B, 32), dtype=torch.uint8, device="cuda")
    issuer.issue_batch_device(issue_kinds, B, req.data_ptr(), cred.data_ptr(), status.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(status.sum().item()) == 0
    parts = [cred[0:3]] + show_attr
    if h_p:
        kp = np.frombuffer(open(os.path.join(ROOT, "bench_data", keypair_file), "rb").read(), np.uint8).reshape(4, 1, 32)
        parts.append(torch.from_numpy(np.ascontiguousarray(np.broadcast_to(kp, (4, B, 32)))).cuda())
    parts.append(rand_words(2 * (1 + 3 + h_s + 6 * h_p)))
    show_in = torch.cat(parts)
    assert show_in.shape[0] == issuer._b.L.afx_show_num_fields(n, kinds)
    pres = torch.empty((issuer.num_fields(kinds), B, 32), dtype=torch.uint8, device="cuda")
    issuer.show_batch_device(kinds, B, show_in.data_ptr(), pres.data_ptr(), status.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(status.sum().item()) == 0
    return pres


def corrupt_items(items, kinds, idx, rng):
    """Corrupt items[idx] in place, class by class (SURVEY 8d config 5: response+1, challenge+1, C_x_0 / C_V replaced by another valid
    point, a revealed scalar + 1, enc E2 replaced, enc response + 1, an undecodable point, a scalar >= l) plus single-bit flips in any
    word and any byte, byte 31 included.  Every class is rejected by the reference."""
    kinds = list(kinds)
    n = len(kinds)
    h_s = sum(k == 1 for k in kinds)
    rev0 = 7 + h_s + n
    ps = [i for i, k in enumerate(kinds) if k == 0]
    enc0 = rev0 + sum(k in (0, 2) for k in kinds)
    has_enc = 3 in kinds

    def plus1(i, w):
        v = (int.from_bytes(items[i, w].tobytes(), "little") + 1) % L_ORDER
        items[i, w] = np.frombuffer(v.to_bytes(32, "little"), np.uint8)

    for j, i in enumerate(idx):
        c = j % 11
        other = items[int(idx[j - 1]) if j else int(idx[-1])]
        if c == 0:
            plus1(i, 1)
        elif c == 1:
            plus1(i, 0)
        elif c == 2:
            items[i, 4 + h_s] = other[5 + h_s]                    # C_x_0 := another item's C_x_1 (a valid point)
        elif c == 3:
            items[i, 6 + h_s] = other[4 + h_s]                    # C_V := another item's C_x_0
        elif c == 4 and ps:
            plus1(i, rev0 + sum(1 for k in kinds[:ps[0]] if k in (0, 2)))
        elif c == 5 and has_enc:
            items[i, enc0 + 9] = other[enc0 + 8]                  # E2 := another item's E1
        elif c == 6 and has_enc:
            plus1(i, enc0 + 1)
        elif c == 7:
            items[i, 5 + h_s] = np.frombuffer(bytes([3]) + bytes(31), np.uint8)      # odd => negative => not a ristretto encoding
        elif c == 8:
            v = int.from_bytes(items[i, 2].tobytes(), "little") + L_ORDER
            items[i, 2] = np.frombuffer(v.to_bytes(32, "little"), np.uint8)
        elif c == 9:
            items[i, rng.integers(0, items.shape[1]), 31] ^= 1 << rng.integers(0, 8)
        else:
            items[i, rng.integers(0, items.shape[1]), rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)


ALL_CPUS = os.sched_getaffinity(0)


class all_cores:
    """The GPU ranks pin their thread to the CPUs next to their device (afx_bind_thread_to_device); a CPU leg runs on every core."""

    def __enter__(self):
        self.saved = os.sched_getaffinity(0)
        os.sched_setaffinity(0, ALL_CPUS)

    def __exit__(self, *a):
        os.sched_setaffinity(0, self.saved)


def cpu_leg(sp, ip, sk, kinds, items, threads):
    """The restated reference CPU path (oracle/c, reference schedule) on `items` with `threads` host threads."""
    from oracle import coracle as C
    C.build()
    orc = C.Issuer(sp, ip, sk)
    sub = np.ascontiguousarray(items)
    with all_cores():
        t0 = time.perf_counter()
        verdicts, _ = orc.verify_presentations(kinds, sub, threads=threads)
        wall = time.perf_counter() - t0
    return verdicts, len(sub) / wall, wall


def libsodium_anchor(seconds=0.5):
    """crypto_scalarmult_ristretto255 from the bundled libsodium on one host core (BASELINE.md section 3: roughly one of the seven
    constant-time scalar multiplications of the reference's aMAC) -- lets a reader sanity-check the CPU port's speed."""
    import ctypes
    import glob
    for path in glob.glob("/opt/prime-rl/.venv/lib/python3*/site-packages/pyzmq.libs/libsodium*.so*"):
        try:
            lib = ctypes.CDLL(path)
            lib.crypto_scalarmult_ristretto255
            lib.sodium_init()
        except (OSError, AttributeError):
            continue
        B = bytes.fromhex("e2f2ae0a6abc4e71a884a961c500515f58e30b6aa582dd8db6a65945e08d2d76")
        out = ctypes.create_string_buffer(32)
        sc = bytes(range(1, 32)) + b"\x05"
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            for _ in range(200):
                lib.crypto_scalarmult_ristretto255(out, sc, B)
            n += 200
        dt = time.perf_counter() - t0
        return {"op": "libsodium 1.0.20 crypto_scalarmult_ristretto255, one core", "per_s": n / dt, "us": 1e6 * dt / n}
    return None


def time_device(torch, stream, flush, fn, steps, warmup=2):
    """Device ms per call of fn (enqueues on `stream`), L2 flushed before each timed call."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream)
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    return total / steps


def time_wall(fn, steps, warmup=1):
    for _ in range(warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        r = fn()
    return (time.perf_counter() - t0) / steps, r


def stage_fracs(issuer, model, count, imad_peak, kernel_names):
    """Per-kernel fraction of the IMAD peak from the context's stage timers of the run just made."""
    st = issuer.stage_times_ms()
    out = {}
    pts_ms, lad_ms = st["points"], st["amac"] + st["msm"]
    if pts_ms > 0:
        out[kernel_names[0]] = {"ms": pts_ms, "frac_of_imad_peak": 2 * model["points"] * count / (pts_ms * 1e-3) / imad_peak}
    if lad_ms > 0:
        out[kernel_names[1]] = {"ms": lad_ms, "frac_of_imad_peak": 2 * (model["msm"] + model.get("amac", 0)) * count / (lad_ms * 1e-3) / imad_peak}
    out["k_transcript"] = {"ms": st["transcript"]}
    return out


def secondary_measurements(torch, issuer4, items4, local, stream, flush, B, steps, imad_peak, cores):
    """BASELINE configs[2] and configs[3] on the same GPU: batch Issuer::issue and CredentialIssuance::verify of B revealed
    4-attribute requests -- device-resident (CUDA events), end to end through the host-buffer C ABI, per-kernel fraction of the IMAD
    peak, CPU leg on the host cores -- and Issuer::verify of S16 presentations; AnonymousCredential::show and the BatchableProof modes."""
    from aeonflux_b200 import Issuer, PresentationBatch, RequestBatch, compact_to_batchable
    from oracle import coracle as C
    out = {}
    sp4, ip4, sk4 = load_issuer("issuer4.bin")
    # ---- configs[2]: requests [scalar, scalar, point, point]; the point attributes are valid encodings taken from the batch
    kinds = bytes([0, 0, 2, 2])
    rng = np.random.default_rng(1234)
    n, nf = 4, 3 * 4 + 14
    req = torch.empty((nf, B, 32), dtype=torch.uint8).pin_memory()
    rq = req.numpy()
    sc = rng.integers(0, 256, (2, B, 32), dtype=np.uint8); sc[:, :, 31] &= 0x0f       # < 2^252 < l: canonical scalars
    rq[0:2] = sc
    rq[2] = items4[:B, 5]; rq[3] = items4[:B, 6]                                       # C_x_0, C_x_1 of the batch: valid, distinct points
    rq[4:] = rng.integers(0, 256, (nf - 4, B, 32), dtype=np.uint8)                     # rng output for t, U, blindings
    req_dev = req.cuda()
    iss_dev = torch.empty((2 * n + 9, B, 32), dtype=torch.uint8, device="cuda")
    iss_dev[:n] = req_dev[:n]
    status_dev = torch.empty(B, dtype=torch.uint8, device="cuda")
    issuer4.set_stage_timing(True)
    ms = time_device(torch, stream, flush, lambda: issuer4.issue_batch_device(kinds, B, req_dev.data_ptr(), iss_dev[n:].data_ptr(), status_dev.data_ptr(), stream.cuda_stream), steps)
    assert int(status_dev.sum().item()) == 0
    im = issue_model(2, 2)
    kern = stage_fracs(issuer4, im, B, imad_peak, ("k_points", "k_msm_ct"))
    issuer4.set_stage_timing(False)
    rb = RequestBatch(kinds, rq)
    issued_host = issuer4.host_array((2 * n + 9, B, 32))
    e2e_s, (issued, st) = time_wall(lambda: issuer4.issue_batch(rb, out=issued_host), steps)
    assert not st.any()
    orc = C.Issuer(sp4, ip4, sk4)
    sample = min(B, cores * 1024)
    attrs_s = np.ascontiguousarray(rq[:4, :sample].transpose(1, 0, 2))
    rnd_s = np.ascontiguousarray(rq[4:, :sample].transpose(1, 0, 2)).reshape(sample, n + 7, 64)
    with all_cores():
        t0 = time.perf_counter()
        oout, ostatus, _ = orc.issue(kinds, attrs_s, rnd_s, threads=cores)
        cpu_wall = time.perf_counter() - t0
    assert (issued.fields.transpose(1, 0, 2)[:sample, 4:] == oout).all(), "issuances differ from the CPU oracle's given the same rng bytes"
    out["issue_4attr"] = {"workload": "batch Issuer::issue (Amac::tag + ProofOfIssuance::prove) of %d revealed 4-attribute requests (BASELINE configs[2])" % B,
                          "value": B / (ms * 1e-3), "unit": "issuances/s", "ms_per_step": ms,
                          "e2e": {"value": B / e2e_s, "unit": "issuances/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": nf * B * 32, "d2h_bytes_per_step": (n + 9) * B * 32 + B,
                                  "api": "afx_issue: struct-of-arrays request fields in pinned host memory -> issuance words in pinned host memory (afx_host_alloc), status bytes"},
                          "algorithmic_imad_per_item": {k: 2 * v for k, v in im.items()},
                          "frac": (2 * im["total"] * B / (ms * 1e-3)) / imad_peak, "kernels": kern,
                          "cpu_baseline": {"value": sample / cpu_wall, "unit": "issuances/s", "cores": cores, "kind": "port",
                                           "sample": "%d requests of the same batch, %.1f s, oracle/c constant-time schedule; output bytes identical to the GPU's" % (sample, cpu_wall)}}
    # ---- CredentialIssuance::verify of what was just issued
    verdicts_dev = torch.empty(B, dtype=torch.uint8, device="cuda")
    issuer4.set_stage_timing(True)
    ms = time_device(torch, stream, flush, lambda: issuer4.verify_issuance_batch_device(kinds, B, iss_dev.data_ptr(), verdicts_dev.data_ptr(), stream.cuda_stream), steps)
    assert int(verdicts_dev.sum().item()) == 0, "issued credentials failed CredentialIssuance::verify"
    vm = issuance_verify_model(2, 2)
    kern = stage_fracs(issuer4, vm, B, imad_peak, ("k_points", "k_ladders"))
    issuer4.set_stage_timing(False)
    wire = torch.empty((B, 2 * n + 9, 32), dtype=torch.uint8).pin_memory()
    wire.numpy()[:] = issued.fields.transpose(1, 0, 2)
    e2e_s, v = time_wall(lambda: issuer4.verify_wire(kinds, wire.numpy(), issuance=True), steps)
    assert not v.any()
    with all_cores():
        t0 = time.perf_counter()
        ov, _ = orc.verify_issuances(kinds, np.ascontiguousarray(wire.numpy()[:sample]), threads=cores)
        cpu_wall = time.perf_counter() - t0
    assert not ov.any()
    survey_imad = 2.158e6          # SURVEY 8d table, issuance-verify n = 4 [PS,PS,PP,EP]
    out["verify_issuance_4attr"] = {"workload": "batch CredentialIssuance::verify of the %d issuances above (BASELINE configs[2])" % B,
                                    "value": B / (ms * 1e-3), "unit": "issuances/s", "ms_per_step": ms,
                                    "e2e": {"value": B / e2e_s, "unit": "issuances/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": (2 * n + 9) * B * 32, "d2h_bytes_per_step": B,
                                            "api": "afx_verify_issuances_wire: item-major bytes in pinned host memory -> verdict bytes"},
                                    "algorithmic_imad_per_item": {"survey_8d": survey_imad, "formula": {k: 2 * v for k, v in vm.items()}},
                                    "frac": (survey_imad * B / (ms * 1e-3)) / imad_peak, "kernels": kern,
                                    "cpu_baseline": {"value": sample / cpu_wall, "unit": "issuances/s", "cores": cores, "kind": "port",
                                                     "sample": "%d issuances of the same batch, %.1f s, oracle/c reference schedule; verdicts identical" % (sample, cpu_wall)}}
    # ---- AnonymousCredential::show (user-side prover, SURVEY 8f rank 3): the issuances above as credentials of shape
    # [PS, PS, PP, PP] (nothing hidden), fresh rng bytes; the presentations are then verified
    k_show = bytes([0, 0, 2, 2])
    nf_in, nf_out = 3 + 4 + 2 * (1 + 3), 1 + 3 + 3 + 4 + 4
    sh = torch.empty((nf_in, B, 32), dtype=torch.uint8, device="cuda")
    sh[0:3] = iss_dev[n:n + 3]; sh[3:7] = iss_dev[0:4]
    sh[7:] = torch.from_numpy(rng.integers(0, 256, (nf_in - 7, B, 32), dtype=np.uint8)).cuda()
    pres_dev = torch.empty((nf_out, B, 32), dtype=torch.uint8, device="cuda")
    ms = time_device(torch, stream, flush, lambda: issuer4.show_batch_device(k_show, B, sh.data_ptr(), pres_dev.data_ptr(), status_dev.data_ptr(), stream.cuda_stream), steps)
    assert int(status_dev.sum().item()) == 0
    issuer4.verify_batch_device(k_show, B, pres_dev.data_ptr(), verdicts_dev.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    assert int(verdicts_dev.sum().item()) == 0, "presentations made on the device failed Issuer::verify"
    out["show_4attr_revealed"] = {"workload": "batch AnonymousCredential::show of %d all-revealed 4-attribute credentials (user-side prover), verified afterwards" % B,
                                  "value": B / (ms * 1e-3), "unit": "presentations/s", "ms_per_step": ms, "timing": "device-resident, CUDA events"}
    # ---- BatchableProof mode (opt-in, not the reference's encoding): the same presentations re-encoded with their commitments,
    # verified exactly and by one random linear combination per batch (Pippenger); host-buffer calls, wall clock
    comp = PresentationBatch.from_items(KINDS_README4, items4[:B])
    _, dbg = issuer4.verify_batch(comp, debug=True)
    bb_host = torch.from_numpy(compact_to_batchable(KINDS_README4, comp.fields, dbg["commitments"])).pin_memory()
    bb = PresentationBatch(KINDS_README4, bb_host.numpy())
    issuer4.set_stage_timing(True)
    for name, fn in (("verify_batchable_exact", lambda: issuer4.verify_batchable(bb)), ("verify_batchable_rlc", lambda: issuer4.verify_batchable_rlc(bb, bytes(range(32)))[0])):
        dt, v = time_wall(fn, steps)
        assert not v.any()
        out[name] = {"workload": "%d README-4 presentations in BatchableProof form through the host-buffer call (%s), all valid" % (B, "one MSM per constraint" if "exact" in name else "one random linear combination per batch, Pippenger"),
                     "value": B / dt, "unit": "presentations/s", "ms_per_step": dt * 1e3, "timing": "end to end (H2D + kernels + D2H), wall clock"}
    bms, binputs, bwin = issuer4.rlc_bucket_time()
    issuer4.set_stage_timing(False)
    # every per-item point enters one bucket per window (a zero digit, 1 in 2^16, aside): one extended addition (9 M) each
    out["verify_batchable_rlc"]["kernels"] = {"k_rlc_buckets": {"ms": bms, "points": binputs, "windows": bwin,
                                                                "frac_of_imad_peak": (2 * 9 * M_LP * binputs * bwin / (bms * 1e-3)) / imad_peak,
                                                                "note": "gather-latency bound: each thread walks one bucket's points (dependent load -> add chain)"}}
    # ---- S16 presentations (configs[3]) at the config's full batch: 65,536 x 4,576 B in, 4.6 GB of ladder tables
    sp, ip, sk = load_issuer("issuer16.bin")
    issuer16 = Issuer(sp, ip, sk, device=local, max_batch=B)
    f16 = synthesize_on_device(torch, issuer16, B, 4242, stream, KINDS_S16, "keypair16.bin")
    v16 = torch.empty(B, dtype=torch.uint8, device="cuda")
    issuer16.set_stage_timing(True)
    ms = time_device(torch, stream, flush, lambda: issuer16.verify_batch_device(KINDS_S16, B, f16.data_ptr(), v16.data_ptr(), stream.cuda_stream), steps)
    assert int(v16.sum().item()) == 0
    wm = work_model(KINDS_S16)
    kern = stage_fracs(issuer16, wm, B, imad_peak, ("k_points", "k_ladders"))
    kern["k_transcript"]["keccak_f_per_item"] = 80
    kern["k_transcript"]["frac_of_alu_peak"] = 80 * KECCAK_ALU_OPS * B / (kern["k_transcript"]["ms"] * 1e-3) / imad_peak
    issuer16.set_stage_timing(False)
    wire16 = torch.empty((B, WORDS_S16, 32), dtype=torch.uint8).pin_memory()
    wire16.copy_(f16.permute(1, 0, 2))
    w16 = wire16.numpy()
    bad16 = [5, B // 2 - 1, B // 2, B - 7]                      # a few rejects on either side of the library's two half passes
    for j, i in enumerate(bad16):
        w16[i, 3 + 11 * j, 31 if j % 2 else 2] ^= 0x40
    exp16 = np.zeros(B, np.uint8); exp16[bad16] = 1
    e2e_s, v = time_wall(lambda: issuer16.verify_wire(KINDS_S16, w16), steps)
    assert (v == exp16).all(), "S16 end-to-end verdicts differ from the expected set"
    sample16 = min(B, cores * 256)
    cv, rate16, wall16 = cpu_leg(sp, ip, sk, KINDS_S16, w16[:sample16], cores)
    assert (cv == exp16[:sample16]).all(), "the CPU oracle disagrees on S16 presentations made on the device"
    out["verify_s16"] = {"workload": "batch Issuer::verify of %d 16-attribute presentations, 8 hidden plaintext attributes (BASELINE configs[3]); distinct items made on the device" % B,
                         "value": B / (ms * 1e-3), "unit": "presentations/s", "ms_per_step": ms,
                         "e2e": {"value": B / e2e_s, "unit": "presentations/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": B * WORDS_S16 * 32, "d2h_bytes_per_step": B,
                                 "api": "afx_verify_presentations_wire (the library runs an input this large as two pipelined half passes)"},
                         "algorithmic_imad_per_item": {k: 2 * v for k, v in wm.items()},
                         "frac": (B * 2 * wm["total"] / (ms * 1e-3)) / imad_peak, "kernels": kern,
                         "cpu_baseline": {"value": rate16, "unit": "presentations/s", "cores": cores, "kind": "port",
                                          "sample": "%d items of the same batch, %.1f s, oracle/c reference schedule; verdicts identical" % (sample16, wall16)}}
    # ---- small batches: latency of ONE synchronous item-major call (copy in, kernels, verdicts out) -- what a serving front end sees
    def call_ms(iss, kinds, w, count):
        iss.verify_wire(kinds, w[:count])
        ts = []
        for _ in range(9):
            t0 = time.perf_counter()
            v = iss.verify_wire(kinds, w[:count])
            ts.append(time.perf_counter() - t0)
        assert not v[:min(count, 5)].any()
        return 1e3 * float(np.median(ts))
    w4 = torch.empty((8192, WORDS, 32), dtype=torch.uint8).pin_memory()
    w4.numpy()[:] = items4[:8192]
    out["small_batch_latency"] = {"workload": "one synchronous afx_verify_presentations_wire call of 1 / 1,024 / 8,192 presentations from page-locked memory, median wall clock of 9 calls",
                                  "unit": "ms per call",
                                  "readme4": {str(c): call_ms(issuer4, KINDS_README4, w4.numpy(), c) for c in (1, 1024, 8192)},
                                  "s16": {str(c): call_ms(issuer16, KINDS_S16, w16[8:], c) for c in (1, 1024, 8192)},
                                  "note": "passes of at most 8,192 items run the aMAC ladder in parts beside the constraint MSMs (DESIGN.md section 5, Small batches)"}
    issuer16.close()
    return out


def stream_config5(torch, dist, sharded4, rank, world, local, total, stream, cores, with_cpu):
    """BASELINE configs[4]: streamed verification of `total` mixed presentations (README-4 and S16, 50:50, 1 % corrupted) sharded over
    the ranks.  Every rank makes its own contiguous slice of the stream on its device (distinct items), corrupts 1 % of it, and
    pushes it through the library's stream object: records bucketed by shape into page-locked double buffers, each full bucket
    submitted asynchronously (afx_*_wire_submit), verdict bitmap all-gathered at the end.  Timed: push + flush + gather."""
    from aeonflux_b200 import Issuer
    from aeonflux_b200.shard import MixedStream, ShardedIssuer, slice_bounds
    sp16, ip16, sk16 = load_issuer("issuer16.bin")
    chunk = 65536
    lo, hi = slice_bounds(total, rank, world)
    mine = hi - lo
    rng = np.random.default_rng(9000 + rank)
    order_all = np.random.default_rng(55).integers(0, 2, total).astype(np.uint8)       # the same stream order on every rank
    order = order_all[lo:hi]
    n4, n16 = int((order == 0).sum()), int((order == 1).sum())
    issuer4 = sharded4.issuer
    issuer16 = Issuer(sp16, ip16, sk16, device=local, max_batch=chunk)
    # this rank's records: one allocation [README-4 pool | S16 pool]; a record's offset says where it lies (the stream order is
    # carried by the offsets / shape ids, as with buffers handed over by a network stack)
    blob = np.empty(n4 * WORDS * 32 + n16 * WORDS_S16 * 32, np.uint8)
    pool4 = blob[:n4 * WORDS * 32].reshape(n4, WORDS, 32)
    pool16 = blob[n4 * WORDS * 32:].reshape(n16, WORDS_S16, 32)
    t_gen = time.perf_counter()
    for pool, iss, kinds, kp, seed in ((pool4, issuer4, KINDS_README4, "keypair4.bin", 100), (pool16, issuer16, KINDS_S16, "keypair16.bin", 200)):
        for s in range(0, len(pool), chunk):
            m = min(chunk, len(pool) - s)
            dev = synthesize_on_device(torch, iss, m, seed + 1000 * rank + s // chunk, stream, kinds, kp)
            pool[s:s + m] = dev.permute(1, 0, 2).cpu().numpy()
            del dev
    t_gen = time.perf_counter() - t_gen
    expect = np.zeros(mine, np.uint8)
    bad = rng.choice(mine, max(1, mine // 100), replace=False)
    expect[bad] = 1
    pos_in_pool = np.empty(mine, np.int64)
    pos_in_pool[order == 0] = np.arange(n4); pos_in_pool[order == 1] = np.arange(n16)
    for sid, pool, kinds in ((0, pool4, KINDS_README4), (1, pool16, KINDS_S16)):
        sel = bad[order[bad] == sid]
        corrupt_items(pool, kinds, pos_in_pool[sel], rng)
    offsets = np.where(order == 0, pos_in_pool * (WORDS * 32), n4 * WORDS * 32 + pos_in_pool * (WORDS_S16 * 32)).astype(np.uint64)
    ms = MixedStream()
    assert [ms.add_shape(issuer4, KINDS_README4), ms.add_shape(issuer16, KINDS_S16)] == [0, 1]
    # warm-up: one bucket of each shape (workspace allocation, shape compilation), untimed
    w = np.zeros(min(mine, 2 * chunk), np.uint8)
    ms.push(blob, offsets[:len(w)], order[:len(w)], w)
    ms.flush()
    assert (w == expect[:len(w)]).all()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    b0 = ms.buckets_submitted
    tm0 = ms.times()
    t0 = time.perf_counter()
    local_v = np.zeros(mine, np.uint8)
    ms.push(blob, offsets, order, local_v)
    t_push = time.perf_counter()
    ms.flush()
    t_flush = time.perf_counter()
    from aeonflux_b200.shard import pack_bitmap
    allv = sharded4._gather_bitmaps(pack_bitmap(local_v), total) if world > 1 else local_v
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    tm1 = ms.times()
    mine_split = {"rank": rank, "push_s": t_push - t0, "flush_s": t_flush - t_push, "gather_s": wall - (t_flush - t0), "bucketing_memcpy_s": tm1[0] - tm0[0],
                  "enqueue_s": tm1[1] - tm0[1], "blocked_on_device_s": tm1[2] - tm0[2]}
    splits = [mine_split]
    if world > 1:
        splits = [None] * world
        dist.all_gather_object(splits, mine_split)
    mism = int((local_v != expect).sum())
    assert mism == 0, "%d verdict mismatches in the config-5 stream" % mism
    t = torch.tensor([wall, float(mism), float(expect.sum())], dtype=torch.float64, device="cuda")
    tot = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        assert int(allv.sum()) == int(tot[2].item()), "gathered bitmap disagrees with the ranks' reject counts"
    res = {"workload": "streamed verification of %d mixed presentations (README-4 and S16, item-mixed 50:50 in stream order, 1 %% corrupted: 11 classes "
                       "incl. byte-31 bit flips), rank r pushing stream slice r through afx_stream_* (BASELINE configs[4])" % total,
           "value": total / float(t[0].item()), "unit": "presentations/s", "wall_s": float(t[0].item()), "n_gpus": world, "items": total, "rejected": int(tot[2].item()),
           "mismatches": int(tot[1].item()), "buckets_per_rank": ms.buckets_submitted - b0, "bucket_items": chunk,
           "h2d_bytes": int(n4 * WORDS * 32 + n16 * WORDS_S16 * 32),
           "per_rank_seconds": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in sp.items()} for sp in splits],
           "timing": "wall clock: push (bucketing into page-locked double buffers, asynchronous wire submits) + flush + bitmap all-gather, max over ranks; "
                                                                             "one warm-up bucket per shape untimed",
           "input": "every item distinct, issued and shown on the rank's device (%.1f s, untimed)" % t_gen}
    if with_cpu and rank == 0:
        sample = min(mine, cores * 384)
        s4, s16 = np.nonzero(order[:sample] == 0)[0], np.nonzero(order[:sample] == 1)[0]
        sp4, ip4, sk4 = load_issuer("issuer4.bin")
        v4, _, w4 = cpu_leg(sp4, ip4, sk4, KINDS_README4, pool4[pos_in_pool[s4]], cores)
        v16, _, w16 = cpu_leg(sp16, ip16, sk16, KINDS_S16, pool16[pos_in_pool[s16]], cores)
        assert (v4 == local_v[s4]).all() and (v16 == local_v[s16]).all(), "GPU verdicts differ from the CPU port's on the stream sample"
        res["cpu_baseline"] = {"value": sample / (w4 + w16), "unit": "presentations/s", "cores": cores, "kind": "port",
                               "sample": "the first %d records of the same stream (%d README-4, %d S16; %d corrupted), %.1f s, oracle/c reference schedule; verdicts identical to the GPU's"
                                         % (sample, len(s4), len(s16), int(expect[:sample].sum()), w4 + w16)}
    ms.close()
    issuer16.close()
    return res


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: each array as out_dir/<name>.npy in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float32))


def run_reference(args, rank):
    """--impl reference: the reference's own CPU schedule of Issuer::verify on the host cores, on the native arm's config.  The Rust
    crate cannot be built in this image (no rustc/cargo, un-vendored deps), so this is the C restatement of its schedule (oracle/c)."""
    if rank != 0:
        return
    from oracle import coracle as C
    C.build()
    cores = os.cpu_count() or 1
    sp, ip, sk = load_issuer("issuer4.bin")
    orc = C.Issuer(sp, ip, sk)
    B = args.batch
    distinct = min(B, 8192)
    kinds, pres, _ = orc.synth(b"SSPE", [0, 3], b"bench-reference-arm", 0, distinct, want_issuances=False, threads=cores)
    assert kinds == KINDS_README4
    items = np.ascontiguousarray(np.tile(pres, ((B + distinct - 1) // distinct, 1, 1))[:B])
    for _ in range(args.warmup):                                  # warm-up steps run a 1/16 sample
        cpu_leg(sp, ip, sk, KINDS_README4, items[:max(B // 16, cores)], cores)
    t_total, n_total = 0.0, 0
    for _ in range(args.steps):
        v, rate, wall = cpu_leg(sp, ip, sk, KINDS_README4, items, cores)
        assert not v.any()
        t_total += wall; n_total += B
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, verdicts_reference=v)
    value = n_total / t_total
    line = {"impl": "reference", "metric": "presentations_verified_per_sec", "value": value, "unit": "presentations/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 (5x51-bit limbs, like dalek u64_backend)", "data": "synthetic", "config": CONFIG,
            "cpu_baseline": {"value": value, "unit": "presentations/s", "cores": cores, "kind": "port",
                             "sample": "the full %d-item batch per step x %d steps (one batch, whatever N), C restatement of the reference schedule (not the Rust binary)" % (B, args.steps),
                             "anchor": libsodium_anchor()},
            "e2e": {"value": value, "unit": "presentations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the issuance / S16 / BatchableProof measurements (configs[2], configs[3])")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-5 mixed stream")
    ap.add_argument("--stream-items", type=int, default=1 << 22, help="items of the config-5 stream (BASELINE: 2^22)")
    ap.add_argument("--tiled-input", action="store_true", help="tile the 1,024-item CPU-made fixture instead of synthesizing the batch on the device")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the verdicts of the last timed device-resident and end-to-end steps to DIR/<name>.npy "
                                                          "(float32; the inputs are seeded, so runs with the same arguments compare item for item)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist
    from aeonflux_b200 import Issuer, PresentationBatch
    from aeonflux_b200.shard import ShardedIssuer
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    from aeonflux_b200.issuer import bind_thread_to_device
    numa_bound = bind_thread_to_device(local)          # before any pinned allocation: node-local staging for this rank's GPU
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.batch
    cores = os.cpu_count() or 1
    sp, ip, sk, items = load_fixture(B)
    issuer = Issuer(sp, ip, sk, device=local, max_batch=B)
    sharded = ShardedIssuer(issuer)
    assert (sharded.rank, sharded.world) == (rank, world)
    kinds = KINDS_README4
    stream = torch.cuda.current_stream()
    if args.tiled_input:
        fields_dev = torch.from_numpy(np.ascontiguousarray(np.roll(items, rank * 131, axis=0).transpose(1, 0, 2))).cuda()
    else:
        fields_dev = synthesize_on_device(torch, issuer, B, 1000 + rank, stream)
    verdicts_dev = torch.empty(B, dtype=torch.uint8, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        issuer.verify_batch_device(kinds, B, fields_dev.data_ptr(), verdicts_dev.data_ptr(), stream.cuda_stream)
        e1.record(stream)
        return e0, e1

    # ---- kernel-only: inputs resident in HBM --------------------------------------------------------------------
    clocks = ClockSampler(local).start()
    issuer.set_stage_timing(True)
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    launches0 = issuer.launch_count
    stage_sum = {k: 0.0 for k in Issuer.STAGES}
    with clocks.window():
        evs = []
        for _ in range(args.steps):
            evs.append(step_device())
            torch.cuda.synchronize()
            for k, v in issuer.stage_times_ms().items():
                stage_sum[k] += v
        barrier()
    launches = issuer.launch_count - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    assert int(verdicts_dev.sum().item()) == 0, "honest presentations were rejected"
    issuer.set_stage_timing(False)

    # ---- end to end: ONE global batch of world x B items in host memory through the product's sharding layer -----------------
    # every rank holds the whole batch (its own slice made on its device, the others' gathered once, untimed); a few items are
    # corrupted so that the gathered bitmap is not all-zero
    wire_global = torch.empty((world * B, WORDS, 32), dtype=torch.uint8).pin_memory()
    local_items = fields_dev.permute(1, 0, 2).contiguous()
    if world > 1:
        gathered = torch.empty((world * B, WORDS, 32), dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(gathered, local_items)
        wire_global.copy_(gathered)
        del gathered
    else:
        wire_global.copy_(local_items)
    crng = np.random.default_rng(7)
    bad = np.sort(crng.choice(world * B, 16 * world, replace=False))
    corrupt_items(wire_global.numpy(), kinds, bad, crng)
    expect = np.zeros(world * B, np.uint8); expect[bad] = 1
    honest_local = np.ascontiguousarray(local_items.cpu().numpy())
    for _ in range(2):
        assert (sharded.verify_wire(kinds, wire_global.numpy()) == expect).all(), "sharded verdicts differ from the expected set"
    barrier()
    sharded.gather_seconds = 0.0
    with clocks.window():
        t0 = time.perf_counter()
        for _ in range(args.steps):
            v = sharded.verify_wire(kinds, wire_global.numpy())
        barrier()
        e2e_s = time.perf_counter() - t0
    gather_ms = 1e3 * sharded.gather_seconds / args.steps
    assert (v == expect).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, verdicts_device=verdicts_dev.cpu().numpy(), verdicts_e2e=v)
    # also timed, per rank on its own slice (no gather): the struct-of-arrays entry and the streamed submit / wait form
    host = torch.empty((WORDS, B, 32), dtype=torch.uint8).pin_memory()
    host.numpy()[:] = honest_local.transpose(1, 0, 2)
    batch = PresentationBatch(kinds, host.numpy())
    issuer.verify_batch(batch)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        assert not issuer.verify_batch(batch).any()
    barrier()
    e2e_soa_s = time.perf_counter() - t0
    wire_local = torch.from_numpy(honest_local).pin_memory()
    for p in [issuer.submit_wire(kinds, wire_local.numpy()), issuer.submit_wire(kinds, wire_local.numpy())]:
        p.wait()
    barrier()
    with clocks.window():
        t0 = time.perf_counter()
        pend = []
        for _ in range(args.steps):
            pend.append(issuer.submit_wire(kinds, wire_local.numpy()))
            if len(pend) == 2:
                assert not pend.pop(0).wait().any()
        while pend:
            assert not pend.pop(0).wait().any()
        barrier()
        e2e_stream_s = time.perf_counter() - t0
    clocks.stop()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    clk = clocks.summary()
    sm_max = clk.get("sm_max_mhz") or peaks.get("sm_max_mhz") or 1965.0
    imad_peak = 148 * 64 * sm_max * 1e6                       # IMAD issue slots/s at max clock (SURVEY 8d; measured 18.52e12 by tools/microbench)

    # diagnostic: host-to-device bandwidth of every rank with all ranks copying at once (256 MiB from page-locked memory, best of 3)
    hb = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    db = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    best = 1e9
    for _ in range(3):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); db.copy_(hb, non_blocking=True); e1.record(stream)
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    h2d = torch.tensor([(256 << 20) / (best * 1e-3) / 1e9, dev_ms / args.steps], dtype=torch.float64, device="cuda")
    per_rank = [torch.empty_like(h2d) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, h2d)
    else:
        per_rank = [h2d]
    per_rank_diag = {"h2d_GBps_all_ranks_copying": [round(float(x[0]), 1) for x in per_rank], "device_ms_per_step": [round(float(x[1]), 2) for x in per_rank]}
    del hb, db

    secondary = {}
    if world == 1 and not args.no_secondary:
        secondary = secondary_measurements(torch, issuer, honest_local, local, stream, flush, B, min(args.steps, 3), imad_peak, cores)
    if not args.no_stream:
        secondary["stream_config5"] = stream_config5(torch, dist, sharded, rank, world, local, args.stream_items, stream, cores, with_cpu=not args.no_cpu_baseline)

    t = torch.tensor([dev_ms, e2e_s * 1e3, e2e_soa_s * 1e3, e2e_stream_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max, e2e_soa_ms_max, e2e_stream_ms_max = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_items = world * B * args.steps
    value = total_items / (dev_ms_max * 1e-3)
    e2e_value = total_items / (e2e_ms_max * 1e-3)
    wm = work_model(kinds)
    # dominant kernel: k_ladders = the aMAC ladder + every constraint MSM of the batch in one launch (stages "amac" + "msm")
    msm_ms = (stage_sum["msm"] + stage_sum["amac"]) / args.steps
    msm_imad = 2 * (wm["msm"] + wm["amac"]) * B               # algorithmic IMAD slots per launch of k_ladders
    achieved = msm_imad / (msm_ms * 1e-3)
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except (OSError, ValueError):
        pass
    hbm_bytes = B * (WORDS * 32 + 1)
    tx_ms = stage_sum["transcript"] / args.steps
    roofline = {"bound": "imad", "kernel": "k_ladders", "achieved": achieved / 1e12, "peak": imad_peak / 1e12, "unit": "TIMAD/s", "frac": achieved / imad_peak,
                "traffic": (traffic or {}).get("k_ladders"),
                "traffic_source": "NOT measured by this run: dram__bytes_read.sum + dram__bytes_write.sum of one k_ladders launch from the committed ncu --set full capture, "
                                  + str((traffic or {}).get("source")),
                "traffic_note": "~25 GB are the aMAC ladder's constant-address table scans (every entry of every per-item table is read at every step so that no "
                                "address depends on an issuer secret), the rest per-item ladder tables; 17 % of DRAM throughput, the kernel is bound by the IMAD pipe",
                "peak_source": "148 SMs x 64 IMAD/clk x sm_max_mhz; tools/microbench measured 18.52 T IMAD/s and 9.12 T IMAD.WIDE/s (profiles/r01_microbench_imad.json)",
                "algorithmic_imad_per_item": {k: 2 * v for k, v in wm.items()},
                "stage_ms_per_step": {k: v / args.steps for k, v in stage_sum.items()},
                "kernels": {"k_points": {"ms": stage_sum["points"] / args.steps, "frac_of_imad_peak": (2 * wm["points"] * B / (stage_sum["points"] / args.steps * 1e-3)) / imad_peak},
                            "k_ladders": {"ms": msm_ms, "frac_of_imad_peak": achieved / imad_peak},
                            "k_transcript": {"ms": tx_ms, "keccak_f_per_item": 16, "bound": "alu (logic ops; no integer multiplies)",
                                             "frac_of_alu_peak": 16 * KECCAK_ALU_OPS * B / (tx_ms * 1e-3) / imad_peak,
                                             "alu_peak": "148 SMs x 64 lanes/clk x sm_max_mhz (the alu pipe issues at the fma pipe's rate, B300_MICROARCH.md); %d logic ops per Keccak-f" % KECCAK_ALU_OPS},
                            "others": "k_msm_ct under secondary.issue_4attr.kernels, k_rlc_buckets under secondary.verify_batchable_rlc.kernels, S16 kernels under secondary.verify_s16.kernels"},
                "pipeline_frac_of_imad_peak": (B * args.steps * 2 * wm["total"] / (dev_ms * 1e-3)) / imad_peak,
                "pipeline_frac_at_observed_clock": ((B * args.steps * 2 * wm["total"] / (dev_ms * 1e-3)) / (148 * 64 * clk["sm_mhz"] * 1e6)) if clk.get("sm_mhz") else None,
                "hbm": {"algorithmic_GBps": hbm_bytes * args.steps / (dev_ms * 1e-3) / 1e9, "peak_GBps": peaks.get("hbm_gbs", 6650.0),
                        "note": "non-binding: 897 B of input/output per presentation"}}
    bitmap_bytes = (B + 7) // 8 + 1
    line = {"metric": "presentations_verified_per_sec", "value": value, "unit": "presentations/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (8x32-bit limbs, IMAD.WIDE carry chains)",
            "data": "synthetic", "config": CONFIG,
            "clocks": clk, "gpu_launches": launches, "numa_bound": bool(numa_bound), "per_rank": per_rank_diag,
            "e2e": {"value": e2e_value, "unit": "presentations/s", "h2d_bytes_per_step": world * B * WORDS * 32, "d2h_bytes_per_step": world * (B + bitmap_bytes * world),
                    "ms_per_step": e2e_ms_max / args.steps,
                    "api": "ShardedIssuer.verify_wire on ONE global batch of %d x 65,536 items in pinned host memory: contiguous slice per rank -> afx_verify_presentations_wire "
                           "(H2D of the slice, kernels, D2H of its verdicts) -> accept/reject bitmap all-gathered%s; every rank returns all %d verdicts; %d corrupted items, verdict vector checked"
                           % (world, " over NCCL" if world > 1 else " (world 1: no collective)", world * B, len(bad)),
                    "collective_bytes_per_step": bitmap_bytes * world * world if world > 1 else 0,
                    "gather_ms_per_step_rank0": gather_ms, "gather_note": "bitmap pack + all-gather + unpack on rank 0, including the wait for the slowest rank of the step",
                    "soa_api_value": total_items / (e2e_soa_ms_max * 1e-3),
                    "streamed_value": total_items / (e2e_stream_ms_max * 1e-3),
                    "streamed_api": "per rank, no gather: afx_verify_presentations_wire_submit / afx_wait, two submissions in flight (same per-step H2D and D2H bytes; "
                                    "the copy of step k+1 overlaps the kernels of step k)"},
            "roofline": roofline}
    if secondary:
        line["secondary"] = secondary
    if world == 1 and not args.no_cpu_baseline:
        sample = min(B, cores * 2048)                  # ~2-4 s of CPU work at ~1 k presentations/s/core
        cv, rate, wall = cpu_leg(sp, ip, sk, kinds, wire_global.numpy()[:sample], cores)
        assert (cv == expect[:sample]).all(), "GPU verdicts differ from the CPU restatement"
        _, rate1, _ = cpu_leg(sp, ip, sk, kinds, honest_local[:max(sample // cores, 256)], 1)
        line["cpu_baseline"] = {"value": rate, "unit": "presentations/s", "cores": cores, "kind": "port", "single_core_value": rate1,
                                "sample": "%d items of the same batch, %.1f s, C restatement of the reference CPU schedule (oracle/c), verdicts cross-checked with the GPU" % (sample, wall),
                                "anchor": libsodium_anchor()}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
