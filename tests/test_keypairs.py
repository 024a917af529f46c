"""Batch Keypair::derive / Keypair::generate (afx_derive_keypairs, afx_derive_keypairs_device; include/aeonflux_b200.h): parity with
the oracle's recorded keypairs under both bench issuers (tests/golden/keypairs.json), the bench fixture's keypairs, the exact
precondition codes, encryption under derived keypairs, and presentations with one derived keypair per item that verify and decrypt.
Every case runs on the host emulation and, under -m gpu, on the CUDA library; the full-size cases run on the GPU only."""
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest

from tests.test_symmetric import KINDS4, KINDS16, hidden_plaintext_blocks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, ARG = 0, -1
BENCH_SECRET = b"aeonflux-b200 bench keypair".ljust(64, b"\0")
ISSUERS = ("issuer4.bin", "issuer16.bin")


@pytest.fixture(scope="module")
def emu():
    from aeonflux_b200._binding import Binding
    from tests.test_host_logic import build_hostemu
    return Binding(ctypes.CDLL(build_hostemu()))


@pytest.fixture(scope="module", params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def binding(request, emu):
    if request.param == "emu":
        return emu
    from aeonflux_b200._lib import load
    return load()


@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(ROOT, "tests", "golden", "keypairs.json")) as f:
        return json.load(f)


def issuer(binding, name, max_batch, secret=False):
    import bench
    from aeonflux_b200 import Issuer
    sp, ip, sk = bench.load_issuer(name)
    return Issuer(sp, ip, sk if secret else None, device=0, max_batch=max_batch, _binding=binding)


def derive_device(binding, emu, iss, ms, max_batch):
    """afx_derive_keypairs_device in passes of max_batch items -> [count][128].  On the host emulation device memory is host memory."""
    out = []
    for lo in range(0, len(ms), max_batch):
        part = np.array(ms[lo:lo + max_batch])                     # a writable copy: torch takes no read-only arrays
        m = len(part)
        if binding is emu:
            rows = np.zeros((4, m, 32), np.uint8)
            iss.derive_keypairs_device(m, part.ctypes.data, rows.ctypes.data)
        else:
            import torch
            d_ms = torch.from_numpy(part).cuda()
            d_rows = torch.empty((4, m, 32), dtype=torch.uint8, device="cuda")
            iss.derive_keypairs_device(m, d_ms.data_ptr(), d_rows.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            rows = d_rows.cpu().numpy()
        out.append(rows.transpose(1, 0, 2).reshape(m, 128))
    return np.concatenate(out)


def test_golden_covers_the_edge_cases(golden):
    ms = golden["master_secrets"]
    assert ms[:3] == ["00" * 64, "ff" * 64, BENCH_SECRET.hex()] and len(set(ms)) == len(ms) >= 30
    assert golden["keypairs"]["issuer4.bin"][2] != golden["keypairs"]["issuer16.bin"][2]      # pk depends on the system parameters
    assert golden["keypairs"]["issuer4.bin"][2][:192] == golden["keypairs"]["issuer16.bin"][2][:192]   # a, a0, a1 do not


@pytest.mark.parametrize("name", ISSUERS)
def test_derive_matches_oracle(binding, emu, golden, name):
    ms = np.array([list(bytes.fromhex(h)) for h in golden["master_secrets"]], np.uint8)
    expect = np.array([list(bytes.fromhex(h)) for h in golden["keypairs"][name]], np.uint8)
    iss = issuer(binding, name, 3)                                 # 33 items in passes of 3
    assert iss.derive_keypairs(ms).tobytes() == expect.tobytes()
    assert derive_device(binding, emu, iss, ms, 3).tobytes() == expect.tobytes()
    out = np.full((1, 128), 7, np.uint8)
    assert iss.derive_keypairs(ms[2:3], out=out) is out and out.tobytes() == expect[2].tobytes()
    iss.close()


@pytest.mark.parametrize("name", ISSUERS)
def test_bench_fixture_keypairs(binding, emu, name):
    fixture = open(os.path.join(ROOT, "bench_data", name.replace("issuer", "keypair")), "rb").read()
    iss = issuer(binding, name, 4, secret=True)                    # an issuer's context derives like a user's
    ms = np.frombuffer(BENCH_SECRET, np.uint8).reshape(1, 64)
    assert iss.derive_keypairs(ms).tobytes() == fixture
    assert derive_device(binding, emu, iss, ms, 4).tobytes() == fixture
    iss.close()


def test_preconditions(binding):
    import bench
    L = binding.L
    sp, ip, sk = bench.load_issuer("issuer4.bin")
    buf = (ctypes.c_uint8 * 1024)()
    B = ctypes.addressof(buf)
    assert L.afx_derive_keypairs(None, 0, None, None) == ARG
    assert L.afx_derive_keypairs_device(None, 0, None, None, None) == ARG
    for secret in (sk, None):                                      # an issuer context and a user-side context
        h = ctypes.c_void_p()
        assert L.afx_ctx_create(sp, len(sp), ip, secret, len(secret) if secret else 0, 0, 4, ctypes.byref(h)) == OK
        try:
            calls = {
                "host": lambda n, ms=B, kp=B: L.afx_derive_keypairs(h, n, ms, kp),
                "device": lambda n, ms=B, kp=B: L.afx_derive_keypairs_device(h, n, ms, kp, None),
            }
            for name, call in calls.items():
                assert call(0) == OK, name
                assert call(0, ms=None, kp=None) == OK, name      # null buffers are fine when there is nothing to read or write
                assert call(1, ms=None) == ARG, name
                assert call(1, kp=None) == ARG, name
            assert calls["device"](5) == ARG                       # more than max_batch
            t = [ctypes.c_uint64(), ctypes.c_uint64()]
            for k in range(2):                                     # verifying issuances needs no issuer secret
                assert L.afx_verify_issuances_wire_submit(h, 4, bytes([0, 0, 2, 2]), 0, None, None, ctypes.byref(t[k])) == OK
            for name, call in calls.items():
                assert call(0) == ARG, name
                assert call(1) == ARG, name
            assert calls["device"](5) == ARG
            for k in range(2):
                assert L.afx_wait(h, t[k].value) == OK
            assert calls["host"](0) == OK and calls["device"](0) == OK
        finally:
            L.afx_ctx_destroy(h)


def test_python_wrappers_validate_arrays(emu):
    iss = issuer(emu, "issuer4.bin", 4)
    with pytest.raises(ValueError):
        iss.derive_keypairs(np.zeros((2, 63), np.uint8))
    with pytest.raises(ValueError):
        iss.derive_keypairs(np.zeros(64, np.uint8))
    with pytest.raises(ValueError):
        iss.derive_keypairs(np.zeros((2, 64), np.uint8), out=np.zeros((2, 4, 32), np.uint8))
    with pytest.raises(ValueError):
        iss.derive_keypairs(np.zeros((2, 64), np.uint8), out=np.zeros((2, 128), np.uint16))
    iss.close()


def test_round_trip_under_derived_keypairs(binding):
    rng = np.random.default_rng(96)
    iss = issuer(binding, "issuer4.bin", 3)
    kps = iss.derive_keypairs(rng.integers(0, 256, (2, 64), dtype=np.uint8))
    data = rng.integers(0, 256, (5, 30), dtype=np.uint8)
    pts, s0 = iss.encode_plaintexts(data)
    cts, s1 = iss.encrypt(kps[0, :96].tobytes(), pts)
    back, s2 = iss.decrypt(kps[0, :96].tobytes(), cts)
    assert not (s0.any() or s1.any() or s2.any()) and back.tobytes() == data.tobytes()
    back, s3 = iss.decrypt(kps[1].tobytes(), cts)                 # the 128-byte form is taken too
    assert s3.all() and not back.any()
    iss.close()


def test_readme4_presentations_with_per_item_keypairs(binding):
    """encode -> issue -> show -> verify -> decrypt on README-4 items, each with its own derived keypair."""
    import bench
    from aeonflux_b200 import Issuer, RequestBatch
    sp, ip, sk = bench.load_issuer("issuer4.bin")
    count = 6
    rng = np.random.default_rng(128)
    iss = Issuer(sp, ip, sk, device=0, max_batch=4, _binding=binding)
    kps = iss.derive_keypairs(rng.integers(0, 256, (count, 64), dtype=np.uint8))
    assert len({k.tobytes() for k in kps}) == count
    data = rng.integers(0, 256, (count, 30), dtype=np.uint8)
    pts, st = iss.encode_plaintexts(data)
    assert not st.any()
    sc = rng.integers(0, 256, (count, 2, 32), dtype=np.uint8)
    sc[:, :, 31] &= 0x0f
    pt2, _ = iss.selftest_primitive("from_uniform", rng.integers(0, 256, (count, 64), dtype=np.uint8))
    attrs = np.stack([sc[:, 0], sc[:, 1], pt2, pts[:, 0]], axis=1)
    cred, st = iss.issue_batch(RequestBatch.from_request(bytes([0, 0, 2, 2]), attrs, rng.integers(0, 256, (count, 11, 64), dtype=np.uint8)))
    assert not st.any()
    kp_rows = kps.reshape(count, 4, 32).transpose(1, 0, 2)         # a, a0, a1, pk rows, one keypair per item
    rnd = rng.integers(0, 256, (2 * (1 + 3 + 1 + 6), count, 32), dtype=np.uint8)
    fields = np.concatenate([cred.fields[4:7], np.stack([sc[:, 0], sc[:, 1], pt2, pts[:, 0], pts[:, 1], pts[:, 2]]), kp_rows, rnd])
    pres, st = iss.show_batch(KINDS4, fields)
    assert not st.any()
    assert not iss.verify_batch(pres).any()
    e1 = hidden_plaintext_blocks(KINDS4)[0]
    assert pres.fields[e1 - 1].tobytes() == kps[:, 96:].tobytes()   # each presentation carries its item's pk
    ct = np.ascontiguousarray(pres.fields[e1:e1 + 2].transpose(1, 0, 2))
    for i in range(count):
        back, st = iss.decrypt(kps[i, :96].tobytes(), ct[i:i + 1])
        assert st[0] == 0 and back[0].tobytes() == data[i].tobytes(), i
        back, st = iss.decrypt(kps[(i + 1) % count, :96].tobytes(), ct[i:i + 1])
        assert st[0] == 1 and not back.any(), i
    iss.close()


CPP = r"""
#include <cstdio>
#include <fstream>
#include <iterator>
#include "aeonflux_b200.hpp"
int main(int, char** argv) {
    std::ifstream f(argv[1], std::ios::binary);
    std::vector<uint8_t> blob((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    aeonflux::Issuer iss = aeonflux::Issuer::from_bytes(blob, 0, 2);
    std::vector<aeonflux::MasterSecret> ms(3);
    for (size_t i = 0; i < ms.size(); i++) for (size_t k = 0; k < 64; k++) ms[i][k] = (uint8_t)(i * 64 + k);
    std::vector<aeonflux::Keypair> kp = iss.derive_keypairs(ms);
    for (const aeonflux::Keypair& k : kp) {
        for (uint8_t b : k.secret) std::printf("%02x", b);
        for (uint8_t b : k.pk) std::printf("%02x", b);
        std::printf("\n");
    }
    return 0;
}
"""


def test_cpp_mirror_on_emulation(emu, tmp_path):
    """aeonflux::Issuer::derive_keypairs (include/aeonflux_b200.hpp) over the host emulation, in passes of 2."""
    from tests.test_host_logic import build_hostemu
    so = build_hostemu()
    src, exe = tmp_path / "derive.cpp", str(tmp_path / "derive")
    src.write_text(CPP)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src),
                           "-L" + os.path.dirname(so), "-lafx_hostemu", "-Wl,-rpath," + os.path.dirname(so)])
    out = subprocess.run([exe, os.path.join(ROOT, "bench_data", "issuer4.bin")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    ms = np.arange(192, dtype=np.uint8).reshape(3, 64)
    assert out.stdout.split() == [k.tobytes().hex() for k in issuer(emu, "issuer4.bin", 4).derive_keypairs(ms)]


# ---- full size, on the GPU ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_full_size_device_form_against_the_c_oracle():
    import bench
    import torch
    from tests.symoracle import derive as derive_oracle
    N, MB = 65536, 16384
    sp, ip, _ = bench.load_issuer("issuer4.bin")
    rng = np.random.default_rng(65536)
    ms = rng.integers(0, 256, (N, 64), dtype=np.uint8)
    iss = issuer(None, "issuer4.bin", MB)
    d_ms = torch.from_numpy(ms).cuda()
    d_kp = torch.empty((4, N, 32), dtype=torch.uint8, device="cuda")
    for lo in range(0, N, MB):                                    # device calls take at most max_batch items: passes of MB
        kp_pass = torch.empty((4, MB, 32), dtype=torch.uint8, device="cuda")
        iss.derive_keypairs_device(MB, d_ms[lo:lo + MB].data_ptr(), kp_pass.data_ptr())
        torch.cuda.synchronize()
        d_kp[:, lo:lo + MB] = kp_pass
    got = d_kp.cpu().numpy().transpose(1, 0, 2).reshape(N, 128)
    expect, _ = derive_oracle.derive(sp, ip, ms)
    assert (got == expect).all()
    assert (iss.derive_keypairs(ms[:40000]) == expect[:40000]).all()      # the host form, in passes of max_batch
    iss.close()


@pytest.mark.gpu
def test_s16_batch_with_per_item_keypairs_built_on_the_device():
    """derive -> encode -> issue -> show on the device, one derived keypair per item; every item verifies and decrypts."""
    import bench
    import torch
    from aeonflux_b200 import Issuer
    B, n = 4096, 16
    sp, ip, sk = bench.load_issuer("issuer16.bin")
    iss = Issuer(sp, ip, sk, device=0, max_batch=B)
    rng = np.random.default_rng(1616)
    s = torch.cuda.current_stream().cuda_stream
    ms = rng.integers(0, 256, (B, 64), dtype=np.uint8)
    kp = torch.empty((4, B, 32), dtype=torch.uint8, device="cuda")
    iss.derive_keypairs_device(B, torch.from_numpy(ms).cuda().data_ptr(), kp.data_ptr(), s)
    data = rng.integers(0, 256, (8, B, 30), dtype=np.uint8)
    d_data = torch.from_numpy(data).cuda()
    pts = torch.empty((8, 3, B, 32), dtype=torch.uint8, device="cuda")
    status = torch.empty(B, dtype=torch.uint8, device="cuda")
    for j in range(8):
        iss.encode_plaintexts_device(B, d_data[j].data_ptr(), pts[j].data_ptr(), status.data_ptr(), s)
        torch.cuda.synchronize()
        assert int(status.sum()) == 0
    sc = rng.integers(0, 256, (6, B, 32), dtype=np.uint8)
    sc[:, :, 31] &= 0x0f
    pp, _ = iss.selftest_primitive("from_uniform", rng.integers(0, 256, (2 * B, 64), dtype=np.uint8))
    pp = torch.from_numpy(pp.reshape(2, B, 32)).cuda()
    d_sc = torch.from_numpy(sc).cuda()
    attr = [d_sc[k] for k in range(6)] + [pp[0], pp[1]] + [pts[j, 0] for j in range(8)]
    req = torch.cat([torch.stack(attr), torch.from_numpy(rng.integers(0, 256, (2 * (n + 7), B, 32), dtype=np.uint8)).cuda()])
    cred = torch.empty((n + 9, B, 32), dtype=torch.uint8, device="cuda")
    iss.issue_batch_device(bytes(0 if k in (0, 1) else 2 for k in KINDS16), B, req.data_ptr(), cred.data_ptr(), status.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(status.sum()) == 0
    show_attr = [d_sc[k:k + 1] for k in range(6)] + [pp[0:1], pp[1:2]] + [pts[j] for j in range(8)]
    rnd = torch.from_numpy(rng.integers(0, 256, (2 * (1 + 3 + 2 + 6 * 8), B, 32), dtype=np.uint8)).cuda()
    show_in = torch.cat([cred[0:3]] + show_attr + [kp, rnd])        # the derived rows, as they are
    assert show_in.shape[0] == iss._b.L.afx_show_num_fields(n, KINDS16)
    pres = torch.empty((iss.num_fields(KINDS16), B, 32), dtype=torch.uint8, device="cuda")
    iss.show_batch_device(KINDS16, B, show_in.data_ptr(), pres.data_ptr(), status.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(status.sum()) == 0
    verdicts = torch.empty(B, dtype=torch.uint8, device="cuda")
    iss.verify_batch_device(KINDS16, B, pres.data_ptr(), verdicts.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(verdicts.sum()) == 0
    kps = kp.cpu().numpy().transpose(1, 0, 2).reshape(B, 128)
    assert len({k.tobytes() for k in kps}) == B
    pres_h = pres.cpu().numpy()
    blocks = hidden_plaintext_blocks(KINDS16)
    for i in rng.choice(B, 32, replace=False):
        assert all(pres_h[e1 - 1, i].tobytes() == kps[i, 96:].tobytes() for e1 in blocks)
        ct = np.ascontiguousarray(np.stack([pres_h[e1:e1 + 2, i] for e1 in blocks]))   # the item's 8 ciphertexts
        back, st = iss.decrypt(kps[i, :96].tobytes(), ct)
        assert not st.any() and back.tobytes() == data[:, i].tobytes(), i
    iss.close()
