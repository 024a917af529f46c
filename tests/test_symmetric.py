"""Symmetric encryption of attributes (Plaintext::from, Keypair::encrypt, Keypair::decrypt; include/aeonflux_b200.h): parity with the
oracle's recorded answers (tests/golden/symmetric.json), passes of max_batch items, rejections, the exact precondition codes, and
presentations built from real plaintexts that verify and decrypt.  Every case runs on the host emulation and, under -m gpu, on the
CUDA library; the full-size cases run on the GPU only."""
import ctypes
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, ARG, ENCODING = 0, -1, -2
L_ORDER = 2**252 + 27742317777372353535851937790883648493
KINDS4 = bytes([1, 0, 2, 3])
KINDS16 = bytes([1, 1, 0, 0, 0, 0, 2, 2] + [3] * 8)


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
    with open(os.path.join(ROOT, "tests", "golden", "symmetric.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def issuer4(coracle):
    return coracle.make_issuer(4)


def user(binding, issuer_material, max_batch):
    """A user-side context (no issuer secret)."""
    from aeonflux_b200 import Issuer
    sp, ip, _ = issuer_material
    return Issuer(sp, ip, None, device=0, max_batch=max_batch, _binding=binding)


def rows(hexes, width):
    return np.array([list(bytes.fromhex(h)) for h in hexes], np.uint8).reshape(len(hexes), width)


def golden_arrays(g):
    data = rows([it["data"] for it in g["items"]], 30)
    pts = rows(["".join(it["plaintext"]) for it in g["items"]], 96).reshape(-1, 3, 32)
    cts = rows(["".join(it["ciphertext"]) for it in g["items"]], 64).reshape(-1, 2, 32)
    return data, pts, cts


def test_golden_covers_the_edge_cases(golden):
    assert golden["items"][32]["data"] == "00" * 30 and golden["items"][32]["plaintext"][0] == "00" * 32   # M1 = identity
    assert max(it["candidates"] for it in golden["items"]) >= 20


def test_encode_matches_oracle(binding, golden, issuer4):
    data, pts, _ = golden_arrays(golden)
    out, status = user(binding, issuer4, 16).encode_plaintexts(data)
    assert not status.any()
    assert out.tobytes() == pts.tobytes()


def test_encrypt_matches_oracle_in_passes(binding, golden, issuer4):
    _, pts, cts = golden_arrays(golden)
    iss = user(binding, issuer4, 3)                       # 10 items in passes of 3
    out, status = iss.encrypt(bytes.fromhex(golden["keypair"]), pts[:10])
    assert not status.any()
    assert out.tobytes() == cts[:10].tobytes()
    bad = pts[:4].copy()
    bad[0, 0] = 0xff                                      # M1 undecodable
    bad[1, 1, 0] = 1                                      # M2 undecodable (negative)
    bad[2, 2] = np.frombuffer(L_ORDER.to_bytes(32, "little"), np.uint8)   # m3 = l
    out, status = iss.encrypt(bytes.fromhex(golden["keypair"]), bad)
    assert list(status) == [1, 1, 1, 0] and not out[:3].any() and out[3].tobytes() == cts[3].tobytes()


def test_decrypt_matches_oracle(binding, golden, issuer4):
    cases = golden["decrypt"]
    iss = user(binding, issuer4, 8)
    for which in ("keypair", "other"):
        sel = [c for c in cases if c["keypair"] == which]
        ct = rows(["".join(c["ciphertext"]) for c in sel], 64).reshape(-1, 2, 32)
        data, pts, status = iss.decrypt(bytes.fromhex(golden[which]), ct, plaintexts=True)
        for k, c in enumerate(sel):
            if c["result"] is None:
                assert status[k] == 1 and not data[k].any() and not pts[k].any(), c["case"]
            else:
                assert status[k] == 0, c["case"]
                assert data[k].tobytes().hex() == c["result"]["data"]
                assert pts[k].tobytes().hex() == "".join(c["result"]["plaintext"])
    assert {c["case"] for c in cases if c["result"] is None} == {"wrong keypair", "another item's E2", "E1 and E2 swapped", "undecodable E1"}


def test_round_trip(binding, golden, issuer4):
    data, _, _ = golden_arrays(golden)
    iss = user(binding, issuer4, 5)
    kp = bytes.fromhex(golden["keypair"])
    pts, s0 = iss.encode_plaintexts(data)
    cts, s1 = iss.encrypt(kp, pts)
    back, pts2, s2 = iss.decrypt(kp, cts, plaintexts=True)
    assert not (s0.any() or s1.any() or s2.any())
    assert back.tobytes() == data.tobytes() and pts2.tobytes() == pts.tobytes()
    back, s3 = iss.decrypt(bytes.fromhex(golden["other"]), cts)
    assert s3.all() and not back.any()


def test_preconditions(emu, golden, issuer4):
    L = emu.L
    sp, ip, sk = issuer4
    kp = bytes.fromhex(golden["keypair"])
    a_plus_l = (int.from_bytes(kp[:32], "little") + L_ORDER).to_bytes(32, "little") + kp[32:]
    buf = (ctypes.c_uint8 * 4096)()
    B = ctypes.addressof(buf)
    for secret in (sk, None):                             # a user-side context works like an issuer's
        h = ctypes.c_void_p()
        assert L.afx_ctx_create(sp, len(sp), ip, secret, len(secret) if secret else 0, 0, 4, ctypes.byref(h)) == OK
        try:
            calls = {
                "encode": lambda n, k=kp, p=B: L.afx_encode_plaintexts(h, n, p, p, p),
                "encrypt": lambda n, k=kp, p=B: L.afx_encrypt(h, k, n, p, p, p),
                "decrypt": lambda n, k=kp, p=B: L.afx_decrypt(h, k, n, p, p, None, p),
                "encode_device": lambda n, k=kp, p=B: L.afx_encode_plaintexts_device(h, n, p, p, p, None),
                "encrypt_device": lambda n, k=kp, p=B: L.afx_encrypt_device(h, k, n, p, p, p, None),
                "decrypt_device": lambda n, k=kp, p=B: L.afx_decrypt_device(h, k, n, p, p, None, p, None),
            }
            for name, call in calls.items():
                assert call(0) == OK, name
                assert call(1, p=None) == ARG, name
                assert call(0, p=None) == OK, name            # null buffers are fine when there is nothing to read or write
                if name.startswith(("encrypt", "decrypt")):
                    assert call(0, k=None) == ARG, name
                    assert call(1, k=a_plus_l) == ENCODING, name
                    assert call(0, k=a_plus_l) == ENCODING, name
                if name.endswith("_device"):
                    assert call(5) == ARG, name               # more than max_batch
            assert L.afx_decrypt_device(h, kp, 1, B, B, None, None, None) == ARG     # status is required
            if secret:
                t = [ctypes.c_uint64(), ctypes.c_uint64()]
                for k in range(2):
                    assert L.afx_verify_presentations_wire_submit(h, 4, KINDS4, 0, None, None, ctypes.byref(t[k])) == OK
                for name, call in calls.items():
                    assert call(0) == ARG, name
                    if name.startswith(("encrypt", "decrypt")):
                        assert call(0, k=a_plus_l) == ARG, name   # the busy check comes first
                for k in range(2):
                    assert L.afx_wait(h, t[k].value) == OK
                assert calls["encode"](0) == OK
        finally:
            L.afx_ctx_destroy(h)
    # nothing is written when the keypair is refused
    h = ctypes.c_void_p()
    assert L.afx_ctx_create(sp, len(sp), ip, None, 0, 0, 4, ctypes.byref(h)) == OK
    try:
        iss_in = np.zeros((2, 2, 32), np.uint8)
        out = np.full((2, 30), 7, np.uint8)
        st = np.full(2, 7, np.uint8)
        assert L.afx_decrypt(h, a_plus_l, 2, iss_in.ctypes.data, out.ctypes.data, None, st.ctypes.data) == ENCODING
        assert (out == 7).all() and (st == 7).all()
    finally:
        L.afx_ctx_destroy(h)


def test_python_wrappers_validate_arrays(emu, issuer4):
    iss = user(emu, issuer4, 4)
    with pytest.raises(ValueError):
        iss.encode_plaintexts(np.zeros((2, 31), np.uint8))
    with pytest.raises(ValueError):
        iss.encode_plaintexts(np.zeros((2, 30), np.uint8), out=np.zeros((2, 3, 32), np.uint16))
    with pytest.raises(ValueError):
        iss.encrypt(bytes(96), np.zeros((2, 2, 32), np.uint8))
    with pytest.raises(ValueError):
        iss.decrypt(bytes(95), np.zeros((2, 2, 32), np.uint8))
    with pytest.raises(ValueError):
        iss.decrypt(bytes(96), np.zeros((2, 2, 32), np.uint8), out=np.zeros((3, 30), np.uint8))


def hidden_plaintext_blocks(kinds):
    """Word index of E1 in each proof-of-encryption block of a presentation of `kinds` (E2 follows)."""
    n, h_s = len(kinds), sum(k == 1 for k in kinds)
    pos = 1 + 3 + h_s + 3 + n + sum(k in (0, 2) for k in kinds)
    return [pos + 14 * j + 8 for j in range(sum(k == 3 for k in kinds))]


def show_inputs(kinds, attrs, kp128, rng):
    """Flat afx_show input rows after the credential words: attributes, keypair, rng words (include/aeonflux_b200.h)."""
    h_s, h_p = sum(k == 1 for k in kinds), sum(k == 3 for k in kinds)
    count = attrs[0].shape[0]
    return np.concatenate([np.stack(attrs), np.broadcast_to(np.frombuffer(kp128, np.uint8).reshape(4, 1, 32), (4, count, 32)),
                           rng.integers(0, 256, (2 * (1 + 3 + h_s + 6 * h_p), count, 32), dtype=np.uint8)])


def test_presentations_with_real_plaintexts_verify_and_decrypt(binding, coracle):
    """encode -> issue -> show -> verify -> decrypt on README-4 items with the bench issuer and keypair."""
    import bench
    from aeonflux_b200 import Issuer, PresentationBatch, RequestBatch
    sp, ip, sk = bench.load_issuer("issuer4.bin")
    kp128 = open(os.path.join(ROOT, "bench_data", "keypair4.bin"), "rb").read()
    count = 6
    rng = np.random.default_rng(5)
    iss = Issuer(sp, ip, sk, device=0, max_batch=4, _binding=binding)
    data = rng.integers(0, 256, (count, 30), dtype=np.uint8)
    data[0] = 0
    pts, st = iss.encode_plaintexts(data)
    assert not st.any()
    sc = rng.integers(0, 256, (count, 2, 32), dtype=np.uint8)
    sc[:, :, 31] &= 0x0f
    pt2, _ = iss.selftest_primitive("from_uniform", rng.integers(0, 256, (count, 64), dtype=np.uint8))
    attrs = np.stack([sc[:, 0], sc[:, 1], pt2, pts[:, 0]], axis=1)
    req = RequestBatch.from_request(bytes([0, 0, 2, 2]), attrs, rng.integers(0, 256, (count, 11, 64), dtype=np.uint8))
    cred, st = iss.issue_batch(req)
    assert not st.any()
    show_attr = [sc[:, 0], sc[:, 1], pt2, pts[:, 0], pts[:, 1], pts[:, 2]]
    fields = np.concatenate([cred.fields[4:7], show_inputs(KINDS4, show_attr, kp128, rng)])
    pres, st = iss.show_batch(KINDS4, fields)
    assert not st.any()
    assert not iss.verify_batch(pres).any()
    e1 = hidden_plaintext_blocks(KINDS4)[0]
    ct = np.ascontiguousarray(pres.fields[e1:e1 + 2].transpose(1, 0, 2))
    back, st = iss.decrypt(kp128, ct)
    assert not st.any() and back.tobytes() == data.tobytes()


# ---- full size, on the GPU ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_full_size_device_calls_against_the_c_oracle(issuer4):
    import torch
    from tests import symoracle
    from aeonflux_b200 import Issuer
    N, MB = 65536, 16384
    rng = np.random.default_rng(65536)
    kp = open(os.path.join(ROOT, "bench_data", "keypair4.bin"), "rb").read()[:96]
    sp, ip, _ = issuer4
    iss = Issuer(sp, ip, None, device=0, max_batch=MB)
    data = rng.integers(0, 256, (N, 30), dtype=np.uint8)
    d_data = torch.from_numpy(data).cuda()
    d_pt = torch.empty((3, N, 32), dtype=torch.uint8, device="cuda")
    d_ct = torch.empty((2, N, 32), dtype=torch.uint8, device="cuda")
    d_back = torch.empty((N, 30), dtype=torch.uint8, device="cuda")
    d_pt2 = torch.empty((3, N, 32), dtype=torch.uint8, device="cuda")
    st = [torch.empty(N, dtype=torch.uint8, device="cuda") for _ in range(3)]
    tamper = rng.choice(N, N // 100, replace=False)
    for lo in range(0, N, MB):                            # device calls take at most max_batch items: passes of MB
        hi = lo + MB
        pt_pass = torch.empty((3, MB, 32), dtype=torch.uint8, device="cuda")
        ct_pass = torch.empty((2, MB, 32), dtype=torch.uint8, device="cuda")
        iss.encode_plaintexts_device(MB, d_data[lo:hi].data_ptr(), pt_pass.data_ptr(), st[0][lo:hi].data_ptr())
        iss.encrypt_device(kp, MB, pt_pass.data_ptr(), ct_pass.data_ptr(), st[1][lo:hi].data_ptr())
        torch.cuda.synchronize()
        d_pt[:, lo:hi] = pt_pass
        d_ct[:, lo:hi] = ct_pass
    assert int(st[0].sum()) == 0 and int(st[1].sum()) == 0
    ct_host = d_ct.cpu().numpy().transpose(1, 0, 2).copy()
    pt_host = d_pt.cpu().numpy().transpose(1, 0, 2).copy()
    other = ct_host[(tamper + 1) % N, 1].copy()
    ct_host[tamper, 1] = other                            # E2 := another item's E2
    d_ct = torch.from_numpy(np.ascontiguousarray(ct_host.transpose(1, 0, 2))).cuda()
    for lo in range(0, N, MB):
        hi = lo + MB
        ct_pass = d_ct[:, lo:hi].contiguous()
        pt_pass = torch.empty((3, MB, 32), dtype=torch.uint8, device="cuda")
        iss.decrypt_device(kp, MB, ct_pass.data_ptr(), d_back[lo:hi].data_ptr(), st[2][lo:hi].data_ptr(), pt_pass.data_ptr())
        torch.cuda.synchronize()
        d_pt2[:, lo:hi] = pt_pass
    status = st[2].cpu().numpy()
    assert set(np.flatnonzero(status)) == set(tamper.tolist())
    ok = status == 0
    back = d_back.cpu().numpy()
    assert (back[ok] == data[ok]).all() and not back[~ok].any()
    assert (d_pt2.cpu().numpy().transpose(1, 0, 2)[ok] == pt_host[ok]).all()
    # the host calls, in passes of max_batch, agree with the device calls
    pts_h, s = iss.encode_plaintexts(data[:40000])
    assert not s.any() and (pts_h == pt_host[:40000]).all()
    # a 4,096-item sample against the C oracle
    sample = rng.choice(N, 4096, replace=False)
    opt, _ = symoracle.encode(data[sample])
    assert (opt == pt_host[sample]).all()
    oct_, ost, _ = symoracle.encrypt(kp, opt)
    assert not ost.any()
    assert (oct_[:, 0] == ct_host[sample, 0]).all()
    assert (oct_[:, 1][ok[sample]] == ct_host[sample, 1][ok[sample]]).all()
    odata, _, ost2, _ = symoracle.decrypt(kp, ct_host[sample])
    assert (ost2 == status[sample]).all() and (odata == back[sample]).all()
    iss.close()


@pytest.mark.gpu
def test_s16_batch_built_on_the_device_with_real_plaintexts():
    import torch
    import bench
    from aeonflux_b200 import Issuer
    B = 4096
    sp, ip, sk = bench.load_issuer("issuer16.bin")
    kp128 = open(os.path.join(ROOT, "bench_data", "keypair16.bin"), "rb").read()
    iss = Issuer(sp, ip, sk, device=0, max_batch=B)
    rng = np.random.default_rng(16)
    s = torch.cuda.current_stream().cuda_stream
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
    issue_kinds = bytes(0 if k in (0, 1) else 2 for k in KINDS16)
    n = 16
    req = torch.cat([torch.stack(attr), torch.from_numpy(rng.integers(0, 256, (2 * (n + 7), B, 32), dtype=np.uint8)).cuda()])
    cred = torch.empty((n + 9, B, 32), dtype=torch.uint8, device="cuda")
    iss.issue_batch_device(issue_kinds, B, req.data_ptr(), cred.data_ptr(), status.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(status.sum()) == 0
    show_attr = [d_sc[k:k + 1] for k in range(6)] + [pp[0:1], pp[1:2]] + [pts[j] for j in range(8)]
    kp = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(np.frombuffer(kp128, np.uint8).reshape(4, 1, 32), (4, B, 32)))).cuda()
    rnd = torch.from_numpy(rng.integers(0, 256, (2 * (1 + 3 + 2 + 6 * 8), B, 32), dtype=np.uint8)).cuda()
    show_in = torch.cat([cred[0:3]] + show_attr + [kp, rnd])
    assert show_in.shape[0] == iss._b.L.afx_show_num_fields(n, KINDS16)
    pres = torch.empty((iss.num_fields(KINDS16), B, 32), dtype=torch.uint8, device="cuda")
    iss.show_batch_device(KINDS16, B, show_in.data_ptr(), pres.data_ptr(), status.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(status.sum()) == 0
    verdicts = torch.empty(B, dtype=torch.uint8, device="cuda")
    iss.verify_batch_device(KINDS16, B, pres.data_ptr(), verdicts.data_ptr(), s)
    torch.cuda.synchronize()
    assert int(verdicts.sum()) == 0
    back = torch.empty((B, 30), dtype=torch.uint8, device="cuda")
    for j, e1 in enumerate(hidden_plaintext_blocks(KINDS16)):
        ct = pres[e1:e1 + 2].contiguous()
        iss.decrypt_device(kp128, B, ct.data_ptr(), back.data_ptr(), status.data_ptr(), None, s)
        torch.cuda.synchronize()
        assert int(status.sum()) == 0
        assert (back.cpu().numpy() == data[j]).all(), j
    iss.close()
