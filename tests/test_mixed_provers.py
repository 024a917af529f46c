"""Issuing and showing over records of several shapes of one issuer in one call, bucketed by shape on the device
(afx_issue_mixed_wire, afx_show_mixed_wire, afx_multi_issue_mixed_wire; include/aeonflux_b200.h).

Checked on the host emulation and, with -m gpu, on the CUDA library:
- parity: outputs and status byte-identical to the per-shape *_wire calls on the same records and to the C oracle, for requests of
  three request kinds and for show inputs of the four README-4 disclosure patterns, the SURVEY A.6 quirk shapes and an S16 mix,
  with malformed records interleaved at random (status 1 and a zero record exactly where they sit) and a kind vector listed twice;
- round trip: the outputs are what the mixed verify calls take;
- passes of max_batch records of any mix (one-shape passes, absent shapes, a short tail; on the GPU passes that cross the
  256-record tile boundary and end in a partial tile); permuting the records permutes the outputs;
- the exact return code of every precondition, with nothing written to the outputs or the status;
- the multi-device handle gives the single-context bytes; the C++ overloads;
- on the GPU, 65,536 README-4 show inputs in four patterns, 65,536 requests in three kinds and an 8,192-record S16 mix, compared in
  full with the per-shape wire calls."""
import ctypes
import importlib.util
import os
import subprocess
import struct

import numpy as np
import pytest

from aeonflux_b200.shard import interleave_records

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, ARG, SHAPE, NO_SECRET = 0, -1, -5, -6
REQUESTS4 = [b"SSPP", b"SPSP", b"PPPP"]                                                          # request kinds [0,0,2,2] [0,2,0,2] [2,2,2,2]
README4_PATTERNS = [(b"SSPE", [0, 3]), (b"SSPE", [3]), (b"SSPE", [0, 1, 3]), (b"SSPE", [])]     # [SS,PS,PP,SP] [PS,PS,PP,SP] [SS,SS,PP,SP] [PS,PS,PP,PP]
QUIRK_PATTERNS = [(b"ESS", [0]), (b"SES", [1]), (b"SES", [])]                                  # [SP,PS,PS] [PS,SP,PS] [PS,PP,PS]
S16_PATTERNS = [(b"SSSSSSPP" + b"E" * 8, [0, 1] + list(range(8, 16))), (b"SSSSSSPP" + b"E" * 8, list(range(12, 16)))]


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


def scale(binding, emu, small, large):
    return small if binding is emu else large


def shuffled_order(counts, rng):
    return rng.permutation(np.repeat(np.arange(len(counts), dtype=np.uint8), counts)).astype(np.uint8)


def in_record_order(per_shape, order):
    """Arrays per shape (in the shape's own order, first axis = item) -> one array in record order (every shape's items equal-sized)."""
    out = np.zeros((len(order),) + per_shape[0].shape[1:], per_shape[0].dtype)
    for s, v in enumerate(per_shape):
        out[np.nonzero(order == s)[0]] = v
    return out


def make_requests(orc, request_kinds, counts, tag, rng, fraction):
    """Per request kind vector: (kinds, requests [count][3n + 14][32], the oracle's issuances [count][2n + 9][32] (zero where
    malformed), the oracle's status).  ~fraction of the requests are malformed: an undecodable point attribute or a scalar >= l."""
    from aeonflux_b200 import RequestBatch
    out = []
    for k, (rk, cnt) in enumerate(zip(request_kinds, counts)):
        _, _, issu = orc.synth(rk, [], b"%s-%d" % (tag, k), 0, cnt)
        ik = bytes(0 if c == ord("S") else 2 for c in rk)
        n = len(ik)
        A = np.ascontiguousarray(issu[:, :n])
        R = rng.integers(0, 256, (cnt, n + 7, 64), dtype=np.uint8)
        for j, i in enumerate(np.nonzero(rng.random(cnt) < fraction)[0]):
            a = [x for x in range(n) if ik[x] == (2 if j % 2 else 0)] or list(range(n))
            x = a[int(rng.integers(len(a)))]
            if ik[x] == 2:
                A[i, x] = 0; A[i, x, 0] = 1                 # s = 1 is negative: no Ristretto point encodes to it
            else:
                A[i, x] = 0xff                              # a scalar >= l
        o, st, _ = orc.issue(ik, A, R)
        expect = np.concatenate([A, o], axis=1)
        expect[st == 1] = 0
        reqs = np.ascontiguousarray(RequestBatch.from_request(ik, A, R).fields.transpose(1, 0, 2))
        out.append((ik, reqs, expect, st))
    return out


def make_show_inputs(orc, patterns, counts, tag, rng, fraction):
    """Per pattern: (kinds, show inputs [count][Ws][32], the oracle's presentations (zero where malformed), status).  ~fraction of
    the inputs are malformed: t not a canonical scalar, or U not a point encoding."""
    out = []
    for k, ((rk, hide), cnt) in enumerate(zip(patterns, counts)):
        kinds, pres, _, showin = orc.synth(rk, hide, b"%s-%d" % (tag, k), 0, cnt, want_issuances=False, want_show_inputs=True)
        st = np.zeros(cnt, np.uint8)
        for j, i in enumerate(np.nonzero(rng.random(cnt) < fraction)[0]):
            if j % 2:
                showin[i, 1] = 0; showin[i, 1, 0] = 1
            else:
                showin[i, 0, 31] = 0xff
            st[i] = 1
        pres = pres.copy()
        pres[st == 1] = 0
        out.append((kinds, np.ascontiguousarray(showin), pres, st))
    return out


def per_shape_show(iss, pools, order):
    """The per-shape afx_show_wire calls, outputs interleaved in record order, and the status."""
    res = [iss.show_wire(k, x) for k, x, _, _ in pools]
    return interleave_records([r[0] for r in res], order)[0], in_record_order([r[1] for r in res], order)


def test_issue_parity(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(31)
    counts = scale(binding, emu, [9, 8, 10], [900, 800, 1000])
    pools = make_requests(orc, REQUESTS4, counts, b"mixiss", rng, 0.15)
    kinds_list = [p[0] for p in pools]
    assert [list(k) for k in kinds_list] == [[0, 0, 2, 2], [0, 2, 0, 2], [2, 2, 2, 2]]
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records([p[1] for p in pools], order)
    iss = Issuer(sp, ip, sk, max_batch=scale(binding, emu, 8, 65536), _binding=binding)
    out, st = iss.issue_mixed_wire(kinds_list, blob, order)
    expect, est = in_record_order([p[2] for p in pools], order), in_record_order([p[3] for p in pools], order)
    assert 0 < int(est.sum()) < len(order)
    assert (st == est).all() and (out == expect).all(), np.nonzero((out != expect).any(axis=(1, 2)))[0][:10]
    wire = [iss.issue_wire(k, r) for k, r, _, _ in pools]
    assert (out == in_record_order([w[0] for w in wire], order)).all() and (st == in_record_order([w[1] for w in wire], order)).all()
    assert not out[st == 1].any()
    # the same kind vector listed twice: records of either id get the same bytes
    dup = order.copy()
    dup[(order == 0) & (np.arange(len(order)) % 2 == 1)] = 3
    out2, st2 = iss.issue_mixed_wire(kinds_list + [kinds_list[0]], blob, dup)
    assert (out2 == out).all() and (st2 == st).all()
    # round trip: what the mixed issuance verifier takes, on a context without the issuer secret
    user = Issuer(sp, ip, None, max_batch=scale(binding, emu, 8, 65536), _binding=binding)
    assert (user.verify_mixed_wire(kinds_list, out, order, issuance=True) == st).all()


def check_show(binding, emu, coracle, n, patterns, counts, tag, seed, max_batch, expect_kinds=None):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(n)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(seed)
    pools = make_show_inputs(orc, patterns, counts, tag, rng, 0.15)
    kinds_list = [p[0] for p in pools]
    if expect_kinds:
        assert [list(k) for k in kinds_list] == expect_kinds
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records([p[1] for p in pools], order)
    user = Issuer(sp, ip, None, max_batch=max_batch, _binding=binding)          # showing needs no issuer secret
    out, st = user.show_mixed_wire(kinds_list, blob, order)
    expect, _ = interleave_records([p[2] for p in pools], order)
    est = in_record_order([p[3] for p in pools], order)
    assert 0 < int(est.sum()) < len(order)
    assert (st == est).all() and (out == expect).all()
    wire, wst = per_shape_show(user, pools, order)
    assert (out == wire).all() and (st == wst).all()
    off = user.presentation_offsets(kinds_list, order)
    assert off[-1] == out.size
    for i in np.nonzero(st)[0]:
        assert not out[off[i]:off[i + 1]].any()                                  # a zero record exactly where the malformed input sits
    # round trip: the blob is what the mixed verifier takes; it agrees with the oracle's verdicts
    iss = Issuer(sp, ip, sk, max_batch=max_batch, _binding=binding)
    v = iss.verify_mixed_wire(kinds_list, out, order)
    ov = []
    for s, (kinds, _, _, _) in enumerate(pools):
        recs = np.stack([out[off[i]:off[i + 1]].reshape(-1, 32) for i in np.nonzero(order == s)[0]])
        ov.append(orc.verify_presentations(kinds, np.ascontiguousarray(recs))[0])
    assert (v == in_record_order(ov, order)).all()
    assert (v[st == 1] == 1).all()
    return user, iss, kinds_list, pools, order, blob, out, st, v


def test_show_parity_readme4(binding, emu, coracle):
    counts = scale(binding, emu, [7, 6, 5, 8], [700, 600, 500, 800])
    user, iss, kinds_list, pools, order, blob, out, st, v = check_show(
        binding, emu, coracle, 4, README4_PATTERNS, counts, b"mixshow4", 32, scale(binding, emu, 8, 65536),
        [[1, 0, 2, 3], [0, 0, 2, 3], [1, 1, 2, 3], [0, 0, 2, 2]])
    assert (v == st).all()                                                       # every honest presentation verifies
    dup = order.copy()
    dup[(order == 1) & (np.arange(len(order)) % 2 == 0)] = 4
    out2, st2 = user.show_mixed_wire(kinds_list + [kinds_list[1]], blob, dup)
    assert (out2 == out).all() and (st2 == st).all()


def test_show_parity_quirk_shapes(binding, emu, coracle):
    counts = scale(binding, emu, [5, 6, 5], [500, 600, 500])
    *_, v = check_show(binding, emu, coracle, 3, QUIRK_PATTERNS, counts, b"mixquirk", 33, scale(binding, emu, 8, 65536),
                       [[3, 0, 0], [0, 3, 0], [0, 2, 0]])


def test_show_parity_s16(binding, emu, coracle):
    counts = scale(binding, emu, [3, 3], [150, 130])
    check_show(binding, emu, coracle, 16, S16_PATTERNS, counts, b"mixs16", 34, scale(binding, emu, 4, 65536))


def test_passes_of_any_mix(binding, coracle):
    """50 records over max_batch = 8: a pass of one shape only, shapes absent from some passes, a final pass of 2 records; permuting
    the records permutes the outputs."""
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(35)
    order = np.array([1] * 8 + [0, 2, 0, 2, 2, 0, 0, 2] + [3, 1, 0, 3, 3, 1, 2, 0] + [2, 2, 2, 2, 0, 2, 2, 2] +
                     [1, 3, 1, 3, 1, 3, 1, 1] + [0, 1, 2, 3, 3, 2, 1, 0] + [3, 0], np.uint8)
    counts = [int((order == s).sum()) for s in range(4)]
    pools = make_show_inputs(orc, README4_PATTERNS, counts, b"mixpass", rng, 0.1)
    kinds_list = [p[0] for p in pools]
    blob, in_off = interleave_records([p[1] for p in pools], order)
    iss = Issuer(sp, ip, sk, max_batch=8, _binding=binding)
    out, st = iss.show_mixed_wire(kinds_list, blob, order)
    expect, _ = interleave_records([p[2] for p in pools], order)
    assert (out == expect).all() and (st == in_record_order([p[3] for p in pools], order)).all()
    sizes = [p[1].shape[1] * 32 for p in pools]
    off = iss.presentation_offsets(kinds_list, order)
    recs = [blob[int(o):int(o) + sizes[s]] for o, s in zip(in_off, order)]
    perm = np.random.default_rng(1).permutation(len(order))
    out_p, st_p = iss.show_mixed_wire(kinds_list, np.concatenate([recs[i] for i in perm]), order[perm])
    assert (out_p == np.concatenate([out[off[i]:off[i + 1]] for i in perm])).all() and (st_p == st[perm]).all()
    # requests: three kinds, one absent from the first pass, passes of 8 and a tail of 3
    rorder = np.array([0, 1] * 4 + [2] * 8 + [2, 1, 0, 2, 1, 0, 2, 1] + [0, 2, 0], np.uint8)
    rpools = make_requests(orc, REQUESTS4, [int((rorder == s).sum()) for s in range(3)], b"mixpassreq", rng, 0.1)
    rk = [p[0] for p in rpools]
    rblob, _ = interleave_records([p[1] for p in rpools], rorder)
    rout, rst = iss.issue_mixed_wire(rk, rblob, rorder)
    assert (rout == in_record_order([p[2] for p in rpools], rorder)).all() and (rst == in_record_order([p[3] for p in rpools], rorder)).all()
    perm = np.random.default_rng(2).permutation(len(rorder))
    rrecs = rblob.reshape(len(rorder), -1)
    rout_p, rst_p = iss.issue_mixed_wire(rk, rrecs[perm], rorder[perm])
    assert (rout_p == rout[perm]).all() and (rst_p == rst[perm]).all()


@pytest.mark.gpu
def test_passes_cross_tile_boundaries(coracle):
    """1,100 records over max_batch = 600: pass 0 is tiles [0, 256), [256, 512) and a partial [512, 600); pass 1 has 500 records,
    one full tile and a partial one."""
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(36)
    counts = [300, 250, 270, 280]
    pools = make_show_inputs(orc, README4_PATTERNS, counts, b"mixtile", rng, 0.02)
    kinds_list = [p[0] for p in pools]
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records([p[1] for p in pools], order)
    iss = Issuer(sp, ip, sk, max_batch=600)
    out, st = iss.show_mixed_wire(kinds_list, blob, order)
    wire, wst = per_shape_show(iss, pools, order)
    assert (out == wire).all() and (st == wst).all()
    assert (out == interleave_records([p[2] for p in pools], order)[0]).all()
    rpools = make_requests(orc, REQUESTS4, [400, 350, 350], b"mixtilereq", rng, 0.02)
    rorder = shuffled_order([400, 350, 350], rng)
    rblob, _ = interleave_records([p[1] for p in rpools], rorder)
    rout, rst = iss.issue_mixed_wire([p[0] for p in rpools], rblob, rorder)
    assert (rout == in_record_order([p[2] for p in rpools], rorder)).all() and (rst == in_record_order([p[3] for p in rpools], rorder)).all()
    iss.close()


# ---- preconditions (host emulation: the checks run before any device work) ---------------------------------------------------

K4 = [bytes([1, 0, 2, 3]), bytes([0, 0, 2, 2])]
R4 = [bytes([0, 0, 2, 2]), bytes([2, 2, 2, 2])]
DUMMY = ctypes.c_void_p(16)        # a non-null "buffer" that no failing check dereferences


@pytest.fixture(scope="module")
def contexts(emu, coracle):
    sp, ip, sk = (bytes(x) for x in coracle.make_issuer(4))
    L, hs = emu.L, []
    for secret in (sk, None):
        h = ctypes.c_void_p()
        assert L.afx_ctx_create(sp, len(sp), ip, secret, len(secret) if secret else 0, 0, 4, ctypes.byref(h)) == OK
        hs.append(h)
    m = ctypes.c_void_p()
    devs = (ctypes.c_int * 3)(0, 0, 0)
    assert L.afx_multi_create(sp, len(sp), ip, sk, len(sk), devs, 3, 4, ctypes.byref(m)) == OK
    yield hs + [m]
    L.afx_multi_destroy(m)
    for h in hs:
        L.afx_ctx_destroy(h)


def call(L, name, h, kinds_list, ids=(0, 1, 1), null=(), n=4, n_shapes=None):
    """afx_<name> over the given shapes and ids; returns (rc, outputs, status), outputs and status starting as all 7."""
    issue = "issue" in name
    ids = np.asarray(ids, np.uint8)
    fit = [i for i in ids if i < len(kinds_list)]
    nin = sum((3 * n + 14) if issue else L.afx_show_num_fields(n, kinds_list[i]) for i in fit)
    nout = sum((2 * n + 9) if issue else L.afx_presentation_num_fields(n, kinds_list[i]) for i in fit)
    inputs = np.zeros(32 * nin, np.uint8)
    out = np.full(32 * nout + 64, 7, np.uint8)
    status = np.full(len(ids), 7, np.uint8)
    args = [h, n, None if "kinds" in null else b"".join(kinds_list), len(kinds_list) if n_shapes is None else n_shapes, len(ids),
            None if "inputs" in null else inputs.ctypes.data, None if "ids" in null else ids.ctypes.data,
            None if "out" in null else out.ctypes.data, None if "status" in null else status.ctypes.data]
    return getattr(L, "afx_" + name)(*args), out, status


NAMES = ["issue_mixed_wire", "show_mixed_wire", "multi_issue_mixed_wire"]


@pytest.mark.parametrize("name", NAMES)
def test_return_codes(emu, contexts, name):
    L, (ctx, user, multi) = emu.L, contexts
    issue = "issue" in name
    kinds = R4 if issue else K4
    h = multi if name.startswith("multi") else ctx

    def check(expect, **kw):
        rc, out, st = call(L, name, kw.pop("h", h), kw.pop("kinds_list", kinds), **kw)
        assert rc == expect, (kw, rc)
        if rc != OK:
            assert (out == 7).all() and (st == 7).all(), kw            # nothing written on an error
        else:
            assert (out[-64:] == 7).all()                              # nothing written past the outputs
        return out, st

    assert call(L, name, None, kinds)[0] == ARG
    check(ARG, n_shapes=0)
    check(ARG, ids=(), n_shapes=0)
    check(ARG, kinds_list=kinds * 128, n_shapes=256)                   # more than 255 shapes
    check(ARG, ids=(0, 2, 1))                                          # a shape id >= n_shapes
    check(ARG, ids=(0, 1, 255))
    for ptr in ("inputs", "ids", "out", "status", "kinds"):
        check(ARG, null=(ptr,))
    assert call(L, name, h, kinds, ids=(), null=("inputs", "ids", "out", "status"))[0] == OK      # count = 0
    check(ARG, ids=(), null=("kinds",))
    check(OK, ids=())
    check(SHAPE, kinds_list=[kinds[0], bytes([0, 0, 2, 9])])           # a kind byte no shape has
    check(SHAPE, kinds_list=[bytes([0, 0, 2])], ids=(0,), n=3)         # an attribute count different from the issuer's
    if issue:
        check(SHAPE, kinds_list=[kinds[0], bytes([1, 0, 2, 2])])       # a hidden kind in a request
        check(SHAPE, kinds_list=[kinds[0], bytes([0, 0, 2, 3])])
    out, st = check(OK, kinds_list=kinds * 127 + [kinds[0]], ids=(0, 254, 3, 254))    # 255 shapes
    assert (st <= 1).all()
    check(ARG, kinds_list=kinds * 127 + [kinds[0]], ids=(0, 255))
    if not name.startswith("multi"):
        check(NO_SECRET if issue else OK, h=user)
        check(NO_SECRET if issue else SHAPE, h=user, kinds_list=[kinds[0], bytes([0, 0, 2, 9])])
        t = [ctypes.c_uint64(), ctypes.c_uint64()]
        for k in range(2):
            assert L.afx_verify_presentations_wire_submit(ctx, 4, K4[0], 0, DUMMY, DUMMY, ctypes.byref(t[k])) == OK
        check(ARG)                                                     # submissions outstanding
        check(ARG, kinds_list=[kinds[0], bytes([0, 0, 2, 9])])         # refused before the shape is compiled
        for k in range(2):
            assert L.afx_wait(ctx, t[k].value) == OK
        check(OK)


def test_python_wrapper_checks_lengths(emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    iss = Issuer(sp, ip, sk, max_batch=4, _binding=emu)
    with pytest.raises(ValueError):
        iss.issue_mixed_wire(R4, np.zeros((3 * 4 + 14) * 32 + 32, np.uint8), [0])
    with pytest.raises(ValueError):
        iss.show_mixed_wire([K4[0], bytes([0, 0, 2])], np.zeros(32, np.uint8), [0])
    with pytest.raises(ValueError):
        iss.issue_mixed_wire(R4, np.zeros((3 * 4 + 14) * 32, np.uint8), [0], out=np.zeros(32, np.uint8))
    out, st = iss.issue_mixed_wire(R4, np.zeros(0, np.uint8), [])
    assert out.shape == (0, 17, 32) and len(st) == 0


def test_multi_device_handle(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    from aeonflux_b200.shard import MultiGpuIssuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(37)
    counts = scale(binding, emu, [5, 6, 4], [3000, 2500, 2000])
    pools = make_requests(orc, REQUESTS4, counts, b"mixmulti", rng, 0.1)
    kinds_list = [p[0] for p in pools]
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records([p[1] for p in pools], order)
    mb = scale(binding, emu, 4, 4096)
    single = Issuer(sp, ip, sk, max_batch=mb, _binding=binding).issue_mixed_wire(kinds_list, blob, order)
    m = MultiGpuIssuer(sp, ip, sk, devices=scale(binding, emu, [0, 0, 0], [0, 0]), max_batch=mb, _binding=binding)
    out, st = m.issue_mixed_wire(kinds_list, blob, order)
    assert (out == single[0]).all() and (st == single[1]).all()
    assert (out == in_record_order([p[2] for p in pools], order)).all()
    assert len(m.issue_mixed_wire(kinds_list, blob[:0], order[:0])[1]) == 0
    m.close()


# ---- the C++ overloads -----------------------------------------------------------------------------------------------------------

def run_cpp(tmp_path, coracle, lib_dir, lib_name, counts, max_batch):
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(38)
    rpools = make_requests(orc, REQUESTS4, counts, b"mixcpp", rng, 0.1)
    spools = make_show_inputs(orc, README4_PATTERNS, counts + [counts[0]], b"mixcppshow", rng, 0.1)
    rorder, sorder = shuffled_order(counts, rng), shuffled_order(counts + [counts[0]], rng)
    rblob, _ = interleave_records([p[1] for p in rpools], rorder)
    sblob, _ = interleave_records([p[1] for p in spools], sorder)
    fx, res = tmp_path / "mixed.bin", tmp_path / "mixed.out"
    with open(fx, "wb") as f:
        for b in (bytes(sp) + bytes(ip) + bytes(sk), bytes([4]), b"".join(p[0] for p in rpools), rblob.tobytes(), rorder.tobytes(),
                  b"".join(p[0] for p in spools), sblob.tobytes(), sorder.tobytes()):
            f.write(struct.pack("<Q", len(b))); f.write(b)
    exe = str(tmp_path / "mixed_provers")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, os.path.join(ROOT, "tests", "cpp", "mixed_provers.cpp"),
                           "-L" + lib_dir, "-l" + lib_name, "-Wl,-rpath," + lib_dir])
    r = subprocess.run([exe, str(fx), str(res), str(max_batch)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "mixed_provers ok" in r.stdout, r.stdout + r.stderr
    got = []
    with open(res, "rb") as f:
        for _ in range(5):
            (k,) = struct.unpack("<Q", f.read(8))
            got.append(np.frombuffer(f.read(k), np.uint8))
    rout, rst, sout, sst, verdicts = got
    assert (rout.reshape(len(rorder), 17, 32) == in_record_order([p[2] for p in rpools], rorder)).all()
    assert (rst == in_record_order([p[3] for p in rpools], rorder)).all()
    assert (sout == interleave_records([p[2] for p in spools], sorder)[0]).all()
    assert (sst == in_record_order([p[3] for p in spools], sorder)).all() and (verdicts == sst).all()
    return r.stdout


def test_cpp_overloads_on_emulation(tmp_path, coracle):
    from tests.test_host_logic import build_hostemu
    so = build_hostemu()
    assert "host-emulation" in run_cpp(tmp_path, coracle, os.path.dirname(so), "afx_hostemu", [4, 5, 3], 4)


@pytest.mark.gpu
def test_cpp_overloads_on_gpu(tmp_path, coracle):
    from aeonflux_b200.build import CSRC
    assert "cuda sm_100a" in run_cpp(tmp_path, coracle, CSRC, "aeonflux_b200", [300, 200, 250], 256)


# ---- full size on the GPU ------------------------------------------------------------------------------------------------------

def bench_tool():
    spec = importlib.util.spec_from_file_location("bench_mixed_provers", os.path.join(ROOT, "tools", "bench_mixed_provers.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def flip_records(pools, order, fraction, rng, word):
    """Set word `word` of ~fraction of the records to 0xff..ff (not a canonical scalar, not a point encoding); returns their mask."""
    bad = np.zeros(len(order), bool)
    bad[rng.choice(len(order), int(len(order) * fraction), replace=False)] = True
    for s, p in enumerate(pools):
        p[bad[order == s], word] = 0xff
    return bad


@pytest.mark.gpu
def test_full_size_show_readme4_patterns():
    from aeonflux_b200 import Issuer
    from bench import load_issuer
    T = bench_tool()
    sp, ip, sk = load_issuer("issuer4.bin")
    iss = Issuer(sp, ip, sk, device=0, max_batch=65536)
    patterns = T.SHOW_PATTERNS
    pools = [T.show_inputs_on_device(iss, k, 16384, 90 + s) for s, k in enumerate(patterns)]
    rng = np.random.default_rng(7)
    order = shuffled_order([16384] * 4, rng)
    bad = flip_records(pools, order, 0.01, rng, 0)
    blob, _ = interleave_records(pools, order)
    pinned = iss.host_array(blob.shape)
    pinned[:] = blob
    out, st = iss.show_mixed_wire(patterns, pinned, order, out=iss.host_array(int(iss.presentation_offsets(patterns, order)[-1])))
    assert (st == bad).all()
    res = [iss.show_wire(k, p) for k, p in zip(patterns, pools)]
    assert (out == interleave_records([r[0] for r in res], order)[0]).all()
    assert (st == in_record_order([r[1] for r in res], order)).all()
    assert (iss.verify_mixed_wire(patterns, out, order) == bad).all()
    iss.close()


@pytest.mark.gpu
def test_full_size_issue_three_kinds():
    from aeonflux_b200 import Issuer
    from bench import load_issuer
    T = bench_tool()
    sp, ip, sk = load_issuer("issuer4.bin")
    iss = Issuer(sp, ip, sk, device=0, max_batch=65536)
    counts = [21846, 21845, 21845]
    pools = [T.requests_for(iss, k, c, 95 + s) for s, (k, c) in enumerate(zip(T.REQUEST_KINDS, counts))]
    rng = np.random.default_rng(8)
    order = shuffled_order(counts, rng)
    bad = flip_records(pools, order, 0.01, rng, 1)
    blob, _ = interleave_records(pools, order)
    out, st = iss.issue_mixed_wire(T.REQUEST_KINDS, blob, order)
    assert (st == bad).all()
    res = [iss.issue_wire(k, p) for k, p in zip(T.REQUEST_KINDS, pools)]
    assert (out == in_record_order([r[0] for r in res], order)).all() and (st == in_record_order([r[1] for r in res], order)).all()
    assert (iss.verify_mixed_wire(T.REQUEST_KINDS, out, order, issuance=True) == bad).all()
    iss.close()


@pytest.mark.gpu
def test_s16_mix():
    from aeonflux_b200 import Issuer
    from bench import KINDS_S16, load_issuer
    T = bench_tool()
    sp, ip, sk = load_issuer("issuer16.bin")
    iss = Issuer(sp, ip, sk, device=0, max_batch=8192)
    patterns = [KINDS_S16, bytes([0] * 6 + [2, 2] + [3] * 4 + [2] * 4)]
    pools = [T.show_inputs_on_device(iss, k, 4096, 97 + s, "keypair16.bin") for s, k in enumerate(patterns)]
    rng = np.random.default_rng(9)
    order = shuffled_order([4096, 4096], rng)
    bad = flip_records(pools, order, 0.01, rng, 0)
    blob, _ = interleave_records(pools, order)
    out, st = iss.show_mixed_wire(patterns, blob, order)
    assert (st == bad).all()
    res = [iss.show_wire(k, p) for k, p in zip(patterns, pools)]
    assert (out == interleave_records([r[0] for r in res], order)[0]).all()
    assert (iss.verify_mixed_wire(patterns, out, order) == bad).all()
    iss.close()
