"""Presentations (and issuances) of several disclosure patterns of one issuer in one call, bucketed by shape on the device
(afx_verify_{presentations,issuances}_mixed_wire and their afx_multi_* forms; include/aeonflux_b200.h).

Checked on the host emulation and, with -m gpu, on the CUDA library:
- parity: the verdicts equal the per-shape *_wire calls on the same records and the C oracle's, for the four disclosure patterns of
  request SSPE and for the SURVEY A.6 quirk shapes, with corrupted records interleaved at random and a kind vector listed twice;
- permuting the records permutes the verdicts; passes of max_batch records of any mix (one-shape passes, absent shapes, a short tail);
- issuances of three request kinds, on a context without the issuer secret;
- the exact return code of every precondition, with nothing written to the verdicts;
- the multi-device handle gives the single-context verdicts;
- on the GPU, 65,536 distinct README-4 presentations in four patterns and an 8,192-record S16 mix."""
import ctypes

import numpy as np
import pytest

from aeonflux_b200.shard import interleave_records
from tests.common import corrupt_batch

OK, ARG, SHAPE, NO_SECRET = 0, -1, -5, -6
README4_PATTERNS = [(b"SSPE", [0, 3]), (b"SSPE", [3]), (b"SSPE", [0, 1, 3]), (b"SSPE", [])]     # [SS,PS,PP,SP] [PS,PS,PP,SP] [SS,SS,PP,SP] [PS,PS,PP,PP]
QUIRK_PATTERNS = [(b"ESS", [0]), (b"SES", [1]), (b"SES", [])]                                  # [SP,PS,PS] [PS,SP,PS] [PS,PP,PS]


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


def make_pools(orc, patterns, counts, tag, rng, fraction):
    """Presentations of every pattern (kinds, items), ~fraction of each pattern's items corrupted, and the oracle's verdicts."""
    kinds_list, pools, expect = [], [], []
    for k, ((rk, hide), cnt) in enumerate(zip(patterns, counts)):
        kinds, pres, _ = orc.synth(rk, hide, b"%s-%d" % (tag, k), 0, cnt, want_issuances=False)
        pts = pres[:4, 4:7].reshape(-1, 32).copy()
        corrupt_batch(pres, kinds, rng, fraction, pts)
        kinds_list.append(kinds); pools.append(pres); expect.append(orc.verify_presentations(kinds, pres)[0])
    return kinds_list, pools, expect


def in_record_order(per_shape, order):
    """Verdicts per shape (in the shape's own order) -> verdicts in record order."""
    out = np.zeros(len(order), np.uint8)
    for s, v in enumerate(per_shape):
        out[np.nonzero(order == s)[0]] = v
    return out


def shuffled_order(counts, rng):
    return rng.permutation(np.repeat(np.arange(len(counts), dtype=np.uint8), counts)).astype(np.uint8)


def split_records(blob, offsets, sizes, order):
    return [blob[int(o):int(o) + int(sizes[s])] for o, s in zip(offsets, order)]


def test_parity_readme4_patterns(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(11)
    counts = scale(binding, emu, [13, 11, 9, 12], [1500, 1300, 1100, 1200])
    kinds_list, pools, expect = make_pools(orc, README4_PATTERNS, counts, b"mix4", rng, 0.05 if binding is not emu else 0.15)
    assert [list(k) for k in kinds_list] == [[1, 0, 2, 3], [0, 0, 2, 3], [1, 1, 2, 3], [0, 0, 2, 2]]
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records(pools, order)
    iss = Issuer(sp, ip, sk, max_batch=scale(binding, emu, 64, 65536), _binding=binding)
    v = iss.verify_mixed_wire(kinds_list, blob, order)
    oracle = in_record_order(expect, order)
    assert 0 < int(oracle.sum()) < len(order)
    assert (v == oracle).all(), np.nonzero(v != oracle)[0][:10]
    per_shape = in_record_order([iss.verify_wire(k, p) for k, p in zip(kinds_list, pools)], order)
    assert (v == per_shape).all()
    # the same kind vector listed twice: records of either id get the verdicts of their shape
    dup = order.copy()
    dup[(order == 0) & (np.arange(len(order)) % 2 == 1)] = 4
    assert (iss.verify_mixed_wire(kinds_list + [kinds_list[0]], blob, dup) == oracle).all()


def test_parity_quirk_shapes(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(3)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(12)
    counts = scale(binding, emu, [7, 9, 8], [700, 900, 800])
    kinds_list, pools, expect = make_pools(orc, QUIRK_PATTERNS, counts, b"quirk", rng, 0.05)
    assert [list(k) for k in kinds_list] == [[3, 0, 0], [0, 3, 0], [0, 2, 0]]
    assert expect[0].all()                                      # [SP,PS,PS] never verifies (SURVEY A.6)
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records(pools, order)
    iss = Issuer(sp, ip, sk, max_batch=scale(binding, emu, 16, 65536), _binding=binding)
    v = iss.verify_mixed_wire(kinds_list, blob, order)
    assert (v == in_record_order(expect, order)).all()


def test_permuting_records_permutes_verdicts(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(13)
    counts = scale(binding, emu, [6, 5, 7, 6], [600, 500, 700, 600])
    kinds_list, pools, _ = make_pools(orc, README4_PATTERNS, counts, b"perm", rng, 0.2)
    order = shuffled_order(counts, rng)
    blob, offsets = interleave_records(pools, order)
    iss = Issuer(sp, ip, sk, max_batch=scale(binding, emu, 10, 1000), _binding=binding)
    v = iss.verify_mixed_wire(kinds_list, blob, order)
    sizes = [p.shape[1] * 32 for p in pools]
    recs = split_records(blob, offsets, sizes, order)
    for seed in (1, 2):
        perm = np.random.default_rng(seed).permutation(len(order))
        blob2 = np.concatenate([recs[i] for i in perm])
        assert (iss.verify_mixed_wire(kinds_list, blob2, order[perm]) == v[perm]).all()


def test_passes_of_any_mix(binding, coracle):
    """50 records over max_batch = 8: a pass of one shape only, shapes absent from some passes, a final pass of 2 records."""
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(14)
    order = np.array([1] * 8 +                                  # pass 0: shape 1 only
                     [0, 2, 0, 2, 2, 0, 0, 2] +                 # pass 1: shapes 1 and 3 absent
                     [3, 1, 0, 3, 3, 1, 2, 0] +
                     [2, 2, 2, 2, 0, 2, 2, 2] +
                     [1, 3, 1, 3, 1, 3, 1, 1] +
                     [0, 1, 2, 3, 3, 2, 1, 0] +
                     [3, 0], np.uint8)                          # pass 6: two records
    counts = [int((order == s).sum()) for s in range(4)]
    kinds_list, pools, expect = make_pools(orc, README4_PATTERNS, counts, b"passes", rng, 0.15)
    blob, _ = interleave_records(pools, order)
    iss = Issuer(sp, ip, sk, max_batch=8, _binding=binding)
    v = iss.verify_mixed_wire(kinds_list, blob, order)
    oracle = in_record_order(expect, order)
    assert 0 < int(oracle.sum()) and (v == oracle).all(), np.nonzero(v != oracle)[0]
    assert (v == in_record_order([iss.verify_wire(k, p) for k, p in zip(kinds_list, pools)], order)).all()


def test_issuances_of_several_request_kinds(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(15)
    requests = [b"SSPP", b"SPSP", b"PPPP"]
    counts = scale(binding, emu, [9, 8, 10], [900, 800, 1000])
    kinds_list, pools, expect = [], [], []
    for k, (rk, cnt) in enumerate(zip(requests, counts)):
        _, _, issu = orc.synth(rk, [], b"issu-%d" % k, 0, cnt)
        ik = bytes(0 if c == ord("S") else 2 for c in rk)
        for j, i in enumerate(np.nonzero(rng.random(cnt) < 0.1)[0]):
            issu[i, int(rng.integers(issu.shape[1])), 31 if j % 3 == 0 else int(rng.integers(32))] ^= 1 << int(rng.integers(8))
        kinds_list.append(ik); pools.append(issu); expect.append(orc.verify_issuances(ik, issu)[0])
    assert [list(k) for k in kinds_list] == [[0, 0, 2, 2], [0, 2, 0, 2], [2, 2, 2, 2]]
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records(pools, order)
    user = Issuer(sp, ip, None, max_batch=scale(binding, emu, 12, 65536), _binding=binding)      # needs no issuer secret
    v = user.verify_mixed_wire(kinds_list, blob, order, issuance=True)
    oracle = in_record_order(expect, order)
    assert 0 < int(oracle.sum()) and (v == oracle).all()
    assert (v == in_record_order([user.verify_wire(k, p, issuance=True) for k, p in zip(kinds_list, pools)], order)).all()


# ---- preconditions (host emulation: the checks run before any device work) ---------------------------------------------------

K4 = [bytes([1, 0, 2, 3]), bytes([0, 0, 2, 2])]
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


def call(L, name, h, kinds_list=K4, ids=(0, 1, 1), records="fit", null=(), n=4, n_shapes=None):
    """afx_<name> over the given shapes and ids; returns (rc, the verdict array, which starts as all 7)."""
    issuance = "issuances" in name
    nf = [(2 * n + 9) if issuance else L.afx_presentation_num_fields(n, k) for k in kinds_list]
    ids = np.asarray(ids, np.uint8)
    rec = np.zeros(sum(32 * nf[i] for i in ids if i < len(nf)) if records == "fit" else 0, np.uint8)
    verdicts = np.full(len(ids), 7, np.uint8)
    blob = b"".join(kinds_list)
    args = [h, n, None if "kinds" in null else blob, len(kinds_list) if n_shapes is None else n_shapes, len(ids),
            None if "records" in null else rec.ctypes.data, None if "ids" in null else ids.ctypes.data,
            None if "verdicts" in null else verdicts.ctypes.data]
    return getattr(L, "afx_" + name)(*args), verdicts


NAMES = ["verify_presentations_mixed_wire", "verify_issuances_mixed_wire", "multi_verify_presentations_mixed_wire",
         "multi_verify_issuances_mixed_wire"]


@pytest.mark.parametrize("name", NAMES)
def test_return_codes(emu, contexts, name):
    L, (ctx, user, multi) = emu.L, contexts
    issuance = "issuances" in name
    kinds = [bytes([0, 0, 2, 2]), bytes([2, 2, 2, 2])] if issuance else K4
    h = multi if name.startswith("multi") else ctx

    def check(expect, **kw):
        rc, v = call(L, name, kw.pop("h", h), kinds_list=kw.pop("kinds_list", kinds), **kw)
        assert rc == expect, (kw, rc)
        if rc != OK:
            assert (v == 7).all(), kw                             # nothing written on an error
        return v

    assert call(L, name, None, kinds)[0] == ARG
    check(ARG, n_shapes=0)
    check(ARG, ids=(), n_shapes=0)
    check(ARG, kinds_list=kinds * 128, n_shapes=256)              # more than 255 shapes
    check(ARG, ids=(0, 2, 1))                                     # a shape id >= n_shapes
    check(ARG, ids=(0, 1, 255))
    for ptr in ("records", "ids", "verdicts", "kinds"):
        check(ARG, null=(ptr,))
    assert call(L, name, h, kinds, ids=(), null=("records", "ids", "verdicts"))[0] == OK      # count = 0
    check(ARG, ids=(), null=("kinds",))
    check(OK, ids=())
    check(SHAPE, kinds_list=[kinds[0], bytes([0, 0, 2, 9])])                                  # a kind vector the issuer cannot verify
    check(SHAPE, kinds_list=[bytes([0, 0, 2])], ids=(0,), n=3)                                # an attribute count different from the issuer's
    if issuance:
        check(SHAPE, kinds_list=[kinds[0], bytes([1, 0, 2, 2])])                              # a hidden kind in a request
    v = check(OK, kinds_list=kinds * 127 + [kinds[0]], ids=(0, 254, 3, 254))                  # 255 shapes; all-zero records are rejected
    assert (v == 1).all()
    kinds255 = kinds * 127 + [kinds[0]]
    check(ARG, kinds_list=kinds255, ids=(0, 255))
    if not name.startswith("multi"):
        check(OK if issuance else NO_SECRET, h=user)
        check(NO_SECRET if not issuance else SHAPE, h=user, kinds_list=[kinds[0], bytes([0, 0, 2, 9])])
        t = [ctypes.c_uint64(), ctypes.c_uint64()]
        for k in range(2):
            assert L.afx_verify_presentations_wire_submit(ctx, 4, K4[0], 0, DUMMY, DUMMY, ctypes.byref(t[k])) == OK
        check(ARG)                                                # submissions outstanding
        check(ARG, kinds_list=[kinds[0], bytes([0, 0, 2, 9])])    # refused before the shape is compiled
        for k in range(2):
            assert L.afx_wait(ctx, t[k].value) == OK
        check(OK)


def test_python_wrapper_checks_the_blob_length(emu, coracle):
    from aeonflux_b200 import Issuer
    sp, ip, sk = coracle.make_issuer(4)
    iss = Issuer(sp, ip, sk, max_batch=4, _binding=emu)
    nf = iss.num_fields(K4[0])
    with pytest.raises(ValueError):
        iss.verify_mixed_wire(K4, np.zeros(nf * 32 + 32, np.uint8), [0])
    with pytest.raises(ValueError):
        iss.verify_mixed_wire([K4[0], bytes([0, 0, 2])], np.zeros(nf * 32, np.uint8), [0])


def test_multi_device_handle(binding, emu, coracle):
    from aeonflux_b200 import Issuer
    from aeonflux_b200.shard import MultiGpuIssuer
    sp, ip, sk = coracle.make_issuer(4)
    orc = coracle.Issuer(sp, ip, sk)
    rng = np.random.default_rng(16)
    counts = scale(binding, emu, [8, 7, 9, 6], [3000, 2500, 2000, 2700])
    kinds_list, pools, expect = make_pools(orc, README4_PATTERNS, counts, b"multi", rng, 0.1)
    order = shuffled_order(counts, rng)
    blob, _ = interleave_records(pools, order)
    mb = scale(binding, emu, 4, 4096)
    single = Issuer(sp, ip, sk, max_batch=mb, _binding=binding).verify_mixed_wire(kinds_list, blob, order)
    m = MultiGpuIssuer(sp, ip, sk, devices=scale(binding, emu, [0, 0, 0], [0, 0]), max_batch=mb, _binding=binding)
    assert (m.verify_mixed_wire(kinds_list, blob, order) == single).all()
    assert (single == in_record_order(expect, order)).all()
    assert len(m.verify_mixed_wire(kinds_list, blob[:0], order[:0])) == 0
    m.close()


# ---- full size on the GPU ------------------------------------------------------------------------------------------------------

def device_pools(torch, iss, patterns, per_pattern, seed, keypair_file):
    from bench import synthesize_on_device
    pools = []
    for k, kinds in enumerate(patterns):
        dev = synthesize_on_device(torch, iss, per_pattern, seed + k, torch.cuda.current_stream(), kinds, keypair_file)
        pools.append(np.ascontiguousarray(dev.cpu().numpy().transpose(1, 0, 2)))
        del dev
    return pools


def flip_bits(pools, order, fraction, rng):
    """One flipped bit in ~fraction of the records (any word, byte 31 every fourth time); returns the expected verdicts."""
    expect = np.zeros(len(order), np.uint8)
    bad = rng.choice(len(order), int(len(order) * fraction), replace=False)
    expect[bad] = 1
    for j, i in enumerate(bad):
        s = order[i]
        item = int((order[:i] == s).sum())
        p = pools[s]
        p[item, rng.integers(0, p.shape[1]), 31 if j % 4 == 0 else rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)
    return expect


@pytest.mark.gpu
def test_full_size_readme4_patterns(coracle):
    import torch
    from aeonflux_b200 import Issuer
    from bench import load_issuer
    sp, ip, sk = load_issuer("issuer4.bin")
    orc = coracle.Issuer(sp, ip, sk)
    iss = Issuer(sp, ip, sk, device=0, max_batch=65536)
    patterns = [bytes([1, 0, 2, 3]), bytes([0, 0, 2, 3]), bytes([1, 1, 2, 3]), bytes([0, 0, 2, 2])]
    pools = device_pools(torch, iss, patterns, 16384, 90, "keypair4.bin")
    assert len(np.unique(np.concatenate([p[:, 4:7].reshape(16384, -1) for p in pools]), axis=0)) == 65536   # distinct records
    rng = np.random.default_rng(5)
    order = shuffled_order([16384] * 4, rng)
    expect = flip_bits(pools, order, 0.01, rng)
    blob, offsets = interleave_records(pools, order)
    pinned = iss.host_array(blob.shape)
    pinned[:] = blob
    v = iss.verify_mixed_wire(patterns, pinned, order)
    assert (v == expect).all(), np.nonzero(v != expect)[0][:10]
    sample = rng.choice(65536, 4096, replace=False)
    got = np.zeros(len(sample), np.uint8)
    for s, kinds in enumerate(patterns):
        sel = np.nonzero(order[sample] == s)[0]
        items = np.stack([blob[int(offsets[sample[j]]):int(offsets[sample[j]]) + pools[s].shape[1] * 32].reshape(-1, 32) for j in sel])
        got[sel] = orc.verify_presentations(kinds, np.ascontiguousarray(items))[0]
    assert (v[sample] == got).all()
    iss.close()


@pytest.mark.gpu
def test_s16_two_patterns(coracle):
    import torch
    from aeonflux_b200 import Issuer
    from bench import KINDS_S16, load_issuer
    sp, ip, sk = load_issuer("issuer16.bin")
    orc = coracle.Issuer(sp, ip, sk)
    iss = Issuer(sp, ip, sk, device=0, max_batch=8192)
    patterns = [KINDS_S16, bytes([0] * 6 + [2, 2] + [3] * 4 + [2] * 4)]
    pools = device_pools(torch, iss, patterns, 4096, 95, "keypair16.bin")
    rng = np.random.default_rng(6)
    order = shuffled_order([4096, 4096], rng)
    expect = flip_bits(pools, order, 0.01, rng)
    blob, _ = interleave_records(pools, order)
    v = iss.verify_mixed_wire(patterns, blob, order)
    assert (v == expect).all(), np.nonzero(v != expect)[0][:10]
    assert (v == in_record_order([iss.verify_wire(k, p) for k, p in zip(patterns, pools)], order)).all()
    for s, kinds in enumerate(patterns):
        ov, _ = orc.verify_presentations(kinds, np.ascontiguousarray(pools[s][:96]))
        pos = np.nonzero(order == s)[0][:96]
        assert (v[pos] == ov).all()
    iss.close()
