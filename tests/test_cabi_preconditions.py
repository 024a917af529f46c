"""Exact return codes of the C ABI's precondition checks (include/aeonflux_b200.h), on the host emulation through the raw
library: null arguments, batches larger than max_batch, a context without the issuer secret, invalid attribute kinds, a
field count that does not match the shape, and synchronous calls while submissions are outstanding.  Empty batches
(count = 0) pass every check that does not concern the buffers, so each case runs no kernel."""
import ctypes

import pytest

from aeonflux_b200._binding import afx_issuance_out, afx_presentation_batch

OK, ARG, SHAPE, NO_SECRET = 0, -1, -5, -6
N, MAX = 4, 4
KINDS = bytes([0, 0, 2, 2])       # presentation / request kinds the issuer of N attributes accepts
BAD = bytes([0, 0, 2, 9])         # kind 9 does not exist
HIDDEN = bytes([1, 0, 2, 3])      # a valid presentation shape, but hidden kinds cannot be issued or form an issuance
SEED = bytes(32)
DUMMY = ctypes.c_void_p(16)       # a non-null "buffer" that no failing check dereferences


@pytest.fixture(scope="module")
def L(coracle):
    from aeonflux_b200._binding import Binding
    from tests.test_host_logic import build_hostemu
    return Binding(ctypes.CDLL(build_hostemu())).L


@pytest.fixture(scope="module")
def issuer_material(coracle):
    return tuple(bytes(x) for x in coracle.make_issuer(N))


def make_ctx(L, issuer_material, with_secret):
    sp, ip, sk = issuer_material
    h = ctypes.c_void_p()
    assert L.afx_ctx_create(sp, len(sp), ip, sk if with_secret else None, len(sk) if with_secret else 0, 0, MAX, ctypes.byref(h)) == OK
    return h


@pytest.fixture(scope="module")
def ctx(L, issuer_material):
    h = make_ctx(L, issuer_material, True)
    yield h
    L.afx_ctx_destroy(h)


@pytest.fixture(scope="module")
def user_ctx(L, issuer_material):
    h = make_ctx(L, issuer_material, False)
    yield h
    L.afx_ctx_destroy(h)


class Calls:
    """Every entry point that takes a batch, called with (kinds, count, n_fields) and buffers that are null only where asked."""

    def __init__(self, L):
        self.L = L

    def soa(self, n, kinds, count, n_fields, null):
        fields = None if null else ctypes.cast((ctypes.c_void_p * max(n_fields, 1))(), ctypes.POINTER(ctypes.c_void_p))
        self.keep = afx_presentation_batch(n, kinds, count, fields, n_fields)
        return ctypes.byref(self.keep)

    def out(self, n_fields, null):
        fields = None if null else ctypes.cast((ctypes.c_void_p * max(n_fields, 1))(), ctypes.POINTER(ctypes.c_void_p))
        self.keep_out = afx_issuance_out(fields, n_fields)
        return ctypes.byref(self.keep_out)

    def nf(self, name, kinds):
        L = self.L
        if "issue" in name:
            return L.afx_request_num_fields(len(kinds))
        if "show" in name:
            return L.afx_show_num_fields(len(kinds), kinds)
        if "issuances_batchable" in name:
            return L.afx_issuance_batchable_num_fields(len(kinds))
        if "issuances" in name:
            return 2 * len(kinds) + 9
        if "batchable" in name:
            return L.afx_batchable_num_fields(len(kinds), kinds)
        return L.afx_presentation_num_fields(len(kinds), kinds)

    def out_nf(self, name, kinds):
        return len(kinds) + 9 if "issue" in name else self.L.afx_presentation_num_fields(len(kinds), kinds)

    def __call__(self, name, c, kinds=KINDS, count=0, null=False, nf_delta=0, out_nf_delta=0):
        """Calls afx_<name>; null = pass null for every data buffer (the context and kinds stay as given).  A submission that is
        accepted is waited for, so that the context is idle again."""
        ticket = ctypes.c_uint64()
        rc = self.call(name, c, kinds, count, null, nf_delta, out_nf_delta, ticket)
        if rc == OK and name.endswith("_submit"):
            assert self.L.afx_wait(c, ticket.value) == OK
        return rc

    def call(self, name, c, kinds, count, null, nf_delta, out_nf_delta, ticket):
        L, buf = self.L, (None if null else DUMMY)
        fn = getattr(L, "afx_" + name)
        n = N if kinds is None else len(kinds)
        nf = self.nf(name, KINDS if kinds is None else kinds) + nf_delta
        if name.endswith("_device"):
            if name in ("issue_device", "show_device"):
                return fn(c, n, kinds, count, buf, buf, buf, None)
            return fn(c, n, kinds, count, buf, buf, None)
        if name.endswith("wire_submit"):
            return fn(c, n, kinds, count, buf, buf, ctypes.byref(ticket))
        if name.endswith("_submit"):
            return fn(c, self.soa(n, kinds, count, nf, null), buf, ctypes.byref(ticket))
        if name.endswith("_rlc"):
            return fn(c, self.soa(n, kinds, count, nf, null), SEED, buf, None)
        if name.endswith("_wire"):
            if name in ("issue_wire", "show_wire", "show_linked_wire"):
                return fn(c, n, kinds, count, buf, buf, buf)
            return fn(c, n, kinds, count, buf, buf)
        if name in ("issue", "show", "show_linked"):
            return fn(c, self.soa(n, kinds, count, nf, null), self.out(self.out_nf(name, KINDS if kinds is None else kinds) + out_nf_delta, null), buf, None)
        return fn(c, self.soa(n, kinds, count, nf, null), buf, None)


PRESENTATION_VERIFY = ["verify_presentations", "verify_presentations_wire", "verify_presentations_device", "verify_presentations_batchable",
                       "verify_presentations_batchable_rlc", "verify_presentations_linked", "verify_presentations_linked_wire"]
PRESENTATION_SUBMIT = ["verify_presentations_submit", "verify_presentations_wire_submit"]
ISSUANCE_VERIFY = ["verify_issuances", "verify_issuances_wire", "verify_issuances_device", "verify_issuances_batchable",
                   "verify_issuances_batchable_rlc"]
ISSUANCE_SUBMIT = ["verify_issuances_submit", "verify_issuances_wire_submit"]
ISSUE = ["issue", "issue_wire", "issue_device"]
SHOW = ["show", "show_wire", "show_device", "show_linked", "show_linked_wire"]
SYNC = PRESENTATION_VERIFY + ISSUANCE_VERIFY + ISSUE + SHOW
ALL = SYNC + PRESENTATION_SUBMIT + ISSUANCE_SUBMIT
DEVICE = [n for n in ALL if n.endswith("_device")]
SOA = [n for n in ALL if not n.endswith(("_device", "_wire", "_wire_submit"))]


def kinds_for(name):
    return HIDDEN if name in PRESENTATION_VERIFY + PRESENTATION_SUBMIT + SHOW and "batchable" not in name else KINDS


@pytest.mark.parametrize("name", ALL)
def test_null_arguments(L, ctx, name):
    call = Calls(L)
    assert call(name, None) == ARG                                  # null context, empty batch
    assert call(name, None, count=1) == ARG
    assert call(name, ctx, kinds=None) == ARG                       # null kinds
    assert call(name, ctx, count=1, null=True) == ARG               # null buffers with items to process
    assert call(name, ctx, count=0, null=True) == OK                # ... which an empty batch does not need


@pytest.mark.parametrize("name", DEVICE + PRESENTATION_SUBMIT + ISSUANCE_SUBMIT)
def test_device_and_submit_calls_take_at_most_max_batch(L, ctx, user_ctx, name):
    call = Calls(L)
    assert call(name, ctx, count=MAX + 1) == ARG
    needs_secret = name in ("verify_presentations_device", "issue_device") or name in PRESENTATION_SUBMIT
    assert call(name, user_ctx, count=MAX + 1) == (NO_SECRET if needs_secret else ARG)     # the secret is checked first


@pytest.mark.parametrize("name", PRESENTATION_VERIFY + PRESENTATION_SUBMIT + ISSUE)
def test_calls_that_need_the_issuer_secret(L, user_ctx, name):
    call = Calls(L)
    assert call(name, user_ctx) == NO_SECRET
    assert call(name, user_ctx, kinds=BAD) == NO_SECRET             # before the shape is compiled
    assert call(name, user_ctx, nf_delta=1) == NO_SECRET


@pytest.mark.parametrize("name", ISSUANCE_VERIFY + ISSUANCE_SUBMIT + SHOW)
def test_calls_without_the_issuer_secret(L, user_ctx, name):
    assert Calls(L)(name, user_ctx, kinds=kinds_for(name)) == OK


def test_stream_shapes_and_the_issuer_secret(L, ctx, user_ctx):
    st = ctypes.c_void_p()
    assert L.afx_stream_create(ctypes.byref(st)) == OK
    sid, rb = ctypes.c_int(), ctypes.c_size_t()
    try:
        assert L.afx_stream_add_shape(st, user_ctx, 0, N, KINDS, ctypes.byref(sid), ctypes.byref(rb)) == NO_SECRET
        assert L.afx_stream_add_shape(st, user_ctx, 0, N, BAD, ctypes.byref(sid), ctypes.byref(rb)) == NO_SECRET
        assert L.afx_stream_add_shape(st, user_ctx, 1, N, KINDS, ctypes.byref(sid), ctypes.byref(rb)) == OK
        assert rb.value == (2 * N + 9) * 32
        assert L.afx_stream_add_shape(st, user_ctx, 1, N, BAD, ctypes.byref(sid), ctypes.byref(rb)) == SHAPE
        assert L.afx_stream_add_shape(st, user_ctx, 1, N, HIDDEN, ctypes.byref(sid), ctypes.byref(rb)) == SHAPE
        assert L.afx_stream_add_shape(st, ctx, 0, N, BAD, ctypes.byref(sid), ctypes.byref(rb)) == SHAPE
        assert L.afx_stream_add_shape(st, ctx, 0, N, HIDDEN, ctypes.byref(sid), ctypes.byref(rb)) == OK
        assert rb.value == L.afx_presentation_num_fields(N, HIDDEN) * 32
        assert L.afx_stream_add_shape(None, ctx, 0, N, KINDS, ctypes.byref(sid), ctypes.byref(rb)) == ARG
        assert L.afx_stream_add_shape(st, None, 0, N, KINDS, ctypes.byref(sid), ctypes.byref(rb)) == ARG
        assert L.afx_stream_add_shape(st, ctx, 0, N, None, ctypes.byref(sid), ctypes.byref(rb)) == ARG
        assert L.afx_stream_add_shape(st, ctx, 0, N, KINDS, None, ctypes.byref(rb)) == ARG
    finally:
        L.afx_stream_destroy(st)


@pytest.mark.parametrize("name", ALL)
def test_invalid_kinds(L, ctx, name):
    call = Calls(L)
    assert call(name, ctx, kinds=BAD) == SHAPE
    assert call(name, ctx, kinds=BAD, nf_delta=1) == SHAPE          # the shape is compiled before the field count is compared
    assert call(name, ctx, kinds=bytes([0, 0, 2])) == SHAPE         # an attribute count different from the issuer's
    if name in ISSUANCE_VERIFY + ISSUANCE_SUBMIT + ISSUE:
        assert call(name, ctx, kinds=HIDDEN) == SHAPE               # requests and issuances have no hidden kinds


@pytest.mark.parametrize("name", SOA)
def test_field_count_mismatch(L, ctx, name):
    call = Calls(L)
    kinds = kinds_for(name)
    assert call(name, ctx, kinds=kinds) == OK
    assert call(name, ctx, kinds=kinds, nf_delta=1) == ARG
    assert call(name, ctx, kinds=kinds, nf_delta=-1) == ARG
    if name in ("issue", "show", "show_linked"):
        assert call(name, ctx, kinds=kinds, out_nf_delta=1) == ARG  # the output descriptor is checked too


def test_calls_while_two_submissions_are_outstanding(L, issuer_material):
    c = make_ctx(L, issuer_material, True)
    call = Calls(L)
    try:
        t = [ctypes.c_uint64(), ctypes.c_uint64()]
        assert call.call("verify_presentations_submit", c, KINDS, 0, False, 0, 0, t[0]) == OK
        assert call.call("verify_presentations_wire_submit", c, KINDS, 0, False, 0, 0, t[1]) == OK
        for name in SYNC:
            assert call(name, c, kinds=kinds_for(name)) == ARG, name
            assert call(name, c, kinds=BAD) == ARG, name            # refused before the shape is compiled
        for name in PRESENTATION_SUBMIT + ISSUANCE_SUBMIT:
            assert call(name, c) == ARG, name                       # a third submission
            assert call(name, c, kinds=BAD) == SHAPE, name          # ... whose shape is compiled before its slot is checked
        sid, rb, st = ctypes.c_int(), ctypes.c_size_t(), ctypes.c_void_p()
        assert L.afx_stream_create(ctypes.byref(st)) == OK
        assert L.afx_stream_add_shape(st, c, 0, N, KINDS, ctypes.byref(sid), ctypes.byref(rb)) == OK   # registering compiles only
        L.afx_stream_destroy(st)
        assert L.afx_wait(c, t[1].value + 1) == ARG
        assert L.afx_wait(c, t[1].value) == OK
        assert L.afx_wait(c, t[1].value) == ARG                     # waited already
        assert call("verify_presentations", c) == ARG               # one is still outstanding
        assert L.afx_wait(c, t[0].value) == OK
        for name in SYNC:
            assert call(name, c, kinds=kinds_for(name)) == OK, name
    finally:
        L.afx_ctx_destroy(c)
