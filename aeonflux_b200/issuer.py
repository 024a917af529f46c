"""Host-side mirror of the reference's interface for the hot path (/root/reference/src/issuer.rs), batch form.

    reference (Rust)                                      here
    ----------------------------------------------------  ----------------------------------------------------
    Issuer { system_parameters, issuer_parameters,        Issuer(system_parameters, issuer_parameters, amacs_key)
             amacs_key }                 issuer.rs:61-65    -- the same to_bytes() encodings (parameters.rs:155-184,
                                                               C_W||I, amacs.rs:110-125)
    Issuer::verify(&self, &presentation) issuer.rs:141-147  Issuer.verify_batch(PresentationBatch) -> verdicts
    CredentialIssuance::verify(self, &sp, &ip)              Issuer.verify_issuance_batch(IssuanceBatch) -> verdicts
                                         issuer.rs:48-57      (amacs_key=None suffices: it is the user-side check)
    Issuer::issue(&self, request, &mut rng)                 Issuer.issue_batch(RequestBatch) -> (IssuanceBatch, status)
                                         issuer.rs:111-124    (the rng output is part of the request batch)
    Result<(), CredentialError::VerificationFailure>        verdict 0 / 1 per item (errors.rs:152-156)

The reference defines no wire format for presentations or issuances (presentation.rs:117 "XXX"); the flat
struct-of-arrays layout is documented in include/aeonflux_b200.h.
"""
import ctypes

import numpy as np

from . import _binding as B

KIND_PUBLIC_SCALAR, KIND_SECRET_SCALAR, KIND_PUBLIC_POINT, KIND_SECRET_POINT = 0, 1, 2, 3
AFX_ERR_SHAPE = -5


class PresentationBatch:
    """kinds: bytes of AFX_KIND_*, one per attribute; fields: uint8 array [n_fields][count][32]."""

    def __init__(self, kinds, fields):
        self.kinds = bytes(kinds)
        fields = np.asarray(fields, dtype=np.uint8)
        if fields.ndim != 3 or fields.shape[2] != 32:
            raise ValueError("fields must be [n_fields][count][32] bytes")
        # each field must be one contiguous [count][32] run (that is all the C ABI needs); an item slice of a batch
        # (fields[:, lo:hi]) already is, so sharding a batch copies nothing
        if not all(fields[f].flags.c_contiguous for f in range(fields.shape[0])):
            fields = np.ascontiguousarray(fields)
        self.fields = fields

    @property
    def count(self):
        return self.fields.shape[1]

    @staticmethod
    def from_items(kinds, items, host_array=None):
        """items: uint8 [count][n_fields][32] (item-major, as a list of per-presentation word lists).  host_array: an allocator
        such as Issuer.host_array -- the struct-of-arrays copy is then built in page-locked memory (afx_host_alloc), from which
        the library's host-to-device copies run asynchronously at the full bus rate."""
        items = np.asarray(items, dtype=np.uint8)
        if host_array is None:
            return PresentationBatch(kinds, np.ascontiguousarray(items.transpose(1, 0, 2)))
        fields = host_array((items.shape[1], items.shape[0], 32))
        fields[:] = items.transpose(1, 0, 2)
        return PresentationBatch(kinds, fields)


def compact_to_batchable(kinds, fields, commitments):
    """Re-encode compact presentations as BatchableProof presentations: fields [n_fields][count][32] in the compact layout and
    the blinding commitments their proofs recompute [n_commitments][count][32] (e.g. the `commitments` of verify_batch(debug=True))
    -> fields in the batchable layout (every challenge word replaced by that proof's commitments, include/aeonflux_b200.h)."""
    kinds = list(bytes(kinds))
    n = len(kinds)
    h_s = sum(k == KIND_SECRET_SCALAR for k in kinds)
    r = sum(k in (KIND_PUBLIC_SCALAR, KIND_PUBLIC_POINT) for k in kinds)
    nsp = sum(k != KIND_SECRET_POINT for k in kinds)
    nc = 2 + sum(kinds[i] != KIND_SECRET_POINT for i in range(nsp))
    head = 1 + 3 + h_s + 3 + n + r
    rows = [commitments[j] for j in range(nc)] + [fields[w] for w in range(1, head)]
    pos, cpos = head, nc
    for k in kinds:
        if k == KIND_SECRET_POINT:
            rows += [commitments[cpos + j] for j in range(5)] + [fields[w] for w in range(pos + 1, pos + 14)]
            pos += 14
            cpos += 5
    return np.ascontiguousarray(np.stack(rows))


IssuanceBatch = PresentationBatch   # same container; kinds are 0 (scalar attribute) / 2 (point attribute)


class RequestBatch(PresentationBatch):
    """A batch of CredentialRequests (user.rs:137-139) plus the rng output Issuer::issue would draw for each.

    fields [3n + 14][count][32]: attribute[n], then the low/high 32 bytes of the 64 rng bytes behind t, U and each of the
    n + 5 proof blindings (include/aeonflux_b200.h)."""

    @staticmethod
    def from_request(kinds, attributes, randomness):
        """attributes: uint8 [count][n][32]; randomness: uint8 [count][n + 7][64] (t, U, blinding[n + 5])."""
        attributes = np.asarray(attributes, dtype=np.uint8)
        randomness = np.asarray(randomness, dtype=np.uint8)
        count, n = attributes.shape[0], len(kinds)
        if attributes.shape != (count, n, 32) or randomness.shape != (count, n + 7, 64):
            raise ValueError("attributes must be [count][n][32] and randomness [count][n+7][64]")
        items = np.concatenate([attributes, randomness.reshape(count, 2 * (n + 7), 32)], axis=1)
        return RequestBatch(kinds, np.ascontiguousarray(items.transpose(1, 0, 2)))


def bind_thread_to_device(device: int, _binding=None) -> bool:
    """Pin the calling thread (and with it the page-locked staging it allocates next) to the CPUs local to `device`
    (afx_bind_thread_to_device).  For a one-process-per-GPU program: call it first.  Returns False if the topology is unreadable."""
    if _binding is None:
        from ._lib import load
        _binding = load()
    return _binding.L.afx_bind_thread_to_device(int(device)) == 0


class Issuer:
    """An anonymous credential issuer/verifier bound to one B200 (issuer.rs:61-65)."""

    def __init__(self, system_parameters: bytes, issuer_parameters: bytes, amacs_key: bytes = None, device: int = 0,
                 max_batch: int = 65536, _binding=None):
        if _binding is None:
            from ._lib import load
            _binding = load()
        self._b = _binding
        self.system_parameters = bytes(system_parameters)
        self.issuer_parameters = bytes(issuer_parameters)
        self.number_of_attributes = int.from_bytes(self.system_parameters[:4], "little")
        self.max_batch = max_batch
        if len(self.issuer_parameters) != 64:
            raise ValueError("issuer_parameters must be C_W || I (64 bytes)")
        h = ctypes.c_void_p()
        sp = ctypes.create_string_buffer(self.system_parameters, len(self.system_parameters))
        ip = ctypes.create_string_buffer(self.issuer_parameters, 64)
        sk = ctypes.create_string_buffer(bytes(amacs_key), len(amacs_key)) if amacs_key is not None else None
        rc = self._b.L.afx_ctx_create(ctypes.addressof(sp), len(self.system_parameters), ctypes.addressof(ip),
                                      ctypes.addressof(sk) if sk is not None else None, len(amacs_key) if amacs_key is not None else 0,
                                      device, max_batch, ctypes.byref(h))
        if sk is not None:
            ctypes.memset(sk, 0, len(amacs_key))
        self._b.check(rc)
        self._h = h

    @classmethod
    def from_bytes(cls, blob: bytes, **kw):
        """Issuer::from_bytes (issuer.rs:152-159): sysparams || C_W || I || secret key."""
        from .wire import issuer_from_bytes
        sp, ip, sk = issuer_from_bytes(blob)
        return cls(sp, ip, sk, **kw)

    def close(self):
        if getattr(self, "_h", None):
            self._b.L.afx_ctx_destroy(self._h)
            self._h = None

    __del__ = close

    # -- shape helpers
    def host_array(self, shape):
        """uint8 ndarray in page-locked host memory (afx_host_alloc / afx_host_free)."""
        return self._b.host_array(shape)

    def num_fields(self, kinds):
        return self._b.L.afx_presentation_num_fields(len(kinds), bytes(kinds))

    def num_commitments(self, kinds):
        return self._b.L.afx_presentation_num_commitments(len(kinds), bytes(kinds))

    def num_proofs(self, kinds):
        return self._b.L.afx_presentation_num_proofs(len(kinds), bytes(kinds))

    @property
    def launch_count(self):
        return int(self._b.L.afx_launch_count(self._h))

    STAGES = ("scalar_check", "points", "amac", "msm", "transcript", "verdict")

    def set_stage_timing(self, on: bool):
        self._b.L.afx_set_stage_timing(self._h, 1 if on else 0)

    def stage_times_ms(self):
        """Device time of each stage of the most recent run (CUDA events on the launching stream)."""
        ms = (ctypes.c_float * 6)()
        self._b.check(self._b.L.afx_get_stage_times(self._h, ms, 6))
        return dict(zip(self.STAGES, [float(x) for x in ms]))

    def rlc_bucket_time(self):
        """(ms, points summed, windows) of k_rlc_buckets in the most recent verify_batchable_rlc pass (stage timing must be on)."""
        ms, n, w = ctypes.c_float(0), ctypes.c_uint64(0), ctypes.c_uint32(0)
        self._b.check(self._b.L.afx_get_rlc_bucket_time(self._h, ctypes.byref(ms), ctypes.byref(n), ctypes.byref(w)))
        return float(ms.value), int(n.value), int(w.value)

    def submit_wire(self, kinds, items, issuance=False):
        """Asynchronous verify of one pass of item-major wire bytes [count][n_fields][32] (count <= max_batch) -> pending result."""
        items = np.ascontiguousarray(items, dtype=np.uint8)
        kinds = bytes(kinds)
        verdicts = np.zeros(items.shape[0], np.uint8)
        ticket = ctypes.c_uint64(0)
        fn = self._b.L.afx_verify_issuances_wire_submit if issuance else self._b.L.afx_verify_presentations_wire_submit
        self._b.check(fn(self._h, len(kinds), kinds, items.shape[0], items.ctypes.data, verdicts.ctypes.data, ctypes.byref(ticket)))
        issuer = self

        class Pending:
            def wait(self_inner):
                issuer._b.check(issuer._b.L.afx_wait(issuer._h, ticket.value))
                return verdicts
            _keep = (items,)
        return Pending()

    def _run(self, fn, batch, ncommit, nproofs, debug):
        count = batch.count
        ptrs, keep = B._as_fields(batch.fields)
        cb = B.afx_presentation_batch(len(batch.kinds), batch.kinds, count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        verdicts = np.zeros(count, np.uint8)
        dbg = None
        out = None
        if debug:
            out = {"Z": np.zeros((count, 32), np.uint8), "commitments": np.zeros((ncommit, count, 32), np.uint8),
                   "challenges": np.zeros((nproofs, count, 32), np.uint8), "status": np.zeros(count, np.uint32)}
            dbg = B.afx_debug_dump(out["Z"].ctypes.data, out["commitments"].ctypes.data, out["challenges"].ctypes.data, out["status"].ctypes.data)
        rc = fn(self._h, ctypes.byref(cb), verdicts.ctypes.data, ctypes.byref(dbg) if dbg is not None else None)
        self._b.check(rc)
        return (verdicts, out) if debug else verdicts

    def verify_batch(self, batch: PresentationBatch, debug=False, linked=False):
        """Batch Issuer::verify (issuer.rs:141-147): verdict 0 = Ok(()), 1 = Err(VerificationFailure).  linked: the opt-in statement
        that ties each proof of encryption to the credential proof (include/aeonflux_b200.h, "Linked presentations")."""
        if linked:
            ncm = self._b.L.afx_presentation_linked_num_commitments(len(batch.kinds), batch.kinds)
            return self._run(self._b.L.afx_verify_presentations_linked, batch, ncm, self.num_proofs(batch.kinds), debug)
        return self._run(self._b.L.afx_verify_presentations, batch, self.num_commitments(batch.kinds), self.num_proofs(batch.kinds), debug)

    def submit(self, batch: PresentationBatch, issuance=False):
        """Asynchronous Issuer::verify (or CredentialIssuance::verify) of one pass (count <= max_batch): returns a pending result;
        call .wait() for the verdicts.  Up to two submissions may be outstanding (copy of one under the kernels of the other)."""
        ptrs, keep = B._as_fields(batch.fields)
        cb = B.afx_presentation_batch(len(batch.kinds), batch.kinds, batch.count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        verdicts = np.zeros(batch.count, np.uint8)
        ticket = ctypes.c_uint64(0)
        fn = self._b.L.afx_verify_issuances_submit if issuance else self._b.L.afx_verify_presentations_submit
        self._b.check(fn(self._h, ctypes.byref(cb), verdicts.ctypes.data, ctypes.byref(ticket)))
        issuer = self

        class Pending:
            def wait(self_inner):
                issuer._b.check(issuer._b.L.afx_wait(issuer._h, ticket.value))
                return verdicts
            _keep = (keep, ptrs, cb)
        return Pending()

    def verify_batchable(self, batch: PresentationBatch, debug=False):
        """Batch Issuer::verify for presentations whose proofs are BatchableProofs (commitments instead of challenges, see
        include/aeonflux_b200.h): every constraint of every item is checked exactly."""
        return self._run(self._b.L.afx_verify_presentations_batchable, batch, self.num_commitments(batch.kinds), self.num_proofs(batch.kinds), debug)

    def verify_batchable_rlc(self, batch: PresentationBatch, seed: bytes, issuance=False):
        """BatchableProof presentations (or issuances) checked as one random linear combination per chunk (Pippenger over the whole
        chunk); a chunk that does not vanish is bisected down to 1,024-item leaves, which are re-verified exactly.  seed: 32 bytes
        (the library mixes in a nonce of its own).  Returns (verdicts, number of chunks that needed exact work)."""
        if len(seed) != 32:
            raise ValueError("seed must be 32 bytes")
        ptrs, keep = B._as_fields(batch.fields)
        cb = B.afx_presentation_batch(len(batch.kinds), batch.kinds, batch.count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        verdicts = np.zeros(batch.count, np.uint8)
        sd = ctypes.create_string_buffer(bytes(seed), 32)
        fell_back = ctypes.c_uint32(0)
        fn = self._b.L.afx_verify_issuances_batchable_rlc if issuance else self._b.L.afx_verify_presentations_batchable_rlc
        self._b.check(fn(self._h, ctypes.byref(cb), ctypes.addressof(sd), verdicts.ctypes.data, ctypes.byref(fell_back)))
        return verdicts, int(fell_back.value)

    def verify_issuance_batchable(self, batch: IssuanceBatch, debug=False):
        """Batch CredentialIssuance::verify for issuances whose proof is a BatchableProof: fields attribute[n], t, U, V,
        commitments[3], responses[n + 5]; every constraint checked exactly."""
        return self._run(self._b.L.afx_verify_issuances_batchable, batch, 3, 1, debug)

    def rlc_stats(self):
        """(combination passes run, items re-verified exactly) by the *_rlc calls on this context so far."""
        a, b = ctypes.c_uint64(0), ctypes.c_uint64(0)
        self._b.check(self._b.L.afx_get_rlc_stats(self._h, ctypes.byref(a), ctypes.byref(b)))
        return int(a.value), int(b.value)

    def verify_wire(self, kinds, items, issuance=False, linked=False):
        """Batch Issuer::verify (or CredentialIssuance::verify) over item-major wire bytes: items = uint8 [count][n_fields][32],
        the concatenation of each item's words.  One H2D copy; no per-field scatter on the host."""
        items = np.ascontiguousarray(items, dtype=np.uint8)
        nf = (2 * len(kinds) + 9) if issuance else self.num_fields(kinds)
        if items.ndim != 3 or items.shape[1:] != (nf, 32):
            raise ValueError("items must be [count][%d][32] bytes for this shape" % nf)
        verdicts = np.zeros(items.shape[0], np.uint8)
        fn = self._b.L.afx_verify_issuances_wire if issuance else self._b.L.afx_verify_presentations_linked_wire if linked else self._b.L.afx_verify_presentations_wire
        self._b.check(fn(self._h, len(kinds), bytes(kinds), items.shape[0], items.ctypes.data, verdicts.ctypes.data))
        return verdicts

    def verify_mixed_wire(self, shape_kinds, records, shape_ids, issuance=False):
        """Batch Issuer::verify (or CredentialIssuance::verify) over wire records of several shapes of this issuer in one call:
        shape_kinds = list of kind vectors, records = uint8 array of the records concatenated in order (record i is an item of
        shape shape_ids[i] in the verify_wire layout), shape_ids = uint8 [count].  The records are bucketed by shape on the
        device; verdicts come back in record order."""
        fn = self._b.L.afx_verify_issuances_mixed_wire if issuance else self._b.L.afx_verify_presentations_mixed_wire
        return B.mixed_wire(self._b, fn, self._h, shape_kinds, records, shape_ids, "issuance" if issuance else "presentation")

    def issue_mixed_wire(self, shape_kinds, requests, shape_ids, out=None):
        """Batch Issuer::issue over CredentialRequests of several request kinds in one call: shape_kinds = list of request kind
        vectors, requests = uint8 array of the requests concatenated in order (record i is a request of kinds shape_kinds[shape_ids[i]]
        in the issue_wire layout, 3n + 14 words whatever the kinds), shape_ids = uint8 [count].  Returns (issuances uint8
        [count][2n + 9][32] in record order, status) -- with the same shape_kinds and shape_ids, what verify_mixed_wire(issuance=True)
        takes.  out: optional preallocated (e.g. page-locked) contiguous uint8 array of the result's size."""
        out, status = B.mixed_wire(self._b, self._b.L.afx_issue_mixed_wire, self._h, shape_kinds, requests, shape_ids, "request", "issuance", out)
        n = len(bytes(shape_kinds[0])) if len(shape_kinds) else 0
        return out.reshape(len(status), 2 * n + 9, 32), status

    def show_mixed_wire(self, shape_kinds, inputs, shape_ids, out=None):
        """Batch AnonymousCredential::show over inputs of several disclosure patterns in one call: inputs = uint8 array of the show
        inputs concatenated in order (record i in the show_wire layout of shape_kinds[shape_ids[i]]).  Returns (the presentations
        concatenated in record order as one uint8 blob -- with the same shape_kinds and shape_ids, what verify_mixed_wire takes --,
        status); presentation_offsets gives where each record starts.  out: as for issue_mixed_wire."""
        return B.mixed_wire(self._b, self._b.L.afx_show_mixed_wire, self._h, shape_kinds, inputs, shape_ids, "show", "presentation", out)

    def presentation_offsets(self, shape_kinds, shape_ids):
        """Byte offsets [count + 1] of the presentations in a show_mixed_wire blob: record i is blob[offsets[i]:offsets[i + 1]]."""
        return B.record_offsets(B.mixed_record_bytes(self._b, shape_kinds, "presentation"), shape_ids)

    def verify_issuance_batch(self, batch: IssuanceBatch, debug=False):
        """Batch CredentialIssuance::verify (issuer.rs:48-57)."""
        return self._run(self._b.L.afx_verify_issuances, batch, 3, 1, debug)

    def issue_batch(self, batch: RequestBatch, debug=False, out=None, batchable=False):
        """Batch Issuer::issue (issuer.rs:111-124).  Returns (IssuanceBatch, status): the issuances in the layout
        verify_issuance_batch takes (attribute[n], t, U, V, challenge, responses[n+5]); status 0 = Ok, 1 = malformed request.
        out: optional preallocated uint8 [2n + 9][count][32] array for the result, e.g. from Issuer.host_array -- in page-locked
        memory the device-to-host copy of (n + 9) x 32 bytes per item runs at the bus rate instead of through the driver's staging.
        batchable: the proofs as zkp's prove_batchable returns them, the challenge replaced by the commitments C_W, I, V -- the
        [2n + 11][count][32] layout verify_issuance_batchable and verify_batchable_rlc(issuance=True) take."""
        n, count = len(batch.kinds), batch.count
        if batch.fields.shape[0] != 3 * n + 14:
            raise ValueError("a request batch has 3n + 14 fields")
        ptrs, keep = B._as_fields(batch.fields)
        cb = B.afx_presentation_batch(n, batch.kinds, count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        nw = 2 * n + (11 if batchable else 9)
        if out is None:
            out = np.zeros((nw, count, 32), np.uint8)
        elif out.shape != (nw, count, 32) or out.dtype != np.uint8 or not out.flags.c_contiguous:
            raise ValueError("out must be a contiguous uint8 [%s][count][32] array" % ("2n + 11" if batchable else "2n + 9"))
        out[:n] = batch.fields[:n]
        optrs, okeep = B._as_fields(out[n:])
        ob = B.afx_issuance_out(ctypes.cast(optrs, ctypes.POINTER(ctypes.c_void_p)), len(okeep))
        status = np.zeros(count, np.uint8)
        dbg, dump = None, None
        if debug:
            dump = {"commitments": np.zeros((3, count, 32), np.uint8), "status": np.zeros(count, np.uint32)}
            dbg = B.afx_debug_dump(None, dump["commitments"].ctypes.data, None, dump["status"].ctypes.data)
        fn = self._b.L.afx_issue_batchable if batchable else self._b.L.afx_issue
        self._b.check(fn(self._h, ctypes.byref(cb), ctypes.byref(ob), status.ctypes.data, ctypes.byref(dbg) if dbg is not None else None))
        for i, a in enumerate(okeep):            # _as_fields may have copied non-contiguous rows
            if a is not out[n + i] and not np.shares_memory(a, out):
                out[n + i] = a
        res = IssuanceBatch(batch.kinds, out)
        return (res, status, dump) if debug else (res, status)

    def show_batch(self, kinds, fields, debug=False, linked=False, batchable=False):
        """Batch AnonymousCredential::show (credential.rs:37-46).  kinds: the presentation's attribute kinds; fields: uint8
        [afx_show_num_fields][count][32] in the order documented in include/aeonflux_b200.h (credential, attributes, keypair,
        rng bytes).  Returns (PresentationBatch, status) -- the batch can be passed to verify_batch as is.  batchable: the proofs
        as zkp's prove_batchable returns them (every challenge replaced by that proof's commitments), the layout verify_batchable
        and verify_batchable_rlc take.  There is no linked BatchableProof statement: linked and batchable together raise
        AFX_ERR_SHAPE."""
        kinds = bytes(kinds)
        if linked and batchable:
            self._b.check(AFX_ERR_SHAPE)
        fields = np.ascontiguousarray(fields, dtype=np.uint8)
        nf = self._b.L.afx_show_num_fields(len(kinds), kinds)
        if fields.ndim != 3 or fields.shape[0] != nf or fields.shape[2] != 32:
            raise ValueError("show input must be [%d][count][32] bytes for this shape" % nf)
        count = fields.shape[1]
        ptrs, keep = B._as_fields(fields)
        cb = B.afx_presentation_batch(len(kinds), kinds, count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        nw = self._b.L.afx_batchable_num_fields(len(kinds), kinds) if batchable else self.num_fields(kinds)
        out = np.zeros((nw, count, 32), np.uint8)
        optrs, okeep = B._as_fields(out)
        ob = B.afx_issuance_out(ctypes.cast(optrs, ctypes.POINTER(ctypes.c_void_p)), len(okeep))
        status = np.zeros(count, np.uint8)
        dbg, dump = None, None
        if debug:
            ncm = self._b.L.afx_presentation_linked_num_commitments(len(kinds), kinds) if linked else self.num_commitments(kinds)
            dump = {"commitments": np.zeros((ncm, count, 32), np.uint8), "status": np.zeros(count, np.uint32)}
            dbg = B.afx_debug_dump(None, dump["commitments"].ctypes.data, None, dump["status"].ctypes.data)
        fn = self._b.L.afx_show_linked if linked else self._b.L.afx_show_batchable if batchable else self._b.L.afx_show
        self._b.check(fn(self._h, ctypes.byref(cb), ctypes.byref(ob), status.ctypes.data, ctypes.byref(dbg) if dbg is not None else None))
        res = PresentationBatch(kinds, out)
        return (res, status, dump) if debug else (res, status)

    def issue_wire(self, kinds, requests, out=None):
        """Batch Issuer::issue over item-major requests uint8 [count][3n + 14][32] -> (issuances uint8 [count][2n + 9][32] in the
        layout verify_wire(issuance=True) takes, status).  out: optional preallocated (e.g. page-locked) result array."""
        kinds = bytes(kinds)
        n = len(kinds)
        requests = np.ascontiguousarray(requests, dtype=np.uint8)
        if requests.ndim != 3 or requests.shape[1:] != (3 * n + 14, 32):
            raise ValueError("requests must be [count][3n + 14][32] bytes")
        count = requests.shape[0]
        if out is None:
            out = np.zeros((count, 2 * n + 9, 32), np.uint8)
        elif out.shape != (count, 2 * n + 9, 32) or out.dtype != np.uint8 or not out.flags.c_contiguous:
            raise ValueError("out must be a contiguous uint8 [count][2n + 9][32] array")
        status = np.zeros(count, np.uint8)
        self._b.check(self._b.L.afx_issue_wire(self._h, n, kinds, count, requests.ctypes.data, out.ctypes.data, status.ctypes.data))
        return out, status

    def show_wire(self, kinds, inputs, out=None, linked=False):
        """Batch AnonymousCredential::show over item-major inputs uint8 [count][afx_show_num_fields][32] -> (presentations uint8
        [count][n_fields][32] in the layout verify_wire takes, status)."""
        kinds = bytes(kinds)
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        nf = self._b.L.afx_show_num_fields(len(kinds), kinds)
        if inputs.ndim != 3 or inputs.shape[1:] != (nf, 32):
            raise ValueError("inputs must be [count][%d][32] bytes for this shape" % nf)
        count = inputs.shape[0]
        if out is None:
            out = np.zeros((count, self.num_fields(kinds), 32), np.uint8)
        status = np.zeros(count, np.uint8)
        fn = self._b.L.afx_show_linked_wire if linked else self._b.L.afx_show_wire
        self._b.check(fn(self._h, len(kinds), kinds, count, inputs.ctypes.data, out.ctypes.data, status.ctypes.data))
        return out, status

    def show_batch_device(self, kinds, count, fields_dev_ptr, out_dev_ptr, status_dev_ptr, stream=0, batchable=False):
        """Enqueue show_batch on device memory: out [n_out][count][32] with n_out = num_fields(kinds), or with batchable=True
        afx_batchable_num_fields(kinds); count <= max_batch, no synchronisation."""
        fn = self._b.L.afx_show_batchable_device if batchable else self._b.L.afx_show_device
        self._b.check(fn(self._h, len(kinds), bytes(kinds), count, fields_dev_ptr, out_dev_ptr, status_dev_ptr, stream))

    def issue_batch_device(self, kinds, count, fields_dev_ptr, out_dev_ptr, status_dev_ptr, stream=0, batchable=False):
        """Enqueue issue_batch on device memory: out [n + 9][count][32], or with batchable=True [n + 11][count][32] (t, U, V, the
        commitments C_W, I, V, responses[n + 5]); count <= max_batch, no synchronisation."""
        fn = self._b.L.afx_issue_batchable_device if batchable else self._b.L.afx_issue_device
        self._b.check(fn(self._h, len(kinds), bytes(kinds), count, fields_dev_ptr, out_dev_ptr, status_dev_ptr, stream))

    def verify_issuance_batch_device(self, kinds, count, fields_dev_ptr, verdicts_dev_ptr, stream=0):
        self._b.check(self._b.L.afx_verify_issuances_device(self._h, len(kinds), bytes(kinds), count, fields_dev_ptr, verdicts_dev_ptr, stream))

    # -- symmetric encryption of attributes (encoding.rs, symmetric.rs); the calls need no issuer secret
    @staticmethod
    def _array(name, a, shape):
        if not isinstance(a, np.ndarray) or a.dtype != np.uint8 or a.shape != shape or not a.flags.c_contiguous:
            raise ValueError("%s must be a contiguous uint8 %s array" % (name, "[" + "][".join(str(d) for d in shape) + "]"))
        return a

    @staticmethod
    def _keypair(keypair):
        """keypair: a || a0 || a1 (96 bytes), or the 128-byte keypair show takes (a, a0, a1, pk)."""
        kp = bytes(keypair)
        if len(kp) not in (96, 128):
            raise ValueError("keypair must be a || a0 || a1 (96 bytes) or a || a0 || a1 || pk (128 bytes)")
        return ctypes.create_string_buffer(kp[:96], 96)

    def encode_plaintexts(self, data, out=None):
        """Plaintext::from(&[u8; 30]) for every row of data (uint8 [count][30]) -> (plaintexts uint8 [count][3][32]: M1, M2, m3 --
        the words of a hidden plaintext attribute in show's input, status).  status 1 (all-zero words): no candidate encoding of
        the 8,192 decodes (the reference panics there)."""
        data = np.asarray(data, dtype=np.uint8)
        if data.ndim != 2 or data.shape[1] != 30:
            raise ValueError("data must be [count][30] bytes")
        data = np.ascontiguousarray(data)
        count = data.shape[0]
        out = np.zeros((count, 3, 32), np.uint8) if out is None else self._array("out", out, (count, 3, 32))
        status = np.zeros(count, np.uint8)
        self._b.check(self._b.L.afx_encode_plaintexts(self._h, count, data.ctypes.data, out.ctypes.data, status.ctypes.data))
        return out, status

    def encrypt(self, keypair, plaintexts, out=None):
        """Keypair::encrypt (symmetric.rs:252-261) of every Plaintext (uint8 [count][3][32]: M1, M2, m3) -> (ciphertexts uint8
        [count][2][32]: E1, E2, status).  status 1 (all-zero words): M1 or M2 does not decode, or m3 is not canonical."""
        kp = self._keypair(keypair)
        plaintexts = np.asarray(plaintexts, dtype=np.uint8)
        if plaintexts.ndim != 3 or plaintexts.shape[1:] != (3, 32):
            raise ValueError("plaintexts must be [count][3][32] bytes")
        plaintexts = np.ascontiguousarray(plaintexts)
        count = plaintexts.shape[0]
        out = np.zeros((count, 2, 32), np.uint8) if out is None else self._array("out", out, (count, 2, 32))
        status = np.zeros(count, np.uint8)
        try:
            self._b.check(self._b.L.afx_encrypt(self._h, ctypes.addressof(kp), count, plaintexts.ctypes.data, out.ctypes.data, status.ctypes.data))
        finally:
            ctypes.memset(kp, 0, 96)
        return out, status

    def decrypt(self, keypair, ciphertexts, plaintexts=False, out=None):
        """Keypair::decrypt (symmetric.rs:273-289) of every ciphertext (uint8 [count][2][32]: E1, E2) -> (data uint8 [count][30],
        status), or (data, plaintexts uint8 [count][3][32], status) with plaintexts=True.  status 1 (all-zero output):
        CredentialError::UndecryptableAttribute, or E1 / E2 does not decode."""
        kp = self._keypair(keypair)
        ciphertexts = np.asarray(ciphertexts, dtype=np.uint8)
        if ciphertexts.ndim != 3 or ciphertexts.shape[1:] != (2, 32):
            raise ValueError("ciphertexts must be [count][2][32] bytes")
        ciphertexts = np.ascontiguousarray(ciphertexts)
        count = ciphertexts.shape[0]
        data = np.zeros((count, 30), np.uint8) if out is None else self._array("out", out, (count, 30))
        pts = np.zeros((count, 3, 32), np.uint8) if plaintexts else None
        status = np.zeros(count, np.uint8)
        try:
            self._b.check(self._b.L.afx_decrypt(self._h, ctypes.addressof(kp), count, ciphertexts.ctypes.data, data.ctypes.data,
                                                pts.ctypes.data if plaintexts else None, status.ctypes.data))
        finally:
            ctypes.memset(kp, 0, 96)
        return (data, pts, status) if plaintexts else (data, status)

    def encode_plaintexts_device(self, count, data_dev_ptr, plaintexts_dev_ptr, status_dev_ptr, stream=0):
        """Enqueue encode_plaintexts on device memory: data [count][30] -> plaintexts [3][count][32] (the rows show_batch_device takes
        for a hidden plaintext), status [count]; count <= max_batch, no synchronisation."""
        self._b.check(self._b.L.afx_encode_plaintexts_device(self._h, count, data_dev_ptr, plaintexts_dev_ptr, status_dev_ptr, stream))

    def encrypt_device(self, keypair, count, plaintexts_dev_ptr, ciphertexts_dev_ptr, status_dev_ptr, stream=0):
        """Enqueue encrypt on device memory: plaintexts [3][count][32] -> ciphertexts [2][count][32], status [count]."""
        kp = self._keypair(keypair)
        try:
            self._b.check(self._b.L.afx_encrypt_device(self._h, ctypes.addressof(kp), count, plaintexts_dev_ptr, ciphertexts_dev_ptr,
                                                       status_dev_ptr, stream))
        finally:
            ctypes.memset(kp, 0, 96)

    def decrypt_device(self, keypair, count, ciphertexts_dev_ptr, data_dev_ptr, status_dev_ptr, plaintexts_dev_ptr=None, stream=0):
        """Enqueue decrypt on device memory: ciphertexts [2][count][32] -> data [count][30], optional plaintexts [3][count][32],
        status [count]."""
        kp = self._keypair(keypair)
        try:
            self._b.check(self._b.L.afx_decrypt_device(self._h, ctypes.addressof(kp), count, ciphertexts_dev_ptr, data_dev_ptr,
                                                       plaintexts_dev_ptr, status_dev_ptr, stream))
        finally:
            ctypes.memset(kp, 0, 96)

    def derive_keypairs(self, master_secrets, out=None):
        """Keypair::derive (symmetric.rs:197-215) of every 64-byte master secret (uint8 [count][64]) under this context's system
        parameters -> keypairs uint8 [count][128]: a || a0 || a1 || pk, the keypair show takes (its first 96 bytes are what
        encrypt and decrypt take).  Keypair::generate is this applied to 64 rng bytes."""
        ms = np.asarray(master_secrets, dtype=np.uint8)
        if ms.ndim != 2 or ms.shape[1] != 64:
            raise ValueError("master_secrets must be [count][64] bytes")
        ms = np.ascontiguousarray(ms)
        count = ms.shape[0]
        out = np.zeros((count, 128), np.uint8) if out is None else self._array("out", out, (count, 128))
        self._b.check(self._b.L.afx_derive_keypairs(self._h, count, ms.ctypes.data, out.ctypes.data))
        return out

    def derive_keypairs_device(self, count, master_secrets_dev_ptr, keypairs_dev_ptr, stream=0):
        """Enqueue derive_keypairs on device memory: master secrets [count][64] -> keypairs [4][count][32] (the a, a0, a1, pk rows
        show_batch_device takes); count <= max_batch, no synchronisation."""
        self._b.check(self._b.L.afx_derive_keypairs_device(self._h, count, master_secrets_dev_ptr, keypairs_dev_ptr, stream))

    PRIMITIVES = {"decompress_compress": (0, 32), "from_uniform": (1, 64), "scalarmult": (2, 64), "wide_reduce": (3, 64), "sc_muladd": (4, 96),
                  "fe_mul": (5, 64), "fe_sq": (6, 64), "fe_add": (7, 64), "fe_sub": (8, 64), "fe_chain": (9, 64), "ladder_scalarmult": (10, 64), "recode4096": (11, 32),
                  "recode65536": (12, 32)}

    def selftest_primitive(self, name, inputs):
        """Run one field/group/scalar primitive of the engine over raw inputs (uint8 [count][in_bytes]) -> (out [count][32], ok [count])."""
        op, width = self.PRIMITIVES[name]
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8).reshape(-1, width)
        out = np.zeros((inputs.shape[0], 32), np.uint8)
        ok = np.zeros(inputs.shape[0], np.uint8)
        self._b.check(self._b.L.afx_selftest_primitive(self._h, op, inputs.ctypes.data, inputs.shape[0], out.ctypes.data, ok.ctypes.data))
        return out, ok

    def verify_batch_device(self, kinds, count, fields_dev_ptr, verdicts_dev_ptr, stream=0):
        """Enqueue Issuer::verify for a batch already in device memory ([n_fields][count][32]); no synchronisation."""
        self._b.check(self._b.L.afx_verify_presentations_device(self._h, len(kinds), bytes(kinds), count, fields_dev_ptr, verdicts_dev_ptr, stream))
