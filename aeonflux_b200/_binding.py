"""ctypes binding of the C ABI in include/aeonflux_b200.h (the stub a reference maintainer's FFI would mirror,
see INTEGRATION.md).  `Binding` wraps an already-loaded library handle; `aeonflux_b200._lib.load()` is the only place the
package loads one, and it loads the CUDA build or fails."""
import ctypes

import numpy as np

AFX_OK = 0


class afx_presentation_batch(ctypes.Structure):
    _fields_ = [("n_attrs", ctypes.c_uint16), ("kinds", ctypes.c_char_p), ("count", ctypes.c_size_t),
                ("fields", ctypes.POINTER(ctypes.c_void_p)), ("n_fields", ctypes.c_size_t)]


class afx_issuance_out(ctypes.Structure):
    _fields_ = [("fields", ctypes.POINTER(ctypes.c_void_p)), ("n_fields", ctypes.c_size_t)]


class afx_debug_dump(ctypes.Structure):
    _fields_ = [("Z", ctypes.c_void_p), ("commitments", ctypes.c_void_p), ("challenges", ctypes.c_void_p), ("status", ctypes.c_void_p)]


class AfxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("aeonflux_b200 error %d: %s" % (code, msg))
        self.code = code


class Binding:
    SYMBOLS = ["afx_ctx_create", "afx_ctx_destroy", "afx_presentation_num_fields", "afx_presentation_num_commitments",
               "afx_presentation_num_proofs", "afx_verify_presentations", "afx_verify_presentations_device", "afx_verify_issuances",
               "afx_verify_issuances_device", "afx_verify_presentations_submit", "afx_verify_issuances_submit", "afx_wait", "afx_host_alloc", "afx_host_free", "afx_batchable_num_fields", "afx_verify_presentations_batchable", "afx_verify_presentations_batchable_rlc", "afx_verify_presentations_wire", "afx_verify_issuances_wire", "afx_request_num_fields", "afx_issue", "afx_issue_device", "afx_show_num_fields", "afx_show", "afx_show_device", "afx_selftest_primitive", "afx_launch_count", "afx_ctx_device", "afx_bind_thread_to_device", "afx_set_stage_timing", "afx_get_stage_times", "afx_get_rlc_bucket_time", "afx_strerror", "afx_version",
               "afx_multi_create", "afx_multi_destroy", "afx_multi_num_devices", "afx_multi_ctx", "afx_multi_verify_presentations",
               "afx_multi_verify_presentations_wire", "afx_multi_verify_issuances", "afx_multi_verify_issuances_wire", "afx_multi_issue",
               "afx_verify_presentations_wire_submit", "afx_verify_issuances_wire_submit", "afx_stream_create", "afx_stream_destroy",
               "afx_stream_add_shape", "afx_stream_push", "afx_stream_flush", "afx_stream_buckets_submitted", "afx_stream_times",
               "afx_issue_wire", "afx_show_wire", "afx_presentation_linked_num_commitments", "afx_verify_presentations_linked",
               "afx_verify_presentations_linked_wire", "afx_show_linked", "afx_show_linked_wire", "afx_issuance_batchable_num_fields", "afx_verify_issuances_batchable", "afx_verify_issuances_batchable_rlc", "afx_get_rlc_stats",
               "afx_encode_plaintexts", "afx_encrypt", "afx_decrypt", "afx_encode_plaintexts_device", "afx_encrypt_device",
               "afx_decrypt_device", "afx_derive_keypairs", "afx_derive_keypairs_device", "afx_issue_batchable", "afx_issue_batchable_device",
               "afx_show_batchable", "afx_show_batchable_device", "afx_verify_presentations_mixed_wire", "afx_verify_issuances_mixed_wire",
               "afx_multi_verify_presentations_mixed_wire", "afx_multi_verify_issuances_mixed_wire", "afx_issue_mixed_wire",
               "afx_show_mixed_wire", "afx_multi_issue_mixed_wire"]

    def __init__(self, cdll):
        L = self.L = cdll
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        L.afx_ctx_create.restype = ctypes.c_int
        L.afx_ctx_create.argtypes = [vp, sz, vp, vp, sz, ctypes.c_int, sz, ctypes.POINTER(vp)]
        L.afx_ctx_destroy.restype = None
        L.afx_ctx_destroy.argtypes = [vp]
        for f in ("afx_presentation_num_fields", "afx_presentation_num_commitments", "afx_presentation_num_proofs"):
            getattr(L, f).restype = sz
            getattr(L, f).argtypes = [ctypes.c_uint16, ctypes.c_char_p]
        L.afx_verify_presentations.restype = ctypes.c_int
        L.afx_verify_presentations.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, ctypes.POINTER(afx_debug_dump)]
        L.afx_verify_issuances.restype = ctypes.c_int
        L.afx_verify_issuances.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, ctypes.POINTER(afx_debug_dump)]
        L.afx_verify_presentations_device.restype = ctypes.c_int
        L.afx_verify_presentations_device.argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp, vp]
        L.afx_verify_issuances_device.restype = ctypes.c_int
        L.afx_verify_issuances_device.argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp, vp]
        for f in ("afx_verify_presentations_submit", "afx_verify_issuances_submit"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, ctypes.POINTER(ctypes.c_uint64)]
        L.afx_wait.restype = ctypes.c_int
        L.afx_wait.argtypes = [vp, ctypes.c_uint64]
        L.afx_host_alloc.restype = ctypes.c_int
        L.afx_host_alloc.argtypes = [ctypes.POINTER(vp), sz]
        L.afx_host_free.restype = None
        L.afx_host_free.argtypes = [vp]
        L.afx_batchable_num_fields.restype = sz
        L.afx_batchable_num_fields.argtypes = [ctypes.c_uint16, ctypes.c_char_p]
        L.afx_verify_presentations_batchable.restype = ctypes.c_int
        L.afx_verify_presentations_batchable.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, ctypes.POINTER(afx_debug_dump)]
        L.afx_verify_presentations_batchable_rlc.restype = ctypes.c_int
        L.afx_verify_presentations_batchable_rlc.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, vp, ctypes.POINTER(ctypes.c_uint32)]
        L.afx_issuance_batchable_num_fields.restype = sz
        L.afx_issuance_batchable_num_fields.argtypes = [ctypes.c_uint16]
        L.afx_verify_issuances_batchable.restype = ctypes.c_int
        L.afx_verify_issuances_batchable.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, ctypes.POINTER(afx_debug_dump)]
        L.afx_verify_issuances_batchable_rlc.restype = ctypes.c_int
        L.afx_verify_issuances_batchable_rlc.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, vp, ctypes.POINTER(ctypes.c_uint32)]
        L.afx_get_rlc_stats.restype = ctypes.c_int
        L.afx_get_rlc_stats.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
        for f in ("afx_verify_presentations_wire", "afx_verify_issuances_wire"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp]
        L.afx_request_num_fields.restype = sz
        L.afx_request_num_fields.argtypes = [ctypes.c_uint16]
        L.afx_show_num_fields.restype = sz
        L.afx_show_num_fields.argtypes = [ctypes.c_uint16, ctypes.c_char_p]
        for f in ("afx_issue", "afx_show", "afx_issue_batchable", "afx_show_batchable"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.POINTER(afx_presentation_batch), ctypes.POINTER(afx_issuance_out), vp, ctypes.POINTER(afx_debug_dump)]
        for f in ("afx_issue_device", "afx_show_device", "afx_issue_batchable_device", "afx_show_batchable_device"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp, vp, vp]
        L.afx_presentation_linked_num_commitments.restype = sz
        L.afx_presentation_linked_num_commitments.argtypes = [ctypes.c_uint16, ctypes.c_char_p]
        L.afx_verify_presentations_linked.restype = ctypes.c_int
        L.afx_verify_presentations_linked.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp, ctypes.POINTER(afx_debug_dump)]
        L.afx_verify_presentations_linked_wire.restype = ctypes.c_int
        L.afx_verify_presentations_linked_wire.argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp]
        L.afx_show_linked.restype = ctypes.c_int
        L.afx_show_linked.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), ctypes.POINTER(afx_issuance_out), vp, ctypes.POINTER(afx_debug_dump)]
        for f in ("afx_issue_wire", "afx_show_wire", "afx_show_linked_wire"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp, vp]
        L.afx_encode_plaintexts.restype = ctypes.c_int
        L.afx_encode_plaintexts.argtypes = [vp, sz, vp, vp, vp]
        L.afx_encrypt.restype = ctypes.c_int
        L.afx_encrypt.argtypes = [vp, vp, sz, vp, vp, vp]
        L.afx_decrypt.restype = ctypes.c_int
        L.afx_decrypt.argtypes = [vp, vp, sz, vp, vp, vp, vp]
        L.afx_encode_plaintexts_device.restype = ctypes.c_int
        L.afx_encode_plaintexts_device.argtypes = [vp, sz, vp, vp, vp, vp]
        L.afx_encrypt_device.restype = ctypes.c_int
        L.afx_encrypt_device.argtypes = [vp, vp, sz, vp, vp, vp, vp]
        L.afx_decrypt_device.restype = ctypes.c_int
        L.afx_decrypt_device.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp]
        L.afx_derive_keypairs.restype = ctypes.c_int
        L.afx_derive_keypairs.argtypes = [vp, sz, vp, vp]
        L.afx_derive_keypairs_device.restype = ctypes.c_int
        L.afx_derive_keypairs_device.argtypes = [vp, sz, vp, vp, vp]
        L.afx_selftest_primitive.restype = ctypes.c_int
        L.afx_selftest_primitive.argtypes = [vp, ctypes.c_int, vp, sz, vp, vp]
        L.afx_launch_count.restype = ctypes.c_uint64
        L.afx_launch_count.argtypes = [vp]
        L.afx_set_stage_timing.restype = None
        L.afx_set_stage_timing.argtypes = [vp, ctypes.c_int]
        L.afx_get_stage_times.restype = ctypes.c_int
        L.afx_get_stage_times.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.c_int]
        L.afx_get_rlc_bucket_time.restype = ctypes.c_int
        L.afx_get_rlc_bucket_time.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint32)]
        L.afx_ctx_device.restype = ctypes.c_int
        L.afx_ctx_device.argtypes = [vp]
        L.afx_bind_thread_to_device.restype = ctypes.c_int
        L.afx_bind_thread_to_device.argtypes = [ctypes.c_int]
        L.afx_strerror.restype = ctypes.c_char_p
        L.afx_strerror.argtypes = [ctypes.c_int]
        L.afx_version.restype = ctypes.c_char_p
        for f in ("afx_verify_presentations_wire_submit", "afx_verify_issuances_wire_submit"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp, ctypes.POINTER(ctypes.c_uint64)]
        L.afx_stream_create.restype = ctypes.c_int
        L.afx_stream_create.argtypes = [ctypes.POINTER(vp)]
        L.afx_stream_destroy.restype = None
        L.afx_stream_destroy.argtypes = [vp]
        L.afx_stream_add_shape.restype = ctypes.c_int
        L.afx_stream_add_shape.argtypes = [vp, vp, ctypes.c_int, ctypes.c_uint16, ctypes.c_char_p, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(sz)]
        L.afx_stream_push.restype = ctypes.c_int
        L.afx_stream_push.argtypes = [vp, vp, vp, vp, sz, vp]
        L.afx_stream_flush.restype = ctypes.c_int
        L.afx_stream_flush.argtypes = [vp]
        L.afx_stream_times.restype = ctypes.c_int
        L.afx_stream_times.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        L.afx_stream_buckets_submitted.restype = ctypes.c_uint64
        L.afx_stream_buckets_submitted.argtypes = [vp]
        L.afx_multi_create.restype = ctypes.c_int
        L.afx_multi_create.argtypes = [vp, sz, vp, vp, sz, ctypes.POINTER(ctypes.c_int), ctypes.c_int, sz, ctypes.POINTER(vp)]
        L.afx_multi_destroy.restype = None
        L.afx_multi_destroy.argtypes = [vp]
        L.afx_multi_num_devices.restype = ctypes.c_int
        L.afx_multi_num_devices.argtypes = [vp]
        L.afx_multi_ctx.restype = vp
        L.afx_multi_ctx.argtypes = [vp, ctypes.c_int]
        for f in ("afx_multi_verify_presentations", "afx_multi_verify_issuances"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.POINTER(afx_presentation_batch), vp]
        for f in ("afx_multi_verify_presentations_wire", "afx_multi_verify_issuances_wire"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, vp, vp]
        for f in ("afx_verify_presentations_mixed_wire", "afx_verify_issuances_mixed_wire", "afx_multi_verify_presentations_mixed_wire",
                  "afx_multi_verify_issuances_mixed_wire"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, sz, vp, vp, vp]
        for f in ("afx_issue_mixed_wire", "afx_show_mixed_wire", "afx_multi_issue_mixed_wire"):
            getattr(L, f).restype = ctypes.c_int
            getattr(L, f).argtypes = [vp, ctypes.c_uint16, ctypes.c_char_p, sz, sz, vp, vp, vp, vp]
        L.afx_multi_issue.restype = ctypes.c_int
        L.afx_multi_issue.argtypes = [vp, ctypes.POINTER(afx_presentation_batch), ctypes.POINTER(afx_issuance_out), vp]

    def check(self, rc):
        if rc != AFX_OK:
            raise AfxError(rc, self.L.afx_strerror(rc).decode())

    def version(self):
        return self.L.afx_version().decode()

    def host_array(self, shape):
        """uint8 ndarray of `shape` in page-locked host memory (afx_host_alloc), freed when the array is collected."""
        import weakref
        n = int(np.prod(shape))
        p = ctypes.c_void_p()
        self.check(self.L.afx_host_alloc(ctypes.byref(p), n))
        buf = (ctypes.c_uint8 * max(n, 1)).from_address(p.value)
        weakref.finalize(buf, self.L.afx_host_free, p.value)
        return np.frombuffer(buf, dtype=np.uint8, count=n).reshape(shape)


def _as_fields(fields):
    """fields: ndarray [n_fields][count][32] uint8 (or a list of [count][32] arrays) -> (ctypes pointer array, keepalive)"""
    arrs = [np.ascontiguousarray(f, dtype=np.uint8) for f in fields]
    ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    return ptrs, arrs


def mixed_record_bytes(binding, shape_kinds, what):
    """Record length in bytes of every kind vector of a mixed call: what = "request", "issuance", "show" (a show input) or
    "presentation"."""
    L = binding.L
    size = {"request": lambda k: 3 * len(k) + 14, "issuance": lambda k: 2 * len(k) + 9,
            "show": lambda k: L.afx_show_num_fields(len(k), k), "presentation": lambda k: L.afx_presentation_num_fields(len(k), k)}[what]
    return np.array([32 * size(bytes(k)) for k in shape_kinds], np.int64)


def record_offsets(sizes, shape_ids):
    """Byte offsets [count + 1] of records concatenated in order, record i of sizes[shape_ids[i]] bytes: record i is
    blob[offsets[i]:offsets[i + 1]]."""
    ids = np.asarray(shape_ids, np.uint8).reshape(-1)
    offsets = np.zeros(len(ids) + 1, np.int64)
    np.cumsum(np.asarray(sizes, np.int64)[ids], out=offsets[1:])
    return offsets


def mixed_wire(binding, fn, handle, shape_kinds, records, shape_ids, what, out_what=None, out=None):
    """Marshals the mixed-shape calls: shape_kinds = the kind vectors of the call, records = uint8 array holding the input records
    concatenated in order, record i a `what` record (see mixed_record_bytes) of shape shape_ids[i], shape_ids = uint8 [count].
    afx_[multi_]verify_{presentations,issuances}_mixed_wire (out_what None) return the verdicts.  afx_[multi_]{issue,show}_mixed_wire
    (out_what "issuance" or "presentation") return (the output records concatenated in order as a flat uint8 array, status); out:
    optional preallocated (e.g. page-locked) contiguous uint8 array of exactly the output size, returned flattened."""
    shape_kinds = [bytes(k) for k in shape_kinds]
    n = len(shape_kinds[0]) if shape_kinds else 0
    if any(len(k) != n for k in shape_kinds):
        raise ValueError("every kind vector of a call has the issuer's attribute count")
    records = np.ascontiguousarray(records, dtype=np.uint8).reshape(-1)
    ids = np.ascontiguousarray(shape_ids, dtype=np.uint8).reshape(-1)
    out_bytes = 0
    if len(ids) and int(ids.max()) < len(shape_kinds):      # an unknown shape id is the library's error to report
        if int(mixed_record_bytes(binding, shape_kinds, what)[ids].sum()) != records.size:
            raise ValueError("%s must hold exactly one record of its shape per shape id" % ("inputs" if out_what else "records"))
        if out_what:
            out_bytes = int(mixed_record_bytes(binding, shape_kinds, out_what)[ids].sum())
    status = np.zeros(len(ids), np.uint8)
    args = [handle, n, b"".join(shape_kinds), len(shape_kinds), len(ids), records.ctypes.data, ids.ctypes.data]
    if not out_what:
        binding.check(fn(*args, status.ctypes.data))
        return status
    if out is None:
        out = np.zeros(out_bytes, np.uint8)
    elif out.dtype != np.uint8 or not out.flags.c_contiguous or out.size != out_bytes:
        raise ValueError("out must be a contiguous uint8 array of %d bytes" % out_bytes)
    out = out.reshape(-1)
    binding.check(fn(*args, out.ctypes.data, status.ctypes.data))
    return out, status
