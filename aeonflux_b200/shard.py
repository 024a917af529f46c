"""Multi-GPU sharding and mixed-shape streaming for the batch engine (SURVEY 8e, BASELINE config 5).

Every presentation / issuance is an independent unit of work (the reference's CompactProof forbids cross-item aggregation,
/root/reference/src/nizk/presentation.rs:31), so the path shards with no data-path collective:

  * one process per GPU, each holding a replicated issuer context (`Issuer`);
  * rank k of G takes the contiguous item range [k*N/G, (k+1)*N/G) of every batch;
  * only the accept/reject bitmap (1 bit per item) is gathered -- `torch.distributed.all_gather` over whatever backend the
    process group was created with (NCCL on the GPU box, gloo in the CPU tests).  The math never touches a collective.

`bucket_by_shape` / `ShardedIssuer.verify_mixed` implement the streamed mixed-shape workload: items are bucketed by their
attribute-kind vector (one compiled shape program per bucket), cut into chunks of at most `max_batch`, verified chunk by
chunk and scattered back into the caller's order.
"""
import numpy as np

from .issuer import PresentationBatch


def slice_bounds(total: int, rank: int, world: int):
    """Contiguous slice of `total` items owned by `rank` (SURVEY 8e): [rank*total/world, (rank+1)*total/world)."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    return (rank * total) // world, ((rank + 1) * total) // world


def pack_bitmap(verdicts) -> np.ndarray:
    """verdict bytes (0 = Ok, non-zero = VerificationFailure) -> little-endian bitmap, 1 bit per item (1 = rejected)."""
    return np.packbits(np.asarray(verdicts, dtype=np.uint8) != 0, bitorder="little")


def unpack_bitmap(bitmap, count: int) -> np.ndarray:
    return np.unpackbits(np.asarray(bitmap, dtype=np.uint8), count=count, bitorder="little").astype(np.uint8)


def bucket_by_shape(kinds_list):
    """kinds_list: one attribute-kind vector (bytes) per item -> {kinds: ndarray of item indices, in stream order}."""
    buckets = {}
    for i, k in enumerate(kinds_list):
        buckets.setdefault(bytes(k), []).append(i)
    return {k: np.asarray(v, dtype=np.int64) for k, v in buckets.items()}


class ShardedIssuer:
    """Data-parallel wrapper around one `Issuer` per process.  With no process group (world 1) it degenerates to the
    single-GPU path, so the same code drives 1, 2, 4 or 8 B200s."""

    def __init__(self, issuer, rank=None, world=None, group=None):
        self.issuer = issuer
        self.group = group
        if rank is None or world is None:
            rank, world = 0, 1
            try:
                import torch.distributed as dist
                if dist.is_available() and dist.is_initialized():
                    rank, world = dist.get_rank(group), dist.get_world_size(group)
            except ImportError:
                pass
        self.rank, self.world = rank, world
        self.gather_seconds = 0.0

    # -- the only communication on the path: the verdict bitmap ------------------------------------------------------
    def _gather_bitmaps(self, local_bits: np.ndarray, total: int) -> np.ndarray:
        if self.world == 1:
            return unpack_bitmap(local_bits, total)
        import time
        import torch
        t0 = time.perf_counter()
        import torch.distributed as dist
        width = (-(-total // self.world) + 7) // 8 + 1          # bytes of the largest slice's bitmap
        dev = "cuda" if dist.get_backend(self.group) == "nccl" else "cpu"
        mine = torch.zeros(width, dtype=torch.uint8)
        mine[:len(local_bits)] = torch.from_numpy(local_bits)
        mine = mine.to(dev)
        allbits = torch.empty(self.world * width, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allbits, mine, group=self.group)          # the only collective on the path: 1 bit per item
        parts = allbits.cpu().numpy().reshape(self.world, width)
        out = np.empty(total, np.uint8)
        for r in range(self.world):
            lo, hi = slice_bounds(total, r, self.world)
            out[lo:hi] = unpack_bitmap(parts[r], hi - lo)
        self.gather_seconds += time.perf_counter() - t0      # includes waiting for the slowest rank
        return out

    def local_slice(self, batch: PresentationBatch) -> PresentationBatch:
        lo, hi = slice_bounds(batch.count, self.rank, self.world)
        return PresentationBatch(batch.kinds, batch.fields[:, lo:hi])

    def verify_batch(self, batch: PresentationBatch) -> np.ndarray:
        """Batch Issuer::verify over the global batch: this rank verifies its slice; every rank returns all verdicts."""
        local = self.issuer.verify_batch(self.local_slice(batch)) if batch.count else np.zeros(0, np.uint8)
        return self._gather_bitmaps(pack_bitmap(local), batch.count)

    def verify_issuance_batch(self, batch: PresentationBatch) -> np.ndarray:
        local = self.issuer.verify_issuance_batch(self.local_slice(batch)) if batch.count else np.zeros(0, np.uint8)
        return self._gather_bitmaps(pack_bitmap(local), batch.count)

    def verify_wire(self, kinds, items, issuance=False) -> np.ndarray:
        """The same over item-major wire bytes [count][n_fields][32]: this rank's slice is one contiguous byte range (one
        host-to-device copy); every rank returns all verdicts."""
        lo, hi = slice_bounds(len(items), self.rank, self.world)
        local = self.issuer.verify_wire(kinds, items[lo:hi], issuance=issuance) if hi > lo else np.zeros(0, np.uint8)
        return self._gather_bitmaps(pack_bitmap(local), len(items))

    def verify_stream(self, stream, records, offsets, shape_ids) -> np.ndarray:
        """Streamed verification of a mixed-shape record stream (BASELINE configs[4]): this rank pushes the contiguous slice
        [rank*T/world, (rank+1)*T/world) of the stream through its `MixedStream` (whose shapes are registered with this rank's
        issuer contexts); only the verdict bitmap is gathered.  Every rank returns all T verdicts."""
        total = len(offsets)
        lo, hi = slice_bounds(total, self.rank, self.world)
        local = np.zeros(hi - lo, np.uint8)
        if hi > lo:
            stream.push(records, offsets[lo:hi], shape_ids[lo:hi], local)
        stream.flush()
        return self._gather_bitmaps(pack_bitmap(local), total)

    def verify_mixed(self, kinds_list, items, issuers=None) -> np.ndarray:
        """Streamed verification of presentations of mixed shapes (BASELINE config 5).

        kinds_list[i] is item i's attribute-kind vector and items[i] its words, uint8 [n_fields(kinds)][32].  Shapes with a
        different attribute count belong to different issuers: pass `issuers` = {n_attrs: Issuer}; by default every item
        goes to self.issuer.  Items are bucketed by shape, verified in chunks of at most max_batch, and the verdicts are
        returned in stream order."""
        total = len(kinds_list)
        out = np.zeros(total, np.uint8)
        for kinds, idx in sorted(bucket_by_shape(kinds_list).items()):
            issuer = issuers[len(kinds)] if issuers else self.issuer
            step = issuer.max_batch * self.world
            for s in range(0, len(idx), step):
                sel = idx[s:s + step]
                fields = np.ascontiguousarray(np.stack([items[i] for i in sel], axis=1))
                lo, hi = slice_bounds(len(sel), self.rank, self.world)
                local = issuer.verify_batch(PresentationBatch(kinds, fields[:, lo:hi])) if hi > lo else np.zeros(0, np.uint8)
                out[sel] = self._gather_bitmaps(pack_bitmap(local), len(sel))
        return out


class MultiGpuIssuer:
    """ONE process driving several B200s through the C ABI's multi-device handle (afx_multi_*, SURVEY 8b/8e): the library
    replicates the issuer context on every listed device, keeps one host thread + stream set per device, cuts every batch into
    contiguous item slices [k*N/G, (k+1)*N/G) and lets each device write its slice of the verdict array.  This is the form a
    single-process caller -- the reference is a library, its `Issuer::verify_batch` shim runs inside the application -- uses
    instead of one process per GPU.  This class only marshals arguments."""

    def __init__(self, system_parameters, issuer_parameters, amacs_key=None, devices=(0,), max_batch=65536, _binding=None):
        import ctypes
        if _binding is None:
            from ._lib import load
            _binding = load()
        if not devices:
            raise ValueError("at least one device")
        self._b = _binding
        self.devices = list(devices)
        self.max_batch = max_batch
        sp, ip = bytes(system_parameters), bytes(issuer_parameters)
        if len(ip) != 64:
            raise ValueError("issuer_parameters must be C_W || I (64 bytes)")
        self.number_of_attributes = int.from_bytes(sp[:4], "little")
        sk = ctypes.create_string_buffer(bytes(amacs_key), len(amacs_key)) if amacs_key is not None else None
        devs = (ctypes.c_int * len(self.devices))(*self.devices)
        h = ctypes.c_void_p()
        rc = self._b.L.afx_multi_create(sp, len(sp), ip, ctypes.addressof(sk) if sk is not None else None, len(amacs_key) if amacs_key is not None else 0,
                                        devs, len(self.devices), max_batch, ctypes.byref(h))
        if sk is not None:
            ctypes.memset(sk, 0, len(amacs_key))
        self._b.check(rc)
        self._h = h

    def host_array(self, shape):
        return self._b.host_array(shape)

    def _soa(self, fn, batch):
        import ctypes
        from . import _binding as B
        ptrs, keep = B._as_fields(batch.fields)
        cb = B.afx_presentation_batch(len(batch.kinds), batch.kinds, batch.count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        verdicts = np.zeros(batch.count, np.uint8)
        self._b.check(fn(self._h, ctypes.byref(cb), verdicts.ctypes.data))
        return verdicts

    def verify_batch(self, batch: PresentationBatch) -> np.ndarray:
        """Batch Issuer::verify: device k verifies items [k*N/G, (k+1)*N/G); verdicts in item order."""
        return self._soa(self._b.L.afx_multi_verify_presentations, batch)

    def verify_issuance_batch(self, batch: PresentationBatch) -> np.ndarray:
        return self._soa(self._b.L.afx_multi_verify_issuances, batch)

    def verify_wire(self, kinds, items, issuance=False) -> np.ndarray:
        """The same over item-major wire bytes [count][n_fields][32]: each device copies its contiguous byte range."""
        items = np.ascontiguousarray(items, dtype=np.uint8)
        kinds = bytes(kinds)
        nf = (2 * len(kinds) + 9) if issuance else self._b.L.afx_presentation_num_fields(len(kinds), kinds)
        if items.ndim != 3 or items.shape[1:] != (nf, 32):
            raise ValueError("items must be [count][%d][32] bytes for this shape" % nf)
        verdicts = np.zeros(items.shape[0], np.uint8)
        fn = self._b.L.afx_multi_verify_issuances_wire if issuance else self._b.L.afx_multi_verify_presentations_wire
        self._b.check(fn(self._h, len(kinds), kinds, items.shape[0], items.ctypes.data, verdicts.ctypes.data))
        return verdicts

    def verify_mixed_wire(self, shape_kinds, records, shape_ids, issuance=False) -> np.ndarray:
        """Issuer.verify_mixed_wire across the devices: device k takes records [k*N/G, (k+1)*N/G) and buckets them itself."""
        from . import _binding as B
        fn = self._b.L.afx_multi_verify_issuances_mixed_wire if issuance else self._b.L.afx_multi_verify_presentations_mixed_wire
        return B.mixed_wire(self._b, fn, self._h, shape_kinds, records, shape_ids, "issuance" if issuance else "presentation")

    def issue_mixed_wire(self, shape_kinds, requests, shape_ids):
        """Issuer.issue_mixed_wire across the devices: device k issues records [k*N/G, (k+1)*N/G) -> (issuances, status)."""
        from . import _binding as B
        out, status = B.mixed_wire(self._b, self._b.L.afx_multi_issue_mixed_wire, self._h, shape_kinds, requests, shape_ids, "request", "issuance")
        n = len(bytes(shape_kinds[0])) if len(shape_kinds) else 0
        return out.reshape(len(status), 2 * n + 9, 32), status

    def issue_batch(self, batch):
        """Batch Issuer::issue across the devices (request layout of Issuer.issue_batch) -> (IssuanceBatch, status)."""
        import ctypes
        from . import _binding as B
        n, count = len(batch.kinds), batch.count
        if batch.fields.shape[0] != 3 * n + 14:
            raise ValueError("a request batch has 3n + 14 fields")
        ptrs, keep = B._as_fields(batch.fields)
        cb = B.afx_presentation_batch(n, batch.kinds, count, ctypes.cast(ptrs, ctypes.POINTER(ctypes.c_void_p)), len(keep))
        out = np.zeros((2 * n + 9, count, 32), np.uint8)
        out[:n] = batch.fields[:n]
        optrs, okeep = B._as_fields(out[n:])
        ob = B.afx_issuance_out(ctypes.cast(optrs, ctypes.POINTER(ctypes.c_void_p)), len(okeep))
        status = np.zeros(count, np.uint8)
        self._b.check(self._b.L.afx_multi_issue(self._h, ctypes.byref(cb), ctypes.byref(ob), status.ctypes.data))
        return PresentationBatch(batch.kinds, out), status

    def close(self):
        if getattr(self, "_h", None):
            self._b.L.afx_multi_destroy(self._h)
            self._h = None

    __del__ = close


class MixedStream:
    """Streamed verification of mixed shapes through the library's stream object (afx_stream_*, BASELINE configs[4]): records of
    several shapes arrive interleaved; the library buckets them by shape into page-locked buckets (three per shape: one filling, two in flight) and submits every full
    bucket asynchronously, so bucketing, copies and kernels overlap.  Shapes of different attribute counts belong to different
    issuers: register each with the `Issuer` that verifies it."""

    def __init__(self, _binding=None):
        import ctypes
        if _binding is None:
            from ._lib import load
            _binding = load()
        self._b = _binding
        h = ctypes.c_void_p()
        self._b.check(self._b.L.afx_stream_create(ctypes.byref(h)))
        self._h = h
        self.record_bytes = []
        self._keep = []

    def add_shape(self, issuer, kinds, issuance=False) -> int:
        import ctypes
        sid, rb = ctypes.c_int(-1), ctypes.c_size_t(0)
        kinds = bytes(kinds)
        self._b.check(self._b.L.afx_stream_add_shape(self._h, issuer._h, 1 if issuance else 0, len(kinds), kinds, ctypes.byref(sid), ctypes.byref(rb)))
        self.record_bytes.append(int(rb.value))
        self._keep.append(issuer)
        return int(sid.value)

    def push(self, records, offsets, shape_ids, verdicts):
        """records: uint8 blob; offsets: uint64 [n] byte offset of each record; shape_ids: uint8 [n]; verdicts: uint8 [n], filled in
        by the time flush() returns (keep it alive until then)."""
        records = np.ascontiguousarray(records, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        shape_ids = np.ascontiguousarray(shape_ids, dtype=np.uint8)
        if not (verdicts.dtype == np.uint8 and verdicts.flags.c_contiguous and len(verdicts) == len(offsets) == len(shape_ids)):
            raise ValueError("verdicts must be a contiguous uint8 array with one entry per record")
        if len(offsets) and int(shape_ids.max()) < len(self.record_bytes):      # an unknown shape id is the library's error to report
            ends = offsets + np.asarray(self.record_bytes, np.uint64)[shape_ids]
            if int(ends.max()) > records.size:
                raise ValueError("a record reaches past the end of the blob")
        self._keep.append((records, verdicts))
        self._b.check(self._b.L.afx_stream_push(self._h, records.ctypes.data, offsets.ctypes.data, shape_ids.ctypes.data, len(offsets), verdicts.ctypes.data))

    def flush(self):
        self._b.check(self._b.L.afx_stream_flush(self._h))
        self._keep = [k for k in self._keep if not isinstance(k, tuple)]

    def times(self):
        """Cumulative host seconds of the driving thread: (copying records into buckets, enqueueing submissions, blocked on the device)."""
        import ctypes
        a, b, c = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
        self._b.check(self._b.L.afx_stream_times(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    @property
    def buckets_submitted(self):
        return int(self._b.L.afx_stream_buckets_submitted(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._b.L.afx_stream_destroy(self._h)
            self._h = None

    __del__ = close


def interleave_records(pools, order):
    """pools[s]: uint8 [count_s][n_fields_s][32] items of shape s; order: uint8 [total] shape id of every stream position (shape s
    must occur count_s times) -> (blob, offsets): the stream as one byte blob of variable-length records, in `order`."""
    order = np.asarray(order, dtype=np.uint8)
    sizes = np.asarray([p.shape[1] * 32 for p in pools], np.uint64)
    rec = sizes[order]
    offsets = np.zeros(len(order), np.uint64)
    np.cumsum(rec[:-1], out=offsets[1:])
    blob = np.empty(int(rec.sum()), np.uint8)
    for sid, p in enumerate(pools):
        pos = np.nonzero(order == sid)[0]
        if len(pos) != len(p):
            raise ValueError("order does not match the pool sizes")
        w = p.shape[1] * 32
        # scatter the pool's items to their stream offsets (row gather through an index matrix, chunked to bound memory)
        flat = p.reshape(len(p), w)
        for lo in range(0, len(pos), 1 << 16):
            o = offsets[pos[lo:lo + (1 << 16)]].astype(np.int64)
            blob[(o[:, None] + np.arange(w, dtype=np.int64)[None, :]).ravel()] = flat[lo:lo + (1 << 16)].ravel()
    return blob, offsets
