//! Safe wrappers over `libaeonflux_b200.so` (include/aeonflux_b200.h) for the batch entry points INTEGRATION.md adds beside
//! `Issuer::verify`, `Issuer::issue` and `CredentialIssuance::verify`.
//!
//! NEVER COMPILED in this repository: its build image has no Rust toolchain (rust/README.md).  The raw FFI -- extern block,
//! #[repr(C)] descriptors, constants -- is `ffi.rs`, GENERATED from the header by tools/gen_rust_ffi.py (a CPU test regenerates it
//! and compares, so it cannot drift); this file is hand-written and review-sized.  Everything is expressed over the reference's own
//! byte encodings: `SystemParameters::to_bytes()` (src/parameters.rs:155-184), the 64 bytes `C_W || I` (src/issuer.rs:155,163),
//! `amacs::SecretKey::to_bytes()` (src/amacs.rs:110-125), canonical scalars and compressed points.

use std::os::raw::c_int;

#[path = "ffi.rs"]
mod ffi;
pub use ffi::*;

/// `afx_presentation_batch`, `afx_issuance_batch`, `afx_request_batch` and `afx_show_batch` share one layout.
type afx_batch = afx_presentation_batch;
type afx_out = afx_issuance_out;

/// A byte buffer in page-locked host memory (`afx_host_alloc`).  Build the struct-of-arrays fields of a batch in these:
/// the library's host-to-device copies then run asynchronously at the full bus rate instead of being staged by the driver.
pub struct PinnedBytes {
    ptr: *mut u8,
    len: usize,
}

unsafe impl Send for PinnedBytes {}

impl PinnedBytes {
    pub fn new(len: usize) -> Result<PinnedBytes, B200Error> {
        let mut p: *mut std::os::raw::c_void = std::ptr::null_mut();
        let rc = unsafe { afx_host_alloc(&mut p, len) };
        if rc != 0 { return Err(B200Error(rc)); }
        unsafe { std::ptr::write_bytes(p as *mut u8, 0, len) };
        Ok(PinnedBytes { ptr: p as *mut u8, len })
    }
}

impl std::ops::Deref for PinnedBytes {
    type Target = [u8];
    fn deref(&self) -> &[u8] { unsafe { std::slice::from_raw_parts(self.ptr, self.len) } }
}

impl std::ops::DerefMut for PinnedBytes {
    fn deref_mut(&mut self) -> &mut [u8] { unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) } }
}

impl Drop for PinnedBytes {
    fn drop(&mut self) { unsafe { afx_host_free(self.ptr as *mut std::os::raw::c_void) } }
}

/// A non-zero return code of the C ABI (`AFX_ERR_*`).
#[derive(Clone, Copy, Debug, Eq, PartialEq)]
pub struct B200Error(pub i32);

impl std::fmt::Display for B200Error {
    fn fmt(&self, f: &mut std::fmt::Formatter) -> std::fmt::Result {
        let msg = unsafe { std::ffi::CStr::from_ptr(afx_strerror(self.0)) };
        write!(f, "aeonflux_b200 error {}: {}", self.0, msg.to_string_lossy())
    }
}

/// One issuer context on one B200.  Replicate it per GPU; every item of a batch is independent.
pub struct B200Context {
    ctx: *mut afx_ctx,
}

// One thread at a time per context (it owns one set of CUDA streams and one workspace).
unsafe impl Send for B200Context {}

impl B200Context {
    /// `secret_key = None` gives a user-side context: `verify_issuances*` and `show` work, `verify_presentations*` and `issue` do not.
    pub fn new(system_parameters: &[u8], issuer_parameters: &[u8; 64], secret_key: Option<&[u8]>, device: i32, max_batch: usize)
        -> Result<B200Context, B200Error>
    {
        let mut ctx: *mut afx_ctx = std::ptr::null_mut();
        let (sk, sk_len) = match secret_key { Some(s) => (s.as_ptr(), s.len()), None => (std::ptr::null(), 0) };
        let rc = unsafe {
            afx_ctx_create(system_parameters.as_ptr(), system_parameters.len(), issuer_parameters.as_ptr(), sk, sk_len,
                           device as c_int, max_batch, &mut ctx)
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(B200Context { ctx })
    }

    fn check_fields(fields: &[&[u8]], expected: usize) -> Result<usize, B200Error> {
        if fields.len() != expected { return Err(B200Error(-1)); }
        let count = if fields.is_empty() { 0 } else { fields[0].len() / 32 };
        if fields.iter().any(|f| f.len() != count * 32) { return Err(B200Error(-1)); }
        Ok(count)
    }

    /// Batch `Issuer::verify` over struct-of-arrays fields: verdict 0 = `Ok(())`, 1 = `Err(VerificationFailure)`.
    pub fn verify_presentations(&self, kinds: &[u8], fields: &[&[u8]]) -> Result<Vec<u8>, B200Error> {
        let n_fields = unsafe { afx_presentation_num_fields(kinds.len() as u16, kinds.as_ptr()) };
        let count = Self::check_fields(fields, n_fields)?;
        let ptrs: Vec<*const u8> = fields.iter().map(|f| f.as_ptr()).collect();
        let batch = afx_batch { n_attrs: kinds.len() as u16, kinds: kinds.as_ptr(), count, fields: ptrs.as_ptr(), n_fields };
        let mut verdicts = vec![0u8; count];
        let rc = unsafe { afx_verify_presentations(self.ctx, &batch, verdicts.as_mut_ptr(), std::ptr::null_mut()) };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }

    /// Asynchronous `Issuer::verify` of one pass (`count <= max_batch`): enqueues the copy, the kernels and the verdict
    /// read-back and returns a ticket for `wait`.  Two submissions may be outstanding, so the copy of one runs under the
    /// kernels of the other.  `fields` and `verdicts` must stay alive and untouched until `wait(ticket)` returns -- hence
    /// `unsafe`; a safe wrapper would own both in the returned handle.
    pub unsafe fn submit_presentations(&self, kinds: &[u8], fields: &[&[u8]], verdicts: &mut [u8]) -> Result<u64, B200Error> {
        let n_fields = afx_presentation_num_fields(kinds.len() as u16, kinds.as_ptr());
        let count = Self::check_fields(fields, n_fields)?;
        if verdicts.len() != count { return Err(B200Error(-1)); }
        let ptrs: Vec<*const u8> = fields.iter().map(|f| f.as_ptr()).collect();
        let batch = afx_batch { n_attrs: kinds.len() as u16, kinds: kinds.as_ptr(), count, fields: ptrs.as_ptr(), n_fields };
        let mut ticket = 0u64;
        let rc = afx_verify_presentations_submit(self.ctx, &batch, verdicts.as_mut_ptr(), &mut ticket);
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(ticket)
    }

    /// Blocks until the submission's verdicts are in the array given to `submit_presentations`.
    pub fn wait(&self, ticket: u64) -> Result<(), B200Error> {
        let rc = unsafe { afx_wait(self.ctx, ticket) };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(())
    }

    /// Batch `Issuer::verify` over item-major wire bytes (`count * n_fields * 32` bytes, as received).
    pub fn verify_presentations_wire(&self, kinds: &[u8], items: &[u8]) -> Result<Vec<u8>, B200Error> {
        let n_fields = unsafe { afx_presentation_num_fields(kinds.len() as u16, kinds.as_ptr()) };
        if n_fields == 0 || items.len() % (n_fields * 32) != 0 { return Err(B200Error(-1)); }
        let count = items.len() / (n_fields * 32);
        let mut verdicts = vec![0u8; count];
        let rc = unsafe {
            afx_verify_presentations_wire(self.ctx, kinds.len() as u16, kinds.as_ptr(), count, items.as_ptr(), verdicts.as_mut_ptr())
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }

    /// Batch `Issuer::verify` (issuance: `CredentialIssuance::verify`) over wire records of several shapes of this issuer:
    /// `records` = the records concatenated in order, record i of shape `shape_kinds[shape_ids[i]]`; bucketed on the device.
    pub fn verify_mixed_wire(&self, issuance: bool, shape_kinds: &[&[u8]], records: &[u8], shape_ids: &[u8]) -> Result<Vec<u8>, B200Error> {
        let (n, flat) = mixed_shapes(issuance, shape_kinds, records, shape_ids)?;
        let mut verdicts = vec![0u8; shape_ids.len()];
        let f = if issuance { afx_verify_issuances_mixed_wire } else { afx_verify_presentations_mixed_wire };
        let rc = unsafe { f(self.ctx, n, flat.as_ptr(), shape_kinds.len(), shape_ids.len(), records.as_ptr(), shape_ids.as_ptr(), verdicts.as_mut_ptr()) };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }

    /// Batch `Issuer::issue` over wire requests of several request kind vectors: `requests` = the requests concatenated in order
    /// (`3n + 14` words each), request i of kinds `shape_kinds[shape_ids[i]]`.  Returns the issuances in record order (`2n + 9` words
    /// each, what `verify_mixed_wire(true, ..)` takes) and a status byte per request.
    pub fn issue_mixed_wire(&self, shape_kinds: &[&[u8]], requests: &[u8], shape_ids: &[u8]) -> Result<(Vec<u8>, Vec<u8>), B200Error> {
        let (n, flat, out_len) = mixed_prover_shapes(true, shape_kinds, requests, shape_ids)?;
        let (mut out, mut status) = (vec![0u8; out_len], vec![0u8; shape_ids.len()]);
        let rc = unsafe {
            afx_issue_mixed_wire(self.ctx, n, flat.as_ptr(), shape_kinds.len(), shape_ids.len(), requests.as_ptr(), shape_ids.as_ptr(),
                                 out.as_mut_ptr(), status.as_mut_ptr())
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok((out, status))
    }

    /// Batch `AnonymousCredential::show` over wire show inputs of several disclosure patterns: `inputs` = the inputs concatenated in
    /// order, input i of shape `shape_kinds[shape_ids[i]]`.  Returns the presentations concatenated in record order (what
    /// `verify_mixed_wire(false, ..)` takes) and a status byte per input.
    pub fn show_mixed_wire(&self, shape_kinds: &[&[u8]], inputs: &[u8], shape_ids: &[u8]) -> Result<(Vec<u8>, Vec<u8>), B200Error> {
        let (n, flat, out_len) = mixed_prover_shapes(false, shape_kinds, inputs, shape_ids)?;
        let (mut out, mut status) = (vec![0u8; out_len], vec![0u8; shape_ids.len()]);
        let rc = unsafe {
            afx_show_mixed_wire(self.ctx, n, flat.as_ptr(), shape_kinds.len(), shape_ids.len(), inputs.as_ptr(), shape_ids.as_ptr(),
                                out.as_mut_ptr(), status.as_mut_ptr())
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok((out, status))
    }

    /// Batch `CredentialIssuance::verify` over struct-of-arrays fields (`attribute[n], t, U, V, challenge, responses[n+5]`).
    pub fn verify_issuances(&self, kinds: &[u8], fields: &[&[u8]]) -> Result<Vec<u8>, B200Error> {
        let n_fields = 2 * kinds.len() + 9;
        let count = Self::check_fields(fields, n_fields)?;
        let ptrs: Vec<*const u8> = fields.iter().map(|f| f.as_ptr()).collect();
        let batch = afx_batch { n_attrs: kinds.len() as u16, kinds: kinds.as_ptr(), count, fields: ptrs.as_ptr(), n_fields };
        let mut verdicts = vec![0u8; count];
        let rc = unsafe { afx_verify_issuances(self.ctx, &batch, verdicts.as_mut_ptr(), std::ptr::null_mut()) };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }

    fn prove(&self, issue: bool, kinds: &[u8], fields: &[&[u8]], n_in: usize, n_out: usize) -> Result<(Vec<Vec<u8>>, Vec<u8>), B200Error> {
        let count = Self::check_fields(fields, n_in)?;
        let ptrs: Vec<*const u8> = fields.iter().map(|f| f.as_ptr()).collect();
        let batch = afx_batch { n_attrs: kinds.len() as u16, kinds: kinds.as_ptr(), count, fields: ptrs.as_ptr(), n_fields: n_in };
        let mut out: Vec<Vec<u8>> = vec![vec![0u8; 32 * count]; n_out];
        let out_ptrs: Vec<*mut u8> = out.iter_mut().map(|f| f.as_mut_ptr()).collect();
        let out_desc = afx_out { fields: out_ptrs.as_ptr(), n_fields: n_out };
        let mut status = vec![0u8; count];
        let rc = unsafe {
            if issue { afx_issue(self.ctx, &batch, &out_desc, status.as_mut_ptr(), std::ptr::null_mut()) }
            else { afx_show(self.ctx, &batch, &out_desc, status.as_mut_ptr(), std::ptr::null_mut()) }
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok((out, status))
    }

    /// Batch `Issuer::issue`: fields = `attribute[n]` then the (lo, hi) halves of the 64 rng bytes of `t`, `U` and the `n+5`
    /// blindings.  Returns the output words `t, U, V, challenge, responses[n+5]` and a status byte per request.
    pub fn issue(&self, kinds: &[u8], fields: &[&[u8]]) -> Result<(Vec<Vec<u8>>, Vec<u8>), B200Error> {
        let n = kinds.len();
        self.prove(true, kinds, fields, unsafe { afx_request_num_fields(n as u16) }, n + 9)
    }

    /// Batch `AnonymousCredential::show`: fields per `afx_show`; returns the presentation's words.
    pub fn show(&self, kinds: &[u8], fields: &[&[u8]]) -> Result<(Vec<Vec<u8>>, Vec<u8>), B200Error> {
        let n_in = unsafe { afx_show_num_fields(kinds.len() as u16, kinds.as_ptr()) };
        let n_out = unsafe { afx_presentation_num_fields(kinds.len() as u16, kinds.as_ptr()) };
        self.prove(false, kinds, fields, n_in, n_out)
    }
}

impl Drop for B200Context {
    /// Zeroizes the device and host copies of the secret key (src/amacs.rs:64-82 semantics) and frees the context.
    fn drop(&mut self) {
        unsafe { afx_ctx_destroy(self.ctx) }
    }
}


/// The kind vectors of a mixed-shape call, flattened, after checking that `records` holds exactly one record per shape id (the
/// library takes no length and reads the records the shape ids describe).
fn mixed_shapes(issuance: bool, shape_kinds: &[&[u8]], records: &[u8], shape_ids: &[u8]) -> Result<(u16, Vec<u8>), B200Error> {
    let n = shape_kinds.first().map_or(0, |k| k.len());
    if shape_kinds.iter().any(|k| k.len() != n) { return Err(B200Error(-1)); }
    let bytes: Vec<usize> = shape_kinds.iter()
        .map(|k| 32 * if issuance { 2 * n + 9 } else { unsafe { afx_presentation_num_fields(n as u16, k.as_ptr()) } }).collect();
    let mut total = 0usize;
    for &s in shape_ids { match bytes.get(s as usize) { Some(b) => total += b, None => return Err(B200Error(-1)) } }
    if total != records.len() { return Err(B200Error(-1)); }
    Ok((n as u16, shape_kinds.concat()))
}

/// The kind vectors of a mixed-shape prover call, flattened, and the length of its output, after checking that `inputs` holds
/// exactly one input record per shape id (requests for `issue`, show inputs otherwise).
fn mixed_prover_shapes(issue: bool, shape_kinds: &[&[u8]], inputs: &[u8], shape_ids: &[u8]) -> Result<(u16, Vec<u8>, usize), B200Error> {
    let n = shape_kinds.first().map_or(0, |k| k.len());
    if shape_kinds.iter().any(|k| k.len() != n) { return Err(B200Error(-1)); }
    let sizes: Vec<(usize, usize)> = shape_kinds.iter().map(|k| unsafe {
        if issue { (32 * (3 * n + 14), 32 * (2 * n + 9)) }
        else { (32 * afx_show_num_fields(n as u16, k.as_ptr()), 32 * afx_presentation_num_fields(n as u16, k.as_ptr())) }
    }).collect();
    let (mut total_in, mut total_out) = (0usize, 0usize);
    for &s in shape_ids {
        match sizes.get(s as usize) { Some(&(i, o)) => { total_in += i; total_out += o; } None => return Err(B200Error(-1)) }
    }
    if total_in != inputs.len() { return Err(B200Error(-1)); }
    Ok((n as u16, shape_kinds.concat(), total_out))
}

/// Several B200s behind one handle (`afx_multi_*`): the library replicates the issuer context on every listed device, keeps one
/// host thread per device, cuts a batch into contiguous item slices (device k of G takes `[k*N/G, (k+1)*N/G)`) and lets every
/// device write its slice of the verdict array.  This is what `Issuer::verify_batch` binds when the box has more than one GPU.
pub struct B200Multi {
    m: *mut afx_multi,
}

unsafe impl Send for B200Multi {}

impl B200Multi {
    pub fn new(system_parameters: &[u8], issuer_parameters: &[u8; 64], secret_key: Option<&[u8]>, devices: &[i32], max_batch_per_device: usize)
        -> Result<B200Multi, B200Error>
    {
        let mut m: *mut afx_multi = std::ptr::null_mut();
        let (sk, sk_len) = match secret_key { Some(s) => (s.as_ptr(), s.len()), None => (std::ptr::null(), 0) };
        let devs: Vec<c_int> = devices.iter().map(|d| *d as c_int).collect();
        let rc = unsafe {
            afx_multi_create(system_parameters.as_ptr(), system_parameters.len(), issuer_parameters.as_ptr(), sk, sk_len,
                             devs.as_ptr(), devs.len() as c_int, max_batch_per_device, &mut m)
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(B200Multi { m })
    }

    /// Batch `Issuer::verify` over item-major wire bytes, sharded over the devices.
    pub fn verify_presentations_wire(&self, kinds: &[u8], items: &[u8]) -> Result<Vec<u8>, B200Error> {
        let n_fields = unsafe { afx_presentation_num_fields(kinds.len() as u16, kinds.as_ptr()) };
        if n_fields == 0 || items.len() % (n_fields * 32) != 0 { return Err(B200Error(-1)); }
        let count = items.len() / (n_fields * 32);
        let mut verdicts = vec![0u8; count];
        let rc = unsafe {
            afx_multi_verify_presentations_wire(self.m, kinds.len() as u16, kinds.as_ptr(), count, items.as_ptr(), verdicts.as_mut_ptr())
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }

    /// `B200Context::verify_mixed_wire` sharded over the devices: each device buckets its own slice of records.
    pub fn verify_mixed_wire(&self, issuance: bool, shape_kinds: &[&[u8]], records: &[u8], shape_ids: &[u8]) -> Result<Vec<u8>, B200Error> {
        let (n, flat) = mixed_shapes(issuance, shape_kinds, records, shape_ids)?;
        let mut verdicts = vec![0u8; shape_ids.len()];
        let f = if issuance { afx_multi_verify_issuances_mixed_wire } else { afx_multi_verify_presentations_mixed_wire };
        let rc = unsafe { f(self.m, n, flat.as_ptr(), shape_kinds.len(), shape_ids.len(), records.as_ptr(), shape_ids.as_ptr(), verdicts.as_mut_ptr()) };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }

    /// `B200Context::issue_mixed_wire` sharded over the devices: device k issues requests `[k*N/G, (k+1)*N/G)`.
    pub fn issue_mixed_wire(&self, shape_kinds: &[&[u8]], requests: &[u8], shape_ids: &[u8]) -> Result<(Vec<u8>, Vec<u8>), B200Error> {
        let (n, flat, out_len) = mixed_prover_shapes(true, shape_kinds, requests, shape_ids)?;
        let (mut out, mut status) = (vec![0u8; out_len], vec![0u8; shape_ids.len()]);
        let rc = unsafe {
            afx_multi_issue_mixed_wire(self.m, n, flat.as_ptr(), shape_kinds.len(), shape_ids.len(), requests.as_ptr(), shape_ids.as_ptr(),
                                       out.as_mut_ptr(), status.as_mut_ptr())
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok((out, status))
    }

    /// Batch `CredentialIssuance::verify` over item-major wire bytes (`attribute[n], t, U, V, challenge, responses[n+5]` per item).
    pub fn verify_issuances_wire(&self, kinds: &[u8], items: &[u8]) -> Result<Vec<u8>, B200Error> {
        let n_fields = 2 * kinds.len() + 9;
        if items.len() % (n_fields * 32) != 0 { return Err(B200Error(-1)); }
        let count = items.len() / (n_fields * 32);
        let mut verdicts = vec![0u8; count];
        let rc = unsafe {
            afx_multi_verify_issuances_wire(self.m, kinds.len() as u16, kinds.as_ptr(), count, items.as_ptr(), verdicts.as_mut_ptr())
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(verdicts)
    }
}

impl Drop for B200Multi {
    fn drop(&mut self) {
        unsafe { afx_multi_destroy(self.m) }
    }
}

/// Records of several shapes arriving interleaved (`afx_stream_*`; BASELINE configs[4]): each record is bucketed by shape into
/// page-locked buffers and every full bucket is verified asynchronously.  The library writes a record's verdict to the address it
/// was given at `push` whenever that record's bucket completes, so the verdict bytes must not move or be read before `flush`: the
/// stream owns them (a `Vec` allocated once for `max_records`, never grown) and hands them out only from `flush`.
/// The contexts registered with `add_shape` must outlive the stream (`'a`).
pub struct B200Stream<'a> {
    s: *mut afx_stream,
    record_bytes: Vec<usize>,
    verdicts: Vec<u8>,          // len = records pushed since the last flush; capacity fixed at construction
    _contexts: std::marker::PhantomData<&'a B200Context>,
}

impl<'a> B200Stream<'a> {
    /// `max_records`: the most records that will be pushed between two flushes.
    pub fn new(max_records: usize) -> Result<B200Stream<'a>, B200Error> {
        let mut s: *mut afx_stream = std::ptr::null_mut();
        let rc = unsafe { afx_stream_create(&mut s) };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(B200Stream { s, record_bytes: Vec::new(), verdicts: Vec::with_capacity(max_records), _contexts: std::marker::PhantomData })
    }

    /// Registers a shape (presentations of `kinds`, or issuances when `issuance`) verified on `ctx`; returns its shape id.
    pub fn add_shape(&mut self, ctx: &'a B200Context, issuance: bool, kinds: &[u8]) -> Result<u8, B200Error> {
        let (mut id, mut bytes): (c_int, usize) = (0, 0);
        let rc = unsafe { afx_stream_add_shape(self.s, ctx.ctx, issuance as c_int, kinds.len() as u16, kinds.as_ptr(), &mut id, &mut bytes) };
        if rc != 0 { return Err(B200Error(rc)); }
        self.record_bytes.push(bytes);
        Ok(id as u8)
    }

    /// `records`: concatenated records (copied into the stream's buckets before this returns); `offsets[i]` / `shape_ids[i]`: where
    /// record i starts and which registered shape it has.  Returns the position of the first of these records in the verdict
    /// vector `flush` will return.
    pub fn push(&mut self, records: &[u8], offsets: &[u64], shape_ids: &[u8]) -> Result<usize, B200Error> {
        let n = offsets.len();
        if shape_ids.len() != n || self.verdicts.len() + n > self.verdicts.capacity() { return Err(B200Error(-1)); }
        for (o, id) in offsets.iter().zip(shape_ids.iter()) {
            match self.record_bytes.get(*id as usize) {
                Some(len) if (*o as usize).checked_add(*len).map_or(false, |end| end <= records.len()) => {},
                _ => return Err(B200Error(-1)),
            }
        }
        let first = self.verdicts.len();
        self.verdicts.resize(first + n, 0);          // within the capacity: the buffer does not move
        let rc = unsafe {
            afx_stream_push(self.s, records.as_ptr(), offsets.as_ptr(), shape_ids.as_ptr(), n, self.verdicts.as_mut_ptr().add(first))
        };
        if rc != 0 { return Err(B200Error(rc)); }
        Ok(first)
    }

    /// Submits the partly filled buckets, waits for everything in flight and returns the verdicts of every record pushed since the
    /// last flush, in push order (0 = Ok, 1 = VerificationFailure).
    pub fn flush(&mut self) -> Result<Vec<u8>, B200Error> {
        let rc = unsafe { afx_stream_flush(self.s) };
        if rc != 0 { return Err(B200Error(rc)); }
        let cap = self.verdicts.capacity();
        Ok(std::mem::replace(&mut self.verdicts, Vec::with_capacity(cap)))
    }
}

impl<'a> Drop for B200Stream<'a> {
    fn drop(&mut self) {
        unsafe { afx_stream_destroy(self.s) }      // waits for outstanding buckets (they write into self.verdicts) before anything is freed
    }
}
