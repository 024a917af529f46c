/* aeonflux_b200 -- C ABI of the B200 batch engine for aeonflux's issuer hot path.
 *
 * The reference (isislovecruft/aeonflux, Rust) has no FFI layer; its boundary for this path is the method surface
 *     Issuer::verify(&self, &ProofOfValidCredential)            src/issuer.rs:141-147
 *     Issuer::issue(&self, CredentialRequest, &mut rng)         src/issuer.rs:111-124
 *     CredentialIssuance::verify(self, &SystemParameters, &IssuerParameters)   src/issuer.rs:48-57
 * A batch entry point added beside each of those (Issuer::verify_batch, Issuer::issue_batch,
 * CredentialIssuance::verify_batch -- see INTEGRATION.md for the Rust shim) flattens its arguments to the plain
 * buffers below and binds exactly these symbols.  Plain pointers and sizes only; the caller owns every buffer; the
 * library copies what it keeps.  All functions are synchronous unless they take a stream.  A context owns one workspace and
 * its CUDA streams, so calls on ONE context serialise on an internal lock (safe from several threads, never concurrent);
 * replicate the context per GPU and per concurrent caller -- or use the afx_multi_* entry points, which do that.
 *
 * Batch data is struct-of-arrays: "field f" is an array [count][32 bytes].  A 32-byte word is either a canonical
 * little-endian Scalar or a CompressedRistretto -- the same encodings the reference's to_bytes() methods emit
 * (src/parameters.rs:155-184, src/amacs.rs:110-125).
 *
 * Presentation fields for attribute kinds k[0..n) (0 = revealed scalar, 1 = hidden scalar, 2 = revealed point,
 * 3 = hidden/encrypted point), h_s = #hidden scalars:
 *     challenge, responses[3 + h_s], C_x_0, C_x_1, C_V, C_y[n],
 *     revealed value of each kind-0 / kind-2 attribute in index order,
 *     then per kind-3 attribute in index order: enc_challenge, enc_responses[6], pk, E1, E2, C_y_1, C_y_2, C_y_3, C_y_2'
 * (struct fields of ProofOfValidCredential, src/nizk/presentation.rs:118-127, and ProofOfEncryption,
 *  src/nizk/encryption.rs:32-41; hidden_scalar_indices and the enc proofs' indices are implied by kinds).
 *
 * Issuance fields for request kinds k[0..n) (0 = scalar attribute, 2 = point attribute -- a revealed point or the M1 of a
 * plaintext, src/amacs.rs:224-244):
 *     attribute[n], t, U, V, challenge, responses[n + 5]
 * (CredentialIssuance = ProofOfIssuance(CompactProof) + AnonymousCredential{amac:{t,U,V}, attributes}, src/issuer.rs:42-45).
 *
 * Verdicts: 0 = Ok(()), 1 = Err(CredentialError::VerificationFailure) -- the only error these verify paths can return
 * (src/errors.rs:152-156).  Byte strings the Rust types could never hold (undecodable point, scalar >= l) also give 1.
 */
#ifndef AEONFLUX_B200_H
#define AEONFLUX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct afx_ctx afx_ctx;

enum { AFX_OK = 0, AFX_ERR_ARG = -1, AFX_ERR_ENCODING = -2, AFX_ERR_CUDA = -3, AFX_ERR_ALLOC = -4, AFX_ERR_SHAPE = -5, AFX_ERR_NO_SECRET = -6 };
enum { AFX_KIND_PUBLIC_SCALAR = 0, AFX_KIND_SECRET_SCALAR = 1, AFX_KIND_PUBLIC_POINT = 2, AFX_KIND_SECRET_POINT = 3 };

/* Replaces Issuer::from_bytes / holding an `Issuer` (src/issuer.rs:61-65,152-159).
 *   sysparams  = SystemParameters::to_bytes()   (src/parameters.rs:155-184)
 *   issuer_pub = C_W || I                        (the 64 bytes src/issuer.rs:155,163 reserve for IssuerParameters)
 *   secret     = amacs::SecretKey::to_bytes()    (src/amacs.rs:110-125); NULL for a user-side context, which runs
 *                afx_verify_issuances* and afx_show* but neither afx_verify_presentations* nor afx_issue* (AFX_ERR_NO_SECRET)
 *   device     = CUDA device ordinal
 * Validates every encoding (AFX_ERR_ENCODING), builds the per-issuer constant tables and transcript midstates on the
 * device (about 3.3 MB of device memory per generator -- 66 MB for 4 attributes, 145 MB for 16 -- or 0.25 MB per generator
 * beyond a 200 MB budget or when that allocation fails).  max_batch = number of items one device pass handles (the workspace is sized for it); host calls with a larger
 * `count` are split into passes of max_batch items and pipelined (copy of pass i+1 under the kernels of pass i), the *_device
 * calls take at most max_batch items. */
int afx_ctx_create(const uint8_t* sysparams, size_t sysparams_len, const uint8_t issuer_pub[64], const uint8_t* secret,
                   size_t secret_len, int device, size_t max_batch, afx_ctx** out);

/* Drop for Issuer: zeroizes host and device copies of the secret key (src/amacs.rs:64-82) and frees everything. */
void afx_ctx_destroy(afx_ctx* ctx);

typedef struct {
    uint16_t n_attrs;
    const uint8_t* kinds;          /* [n_attrs] AFX_KIND_* ; identical for all items of the call */
    size_t count;
    const uint8_t* const* fields;  /* [n_fields] pointers, each to [count][32] bytes */
    size_t n_fields;               /* must equal afx_presentation_num_fields(n_attrs, kinds) */
} afx_presentation_batch;

typedef struct {                   /* optional parity hooks (debug-transcript equivalent, SURVEY section 5) */
    uint8_t* Z;                    /* [count][32]              recomputed Z, compressed; nullable */
    uint8_t* commitments;          /* [n_commitments][count][32] recomputed blinding commitments, constraint order; nullable */
    uint8_t* challenges;           /* [n_proofs][count][32]    recomputed challenge scalars; nullable */
    uint32_t* status;              /* [count] internal failure bits (1 bad point, 2 bad scalar, 4 identity, 8 challenge); nullable */
} afx_debug_dump;

size_t afx_presentation_num_fields(uint16_t n_attrs, const uint8_t* kinds);
size_t afx_presentation_num_commitments(uint16_t n_attrs, const uint8_t* kinds);
size_t afx_presentation_num_proofs(uint16_t n_attrs, const uint8_t* kinds);

/* Batch Issuer::verify (src/issuer.rs:141-147).  Host buffers in, host verdicts out. */
int afx_verify_presentations(afx_ctx* ctx, const afx_presentation_batch* batch, uint8_t* verdicts, afx_debug_dump* dbg);

/* Same, with the batch already resident on the context's device: fields_dev = [n_fields][count][32] contiguous device
 * memory, verdicts_dev = [count] device bytes; enqueued on `stream` (a cudaStream_t; NULL = default stream) without
 * synchronizing.  This is what bench.py times for the kernel-only figure. */
int afx_verify_presentations_device(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const void* fields_dev,
                                    void* verdicts_dev, void* stream);

typedef struct {
    uint16_t n_attrs;
    const uint8_t* kinds;          /* [n_attrs] 0 = scalar attribute, 2 = point attribute */
    size_t count;
    const uint8_t* const* fields;  /* [2*n_attrs + 9] pointers: attribute[n], t, U, V, challenge, responses[n+5] */
    size_t n_fields;
} afx_issuance_batch;

/* Batch CredentialIssuance::verify (src/issuer.rs:48-57 -> src/nizk/issuance.rs:132-218).  Needs no secret key. */
int afx_verify_issuances(afx_ctx* ctx, const afx_issuance_batch* batch, uint8_t* verdicts, afx_debug_dump* dbg);

/* Asynchronous host calls for a caller that streams batches (SURVEY 8b "optional async/stream variant"): submit enqueues the
 * copy, the kernels and the verdict read-back of one pass (count <= max_batch) and returns a ticket; afx_wait(ticket) blocks until
 * the verdicts are in the array given at submission.  Up to two submissions may be outstanding per context, so the copy of one
 * overlaps the kernels of the other; a third submit, or any synchronous call, while submissions are outstanding returns
 * AFX_ERR_ARG.  The workspace is (re)sized only while nothing is in flight: a submit whose shape needs more of any workspace
 * array than the outstanding submission was sized for also returns AFX_ERR_ARG -- wait, then submit (streams of one shape, or of
 * shapes submitted largest first, never hit this).  The field buffers and the verdict array must stay valid until afx_wait returns. */
int afx_verify_presentations_submit(afx_ctx* ctx, const afx_presentation_batch* batch, uint8_t* verdicts, uint64_t* ticket);
int afx_verify_issuances_submit(afx_ctx* ctx, const afx_issuance_batch* batch, uint8_t* verdicts, uint64_t* ticket);
int afx_wait(afx_ctx* ctx, uint64_t ticket);
/* The same for item-major wire bytes ([count][n_fields][32], see the *_wire calls below): one host-to-device copy per pass. */
int afx_verify_presentations_wire_submit(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                                         uint8_t* verdicts, uint64_t* ticket);
int afx_verify_issuances_wire_submit(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                                     uint8_t* verdicts, uint64_t* ticket);

/* Page-locked host memory for batch buffers (optional: every entry point accepts any host memory).  A host-to-device copy
 * from page-locked memory runs at the full bus rate and asynchronously; from pageable memory the driver stages it at a
 * fraction of that rate on the calling thread, which exposes the copy of every pass of a multi-pass call (S16: 300 MB per
 * 65,536 items).  A shim that flattens its presentations into struct-of-arrays buffers should build them here.  The memory is
 * not tied to a context; free it with afx_host_free (NULL is ignored). */
int afx_host_alloc(void** out, size_t bytes);
void afx_host_free(void* p);

/* BatchableProof form (SURVEY 8f rank 2; opt-in, NOT the reference's encoding).  The reference proves with zkp's CompactProof
 * (challenge + responses); its authors left zkp's BatchVerifier commented out (src/nizk/presentation.rs:33-34), which needs the
 * other zkp encoding, BatchableProof = blinding commitments + responses.  These entry points verify presentations whose proofs
 * travel in that form: the field layout is the presentation layout above with every challenge word replaced by that proof's
 * commitments in constraint order (main proof: Z, C_x_1, then the C_y constraints; proof of encryption: pk, C_y_1-E2, C_y_2',
 * E1, C_y_3), i.e. afx_batchable_num_fields() words.  Semantics = zkp 0.7 Verifier::verify_batchable per proof: commitments are
 * validated (identity / undecodable => reject) and absorbed, the challenge is derived from the transcript, and every constraint
 * must satisfy sum resp_k*P_k - c*LHS == commitment.  The aMAC recomputation of Z is unchanged (constant schedule).
 *   afx_verify_presentations_batchable      checks every constraint of every item exactly (one MSM per constraint);
 *   afx_verify_presentations_batchable_rlc  checks one random linear combination of all constraints of all items of a chunk as
 *       a single Pippenger multiscalar multiplication.  A chunk whose combination does not vanish is bisected: its halves get fresh
 *       coefficients and their own pass, down to leaves of 1,024 items, which are re-verified exactly; after 16 failing nodes, or
 *       when the suspect leaves cover more than half the chunk, the rest is checked exactly.  So the verdicts are the exact ones
 *       except with probability ~2^-120 per pass; one bad item in a chunk costs a few small passes and one leaf, many bad items
 *       cost the exact check plus a bounded number of wasted passes (fast when rejects are rare).
 *       Coefficients: 127 bits each, derived from `seed` AND a nonce the library draws from the operating system for every call,
 *       so they are unpredictable to the provers even if a caller reuses or mis-generates its seed (pass 32 zero bytes if you have
 *       nothing better; the seed only adds entropy).
 * The same two calls exist for issuances (afx_verify_issuances_batchable{,_rlc}: the BatchVerifier the reference left commented out
 * at src/nizk/issuance.rs:21-22): fields attribute[n], t, U, V, commitments[3] (constraint order C_W, I, V), responses[n + 5],
 * i.e. afx_issuance_batchable_num_fields(n) = 2n + 11 words. */
size_t afx_batchable_num_fields(uint16_t n_attrs, const uint8_t* kinds);
int afx_verify_presentations_batchable(afx_ctx* ctx, const afx_presentation_batch* batch, uint8_t* verdicts, afx_debug_dump* dbg);
/* exact_chunks (nullable): how many chunks of max_batch items held a combination that did not vanish (and needed exact work). */
int afx_verify_presentations_batchable_rlc(afx_ctx* ctx, const afx_presentation_batch* batch, const uint8_t seed[32], uint8_t* verdicts,
                                           uint32_t* exact_chunks);
size_t afx_issuance_batchable_num_fields(uint16_t n_attrs);
int afx_verify_issuances_batchable(afx_ctx* ctx, const afx_issuance_batch* batch, uint8_t* verdicts, afx_debug_dump* dbg);
int afx_verify_issuances_batchable_rlc(afx_ctx* ctx, const afx_issuance_batch* batch, const uint8_t seed[32], uint8_t* verdicts,
                                       uint32_t* exact_chunks);
/* Cumulative counters of the *_rlc calls on this context: combination passes run, items re-verified exactly. */
int afx_get_rlc_stats(afx_ctx* ctx, uint64_t* rlc_passes, uint64_t* exact_items);

/* Item-major ("wire") variants.  The reference defines no serialization for a presentation or an issuance
 * (src/nizk/presentation.rs:117 "XXX"; SURVEY 8f rank 1); the natural one is the concatenation of the item's 32-byte words in
 * the field order documented above, and a batch is the concatenation of its items:
 *     items = [count][n_fields][32] contiguous bytes.
 * These take such a blob as received -- one host-to-device copy, no scatter into per-field arrays; the kernels read the
 * item-major layout directly (32 contiguous bytes per word either way).  Verdicts and chunking/pipelining as above. */
int afx_verify_presentations_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                                  uint8_t* verdicts);
int afx_verify_issuances_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                              uint8_t* verdicts);

/* Wire records of SEVERAL shapes of the context's issuer in one call: the batch form of Issuer::verify over whatever presentations
 * the issuer receives, each user having chosen which attributes to hide (src/credential.rs:53-97), or of CredentialIssuance::verify
 * over issuances of several request kinds.
 *   shape_kinds = [n_shapes][n_attrs] the kind vectors of the call, 1 <= n_shapes <= 255 (a vector may be listed twice)
 *   shape_ids   = [count] shape of each record, < n_shapes
 *   records     = the records concatenated in order, record i being its shape's item in the *_wire layout above:
 *                 afx_presentation_num_fields(n_attrs, kinds) * 32 bytes, or (2 * n_attrs + 9) * 32 bytes for an issuance
 * verdicts[i] is what afx_verify_{presentations,issuances}_wire gives record i alone under its shape.  Checked before any device work
 * and before anything is written to verdicts: AFX_ERR_ARG for n_shapes out of range, a shape id >= n_shapes, a null pointer with
 * count > 0 (shape_kinds: always) or submissions outstanding; AFX_ERR_SHAPE for a kind vector the issuer cannot verify;
 * AFX_ERR_NO_SECRET for presentations on a context without the issuer secret.  count = 0 is AFX_OK.
 * The call works in passes of at most max_batch consecutive records of any mix.  Each pass's bytes are copied to the device once,
 * as received (the copy of pass i + 1 under the kernels of pass i); a kernel copies every record into the item-major bucket of its
 * shape, keeping the record order, the verify program of each shape present runs over its bucket, and the verdicts are put back in
 * record order before one copy to the host.  The host reads only the shape ids.  Device memory: the workspace of the largest shape
 * of the call at max_batch items, plus three [max_batch][largest record] buffers (the pass as received, twice, and the buckets),
 * plus about 2 * (6 + (4 * n_shapes + 16) / 256) bytes of bucketing arrays per record of max_batch. */
int afx_verify_presentations_mixed_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                                        const uint8_t* records, const uint8_t* shape_ids, uint8_t* verdicts);
int afx_verify_issuances_mixed_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                                    const uint8_t* records, const uint8_t* shape_ids, uint8_t* verdicts);

/* Same as afx_verify_issuances with the batch resident on the device ([2*n_attrs + 9][count][32] contiguous). */
int afx_verify_issuances_device(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const void* fields_dev,
                                void* verdicts_dev, void* stream);

/* Batch Issuer::issue (src/issuer.rs:111-124 = Amac::tag, src/amacs.rs:276-294, + ProofOfIssuance::prove,
 * src/nizk/issuance.rs:40-129).  The reference draws t, U and the proof's blindings from the caller's rng
 * (`&mut rng` argument / zkp's TranscriptRng); here the caller passes that rng output explicitly, 64 bytes per random
 * value exactly as Scalar::random / RistrettoPoint::random consume them, so that the result is a deterministic function
 * of its inputs (and byte-identical to the reference given the same rng bytes).
 *
 * Request fields for request kinds k[0..n) (0 = scalar attribute, 2 = point attribute -- a revealed point or the M1 of a
 * plaintext): attribute[n], then two 32-byte words (low, high half of the 64 rng bytes) for each of
 *     t, U, blinding[n + 5]   (blindings in witness order w, w', x_0, x_1, y[n], "1"; src/nizk/issuance.rs:52-68)
 * i.e. 3*n + 14 fields.  Output fields: t, U, V, challenge, responses[n + 5]  (n + 9 fields, each [count][32]) -- together
 * with the request's attribute fields this is exactly the afx_issuance_batch layout, so an issued batch can be handed to
 * afx_verify_issuances unchanged.  status: 0 = Ok, 1 = the request holds bytes the Rust types could never hold
 * (undecodable point / scalar >= l); its output words are all-zero.  An attribute count different from the issuer's is
 * AFX_ERR_SHAPE for the whole call (CredentialError::MacCreation, src/amacs.rs:285-287).
 * Every scalar on this path is secret (key material, blindings, t): all ladders run a constant schedule with
 * constant-address table scans (dalek's constant-time `*` and multiscalar_mul). */
typedef struct {
    uint16_t n_attrs;
    const uint8_t* kinds;          /* [n_attrs] 0 = scalar attribute, 2 = point attribute */
    size_t count;
    const uint8_t* const* fields;  /* [3*n_attrs + 14] pointers, each to [count][32] bytes */
    size_t n_fields;               /* must equal afx_request_num_fields(n_attrs) */
} afx_request_batch;

typedef struct {
    uint8_t* const* fields;        /* [n_attrs + 9] pointers, each to [count][32] bytes: t, U, V, challenge, responses[n+5] */
    size_t n_fields;
} afx_issuance_out;

size_t afx_request_num_fields(uint16_t n_attrs);
/* dbg (nullable): commitments = the three blinding commitments [3][count][32]; status. */
int afx_issue(afx_ctx* ctx, const afx_request_batch* batch, const afx_issuance_out* out, uint8_t* status, afx_debug_dump* dbg);
/* Device-resident variant: fields_dev = [3*n_attrs + 14][count][32], out_dev = [n_attrs + 9][count][32], status_dev = [count]. */
int afx_issue_device(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const void* fields_dev, void* out_dev,
                     void* status_dev, void* stream);

/* Item-major ("wire") form of afx_issue: a CredentialRequest (src/user.rs:137-139) travels as the concatenation of its words --
 * attribute[n] followed by the rng halves, 3n + 14 words -- and a batch as the concatenation of its requests,
 *     requests = [count][3n + 14][32];   issuances = [count][2n + 9][32]: attribute[n] (echoed), t, U, V, challenge, responses[n + 5]
 * i.e. each issuance comes back in exactly the layout afx_verify_issuances_wire takes.  One copy each way per pass of max_batch
 * items.  status as afx_issue (a malformed request gives status 1 and an all-zero issuance). */
int afx_issue_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* requests, uint8_t* issuances,
                   uint8_t* status);

/* Batch AnonymousCredential::show (src/credential.rs:37-46 = ProofOfValidCredential::prove, src/nizk/presentation.rs:139-321, plus
 * one ProofOfEncryption::prove, src/nizk/encryption.rs:58-142, with Keypair::encrypt, src/symmetric.rs:252-261, per hidden
 * plaintext attribute).  The USER-side batch operation (SURVEY 8f rank 3): it needs no issuer secret, so a context created with
 * secret = NULL suffices.  As with afx_issue the rng output (z and the blindings) is passed explicitly, 64 bytes per value.
 *
 * kinds = the attribute kinds of the presentation to produce (AFX_KIND_*), h_s = #hidden scalars, h_p = #hidden plaintexts.
 * Input fields:  t, U, V   (the credential's aMAC, src/amacs.rs:248-252),
 *                per attribute in index order: the scalar m_i (kinds 0, 1) | the point M_i (kind 2; for a revealed plaintext its
 *                M1) | the plaintext M1, M2, m3 (kind 3; src/symmetric.rs:89-96),
 *                a, a0, a1, pk of the symmetric keypair (src/symmetric.rs:74-79) -- present only when h_p > 0,
 *                then (lo, hi) 32-byte halves of the rng bytes of: z, the 3 + h_s blindings of the presentation proof (witness
 *                order z, z_0, t, m...), and 6 blindings per hidden plaintext (a, a0, a1, m3, z, z1).
 * Output fields: exactly the presentation layout documented at the top of this header, so the result can be handed to
 * afx_verify_presentations unchanged.  status: 0 = Ok, 1 = undecodable point / non-canonical scalar in the input (all-zero output). */
typedef afx_request_batch afx_show_batch;
typedef afx_issuance_out afx_presentation_out;
size_t afx_show_num_fields(uint16_t n_attrs, const uint8_t* kinds);
int afx_show(afx_ctx* ctx, const afx_show_batch* batch, const afx_presentation_out* out, uint8_t* status, afx_debug_dump* dbg);
int afx_show_device(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const void* fields_dev, void* out_dev,
                    void* status_dev, void* stream);
/* Item-major form: inputs = [count][afx_show_num_fields][32], presentations = [count][afx_presentation_num_fields][32] -- what
 * afx_verify_presentations_wire takes. */
int afx_show_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* inputs, uint8_t* presentations,
                  uint8_t* status);

/* Issue or show over records of SEVERAL shapes of the context's issuer in one call, bucketed on the device: Issuer::issue over
 * CredentialRequests of several request kinds, or AnonymousCredential::show for users who each chose which attributes to hide.
 *   shape_kinds = [n_shapes][n_attrs] the kind vectors of the call, 1 <= n_shapes <= 255 (a vector may be listed twice)
 *   shape_ids   = [count] shape of each record, < n_shapes
 *   requests / inputs = the input records concatenated in order, record i being one item of its shape as afx_issue_wire /
 *                 afx_show_wire take it: (3 * n_attrs + 14) * 32 bytes for every request kind vector, or
 *                 afx_show_num_fields(n_attrs, kinds) * 32 bytes
 *   issuances / presentations = the output records concatenated in the same order, record i being what the per-shape call writes
 *                 for it: (2 * n_attrs + 9) * 32 bytes (the attributes echoed), or afx_presentation_num_fields(n_attrs, kinds) * 32
 *                 bytes.  So the outputs, with the same shape_kinds and shape_ids, are exactly the records argument of
 *                 afx_verify_issuances_mixed_wire / afx_verify_presentations_mixed_wire.
 * Output bytes and status[i] are byte-identical to the per-shape *_wire call on record i: status 1 and an all-zero output record for
 * a malformed input.  Checked before any device work and before anything is written to the outputs or status: AFX_ERR_ARG for
 * n_shapes out of range, a shape id >= n_shapes, a null pointer with count > 0 (shape_kinds: always) or submissions outstanding;
 * AFX_ERR_SHAPE for a kind vector that cannot be issued (a request kind other than 0 or 2, or an attribute count other than the
 * issuer's) or shown; AFX_ERR_NO_SECRET for issuing on a context without the issuer secret (showing needs none).  count = 0 is AFX_OK.
 * The call works in passes of at most max_batch consecutive records of any mix: the pass's inputs are copied to the device once, as
 * received; a kernel copies every record into the item-major bucket of its shape; the prover program of each shape present writes
 * its outputs into a region of its own; a second kernel puts the outputs and status bytes back in record order.  The outputs go
 * straight into the caller's buffer in one copy; the status bytes go through the library's page-locked staging, so the status array
 * need not be page-locked.  With the inputs and outputs in page-locked memory the copy in of pass i + 1 and the copy out of pass
 * i - 1 run under the kernels of pass i.  The library keeps no host copy of the inputs, and wipes the device buffers that held them
 * (request rng bytes, the credential's t, hidden attributes, keypairs) before it returns.  Device memory: the workspace of the
 * largest shape of the call at max_batch items, plus three [max_batch][largest input record] buffers (the pass as received, twice, and the buckets), two
 * [max_batch][largest output record] buffers (the outputs in record order, double-buffered), and about
 * 2 * (6 + (4 * n_shapes + 16) / 256) bytes of bucketing arrays per record of max_batch. */
int afx_issue_mixed_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                         const uint8_t* requests, const uint8_t* shape_ids, uint8_t* issuances, uint8_t* status);
int afx_show_mixed_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                        const uint8_t* inputs, const uint8_t* shape_ids, uint8_t* presentations, uint8_t* status);

/* Issue and show in BatchableProof form: zkp 0.7's prove_batchable instead of prove_compact.  The prover is the same (same inputs,
 * blindings, commitments and transcripts, hence the same challenges and responses); only its return value differs: the blinding
 * commitments in place of each challenge.  The outputs are exactly what the BatchableProof verifiers above take:
 *   afx_issue_batchable: output fields t, U, V, commitments[3] (constraint order C_W, I, V), responses[n + 5], i.e. n + 11 fields,
 *       which with the request's attribute[n] in front is the afx_issuance_batchable_num_fields(n) = 2n + 11 layout of
 *       afx_verify_issuances_batchable{,_rlc}.  Needs the issuer secret, like afx_issue.
 *   afx_show_batchable: output fields in the afx_batchable_num_fields(n, kinds) layout of afx_verify_presentations_batchable{,_rlc}
 *       (the main proof's challenge replaced by its commitments Z, C_x_1, then the C_y constraints; each proof of encryption's by
 *       pk, C_y_1-E2, C_y_2', E1, C_y_3).  Needs no issuer secret, like afx_show.
 * Inputs, status, chunking beyond max_batch, dbg and the *_device forms (count <= max_batch, out_dev = [n_out][count][32]) are those
 * of afx_issue / afx_show.  A commitment that is the identity (possible only when blindings are zero) is written as its encoding,
 * 32 zero bytes, with status 0: zkp's prover appends commitments without validating them.  zkp's verify_batchable, and the
 * afx_verify_*_batchable calls, reject such a proof.  There is no linked BatchableProof statement. */
int afx_issue_batchable(afx_ctx* ctx, const afx_request_batch* batch, const afx_issuance_out* out, uint8_t* status, afx_debug_dump* dbg);
int afx_issue_batchable_device(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const void* fields_dev, void* out_dev,
                               void* status_dev, void* stream);
int afx_show_batchable(afx_ctx* ctx, const afx_show_batch* batch, const afx_presentation_out* out, uint8_t* status, afx_debug_dump* dbg);
int afx_show_batchable_device(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const void* fields_dev, void* out_dev,
                              void* status_dev, void* stream);

/* Symmetric encryption of attributes: Plaintext::from(&[u8; 30]) (src/symmetric.rs:135-143 -> src/encoding.rs:56-70),
 * Keypair::encrypt (src/symmetric.rs:252-261) and Keypair::decrypt (src/symmetric.rs:273-289), in batch form.  User-side and
 * key-holder operations: they need no issuer secret (a context created with secret = NULL suffices) and do not use the system
 * parameters.  Calls lock the context like every other call.
 *   data       = [count][30] bytes, the attribute's plaintext bytes
 *   plaintext  = the words M1, M2, m3 (src/symmetric.rs:89-96): exactly the three words a kind-3 attribute takes in afx_show's input
 *   ciphertext = the words E1, E2 (src/symmetric.rs:252-261): words 8 and 9 of a presentation's 14-word proof-of-encryption block
 *   keypair    = a || a0 || a1, 96 bytes of canonical scalars (src/symmetric.rs:74-79): the first 96 bytes of the 128-byte keypair
 *                afx_show takes.  A scalar >= l is AFX_ERR_ENCODING, and nothing is written.
 * Host calls are item-major (plaintexts [count][3][32], ciphertexts [count][2][32]) and run in passes of max_batch items.  The
 * *_device calls take struct-of-arrays device memory (plaintexts [3][count][32], ciphertexts [2][count][32]; data [count][30]),
 * count <= max_batch, and are enqueued on `stream` (a cudaStream_t; NULL = default stream) without synchronizing, so the rows
 * afx_encode_plaintexts_device writes can be handed to afx_show_device as they are.
 * status: 0 = Ok, 1 = the item's output words are all zero and:
 *   encode:  none of the 8,192 candidate encodings of M1 decodes (the reference panics; no such input is known);
 *   encrypt: M1 or M2 does not decode, or m3 is not canonical;
 *   decrypt: E1 or E2 does not decode, or (a0 + a1*m3')*M2' != E1 (CredentialError::UndecryptableAttribute, src/errors.rs).
 * Timing: encrypt and decrypt run constant-schedule ladders with constant-address table scans (the keypair, m3 and the plaintext are
 * secrets); the device copy of the keypair, the scalars derived from it and decrypt's ladder tables are zeroed on the stream at the
 * end of every pass.  Encode runs in variable time, in the number of candidates tried, as the reference's loop does. */
int afx_encode_plaintexts(afx_ctx* ctx, size_t count, const uint8_t* data, uint8_t* plaintexts, uint8_t* status);
int afx_encrypt(afx_ctx* ctx, const uint8_t keypair[96], size_t count, const uint8_t* plaintexts, uint8_t* ciphertexts, uint8_t* status);
/* plaintexts (nullable): the Plaintext (M1', M2', m3') the reference returns. */
int afx_decrypt(afx_ctx* ctx, const uint8_t keypair[96], size_t count, const uint8_t* ciphertexts, uint8_t* data, uint8_t* plaintexts,
                uint8_t* status);
int afx_encode_plaintexts_device(afx_ctx* ctx, size_t count, const void* data_dev, void* plaintexts_dev, void* status_dev, void* stream);
int afx_encrypt_device(afx_ctx* ctx, const uint8_t keypair[96], size_t count, const void* plaintexts_dev, void* ciphertexts_dev,
                       void* status_dev, void* stream);
int afx_decrypt_device(afx_ctx* ctx, const uint8_t keypair[96], size_t count, const void* ciphertexts_dev, void* data_dev,
                       void* plaintexts_dev, void* status_dev, void* stream);

/* Batch Keypair::derive (src/symmetric.rs:197-215): from each 64-byte master secret,
 *     a = SHA-512(master_secret) mod l,  a0 = SHA-512(a) mod l,  a1 = SHA-512(a0) mod l,  pk = a*G_a + a0*G_a0 + a1*G_a1
 * (wide reductions; G_a, G_a0, G_a1 of the context's SystemParameters, so the same master secret gives different keypairs under
 * different issuers).  Keypair::generate (src/symmetric.rs:227-241) is this call applied to 64 bytes of rng output: as with
 * afx_issue and afx_show the caller supplies the rng bytes, and they are the master secret generate returns.  The call needs no
 * issuer secret (a context created with secret = NULL suffices).  Every 64-byte string derives a keypair: there is no status.
 *   master_secrets = [count][64] bytes
 *   keypairs       = [count][128] bytes a || a0 || a1 || pk: exactly the keypair afx_show takes, whose first 96 bytes are the keypair
 *                    afx_encrypt and afx_decrypt take.  Runs in passes of max_batch items.
 * The device form takes device memory: master_secrets_dev = [count][64], keypairs_dev = [4][count][32], the rows a, a0, a1, pk --
 * the four keypair rows of afx_show_device's input, so they can be handed over without a host round trip.  count <= max_batch;
 * enqueued on `stream` (a cudaStream_t; NULL = default stream) without synchronizing.
 * Timing: the hashes run one thread per item with no branch or address depending on the master secret, and pk is a comb over the
 * three generators with constant-address table scans.  The device copies of the master secrets and of a, a0, a1 the call makes are
 * zeroed on the stream at the end of every pass. */
int afx_derive_keypairs(afx_ctx* ctx, size_t count, const uint8_t* master_secrets, uint8_t* keypairs);
int afx_derive_keypairs_device(afx_ctx* ctx, size_t count, const void* master_secrets_dev, void* keypairs_dev, void* stream);

/* Linked presentations (opt-in; NOT the reference's protocol but the fix its authors left as a TODO: README.md:119-122,
 * src/nizk/presentation.rs:292 "don't we also need DLEQ between the plaintext here and that in the commitments above?").  In the
 * reference nothing ties the proof of encryption's commitment C_y_1 = z*G_y[0] + M1 to the credential proof's C_y[i] = z*G_y[i] + M1:
 * a prover can present a valid credential and attach the encryption of ANOTHER plaintext, and Issuer::verify accepts.  The linked
 * statement adds to the credential proof, per hidden plaintext attribute at index i > 0, the allocated points G_y[i] - G_y[0] (label
 * "G_y-G_y_1") and C_y[i] - C_y_1 (label "C_y-C_y_1") -- after the G_m points, before Z -- and the constraint
 *     C_y[i] - C_y_1 = z * (G_y[i] - G_y[0])        (a DLEQ with Z = z*I: the same z, hence the same M1)
 * after the C_y constraints; at index 0 both commitments use G_y[0] and the two wire words must be equal.  The wire layout is
 * unchanged (only challenge and responses differ), so afx_show_linked's output has the presentation layout and
 * afx_verify_presentations_linked takes it; a presentation made by afx_show / the reference fails the linked verifier and vice versa
 * (different transcripts), except for shapes without a hidden plaintext at an index > 0.  dbg->commitments then holds
 * afx_presentation_linked_num_commitments() rows (the link constraints follow the C_y constraints of the main proof). */
size_t afx_presentation_linked_num_commitments(uint16_t n_attrs, const uint8_t* kinds);
int afx_verify_presentations_linked(afx_ctx* ctx, const afx_presentation_batch* batch, uint8_t* verdicts, afx_debug_dump* dbg);
int afx_verify_presentations_linked_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                                         uint8_t* verdicts);
int afx_show_linked(afx_ctx* ctx, const afx_show_batch* batch, const afx_presentation_out* out, uint8_t* status, afx_debug_dump* dbg);
int afx_show_linked_wire(afx_ctx* ctx, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* inputs,
                         uint8_t* presentations, uint8_t* status);

/* Several B200s behind one handle -- the `devices[], n_devices` form of SURVEY 8b, so that a caller (the Rust shim's
 * Issuer::verify_batch) gets the whole box from one call and builds no threads of its own.  afx_multi_create replicates the
 * issuer context on every listed device (the same arguments as afx_ctx_create; max_batch is per device) and starts one host
 * thread per device.  A batch call cuts the batch into contiguous item slices -- device k of G takes [k*N/G, (k+1)*N/G), SURVEY
 * 8e -- runs the single-device entry point on each slice concurrently (a slice longer than max_batch is pipelined in passes, as
 * there), and every device writes its slice of the caller's verdict array: no collective, nothing but the verdicts is gathered.
 * Results are identical to the single-device call on the whole batch.  Calls on one handle serialise.
 * afx_multi_ctx(m, k) is device k's context (owned by the handle) for the per-device calls that have no multi form. */
typedef struct afx_multi afx_multi;
int afx_multi_create(const uint8_t* sysparams, size_t sysparams_len, const uint8_t issuer_pub[64], const uint8_t* secret,
                     size_t secret_len, const int* devices, int n_devices, size_t max_batch, afx_multi** out);
void afx_multi_destroy(afx_multi* m);
int afx_multi_num_devices(const afx_multi* m);
afx_ctx* afx_multi_ctx(afx_multi* m, int k);
int afx_multi_verify_presentations(afx_multi* m, const afx_presentation_batch* batch, uint8_t* verdicts);
int afx_multi_verify_presentations_wire(afx_multi* m, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                                        uint8_t* verdicts);
int afx_multi_verify_issuances(afx_multi* m, const afx_issuance_batch* batch, uint8_t* verdicts);
int afx_multi_verify_issuances_wire(afx_multi* m, uint16_t n_attrs, const uint8_t* kinds, size_t count, const uint8_t* items,
                                    uint8_t* verdicts);
/* The mixed-shape calls across the devices: contiguous record slices as above, each device bucketing its own slice. */
int afx_multi_verify_presentations_mixed_wire(afx_multi* m, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                                              const uint8_t* records, const uint8_t* shape_ids, uint8_t* verdicts);
int afx_multi_verify_issuances_mixed_wire(afx_multi* m, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                                          const uint8_t* records, const uint8_t* shape_ids, uint8_t* verdicts);
int afx_multi_issue(afx_multi* m, const afx_request_batch* batch, const afx_issuance_out* out, uint8_t* status);
/* afx_issue_mixed_wire across the devices: device k issues records [k*N/G, (k+1)*N/G) and writes that slice of issuances and status
 * (requests and issuances have one length whatever the request kinds). */
int afx_multi_issue_mixed_wire(afx_multi* m, uint16_t n_attrs, const uint8_t* shape_kinds, size_t n_shapes, size_t count,
                               const uint8_t* requests, const uint8_t* shape_ids, uint8_t* issuances, uint8_t* status);

/* Streamed verification of MIXED shapes (BASELINE configs[4]; SURVEY 8d config 5: "bucketed by shape into chunks").  A stream is a
 * sequence of records of several registered shapes, each record the item-major wire bytes of one presentation (issuance = 1: of
 * one issuance).  Register every shape with the context that verifies it (shapes with different attribute counts belong to
 * different issuers, hence different contexts; max_batch of the context = the bucket size; give each shape its own context for
 * full overlap -- shapes sharing one are still correct but take turns).  afx_stream_push takes `n` records: record i is
 * record_bytes(shape_ids[i]) bytes at records + offsets[i]; it is copied into the page-locked bucket of its shape, and a full
 * bucket is submitted asynchronously (afx_*_wire_submit) while another of the shape's three buckets fills, so bucketing, copies and kernels
 * overlap (the first buckets after a flush are submitted at 1/8, 1/4, 1/2 of the bucket size so that the device starts early).  verdicts[i] is written when the record's bucket retires -- at the latest in afx_stream_flush, which submits the
 * partial buckets and waits for everything; the verdict array of every push must stay valid until then.  The contexts must not
 * be used for other calls between the first push and the flush.  One thread drives a stream. */
typedef struct afx_stream afx_stream;
int afx_stream_create(afx_stream** out);
void afx_stream_destroy(afx_stream* stream);
int afx_stream_add_shape(afx_stream* stream, afx_ctx* ctx, int issuance, uint16_t n_attrs, const uint8_t* kinds, int* shape_id,
                         size_t* record_bytes);
int afx_stream_push(afx_stream* stream, const uint8_t* records, const uint64_t* offsets, const uint8_t* shape_ids, size_t n,
                    uint8_t* verdicts);
int afx_stream_flush(afx_stream* stream);
uint64_t afx_stream_buckets_submitted(const afx_stream* stream);
/* Cumulative host time of the driving thread: copying records into buckets, enqueueing submissions, blocked waiting for the device. */
int afx_stream_times(const afx_stream* stream, double* fill_s, double* submit_s, double* wait_s);

/* Primitive self-test (parity hooks for the field / group / scalar code, independent of the protocol flows).  `in` is
 * item-major, `out` is [count][32], ok[i] = 1 unless an input encoding was rejected.
 *   op 0: in [count][32] encoding               -> compress(decompress(in))           (CompressedRistretto::decompress / compress)
 *   op 1: in [count][64] uniform bytes          -> compress(from_uniform_bytes(in))   (RistrettoPoint::from_uniform_bytes)
 *   op 2: in [count][2][32] scalar, encoding    -> compress(scalar * point)
 *   op 3: in [count][64] bytes                  -> the integer mod l                  (Scalar::from_bytes_mod_order_wide)
 *   op 4: in [count][3][32] scalars a, b, c     -> a*b + c mod l
 *   op 5..8: in [count][2][32] raw 256-bit limb vectors a, b (any value in [0, 2^256) is a legal lazily reduced field element)
 *                                               -> canonical bytes of a*b, a^2, a+b, a-b mod 2^255-19
 *   op 9: same inputs                           -> canonical ((a+b)(a-b))^2 (a-b) + a     (chained unreduced intermediates)
 *   op 10: in [count][2][32] scalar, encoding   -> compress(scalar * point) through the completed-coordinates ladder forms
 *   op 11: in [count][32] a 256-bit integer     -> the integer recomposed from its biased radix-4096 digits (the recoding of the
 *                                                  constant-base terms); ok = every digit within [-2048, 2048]
 *   op 12: in [count][32] a 256-bit integer     -> the integer recomposed from its biased radix-2^16 digits (the recoding of the
 *                                                  constant-base terms with the wide tables); ok = every low digit within
 *                                                  [-32768, 32767] and the top digit at most 2^13 + 1 */
int afx_selftest_primitive(afx_ctx* ctx, int op, const uint8_t* in, size_t count, uint8_t* out, uint8_t* ok);

/* Number of kernels this library launched on behalf of `ctx` so far (bench.py's gpu_launches). */
uint64_t afx_launch_count(const afx_ctx* ctx);

/* Per-stage device timing for the roofline report.  When enabled, every pipeline run records CUDA events between its
 * stages on the launching stream; afx_get_stage_times waits for the last run and returns the AFX_NUM_STAGES durations in
 * milliseconds, in order: scalar checks, points (decompress + tables), aMAC ladder, constraint MSMs, transcripts, verdict. */
#define AFX_NUM_STAGES 6
void afx_set_stage_timing(afx_ctx* ctx, int on);
int afx_get_stage_times(afx_ctx* ctx, float* ms, int n);
/* With stage timing on: device time of the Pippenger bucket-sum kernel (k_rlc_buckets) of the most recent random-linear-combination
 * pass, the number of per-item points it summed and the number of windows (each point enters one bucket per window). */
int afx_get_rlc_bucket_time(afx_ctx* ctx, float* ms, uint64_t* inputs, uint32_t* windows);

/* Device time of the most recent *_device / host call's kernel sequence is measured by the caller with events on the
 * stream it passed; this returns the ordinal of the CUDA device the context lives on. */
int afx_ctx_device(const afx_ctx* ctx);

/* NUMA placement for the thread that drives a device (optional, best effort).  Pins the CALLING thread to the CPUs local to the
 * device's PCI function (sysfs local_cpulist), so that page-locked staging it allocates afterwards is node-local and its copies do
 * not cross the socket interconnect: call it before afx_ctx_create / afx_host_alloc in a one-process-per-GPU or one-thread-per-GPU
 * program (measured on an 8 x B200 box: the config-5 stream of the four far-socket ranks ran 9 % slower without it).  The
 * library's own device threads (afx_multi_*) do this themselves.  AFX_ERR_ARG when the topology cannot be read (nothing changes). */
int afx_bind_thread_to_device(int device);

const char* afx_strerror(int code);
const char* afx_version(void);

/* Environment (read by the library, all optional):
 *   AFX_CTAB16_BUDGET_MB   device-memory budget for the radix-2^16 constant tables of one issuer (default 200; 0 = radix 4096 only)
 *   AFX_AMAC_SPLIT         0: never cut the aMAC ladder of a small pass into parts; g > 0: g terms per part for every pass of at most
 *                          32,768 items (default: passes of at most 8,192 items, 2 or 4 terms per part -- DESIGN.md section 5)
 *   AFX_RLC_LEAF           smallest range the bisection of a failing random-linear-combination chunk descends to (default 1024)
 *   AFX_STREAM_TRACE       non-empty: afx_stream_* logs every bucket submission and retirement with timestamps to stderr */

#ifdef __cplusplus
}
#endif
#endif
