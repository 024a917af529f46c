// aeonflux_b200.hpp -- C++ host-side mirror of the reference's interface for the hot path, over the C ABI of
// aeonflux_b200.h.  The reference is a Rust crate; no Rust toolchain exists in this image, so the host code above the C ABI
// is C++ (header-only, links against libaeonflux_b200.so) and mirrors the reference's names, argument meaning and error
// behaviour so that callers and tests read like the reference's own:
//
//   reference (Rust)                                                   here (namespace aeonflux)
//   -----------------------------------------------------------------  -----------------------------------------------------
//   enum CredentialError { ..., VerificationFailure, MacCreation }     enum class CredentialError          src/errors.rs:73-89
//   Result<T, CredentialError>                                         Result<T>
//   Issuer { system_parameters, issuer_parameters, amacs_key }         class Issuer                        src/issuer.rs:61-65
//   Issuer::from_bytes / to_bytes                                      Issuer::from_bytes / to_bytes       src/issuer.rs:152-174
//   Issuer::verify(&self, &ProofOfValidCredential)                     Issuer::verify_batch(PresentationBatch)    :141-147
//   Issuer::issue(&self, CredentialRequest, &mut rng)                  Issuer::issue_batch(RequestBatch)          :111-124
//   CredentialIssuance::verify(self, &sysparams, &issuer_params)       CredentialIssuance::verify_batch(Issuer&, IssuanceBatch)  :48-57
//   AnonymousCredential::show(...)                                     Issuer::show_batch(ShowBatch)  (user side, no secret key)
//   (zkp prove_batchable instead of prove_compact)                     issue_batch / show_batch with batchable = true
//
// A batch is one attribute shape (the kinds vector) and struct-of-arrays fields, each `count` x 32 bytes; the field orders are
// documented in aeonflux_b200.h.  Structural mistakes (wrong field count, wrong attribute count) throw std::invalid_argument /
// aeonflux::Error, the analogue of the reference's panics and constructor errors; per-item outcomes are Results.
#ifndef AEONFLUX_B200_HPP
#define AEONFLUX_B200_HPP

#include <array>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "aeonflux_b200.h"

namespace aeonflux {

enum class CredentialError {   // src/errors.rs:73-89, same variants
    BadAttribute, CredentialIssuance, MacCreation, MacVerification, MissingData, NoSymmetricKey, NoIssuerKey, NoIssuerParameters,
    NoSystemParameters, PointDecompressionError, ScalarFormatError, UndecryptableAttribute, VerificationFailure,
    WrongNumberOfAttributes, WrongNumberOfBytes
};

// Result<(), CredentialError> / Result<T, CredentialError>
template <typename T = void> struct Result;
template <> struct Result<void> {
    bool ok; CredentialError error;
    static Result Ok() { return {true, CredentialError::VerificationFailure}; }
    static Result Err(CredentialError e) { return {false, e}; }
    bool is_ok() const { return ok; }
    bool is_err() const { return !ok; }
};

struct Error : std::runtime_error {   // a non-zero afx_* return code
    int code;
    Error(int c) : std::runtime_error(std::string("aeonflux_b200: ") + afx_strerror(c)), code(c) {}
};

typedef std::array<uint8_t, 32> Word;   // a canonical Scalar or a CompressedRistretto

// Symmetric encryption of attributes (src/symmetric.rs): the 30 data bytes, Plaintext (M1, M2, m3), Ciphertext (E1, E2) and the
// keypair's secret scalars a || a0 || a1, laid out as the C ABI takes them.
typedef std::array<uint8_t, 30> AttributeData;
struct Plaintext { Word M1, M2, m3; };
struct Ciphertext { Word E1, E2; };
typedef std::array<uint8_t, 96> KeypairSecret;
static_assert(sizeof(Plaintext) == 96 && sizeof(Ciphertext) == 64 && sizeof(AttributeData) == 30, "C ABI layouts");
// Keypair::derive's input and output (src/symmetric.rs:74-79,197-215): the 64-byte master secret, and a || a0 || a1 || pk -- the
// keypair afx_show takes, whose first 96 bytes (secret) are what encrypt_batch and decrypt_batch take.
typedef std::array<uint8_t, 64> MasterSecret;
struct Keypair { KeypairSecret secret; Word pk; };
static_assert(sizeof(MasterSecret) == 64 && sizeof(Keypair) == 128 && offsetof(Keypair, pk) == 96, "C ABI layouts");

// One shape, struct-of-arrays.  fields[f] holds count * 32 bytes.
struct Batch {
    std::vector<uint8_t> kinds;
    std::vector<std::vector<uint8_t>> fields;
    size_t count() const { return fields.empty() ? 0 : fields[0].size() / 32; }
    // item-major words ([count][n_fields][32], e.g. as received from the wire) -> struct of arrays
    static Batch from_items(const std::vector<uint8_t>& kinds, const uint8_t* items, size_t count, size_t n_fields) {
        Batch b; b.kinds = kinds; b.fields.assign(n_fields, std::vector<uint8_t>(count * 32));
        for (size_t i = 0; i < count; i++)
            for (size_t f = 0; f < n_fields; f++) std::memcpy(&b.fields[f][32 * i], items + (i * n_fields + f) * 32, 32);
        return b;
    }
    std::vector<const uint8_t*> pointers() const {
        std::vector<const uint8_t*> p;
        for (const auto& f : fields) { if (f.size() != count() * 32) throw std::invalid_argument("ragged batch"); p.push_back(f.data()); }
        return p;
    }
};
typedef Batch PresentationBatch;   // kinds AFX_KIND_*; fields: challenge, responses, C_x_0, C_x_1, C_V, C_y[n], revealed..., enc proofs
typedef Batch IssuanceBatch;       // kinds 0 scalar / 2 point; fields: attribute[n], t, U, V, challenge, responses[n+5]
typedef Batch RequestBatch;        // fields: attribute[n], then (lo, hi) halves of the rng bytes of t, U, blinding[n+5]
typedef Batch ShowBatch;           // fields: t, U, V, attributes, keypair, rng bytes (afx_show)

class Issuer {
public:
    // Issuer::new's result restored from its parts: SystemParameters::to_bytes, C_W || I, SecretKey::to_bytes (empty = user side)
    Issuer(const std::vector<uint8_t>& system_parameters, const std::vector<uint8_t>& issuer_parameters, const std::vector<uint8_t>& amacs_key,
           int device = 0, size_t max_batch = 65536)
        : sp_(system_parameters), ip_(issuer_parameters), sk_(amacs_key) {
        if (ip_.size() != 64) throw std::invalid_argument("issuer_parameters must be C_W || I (64 bytes)");
        int rc = afx_ctx_create(sp_.data(), sp_.size(), ip_.data(), sk_.empty() ? nullptr : sk_.data(), sk_.size(), device, max_batch, &ctx_);
        if (rc != AFX_OK) throw Error(rc);
    }
    // Issuer::from_bytes (src/issuer.rs:152-159): sysparams || C_W || I || secret key
    static Issuer from_bytes(const std::vector<uint8_t>& b, int device = 0, size_t max_batch = 65536) {
        if (b.size() < 4) throw std::invalid_argument("NoIssuerParameters");
        uint32_t n; std::memcpy(&n, b.data(), 4);
        size_t a = n < 3 ? 32 * (size_t)(5 + 3 + n + 4) + 4 : 32 * (size_t)(5 + 2 * n + 4) + 4, k = 32 * (size_t)(5 + n) + 4;   // parameters.rs:34-40, amacs.rs:44-46
        if (n == 0 || b.size() != a + 64 + k) throw std::invalid_argument("NoIssuerParameters");
        return Issuer(std::vector<uint8_t>(b.begin(), b.begin() + a), std::vector<uint8_t>(b.begin() + a, b.begin() + a + 64),
                      std::vector<uint8_t>(b.begin() + a + 64, b.end()), device, max_batch);
    }
    // Issuer::to_bytes (src/issuer.rs:162-174; panics in the reference because IssuerParameters::to_bytes is unimplemented!())
    std::vector<uint8_t> to_bytes() const { std::vector<uint8_t> v(sp_); v.insert(v.end(), ip_.begin(), ip_.end()); v.insert(v.end(), sk_.begin(), sk_.end()); return v; }
    ~Issuer() { if (ctx_) afx_ctx_destroy(ctx_); for (volatile uint8_t& x : sk_) x = 0; }   // Drop: zeroize (src/amacs.rs:64-82)
    Issuer(Issuer&& o) noexcept : sp_(std::move(o.sp_)), ip_(std::move(o.ip_)), sk_(std::move(o.sk_)), ctx_(o.ctx_) { o.ctx_ = nullptr; }
    Issuer(const Issuer&) = delete;
    Issuer& operator=(const Issuer&) = delete;

    uint32_t number_of_attributes() const { uint32_t n; std::memcpy(&n, sp_.data(), 4); return n; }
    afx_ctx* raw() const { return ctx_; }

    // Batch Issuer::verify: Ok(()) or Err(VerificationFailure) per presentation (src/errors.rs:152-156)
    std::vector<Result<>> verify_batch(const PresentationBatch& p) const {
        if (p.fields.size() != afx_presentation_num_fields((uint16_t)p.kinds.size(), p.kinds.data())) throw std::invalid_argument("wrong number of presentation fields");
        auto ptrs = p.pointers();
        afx_presentation_batch b{(uint16_t)p.kinds.size(), p.kinds.data(), p.count(), ptrs.data(), ptrs.size()};
        std::vector<uint8_t> v(p.count());
        int rc = afx_verify_presentations(ctx_, &b, v.data(), nullptr);
        if (rc != AFX_OK) throw Error(rc);
        return to_results(v);
    }
    // Opt-in BatchableProof form (commitments instead of challenges; not the reference's encoding, see aeonflux_b200.h):
    // exact per-constraint check, or one random linear combination per chunk with the exact check as fallback.
    std::vector<Result<>> verify_batchable(const PresentationBatch& p, const uint8_t* rlc_seed32 = nullptr) const {
        if (p.fields.size() != afx_batchable_num_fields((uint16_t)p.kinds.size(), p.kinds.data())) throw std::invalid_argument("wrong number of batchable fields");
        auto ptrs = p.pointers();
        afx_presentation_batch b{(uint16_t)p.kinds.size(), p.kinds.data(), p.count(), ptrs.data(), ptrs.size()};
        std::vector<uint8_t> v(p.count());
        int rc = rlc_seed32 ? afx_verify_presentations_batchable_rlc(ctx_, &b, rlc_seed32, v.data(), nullptr)
                            : afx_verify_presentations_batchable(ctx_, &b, v.data(), nullptr);
        if (rc != AFX_OK) throw Error(rc);
        return to_results(v);
    }
    // ... over item-major wire bytes ([count][n_fields][32])
    std::vector<Result<>> verify_wire(const std::vector<uint8_t>& kinds, const uint8_t* items, size_t count) const {
        std::vector<uint8_t> v(count);
        int rc = afx_verify_presentations_wire(ctx_, (uint16_t)kinds.size(), kinds.data(), count, items, v.data());
        if (rc != AFX_OK) throw Error(rc);
        return to_results(v);
    }
    // ... over presentations of any of `shape_kinds` (each user hides what it chooses): records = the wire records concatenated in
    // order, record i of shape shape_ids[i]; bucketed by shape on the device, results in record order
    std::vector<Result<>> verify_batch(const std::vector<std::vector<uint8_t>>& shape_kinds, const uint8_t* records,
                                       const std::vector<uint8_t>& shape_ids) const {
        const std::vector<uint8_t> flat = flatten_kinds(shape_kinds);
        const uint16_t n = shape_kinds.empty() ? 0 : (uint16_t)shape_kinds[0].size();
        std::vector<uint8_t> v(shape_ids.size());
        int rc = afx_verify_presentations_mixed_wire(ctx_, n, flat.data(), shape_kinds.size(), shape_ids.size(), records, shape_ids.data(), v.data());
        if (rc != AFX_OK) throw Error(rc);
        return to_results(v);
    }
    // Batch Issuer::issue.  Err(MacCreation) for the whole batch when the attribute count is not the issuer's (src/amacs.rs:285-287);
    // otherwise the issuances (in IssuanceBatch layout) and a per-item Result.  batchable: zkp's prove_batchable form, the
    // challenge replaced by the commitments C_W, I, V (2n + 11 fields, what afx_verify_issuances_batchable takes).
    std::pair<IssuanceBatch, std::vector<Result<>>> issue_batch(const RequestBatch& r, bool batchable = false) const {
        size_t n = r.kinds.size(), count = r.count(), nw = 2 * n + (batchable ? 11 : 9);
        IssuanceBatch out; out.kinds = r.kinds;
        if (n != number_of_attributes()) return {out, std::vector<Result<>>(count, Result<>::Err(CredentialError::MacCreation))};
        if (r.fields.size() != afx_request_num_fields((uint16_t)n)) throw std::invalid_argument("wrong number of request fields");
        out.fields.assign(nw, std::vector<uint8_t>(count * 32));
        for (size_t i = 0; i < n; i++) out.fields[i] = r.fields[i];
        auto in = r.pointers();
        std::vector<uint8_t*> op;
        for (size_t w = n; w < nw; w++) op.push_back(out.fields[w].data());
        afx_request_batch b{(uint16_t)n, r.kinds.data(), count, in.data(), in.size()};
        afx_issuance_out o{op.data(), op.size()};
        std::vector<uint8_t> st(count);
        int rc = batchable ? afx_issue_batchable(ctx_, &b, &o, st.data(), nullptr) : afx_issue(ctx_, &b, &o, st.data(), nullptr);
        if (rc != AFX_OK) throw Error(rc);
        std::vector<Result<>> res;
        for (uint8_t s : st) res.push_back(s == 0 ? Result<>::Ok() : Result<>::Err(CredentialError::BadAttribute));
        return {out, res};
    }
    // ... over CredentialRequests of any of `shape_kinds` in one call: requests = the wire requests concatenated in order (3n + 14
    // words each), request i of kinds shape_kinds[shape_ids[i]]; bucketed by shape on the device.  Returns the issuances in record
    // order ([count][2n + 9][32], what the mixed verify_issuances call takes) and a per-item Result.
    std::pair<std::vector<uint8_t>, std::vector<Result<>>> issue_batch(const std::vector<std::vector<uint8_t>>& shape_kinds, const uint8_t* requests,
                                                                       const std::vector<uint8_t>& shape_ids) const {
        const std::vector<uint8_t> flat = flatten_kinds(shape_kinds);
        const uint16_t n = shape_kinds.empty() ? 0 : (uint16_t)shape_kinds[0].size();
        std::vector<uint8_t> out(shape_ids.size() * (2 * (size_t)n + 9) * 32), st(shape_ids.size());
        int rc = afx_issue_mixed_wire(ctx_, n, flat.data(), shape_kinds.size(), shape_ids.size(), requests, shape_ids.data(), out.data(), st.data());
        if (rc != AFX_OK) throw Error(rc);
        return {out, status_results(st, CredentialError::BadAttribute)};
    }
    // Batch AnonymousCredential::show over inputs of any of `shape_kinds` in one call (each user hides what it chooses): inputs = the
    // wire show inputs concatenated in order, input i of shape shape_ids[i].  Returns the presentations concatenated in record order
    // (what the mixed verify_batch takes) and a per-item Result.
    std::pair<std::vector<uint8_t>, std::vector<Result<>>> show_batch(const std::vector<std::vector<uint8_t>>& shape_kinds, const uint8_t* inputs,
                                                                      const std::vector<uint8_t>& shape_ids) const {
        const std::vector<uint8_t> flat = flatten_kinds(shape_kinds);
        const uint16_t n = shape_kinds.empty() ? 0 : (uint16_t)shape_kinds[0].size();
        size_t bytes = 0;
        for (uint8_t s : shape_ids) if (s < shape_kinds.size()) bytes += 32 * afx_presentation_num_fields(n, shape_kinds[s].data());
        std::vector<uint8_t> out(bytes), st(shape_ids.size());
        int rc = afx_show_mixed_wire(ctx_, n, flat.data(), shape_kinds.size(), shape_ids.size(), inputs, shape_ids.data(), out.data(), st.data());
        if (rc != AFX_OK) throw Error(rc);
        return {out, status_results(st, CredentialError::BadAttribute)};
    }
    // Batch AnonymousCredential::show (user side; works on a context without the secret key).  batchable: zkp's prove_batchable
    // form, every challenge replaced by that proof's commitments (what verify_batchable takes).
    std::pair<PresentationBatch, std::vector<Result<>>> show_batch(const ShowBatch& s, bool batchable = false) const {
        size_t count = s.count();
        if (s.fields.size() != afx_show_num_fields((uint16_t)s.kinds.size(), s.kinds.data())) throw std::invalid_argument("wrong number of show fields");
        PresentationBatch out; out.kinds = s.kinds;
        size_t nw = batchable ? afx_batchable_num_fields((uint16_t)s.kinds.size(), s.kinds.data())
                              : afx_presentation_num_fields((uint16_t)s.kinds.size(), s.kinds.data());
        out.fields.assign(nw, std::vector<uint8_t>(count * 32));
        auto in = s.pointers();
        std::vector<uint8_t*> op;
        for (auto& f : out.fields) op.push_back(f.data());
        afx_show_batch b{(uint16_t)s.kinds.size(), s.kinds.data(), count, in.data(), in.size()};
        afx_presentation_out o{op.data(), op.size()};
        std::vector<uint8_t> st(count);
        int rc = batchable ? afx_show_batchable(ctx_, &b, &o, st.data(), nullptr) : afx_show(ctx_, &b, &o, st.data(), nullptr);
        if (rc != AFX_OK) throw Error(rc);
        std::vector<Result<>> res;
        for (uint8_t x : st) res.push_back(x == 0 ? Result<>::Ok() : Result<>::Err(CredentialError::BadAttribute));
        return {out, res};
    }
    // Plaintext::from(&[u8; 30]) per item (src/symmetric.rs:135-143); Err(BadAttribute) where no candidate encoding decodes
    std::pair<std::vector<Plaintext>, std::vector<Result<>>> encode_batch(const std::vector<AttributeData>& data) const {
        std::vector<Plaintext> out(data.size());
        std::vector<uint8_t> st(data.size());
        int rc = afx_encode_plaintexts(ctx_, data.size(), data.empty() ? nullptr : data[0].data(), (uint8_t*)out.data(), st.data());
        if (rc != AFX_OK) throw Error(rc);
        return {out, status_results(st, CredentialError::BadAttribute)};
    }
    // Keypair::encrypt per item (src/symmetric.rs:252-261); Err(BadAttribute) for a Plaintext the Rust type could never hold
    std::pair<std::vector<Ciphertext>, std::vector<Result<>>> encrypt_batch(const KeypairSecret& keypair, const std::vector<Plaintext>& pts) const {
        std::vector<Ciphertext> out(pts.size());
        std::vector<uint8_t> st(pts.size());
        int rc = afx_encrypt(ctx_, keypair.data(), pts.size(), (const uint8_t*)pts.data(), (uint8_t*)out.data(), st.data());
        if (rc != AFX_OK) throw Error(rc);
        return {out, status_results(st, CredentialError::BadAttribute)};
    }
    // Keypair::derive per item (src/symmetric.rs:197-215) under this issuer's system parameters; Keypair::generate is this on 64 rng bytes
    std::vector<Keypair> derive_keypairs(const std::vector<MasterSecret>& master_secrets) const {
        std::vector<Keypair> out(master_secrets.size());
        int rc = afx_derive_keypairs(ctx_, master_secrets.size(), master_secrets.empty() ? nullptr : master_secrets[0].data(), (uint8_t*)out.data());
        if (rc != AFX_OK) throw Error(rc);
        return out;
    }
    // Keypair::decrypt per item (src/symmetric.rs:273-289): the data and the Plaintext, or Err(UndecryptableAttribute)
    std::pair<std::vector<std::pair<AttributeData, Plaintext>>, std::vector<Result<>>> decrypt_batch(const KeypairSecret& keypair,
                                                                                                       const std::vector<Ciphertext>& cts) const {
        std::vector<AttributeData> data(cts.size());
        std::vector<Plaintext> pts(cts.size());
        std::vector<uint8_t> st(cts.size());
        int rc = afx_decrypt(ctx_, keypair.data(), cts.size(), (const uint8_t*)cts.data(), (uint8_t*)data.data(), (uint8_t*)pts.data(), st.data());
        if (rc != AFX_OK) throw Error(rc);
        std::vector<std::pair<AttributeData, Plaintext>> out;
        for (size_t i = 0; i < cts.size(); i++) out.push_back({data[i], pts[i]});
        return {out, status_results(st, CredentialError::UndecryptableAttribute)};
    }

private:
    static std::vector<Result<>> status_results(const std::vector<uint8_t>& st, CredentialError e) {
        std::vector<Result<>> r;
        for (uint8_t x : st) r.push_back(x == 0 ? Result<>::Ok() : Result<>::Err(e));
        return r;
    }
    static std::vector<Result<>> to_results(const std::vector<uint8_t>& v) {
        std::vector<Result<>> r;
        for (uint8_t x : v) r.push_back(x == 0 ? Result<>::Ok() : Result<>::Err(CredentialError::VerificationFailure));
        return r;
    }
    // the kind vectors of a mixed-shape call, concatenated; they all have one attribute count
    static std::vector<uint8_t> flatten_kinds(const std::vector<std::vector<uint8_t>>& shape_kinds) {
        std::vector<uint8_t> flat;
        for (const auto& k : shape_kinds) {
            if (k.size() != shape_kinds[0].size()) throw std::invalid_argument("every kind vector has the issuer's attribute count");
            flat.insert(flat.end(), k.begin(), k.end());
        }
        return flat;
    }
    std::vector<uint8_t> sp_, ip_, sk_;
    afx_ctx* ctx_ = nullptr;
    friend struct CredentialIssuance;
    friend class MultiGpuIssuer;
};

// One process driving several B200s through the C ABI's multi-device handle (afx_multi_*, SURVEY 8b/8e): the library keeps a
// replicated context and one host thread per device; device k verifies the contiguous item slice [k*N/G, (k+1)*N/G); nothing
// but the verdicts is gathered.  The single-process counterpart of bench.py's one-process-per-GPU launch.
class MultiGpuIssuer {
public:
    MultiGpuIssuer(const std::vector<uint8_t>& system_parameters, const std::vector<uint8_t>& issuer_parameters, const std::vector<uint8_t>& amacs_key,
                   const std::vector<int>& devices, size_t max_batch = 65536) {
        if (devices.empty()) throw std::invalid_argument("at least one device");
        if (issuer_parameters.size() != 64) throw std::invalid_argument("issuer_parameters must be C_W || I (64 bytes)");
        int rc = afx_multi_create(system_parameters.data(), system_parameters.size(), issuer_parameters.data(), amacs_key.empty() ? nullptr : amacs_key.data(),
                                  amacs_key.size(), devices.data(), (int)devices.size(), max_batch, &m_);
        if (rc != AFX_OK) throw Error(rc);
    }
    ~MultiGpuIssuer() { if (m_) afx_multi_destroy(m_); }
    MultiGpuIssuer(const MultiGpuIssuer&) = delete;
    MultiGpuIssuer& operator=(const MultiGpuIssuer&) = delete;
    size_t devices() const { return (size_t)afx_multi_num_devices(m_); }
    std::vector<Result<>> verify_batch(const PresentationBatch& p) const {
        if (p.fields.size() != afx_presentation_num_fields((uint16_t)p.kinds.size(), p.kinds.data())) throw std::invalid_argument("wrong number of presentation fields");
        auto ptrs = p.pointers();   // rejects a ragged batch
        afx_presentation_batch b{(uint16_t)p.kinds.size(), p.kinds.data(), p.count(), ptrs.data(), ptrs.size()};
        std::vector<uint8_t> v(p.count());
        int rc = afx_multi_verify_presentations(m_, &b, v.data());
        if (rc != AFX_OK) throw Error(rc);
        return Issuer::to_results(v);
    }
    std::vector<Result<>> verify_wire(const std::vector<uint8_t>& kinds, const uint8_t* items, size_t count) const {
        std::vector<uint8_t> v(count);
        int rc = afx_multi_verify_presentations_wire(m_, (uint16_t)kinds.size(), kinds.data(), count, items, v.data());
        if (rc != AFX_OK) throw Error(rc);
        return Issuer::to_results(v);
    }

private:
    afx_multi* m_ = nullptr;
};

// CredentialIssuance::verify (src/issuer.rs:48-57), batch form; needs only the public parameters held by `params`.
struct CredentialIssuance {
    static std::vector<Result<>> verify_batch(const Issuer& params, const IssuanceBatch& i) {
        if (i.fields.size() != 2 * i.kinds.size() + 9) throw std::invalid_argument("wrong number of issuance fields");
        auto ptrs = i.pointers();
        afx_issuance_batch b{(uint16_t)i.kinds.size(), i.kinds.data(), i.count(), ptrs.data(), ptrs.size()};
        std::vector<uint8_t> v(i.count());
        int rc = afx_verify_issuances(params.raw(), &b, v.data(), nullptr);
        if (rc != AFX_OK) throw Error(rc);
        return Issuer::to_results(v);
    }
};

}  // namespace aeonflux
#endif
