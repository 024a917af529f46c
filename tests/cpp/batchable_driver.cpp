// C++ driver of the BatchableProof provers through include/aeonflux_b200.hpp: Issuer::issue_batch and Issuer::show_batch with
// batchable = true, then the BatchableProof verifiers (afx_verify_issuances_batchable, Issuer::verify_batchable exact and with a
// random linear combination), against the oracle's compact issuances and presentations in the fixture tests/test_cpp_host.py writes.
// Linked against libaeonflux_b200.so (GPU, `-m gpu`) or the test-only host emulation of the same C ABI (CPU tests).
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>

#include "../../include/aeonflux_b200.hpp"

using namespace aeonflux;

static std::vector<uint8_t> rd(std::ifstream& f, size_t n) { std::vector<uint8_t> v(n); f.read((char*)v.data(), (std::streamsize)n); if (!f) { std::cerr << "short fixture\n"; std::exit(2); } return v; }
static uint32_t rd32(std::ifstream& f) { auto v = rd(f, 4); uint32_t x; std::memcpy(&x, v.data(), 4); return x; }
#define CHECK(cond) do { if (!(cond)) { std::fprintf(stderr, "CHECK failed at %s:%d: %s\n", __FILE__, __LINE__, #cond); return 1; } } while (0)

int main(int argc, char** argv) {
    if (argc < 2) { std::cerr << "usage: batchable_driver <fixture> [max_batch]\n"; return 2; }
    size_t max_batch = argc > 2 ? (size_t)std::atoi(argv[2]) : 64;
    std::ifstream f(argv[1], std::ios::binary);
    uint32_t n = rd32(f), count = rd32(f);
    auto issuer_bytes = rd(f, rd32(f));
    auto request_kinds = rd(f, n);
    auto attrs = rd(f, (size_t)count * n * 32);
    auto rnd = rd(f, (size_t)count * (n + 7) * 64);
    auto expect_issued = rd(f, (size_t)count * (n + 9) * 32); // compact: t, U, V, challenge, responses[n + 5]
    auto pres_kinds = rd(f, n);
    uint32_t Ws = rd32(f), W = rd32(f);
    auto show_in = rd(f, (size_t)count * Ws * 32);
    auto expect_pres = rd(f, (size_t)count * W * 32);         // compact presentations

    Issuer issuer = Issuer::from_bytes(issuer_bytes, 0, max_batch);
    size_t a = issuer_bytes.size() - 64 - (32 * (size_t)(5 + n) + 4);
    Issuer user(std::vector<uint8_t>(issuer_bytes.begin(), issuer_bytes.begin() + a), std::vector<uint8_t>(issuer_bytes.begin() + a, issuer_bytes.begin() + a + 64), {}, 0, max_batch);

    // Issuer::issue in BatchableProof form: t, U, V and the responses are the compact proof's, the challenge becomes C_W, I, V
    std::vector<uint8_t> req_items((size_t)count * (3 * n + 14) * 32);
    for (uint32_t i = 0; i < count; i++) {
        std::memcpy(&req_items[(size_t)i * (3 * n + 14) * 32], &attrs[(size_t)i * n * 32], (size_t)n * 32);
        std::memcpy(&req_items[((size_t)i * (3 * n + 14) + n) * 32], &rnd[(size_t)i * (n + 7) * 64], (size_t)(n + 7) * 64);
    }
    auto issued = issuer.issue_batch(Batch::from_items(request_kinds, req_items.data(), count, 3 * n + 14), true);
    for (auto& r : issued.second) CHECK(r.is_ok());
    CHECK(issued.first.fields.size() == afx_issuance_batchable_num_fields((uint16_t)n));
    for (uint32_t i = 0; i < count; i++)
        for (uint32_t w = 0; w < n + 9; w++) {
            if (w == 3) continue;
            const uint32_t bw = w < 3 ? n + w : n + w + 2;
            CHECK(std::memcmp(&issued.first.fields[bw][32 * i], &expect_issued[((size_t)i * (n + 9) + w) * 32], 32) == 0);
        }
    auto verify_issuances = [&](const IssuanceBatch& b) {
        auto ptrs = b.pointers();
        afx_issuance_batch ib{(uint16_t)n, b.kinds.data(), b.count(), ptrs.data(), ptrs.size()};
        std::vector<uint8_t> v(b.count());
        int rc = afx_verify_issuances_batchable(user.raw(), &ib, v.data(), nullptr);
        if (rc != AFX_OK) throw Error(rc);
        return v;
    };
    for (uint8_t v : verify_issuances(issued.first)) CHECK(v == 0);
    {
        IssuanceBatch bad = issued.first; bad.fields[n + 6][0] ^= 1;   // item 0's response w
        auto v = verify_issuances(bad);
        CHECK(v[0] == 1);
        for (uint32_t i = 1; i < count; i++) CHECK(v[i] == 0);
    }

    // AnonymousCredential::show in BatchableProof form, user side
    auto shown = user.show_batch(Batch::from_items(pres_kinds, show_in.data(), count, Ws), true);
    for (auto& r : shown.second) CHECK(r.is_ok());
    const size_t Wb = afx_batchable_num_fields((uint16_t)n, pres_kinds.data());
    CHECK(shown.first.fields.size() == Wb);
    size_t hp = 0, hs = 0;
    for (uint8_t k : pres_kinds) { hp += k == AFX_KIND_SECRET_POINT; hs += k == AFX_KIND_SECRET_SCALAR; }
    const size_t nc = Wb + 1 - W - 4 * hp, head = 1 + 3 + hs + 3 + n;   // main-proof commitments; words up to C_y[n]
    for (uint32_t i = 0; i < count; i++)                      // the responses, C_x_0, C_x_1, C_V, C_y: the compact proof's
        for (size_t w = 1; w < head; w++) CHECK(std::memcmp(&shown.first.fields[nc + w - 1][32 * i], &expect_pres[((size_t)i * W + w) * 32], 32) == 0);
    const uint8_t seed[32] = {7};
    for (auto& r : issuer.verify_batchable(shown.first)) CHECK(r.is_ok());
    for (auto& r : issuer.verify_batchable(shown.first, seed)) CHECK(r.is_ok());
    {
        PresentationBatch bad = shown.first; bad.fields[nc][32 * (count - 1)] ^= 1;   // the last item's response z
        for (const uint8_t* s : {(const uint8_t*)nullptr, seed}) {
            auto v = issuer.verify_batchable(bad, s);
            for (uint32_t i = 0; i < count; i++) CHECK(v[i].is_ok() == (i + 1 < count));
            CHECK(v[count - 1].error == CredentialError::VerificationFailure);
        }
    }
    std::printf("batchable_driver ok: %u items, %s\n", count, afx_version());
    return 0;
}
