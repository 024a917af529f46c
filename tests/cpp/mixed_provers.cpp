// C++ driver of the mixed-shape prover overloads of include/aeonflux_b200.hpp: Issuer::issue_batch and Issuer::show_batch over
// records of several shapes in one call, then the mixed verify_batch over the presentations they return.  The fixture and the
// result are sequences of length-prefixed byte strings (u64 little-endian length, then the bytes), written and checked by
// tests/test_mixed_provers.py:
//   in:  issuer bytes (Issuer::to_bytes), n, request kind vectors (concatenated), requests, their shape ids,
//        show kind vectors (concatenated), show inputs, their shape ids
//   out: issuances, issue status, presentations, show status, verdicts of the presentations
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>

#include "../../include/aeonflux_b200.hpp"

using namespace aeonflux;

static std::vector<uint8_t> rd(std::ifstream& f) {
    uint64_t n = 0;
    f.read((char*)&n, 8);
    std::vector<uint8_t> v(n);
    f.read((char*)v.data(), (std::streamsize)n);
    if (!f) { std::cerr << "short fixture\n"; std::exit(2); }
    return v;
}
static void wr(std::ofstream& f, const std::vector<uint8_t>& v) {
    uint64_t n = v.size();
    f.write((const char*)&n, 8);
    f.write((const char*)v.data(), (std::streamsize)n);
}
static std::vector<std::vector<uint8_t>> split_kinds(const std::vector<uint8_t>& flat, size_t n) {
    std::vector<std::vector<uint8_t>> r;
    for (size_t i = 0; i + n <= flat.size(); i += n) r.emplace_back(flat.begin() + i, flat.begin() + i + n);
    return r;
}
static std::vector<uint8_t> status_bytes(const std::vector<Result<>>& r) {
    std::vector<uint8_t> v;
    for (const auto& x : r) v.push_back(x.is_ok() ? 0 : 1);
    return v;
}

int main(int argc, char** argv) {
    if (argc < 4) { std::cerr << "usage: mixed_provers <fixture> <result> <max_batch>\n"; return 2; }
    std::ifstream f(argv[1], std::ios::binary);
    auto issuer_bytes = rd(f);
    const size_t n = rd(f)[0];
    auto issue_kinds = split_kinds(rd(f), n);
    auto requests = rd(f), issue_ids = rd(f);
    auto show_kinds = split_kinds(rd(f), n);
    auto inputs = rd(f), show_ids = rd(f);

    Issuer issuer = Issuer::from_bytes(issuer_bytes, 0, (size_t)std::atoi(argv[3]));
    auto issued = issuer.issue_batch(issue_kinds, requests.data(), issue_ids);
    auto shown = issuer.show_batch(show_kinds, inputs.data(), show_ids);
    auto verdicts = issuer.verify_batch(show_kinds, shown.first.data(), show_ids);
    bool threw = false;
    try {
        issuer.show_batch({show_kinds[0], std::vector<uint8_t>(n + 1, 0)}, inputs.data(), show_ids);
    } catch (const std::invalid_argument&) { threw = true; }
    if (!threw) { std::cerr << "kind vectors of different lengths were accepted\n"; return 1; }

    std::ofstream o(argv[2], std::ios::binary);
    wr(o, issued.first); wr(o, status_bytes(issued.second));
    wr(o, shown.first); wr(o, status_bytes(shown.second));
    wr(o, status_bytes(verdicts));
    std::printf("mixed_provers ok: %zu issued, %zu shown (%s)\n", issue_ids.size(), show_ids.size(), afx_version());
    return 0;
}
