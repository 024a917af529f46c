// Host-side "shape compiler": turns an attribute-kind vector into the stage descriptors engine.cuh executes.
//
// It restates, as data, the statement structure of
//   ProofOfValidCredential::verify   /root/reference/src/nizk/presentation.rs:324-443
//   ProofOfEncryption::verify        /root/reference/src/nizk/encryption.rs:154-210
//   ProofOfIssuance::verify          /root/reference/src/nizk/issuance.rs:132-218
// and of the zkp 0.7 toolbox / merlin framing they drive (SURVEY A.3-A.5): which points are allocated under which
// labels and in which order, which constraints exist, and every quirk of SURVEY A.6 (compacted-index constraint loop,
// G_y padded to >= 3, singular/plural transcript labels, identity rejection only for allocated points).  Each statement's
// constraint order, wire layout and transcript schedule are written once, and its prover and verifier compilers both use them.
// Pure byte/bookkeeping work: no field arithmetic happens on the host.
#pragma once
#include <algorithm>
#include <array>
#include <cstring>
#include <iterator>
#include <stdexcept>
#include <string>
#include <vector>

#include "engine.cuh"

namespace afx {

// ---- per-issuer constants -------------------------------------------------------------------------
// Constant point ids follow the SystemParameters::to_bytes order (parameters.rs:155-184), then C_W, I.
struct IssuerConsts {
    u32 n = 0, ny = 0;
    std::vector<std::array<uint8_t, 32>> enc;      // compressed encoding of constant point id
    std::vector<std::array<uint8_t, 32>> enc_neg;  // compressed encoding of its negation (filled by device setup)
    std::vector<std::array<uint8_t, 32>> enc_link; // [ny] encoding of G_y[i] - G_y[0] (linked presentations; filled by device setup; entry 0 unused)
    u32 id_G() const { return 0; }
    u32 id_Gw() const { return 1; }
    u32 id_Gwp() const { return 2; }
    u32 id_Gx0() const { return 3; }
    u32 id_Gx1() const { return 4; }
    u32 id_Gy(u32 i) const { return 5 + i; }
    u32 id_Gm(u32 i) const { return 5 + ny + i; }
    u32 id_GV() const { return 5 + ny + n; }
    u32 id_Ga() const { return 6 + ny + n; }
    u32 id_Ga0() const { return 7 + ny + n; }
    u32 id_Ga1() const { return 8 + ny + n; }
    u32 id_CW() const { return 9 + ny + n; }
    u32 id_I() const { return 10 + ny + n; }
    u32 count() const { return 11 + ny + n; }
};
// secret rows (secdig / secsc): 0 = x_0, 1 = x_1, 2 + i = y_i, then w, w'
inline u32 sec_x0() { return 0; }
inline u32 sec_x1() { return 1; }
inline u32 sec_y(u32 i) { return 2 + i; }

inline size_t sysparams_size(u32 n) { return n < 3 ? 32 * (5 + 3 + n + 4) + 4 : 32 * (5 + 2 * n + 4) + 4; }  // parameters.rs:34-40
inline size_t secret_size(u32 n) { return 32 * (5 + n) + 4; }                                                // amacs.rs:44-46

// ---- transcript template builder (symbolic STROBE-128, SURVEY A.3) ----------------------------------
struct PointSrc { u32 kind, idx; };   // where an allocated point's encoding comes from: SRC_FIELD / SRC_COMP / SRC_COMMIT and its index
struct TxBuilder {
    std::vector<std::array<uint8_t, 168>> blocks;
    std::array<uint8_t, 168> cur{};
    int pos = 0, pos_begin = 0, cur_flags = 0;
    std::vector<TxHole> holes;
    std::vector<TxIdCheck> ids;
    bool init_done = false;

    void run_f() {
        cur[pos] ^= (uint8_t)pos_begin; cur[pos + 1] ^= 0x04; cur[167] ^= 0x80;
        blocks.push_back(cur); cur.fill(0); pos = 0; pos_begin = 0;
    }
    void absorb(const uint8_t* d, size_t n) {
        for (size_t i = 0; i < n; i++) { cur[pos++] ^= d[i]; if (pos == 166) run_f(); }
    }
    void absorb_hole(u32 kind, u32 idx) {
        u32 done = 0;
        while (done < 32) {
            u32 room = 166 - pos, take = (32 - done) < room ? (32 - done) : room;
            TxHole h; h.block = (u16)blocks.size(); h.off = (u16)pos; h.len = (u16)take; h.src_off = (u16)done; h.src_kind = (u16)kind; h.src_idx = (u16)idx;
            holes.push_back(h);
            pos += take; done += take;
            if (pos == 166) run_f();
        }
    }
    void begin_op(int flags, bool more) {
        if (more) return;
        uint8_t hdr[2] = {(uint8_t)pos_begin, (uint8_t)flags};
        pos_begin = pos + 1; cur_flags = flags;
        absorb(hdr, 2);
        if ((flags & (4 | 32)) && pos != 0) run_f();
    }
    void meta_ad(const void* d, size_t n, bool more) { begin_op(16 | 2, more); absorb((const uint8_t*)d, n); }
    void ad(const void* d, size_t n, bool more) { begin_op(2, more); absorb((const uint8_t*)d, n); }
    void start(const char* transcript_label) {
        // Strobe128::new("Merlin v1.0"): the initial permutation is a block whose mask is the 18 header bytes
        static const uint8_t hdr[6] = {1, 168, 1, 0, 1, 96};
        std::memcpy(cur.data(), hdr, 6); std::memcpy(cur.data() + 6, "STROBEv1.0.2", 12);
        blocks.push_back(cur); cur.fill(0); pos = 0; pos_begin = 0;
        meta_ad("Merlin v1.0", 11, false);
        append_message("dom-sep", transcript_label, std::strlen(transcript_label));
    }
    void append_header(const char* label, u32 len) {
        meta_ad(label, std::strlen(label), false);
        uint8_t l4[4] = {(uint8_t)len, (uint8_t)(len >> 8), (uint8_t)(len >> 16), (uint8_t)(len >> 24)};
        meta_ad(l4, 4, true);
    }
    void append_message(const char* label, const void* msg, size_t len) { append_header(label, (u32)len); ad(msg, len, false); }
    // zkp TranscriptProtocol (SURVEY A.4)
    void domain_sep(const char* label) {
        append_message("dom-sep", "schnorrzkp/1.0/ristretto255", 27);
        append_message("dom-sep", label, std::strlen(label));
    }
    void scalar_var(const char* label) { append_message("scvar", label, std::strlen(label)); }
    void point_var_const(const char* label, const uint8_t enc[32]) {  // per-issuer constant: identity checked at ctx creation
        append_message("ptvar", label, std::strlen(label)); append_message("val", enc, 32);
    }
    // verifier: validate_and_append_point_var (identity rejected); prover: append_point_var (no check, SURVEY A.4)
    void point_var(const char* label, PointSrc s, bool check_identity) {
        if (check_identity) { TxIdCheck c; c.src_kind = (u16)s.kind; c.src_idx = (u16)s.idx; ids.push_back(c); }
        append_message("ptvar", label, std::strlen(label));
        append_header("val", 32); begin_op(2, false); absorb_hole(s.kind, s.idx);
    }
    void blinding_commitment_wire(const char* label, u32 field) {   // verify_batchable: validate_and_append_blinding_commitment
        TxIdCheck c; c.src_kind = (u16)SRC_FIELD; c.src_idx = (u16)field; ids.push_back(c);
        append_message("blindcom", label, std::strlen(label));
        append_header("val", 32); begin_op(2, false); absorb_hole(SRC_FIELD, field);
    }
    void blinding_commitment(const char* label, u32 commit_slot) {
        append_message("blindcom", label, std::strlen(label));
        append_header("val", 32); begin_op(2, false); absorb_hole(SRC_COMMIT, commit_slot);
    }
    void challenge() {  // get_challenge("chal"): 64 bytes; the output is the head of the state after the last block
        append_header("chal", 64);
        int nb = (int)blocks.size();
        begin_op(1 | 2 | 4, false);
        if ((int)blocks.size() == nb) throw std::logic_error("transcript: prf did not close a block");
        if (pos != 0) throw std::logic_error("transcript: dangling bytes");
    }
};

// ---- compiled program --------------------------------------------------------------------------------
struct ShapeProgram {
    u32 n_fields = 0, n_tables = 0, n_atabs = 0, n_ext = 0, n_comp = 0, n_msm = 0, n_proofs = 0;
    bool batchable = false;            // BatchableProof form: commitments on the wire, challenges derived (transcripts run before the MSMs)
    u32 n_point_jobs_amac = 0;         // the first point jobs feed the aMAC ladder (batchable mode runs the rest beside it)
    std::vector<CmpPair> cmp_pairs;    // (recomputed commitment slot, wire commitment field)
    std::vector<u16> commit_ext;       // extended-coordinates slot of each wire commitment, same order as cmp_pairs' fields
    std::vector<RlcDesc> rlc;          // one descriptor (batchable mode): inputs / constant terms of the random linear combination
    std::vector<CmpPair> eq_fields;    // linked presentations: wire words that must be equal (commit_slot = 0x8000 | field a, field = field b)
    std::vector<u32> pre_msms;         // batchable mode: MSM jobs whose outputs the transcript absorbs (tU, M_i of an issuance): they run before it
    bool is_issue = false;             // Issuer::issue: constant-schedule MSMs, derived scalars, output words instead of verdicts
    std::vector<DeriveOp> derived;     // per-item derived scalars, slot k = op k
    std::vector<OutWord> out_words;    // prover output words
    std::vector<u16> scalar_fields;
    std::vector<PointJob> point_jobs;
    bool has_amac = false;
    AmacDesc amac{};
    std::vector<MsmDesc> msms;
    std::vector<TxDesc> txs;
    std::vector<u64> lanes;
    std::vector<TxHole> holes;
    std::vector<TxIdCheck> ids;
    u32 z_comp_slot = 0;          // where the recomputed Z encoding lands (debug dump)
    u32 z_msm = 0;                // index of the one MSM that reads Z's ladder table (constraint "Z")
    std::vector<u32> dump_commit; // commit slots that are blinding commitments, in constraint order (debug dump)
};

inline u32 sref_secret(u32 row) { return SREF_SECRET | row; }
inline u32 sref_derived(u32 slot) { return SREF_DERIVED | slot; }
inline ScalarSrc sc_field(u32 f) { ScalarSrc s; s.op = SC_FIELD; s.f0 = (u16)f; s.f1 = s.f2 = 0; return s; }
inline ScalarSrc sc_mul2(u32 a, u32 b) { ScalarSrc s; s.op = SC_MUL; s.f0 = (u16)a; s.f1 = (u16)b; s.f2 = 0; return s; }
inline ScalarSrc sc_muladd3(u32 a, u32 b, u32 c) { ScalarSrc s; s.op = SC_MULADD; s.f0 = (u16)a; s.f1 = (u16)b; s.f2 = (u16)c; return s; }

struct MsmBuilder {
    MsmDesc d{};
    const std::vector<int>& tab2ext;   // extended-coordinates slot of each ladder table's base (-1 = none: only BatchableProof verifiers keep them)
    MsmBuilder(u32 out_slot, const std::vector<int>& t2e) : tab2ext(t2e) { std::memset(&d, 0, sizeof d); d.out_slot = (u16)out_slot; }
    void add_ext(u32 ext_slot) { d.flags |= MSM_ADD_EXT; d.add_ext = (u16)ext_slot; }
    void var(u32 table_slot, ScalarSrc s, bool neg = false) {
        if (d.nvar >= MAX_VAR_TERMS) throw std::length_error("too many variable-base terms");
        VarTerm& t = d.var[d.nvar++]; t.table_slot = (u16)table_slot; t.neg = neg; t.s = s;
        t.ext_slot = (u16)(table_slot < tab2ext.size() ? tab2ext[table_slot] : -1); t.pad = 0;
    }
    void con(u32 ctab, ScalarSrc s, bool neg = false) {
        if (d.ncon >= MAX_CONST_TERMS) throw std::length_error("too many constant-base terms");
        ConstTerm& t = d.con[d.ncon++]; t.ctab = (u16)ctab; t.neg = neg; t.s = s;
    }
};

// A job with constant bases only runs on the comb tables (64 mixed adds per term, no doublings) when that beats the ladder:
// verify paths, public digits: 252 shared doublings + 16..22 wide-table adds per term, i.e. fewer than 5 terms;
// prover paths, secret digits: the ladder also needs 64 scanned adds per term, so the comb always saves the 252 doublings, but its
// scans walk 48 KiB per generator instead of 768 B; measured on 4 attributes (7-term commitments: issue 4.35 -> 4.64 M/s), so the
// limit is set just above that (fewer than 9 terms).
inline void mark_comb_jobs(ShapeProgram& P) {
    const u32 limit = P.is_issue ? 9 : 5;
    for (MsmDesc& d : P.msms) if (d.nvar == 0 && d.ncon > 0 && d.ncon < limit && !(d.flags & MSM_ADD_W)) d.flags |= MSM_COMB;
}

// Fold the hole-free leading blocks into a midstate, append the rest to the program.
inline void finish_transcript(ShapeProgram& P, TxBuilder& tb, u32 chal_field, u32 out_slot) {
    TxDesc d; std::memset(&d, 0, sizeof d);
    u32 first_hole_block = tb.holes.empty() ? (u32)tb.blocks.size() - 1 : tb.holes.front().block;
    if (first_hole_block > tb.blocks.size() - 1) first_hole_block = (u32)tb.blocks.size() - 1;  // keep >= 1 block on the device
    u64 st[25]; for (int i = 0; i < 25; i++) st[i] = 0;
    for (u32 b = 0; b < first_hole_block; b++) {
        for (int i = 0; i < 21; i++) { u64 lane; std::memcpy(&lane, tb.blocks[b].data() + 8 * i, 8); st[i] ^= lane; }
        keccak_f1600(st);
    }
    for (int i = 0; i < 25; i++) d.midstate[i] = st[i];
    d.block_ofs = (u32)(P.lanes.size() / 21);
    d.nblocks = (u32)tb.blocks.size() - first_hole_block;
    for (u32 b = first_hole_block; b < tb.blocks.size(); b++)
        for (int i = 0; i < 21; i++) { u64 lane; std::memcpy(&lane, tb.blocks[b].data() + 8 * i, 8); P.lanes.push_back(lane); }
    d.hole_ofs = (u32)P.holes.size(); d.nholes = (u32)tb.holes.size();
    for (TxHole h : tb.holes) { h.block = (u16)(h.block - first_hole_block); P.holes.push_back(h); }
    d.id_ofs = (u32)P.ids.size(); d.nid = (u32)tb.ids.size();
    for (const TxIdCheck& c : tb.ids) P.ids.push_back(c);
    d.chal_field = (u16)chal_field; d.out_slot = (u16)out_slot;
    P.txs.push_back(d);
}

// BatchableProof mode: the constraints of a compiled shape as inputs of one random linear combination per chunk (engine.cuh, RLC section)
inline void build_rlc(ShapeProgram& P) {
    RlcDesc R; std::memset(&R, 0, sizeof R);
    u32 ni = 0, nt = 0;
    if (P.cmp_pairs.size() > RLC_MAX_CONS) throw std::length_error("too many constraints");
    for (size_t j = 0; j < P.cmp_pairs.size(); j++) {
        const MsmDesc& m = P.msms[P.cmp_pairs[j].commit_slot];
        R.first_input[j] = (u16)ni; R.first_cterm[j] = (u16)nt;
        if (ni + m.nvar + 1 > RLC_MAX_INPUTS || nt + m.ncon > RLC_MAX_CTERMS) throw std::length_error("too many RLC terms");
        for (u32 k = 0; k < m.nvar; k++) {
            if (m.var[k].ext_slot == 0xffff) throw std::logic_error("ladder base without extended coordinates");
            R.in_ext[ni] = m.var[k].ext_slot; R.in_neg[ni] = m.var[k].neg; R.in_s[ni] = m.var[k].s; ni++;
        }
        R.in_ext[ni] = P.commit_ext[j]; R.in_neg[ni] = 1; R.in_s[ni].op = 0xffff; ni++;      // - rho * R_wire
        for (u32 k = 0; k < m.ncon; k++) { R.ct_ctab[nt] = m.con[k].ctab; R.ct_neg[nt] = m.con[k].neg; R.ct_s[nt] = m.con[k].s; nt++; }
    }
    R.ncons = (u16)P.cmp_pairs.size(); R.ninputs = (u16)ni; R.ncterms = (u16)nt;
    R.first_input[R.ncons] = (u16)ni; R.first_cterm[R.ncons] = (u16)nt;
    P.rlc.push_back(R);
}

// ---- program builder: the slot counters and descriptor appends of every compiler ---------------------------------------------
enum : u32 { W_TABLE = 1, W_ATAB = 2, W_EXT = 4, W_COMP = 8, W_COMPNEG = 16 };   // the slots a point job writes
struct ProgramBuilder {
    ShapeProgram P;
    u32 n_tables = 0, n_atabs = 0, n_ext = 0, n_comp = 0, n_msm = 0;
    std::vector<int> tab2ext;   // extended-coordinates slot of each ladder table's base, -1 = none

    u32 table(int ext_slot = -1) { tab2ext.push_back(ext_slot); return n_tables++; }
    u32 atab() { return n_atabs++; }
    u32 ext() { return n_ext++; }
    u32 comp() { return n_comp++; }
    struct Slots { int table, atab, ext, comp, compneg; };
    // A BatchableProof verifier keeps every ladder base in extended coordinates too: its RLC path adds the bases themselves, not table entries.
    Slots point(int field_a, int field_b, u32 op, u32 want) {
        if (P.batchable && (want & W_TABLE)) want |= W_EXT;
        Slots o;
        o.ext = (want & W_EXT) ? (int)ext() : -1;
        o.table = (want & W_TABLE) ? (int)table(o.ext) : -1;
        o.atab = (want & W_ATAB) ? (int)atab() : -1;
        o.comp = (want & W_COMP) ? (int)comp() : -1;
        o.compneg = (want & W_COMPNEG) ? (int)comp() : -1;
        PointJob j; j.field_a = (int16_t)field_a; j.field_b = (int16_t)field_b; j.op = (u16)op; j.atab_slot = (int16_t)o.atab;
        j.table_slot = (int16_t)o.table; j.ext_slot = (int16_t)o.ext; j.comp_slot = (int16_t)o.comp; j.compneg_slot = (int16_t)o.compneg;
        P.point_jobs.push_back(j);
        return o;
    }
    // a derived scalar; returns its scalar ref
    u32 derive(u32 op, u32 a, u32 b, u32 c = 0) {
        DeriveOp d; d.op = (u16)op; d.a = (u16)a; d.b = (u16)b; d.c = (u16)c; P.derived.push_back(d);
        return sref_derived((u32)P.derived.size() - 1);
    }
    u32 wide(u32 lo) { return derive(DV_WIDE, lo, lo + 1); }
    // an MSM whose terms `terms` adds; returns its commit slot
    template <class F> u32 msm(F&& terms) { MsmBuilder m(n_msm, tab2ext); terms(m); P.msms.push_back(m.d); return n_msm++; }
    // a prover's output: n words per item, each placed by word() exactly once
    void outputs(u32 n) { OutWord unset; unset.kind = 0xffff; unset.a = unset.b = unset.c = 0; P.out_words.assign(n, unset); }
    void word(u32 pos, u32 kind, u32 a, u32 b = 0, u32 c = 0) { OutWord& o = P.out_words.at(pos); o.kind = (u16)kind; o.a = (u16)a; o.b = (u16)b; o.c = (u16)c; }
    ShapeProgram finish() {
        for (const OutWord& o : P.out_words) if (o.kind == 0xffff) throw std::logic_error("output word not written");
        if (P.batchable)   // wire commitments must decode (verify_batchable decompresses them); their extended form feeds the RLC path
            for (const CmpPair& cp : P.cmp_pairs) { P.commit_ext.push_back((u16)n_ext); point(cp.field, -1, PJ_COPY, W_EXT); }
        P.n_tables = n_tables; P.n_atabs = n_atabs; P.n_ext = n_ext; P.n_comp = n_comp; P.n_msm = n_msm; P.n_proofs = (u32)P.txs.size();
        mark_comb_jobs(P);
        if (P.batchable) build_rlc(P);
        return std::move(P);
    }
};

// ---- statements: constraint order, wire layout and transcript schedule, shared by each prover and its verifier ------------------
// How one side of a proof drives its transcript: the verifier checks its allocated points for the identity; the BatchableProof verifier
// absorbs the wire commitments at commit_field + k (and compares each with its recomputed slot) instead of its recomputed ones;
// chal_field is the wire challenge the verifier compares (0xffff = none).
struct TxSide { bool check_ids; int commit_field; u32 chal_field; };
// f = the proof's first wire word: the challenge, or in the BatchableProof form the first commitment
inline TxSide verifier_side(bool batchable, u32 f) { return batchable ? TxSide{true, (int)f, 0xffff} : TxSide{true, -1, f}; }
inline TxSide prover_side() { return TxSide{false, -1, 0xffff}; }

// The proof's blinding commitments in constraint order, the challenge, and the finished template.
inline void finish_proof(ShapeProgram& P, TxBuilder& tb, const char* const* labels, const u32* slots, size_t ncons, const TxSide& side, u32 proof) {
    for (size_t k = 0; k < ncons; k++) {
        if (side.commit_field >= 0) {
            const u32 f = (u32)side.commit_field + (u32)k;
            tb.blinding_commitment_wire(labels[k], f);
            CmpPair cp; cp.commit_slot = (u16)slots[k]; cp.field = (u16)f; P.cmp_pairs.push_back(cp);
        } else tb.blinding_commitment(labels[k], slots[k]);
        P.dump_commit.push_back(slots[k]);
    }
    tb.challenge();
    finish_transcript(P, tb, side.chal_field, proof);
}

// ProofOfValidCredential's constraints in the order zkp allocates them (presentation.rs:416-433): Z, C_x_1, the C_y constraints of the
// compacted-index loop (SURVEY A.6.1: i runs over the count of non-hidden-plaintext attributes and indexes kinds, G_y and G_m, while the
// commitment is the i-th entry of the compacted C_y list) and, in a linked presentation, C_y[i] - C_y_1 = z * (G_y[i] - G_y[0]) for each
// hidden plaintext at an index i > 0.  kinds is not validated: a byte other than 3 is not a hidden plaintext, as the C ABI counters take it.
enum : u32 { CON_Z, CON_CX1, CON_CY, CON_LINK };
struct MainConstraint {
    u32 type, attr;     // attr: the attribute whose G_y (and G_m) the constraint uses
    u32 cy;             // CON_CY: the attribute whose C_y the constraint proves
    int m;              // CON_CY: the index of attr's response among m[h_s] if attr is a hidden scalar, else -1
    const char* label;
};
inline std::vector<MainConstraint> presentation_constraints(u32 n, const uint8_t* kinds, bool linked) {
    std::vector<MainConstraint> cons{{CON_Z, 0, 0, -1, "Z"}, {CON_CX1, 0, 0, -1, "C_x_1"}};
    std::vector<u32> nsp;   // the compacted C_y list: the attributes that are not hidden plaintexts
    for (u32 i = 0; i < n; i++) if (kinds[i] != 3) nsp.push_back(i);
    int m = 0;              // hidden scalars before attribute i
    for (u32 i = 0; i < nsp.size(); i++) {
        if (kinds[i] != 3) cons.push_back({CON_CY, i, nsp[i], kinds[i] == 1 ? m : -1, "C_y"});
        m += kinds[i] == 1;
    }
    if (linked) for (u32 i = 1; i < n; i++) if (kinds[i] == 3) cons.push_back({CON_LINK, i, 0, -1, "C_y-C_y_1"});
    return cons;
}
// ProofOfEncryption's constraints (encryption.rs:154-210) and ProofOfIssuance's (issuance.rs:195-215), in order.
inline constexpr const char* ENC_CONSTRAINTS[5] = {"pk", "C_y_1-E2", "C_y_2'", "E1", "C_y_3"};
inline constexpr const char* ISSUANCE_CONSTRAINTS[3] = {"C_W", "I", "V"};

// The presentation wire layout of include/aeonflux_b200.h: the challenge, responses z, z_0, t, m[h_s], C_x_0, C_x_1, C_V, C_y[n], the revealed
// attributes (kinds 0 and 2) in attribute order, then one block per hidden plaintext: challenge, responses a, a0, a1, m3, z, z1, pk, E1, E2,
// C_y_1, C_y_2, C_y_3, C_y_2'.  The BatchableProof form replaces each challenge word by that proof's commitments in constraint order.
// kinds is not validated here either.
struct PresentationLayout {
    struct Enc { u32 attr, chal, resp, pk, e1, e2, cy1, cy2, cy3, cy2p; };   // chal: the challenge or the first commitment
    u32 hs = 0, chal = 0, resp = 0, cx0 = 0, cx1 = 0, cv = 0, cy = 0, size = 0;
    std::vector<int> rev;   // [n] field of each revealed attribute, -1 for the others
    std::vector<Enc> enc;   // one block per hidden plaintext, in attribute order
};
inline PresentationLayout presentation_layout(u32 n, const uint8_t* kinds, bool batchable) {
    PresentationLayout L; L.rev.assign(n, -1);
    for (u32 i = 0; i < n; i++) L.hs += kinds[i] == 1;
    u32 f = batchable ? (u32)presentation_constraints(n, kinds, false).size() : 1;
    L.resp = f; f += 3 + L.hs;
    L.cx0 = f++; L.cx1 = f++; L.cv = f++; L.cy = f; f += n;
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0 || kinds[i] == 2) L.rev[i] = (int)f++;
    for (u32 i = 0; i < n; i++) if (kinds[i] == 3) {
        PresentationLayout::Enc e; e.attr = i; e.chal = f; f += batchable ? (u32)std::size(ENC_CONSTRAINTS) : 1;
        e.resp = f; f += 6;
        e.pk = f++; e.e1 = f++; e.e2 = f++; e.cy1 = f++; e.cy2 = f++; e.cy3 = f++; e.cy2p = f++;
        L.enc.push_back(e);
    }
    L.size = f;
    return L;
}
inline size_t presentation_num_fields(u32 n, const uint8_t* kinds) { return presentation_layout(n, kinds, false).size; }
inline size_t batchable_num_fields(u32 n, const uint8_t* kinds) { return presentation_layout(n, kinds, true).size; }
// the recomputed commitments of a presentation: the main proof's, then those of each proof of encryption
inline size_t presentation_num_commitments(u32 n, const uint8_t* kinds, bool linked) {
    return presentation_constraints(n, kinds, linked).size() + std::size(ENC_CONSTRAINTS) * presentation_layout(n, kinds, false).enc.size();
}

// The main proof's transcript (presentation.rs:355-412).  Its allocated points other than the per-issuer constants come from the caller:
// C_y and link are indexed by attribute (link: the linked attributes' C_y[i] - C_y_1 only).
struct PresentationPoints { PointSrc cx0, cx1, z; std::vector<PointSrc> cy, link; };
inline void presentation_transcript(ShapeProgram& P, const IssuerConsts& ic, u32 n, const uint8_t* kinds, const std::vector<MainConstraint>& cons,
                                    const std::vector<u32>& slots, const PresentationPoints& pt, const TxSide& side) {
    TxBuilder tb; tb.start("2019/1416 anonymous credential"); tb.domain_sep("2019/1416 presentation proof");
    tb.scalar_var("z"); tb.scalar_var("z_0"); tb.scalar_var("t");
    for (u32 i = 0; i < n; i++) if (kinds[i] == 1) tb.scalar_var("m");
    tb.point_var_const("I", ic.enc[ic.id_I()].data());
    tb.point_var("C_x_1", pt.cx1, side.check_ids); tb.point_var("C_x_0", pt.cx0, side.check_ids);
    tb.point_var_const("G_x_0", ic.enc[ic.id_Gx0()].data()); tb.point_var_const("G_x_1", ic.enc[ic.id_Gx1()].data());
    for (u32 i = 0; i < n; i++) if (kinds[i] != 3) tb.point_var("C_y", pt.cy[i], side.check_ids);
    for (u32 i = 0; i < ic.ny; i++) tb.point_var_const("G_y", ic.enc[ic.id_Gy(i)].data());
    for (u32 i = 0; i < n; i++) if (kinds[i] == 1) tb.point_var_const("G_m", ic.enc[ic.id_Gm(i)].data());
    for (const MainConstraint& c : cons)
        if (c.type == CON_LINK) { tb.point_var_const("G_y-G_y_1", ic.enc_link.at(c.attr).data()); tb.point_var("C_y-C_y_1", pt.link[c.attr], side.check_ids); }
    tb.point_var("Z", pt.z, side.check_ids);
    std::vector<const char*> labels;
    for (const MainConstraint& c : cons) labels.push_back(c.label);
    finish_proof(P, tb, labels.data(), slots.data(), cons.size(), side, 0);
}

// A proof of encryption's transcript (encryption.rs:154-210) for the hidden plaintext at attribute attr; d = C_y_1 - E2.
struct EncryptionPoints { PointSrc pk, cy2, cy3, cy2p, d, e1, neg_e1; };
inline void encryption_transcript(ShapeProgram& P, const IssuerConsts& ic, u32 attr, const EncryptionPoints& pt, const u32* slots, const TxSide& side, u32 proof) {
    TxBuilder tb; tb.start("2019/1416 anonymous credentials"); tb.domain_sep("2019/1416 proof of encryption");
    for (const char* s : {"a", "a0", "a1", "m3", "z", "z1"}) tb.scalar_var(s);
    tb.point_var("pk", pt.pk, side.check_ids);
    tb.point_var_const("G_a", ic.enc[ic.id_Ga()].data()); tb.point_var_const("G_a_0", ic.enc[ic.id_Ga0()].data());
    tb.point_var_const("G_a_1", ic.enc[ic.id_Ga1()].data());
    tb.point_var_const("G_y_1", ic.enc[ic.id_Gy(0)].data()); tb.point_var_const("G_y_2", ic.enc[ic.id_Gy(1)].data());
    tb.point_var_const("G_y_3", ic.enc[ic.id_Gy(2)].data()); tb.point_var_const("G_m_3", ic.enc[ic.id_Gm(attr)].data());
    tb.point_var("C_y_2", pt.cy2, side.check_ids); tb.point_var("C_y_3", pt.cy3, side.check_ids); tb.point_var("C_y_2'", pt.cy2p, side.check_ids);
    tb.point_var("C_y_1-E2", pt.d, side.check_ids);
    tb.point_var("E1", pt.e1, side.check_ids);
    tb.point_var("-E1", pt.neg_e1, side.check_ids);
    finish_proof(P, tb, ENC_CONSTRAINTS, slots, std::size(ENC_CONSTRAINTS), side, proof);
}

// The issuance wire layout: attribute[n], t, U, V, the challenge (BatchableProof form: the commitments C_W, I, V), responses w, w', x_0,
// x_1, y[n], 1 (issuance.rs:146-159).
struct IssuanceLayout { u32 t, u, v, chal, resp, size; };
inline IssuanceLayout issuance_layout(u32 n, bool batchable) {
    IssuanceLayout L; L.t = n; L.u = n + 1; L.v = n + 2; L.chal = n + 3;
    L.resp = L.chal + (batchable ? (u32)std::size(ISSUANCE_CONSTRAINTS) : 1); L.size = L.resp + n + 5;
    return L;
}
inline size_t issuance_num_fields(u32 n) { return issuance_layout(n, false).size; }
inline size_t issuance_batchable_num_fields(u32 n) { return issuance_layout(n, true).size; }

// The issuance proof's transcript (issuance.rs:160-190); m = M_i per attribute.
struct IssuancePoints { PointSrc u, v, tu; std::vector<PointSrc> m; };
inline void issuance_transcript(ShapeProgram& P, const IssuerConsts& ic, u32 n, const IssuancePoints& pt, const u32* slots, const TxSide& side) {
    TxBuilder tb; tb.start("2019/1416 anonymous credential"); tb.domain_sep("2019/1416 issuance proof");
    tb.scalar_var("w"); tb.scalar_var("w'"); tb.scalar_var("x_0"); tb.scalar_var("x_1");
    for (u32 i = 0; i < n; i++) tb.scalar_var("y");
    tb.scalar_var("1");
    tb.point_var_const("G_V", ic.enc[ic.id_GV()].data()); tb.point_var_const("G_w", ic.enc[ic.id_Gw()].data());
    tb.point_var_const("G_w_prime", ic.enc[ic.id_Gwp()].data());
    tb.point_var_const("-G_x_0", ic.enc_neg[ic.id_Gx0()].data()); tb.point_var_const("-G_x_1", ic.enc_neg[ic.id_Gx1()].data());
    for (u32 i = 0; i < ic.ny; i++) tb.point_var_const("-G_y", ic.enc_neg[ic.id_Gy(i)].data());
    tb.point_var_const("C_W", ic.enc[ic.id_CW()].data()); tb.point_var_const("I", ic.enc[ic.id_I()].data());
    tb.point_var("U", pt.u, side.check_ids); tb.point_var("V", pt.v, side.check_ids); tb.point_var("tU", pt.tu, side.check_ids);
    for (u32 i = 0; i < n; i++) tb.point_var("M", pt.m[i], side.check_ids);
    finish_proof(P, tb, ISSUANCE_CONSTRAINTS, slots, std::size(ISSUANCE_CONSTRAINTS), side, 0);
}

// ProofOfValidCredential::verify as a program (presentation.rs:324-443).  batchable = the same statement verified from a
// BatchableProof (zkp verify_batchable): each challenge word of the layout is replaced by that proof's blinding commitments.
// linked = the opt-in statement that ties each proof of encryption to the credential proof (the DLEQ the reference leaves as a
// TODO, README.md:119-122, presentation.rs:292; oracle/pyoracle/aeonflux.py:presentation_prove spells the statement out): per hidden
// plaintext at index i > 0 two more allocated points, G_y[i] - G_y[0] ("G_y-G_y_1", a per-issuer constant) and C_y[i] - C_y_1
// ("C_y-C_y_1"), after the G_m points and before Z, and the constraint C_y[i] - C_y_1 = z * (G_y[i] - G_y[0]) after the C_y constraints
// (evaluated over the existing generators: z*G_y[i] - z*G_y[0] - c*D); at index 0 the two wire words must be equal.  Same wire layout.
inline ShapeProgram compile_presentation(const IssuerConsts& ic, u32 n, const uint8_t* kinds, bool batchable = false, bool linked = false) {
    if (n != ic.n || n == 0 || n > MAX_ATTRS) throw std::invalid_argument("attribute count does not match the issuer's");
    for (u32 i = 0; i < n; i++) if (kinds[i] > 3) throw std::invalid_argument("bad attribute kind");
    if (batchable && linked) throw std::invalid_argument("the linked statement is only built for compact proofs");
    ProgramBuilder B; ShapeProgram& P = B.P;
    P.batchable = batchable;
    const PresentationLayout L = presentation_layout(n, kinds, batchable);
    const std::vector<MainConstraint> cons = presentation_constraints(n, kinds, linked);
    P.n_fields = L.size;
    if (!batchable) P.scalar_fields.push_back((u16)L.chal);
    for (u32 k = 0; k < 3 + L.hs; k++) P.scalar_fields.push_back((u16)(L.resp + k));
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) P.scalar_fields.push_back((u16)L.rev[i]);
    for (const PresentationLayout::Enc& b : L.enc) {
        if (!batchable) P.scalar_fields.push_back((u16)b.chal);
        for (u32 k = 0; k < 6; k++) P.scalar_fields.push_back((u16)(b.resp + k));
    }

    // ---- point jobs
    // C_x_0, C_x_1: bases of the aMAC ladder (transposed copy) and of the C_x_1 constraint (standard table)
    const ProgramBuilder::Slots s_cx0 = B.point((int)L.cx0, -1, PJ_COPY, W_TABLE | W_ATAB), s_cx1 = B.point((int)L.cx1, -1, PJ_COPY, W_TABLE | W_ATAB);
    const int E_CV = B.point((int)L.cv, -1, PJ_COPY, W_EXT).ext;
    std::vector<int> T_CY(n, -1), A_X(n, -1);   // A_X[i]: aMAC table of X_i (presentation.rs:344-350)
    for (u32 i = 0; i < n; i++) {
        if (kinds[i] == 2) {
            T_CY[i] = B.point((int)(L.cy + i), -1, PJ_COPY, W_TABLE).table;
            A_X[i] = B.point((int)(L.cy + i), L.rev[i], PJ_ADD, W_ATAB).atab;                       // X_i = C_y[i] + M_i (:348)
        } else {
            const ProgramBuilder::Slots o = B.point((int)(L.cy + i), -1, PJ_COPY, (kinds[i] == 3 ? 0u : (u32)W_TABLE) | W_ATAB);   // a hidden point's C_y is only a ladder base
            T_CY[i] = o.table; A_X[i] = o.atab;
        }
    }
    P.n_point_jobs_amac = (u32)P.point_jobs.size();
    std::vector<ProgramBuilder::Slots> s_pk, s_e1, s_cy2, s_cy3, s_cy2p, s_d;
    for (const PresentationLayout::Enc& b : L.enc) {
        s_pk.push_back(B.point((int)b.pk, -1, PJ_COPY, W_TABLE));
        s_e1.push_back(B.point((int)b.e1, -1, PJ_COPY, W_TABLE | W_COMPNEG));                           // E1 and compress(-E1) (encryption.rs:184-185)
        s_cy2.push_back(B.point((int)b.cy2, -1, PJ_COPY, W_TABLE));
        s_cy3.push_back(B.point((int)b.cy3, -1, PJ_COPY, W_TABLE));
        s_cy2p.push_back(B.point((int)b.cy2p, -1, PJ_COPY, W_TABLE));
        s_d.push_back(B.point((int)b.cy1, (int)b.e2, PJ_SUB, W_TABLE | W_COMP));                        // C_y_1 - E2 (encryption.rs:183)
    }
    // linked statement: D_i = C_y[i] - C_y_1 of hidden plaintext i > 0 (ladder base + encoding); at index 0 an equality check
    std::vector<ProgramBuilder::Slots> s_link(n);
    if (linked)
        for (const PresentationLayout::Enc& b : L.enc) {
            if (b.attr == 0) { CmpPair cp; cp.commit_slot = (u16)(0x8000u | L.cy); cp.field = (u16)b.cy1; P.eq_fields.push_back(cp); continue; }
            s_link[b.attr] = B.point((int)(L.cy + b.attr), (int)b.cy1, PJ_SUB, W_TABLE | W_COMP);
        }
    // ---- aMAC (presentation.rs:342-352)
    P.has_amac = true;
    AmacDesc& A = P.amac; std::memset(&A, 0, sizeof A);
    A.ext_cv = (u16)E_CV;
    A.var[A.nvar].atab_slot = (u16)s_cx0.atab; A.var[A.nvar++].digit_row = (u16)sec_x0();
    A.var[A.nvar].atab_slot = (u16)s_cx1.atab; A.var[A.nvar++].digit_row = (u16)sec_x1();
    for (u32 i = 0; i < n; i++) {
        A.var[A.nvar].atab_slot = (u16)A_X[i]; A.var[A.nvar++].digit_row = (u16)sec_y(i);
        if (kinds[i] == 0) { AmacPs& p = A.ps[A.nps++]; p.ctab = (u16)ic.id_Gm(i); p.y_row = (u16)sec_y(i); p.field_m = (u16)L.rev[i]; p.pad = 0; }  // (:346)
    }
    const int E_Z = batchable ? (int)B.ext() : -1;
    const u32 T_Z = B.table(E_Z), C_Z = B.comp();
    A.out_table_slot = (u16)T_Z; A.out_comp_slot = (u16)C_Z; A.out_ext_slot = (u16)E_Z; P.z_comp_slot = C_Z;

    // ---- main proof: constraints (:416-433) and transcript (:355-412)
    const ScalarSrc R_z = sc_field(L.resp + 0), R_z0 = sc_field(L.resp + 1), R_t = sc_field(L.resp + 2),
                    C_main = batchable ? sc_field(SREF_CHAL | 0) : sc_field(L.chal);
    std::vector<u32> slots;
    for (const MainConstraint& k : cons)
        slots.push_back(B.msm([&](MsmBuilder& m) {
            switch (k.type) {
                case CON_Z: m.con(ic.id_I(), R_z); m.var(T_Z, C_main, true); break;
                case CON_CX1: m.var((u32)s_cx0.table, R_t); m.con(ic.id_Gx0(), R_z0); m.con(ic.id_Gx1(), R_z); m.var((u32)s_cx1.table, C_main, true); break;
                case CON_CY:
                    m.con(ic.id_Gy(k.attr), R_z);
                    if (k.m >= 0) m.con(ic.id_Gm(k.attr), sc_field(L.resp + 3 + (u32)k.m));
                    m.var((u32)T_CY[k.cy], C_main, true);
                    break;
                default: m.con(ic.id_Gy(k.attr), R_z); m.con(ic.id_Gy(0), R_z, true); m.var((u32)s_link[k.attr].table, C_main, true);
            }
        }));
    PresentationPoints pt{{SRC_FIELD, L.cx0}, {SRC_FIELD, L.cx1}, {SRC_COMP, C_Z}, {}, {}};
    for (u32 i = 0; i < n; i++) { pt.cy.push_back({SRC_FIELD, L.cy + i}); pt.link.push_back({SRC_COMP, (u32)s_link[i].comp}); }
    presentation_transcript(P, ic, n, kinds, cons, slots, pt, verifier_side(batchable, L.chal));
    // ---- proofs of encryption (encryption.rs:154-210), one per hidden plaintext attribute (presentation.rs:438-440)
    for (size_t e = 0; e < L.enc.size(); e++) {
        const PresentationLayout::Enc& b = L.enc[e];
        const ScalarSrc c = batchable ? sc_field(SREF_CHAL | (u32)(1 + e)) : sc_field(b.chal), r_a = sc_field(b.resp), r_a0 = sc_field(b.resp + 1),
                        r_a1 = sc_field(b.resp + 2), r_m3 = sc_field(b.resp + 3), r_z = sc_field(b.resp + 4), r_z1 = sc_field(b.resp + 5);
        const u32 T_PK = (u32)s_pk[e].table, T_E1 = (u32)s_e1[e].table, T_CY2 = (u32)s_cy2[e].table, T_CY3 = (u32)s_cy3[e].table,
                  T_CY2P = (u32)s_cy2p[e].table, T_D = (u32)s_d[e].table;
        const u32 eslots[5] = {
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Ga(), r_a); m.con(ic.id_Ga0(), r_a0); m.con(ic.id_Ga1(), r_a1); m.var(T_PK, c, true); }),
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(0), r_z); m.var(T_E1, r_a, true); m.var(T_D, c, true); }),
            B.msm([&](MsmBuilder& m) { m.var(T_CY2, r_a1); m.var(T_CY2P, c, true); }),
            B.msm([&](MsmBuilder& m) { m.var(T_CY2, r_a0); m.var(T_CY2P, r_m3); m.con(ic.id_Gy(1), r_z1); m.var(T_E1, c, true); }),
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(2), r_z); m.con(ic.id_Gm(b.attr), r_m3); m.var(T_CY3, c, true); })};
        const EncryptionPoints ept{{SRC_FIELD, b.pk}, {SRC_FIELD, b.cy2}, {SRC_FIELD, b.cy3}, {SRC_FIELD, b.cy2p},
                                   {SRC_COMP, (u32)s_d[e].comp}, {SRC_FIELD, b.e1}, {SRC_COMP, (u32)s_e1[e].compneg}};
        encryption_transcript(P, ic, b.attr, ept, eslots, verifier_side(batchable, b.chal), (u32)(1 + e));
    }
    if (!batchable) {   // longest point jobs first, so that the short ones fill the tail of the k_points grid (slots are already assigned)
        auto cost = [](const PointJob& j) {
            return 13 * (j.op == PJ_COPY ? 1 : 2) + ((j.table_slot >= 0 || j.atab_slot >= 0) ? 4 : 0) + 13 * ((j.comp_slot >= 0) + (j.compneg_slot >= 0));
        };
        std::stable_sort(P.point_jobs.begin(), P.point_jobs.end(), [&](const PointJob& a, const PointJob& b) { return cost(a) > cost(b); });
    }
    return B.finish();
}

// CredentialIssuance::verify as a program (issuer.rs:48-57 -> issuance.rs:132-218).
// kinds: 0 = scalar attribute (M_i = m_i * G_m[i]), 2 = point attribute.  Fields: the issuance layout (issuance_layout).
// batchable = the same statement verified from a BatchableProof (the commented-out BatchVerifier of issuance.rs:21-22).
inline ShapeProgram compile_issuance_verify(const IssuerConsts& ic, u32 n, const uint8_t* kinds, bool batchable = false) {
    if (n != ic.n || n == 0 || n > MAX_ATTRS) throw std::invalid_argument("attribute count does not match the issuer's");
    for (u32 i = 0; i < n; i++) if (kinds[i] != 0 && kinds[i] != 2) throw std::invalid_argument("bad request kind");
    ProgramBuilder B; ShapeProgram& P = B.P;
    P.batchable = batchable;
    const IssuanceLayout L = issuance_layout(n, batchable);
    P.n_fields = L.size;
    const u32 R_w = L.resp, R_wp = L.resp + 1, R_x0 = L.resp + 2, R_x1 = L.resp + 3, R_y = L.resp + 4, R_one = L.resp + 4 + n;
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) P.scalar_fields.push_back((u16)i);
    P.scalar_fields.push_back((u16)L.t);
    if (!batchable) P.scalar_fields.push_back((u16)L.chal);
    for (u32 k = 0; k < n + 5; k++) P.scalar_fields.push_back((u16)(L.resp + k));
    // PJ_KEEP_TABLE: U's ladder table feeds tU = t*U, which the transcript absorbs -- it is needed even when the random-linear-combination
    // pass skips the other tables
    const u32 T_U = (u32)B.point((int)L.u, -1, PJ_COPY | PJ_KEEP_TABLE, W_TABLE).table, T_V = (u32)B.point((int)L.v, -1, PJ_COPY, W_TABLE).table;
    std::vector<int> T_M(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 2) T_M[i] = B.point((int)i, -1, PJ_COPY, W_TABLE).table;
    const ScalarSrc c = batchable ? sc_field(SREF_CHAL | 0) : sc_field(L.chal);
    // derived allocated points that are not inputs: tU = t*U (:180) and M_i = m_i * G_m[i] for scalar attributes (:184)
    const u32 S_tU = B.msm([&](MsmBuilder& m) { m.var(T_U, sc_field(L.t)); });
    P.pre_msms.push_back(S_tU);
    std::vector<u32> S_M(n, 0);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) { S_M[i] = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gm(i), sc_field(i)); }); P.pre_msms.push_back(S_M[i]); }
    // constraints (:195-215)
    const u32 slots[3] = {
        B.msm([&](MsmBuilder& m) { m.con(ic.id_Gw(), sc_field(R_w)); m.con(ic.id_Gwp(), sc_field(R_wp)); m.con(ic.id_CW(), c, true); }),
        B.msm([&](MsmBuilder& m) {
            m.con(ic.id_GV(), sc_field(R_one)); m.con(ic.id_Gx0(), sc_field(R_x0), true); m.con(ic.id_Gx1(), sc_field(R_x1), true);
            for (u32 i = 0; i < n; i++) m.con(ic.id_Gy(i), sc_field(R_y + i), true);
            m.con(ic.id_I(), c, true);
        }),
        B.msm([&](MsmBuilder& m) {
            m.con(ic.id_Gw(), sc_field(R_w));
            m.var(T_U, sc_muladd3(R_x0, R_x1, L.t));               // x_0*U + x_1*(t*U) = (x_0 + x_1*t)*U
            for (u32 i = 0; i < n; i++) {
                if (kinds[i] == 0) m.con(ic.id_Gm(i), sc_mul2(R_y + i, i));  // y_i * (m_i*G_m[i])
                else m.var((u32)T_M[i], sc_field(R_y + i));
            }
            m.var(T_V, c, true);
        })};
    IssuancePoints pt{{SRC_FIELD, L.u}, {SRC_FIELD, L.v}, {SRC_COMMIT, S_tU}, {}};
    for (u32 i = 0; i < n; i++) pt.m.push_back(kinds[i] == 0 ? PointSrc{SRC_COMMIT, S_M[i]} : PointSrc{SRC_FIELD, i});
    issuance_transcript(P, ic, n, pt, slots, verifier_side(batchable, L.chal));
    return B.finish();
}


// Issuer::issue as a program (issuer.rs:111-124: Amac::tag amacs.rs:276-294 + ProofOfIssuance::prove issuance.rs:40-129),
// with the rng output supplied by the caller.  kinds: 0 = scalar attribute, 2 = point attribute.
// Fields: attr[n], then two 32-byte words (the 64 rng bytes) per random value: t, U, blinding[n+5] in the order the
// witnesses are allocated (w, w', x_0, x_1, y[n], "1"; issuance.rs:52-68).  Output words: the issuance layout from t on (the
// attributes in front of it are the request's own), compact or, with batchable, as zkp's prove_batchable returns the proof: the
// commitments in place of the challenge.  The transcript and the responses do not change.
inline size_t issue_num_fields(u32 n) { return (size_t)n + 2 * ((size_t)n + 7); }
inline ShapeProgram compile_issue(const IssuerConsts& ic, u32 n, const uint8_t* kinds, bool batchable = false) {
    if (n != ic.n || n == 0 || n > MAX_ATTRS) throw std::invalid_argument("attribute count does not match the issuer's");  // amacs.rs:285-287
    for (u32 i = 0; i < n; i++) if (kinds[i] != 0 && kinds[i] != 2) throw std::invalid_argument("bad request kind");
    ProgramBuilder B; ShapeProgram& P = B.P; P.is_issue = true;
    const u32 F_ATTR = 0, F_TSEED = n, F_USEED = n + 2, F_BSEED = n + 4;
    P.n_fields = (u32)issue_num_fields(n);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) P.scalar_fields.push_back((u16)(F_ATTR + i));
    const u32 D_t = B.wide(F_TSEED);
    std::vector<u32> D_b(n + 5);   // blindings of w, w', x_0, x_1, y[n], "1"
    for (u32 k = 0; k < n + 5; k++) D_b[k] = B.wide(F_BSEED + 2 * k);
    const u32 S_x0 = sref_secret(sec_x0()), S_x1 = sref_secret(sec_x1());
    // points: U = from_uniform(seed) with its ladder table and encoding; one ladder table per point attribute.  Every lookup
    // on this path is a constant-address scan, so the tables only exist in the warp-transposed layout (table_slot of a
    // variable term = transposed slot).
    const ProgramBuilder::Slots s_u = B.point((int)F_USEED, (int)(F_USEED + 1), PJ_UNIFORM, W_ATAB | W_COMP);
    const u32 T_U = (u32)s_u.atab;
    std::vector<int> T_M(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 2) T_M[i] = B.point((int)(F_ATTR + i), -1, PJ_COPY, W_ATAB).atab;
    // M_i = m_i * G_m[i] (amacs.rs:234-235), tU = t * U (issuance.rs:91)
    std::vector<u32> S_M(n, 0);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) S_M[i] = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gm(i), sc_field(F_ATTR + i)); });
    const u32 S_tU = B.msm([&](MsmBuilder& m) { m.var(T_U, sc_field(D_t)); });
    // V = W + x_0*U + (x_1*t)*U + sum y_i*M_i (amacs.rs:267-270), as one ladder: (x_0 + x_1*t)*U + sum (y_i*m_i)*G_m[i] + sum y_i*M_i, then + W
    const u32 S_V = B.msm([&](MsmBuilder& m) {
        m.d.flags = MSM_ADD_W;
        m.var(T_U, sc_muladd3(S_x0, S_x1, D_t));
        for (u32 i = 0; i < n; i++) {
            if (kinds[i] == 0) m.con(ic.id_Gm(i), sc_mul2(sref_secret(sec_y(i)), F_ATTR + i));
            else m.var((u32)T_M[i], sc_field(sref_secret(sec_y(i))));
        }
    });
    // blinding commitments of the three constraints (issuance.rs:106-126; zkp prove_compact)
    const u32 slots[3] = {
        B.msm([&](MsmBuilder& m) { m.con(ic.id_Gw(), sc_field(D_b[0])); m.con(ic.id_Gwp(), sc_field(D_b[1])); }),
        B.msm([&](MsmBuilder& m) {
            m.con(ic.id_GV(), sc_field(D_b[4 + n])); m.con(ic.id_Gx0(), sc_field(D_b[2]), true); m.con(ic.id_Gx1(), sc_field(D_b[3]), true);
            for (u32 i = 0; i < n; i++) m.con(ic.id_Gy(i), sc_field(D_b[4 + i]), true);
        }),
        B.msm([&](MsmBuilder& m) {
            m.con(ic.id_Gw(), sc_field(D_b[0]));
            m.var(T_U, sc_muladd3(D_b[2], D_b[3], D_t));                                   // b_x0*U + b_x1*(t*U)
            for (u32 i = 0; i < n; i++) {
                if (kinds[i] == 0) m.con(ic.id_Gm(i), sc_mul2(D_b[4 + i], F_ATTR + i));      // b_y_i * (m_i*G_m[i])
                else m.var((u32)T_M[i], sc_field(D_b[4 + i]));
            }
        })};
    IssuancePoints pt{{SRC_COMP, (u32)s_u.comp}, {SRC_COMMIT, S_V}, {SRC_COMMIT, S_tU}, {}};
    for (u32 i = 0; i < n; i++) pt.m.push_back(kinds[i] == 0 ? PointSrc{SRC_COMMIT, S_M[i]} : PointSrc{SRC_FIELD, F_ATTR + i});
    issuance_transcript(P, ic, n, pt, slots, prover_side());
    const IssuanceLayout L = issuance_layout(n, batchable);
    const u32 o = L.t;
    B.outputs(L.size - o);
    B.word(L.t - o, OW_DERIVED, D_t & SREF_MASK); B.word(L.u - o, OW_COMP, (u32)s_u.comp); B.word(L.v - o, OW_COMMIT, S_V);
    if (batchable) for (u32 k = 0; k < 3; k++) B.word(L.chal - o + k, OW_COMMIT, slots[k]);
    else B.word(L.chal - o, OW_CHAL, 0);
    const u32 wit[4] = {sref_secret(2 + n), sref_secret(3 + n), S_x0, S_x1};   // w, w', x_0, x_1, then y[n] and the witness "1"
    for (u32 k = 0; k < n + 5; k++) B.word(L.resp - o + k, OW_RESP, 0, k < 4 ? wit[k] : k < 4 + n ? sref_secret(sec_y(k - 4)) : 0xffff, D_b[k]);
    return B.finish();
}

// AnonymousCredential::show as a program (credential.rs:37-46 -> ProofOfValidCredential::prove presentation.rs:139-321 and, per
// hidden plaintext attribute, ProofOfEncryption::prove encryption.rs:58-142 with Keypair::encrypt symmetric.rs:252-261),
// with the rng output supplied by the caller.  The user-side batch operation: it needs no issuer secret.
// kinds = the presentation's attribute kinds (0 revealed scalar, 1 hidden scalar, 2 revealed point, 3 hidden plaintext).
// Fields: t, U, V, then per attribute: scalar m_i (kinds 0/1) | point M_i (kind 2) | plaintext M1, M2, m3 (kind 3);
//         then a, a0, a1, pk of the symmetric keypair (only if some kind is 3); then two 32-byte words (64 rng bytes) per
//         random value: z, the main proof's 3 + h_s blindings, then 6 blindings per hidden plaintext.
// Output words: the presentation layout (presentation_layout), compact or, with batchable, as zkp's prove_batchable returns the proofs:
// the commitments in place of each challenge.  The challenges are still derived: the responses need them.  Like compile_presentation,
// the linked statement has no batchable form.
// Every commitment is rewritten over the per-issuer generators and the *input* points (U, M2): e.g. the blinding commitment
// b_t*C_x_0 + b_z0*G_x_0 + b_z*G_x_1 with C_x_0 = z*G_x_0 + U becomes (b_z0 + b_t*z)*G_x_0 + b_z*G_x_1 + b_t*U, so no ladder
// has to wait for another ladder's output and every job of an item runs in one launch.
inline size_t show_num_fields(u32 n, const uint8_t* kinds) {
    size_t f = 3, hs = 0, hp = 0;
    for (u32 i = 0; i < n; i++) { f += kinds[i] == 3 ? 3 : 1; hs += kinds[i] == 1; hp += kinds[i] == 3; }
    return f + (hp ? 4 : 0) + 2 + 2 * (3 + hs) + 12 * hp;
}
inline ShapeProgram compile_show(const IssuerConsts& ic, u32 n, const uint8_t* kinds, bool linked = false, bool batchable = false) {
    if (n != ic.n || n == 0 || n > MAX_ATTRS) throw std::invalid_argument("attribute count does not match the issuer's");
    for (u32 i = 0; i < n; i++) if (kinds[i] > 3) throw std::invalid_argument("bad attribute kind");
    if (batchable && linked) throw std::invalid_argument("the linked statement is only built for compact proofs");
    ProgramBuilder B; ShapeProgram& P = B.P; P.is_issue = true;
    const PresentationLayout L = presentation_layout(n, kinds, batchable);
    const std::vector<MainConstraint> cons = presentation_constraints(n, kinds, linked);
    const u32 hs = L.hs, hp = (u32)L.enc.size();
    // ---- field map
    const u32 F_T = 0, F_U = 1, F_V = 2;
    u32 f = 3;
    std::vector<u32> F_ATTR(n);
    for (u32 i = 0; i < n; i++) { F_ATTR[i] = f; f += kinds[i] == 3 ? 3 : 1; }
    u32 F_A = 0, F_A0 = 0, F_A1 = 0, F_PK = 0;
    if (hp) { F_A = f++; F_A0 = f++; F_A1 = f++; F_PK = f++; }
    const u32 F_ZSEED = f; f += 2;
    const u32 F_BSEED = f; f += 2 * (3 + hs);
    const u32 F_EBSEED = f; f += 12 * hp;
    P.n_fields = f;
    P.scalar_fields.push_back((u16)F_T);
    for (u32 i = 0; i < n; i++) { if (kinds[i] <= 1) P.scalar_fields.push_back((u16)F_ATTR[i]); if (kinds[i] == 3) P.scalar_fields.push_back((u16)(F_ATTR[i] + 2)); }
    if (hp) for (u32 k : {F_A, F_A0, F_A1}) P.scalar_fields.push_back((u16)k);
    // ---- derived scalars
    const u32 D_z = B.wide(F_ZSEED);
    const u32 D_z0 = B.derive(DV_NEGMUL, F_T, D_z);                                // z_0 = -t*z (presentation.rs:163)
    const u32 D_bz = B.wide(F_BSEED), D_bz0 = B.wide(F_BSEED + 2), D_bt = B.wide(F_BSEED + 4);
    std::vector<u32> D_bm(hs);
    for (u32 k = 0; k < hs; k++) D_bm[k] = B.wide(F_BSEED + 6 + 2 * k);
    const u32 D_g0 = B.derive(DV_MULADD, D_bz0, D_bt, D_z);                         // b_z0 + b_t*z
    // ---- points
    const ProgramBuilder::Slots s_u = B.point((int)F_U, -1, PJ_COPY, W_ATAB | W_EXT);
    const u32 A_U = (u32)s_u.atab, E_V = (u32)B.point((int)F_V, -1, PJ_COPY, W_EXT).ext;
    std::vector<int> E_M1(n, -1), A_M2(n, -1), E_M2(n, -1);
    for (u32 i = 0; i < n; i++) {
        if (kinds[i] == 2) B.point((int)F_ATTR[i], -1, PJ_COPY, 0);     // revealed point: only has to decode
        if (kinds[i] == 3) {
            E_M1[i] = B.point((int)F_ATTR[i], -1, PJ_COPY, W_EXT).ext;
            const ProgramBuilder::Slots o = B.point((int)(F_ATTR[i] + 1), -1, PJ_COPY, W_ATAB | W_EXT); A_M2[i] = o.atab; E_M2[i] = o.ext;
        }
    }
    if (hp) B.point((int)F_PK, -1, PJ_COPY, 0);
    // ---- ladders (every scalar is a user secret: constant-schedule jobs; a variable term's table_slot is its transposed table)
    auto R = [](u32 ref) { return sc_field(ref); };
    const u32 S_CX0 = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gx0(), R(D_z)); m.add_ext((u32)s_u.ext); });         // C_x_0 = z*G_x_0 + U   (:181)
    const u32 S_CX1 = B.msm([&](MsmBuilder& m) { m.var(A_U, R(F_T)); m.con(ic.id_Gx1(), R(D_z)); });               // C_x_1 = z*G_x_1 + t*U (:182)
    const u32 S_CV = B.msm([&](MsmBuilder& m) { m.con(ic.id_GV(), R(D_z)); m.add_ext(E_V); });                     // C_V = z*G_V + V       (:183)
    std::vector<u32> S_CY(n);
    for (u32 i = 0; i < n; i++)                                                                                      // (:169-180)
        S_CY[i] = B.msm([&](MsmBuilder& m) {
            m.con(ic.id_Gy(i), R(D_z));
            if (kinds[i] == 1) m.con(ic.id_Gm(i), R(F_ATTR[i]));
            if (kinds[i] == 3) m.add_ext((u32)E_M1[i]);
        });
    // the constraints' blinding commitments; Z = z*I (:184) and, linked, D_i = C_y[i] - C_y_1 = z*G_y[i] - z*G_y[0] just before theirs
    u32 S_Z = 0;
    std::vector<u32> S_D(n, 0), slots;
    for (const MainConstraint& k : cons) {
        switch (k.type) {
            case CON_Z:
                S_Z = B.msm([&](MsmBuilder& m) { m.con(ic.id_I(), R(D_z)); });
                slots.push_back(B.msm([&](MsmBuilder& m) { m.con(ic.id_I(), R(D_bz)); }));
                break;
            case CON_CX1: slots.push_back(B.msm([&](MsmBuilder& m) { m.var(A_U, R(D_bt)); m.con(ic.id_Gx0(), R(D_g0)); m.con(ic.id_Gx1(), R(D_bz)); })); break;
            case CON_CY:
                slots.push_back(B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(k.attr), R(D_bz)); if (k.m >= 0) m.con(ic.id_Gm(k.attr), R(D_bm[(u32)k.m])); }));
                break;
            default:
                S_D[k.attr] = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(k.attr), R(D_z)); m.con(ic.id_Gy(0), R(D_z), true); });
                slots.push_back(B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(k.attr), R(D_bz)); m.con(ic.id_Gy(0), R(D_bz), true); }));
        }
    }
    PresentationPoints pt{{SRC_COMMIT, S_CX0}, {SRC_COMMIT, S_CX1}, {SRC_COMMIT, S_Z}, {}, {}};
    for (u32 i = 0; i < n; i++) { pt.cy.push_back({SRC_COMMIT, S_CY[i]}); pt.link.push_back({SRC_COMMIT, S_D[i]}); }
    presentation_transcript(P, ic, n, kinds, cons, slots, pt, prover_side());
    B.outputs(L.size);
    if (batchable) for (u32 k = 0; k < slots.size(); k++) B.word(L.chal + k, OW_COMMIT, slots[k]);
    else B.word(L.chal, OW_CHAL, 0);
    B.word(L.resp, OW_RESP, 0, D_z, D_bz); B.word(L.resp + 1, OW_RESP, 0, D_z0, D_bz0); B.word(L.resp + 2, OW_RESP, 0, F_T, D_bt);
    for (u32 i = 0, k = 0; i < n; i++) if (kinds[i] == 1) { B.word(L.resp + 3 + k, OW_RESP, 0, F_ATTR[i], D_bm[k]); k++; }
    B.word(L.cx0, OW_COMMIT, S_CX0); B.word(L.cx1, OW_COMMIT, S_CX1); B.word(L.cv, OW_COMMIT, S_CV);
    for (u32 i = 0; i < n; i++) B.word(L.cy + i, OW_COMMIT, S_CY[i]);
    for (u32 i = 0; i < n; i++) if (L.rev[i] >= 0) B.word((u32)L.rev[i], OW_FIELD, F_ATTR[i]);
    // ---- proofs of encryption, one per hidden plaintext (presentation.rs:293-309 -> encryption.rs:58-142)
    for (u32 e = 0; e < hp; e++) {
        const PresentationLayout::Enc& b = L.enc[e];
        const u32 idx = b.attr, F_M3 = F_ATTR[idx] + 2, AM2 = (u32)A_M2[idx], EM1 = (u32)E_M1[idx], EM2 = (u32)E_M2[idx];
        const u32 D_u = B.derive(DV_MULADD, F_A0, F_A1, F_M3);                    // a0 + a1*m3 (symmetric.rs:257)
        const u32 D_au = B.derive(DV_MUL, F_A, D_u);
        const u32 D_z1 = B.derive(DV_NEGMUL, D_z, D_u);                            // z1 = -z*(a0 + a1*m3) (encryption.rs:78)
        const u32 D_a1z = B.derive(DV_MUL, F_A1, D_z);
        const u32 B0 = F_EBSEED + 12 * e;
        const u32 D_ba = B.wide(B0), D_ba0 = B.wide(B0 + 2), D_ba1 = B.wide(B0 + 4), D_bm3 = B.wide(B0 + 6), D_bze = B.wide(B0 + 8), D_bz1 = B.wide(B0 + 10);
        const u32 D_bau = B.derive(DV_MUL, D_ba, D_u);
        const u32 D_ba1z = B.derive(DV_MUL, D_ba1, D_z);
        const u32 D_s1 = B.derive(DV_MULADD, D_ba0, D_bm3, F_A1);                  // b_a0 + b_m3*a1
        const u32 D_s2 = B.derive(DV_MULADD, D_bz1, D_s1, D_z);                    // b_z1 + (b_a0 + b_m3*a1)*z
        const u32 S_E1 = B.msm([&](MsmBuilder& m) { m.var(AM2, R(D_u)); });                                                 // E1 = (a0 + a1*m3)*M2
        const u32 S_E2 = B.msm([&](MsmBuilder& m) { m.var(AM2, R(D_au)); m.add_ext(EM1); });                                // E2 = a*E1 + M1
        const u32 S_CY1 = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(0), R(D_z)); m.add_ext(EM1); });                        // C_y_1 = z*G_y[0] + M1
        const u32 S_CY2 = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(1), R(D_z)); m.add_ext(EM2); });                        // C_y_2 = z*G_y[1] + M2
        const u32 S_CY3 = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(2), R(D_z)); m.con(ic.id_Gm(idx), R(F_M3)); });         // C_y_3 = z*G_y[2] + m3*G_m[idx]
        const u32 S_CY2P = B.msm([&](MsmBuilder& m) { m.var(AM2, R(F_A1)); m.con(ic.id_Gy(1), R(D_a1z)); });                // C_y_2' = a1*C_y_2
        const u32 S_ED = B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(0), R(D_z)); m.var(AM2, R(D_au), true); });              // C_y_1 - E2 (M1 cancels)
        const u32 S_NE1 = B.msm([&](MsmBuilder& m) { m.var(AM2, R(D_u), true); });                                          // -E1
        const u32 eslots[5] = {
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Ga(), R(D_ba)); m.con(ic.id_Ga0(), R(D_ba0)); m.con(ic.id_Ga1(), R(D_ba1)); }),
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(0), R(D_bze)); m.var(AM2, R(D_bau), true); }),                   // b_z*G_y_1 + b_a*(-E1)
            B.msm([&](MsmBuilder& m) { m.var(AM2, R(D_ba1)); m.con(ic.id_Gy(1), R(D_ba1z)); }),                        // b_a1*C_y_2
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(1), R(D_s2)); m.var(AM2, R(D_s1)); }),                           // b_a0*C_y_2 + b_m3*C_y_2' + b_z1*G_y_2
            B.msm([&](MsmBuilder& m) { m.con(ic.id_Gy(2), R(D_bze)); m.con(ic.id_Gm(idx), R(D_bm3)); })};
        const EncryptionPoints ept{{SRC_FIELD, F_PK}, {SRC_COMMIT, S_CY2}, {SRC_COMMIT, S_CY3}, {SRC_COMMIT, S_CY2P},
                                   {SRC_COMMIT, S_ED}, {SRC_COMMIT, S_E1}, {SRC_COMMIT, S_NE1}};
        encryption_transcript(P, ic, idx, ept, eslots, prover_side(), 1 + e);
        if (batchable) for (u32 k = 0; k < 5; k++) B.word(b.chal + k, OW_COMMIT, eslots[k]);
        else B.word(b.chal, OW_CHAL, 1 + e);
        const u32 wit[6] = {F_A, F_A0, F_A1, F_M3, D_z, D_z1}, bl[6] = {D_ba, D_ba0, D_ba1, D_bm3, D_bze, D_bz1};
        for (u32 k = 0; k < 6; k++) B.word(b.resp + k, OW_RESP, 1 + e, wit[k], bl[k]);
        B.word(b.pk, OW_FIELD, F_PK);
        B.word(b.e1, OW_COMMIT, S_E1); B.word(b.e2, OW_COMMIT, S_E2); B.word(b.cy1, OW_COMMIT, S_CY1);
        B.word(b.cy2, OW_COMMIT, S_CY2); B.word(b.cy3, OW_COMMIT, S_CY3); B.word(b.cy2p, OW_COMMIT, S_CY2P);
    }
    return B.finish();
}

// Keypair::encrypt (symmetric.rs:252-261) as a program: the two ladders of show's proof of encryption (compile_show),
//     E1 = (a0 + a1*m3)*M2,   E2 = (a*(a0 + a1*m3))*M2 + M1.
// Fields: the Plaintext M1, M2, m3.  The keypair a, a0, a1 is the call's: the pass puts it in the secret rows (ws.secsc) 0, 1, 2.
// Output words: E1, E2.  Every scalar is secret (constant-schedule ladders); the derived scalars are wiped after each pass.
inline ShapeProgram compile_encrypt() {
    ProgramBuilder B; ShapeProgram& P = B.P; P.is_issue = true;
    const u32 F_M1 = 0, F_M2 = 1, F_M3 = 2;
    P.n_fields = 3;
    P.scalar_fields.push_back((u16)F_M3);
    const u32 D_u = B.derive(DV_MULADD, sref_secret(1), sref_secret(2), F_M3);      // a0 + a1*m3
    const u32 D_au = B.derive(DV_MUL, sref_secret(0), D_u);
    const u32 E_M1 = (u32)B.point((int)F_M1, -1, PJ_COPY, W_EXT).ext, A_M2 = (u32)B.point((int)F_M2, -1, PJ_COPY, W_ATAB).atab;
    B.outputs(2);
    B.word(0, OW_COMMIT, B.msm([&](MsmBuilder& m) { m.var(A_M2, sc_field(D_u)); }));
    B.word(1, OW_COMMIT, B.msm([&](MsmBuilder& m) { m.var(A_M2, sc_field(D_au)); m.add_ext(E_M1); }));
    return B.finish();
}

// Keypair::derive (symmetric.rs:197-215) as a program: pk = a*G_a + a0*G_a0 + a1*G_a1 over the context's system parameters, one MSM of
// constant bases with secret scalars, which mark_comb_jobs puts on the radix-16 comb (constant-address scans).
// Fields: a, a0, a1, the rows the hashes of keypair_scalars_job (engine.cuh) leave.  Output words: a, a0, a1, pk -- the 128-byte
// keypair afx_show takes.
inline ShapeProgram compile_keypair(const IssuerConsts& ic) {
    ProgramBuilder B; ShapeProgram& P = B.P; P.is_issue = true;
    P.n_fields = 3;
    const u32 S_PK = B.msm([&](MsmBuilder& m) { m.con(ic.id_Ga(), sc_field(0)); m.con(ic.id_Ga0(), sc_field(1)); m.con(ic.id_Ga1(), sc_field(2)); });
    B.outputs(4);
    for (u32 k = 0; k < 3; k++) B.word(k, OW_FIELD, k);
    B.word(3, OW_COMMIT, S_PK);
    return B.finish();
}

}  // namespace afx
