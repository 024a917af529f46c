// Host-side "shape compiler": turns an attribute-kind vector into the stage descriptors engine.cuh executes.
//
// It restates, as data, the statement structure of
//   ProofOfValidCredential::verify   /root/reference/src/nizk/presentation.rs:324-443
//   ProofOfEncryption::verify        /root/reference/src/nizk/encryption.rs:154-210
//   ProofOfIssuance::verify          /root/reference/src/nizk/issuance.rs:132-218
// and of the zkp 0.7 toolbox / merlin framing they drive (SURVEY A.3-A.5): which points are allocated under which
// labels and in which order, which constraints exist, and every quirk of SURVEY A.6 (compacted-index constraint loop,
// G_y padded to >= 3, singular/plural transcript labels, identity rejection only for allocated points).
// Pure byte/bookkeeping work: no field arithmetic happens on the host.
#pragma once
#include <algorithm>
#include <array>
#include <cstring>
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
    void point_var(const char* label, u32 kind, u32 idx, bool check_identity = true) {
        if (check_identity) { TxIdCheck c; c.src_kind = (u16)kind; c.src_idx = (u16)idx; ids.push_back(c); }
        append_message("ptvar", label, std::strlen(label));
        append_header("val", 32); begin_op(2, false); absorb_hole(kind, idx);
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
    explicit MsmBuilder(u32 out_slot) { std::memset(&d, 0, sizeof d); d.out_slot = (u16)out_slot; }
    void add_ext(u32 ext_slot) { d.flags |= MSM_ADD_EXT; d.add_ext = (u16)ext_slot; }
    const std::vector<int>* tab2ext = nullptr;   // batchable mode: extended-coordinates slot of each table's base
    void var(u32 table_slot, ScalarSrc s, bool neg = false) {
        if (d.nvar >= MAX_VAR_TERMS) throw std::length_error("too many variable-base terms");
        VarTerm& t = d.var[d.nvar++]; t.table_slot = (u16)table_slot; t.neg = neg; t.s = s;
        t.ext_slot = (u16)((tab2ext && table_slot < tab2ext->size()) ? (*tab2ext)[table_slot] : 0xffff); t.pad = 0;
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

inline size_t presentation_num_fields(u32 n, const uint8_t* kinds) {
    size_t hs = 0, r = 0, hp = 0;
    for (u32 i = 0; i < n; i++) { hs += kinds[i] == 1; r += (kinds[i] == 0 || kinds[i] == 2); hp += kinds[i] == 3; }
    return 1 + 3 + hs + 3 + n + r + 14 * hp;
}

inline size_t presentation_num_main_constraints(u32 n, const uint8_t* kinds) {
    size_t nsp = 0, cons = 2;
    for (u32 i = 0; i < n; i++) nsp += kinds[i] != 3;
    for (size_t i = 0; i < nsp; i++) cons += kinds[i] != 3;
    return cons;
}
inline size_t batchable_num_fields(u32 n, const uint8_t* kinds) {
    size_t hp = 0; for (u32 i = 0; i < n; i++) hp += kinds[i] == 3;
    return presentation_num_fields(n, kinds) - 1 + presentation_num_main_constraints(n, kinds) + 4 * hp;
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
    ShapeProgram P;
    // ---- field map
    u32 hs = 0; std::vector<int> ss_rank(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 1) ss_rank[i] = (int)hs++;
    P.batchable = batchable;
    const u32 nc_main = (u32)presentation_num_main_constraints(n, kinds), ENC_SH = batchable ? 4 : 0;
    u32 f = 0;
    const u32 F_CHAL = f; f += batchable ? nc_main : 1;      // the challenge, or the main proof's commitments
    const u32 F_RESP = f; f += 3 + hs;
    const u32 F_CX0 = f++, F_CX1 = f++, F_CV = f++; const u32 F_CY = f; f += n;
    std::vector<int> F_REV(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0 || kinds[i] == 2) F_REV[i] = (int)f++;
    std::vector<u32> enc_base, enc_attr;
    for (u32 i = 0; i < n; i++) if (kinds[i] == 3) { enc_base.push_back(f); enc_attr.push_back(i); f += 14 + ENC_SH; }
    P.n_fields = f;
    if (!batchable) P.scalar_fields.push_back((u16)F_CHAL);
    for (u32 k = 0; k < 3 + hs; k++) P.scalar_fields.push_back((u16)(F_RESP + k));
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) P.scalar_fields.push_back((u16)F_REV[i]);
    for (u32 b : enc_base) for (u32 k = batchable ? 5 : 0; k < 7 + ENC_SH; k++) P.scalar_fields.push_back((u16)(b + k));

    // ---- point jobs
    u32 ntab = 0, natab = 0, next = 0, ncomp = 0;
    enum : u32 { W_TABLE = 1, W_ATAB = 2, W_EXT = 4, W_COMP = 8, W_COMPNEG = 16 };
    struct Slots { int table = -1, atab = -1, ext = -1, comp = -1, compneg = -1; };
    std::vector<int> tab2ext;
    auto job = [&](int fa, int fb, u32 op, u32 want) {
        if (batchable && (want & W_TABLE)) want |= W_EXT;            // the RLC path adds the bases themselves, not table entries
        Slots o;
        PointJob j; j.field_a = (int16_t)fa; j.field_b = (int16_t)fb; j.op = (u16)op;
        j.table_slot = (int16_t)(o.table = (want & W_TABLE) ? (int)ntab++ : -1);
        j.atab_slot = (int16_t)(o.atab = (want & W_ATAB) ? (int)natab++ : -1);
        j.ext_slot = (int16_t)(o.ext = (want & W_EXT) ? (int)next++ : -1);
        j.comp_slot = (int16_t)(o.comp = (want & W_COMP) ? (int)ncomp++ : -1);
        j.compneg_slot = (int16_t)(o.compneg = (want & W_COMPNEG) ? (int)ncomp++ : -1);
        if (o.table >= 0) { tab2ext.resize((size_t)o.table + 1, -1); tab2ext[(size_t)o.table] = o.ext; }
        P.point_jobs.push_back(j);
        return o;
    };
    // C_x_0, C_x_1: bases of the aMAC ladder (transposed copy) and of the C_x_1 constraint (standard table)
    const Slots s_cx0 = job((int)F_CX0, -1, PJ_COPY, W_TABLE | W_ATAB), s_cx1 = job((int)F_CX1, -1, PJ_COPY, W_TABLE | W_ATAB);
    const int T_CX0 = s_cx0.table, T_CX1 = s_cx1.table;
    const int E_CV = job((int)F_CV, -1, PJ_COPY, W_EXT).ext;
    std::vector<int> T_CY(n, -1), A_X(n, -1);   // A_X[i]: aMAC table of X_i (presentation.rs:344-350)
    for (u32 i = 0; i < n; i++) {
        if (kinds[i] == 2) {
            T_CY[i] = job((int)(F_CY + i), -1, PJ_COPY, W_TABLE).table;
            A_X[i] = job((int)(F_CY + i), F_REV[i], PJ_ADD, W_ATAB).atab;                        // X_i = C_y[i] + M_i (:348)
        } else {
            Slots o = job((int)(F_CY + i), -1, PJ_COPY, (kinds[i] == 3 ? 0u : (u32)W_TABLE) | W_ATAB);   // a hidden point's C_y is only a ladder base
            T_CY[i] = o.table; A_X[i] = o.atab;
        }
    }
    P.n_point_jobs_amac = (u32)P.point_jobs.size();
    struct EncSlots { int T_PK, T_E1, C_NEG_E1, T_CY2, T_CY3, T_CY2P, T_D, C_D; };
    std::vector<EncSlots> es(enc_base.size());
    for (size_t e = 0; e < enc_base.size(); e++) {
        u32 b = enc_base[e];
        b += ENC_SH;                                                                              // the point words sit 4 further in the batchable layout
        es[e].T_PK = job((int)(b + 7), -1, PJ_COPY, W_TABLE).table;
        { Slots o = job((int)(b + 8), -1, PJ_COPY, W_TABLE | W_COMPNEG); es[e].T_E1 = o.table; es[e].C_NEG_E1 = o.compneg; }  // E1 and compress(-E1) (encryption.rs:184-185)
        es[e].T_CY2 = job((int)(b + 11), -1, PJ_COPY, W_TABLE).table;
        es[e].T_CY3 = job((int)(b + 12), -1, PJ_COPY, W_TABLE).table;
        es[e].T_CY2P = job((int)(b + 13), -1, PJ_COPY, W_TABLE).table;
        { Slots o = job((int)(b + 10), (int)(b + 9), PJ_SUB, W_TABLE | W_COMP); es[e].T_D = o.table; es[e].C_D = o.comp; }    // C_y_1 - E2 (encryption.rs:183)
    }
    // linked statement: D_i = C_y[i] - C_y_1 of hidden plaintext i > 0 (ladder base + encoding); at index 0 an equality check
    struct LinkSlots { u32 attr; int T_D, C_D; };
    std::vector<LinkSlots> links;
    if (linked)
        for (size_t e = 0; e < enc_base.size(); e++) {
            const u32 idx = enc_attr[e], f_cy1 = enc_base[e] + 10;
            if (idx == 0) { CmpPair cp; cp.commit_slot = (u16)(0x8000u | (F_CY + 0)); cp.field = (u16)f_cy1; P.eq_fields.push_back(cp); continue; }
            Slots o = job((int)(F_CY + idx), (int)f_cy1, PJ_SUB, W_TABLE | W_COMP);
            links.push_back({idx, o.table, o.comp});
        }
    // ---- aMAC (presentation.rs:342-352)
    P.has_amac = true;
    AmacDesc& A = P.amac; std::memset(&A, 0, sizeof A);
    A.ext_cv = (u16)E_CV;
    A.var[A.nvar].atab_slot = (u16)s_cx0.atab; A.var[A.nvar++].digit_row = (u16)sec_x0();
    A.var[A.nvar].atab_slot = (u16)s_cx1.atab; A.var[A.nvar++].digit_row = (u16)sec_x1();
    for (u32 i = 0; i < n; i++) {
        A.var[A.nvar].atab_slot = (u16)A_X[i]; A.var[A.nvar++].digit_row = (u16)sec_y(i);
        if (kinds[i] == 0) { AmacPs& p = A.ps[A.nps++]; p.ctab = (u16)ic.id_Gm(i); p.y_row = (u16)sec_y(i); p.field_m = (u16)F_REV[i]; p.pad = 0; }  // (:346)
    }
    const u32 T_Z = ntab++; const u32 C_Z = ncomp++;
    A.out_table_slot = (u16)T_Z; A.out_comp_slot = (u16)C_Z; P.z_comp_slot = C_Z;
    A.out_ext_slot = 0xffff;
    if (batchable) { A.out_ext_slot = (u16)next; tab2ext.resize((size_t)T_Z + 1, -1); tab2ext[T_Z] = (int)next++; }
    // wire commitments must decode (verify_batchable decompresses them); their extended form feeds the RLC path
    std::vector<u32> F_COMMITS;     // every commitment field, main proof first, constraint order
    if (batchable) {
        for (u32 k = 0; k < nc_main; k++) F_COMMITS.push_back(F_CHAL + k);
        for (u32 b : enc_base) for (u32 k = 0; k < 5; k++) F_COMMITS.push_back(b + k);
        for (u32 fc : F_COMMITS) { P.commit_ext.push_back((u16)next); job((int)fc, -1, PJ_COPY, W_EXT); }
    }
    P.n_tables = ntab; P.n_atabs = natab; P.n_ext = next; P.n_comp = ncomp;

    // ---- main proof: constraints (:416-433) and transcript (:355-412)
    const ScalarSrc R_z = sc_field(F_RESP + 0), R_z0 = sc_field(F_RESP + 1), R_t = sc_field(F_RESP + 2),
                    C_main = batchable ? sc_field(SREF_CHAL | 0) : sc_field(F_CHAL);
    const std::vector<int>* t2e = batchable ? &tab2ext : nullptr;
    std::vector<u32> nsp;  // original indices of the non-SecretPoint attributes (the compacted C_y list)
    for (u32 i = 0; i < n; i++) if (kinds[i] != 3) nsp.push_back(i);
    u32 slot = 0;
    struct Con { u32 slot; const char* label; };
    std::vector<Con> main_cons;
    { MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_I(), R_z); m.var(T_Z, C_main, true); P.msms.push_back(m.d); main_cons.push_back({slot++, "Z"}); }
    { MsmBuilder m(slot); m.tab2ext = t2e; m.var(T_CX0, R_t); m.con(ic.id_Gx0(), R_z0); m.con(ic.id_Gx1(), R_z); m.var(T_CX1, C_main, true);
      P.msms.push_back(m.d); main_cons.push_back({slot++, "C_x_1"}); }
    for (u32 i = 0; i < nsp.size(); i++) {  // compacted-index loop: i indexes kinds / G_y / G_m, nsp[i] is the commitment (SURVEY A.6.1)
        if (kinds[i] == 3) continue;
        MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_Gy(i), R_z);
        if (kinds[i] == 1) m.con(ic.id_Gm(i), sc_field(F_RESP + 3 + ss_rank[i]));
        m.var(T_CY[nsp[i]], C_main, true);
        P.msms.push_back(m.d); main_cons.push_back({slot++, "C_y"});
    }
    for (const LinkSlots& l : links) {      // C_y[i] - C_y_1 = z * (G_y[i] - G_y[0])
        MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_Gy(l.attr), R_z); m.con(ic.id_Gy(0), R_z, true); m.var((u32)l.T_D, C_main, true);
        P.msms.push_back(m.d); main_cons.push_back({slot++, "C_y-C_y_1"});
    }
    {
        TxBuilder tb; tb.start("2019/1416 anonymous credential"); tb.domain_sep("2019/1416 presentation proof");
        tb.scalar_var("z"); tb.scalar_var("z_0"); tb.scalar_var("t");
        for (u32 k = 0; k < hs; k++) tb.scalar_var("m");
        tb.point_var_const("I", ic.enc[ic.id_I()].data());
        tb.point_var("C_x_1", SRC_FIELD, F_CX1); tb.point_var("C_x_0", SRC_FIELD, F_CX0);
        tb.point_var_const("G_x_0", ic.enc[ic.id_Gx0()].data()); tb.point_var_const("G_x_1", ic.enc[ic.id_Gx1()].data());
        for (u32 i : nsp) tb.point_var("C_y", SRC_FIELD, F_CY + i);
        for (u32 i = 0; i < ic.ny; i++) tb.point_var_const("G_y", ic.enc[ic.id_Gy(i)].data());
        for (u32 i = 0; i < n; i++) if (kinds[i] == 1) tb.point_var_const("G_m", ic.enc[ic.id_Gm(i)].data());
        for (const LinkSlots& l : links) { tb.point_var_const("G_y-G_y_1", ic.enc_link.at(l.attr).data()); tb.point_var("C_y-C_y_1", SRC_COMP, (u32)l.C_D); }
        tb.point_var("Z", SRC_COMP, C_Z);
        for (size_t k = 0; k < main_cons.size(); k++) {
            const Con& c = main_cons[k];
            if (batchable) { tb.blinding_commitment_wire(c.label, F_CHAL + (u32)k); CmpPair cp; cp.commit_slot = (u16)c.slot; cp.field = (u16)(F_CHAL + k); P.cmp_pairs.push_back(cp); }
            else tb.blinding_commitment(c.label, c.slot);
            P.dump_commit.push_back(c.slot);
        }
        if (batchable && main_cons.size() != nc_main) throw std::logic_error("constraint count");
        tb.challenge();
        finish_transcript(P, tb, batchable ? 0xffff : F_CHAL, 0);
    }
    // ---- proofs of encryption (encryption.rs:154-210), one per hidden plaintext attribute (presentation.rs:438-440)
    for (size_t e = 0; e < enc_base.size(); e++) {
        const u32 b0 = enc_base[e], idx = enc_attr[e];
        const u32 b = b0 + ENC_SH;                       // responses at b+1.., points at b+7.. in either layout; commitments at b0..b0+4
        const ScalarSrc c = batchable ? sc_field(SREF_CHAL | (u32)(1 + e)) : sc_field(b0), r_a = sc_field(b + 1), r_a0 = sc_field(b + 2),
                        r_a1 = sc_field(b + 3), r_m3 = sc_field(b + 4), r_z = sc_field(b + 5), r_z1 = sc_field(b + 6);
        u32 s_pk, s_d, s_c2p, s_e1, s_c3;
        { MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_Ga(), r_a); m.con(ic.id_Ga0(), r_a0); m.con(ic.id_Ga1(), r_a1); m.var(es[e].T_PK, c, true); P.msms.push_back(m.d); s_pk = slot++; }
        { MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_Gy(0), r_z); m.var(es[e].T_E1, r_a, true); m.var(es[e].T_D, c, true); P.msms.push_back(m.d); s_d = slot++; }
        { MsmBuilder m(slot); m.tab2ext = t2e; m.var(es[e].T_CY2, r_a1); m.var(es[e].T_CY2P, c, true); P.msms.push_back(m.d); s_c2p = slot++; }
        { MsmBuilder m(slot); m.tab2ext = t2e; m.var(es[e].T_CY2, r_a0); m.var(es[e].T_CY2P, r_m3); m.con(ic.id_Gy(1), r_z1); m.var(es[e].T_E1, c, true); P.msms.push_back(m.d); s_e1 = slot++; }
        { MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_Gy(2), r_z); m.con(ic.id_Gm(idx), r_m3); m.var(es[e].T_CY3, c, true); P.msms.push_back(m.d); s_c3 = slot++; }
        TxBuilder tb; tb.start("2019/1416 anonymous credentials"); tb.domain_sep("2019/1416 proof of encryption");
        tb.scalar_var("a"); tb.scalar_var("a0"); tb.scalar_var("a1"); tb.scalar_var("m3"); tb.scalar_var("z"); tb.scalar_var("z1");
        tb.point_var("pk", SRC_FIELD, b + 7);
        tb.point_var_const("G_a", ic.enc[ic.id_Ga()].data()); tb.point_var_const("G_a_0", ic.enc[ic.id_Ga0()].data());
        tb.point_var_const("G_a_1", ic.enc[ic.id_Ga1()].data());
        tb.point_var_const("G_y_1", ic.enc[ic.id_Gy(0)].data()); tb.point_var_const("G_y_2", ic.enc[ic.id_Gy(1)].data());
        tb.point_var_const("G_y_3", ic.enc[ic.id_Gy(2)].data()); tb.point_var_const("G_m_3", ic.enc[ic.id_Gm(idx)].data());
        tb.point_var("C_y_2", SRC_FIELD, b + 11); tb.point_var("C_y_3", SRC_FIELD, b + 12); tb.point_var("C_y_2'", SRC_FIELD, b + 13);
        tb.point_var("C_y_1-E2", SRC_COMP, (u32)es[e].C_D);
        tb.point_var("E1", SRC_FIELD, b + 8);
        tb.point_var("-E1", SRC_COMP, (u32)es[e].C_NEG_E1);
        const char* enc_labels[5] = {"pk", "C_y_1-E2", "C_y_2'", "E1", "C_y_3"};
        const u32 enc_slots[5] = {s_pk, s_d, s_c2p, s_e1, s_c3};
        for (u32 k = 0; k < 5; k++) {
            if (batchable) { tb.blinding_commitment_wire(enc_labels[k], b0 + k); CmpPair cp; cp.commit_slot = (u16)enc_slots[k]; cp.field = (u16)(b0 + k); P.cmp_pairs.push_back(cp); }
            else tb.blinding_commitment(enc_labels[k], enc_slots[k]);
            P.dump_commit.push_back(enc_slots[k]);
        }
        tb.challenge();
        finish_transcript(P, tb, batchable ? 0xffff : b0, (u32)(1 + e));
    }
    P.n_msm = slot; P.n_proofs = (u32)P.txs.size();
    mark_comb_jobs(P);
    if (!batchable) {   // longest point jobs first, so that the short ones fill the tail of the k_points grid (slots are already assigned)
        auto cost = [](const PointJob& j) {
            return 13 * (j.op == PJ_COPY ? 1 : 2) + ((j.table_slot >= 0 || j.atab_slot >= 0) ? 4 : 0) + 13 * ((j.comp_slot >= 0) + (j.compneg_slot >= 0));
        };
        std::stable_sort(P.point_jobs.begin(), P.point_jobs.end(), [&](const PointJob& a, const PointJob& b) { return cost(a) > cost(b); });
    }
    if (batchable) build_rlc(P);
    return P;
}

// CredentialIssuance::verify as a program (issuer.rs:48-57 -> issuance.rs:132-218).
// kinds: 0 = scalar attribute (M_i = m_i * G_m[i]), 2 = point attribute.  Fields: attr[n], t, U, V, challenge, responses[n+5].
// batchable = the same statement verified from a BatchableProof (the commented-out BatchVerifier of issuance.rs:21-22): the
// challenge word is replaced by the three blinding commitments (constraint order C_W, I, V), i.e. 2n + 11 fields.
inline size_t issuance_num_fields(u32 n) { return 2 * (size_t)n + 9; }
inline size_t issuance_batchable_num_fields(u32 n) { return 2 * (size_t)n + 11; }
inline ShapeProgram compile_issuance_verify(const IssuerConsts& ic, u32 n, const uint8_t* kinds, bool batchable = false) {
    if (n != ic.n || n == 0 || n > MAX_ATTRS) throw std::invalid_argument("attribute count does not match the issuer's");
    for (u32 i = 0; i < n; i++) if (kinds[i] != 0 && kinds[i] != 2) throw std::invalid_argument("bad request kind");
    ShapeProgram P;
    P.batchable = batchable;
    const u32 F_ATTR = 0, F_T = n, F_U = n + 1, F_V = n + 2, F_CHAL = n + 3, F_RESP = n + 4 + (batchable ? 2 : 0);
    P.n_fields = (u32)(batchable ? issuance_batchable_num_fields(n) : issuance_num_fields(n));
    // responses: w, w', x_0, x_1, y[n], 1  (issuance.rs:146-159)
    const u32 R_w = F_RESP, R_wp = F_RESP + 1, R_x0 = F_RESP + 2, R_x1 = F_RESP + 3, R_y = F_RESP + 4, R_one = F_RESP + 4 + n;
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) P.scalar_fields.push_back((u16)(F_ATTR + i));
    P.scalar_fields.push_back((u16)F_T);
    if (!batchable) P.scalar_fields.push_back((u16)F_CHAL);
    for (u32 k = 0; k < n + 5; k++) P.scalar_fields.push_back((u16)(F_RESP + k));
    u32 ntab = 0, next = 0;
    std::vector<int> tab2ext;
    // keep_table: U's ladder table feeds tU = t*U, which the transcript absorbs -- it is needed even when the random-linear-combination
    // pass skips the other tables
    auto table_job = [&](u32 field, bool keep_table = false) {
        PointJob j; j.field_a = (int16_t)field; j.field_b = -1; j.op = (u16)(PJ_COPY | (keep_table ? PJ_KEEP_TABLE : 0)); j.atab_slot = -1; j.table_slot = (int16_t)ntab;
        j.ext_slot = (int16_t)(batchable ? (int)next++ : -1); j.comp_slot = -1; j.compneg_slot = -1; P.point_jobs.push_back(j);
        tab2ext.push_back(j.ext_slot);
        return ntab++; };
    const u32 T_U = table_job(F_U, true), T_V = table_job(F_V);
    std::vector<int> T_M(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 2) T_M[i] = (int)table_job(F_ATTR + i);
    if (batchable)       // wire commitments must decode (verify_batchable decompresses them); their extended form feeds the RLC path
        for (u32 k = 0; k < 3; k++) {
            PointJob j; j.field_a = (int16_t)(F_CHAL + k); j.field_b = -1; j.op = PJ_COPY; j.atab_slot = -1; j.table_slot = -1; j.ext_slot = (int16_t)next;
            j.comp_slot = -1; j.compneg_slot = -1; P.point_jobs.push_back(j); P.commit_ext.push_back((u16)next++);
        }
    P.n_tables = ntab; P.n_ext = next; P.n_comp = 0;
    const std::vector<int>* t2e = batchable ? &tab2ext : nullptr;
    const ScalarSrc c = batchable ? sc_field(SREF_CHAL | 0) : sc_field(F_CHAL);
    u32 slot = 0;
    // derived allocated points that are not inputs: tU = t*U (:180) and M_i = m_i * G_m[i] for scalar attributes (:184)
    u32 S_tU; { MsmBuilder m(slot); m.tab2ext = t2e; m.var(T_U, sc_field(F_T)); P.msms.push_back(m.d); P.pre_msms.push_back(slot); S_tU = slot++; }
    std::vector<int> S_M(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) { MsmBuilder m(slot); m.con(ic.id_Gm(i), sc_field(F_ATTR + i)); P.msms.push_back(m.d); P.pre_msms.push_back(slot); S_M[i] = (int)slot++; }
    // constraints (:195-215)
    u32 S_CW, S_I, S_V;
    { MsmBuilder m(slot); m.con(ic.id_Gw(), sc_field(R_w)); m.con(ic.id_Gwp(), sc_field(R_wp)); m.con(ic.id_CW(), c, true); P.msms.push_back(m.d); S_CW = slot++; }
    { MsmBuilder m(slot); m.con(ic.id_GV(), sc_field(R_one)); m.con(ic.id_Gx0(), sc_field(R_x0), true); m.con(ic.id_Gx1(), sc_field(R_x1), true);
      for (u32 i = 0; i < n; i++) m.con(ic.id_Gy(i), sc_field(R_y + i), true);
      m.con(ic.id_I(), c, true); P.msms.push_back(m.d); S_I = slot++; }
    { MsmBuilder m(slot); m.tab2ext = t2e; m.con(ic.id_Gw(), sc_field(R_w));
      m.var(T_U, sc_muladd3(R_x0, R_x1, F_T));               // x_0*U + x_1*(t*U) = (x_0 + x_1*t)*U
      for (u32 i = 0; i < n; i++) {
          if (kinds[i] == 0) m.con(ic.id_Gm(i), sc_mul2(R_y + i, F_ATTR + i));  // y_i * (m_i*G_m[i])
          else m.var((u32)T_M[i], sc_field(R_y + i));
      }
      m.var(T_V, c, true); P.msms.push_back(m.d); S_V = slot++; }
    TxBuilder tb; tb.start("2019/1416 anonymous credential"); tb.domain_sep("2019/1416 issuance proof");
    tb.scalar_var("w"); tb.scalar_var("w'"); tb.scalar_var("x_0"); tb.scalar_var("x_1");
    for (u32 i = 0; i < n; i++) tb.scalar_var("y");
    tb.scalar_var("1");
    tb.point_var_const("G_V", ic.enc[ic.id_GV()].data()); tb.point_var_const("G_w", ic.enc[ic.id_Gw()].data());
    tb.point_var_const("G_w_prime", ic.enc[ic.id_Gwp()].data());
    tb.point_var_const("-G_x_0", ic.enc_neg[ic.id_Gx0()].data()); tb.point_var_const("-G_x_1", ic.enc_neg[ic.id_Gx1()].data());
    for (u32 i = 0; i < ic.ny; i++) tb.point_var_const("-G_y", ic.enc_neg[ic.id_Gy(i)].data());
    tb.point_var_const("C_W", ic.enc[ic.id_CW()].data()); tb.point_var_const("I", ic.enc[ic.id_I()].data());
    tb.point_var("U", SRC_FIELD, F_U); tb.point_var("V", SRC_FIELD, F_V); tb.point_var("tU", SRC_COMMIT, S_tU);
    for (u32 i = 0; i < n; i++) { if (kinds[i] == 0) tb.point_var("M", SRC_COMMIT, (u32)S_M[i]); else tb.point_var("M", SRC_FIELD, F_ATTR + i); }
    const char* labels[3] = {"C_W", "I", "V"};
    const u32 slots[3] = {S_CW, S_I, S_V};
    for (u32 k = 0; k < 3; k++) {
        if (batchable) { tb.blinding_commitment_wire(labels[k], F_CHAL + k); CmpPair cp; cp.commit_slot = (u16)slots[k]; cp.field = (u16)(F_CHAL + k); P.cmp_pairs.push_back(cp); }
        else tb.blinding_commitment(labels[k], slots[k]);
        P.dump_commit.push_back(slots[k]);
    }
    tb.challenge();
    finish_transcript(P, tb, batchable ? 0xffff : F_CHAL, 0);
    P.n_msm = slot; P.n_proofs = 1;
    mark_comb_jobs(P);
    if (batchable) build_rlc(P);
    return P;
}


// Issuer::issue as a program (issuer.rs:111-124: Amac::tag amacs.rs:276-294 + ProofOfIssuance::prove issuance.rs:40-129),
// with the rng output supplied by the caller.  kinds: 0 = scalar attribute, 2 = point attribute.
// Fields: attr[n], then two 32-byte words (the 64 rng bytes) per random value: t, U, blinding[n+5] in the order the
// witnesses are allocated (w, w', x_0, x_1, y[n], "1"; issuance.rs:52-68).  Output words: t, U, V, challenge, responses[n+5].
// batchable = the same proof returned as zkp's prove_batchable returns it: the challenge word is replaced by the encodings of the
// three blinding commitments (constraint order C_W, I, V), n + 11 output words, which with attribute[n] in front is the layout
// compile_issuance_verify(..., batchable = true) takes.  The transcript and the responses do not change.
inline size_t issue_num_fields(u32 n) { return (size_t)n + 2 * ((size_t)n + 7); }
inline ShapeProgram compile_issue(const IssuerConsts& ic, u32 n, const uint8_t* kinds, bool batchable = false) {
    if (n != ic.n || n == 0 || n > MAX_ATTRS) throw std::invalid_argument("attribute count does not match the issuer's");  // amacs.rs:285-287
    for (u32 i = 0; i < n; i++) if (kinds[i] != 0 && kinds[i] != 2) throw std::invalid_argument("bad request kind");
    ShapeProgram P; P.is_issue = true;
    const u32 F_ATTR = 0, F_TSEED = n, F_USEED = n + 2, F_BSEED = n + 4;
    P.n_fields = (u32)issue_num_fields(n);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) P.scalar_fields.push_back((u16)(F_ATTR + i));
    // derived scalars: slot 0 = t, 1 + k = blinding k
    const u32 D_T = 0;
    auto D_B = [](u32 k) { return 1 + k; };
    auto wide = [&](u32 lo) { DeriveOp w; w.op = DV_WIDE; w.a = (u16)lo; w.b = (u16)(lo + 1); w.c = 0; P.derived.push_back(w); };
    wide(F_TSEED);
    for (u32 k = 0; k < n + 5; k++) wide(F_BSEED + 2 * k);
    const u32 B_w = D_B(0), B_wp = D_B(1), B_x0 = D_B(2), B_x1 = D_B(3), B_one = D_B(4 + n);
    auto B_y = [&](u32 i) { return D_B(4 + i); };
    const u32 S_w = sref_secret(2 + n), S_wp = sref_secret(3 + n), S_x0 = sref_secret(sec_x0()), S_x1 = sref_secret(sec_x1());
    (void)S_w; (void)S_wp;
    // points: U = from_uniform(seed) with its ladder table and encoding; one ladder table per point attribute.  Every lookup
    // on this path is a constant-address scan, so the tables only exist in the warp-transposed layout (table_slot of a
    // variable term = transposed slot).
    u32 ntab = 0, ncomp = 0;
    u32 T_U, C_U;
    { PointJob j; j.field_a = (int16_t)F_USEED; j.field_b = (int16_t)(F_USEED + 1); j.op = PJ_UNIFORM; j.table_slot = -1; j.atab_slot = (int16_t)(T_U = ntab++);
      j.ext_slot = -1; j.comp_slot = (int16_t)(C_U = ncomp++); j.compneg_slot = -1; P.point_jobs.push_back(j); }
    std::vector<int> T_M(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 2) {
        PointJob j; j.field_a = (int16_t)(F_ATTR + i); j.field_b = -1; j.op = PJ_COPY; j.table_slot = -1; j.atab_slot = (int16_t)(T_M[i] = (int)ntab++);
        j.ext_slot = -1; j.comp_slot = -1; j.compneg_slot = -1; P.point_jobs.push_back(j);
    }
    P.n_tables = 0; P.n_atabs = ntab; P.n_ext = 0; P.n_comp = ncomp;
    u32 slot = 0;
    auto D = [](u32 d) { return sc_field(sref_derived(d)); };
    // M_i = m_i * G_m[i] (amacs.rs:234-235), tU = t * U (issuance.rs:91)
    std::vector<int> S_M(n, -1);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0) { MsmBuilder m(slot); m.con(ic.id_Gm(i), sc_field(F_ATTR + i)); P.msms.push_back(m.d); S_M[i] = (int)slot++; }
    u32 S_tU; { MsmBuilder m(slot); m.var(T_U, D(D_T)); P.msms.push_back(m.d); S_tU = slot++; }
    // V = W + x_0*U + (x_1*t)*U + sum y_i*M_i (amacs.rs:267-270), as one ladder: (x_0 + x_1*t)*U + sum (y_i*m_i)*G_m[i] + sum y_i*M_i, then + W
    u32 S_V;
    { MsmBuilder m(slot); m.d.flags = MSM_ADD_W;
      m.var(T_U, sc_muladd3(S_x0, S_x1, sref_derived(D_T)));
      for (u32 i = 0; i < n; i++) {
          if (kinds[i] == 0) m.con(ic.id_Gm(i), sc_mul2(sref_secret(sec_y(i)), F_ATTR + i));
          else m.var((u32)T_M[i], sc_field(sref_secret(sec_y(i))));
      }
      P.msms.push_back(m.d); S_V = slot++; }
    // blinding commitments of the three constraints (issuance.rs:106-126; zkp prove_compact)
    u32 S_CW, S_I, S_CV;
    { MsmBuilder m(slot); m.con(ic.id_Gw(), D(B_w)); m.con(ic.id_Gwp(), D(B_wp)); P.msms.push_back(m.d); S_CW = slot++; }
    { MsmBuilder m(slot); m.con(ic.id_GV(), D(B_one)); m.con(ic.id_Gx0(), D(B_x0), true); m.con(ic.id_Gx1(), D(B_x1), true);
      for (u32 i = 0; i < n; i++) m.con(ic.id_Gy(i), D(B_y(i)), true);
      P.msms.push_back(m.d); S_I = slot++; }
    { MsmBuilder m(slot); m.con(ic.id_Gw(), D(B_w));
      m.var(T_U, sc_muladd3(sref_derived(B_x0), sref_derived(B_x1), sref_derived(D_T)));      // b_x0*U + b_x1*(t*U)
      for (u32 i = 0; i < n; i++) {
          if (kinds[i] == 0) m.con(ic.id_Gm(i), sc_mul2(sref_derived(B_y(i)), F_ATTR + i));    // b_y_i * (m_i*G_m[i])
          else m.var((u32)T_M[i], D(B_y(i)));
      }
      P.msms.push_back(m.d); S_CV = slot++; }
    TxBuilder tb; tb.start("2019/1416 anonymous credential"); tb.domain_sep("2019/1416 issuance proof");
    tb.scalar_var("w"); tb.scalar_var("w'"); tb.scalar_var("x_0"); tb.scalar_var("x_1");
    for (u32 i = 0; i < n; i++) tb.scalar_var("y");
    tb.scalar_var("1");
    tb.point_var_const("G_V", ic.enc[ic.id_GV()].data()); tb.point_var_const("G_w", ic.enc[ic.id_Gw()].data());
    tb.point_var_const("G_w_prime", ic.enc[ic.id_Gwp()].data());
    tb.point_var_const("-G_x_0", ic.enc_neg[ic.id_Gx0()].data()); tb.point_var_const("-G_x_1", ic.enc_neg[ic.id_Gx1()].data());
    for (u32 i = 0; i < ic.ny; i++) tb.point_var_const("-G_y", ic.enc_neg[ic.id_Gy(i)].data());
    tb.point_var_const("C_W", ic.enc[ic.id_CW()].data()); tb.point_var_const("I", ic.enc[ic.id_I()].data());
    tb.point_var("U", SRC_COMP, C_U, false); tb.point_var("V", SRC_COMMIT, S_V, false); tb.point_var("tU", SRC_COMMIT, S_tU, false);
    for (u32 i = 0; i < n; i++) { if (kinds[i] == 0) tb.point_var("M", SRC_COMMIT, (u32)S_M[i], false); else tb.point_var("M", SRC_FIELD, F_ATTR + i, false); }
    tb.blinding_commitment("C_W", S_CW); tb.blinding_commitment("I", S_I); tb.blinding_commitment("V", S_CV);
    for (u32 s : {S_CW, S_I, S_CV}) P.dump_commit.push_back(s);
    tb.challenge();
    finish_transcript(P, tb, 0xffff, 0);
    P.n_msm = slot; P.n_proofs = 1;
    auto word = [&](u32 kind, u32 a, u32 b = 0, u32 c = 0) { OutWord o; o.kind = (u16)kind; o.a = (u16)a; o.b = (u16)b; o.c = (u16)c; P.out_words.push_back(o); };
    word(OW_DERIVED, D_T); word(OW_COMP, C_U); word(OW_COMMIT, S_V);
    if (batchable) for (u32 s : {S_CW, S_I, S_CV}) word(OW_COMMIT, s);
    else word(OW_CHAL, 0);
    const u32 wit[4] = {sref_secret(2 + n), sref_secret(3 + n), sref_secret(sec_x0()), sref_secret(sec_x1())};   // w, w', x_0, x_1
    for (u32 k = 0; k < 4; k++) word(OW_RESP, 0, wit[k], sref_derived(D_B(k)));
    for (u32 i = 0; i < n; i++) word(OW_RESP, 0, sref_secret(sec_y(i)), sref_derived(D_B(4 + i)));
    word(OW_RESP, 0, 0xffff, sref_derived(D_B(4 + n)));                                                          // the witness "1"
    mark_comb_jobs(P);
    return P;
}

// AnonymousCredential::show as a program (credential.rs:37-46 -> ProofOfValidCredential::prove presentation.rs:139-321 and, per
// hidden plaintext attribute, ProofOfEncryption::prove encryption.rs:58-142 with Keypair::encrypt symmetric.rs:252-261),
// with the rng output supplied by the caller.  The user-side batch operation: it needs no issuer secret.
// kinds = the presentation's attribute kinds (0 revealed scalar, 1 hidden scalar, 2 revealed point, 3 hidden plaintext).
// Fields: t, U, V, then per attribute: scalar m_i (kinds 0/1) | point M_i (kind 2) | plaintext M1, M2, m3 (kind 3);
//         then a, a0, a1, pk of the symmetric keypair (only if some kind is 3); then two 32-byte words (64 rng bytes) per
//         random value: z, the main proof's 3 + h_s blindings, then 6 blindings per hidden plaintext.
// Output words: exactly the presentation layout of include/aeonflux_b200.h.  batchable = zkp's prove_batchable: every challenge word
// is replaced by that proof's blinding commitments in constraint order (main proof: Z, C_x_1, the C_y constraints; proof of
// encryption: pk, C_y_1-E2, C_y_2', E1, C_y_3), which is the layout compile_presentation(..., batchable = true) takes.  The
// challenges are still derived: the responses need them.  Like compile_presentation, the linked statement has no batchable form.
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
    ShapeProgram P; P.is_issue = true;
    u32 hs = 0, hp = 0; std::vector<int> ss_rank(n, -1);
    for (u32 i = 0; i < n; i++) { if (kinds[i] == 1) ss_rank[i] = (int)hs++; hp += kinds[i] == 3; }
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
    auto dv = [&](u32 op, u32 a, u32 b, u32 c = 0) { DeriveOp d; d.op = (u16)op; d.a = (u16)a; d.b = (u16)b; d.c = (u16)c; P.derived.push_back(d); return sref_derived((u32)P.derived.size() - 1); };
    auto wide = [&](u32 lo) { return dv(DV_WIDE, lo, lo + 1); };
    const u32 D_z = wide(F_ZSEED);
    const u32 D_z0 = dv(DV_NEGMUL, F_T, D_z);                                   // z_0 = -t*z (presentation.rs:163)
    const u32 D_bz = wide(F_BSEED), D_bz0 = wide(F_BSEED + 2), D_bt = wide(F_BSEED + 4);
    std::vector<u32> D_bm(hs);
    for (u32 k = 0; k < hs; k++) D_bm[k] = wide(F_BSEED + 6 + 2 * k);
    const u32 D_g0 = dv(DV_MULADD, D_bz0, D_bt, D_z);                            // b_z0 + b_t*z
    // ---- points
    u32 natab = 0, next = 0;
    auto pjob = [&](u32 field, bool atab, bool ext, int* a_out, int* e_out) {
        PointJob j; j.field_a = (int16_t)field; j.field_b = -1; j.op = PJ_COPY; j.table_slot = -1; j.comp_slot = -1; j.compneg_slot = -1;
        j.atab_slot = (int16_t)(atab ? (int)natab++ : -1); j.ext_slot = (int16_t)(ext ? (int)next++ : -1);
        if (a_out) *a_out = j.atab_slot; if (e_out) *e_out = j.ext_slot;
        P.point_jobs.push_back(j);
    };
    int A_U, E_U, E_V;
    pjob(F_U, true, true, &A_U, &E_U); pjob(F_V, false, true, nullptr, &E_V);
    std::vector<int> E_M1(n, -1), A_M2(n, -1), E_M2(n, -1);
    for (u32 i = 0; i < n; i++) {
        if (kinds[i] == 2) pjob(F_ATTR[i], false, false, nullptr, nullptr);     // revealed point: only has to decode
        if (kinds[i] == 3) { pjob(F_ATTR[i], false, true, nullptr, &E_M1[i]); pjob(F_ATTR[i] + 1, true, true, &A_M2[i], &E_M2[i]); }
    }
    if (hp) pjob(F_PK, false, false, nullptr, nullptr);
    P.n_tables = 0; P.n_atabs = natab; P.n_ext = next; P.n_comp = 0;
    // ---- ladders (every scalar is a user secret: constant-schedule jobs; a variable term's table_slot is its transposed table)
    u32 slot = 0;
    auto push = [&](MsmBuilder& m) { P.msms.push_back(m.d); return slot++; };
    auto R = [](u32 ref) { return sc_field(ref); };
    u32 S_CX0, S_CX1, S_CV, S_Z, S_RZ, S_RCX1;
    { MsmBuilder m(slot); m.con(ic.id_Gx0(), R(D_z)); m.add_ext((u32)E_U); S_CX0 = push(m); }                              // C_x_0 = z*G_x_0 + U   (:181)
    { MsmBuilder m(slot); m.var((u32)A_U, R(F_T)); m.con(ic.id_Gx1(), R(D_z)); S_CX1 = push(m); }                          // C_x_1 = z*G_x_1 + t*U (:182)
    { MsmBuilder m(slot); m.con(ic.id_GV(), R(D_z)); m.add_ext((u32)E_V); S_CV = push(m); }                                // C_V = z*G_V + V       (:183)
    std::vector<u32> S_CY(n);
    for (u32 i = 0; i < n; i++) {                                                                                           // (:169-180)
        MsmBuilder m(slot); m.con(ic.id_Gy(i), R(D_z));
        if (kinds[i] == 1) m.con(ic.id_Gm(i), R(F_ATTR[i]));
        if (kinds[i] == 3) m.add_ext((u32)E_M1[i]);
        S_CY[i] = push(m);
    }
    { MsmBuilder m(slot); m.con(ic.id_I(), R(D_z)); S_Z = push(m); }                                                       // Z = z*I (:184)
    { MsmBuilder m(slot); m.con(ic.id_I(), R(D_bz)); S_RZ = push(m); }
    { MsmBuilder m(slot); m.var((u32)A_U, R(D_bt)); m.con(ic.id_Gx0(), R(D_g0)); m.con(ic.id_Gx1(), R(D_bz)); S_RCX1 = push(m); }
    std::vector<u32> nsp;
    for (u32 i = 0; i < n; i++) if (kinds[i] != 3) nsp.push_back(i);
    struct Con { u32 slot; const char* label; };
    std::vector<Con> main_cons; main_cons.push_back({S_RZ, "Z"}); main_cons.push_back({S_RCX1, "C_x_1"});
    for (u32 i = 0; i < nsp.size(); i++) {                    // compacted-index loop (:267-273, SURVEY A.6.1)
        if (kinds[i] == 3) continue;
        MsmBuilder m(slot); m.con(ic.id_Gy(i), R(D_bz));
        if (kinds[i] == 1) m.con(ic.id_Gm(i), R(D_bm[ss_rank[i]]));
        main_cons.push_back({push(m), "C_y"});
    }
    // linked statement (see compile_presentation): D_i = C_y[i] - C_y_1 = z*G_y[i] - z*G_y[0] and its blinding commitment b_z*(G_y[i] - G_y[0])
    struct Link { u32 attr, S_D; };
    std::vector<Link> links;
    if (linked)
        for (u32 i = 1; i < n; i++) if (kinds[i] == 3) {
            u32 S_D;
            { MsmBuilder m(slot); m.con(ic.id_Gy(i), R(D_z)); m.con(ic.id_Gy(0), R(D_z), true); S_D = push(m); }
            { MsmBuilder m(slot); m.con(ic.id_Gy(i), R(D_bz)); m.con(ic.id_Gy(0), R(D_bz), true); main_cons.push_back({push(m), "C_y-C_y_1"}); }
            links.push_back({i, S_D});
        }
    {
        TxBuilder tb; tb.start("2019/1416 anonymous credential"); tb.domain_sep("2019/1416 presentation proof");
        tb.scalar_var("z"); tb.scalar_var("z_0"); tb.scalar_var("t");
        for (u32 k = 0; k < hs; k++) tb.scalar_var("m");
        tb.point_var_const("I", ic.enc[ic.id_I()].data());
        tb.point_var("C_x_1", SRC_COMMIT, S_CX1, false); tb.point_var("C_x_0", SRC_COMMIT, S_CX0, false);
        tb.point_var_const("G_x_0", ic.enc[ic.id_Gx0()].data()); tb.point_var_const("G_x_1", ic.enc[ic.id_Gx1()].data());
        for (u32 i : nsp) tb.point_var("C_y", SRC_COMMIT, S_CY[i], false);
        for (u32 i = 0; i < ic.ny; i++) tb.point_var_const("G_y", ic.enc[ic.id_Gy(i)].data());
        for (u32 i = 0; i < n; i++) if (kinds[i] == 1) tb.point_var_const("G_m", ic.enc[ic.id_Gm(i)].data());
        for (const Link& l : links) { tb.point_var_const("G_y-G_y_1", ic.enc_link.at(l.attr).data()); tb.point_var("C_y-C_y_1", SRC_COMMIT, l.S_D, false); }
        tb.point_var("Z", SRC_COMMIT, S_Z, false);
        for (const Con& c : main_cons) { tb.blinding_commitment(c.label, c.slot); P.dump_commit.push_back(c.slot); }
        tb.challenge();
        finish_transcript(P, tb, 0xffff, 0);
    }
    auto word = [&](u32 kind, u32 a, u32 b = 0, u32 c = 0) { OutWord o; o.kind = (u16)kind; o.a = (u16)a; o.b = (u16)b; o.c = (u16)c; P.out_words.push_back(o); };
    if (batchable) for (const Con& c : main_cons) word(OW_COMMIT, c.slot);
    else word(OW_CHAL, 0);
    word(OW_RESP, 0, D_z, D_bz); word(OW_RESP, 0, D_z0, D_bz0); word(OW_RESP, 0, F_T, D_bt);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 1) word(OW_RESP, 0, F_ATTR[i], D_bm[ss_rank[i]]);
    word(OW_COMMIT, S_CX0); word(OW_COMMIT, S_CX1); word(OW_COMMIT, S_CV);
    for (u32 i = 0; i < n; i++) word(OW_COMMIT, S_CY[i]);
    for (u32 i = 0; i < n; i++) if (kinds[i] == 0 || kinds[i] == 2) word(OW_FIELD, F_ATTR[i]);
    // ---- proofs of encryption, one per hidden plaintext (presentation.rs:293-309 -> encryption.rs:58-142)
    u32 e = 0;
    for (u32 idx = 0; idx < n; idx++) {
        if (kinds[idx] != 3) continue;
        const u32 F_M3 = F_ATTR[idx] + 2, AM2 = (u32)A_M2[idx], EM1 = (u32)E_M1[idx], EM2 = (u32)E_M2[idx];
        const u32 D_u = dv(DV_MULADD, F_A0, F_A1, F_M3);                        // a0 + a1*m3 (symmetric.rs:257)
        const u32 D_au = dv(DV_MUL, F_A, D_u);
        const u32 D_z1 = dv(DV_NEGMUL, D_z, D_u);                                // z1 = -z*(a0 + a1*m3) (encryption.rs:78)
        const u32 D_a1z = dv(DV_MUL, F_A1, D_z);
        const u32 B0 = F_EBSEED + 12 * e;
        const u32 D_ba = wide(B0), D_ba0 = wide(B0 + 2), D_ba1 = wide(B0 + 4), D_bm3 = wide(B0 + 6), D_bze = wide(B0 + 8), D_bz1 = wide(B0 + 10);
        const u32 D_bau = dv(DV_MUL, D_ba, D_u);
        const u32 D_ba1z = dv(DV_MUL, D_ba1, D_z);
        const u32 D_s1 = dv(DV_MULADD, D_ba0, D_bm3, F_A1);                      // b_a0 + b_m3*a1
        const u32 D_s2 = dv(DV_MULADD, D_bz1, D_s1, D_z);                        // b_z1 + (b_a0 + b_m3*a1)*z
        u32 S_E1, S_E2, S_CY1, S_CY2, S_CY3, S_CY2P, S_D, S_NE1, S_Rpk, S_RD, S_RCY2P, S_RE1, S_RCY3;
        { MsmBuilder m(slot); m.var(AM2, R(D_u)); S_E1 = push(m); }                                                         // E1 = (a0 + a1*m3)*M2
        { MsmBuilder m(slot); m.var(AM2, R(D_au)); m.add_ext(EM1); S_E2 = push(m); }                                        // E2 = a*E1 + M1
        { MsmBuilder m(slot); m.con(ic.id_Gy(0), R(D_z)); m.add_ext(EM1); S_CY1 = push(m); }                                // C_y_1 = z*G_y[0] + M1
        { MsmBuilder m(slot); m.con(ic.id_Gy(1), R(D_z)); m.add_ext(EM2); S_CY2 = push(m); }                                // C_y_2 = z*G_y[1] + M2
        { MsmBuilder m(slot); m.con(ic.id_Gy(2), R(D_z)); m.con(ic.id_Gm(idx), R(F_M3)); S_CY3 = push(m); }                 // C_y_3 = z*G_y[2] + m3*G_m[idx]
        { MsmBuilder m(slot); m.var(AM2, R(F_A1)); m.con(ic.id_Gy(1), R(D_a1z)); S_CY2P = push(m); }                        // C_y_2' = a1*C_y_2
        { MsmBuilder m(slot); m.con(ic.id_Gy(0), R(D_z)); m.var(AM2, R(D_au), true); S_D = push(m); }                       // C_y_1 - E2 (M1 cancels)
        { MsmBuilder m(slot); m.var(AM2, R(D_u), true); S_NE1 = push(m); }                                                  // -E1
        { MsmBuilder m(slot); m.con(ic.id_Ga(), R(D_ba)); m.con(ic.id_Ga0(), R(D_ba0)); m.con(ic.id_Ga1(), R(D_ba1)); S_Rpk = push(m); }
        { MsmBuilder m(slot); m.con(ic.id_Gy(0), R(D_bze)); m.var(AM2, R(D_bau), true); S_RD = push(m); }                   // b_z*G_y_1 + b_a*(-E1)
        { MsmBuilder m(slot); m.var(AM2, R(D_ba1)); m.con(ic.id_Gy(1), R(D_ba1z)); S_RCY2P = push(m); }                     // b_a1*C_y_2
        { MsmBuilder m(slot); m.con(ic.id_Gy(1), R(D_s2)); m.var(AM2, R(D_s1)); S_RE1 = push(m); }                          // b_a0*C_y_2 + b_m3*C_y_2' + b_z1*G_y_2
        { MsmBuilder m(slot); m.con(ic.id_Gy(2), R(D_bze)); m.con(ic.id_Gm(idx), R(D_bm3)); S_RCY3 = push(m); }
        TxBuilder tb; tb.start("2019/1416 anonymous credentials"); tb.domain_sep("2019/1416 proof of encryption");
        tb.scalar_var("a"); tb.scalar_var("a0"); tb.scalar_var("a1"); tb.scalar_var("m3"); tb.scalar_var("z"); tb.scalar_var("z1");
        tb.point_var("pk", SRC_FIELD, F_PK, false);
        tb.point_var_const("G_a", ic.enc[ic.id_Ga()].data()); tb.point_var_const("G_a_0", ic.enc[ic.id_Ga0()].data());
        tb.point_var_const("G_a_1", ic.enc[ic.id_Ga1()].data());
        tb.point_var_const("G_y_1", ic.enc[ic.id_Gy(0)].data()); tb.point_var_const("G_y_2", ic.enc[ic.id_Gy(1)].data());
        tb.point_var_const("G_y_3", ic.enc[ic.id_Gy(2)].data()); tb.point_var_const("G_m_3", ic.enc[ic.id_Gm(idx)].data());
        tb.point_var("C_y_2", SRC_COMMIT, S_CY2, false); tb.point_var("C_y_3", SRC_COMMIT, S_CY3, false); tb.point_var("C_y_2'", SRC_COMMIT, S_CY2P, false);
        tb.point_var("C_y_1-E2", SRC_COMMIT, S_D, false);
        tb.point_var("E1", SRC_COMMIT, S_E1, false);
        tb.point_var("-E1", SRC_COMMIT, S_NE1, false);
        tb.blinding_commitment("pk", S_Rpk); tb.blinding_commitment("C_y_1-E2", S_RD); tb.blinding_commitment("C_y_2'", S_RCY2P);
        tb.blinding_commitment("E1", S_RE1); tb.blinding_commitment("C_y_3", S_RCY3);
        for (u32 s2 : {S_Rpk, S_RD, S_RCY2P, S_RE1, S_RCY3}) P.dump_commit.push_back(s2);
        tb.challenge();
        finish_transcript(P, tb, 0xffff, 1 + e);
        if (batchable) for (u32 s2 : {S_Rpk, S_RD, S_RCY2P, S_RE1, S_RCY3}) word(OW_COMMIT, s2);
        else word(OW_CHAL, 1 + e);
        word(OW_RESP, 1 + e, F_A, D_ba); word(OW_RESP, 1 + e, F_A0, D_ba0); word(OW_RESP, 1 + e, F_A1, D_ba1);
        word(OW_RESP, 1 + e, F_M3, D_bm3); word(OW_RESP, 1 + e, D_z, D_bze); word(OW_RESP, 1 + e, D_z1, D_bz1);
        word(OW_FIELD, F_PK);
        word(OW_COMMIT, S_E1); word(OW_COMMIT, S_E2); word(OW_COMMIT, S_CY1); word(OW_COMMIT, S_CY2); word(OW_COMMIT, S_CY3); word(OW_COMMIT, S_CY2P);
        e++;
    }
    P.n_msm = slot; P.n_proofs = (u32)P.txs.size();
    mark_comb_jobs(P);
    return P;
}

// Keypair::encrypt (symmetric.rs:252-261) as a program: the two ladders of show's proof of encryption (compile_show),
//     E1 = (a0 + a1*m3)*M2,   E2 = (a*(a0 + a1*m3))*M2 + M1.
// Fields: the Plaintext M1, M2, m3.  The keypair a, a0, a1 is the call's: the pass puts it in the secret rows (ws.secsc) 0, 1, 2.
// Output words: E1, E2.  Every scalar is secret (constant-schedule ladders); the derived scalars are wiped after each pass.
inline ShapeProgram compile_encrypt() {
    ShapeProgram P; P.is_issue = true;
    const u32 F_M1 = 0, F_M2 = 1, F_M3 = 2;
    P.n_fields = 3;
    P.scalar_fields.push_back((u16)F_M3);
    auto dv = [&](u32 op, u32 a, u32 b, u32 c = 0) { DeriveOp d; d.op = (u16)op; d.a = (u16)a; d.b = (u16)b; d.c = (u16)c; P.derived.push_back(d); return sref_derived((u32)P.derived.size() - 1); };
    const u32 D_u = dv(DV_MULADD, sref_secret(1), sref_secret(2), F_M3);      // a0 + a1*m3
    const u32 D_au = dv(DV_MUL, sref_secret(0), D_u);
    PointJob j; j.field_b = -1; j.op = PJ_COPY; j.table_slot = -1; j.comp_slot = -1; j.compneg_slot = -1;
    j.field_a = (int16_t)F_M1; j.atab_slot = -1; j.ext_slot = 0; P.point_jobs.push_back(j);
    j.field_a = (int16_t)F_M2; j.atab_slot = 0; j.ext_slot = -1; P.point_jobs.push_back(j);
    P.n_tables = 0; P.n_atabs = 1; P.n_ext = 1; P.n_comp = 0;
    { MsmBuilder m(0); m.var(0, sc_field(D_u)); P.msms.push_back(m.d); }
    { MsmBuilder m(1); m.var(0, sc_field(D_au)); m.add_ext(0); P.msms.push_back(m.d); }
    P.n_msm = 2; P.n_proofs = 0;
    for (u32 k = 0; k < 2; k++) { OutWord o; o.kind = OW_COMMIT; o.a = (u16)k; o.b = o.c = 0; P.out_words.push_back(o); }
    return P;
}

// Keypair::derive (symmetric.rs:197-215) as a program: pk = a*G_a + a0*G_a0 + a1*G_a1 over the context's system parameters, one MSM of
// constant bases with secret scalars, which mark_comb_jobs puts on the radix-16 comb (constant-address scans).
// Fields: a, a0, a1, the rows the hashes of keypair_scalars_job (engine.cuh) leave.  Output words: a, a0, a1, pk -- the 128-byte
// keypair afx_show takes.
inline ShapeProgram compile_keypair(const IssuerConsts& ic) {
    ShapeProgram P; P.is_issue = true;
    P.n_fields = 3;
    MsmBuilder m(0); m.con(ic.id_Ga(), sc_field(0)); m.con(ic.id_Ga0(), sc_field(1)); m.con(ic.id_Ga1(), sc_field(2)); P.msms.push_back(m.d);
    P.n_msm = 1; P.n_proofs = 0;
    for (u32 k = 0; k < 4; k++) { OutWord o; o.kind = (u16)(k < 3 ? OW_FIELD : OW_COMMIT); o.a = (u16)(k < 3 ? k : 0); o.b = o.c = 0; P.out_words.push_back(o); }
    mark_comb_jobs(P);
    return P;
}

}  // namespace afx
