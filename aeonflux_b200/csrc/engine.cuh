// The batch engine's stage bodies, shared by the CUDA kernels (afx_b200.cu) and the test-only host emulation
// harness (tests/hostemu).  One "item" = one presentation / issuance of a batch; every stage is data-parallel over
// items with no cross-item state.
//
// Stages for Issuer::verify (/root/reference/src/issuer.rs:141-147 -> nizk/presentation.rs:324-443):
//   points     decompress every input point once, derive sums/differences, build the [1P..8P] Niels table each
//              ladder needs, compress the derived points the transcript absorbs (presentation.rs:373-412 do this with
//              compress()+decompress() per allocated point; SURVEY 8d "minimal schedule")
//   amac       Z = C_V - W - x0*C_x0 - x1*C_x1 - sum y_i*X_i as ONE constant-schedule radix-16 Straus ladder over
//              issuer-secret scalars (presentation.rs:342-352: seven separate constant-time scalar mults)
//   msm        one thread per (item, constraint): R = sum resp_k*P_k - c*LHS, fixed-window ladder sharing 252 doublings,
//              radix-256 affine tables for per-issuer constant bases, radix-16 tables for per-item bases; compress R
//              (zkp verify_compact's vartime_multiscalar_mul per constraint, SURVEY A.4)
//   transcript one thread per (item, proof): Merlin/STROBE/Keccak-f[1600] over the compiled block template, 64-byte
//              challenge squeeze, reduction mod l, compare with the claimed challenge
//   verdict    status word -> 0 (Ok) / 1 (VerificationFailure)
// Symmetric encryption of attributes (encoding.rs, symmetric.rs) has its own per-item bodies at the end of this file.
#pragma once
#include "fe.cuh"
#include "ge.cuh"
#include "keccak.cuh"
#include "sc.cuh"
#include "sha512.cuh"

namespace afx {

#ifndef AFX_SYNC_MASK
#define AFX_SYNC_MASK 0   // ladder CTAs re-align at a barrier every (AFX_SYNC_MASK + 1) windows
#endif
// The constant-schedule ladders (k_msm_ct) stall on their table scans; their barrier policy is separate from the verify ladders':
// AFX_CT_SYNC_MASK as above, AFX_CT_SYNC_GROUPS = 2 re-aligns each half of the CTA on its own named barrier so that one half can
// scan while the other multiplies.
#ifndef AFX_CT_SYNC_MASK
#define AFX_CT_SYNC_MASK 0
#endif
#ifndef AFX_CT_SYNC_GROUPS
#define AFX_CT_SYNC_GROUPS 1
#endif
#if defined(__CUDA_ARCH__) && AFX_CT_SYNC_GROUPS == 2
#define AFX_CT_STEP_SYNC() do { if (threadIdx.x < 128u) asm volatile("bar.sync 1, 128;" ::: "memory"); else asm volatile("bar.sync 2, 128;" ::: "memory"); } while (0)   /* TPB_MSM = 256 */
#elif defined(__CUDA_ARCH__) && AFX_CT_SYNC_GROUPS == 0
#define AFX_CT_STEP_SYNC() do { } while (0)
#else
#define AFX_CT_STEP_SYNC() AFX_STEP_SYNC()
#endif
constexpr int MAX_ATTRS = 32;
constexpr int MAX_VAR_TERMS = MAX_ATTRS + 4;
constexpr int MAX_CONST_TERMS = MAX_ATTRS + 8;
constexpr int CTAB_ENTRIES = 2048; // radix-4096 signed digits: multiples 1..2048 of a constant base (192 KiB per generator, L2-resident)
constexpr int CTAB16_ENTRIES = 32768;  // optional radix-2^16 tables (3 MB per generator), built when all of an issuer's fit the L2 budget

// ---- scalar sources ---------------------------------------------------------------------------
enum : u32 { SC_FIELD = 0, SC_MUL = 1, SC_MULADD = 2 };  // R[f0] | R[f0]*R[f1] | R[f0] + R[f1]*R[f2]
// A scalar reference R[f] names an input field (f < 0x4000), an issuer-secret row (SREF_SECRET | row: x_0, x_1, y_i, w, w')
// or a per-item derived scalar (SREF_DERIVED | slot: the wide-reduced t and blindings of Issuer::issue).
// SREF_CHAL | proof: the challenge recomputed by transcript `proof` of this item (BatchableProof verification, where the wire
// carries the commitments and the challenge is derived, not given).
enum : u32 { SREF_SECRET = 0x4000, SREF_DERIVED = 0x8000, SREF_CHAL = 0xc000, SREF_MASK = 0x3fff };
struct ScalarSrc { u16 op, f0, f1, f2; };

struct VarTerm { u16 table_slot; u16 neg; ScalarSrc s; u16 ext_slot, pad; };   // ext_slot: the base in extended coordinates (batchable mode only)
struct ConstTerm { u16 ctab; u16 neg; ScalarSrc s; };
// flags.  MSM_ADD_W: add the issuer's W after the ladder (Amac::compute_V, amacs.rs:267).  MSM_COMB: a job with constant
// bases only is evaluated on the per-issuer radix-16 comb tables ((e * 16^i) * G for every window i): 64 mixed adds per
// term and no doublings at all.
enum : u32 { MSM_ADD_W = 1, MSM_COMB = 2, MSM_ADD_EXT = 4 };
constexpr int COMB_WINDOWS = 64, COMB_ENTRIES = 8;   // comb[g][i][e-1] = (e * 16^i) * G_g in affine Niels form, 48 KiB per generator
struct MsmDesc {
    u16 nvar, ncon, out_slot, flags;
    u16 add_ext, pad;                  // MSM_ADD_EXT: ext slot of a per-item point added after the ladder
    VarTerm var[MAX_VAR_TERMS];
    ConstTerm con[MAX_CONST_TERMS];
};

enum : u32 { PJ_COPY = 0, PJ_ADD = 1, PJ_SUB = 2, PJ_UNIFORM = 3, PJ_OP_MASK = 0xff,   // PJ_UNIFORM: from_uniform_bytes(field_a || field_b)
              PJ_KEEP_TABLE = 0x100 };  // flag: build the ladder table even when the pass skips tables (ws.no_tables)
struct PointJob {
    int16_t field_a, field_b;      // input point fields (field_b = -1 for PJ_COPY)
    u16 op;
    int16_t atab_slot;             // aMAC-private transposed copy of the ladder table (-1 = none)
    int16_t table_slot, ext_slot;  // -1 = not written
    int16_t comp_slot, compneg_slot;  // compressed encoding of the point / of its negation
};

struct AmacVar { u16 atab_slot, digit_row; };
struct AmacPs { u16 ctab, y_row, field_m, pad; };  // (y_i * m_i) * G_m[i] for a revealed scalar attribute
struct AmacDesc {
    u16 ext_cv, nvar, nps, out_table_slot, out_comp_slot, out_ext_slot;   // out_ext_slot: 0xffff = Z is not kept in extended form
    AmacVar var[MAX_ATTRS + 2];
    AmacPs ps[MAX_ATTRS];
};

enum : u32 { SRC_FIELD = 0, SRC_COMP = 1, SRC_COMMIT = 2 };
struct TxHole { u16 block, off, len, src_off; u16 src_kind, src_idx; };
struct TxIdCheck { u16 src_kind, src_idx; };
struct TxDesc {
    u32 nblocks, block_ofs;   // blocks: 21 u64 lanes each, at lanes[block_ofs*21]
    u32 nholes, hole_ofs;
    u32 nid, id_ofs;
    u16 chal_field, out_slot;
    u64 midstate[25];
};

// Prover paths (Issuer::issue, AnonymousCredential::show): per-item derived scalars and the output words.
// Derived slot k = result of op k, evaluated in order by one thread per item (operands are scalar refs, so an op may use
// the slots before it).
enum : u32 { DV_WIDE = 0, DV_MUL = 1, DV_MULADD = 2, DV_NEGMUL = 3 };
// DV_WIDE:   (F[a] || F[b]) mod l           Scalar::random's wide reduction of 64 rng bytes
// DV_MUL:    R[a] * R[b]        DV_MULADD: R[a] + R[b] * R[c]        DV_NEGMUL: -(R[a] * R[b])
struct DeriveOp { u16 op, a, b, c; };
// One 32-byte output word per (item, OutWord).
enum : u32 { OW_FIELD = 0, OW_COMP = 1, OW_COMMIT = 2, OW_DERIVED = 3, OW_CHAL = 4, OW_RESP = 5 };
// OW_RESP: a = proof index, b = witness scalar ref (0xffff = the constant "1"), c = blinding scalar ref:
//          response = witness * challenge + blinding  (zkp prove_compact)
struct OutWord { u16 kind, a, b, c; };

// ---- workspace ------------------------------------------------------------------------------------
// All arrays are slot-major then item-major; an item's 32-byte word is 8 consecutive u32 (two 128-bit loads).
struct Workspace {
    u32 count;
    const u32* fields;   // struct-of-arrays [n_fields][count][8] (fs_field = count, fs_item = 1) or item-major "wire"
                         // [count][n_fields][8] (fs_field = 1, fs_item = n_fields); strides in 32-byte words
    u32 fs_field, fs_item;
    u32 e_lo, e_hi;      // the early stages (scalar checks, point jobs) of this launch cover items [e_lo, e_hi) only (a batch copied in halves)
    u32 no_tables;       // 1: point jobs skip the standard ladder tables (BatchableProof RLC pass: only its exact fallback walks them)
    u32* tables;         // [n_tables][count][8 entries][32]
    u32* atabs;          // [n_atabs][ceil(count/32)][8 entries][8 quads][32 lanes][4]  aMAC tables, warp-transposed
    u32* ext;            // [n_ext][count][32]
    u32* comp;           // [n_comp][count][8]
    u32* commit;         // [n_msm][count][8]
    u32* chal;           // [n_proofs][count][8]  recomputed challenges
    u32* status;         // [count]   0 = ok so far
    u32* derived;        // [n_derived][count][8]  per-item derived scalars (Issuer::issue only)
    u32 os_word, os_item, os_base;   // prover output strides in 32-byte words: struct-of-arrays (count, 1, 0) or item-major (1, words per item, first word)
    // per-issuer constants
    const u32* ctabs;    // [n_ctab][2048][24]   affine Niels multiples 1..2048
    const u32* ctabs16;  // [n_ctab][32768][24]  multiples 1..32768, or null (the verify-path MSMs then use radix 4096)
    const u32* comb;     // [n_ctab][64][8][24]  radix-16 comb: (e * 16^i) * G
    const u32* secdig;   // [n_secret][8]      radix-16 recoded secret scalars (packed nibbles)
    const u32* secsc;    // [n_secret][8]      the same scalars, canonical words
    const u32* W_pniels; // [32]               W in projective Niels form
    const u64* lanes;    // transcript block masks
    const TxHole* holes;
    const TxIdCheck* idchecks;
    u32* commit_q;       // [n_msm][count][32]  verify MSMs: Q = R/2 in extended coordinates, which commit_encode_job encodes into commit
};

enum : u32 { ST_BAD_POINT = 1, ST_BAD_SCALAR = 2, ST_IDENTITY = 4, ST_CHALLENGE = 8 };

// ---- small helpers ----------------------------------------------------------------------------------
AFX_HD void load8(u32* dst, const u32* src) {
#if defined(__CUDA_ARCH__)
    const uint4* p = reinterpret_cast<const uint4*>(src);
    uint4 a = p[0], b = p[1];
    dst[0] = a.x; dst[1] = a.y; dst[2] = a.z; dst[3] = a.w; dst[4] = b.x; dst[5] = b.y; dst[6] = b.z; dst[7] = b.w;
#else
    for (int i = 0; i < 8; i++) dst[i] = src[i];
#endif
}
AFX_HD void store8(u32* dst, const u32* src) {
#if defined(__CUDA_ARCH__)
    uint4* p = reinterpret_cast<uint4*>(dst);
    p[0] = make_uint4(src[0], src[1], src[2], src[3]); p[1] = make_uint4(src[4], src[5], src[6], src[7]);
#else
    for (int i = 0; i < 8; i++) dst[i] = src[i];
#endif
}
// Pull a 1 KiB ladder table towards L2 ahead of the constant-address scan that will read all of it.
AFX_HD void prefetch_table(const u32* table) {
#if defined(__CUDA_ARCH__)
    for (int e = 0; e < 8; e++) asm volatile("prefetch.global.L2 [%0];" ::"l"(table + 32 * e));
#else
    (void)table;
#endif
}
AFX_HD fe load_fe(const u32* src) { fe r; load8(r.v, src); return r; }
AFX_HD void store_fe(u32* dst, const fe& a) { store8(dst, a.v); }
AFX_HD ge load_ge(const u32* src) { ge p; p.X = load_fe(src); p.Y = load_fe(src + 8); p.Z = load_fe(src + 16); p.T = load_fe(src + 24); return p; }
AFX_HD void store_ge(u32* dst, const ge& p) { store_fe(dst, p.X); store_fe(dst + 8, p.Y); store_fe(dst + 16, p.Z); store_fe(dst + 24, p.T); }
AFX_HD pniels load_pniels(const u32* src) { pniels n; n.YpX = load_fe(src); n.YmX = load_fe(src + 8); n.Z = load_fe(src + 16); n.T2d = load_fe(src + 24); return n; }
AFX_HD void store_pniels(u32* dst, const pniels& n) { store_fe(dst, n.YpX); store_fe(dst + 8, n.YmX); store_fe(dst + 16, n.Z); store_fe(dst + 24, n.T2d); }
AFX_HD aniels load_aniels(const u32* src) { aniels n; n.ypx = load_fe(src); n.ymx = load_fe(src + 8); n.xy2d = load_fe(src + 16); return n; }

// The aMAC ladder reads EVERY entry of a table at every step (constant-address scan), so its tables are kept in a
// warp-transposed layout: the 16-byte quad q of entry e of 32 consecutive items is one contiguous 512-byte run, and a
// warp's scan is 64 fully coalesced loads instead of 64 loads that each touch 32 different lines.
AFX_HD void store4(u32* dst, const u32* src) {
#if defined(__CUDA_ARCH__)
    *reinterpret_cast<uint4*>(dst) = make_uint4(src[0], src[1], src[2], src[3]);
#else
    for (int i = 0; i < 4; i++) dst[i] = src[i];
#endif
}
AFX_HD void load4(u32* dst, const u32* src) {
#if defined(__CUDA_ARCH__)
    uint4 a = *reinterpret_cast<const uint4*>(src);
    dst[0] = a.x; dst[1] = a.y; dst[2] = a.z; dst[3] = a.w;
#else
    for (int i = 0; i < 4; i++) dst[i] = src[i];
#endif
}
constexpr u32 ATAB_QUAD_STRIDE = 128;                       // words between consecutive quads of one item: 32 lanes x 4
constexpr u32 ATAB_BLOCK_WORDS = 64 * ATAB_QUAD_STRIDE;     // 8 entries x 8 quads
AFX_HD void store_pniels_t(u32* dst, int e, const pniels& n) {
    u32* d = dst + (size_t)e * 8 * ATAB_QUAD_STRIDE;
    store4(d, n.YpX.v); store4(d + ATAB_QUAD_STRIDE, n.YpX.v + 4);
    store4(d + 2 * ATAB_QUAD_STRIDE, n.YmX.v); store4(d + 3 * ATAB_QUAD_STRIDE, n.YmX.v + 4);
    store4(d + 4 * ATAB_QUAD_STRIDE, n.Z.v); store4(d + 5 * ATAB_QUAD_STRIDE, n.Z.v + 4);
    store4(d + 6 * ATAB_QUAD_STRIDE, n.T2d.v); store4(d + 7 * ATAB_QUAD_STRIDE, n.T2d.v + 4);
}
struct TableStore {
    u32* dst; u32* tdst;   // standard / transposed destination, either may be null
    AFX_HD void operator()(int e, const pniels& n) const {
        if (dst) store_pniels(dst + 32 * e, n);
        if (tdst) store_pniels_t(tdst, e, n);
    }
};
AFX_HD void store_table8(u32* dst, const ge& p, u32* tdst = nullptr) { TableStore ts{dst, tdst}; ge_table8(p, ts); }

AFX_HD const u32* field_ptr(const Workspace& ws, u32 f, u32 item) { return ws.fields + ((size_t)f * ws.fs_field + (size_t)item * ws.fs_item) * 8; }
AFX_HD u32* table_ptr(const Workspace& ws, u32 slot, u32 item) { return ws.tables + ((size_t)slot * ws.count + item) * 256; }
AFX_HD u32* atab_ptr(const Workspace& ws, u32 slot, u32 item) {
    size_t nblk = ((size_t)ws.count + 31) / 32;
    return ws.atabs + ((size_t)slot * nblk + item / 32) * ATAB_BLOCK_WORDS + (item % 32) * 4;
}
AFX_HD u32* ext_ptr(const Workspace& ws, u32 slot, u32 item) { return ws.ext + ((size_t)slot * ws.count + item) * 32; }
AFX_HD u32* comp_ptr(const Workspace& ws, u32 slot, u32 item) { return ws.comp + ((size_t)slot * ws.count + item) * 8; }
AFX_HD u32* commit_ptr(const Workspace& ws, u32 slot, u32 item) { return ws.commit + ((size_t)slot * ws.count + item) * 8; }
AFX_HD u32* commit_q_ptr(const Workspace& ws, u32 slot, u32 item) { return ws.commit_q + ((size_t)slot * ws.count + item) * 32; }

AFX_HD void status_or(const Workspace& ws, u32 item, u32 bits) {
#if defined(__CUDA_ARCH__)
    atomicOr(ws.status + item, bits);
#else
    ws.status[item] |= bits;
#endif
}

AFX_HD const u32* scalar_ref_ptr(const Workspace& ws, u32 ref, u32 item) {
    if ((ref & SREF_CHAL) == SREF_CHAL) return ws.chal + ((size_t)(ref & SREF_MASK) * ws.count + item) * 8;
    if (ref & SREF_DERIVED) return ws.derived + ((size_t)(ref & SREF_MASK) * ws.count + item) * 8;
    if (ref & SREF_SECRET) return ws.secsc + 8 * (ref & SREF_MASK);
    return field_ptr(ws, ref, item);
}
AFX_HD sc load_sc(const u32* p) { u32 w[8]; load8(w, p); return sc_from_words(w); }
// A scalar that feeds a ladder.  Wire words are attacker-chosen 256-bit strings: one that is not canonical already has its
// ST_BAD_SCALAR bit (k_scalar_check) and the item is rejected whatever the ladders compute, but the recodings below assume
// a < l (sc_digit65536's top digit is the unbiased top halfword, sc_digit4096's the top nibble) and a table index must never
// follow a wire value out of bounds -- so a non-canonical word enters every ladder as 0.  Products (SC_MUL / SC_MULADD) leave
// sc_reduce512 canonical; secret rows are validated at afx_ctx_create; derived scalars and challenges are reduced on the device.
AFX_HD sc eval_scalar(const Workspace& ws, const ScalarSrc& s, u32 item) {
    sc a = load_sc(scalar_ref_ptr(ws, s.f0, item));
    if (s.op == SC_FIELD) {
        if (s.f0 < SREF_SECRET) { u32 m = 0u - sc_is_canonical(a); for (int i = 0; i < 8; i++) a.v[i] &= m; }
        return a;
    }
    sc b = load_sc(scalar_ref_ptr(ws, s.f1, item));
    if (s.op == SC_MUL) return sc_mul(a, b);
    sc c = load_sc(scalar_ref_ptr(ws, s.f2, item));
    return sc_muladd(b, c, a);
}

// ---- stage: scalar canonicity ------------------------------------------------------------------------
AFX_HD void scalar_check_job(const Workspace& ws, u32 field, u32 item) {
    u32 w[8]; load8(w, field_ptr(ws, field, item));
    if (!sc_is_canonical(sc_from_words(w))) status_or(ws, item, ST_BAD_SCALAR);
}

// ---- stage: points --------------------------------------------------------------------------------------
AFX_HD void points_job(const Workspace& ws, const PointJob& j, u32 item) {
    u32 w[8];
    ge p;
    u32 ok = 1;
    const u32 op = j.op & PJ_OP_MASK;
    if (op == PJ_UNIFORM) {       // RistrettoPoint::random: 64 rng bytes through the Elligator map twice (amacs.rs:290)
        u32 u[16];
        load8(u, field_ptr(ws, (u32)j.field_a, item)); load8(u + 8, field_ptr(ws, (u32)j.field_b, item));
        p = ge_from_uniform(u);
    } else {
        load8(w, field_ptr(ws, (u32)j.field_a, item));
        ok = ge_decompress(p, w);
    }
    if (op == PJ_ADD || op == PJ_SUB) {
        ge q;
        load8(w, field_ptr(ws, (u32)j.field_b, item));
        ok &= ge_decompress(q, w);
        p = (op == PJ_ADD) ? ge_add(p, q) : ge_sub(p, q);
    }
    if (!ok) status_or(ws, item, ST_BAD_POINT);
    if (j.ext_slot >= 0) store_ge(ext_ptr(ws, (u32)j.ext_slot, item), p);
    if (j.comp_slot >= 0) { ge_compress(w, p); store8(comp_ptr(ws, (u32)j.comp_slot, item), w); }
    if (j.compneg_slot >= 0) { ge_compress(w, ge_neg(p)); store8(comp_ptr(ws, (u32)j.compneg_slot, item), w); }
    const bool want_table = j.table_slot >= 0 && (!ws.no_tables || (j.op & PJ_KEEP_TABLE));
    if (want_table || j.atab_slot >= 0)
        store_table8(want_table ? table_ptr(ws, (u32)j.table_slot, item) : nullptr, p,
                     j.atab_slot >= 0 ? atab_ptr(ws, (u32)j.atab_slot, item) : nullptr);
}

// Constant-address table reads: every entry is loaded and the wanted one kept with masks, so neither the branch
// pattern nor the address stream depends on the (secret) digit.
AFX_HD pniels pniels_scan_select(const u32* table, int digit, u32 xneg = 0) {
    u32 neg = ((u32)digit >> 31) ^ xneg;
    u32 mag = (u32)((digit ^ (digit >> 31)) - (digit >> 31));
#ifdef AFX_EXPERIMENT_DIRECT
    { pniels r = pniels_identity(); if (mag) r = load_pniels(table + 32 * (mag - 1)); return pniels_cneg(r, neg); }
#endif
    // every entry is read (128 contiguous bytes per load group) and OR-ed in under a mask
    u32 out[32];
    for (int i = 0; i < 32; i++) out[i] = 0;
    for (u32 e = 1; e <= 8; e++) {
        u32 m = 0u - (u32)(e == mag);
        for (int q = 0; q < 4; q++) {
            u32 w[8]; load8(w, table + 32 * (e - 1) + 8 * q);
            for (int i = 0; i < 8; i++) out[8 * q + i] |= w[i] & m;
        }
    }
    u32 z = (mag == 0);   // digit 0 -> the identity (1, 1, 1, 0)
    out[0] |= z; out[8] |= z; out[16] |= z;
    pniels r;
    for (int i = 0; i < 8; i++) { r.YpX.v[i] = out[i]; r.YmX.v[i] = out[8 + i]; r.Z.v[i] = out[16 + i]; r.T2d.v[i] = out[24 + i]; }
    return pniels_cneg(r, neg);
}
// The same scan over a warp-transposed table (tab = atab_ptr(slot, item)).
AFX_HD pniels pniels_scan_select_t(const u32* tab, int digit, u32 xneg = 0) {
    u32 neg = ((u32)digit >> 31) ^ xneg;
    u32 mag = (u32)((digit ^ (digit >> 31)) - (digit >> 31));
    u32 out[32];
    for (int i = 0; i < 32; i++) out[i] = 0;
    for (u32 e = 1; e <= 8; e++) {
        u32 m = 0u - (u32)(e == mag);
        for (int q = 0; q < 8; q++) {
            u32 w[4]; load4(w, tab + ((size_t)(e - 1) * 8 + q) * ATAB_QUAD_STRIDE);
            for (int i = 0; i < 4; i++) out[4 * q + i] |= w[i] & m;
        }
    }
    u32 z = (mag == 0);   // digit 0 -> the identity (1, 1, 1, 0)
    out[0] |= z; out[8] |= z; out[16] |= z;
    pniels r;
    for (int i = 0; i < 8; i++) { r.YpX.v[i] = out[i]; r.YmX.v[i] = out[8 + i]; r.Z.v[i] = out[16 + i]; r.T2d.v[i] = out[24 + i]; }
    return pniels_cneg(r, neg);
}
// Pull the next table block of this warp (32 KiB, contiguous) towards L2: each lane touches 8 of its 256 lines.
AFX_HD void prefetch_atab(const u32* tab_lane0) {
#if defined(__CUDA_ARCH__)
    const u32* base = tab_lane0 + (threadIdx.x & 31u) * 8 * 32;   // lane's 8 consecutive 128-byte lines
#ifdef AFX_CT_PREFETCH_L1
    for (int j = 0; j < 8; j++) asm volatile("prefetch.global.L1 [%0];" ::"l"(base + 32 * j));
#else
    for (int j = 0; j < 8; j++) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + 32 * j));
#endif
#else
    (void)tab_lane0;
#endif
}
AFX_HD aniels aniels_scan_select8(const u32* ctab, int digit, u32 xneg = 0) {
    u32 neg = ((u32)digit >> 31) ^ xneg;
    u32 mag = (u32)((digit ^ (digit >> 31)) - (digit >> 31));
    u32 out[24];
    for (int comp = 0; comp < 3; comp++) {
        u32 acc[8];
        for (int i = 0; i < 8; i++) acc[i] = 0;
        for (u32 e = 1; e <= 8; e++) {
            u32 w[8]; load8(w, ctab + 24 * (e - 1) + 8 * comp);
            u32 m = 0u - (u32)(e == mag);
            for (int i = 0; i < 8; i++) acc[i] |= w[i] & m;
        }
        for (int i = 0; i < 8; i++) out[8 * comp + i] = acc[i];
    }
    u32 z = (mag == 0);
    out[0] |= z; out[8] |= z;
    aniels r;
    for (int i = 0; i < 8; i++) { r.ypx.v[i] = out[i]; r.ymx.v[i] = out[8 + i]; r.xy2d.v[i] = out[16 + i]; }
    return aniels_cneg(r, neg);
}

// ---- stage: aMAC --------------------------------------------------------------------------------------------
// scratch: nps * 8 words per item for the recoded (y_i * m_i) scalars; scratch_stride = distance between words
AFX_HD void amac_job(const Workspace& ws, const AmacDesc& d, u32 item, u32* scratch, u32 scratch_stride, bool active = true) {
    for (u32 k = 0; k < d.nps; k++) {
        sc m = sc_from_words(field_ptr(ws, d.ps[k].field_m, item));
        sc y = sc_from_words(ws.secsc + 8 * d.ps[k].y_row);
        u32 rec[8];
        sc_recode16(rec, sc_mul(y, m));
        for (int w = 0; w < 8; w++) scratch[(k * 8 + w) * scratch_stride] = rec[w];
    }
    gc cacc = gc_identity();
    for (int i = 63; i >= 0; i--) {
#if defined(__CUDA_ARCH__)
        if ((i & AFX_SYNC_MASK) == AFX_SYNC_MASK) AFX_STEP_SYNC();
#endif
        if (i != 63) gc_dbl4(cacc);
#if defined(__CUDA_ARCH__) && defined(AFX_SYNC_FINE)
        AFX_STEP_SYNC();
#endif
        for (u32 k = 0; k < d.nvar; k++) {
            int dig = sc_digit16(ws.secdig + 8 * d.var[k].digit_row, i);
            pniels e = pniels_scan_select_t(atab_ptr(ws, d.var[k].atab_slot, item), dig);
            prefetch_atab(atab_ptr(ws, d.var[k + 1 < d.nvar ? k + 1 : 0].atab_slot, item & ~31u));   // next lookup, hidden behind this add
            GE_LADDER_ADD(cacc, e);
        }
        for (u32 k = 0; k < d.nps; k++) {
            u32 word = scratch[(k * 8 + (i >> 3)) * scratch_stride];
            int dig = ((int)(word << (28 - 4 * (i & 7)))) >> 28;
            aniels e = aniels_scan_select8(ws.ctabs + (size_t)d.ps[k].ctab * CTAB_ENTRIES * 24, dig);
            GE_LADDER_MADD(cacc, e);
        }
    }
    for (u32 k = 0; k < d.nps * 8u; k++) scratch[k * scratch_stride] = 0;   // wipe the recoded y_i * m_i
    ge acc = gc_to_ge(cacc);
    // Z = (C_V - W) - acc
    ge cv = load_ge(ext_ptr(ws, d.ext_cv, item));
    ge z = ge_add_pn(cv, pniels_cneg(load_pniels(ws.W_pniels), 1));
    z = ge_sub(z, acc);
    u32 w[8];
    ge_compress(w, z);
    if (active) {
        store8(comp_ptr(ws, d.out_comp_slot, item), w);
        if (!ws.no_tables) store_table8(table_ptr(ws, d.out_table_slot, item), z);
        if (d.out_ext_slot != 0xffff) store_ge(ext_ptr(ws, d.out_ext_slot, item), z);
    }
}

// Small batches (api_impl.inc:run_pipeline): an item's aMAC ladder is the longest dependent chain of the pipeline -- 2 + n bases
// walked by ONE thread, then the "Z" constraint -- and when the batch cannot fill the chip that chain IS the call's latency.  The
// ladder is then cut into parts: part p takes the variable terms [var_lo, var_hi) and the revealed-scalar terms [ps_lo, ps_hi) of
// the same AmacDesc through the same constant-schedule ladder (every table entry read and masked, no digit skipped) with its own
// doublings and leaves its partial sum in extended coordinates; amac_combine_job subtracts the partial sums from C_V - W.  The
// result is the same group element, hence the same bytes.
struct AmacPart { u16 var_lo, var_hi, ps_lo, ps_hi; };
constexpr int MAX_AMAC_PARTS = 24;
AFX_HD void amac_part_job(const Workspace& ws, const AmacDesc& d, const AmacPart& p, u32* part_out /*[count][32]*/, u32 item, u32* scratch, u32 scratch_stride,
                          bool active = true) {
    for (u32 k = p.ps_lo; k < p.ps_hi; k++) {
        sc m = sc_from_words(field_ptr(ws, d.ps[k].field_m, item));
        sc y = sc_from_words(ws.secsc + 8 * d.ps[k].y_row);
        u32 rec[8];
        sc_recode16(rec, sc_mul(y, m));
        for (int w = 0; w < 8; w++) scratch[((k - p.ps_lo) * 8 + w) * scratch_stride] = rec[w];
    }
    gc cacc = gc_identity();
    for (int i = 63; i >= 0; i--) {
#if defined(__CUDA_ARCH__)
        AFX_STEP_SYNC();
#endif
        if (i != 63) gc_dbl4(cacc);
        for (u32 k = p.var_lo; k < p.var_hi; k++) {
            int dig = sc_digit16(ws.secdig + 8 * d.var[k].digit_row, i);
            pniels e = pniels_scan_select_t(atab_ptr(ws, d.var[k].atab_slot, item), dig);
            GE_LADDER_ADD(cacc, e);
        }
        for (u32 k = p.ps_lo; k < p.ps_hi; k++) {
            u32 word = scratch[((k - p.ps_lo) * 8 + (i >> 3)) * scratch_stride];
            int dig = ((int)(word << (28 - 4 * (i & 7)))) >> 28;
            aniels e = aniels_scan_select8(ws.ctabs + (size_t)d.ps[k].ctab * CTAB_ENTRIES * 24, dig);
            GE_LADDER_MADD(cacc, e);
        }
    }
    for (u32 k = 0; k < (u32)(p.ps_hi - p.ps_lo) * 8u; k++) scratch[k * scratch_stride] = 0;   // wipe the recoded y_i * m_i
    ge acc = gc_to_ge(cacc);
    if (active) store_ge(part_out + (size_t)item * 32, acc);
}
AFX_HD void amac_combine_job(const Workspace& ws, const AmacDesc& d, const u32* parts /*[n_parts][count][32]*/, u32 n_parts, u32 item) {
    ge cv = load_ge(ext_ptr(ws, d.ext_cv, item));
    ge z = ge_add_pn(cv, pniels_cneg(load_pniels(ws.W_pniels), 1));      // Z = (C_V - W) - sum of the parts
    for (u32 g = 0; g < n_parts; g++) z = ge_sub(z, load_ge(parts + ((size_t)g * ws.count + item) * 32));
    u32 w[8];
    ge_compress(w, z);
    store8(comp_ptr(ws, d.out_comp_slot, item), w);
    if (!ws.no_tables) store_table8(table_ptr(ws, d.out_table_slot, item), z);
    if (d.out_ext_slot != 0xffff) store_ge(ext_ptr(ws, d.out_ext_slot, item), z);
}

AFX_HD void ztable_job(const Workspace& ws, const AmacDesc& d, u32 item) {
    store_table8(table_ptr(ws, d.out_table_slot, item), load_ge(ext_ptr(ws, d.out_ext_slot, item)));
}

// Where constant term k's radix-4096 table lives (global memory; 192 KiB per generator stay L2-resident).
struct CtabResolver {
    const u32* global; const MsmDesc* d;
    AFX_HD const u32* operator()(u32 k) const { return global + (size_t)d->con[k].ctab * CTAB_ENTRIES * 24; }
};

// ---- stage: msm -----------------------------------------------------------------------------------------------
// Every scalar is halved mod l, so the job computes Q = R/2 of the constraint's R = sum s_j * P_j and leaves it in commit_q in
// extended coordinates: commit_encode_job then encodes 2Q, which needs one inversion per item instead of a square root per job.
// scratch: (nvar + ncon) * 8 words per item of recoded scalars.  ctab_of(k) returns the table base of constant term k
// (global memory).
template <typename CtabOf>
AFX_HD void msm_job(const Workspace& ws, const MsmDesc& d, u32 item, u32* scratch, u32 scratch_stride, CtabOf ctab_of, bool active = true) {
    if (d.flags & MSM_COMB) {      // constant bases only: radix-16 comb, public digits index it directly, no doublings
        gc cacc = gc_identity();
        for (u32 k = 0; k < d.ncon; k++) {
            u32 rec[8];
            sc_recode16(rec, sc_half(eval_scalar(ws, d.con[k].s, item)));
            const u32* comb = ws.comb + (size_t)d.con[k].ctab * COMB_WINDOWS * COMB_ENTRIES * 24;
            for (int i = 0; i < COMB_WINDOWS; i++) {
                int dig = sc_digit16(rec, i);
                if (dig != 0) {
                    u32 neg = ((u32)dig >> 31) ^ d.con[k].neg;
                    u32 mag = (u32)(dig < 0 ? -dig : dig);
                    aniels e = aniels_cneg(load_aniels(comb + ((size_t)i * COMB_ENTRIES + (mag - 1)) * 24), neg);
                    GE_LADDER_MADD(cacc, e);
                }
            }
        }
        if (active) store_ge(commit_q_ptr(ws, d.out_slot, item), gc_to_ge(cacc));
        return;
    }
    const bool wide = ws.ctabs16 != nullptr;      // radix-2^16 constant tables: a digit every 4th window instead of every 3rd
    for (u32 k = 0; k < d.nvar; k++) {
        u32 rec[8];
        sc_recode16(rec, sc_half(eval_scalar(ws, d.var[k].s, item)));
        for (int w = 0; w < 8; w++) scratch[(k * 8 + w) * scratch_stride] = rec[w];
    }
    for (u32 k = 0; k < d.ncon; k++) {
        u32 rec[8];
        const sc h = sc_half(eval_scalar(ws, d.con[k].s, item));
        if (wide) sc_bias65536(rec, h); else sc_bias4096(rec, h);
        for (int w = 0; w < 8; w++) scratch[((d.nvar + k) * 8 + w) * scratch_stride] = rec[w];
    }
    gc cacc = gc_identity();
    for (int i = 63; i >= 0; i--) {
#if defined(__CUDA_ARCH__)
        if ((i & AFX_SYNC_MASK) == AFX_SYNC_MASK) AFX_STEP_SYNC();
#endif
        if (i != 63) gc_dbl4(cacc);
#if defined(__CUDA_ARCH__) && defined(AFX_SYNC_FINE)
        AFX_STEP_SYNC();
#endif
        for (u32 k = 0; k < d.nvar; k++) {
            u32 word = scratch[(k * 8 + (i >> 3)) * scratch_stride];
            int dig = ((int)(word << (28 - 4 * (i & 7)))) >> 28;
            if (dig != 0) {
                u32 neg = ((u32)dig >> 31) ^ d.var[k].neg;
                u32 mag = (u32)(dig < 0 ? -dig : dig);
                pniels e = load_pniels(table_ptr(ws, d.var[k].table_slot, item) + 32 * (mag - 1));
                e = pniels_cneg(e, neg);
                GE_LADDER_ADD(cacc, e);
            }
        }
        // a constant term contributes one radix-4096 digit every third window (22 mixed additions per term), or one radix-2^16
        // digit every fourth (16 per term) when the issuer's wide tables exist
        if (wide ? (i & 3) == 0 : i % 3 == 0) {
            for (u32 k = 0; k < d.ncon; k++) {
                const u32* rec = scratch + (d.nvar + k) * 8 * scratch_stride;
                int dig = wide ? sc_digit65536(rec, scratch_stride, i >> 2) : sc_digit4096(rec, scratch_stride, i / 3);
                if (dig != 0) {
                    u32 neg = ((u32)dig >> 31) ^ d.con[k].neg;
                    u32 mag = (u32)(dig < 0 ? -dig : dig);
                    aniels e = load_aniels((wide ? ws.ctabs16 + (size_t)d.con[k].ctab * CTAB16_ENTRIES * 24 : ctab_of(k)) + 24 * (size_t)(mag - 1));
                    e = aniels_cneg(e, neg);
                    GE_LADDER_MADD(cacc, e);
                }
            }
        }
    }
    if (active) store_ge(commit_q_ptr(ws, d.out_slot, item), gc_to_ge(cacc));
}

// ---- stage: commitment encoding ----------------------------------------------------------------------------------
// Encodes the verify MSMs' results: commit[slot] = the encoding of 2 * commit_q[slot] for the n slots slots[0 .. n) of one
// item, with one field inversion for all of them (ge.cuh:dac_begin).  2Q encodes as R: every base of a verify MSM is a decoded
// point or a sum of such points, so it lies in 2E, and 2Q - R = sum k_j * l * P_j (k_j in {0, 1}) is 4-torsion.  The prefix
// products of the batch are kept in the commit words they are about to be replaced with.
AFX_HD void commit_encode_job(const Workspace& ws, const u32* slots, u32 n, u32 item) {
    fe acc = fe_one();
    for (u32 k = 0; k < n; k++) {
        u32 zero;
        const fe x = dac_den(dac_begin(load_ge(commit_q_ptr(ws, slots[k], item))), zero);
        store_fe(commit_ptr(ws, slots[k], item), acc);
        acc = fe_mul(acc, x);
    }
    fe inv = fe_invert(acc);
    for (u32 k = n; k-- > 0;) {
        u32 zero;
        const dac_state st = dac_begin(load_ge(commit_q_ptr(ws, slots[k], item)));
        const fe x = dac_den(st, zero);
        u32* out = commit_ptr(ws, slots[k], item);
        const fe inv_k = fe_mul(inv, load_fe(out));
        inv = fe_mul(inv, x);
        enc32 e = dac_finish(st, inv_k, zero);
        store8(out, e.w);
    }
}

// ---- stage: constant-schedule msm (Issuer::issue) ----------------------------------------------------------------
// Same job shape as msm_job but every scalar is a secret (issuer key material, per-item blindings, t): all terms use
// radix-16 digits, no digit is skipped and table entries are fetched by scan-and-mask, so neither the instruction
// stream nor the address stream depends on a scalar (dalek's constant-time `*` / multiscalar_mul, amacs.rs:267-270,
// zkp prove_compact).  scratch: (nvar + ncon) * 8 words per item.
AFX_HD void msm_ct_job(const Workspace& ws, const MsmDesc& d, u32 item, u32* scratch, u32 scratch_stride, bool active = true) {
    if (d.flags & MSM_COMB) {      // constant bases only: radix-16 comb with constant-address scans, no doublings
        gc cacc = gc_identity();
        for (u32 k = 0; k < d.ncon; k++) {
            u32 rec[8];
            sc_recode16(rec, eval_scalar(ws, d.con[k].s, item));
            const u32* comb = ws.comb + (size_t)d.con[k].ctab * COMB_WINDOWS * COMB_ENTRIES * 24;
            for (int i = 0; i < COMB_WINDOWS; i++) {
                aniels e = aniels_scan_select8(comb + (size_t)i * COMB_ENTRIES * 24, sc_digit16(rec, i), d.con[k].neg);
                GE_LADDER_MADD(cacc, e);
            }
            for (int i = 0; i < 8; i++) rec[i] = 0;
        }
        ge acc = gc_to_ge(cacc);
        if (d.flags & MSM_ADD_EXT) acc = ge_add(acc, load_ge(ext_ptr(ws, d.add_ext, item)));
        u32 w[8];
        ge_compress(w, acc);
        if (active) store8(commit_ptr(ws, d.out_slot, item), w);
        return;
    }
    for (u32 k = 0; k < (u32)d.nvar + d.ncon; k++) {
        u32 rec[8];
        sc_recode16(rec, eval_scalar(ws, k < d.nvar ? d.var[k].s : d.con[k - d.nvar].s, item));
        for (int w = 0; w < 8; w++) scratch[(k * 8 + w) * scratch_stride] = rec[w];
    }
    gc cacc = gc_identity();
    for (int i = 63; i >= 0; i--) {
#if defined(__CUDA_ARCH__)
        if ((i & AFX_CT_SYNC_MASK) == AFX_CT_SYNC_MASK) AFX_CT_STEP_SYNC();
#endif
        if (i != 63) gc_dbl4(cacc);
#if defined(__CUDA_ARCH__) && defined(AFX_SYNC_FINE)
        AFX_STEP_SYNC();
#endif
        for (u32 k = 0; k < d.nvar; k++) {
            u32 word = scratch[(k * 8 + (i >> 3)) * scratch_stride];
            int dig = ((int)(word << (28 - 4 * (i & 7)))) >> 28;
            pniels e = pniels_scan_select_t(atab_ptr(ws, d.var[k].table_slot, item), dig, d.var[k].neg);
#ifndef AFX_NO_CT_PREFETCH
            prefetch_atab(atab_ptr(ws, d.var[k + 1 < d.nvar ? k + 1 : 0].table_slot, item & ~31u));   // next scan, hidden behind this add
#endif
            GE_LADDER_ADD(cacc, e);
        }
        for (u32 k = 0; k < d.ncon; k++) {
            u32 word = scratch[((d.nvar + k) * 8 + (i >> 3)) * scratch_stride];
            int dig = ((int)(word << (28 - 4 * (i & 7)))) >> 28;
            aniels e = aniels_scan_select8(ws.ctabs + (size_t)d.con[k].ctab * CTAB_ENTRIES * 24, dig, d.con[k].neg);
            GE_LADDER_MADD(cacc, e);
        }
    }
    for (u32 k = 0; k < ((u32)d.nvar + d.ncon) * 8; k++) scratch[k * scratch_stride] = 0;   // wipe the recoded secrets
    ge acc = gc_to_ge(cacc);
    if (d.flags & MSM_ADD_W) acc = ge_add_pn(acc, load_pniels(ws.W_pniels));
    if (d.flags & MSM_ADD_EXT) acc = ge_add(acc, load_ge(ext_ptr(ws, d.add_ext, item)));
    u32 w[8];
    ge_compress(w, acc);
    if (active) store8(commit_ptr(ws, d.out_slot, item), w);
}

// ---- stage: derived scalars (prover paths) ---------------------------------------------------------------------------
AFX_HD void derive_program_job(const Workspace& ws, const DeriveOp* ops, u32 nops, u32 item) {
    for (u32 k = 0; k < nops; k++) {
        const DeriveOp& d = ops[k];
        sc r;
        if (d.op == DV_WIDE) {     // Scalar::random(rng) = 64 rng bytes reduced mod l (amacs.rs:289; zkp prove_compact's blindings)
            u32 x[16];
            load8(x, field_ptr(ws, d.a, item)); load8(x + 8, field_ptr(ws, d.b, item));
            r = sc_reduce512(x);
        } else {
            sc a = load_sc(scalar_ref_ptr(ws, d.a, item)), b = load_sc(scalar_ref_ptr(ws, d.b, item));
            if (d.op == DV_MUL) r = sc_mul(a, b);
            else if (d.op == DV_NEGMUL) r = sc_neg(sc_mul(a, b));
            else r = sc_muladd(b, load_sc(scalar_ref_ptr(ws, d.c, item)), a);
        }
        store8(ws.derived + ((size_t)k * ws.count + item) * 8, r.v);
    }
}

// ---- stage: prover output --------------------------------------------------------------------------------------------
// A request the Rust types could never hold (status != 0) yields all-zero words.
AFX_HD void out_word_job(const Workspace& ws, const OutWord& d, u32 word, u32 item, u32* out /*[n_out][count][8]*/) {
    u32 w[8];
    if (ws.status[item] != 0) { for (int i = 0; i < 8; i++) w[i] = 0; }
    else if (d.kind == OW_FIELD) load8(w, field_ptr(ws, d.a, item));
    else if (d.kind == OW_COMP) load8(w, comp_ptr(ws, d.a, item));
    else if (d.kind == OW_COMMIT) load8(w, commit_ptr(ws, d.a, item));
    else if (d.kind == OW_DERIVED) load8(w, scalar_ref_ptr(ws, SREF_DERIVED | d.a, item));
    else if (d.kind == OW_CHAL) load8(w, ws.chal + ((size_t)d.a * ws.count + item) * 8);
    else {
        sc c = load_sc(ws.chal + ((size_t)d.a * ws.count + item) * 8);
        sc b = load_sc(scalar_ref_ptr(ws, d.c, item));
        sc s;
        if (d.b == 0xffff) { s = sc_zero(); s.v[0] = 1; } else s = load_sc(scalar_ref_ptr(ws, d.b, item));
        sc r = sc_muladd(s, c, b);
        for (int i = 0; i < 8; i++) w[i] = r.v[i];
    }
    store8(out + ((size_t)word * ws.os_word + (size_t)item * ws.os_item + ws.os_base) * 8, w);
}

// ---- stage: commitment comparison (BatchableProof, exact path) -------------------------------------------------------
// The recomputed sum resp_k*P_k - c*LHS must equal the commitment on the wire (zkp verify_batchable, SURVEY 8f rank 2).
struct CmpPair { u16 commit_slot, field; };
AFX_HD void commit_compare_job(const Workspace& ws, const CmpPair& p, u32 item) {
    u32 a[8], b[8];
    // 0x8000 | field: compare two wire words (linked presentations: C_y[0] must be the proof of encryption's C_y_1)
    load8(a, (p.commit_slot & 0x8000u) ? field_ptr(ws, p.commit_slot & 0x7fffu, item) : commit_ptr(ws, p.commit_slot, item));
    load8(b, field_ptr(ws, p.field, item));
    u32 x = 0;
    for (int i = 0; i < 8; i++) x |= a[i] ^ b[i];
    if (x) status_or(ws, item, ST_CHALLENGE);
}

// ---- random-linear-combination verification of BatchableProofs (SURVEY 8f rank 2) -------------------------------------------
// Every constraint j of every item i of a chunk must satisfy  E_ij = sum_k s_k*P_k - c*LHS - R = 0.  One check replaces all of
// them:  sum_ij rho_ij * E_ij == 0  with independent 127-bit rho_ij derived from a caller-supplied seed.  The sum is one big
// multiscalar multiplication: per-item points (ladder bases, LHS points, wire commitments) go through a Pippenger bucket
// method across the whole chunk; the per-issuer generators only need the chunk-wide sums of their coefficients.
constexpr int RLC_MAX_INPUTS = 6 * MAX_ATTRS + 16, RLC_MAX_CTERMS = 4 * MAX_ATTRS + 16, RLC_MAX_CONS = 6 * MAX_ATTRS + 8;
struct RlcDesc {
    u16 ncons, ninputs, ncterms, pad;
    u16 first_input[RLC_MAX_CONS + 1];   // inputs of constraint j: [first_input[j], first_input[j+1]); the last one is the wire commitment
    u16 first_cterm[RLC_MAX_CONS + 1];
    u16 in_ext[RLC_MAX_INPUTS];          // extended-coordinates slot of input k
    u16 in_neg[RLC_MAX_INPUTS];
    ScalarSrc in_s[RLC_MAX_INPUTS];      // its scalar (op 0xffff = the constant 1, used for the commitment with in_neg = 1)
    u16 ct_ctab[RLC_MAX_CTERMS];         // generator of constant term t
    u16 ct_neg[RLC_MAX_CTERMS];
    ScalarSrc ct_s[RLC_MAX_CTERMS];
};
struct RlcBuffers {
    u32* scal;      // [ninputs][count][8]   coefficient of every per-item point
    u32* cterm;     // [ncterms][count][8]   coefficient contributions of the generators
    u32* csum;      // [ncterms][8]          their chunk-wide sums mod l
    u32* keys;      // [nwin][N]             (bucket << 1) | sign of input n in window w
    u32* sorted;    // [nwin][N]             inputs ordered by bucket: (n << 1) | sign
    u32* hist;      // [nwin][nb + 1]        bucket sizes -> exclusive offsets
    u32* cursor;    // [nwin][nb + 1]
    u32* buckets;   // [nwin][nb][32]        bucket sums (extended coordinates)
    u32* wsum;      // [nwin][32]            per-window sums
    u32* result;    // [9]                   compress(total) and the verdict word
    u32 N, nwin, c, nb;    // inputs of the pass, windows, window bits, buckets per window = 2^(c-1)
    u32 lo, cnt;           // the pass covers items [lo, lo + cnt) of the chunk (bisection of a chunk whose combination did not vanish); N = cnt * ninputs
    u64 seed[4];
};

// rho_ij: 128 bits out of Keccak-f[1600](seed || item || block), twelve per permutation
AFX_HD void rlc_rho_block(const RlcBuffers& rb, u32 item, u32 block, u64* st) {
    for (int i = 0; i < 25; i++) st[i] = 0;
    for (int i = 0; i < 4; i++) st[i] = rb.seed[i];
    st[4] = item; st[5] = block; st[6] = 0x434c522d58464175ull;   // "uAFX-RLC"
    keccak_f1600(st);
}
AFX_HD sc rlc_rho(const u64* st, u32 j) {
    sc r = sc_zero();
    u64 lo = st[2 * (j % 12)], hi = st[2 * (j % 12) + 1];
    // 127 bits: with bit 127 clear the signed-digit recoding of a bare rho (the commitments' coefficient) never carries out of
    // its top window -- a carry would put half of all commitments of the chunk into bucket 1 of the next window
    r.v[0] = (u32)lo; r.v[1] = (u32)(lo >> 32); r.v[2] = (u32)hi; r.v[3] = (u32)(hi >> 32) & 0x7fffffffu;
    return r;
}
// one thread per item (absolute index in [lo, lo + cnt)): the coefficient of every input and constant term
AFX_HD void rlc_scalars_job(const Workspace& ws, const RlcDesc& d, const RlcBuffers& rb, u32 item) {
    u64 st[25];
    for (u32 j = 0; j < d.ncons; j++) {
        if (j % 12 == 0) rlc_rho_block(rb, item, j / 12, st);
        sc rho = rlc_rho(st, j);
        for (u32 k = d.first_input[j]; k < d.first_input[j + 1]; k++) {
            // the sign of an input is applied to its point in the bucket pass, not to the scalar: -rho mod l would share its
            // upper ~125 bits with every other 128-bit rho and pile all those inputs into the same few buckets
            sc v = d.in_s[k].op == 0xffff ? rho : sc_mul(rho, eval_scalar(ws, d.in_s[k], item));
            store8(rb.scal + ((size_t)k * rb.cnt + (item - rb.lo)) * 8, v.v);
        }
        for (u32 t = d.first_cterm[j]; t < d.first_cterm[j + 1]; t++) {
            sc v = sc_mul(rho, eval_scalar(ws, d.ct_s[t], item));
            if (d.ct_neg[t]) v = sc_neg(v);
            store8(rb.cterm + ((size_t)t * rb.cnt + (item - rb.lo)) * 8, v.v);
        }
    }
}
// sum of a column of canonical scalars mod l (sequential form; the device kernel strides and tree-reduces 9-word partials)
AFX_HD void rlc_add288(u32* acc /*9 words*/, const u32* v /*8 words*/) {
    u64 c = 0;
    for (int i = 0; i < 8; i++) { c += (u64)acc[i] + v[i]; acc[i] = (u32)c; c >>= 32; }
    acc[8] += (u32)c;
}
AFX_HD void rlc_add288x(u32* acc, const u32* v /*9 words*/) {
    u64 c = 0;
    for (int i = 0; i < 9; i++) { c += (u64)acc[i] + v[i]; acc[i] = (u32)c; c >>= 32; }
}
AFX_HD sc rlc_reduce288(const u32* acc) {
    u32 x[16];
    for (int i = 0; i < 16; i++) x[i] = i < 9 ? acc[i] : 0;
    return sc_reduce512(x);
}
// signed base-2^c digits of a canonical scalar: digit w in [-2^(c-1), 2^(c-1)]
AFX_HD void rlc_digits_job(const RlcDesc& d, const RlcBuffers& rb, u32 n) {
    u32 v[9]; load8(v, rb.scal + (size_t)n * 8); v[8] = 0;
    const u32 flip = d.in_neg[n / rb.cnt] & 1u;
    u32 carry = 0;
    const u32 half = 1u << (rb.c - 1), mask = (1u << rb.c) - 1u;
    for (u32 w = 0; w < rb.nwin; w++) {
        u32 bit = w * rb.c, word = bit >> 5, sh = bit & 31;
        u64 two = word < 8 ? ((u64)v[word] | ((u64)v[word + 1] << 32)) : 0;
        u32 dgt = (u32)((two >> sh) & mask) + carry;
        u32 neg = dgt > half;
        carry = neg;
        u32 mag = neg ? (1u << rb.c) - dgt : dgt;
        rb.keys[(size_t)w * rb.N + n] = (mag << 1) | (neg ^ flip);
        if (mag) {
#if defined(__CUDA_ARCH__)
            atomicAdd(rb.hist + (size_t)w * (rb.nb + 1) + mag, 1u);
#else
            rb.hist[(size_t)w * (rb.nb + 1) + mag]++;
#endif
        }
    }
}
// hist[w][b] -> exclusive offsets (in place), cursor = copy; hist[w][0] is unused (digit 0 adds nothing)
AFX_HD void rlc_scan_job(const RlcBuffers& rb, u32 w) {
    u32* h = rb.hist + (size_t)w * (rb.nb + 1);
    u32* cur = rb.cursor + (size_t)w * (rb.nb + 1);
    u32 run = 0;
    for (u32 b = 1; b <= rb.nb; b++) { u32 cnt = h[b]; h[b] = run; cur[b] = run; run += cnt; }
    h[0] = run;   // total number of non-zero digits of the window
}
AFX_HD void rlc_scatter_job(const RlcBuffers& rb, u32 n) {
    for (u32 w = 0; w < rb.nwin; w++) {
        u32 key = rb.keys[(size_t)w * rb.N + n], mag = key >> 1;
        if (!mag) continue;
        u32* cur = rb.cursor + (size_t)w * (rb.nb + 1) + mag;
#if defined(__CUDA_ARCH__)
        u32 pos = atomicAdd(cur, 1u);
#else
        u32 pos = (*cur)++;
#endif
        rb.sorted[(size_t)w * rb.N + pos] = (n << 1) | (key & 1u);
    }
}
// one thread per (window, bucket): the sum of the bucket's points
AFX_HD void rlc_bucket_job(const Workspace& ws, const RlcDesc& d, const RlcBuffers& rb, u32 w, u32 b /*1..nb*/) {
    const u32* h = rb.hist + (size_t)w * (rb.nb + 1);
    u32 lo = h[b], hi = b < rb.nb ? h[b + 1] : h[0];
    ge acc = ge_identity();
    for (u32 q = lo; q < hi; q++) {
        u32 e = rb.sorted[(size_t)w * rb.N + q], n = e >> 1;
        u32 k = n / rb.cnt, item = rb.lo + (n - k * rb.cnt);
        ge p = load_ge(ext_ptr(ws, d.in_ext[k], item));
        if (e & 1u) p = ge_neg(p);
        acc = ge_add(acc, p);
    }
    store_ge(rb.buckets + ((size_t)w * rb.nb + (b - 1)) * 32, acc);
}
AFX_HD ge ge_mul_small(const ge& p, u32 m) {     // m < 2^16, public
    ge acc = ge_identity();
    pniels pn = ge_to_pniels(p);
    for (int bit = 15; bit >= 0; bit--) {
        acc = ge_dbl(acc, true);
        if ((m >> bit) & 1u) acc = ge_add_pn(acc, pn, true);
    }
    return acc;
}
// contribution of buckets [lo, hi] (1-based) of window w to sum_b b*B_b: running sums, then (lo-1) * (segment sum)
AFX_HD ge rlc_segment_job(const RlcBuffers& rb, u32 w, u32 lo, u32 hi) {
    ge run = ge_identity(), tot = ge_identity();
    for (u32 b = hi; b >= lo; b--) {
        run = ge_add(run, load_ge(rb.buckets + ((size_t)w * rb.nb + (b - 1)) * 32));
        tot = ge_add(tot, run);
        if (b == lo) break;
    }
    if (lo > 1) tot = ge_add(tot, ge_mul_small(run, lo - 1));
    return tot;
}
// total = sum_w 2^(c*w) * S_w + sum_t csum[t] * G_t ; result = its encoding (all-zero iff the combination vanishes)
AFX_HD ge rlc_horner(const RlcBuffers& rb) {
    ge acc = ge_identity();
    for (int w = (int)rb.nwin - 1; w >= 0; w--) {
        for (u32 k = 0; k < rb.c; k++) acc = ge_dbl(acc, true);
        acc = ge_add(acc, load_ge(rb.wsum + (size_t)w * 32));
    }
    return acc;
}
AFX_HD ge rlc_cterm_point(const Workspace& ws, const RlcDesc& d, const RlcBuffers& rb, u32 t) {   // csum[t] * G_t on the comb tables
    ge acc = ge_identity();
    u32 rec[8];
    sc_recode16(rec, sc_from_words(rb.csum + 8 * t));
    const u32* comb = ws.comb + (size_t)d.ct_ctab[t] * COMB_WINDOWS * COMB_ENTRIES * 24;
    for (int i = 0; i < COMB_WINDOWS; i++) {
        int dig = sc_digit16(rec, i);
        if (dig != 0) {
            u32 mag = (u32)(dig < 0 ? -dig : dig);
            acc = ge_madd(acc, aniels_cneg(load_aniels(comb + ((size_t)i * COMB_ENTRIES + (mag - 1)) * 24), (u32)dig >> 31), true);
        }
    }
    return acc;
}
AFX_HD void rlc_publish(const RlcBuffers& rb, const ge& total) {
    u32 wv[8], x = 0;
    ge_compress(wv, total);
    for (int i = 0; i < 8; i++) { rb.result[i] = wv[i]; x |= wv[i]; }
    rb.result[8] = x == 0;
}
AFX_HD void rlc_final_job(const Workspace& ws, const RlcDesc& d, const RlcBuffers& rb) {
    ge acc = rlc_horner(rb);
    for (u32 t = 0; t < d.ncterms; t++) acc = ge_add(acc, rlc_cterm_point(ws, d, rb, t));
    rlc_publish(rb, acc);
}

// ---- stage: transcript -------------------------------------------------------------------------------------------
AFX_HD const u32* tx_src(const Workspace& ws, u32 kind, u32 idx, u32 item) {
    if (kind == SRC_FIELD) return field_ptr(ws, idx, item);
    if (kind == SRC_COMP) return comp_ptr(ws, idx, item);
    return commit_ptr(ws, idx, item);
}
AFX_HD void transcript_job(const Workspace& ws, const TxDesc& d, u32 item) {
    u64 st[25];
    for (int i = 0; i < 25; i++) st[i] = d.midstate[i];
    for (u32 k = 0; k < d.nid; k++) {
        const TxIdCheck& c = ws.idchecks[d.id_ofs + k];
        u32 w[8]; load8(w, tx_src(ws, c.src_kind, c.src_idx, item));
        u32 x = 0;
        for (int i = 0; i < 8; i++) x |= w[i];
        if (x == 0) status_or(ws, item, ST_IDENTITY);
    }
    u32 h = 0;
    for (u32 b = 0; b < d.nblocks; b++) {
        u64 buf[21];
        const u64* mask = ws.lanes + (size_t)(d.block_ofs + b) * 21;
        for (int i = 0; i < 21; i++) buf[i] = mask[i];
        while (h < d.nholes && ws.holes[d.hole_ofs + h].block == b) {
            const TxHole& hole = ws.holes[d.hole_ofs + h];
            u32 w[8]; load8(w, tx_src(ws, hole.src_kind, hole.src_idx, item));
            for (u32 t = 0; t < hole.len; t++) {
                u32 sb = hole.src_off + t, db = hole.off + t;
                u64 byte = (w[sb >> 2] >> (8 * (sb & 3))) & 0xffu;
                buf[db >> 3] ^= byte << (8 * (db & 7));
            }
            h++;
        }
        for (int i = 0; i < 21; i++) st[i] ^= buf[i];
        keccak_f1600(st);
    }
    u32 x[16];
    for (int i = 0; i < 8; i++) { x[2 * i] = (u32)st[i]; x[2 * i + 1] = (u32)(st[i] >> 32); }
    sc c = sc_reduce512(x);
    if (d.chal_field != 0xffff) {      // verifier: compare with the claimed challenge; prover (Issuer::issue): just emit it
        sc claimed = sc_from_words(field_ptr(ws, d.chal_field, item));
        if (!sc_equal(c, claimed)) status_or(ws, item, ST_CHALLENGE);
    }
    if (ws.chal) store8(ws.chal + ((size_t)d.out_slot * ws.count + item) * 8, c.v);
}

// ---- setup (per issuer): constant tables --------------------------------------------------------------------------
// entry (base b, multiple m in 1..2048) of the radix-4096 table: m*P in affine Niels form.
AFX_HD u32 ctab_entry_job(const u32* enc /*8 words*/, u32 m, u32* out /*24 words*/, int bits = 12) {
    ge p; u32 ok = ge_decompress(p, enc);
    ge acc = ge_identity();
    pniels pn = ge_to_pniels(p);
    for (int bit = bits - 1; bit >= 0; bit--) {
        acc = ge_dbl(acc, true);
        if ((m >> bit) & 1u) acc = ge_add_pn(acc, pn, true);
    }
    // 1/Z = Z^(p-2) = (Z^(2^252-3))^8 * Z^3 ... use pow_p58: Z^(p-2) = Z^(2^255-21) = (Z^(2^252-3))^(8) * Z^3
    fe z = acc.Z;
    fe t = fe_pow_p58(z);               // z^(2^252-3)
    t = fe_sqn(t, 3);                   // z^(2^255-24)
    fe zinv = fe_mul(t, fe_mul(fe_sq(z), z));  // * z^3 -> z^(2^255-21)
    fe x = fe_mul(acc.X, zinv), y = fe_mul(acc.Y, zinv);
    store_fe(out, fe_add(y, x));
    store_fe(out + 8, fe_sub(y, x));
    store_fe(out + 16, fe_mul(fe_mul(x, y), FE_D2()));
    return ok;
}

// ---- primitive self-test (parity hooks for the field / group / scalar code, independent of the protocol flows) ------
enum : u32 { PRIM_DECOMPRESS_COMPRESS = 0, PRIM_FROM_UNIFORM = 1, PRIM_SCALARMULT = 2, PRIM_WIDE_REDUCE = 3, PRIM_SC_MULADD = 4,
             PRIM_FE_MUL = 5, PRIM_FE_SQ = 6, PRIM_FE_ADD = 7, PRIM_FE_SUB = 8, PRIM_FE_CHAIN = 9, PRIM_LADDER_STEP = 10, PRIM_RECODE4096 = 11,
             PRIM_RECODE65536 = 12 };
// in/out are [count][words][8] item-major.  Returns per item ok (1) / rejected encoding (0) in flags.
//   0: in 1 word (encoding)          -> out 1 word: compress(decompress(in)); flag = decodes
//   1: in 2 words (64 uniform bytes) -> out 1 word: compress(from_uniform_bytes(in))
//   2: in 2 words (scalar, encoding) -> out 1 word: compress(scalar * point)  (fixed-window ladder over the [1P..8P] table)
//   3: in 2 words (64 bytes)         -> out 1 word: the integer mod l
//   4: in 3 words (a, b, c)          -> out 1 word: a*b + c mod l
//   5..8: in 2 words (a, b: raw 256-bit limb vectors, NOT reduced -- any value in [0, 2^256) is a legal lazily-reduced
//         field element) -> out 1 word: canonical bytes of a*b, a^2, a+b, a-b mod p
//   9: in 2 words (a, b raw)         -> out 1 word: canonical ((a+b)*(a-b))^2 * (a-b) + a  (unreduced intermediates chained)
//  10: in 2 words (scalar, encoding) -> out 1 word: compress(scalar * point) through the completed-coordinates ladder forms
//         (gc_dbl4 / gc_add_pn_inl / gc_to_ge) that k_ladders and k_msm_ct use
//  11: in 1 word (a 256-bit integer)   -> out 1 word: sum_j digit_j * 4096^j mod 2^256 of its biased radix-4096 recoding
//         (sc_bias4096 / sc_digit4096); equals the input for every input below 2^256 - 2^252; flag = every |digit| <= 2048
//  12: in 1 word (a 256-bit integer)   -> out 1 word: sum_j digit_j * 65536^j mod 2^256 of its biased radix-2^16 recoding
//         (sc_bias65536 / sc_digit65536); equals the input for every input below 2^256 - 2^240; flag = every low digit within
//         [-32768, 32767] and the top digit at most 2^13 + 1
AFX_HD void primitive_job(u32 op, const u32* in, u32* out, u32* flags, u32 item) {
    u32 w[8]; u32 ok = 1;
    if (op == PRIM_DECOMPRESS_COMPRESS) {
        ge p; ok = ge_decompress(p, in + (size_t)item * 8);
        ge_compress(w, p);
    } else if (op == PRIM_FROM_UNIFORM) {
        ge_compress(w, ge_from_uniform(in + (size_t)item * 16));
    } else if (op == PRIM_SCALARMULT) {
        ge p; ok = ge_decompress(p, in + (size_t)item * 16 + 8);
        sc s = sc_from_words(in + (size_t)item * 16);
        ok &= sc_is_canonical(s);
        u32 rec[8]; sc_recode16(rec, s);
        pniels tab[8];
        struct Keep { pniels* t; AFX_HD void operator()(int e, const pniels& n) const { t[e] = n; } };
        Keep keep{tab}; ge_table8(p, keep);
        ge acc = ge_identity();
        for (int i = 63; i >= 0; i--) {
            if (i != 63) { acc = ge_dbl(acc, false); acc = ge_dbl(acc, false); acc = ge_dbl(acc, false); acc = ge_dbl(acc, true); }
            int dig = sc_digit16(rec, i);
            if (dig != 0) { u32 mag = (u32)(dig < 0 ? -dig : dig); acc = ge_add_pn(acc, pniels_cneg(tab[mag - 1], (u32)dig >> 31), true); }
        }
        ge_compress(w, acc);
    } else if (op == PRIM_WIDE_REDUCE) {
        sc r = sc_reduce512(in + (size_t)item * 16);
        for (int i = 0; i < 8; i++) w[i] = r.v[i];
    } else if (op >= PRIM_FE_MUL && op <= PRIM_FE_CHAIN) {
        fe a, b, r;
        for (int i = 0; i < 8; i++) { a.v[i] = in[(size_t)item * 16 + i]; b.v[i] = in[(size_t)item * 16 + 8 + i]; }
        if (op == PRIM_FE_MUL) r = fe_mul(a, b);
        else if (op == PRIM_FE_SQ) r = fe_sq(a);
        else if (op == PRIM_FE_ADD) r = fe_add(a, b);
        else if (op == PRIM_FE_SUB) r = fe_sub(a, b);
        else { fe d = fe_sub(a, b); r = fe_add(fe_mul(fe_sq(fe_mul(fe_add(a, b), d)), d), a); }
        fe_to_bytes_words(w, r);
    } else if (op == PRIM_RECODE4096 || op == PRIM_RECODE65536) {
        const bool wide = op == PRIM_RECODE65536;
        sc a; for (int i = 0; i < 8; i++) a.v[i] = in[(size_t)item * 8 + i];
        u32 rec[8];
        if (wide) sc_bias65536(rec, a); else sc_bias4096(rec, a);
        for (int i = 0; i < 8; i++) w[i] = 0;
        for (int j = 0; j < (wide ? 16 : 22); j++) {
            int dig = wide ? sc_digit65536(rec, 1, j) : sc_digit4096(rec, 1, j);
            ok &= wide ? (u32)(j < 15 ? dig >= -32768 && dig <= 32767 : dig <= 8193) : (u32)(dig >= -2048 && dig <= 2048);
            const u32 bit = (wide ? 16u : 12u) * (u32)j, w0 = bit >> 5;
            const long long v = (long long)dig * (long long)(1ull << (bit & 31u));
            const u32 ext = v < 0 ? 0xffffffffu : 0u;
            u64 c = 0;
            for (u32 k = w0; k < 8; k++) {
                u32 part = k == w0 ? (u32)(u64)v : k == w0 + 1 ? (u32)((u64)v >> 32) : ext;
                c += (u64)w[k] + part; w[k] = (u32)c; c >>= 32;
            }
        }
    } else if (op == PRIM_LADDER_STEP) {
        ge p; ok = ge_decompress(p, in + (size_t)item * 16 + 8);
        sc s = sc_from_words(in + (size_t)item * 16);
        ok &= sc_is_canonical(s);
        u32 rec[8]; sc_recode16(rec, s);
        pniels tab[8];
        struct Keep { pniels* t; AFX_HD void operator()(int e, const pniels& n) const { t[e] = n; } };
        Keep keep{tab}; ge_table8(p, keep);
        gc cacc = gc_identity();
        for (int i = 63; i >= 0; i--) {
            if (i != 63) gc_dbl4(cacc);
            int dig = sc_digit16(rec, i);
            if (dig != 0) { u32 mag = (u32)(dig < 0 ? -dig : dig); pniels e = pniels_cneg(tab[mag - 1], (u32)dig >> 31); GE_LADDER_ADD(cacc, e); }
        }
        ge_compress(w, gc_to_ge(cacc));
    } else {
        const u32* q = in + (size_t)item * 24;
        sc r = sc_muladd(sc_from_words(q), sc_from_words(q + 8), sc_from_words(q + 16));
        for (int i = 0; i < 8; i++) w[i] = r.v[i];
    }
    for (int i = 0; i < 8; i++) out[(size_t)item * 8 + i] = w[i];
    flags[item] = ok;
}

// encoding of G_y[i] - G_y[0] (the base of the linked presentation's extra constraint), i = 1..ny-1
AFX_HD void link_entry_job(const u32* enc_gy /*[ny][8]*/, u32 i, u32* out /*8 words*/) {
    ge a, b; ge_decompress(a, enc_gy + 8 * i); ge_decompress(b, enc_gy);
    ge_compress(out, ge_sub(a, b));
}

// entry (base b, window i, multiple e in 1..8) of the radix-16 comb: (e * 16^i) * P in affine Niels form.
AFX_HD void comb_entry_job(const u32* enc /*8 words*/, u32 i, u32 e, u32* out /*24 words*/) {
    ge p; ge_decompress(p, enc);
    pniels pn = ge_to_pniels(p);
    ge acc = ge_identity();
    for (int bit = 3; bit >= 0; bit--) {
        acc = ge_dbl(acc, true);
        if ((e >> bit) & 1u) acc = ge_add_pn(acc, pn, true);
    }
    for (u32 k = 0; k < 4 * i; k++) acc = ge_dbl(acc, true);
    fe z = acc.Z;
    fe t = fe_sqn(fe_pow_p58(z), 3);
    fe zinv = fe_mul(t, fe_mul(fe_sq(z), z));
    fe x = fe_mul(acc.X, zinv), y = fe_mul(acc.Y, zinv);
    store_fe(out, fe_add(y, x));
    store_fe(out + 8, fe_sub(y, x));
    store_fe(out + 16, fe_mul(fe_mul(x, y), FE_D2()));
}

// ---- symmetric encryption of attributes (encoding.rs:56-82, symmetric.rs:89-96,135-143,197-215,252-261,273-289) ------------------
// Keypair::encrypt is a program of the prover stages (program.hpp:compile_encrypt); encoding and decryption are one thread per item.
// Keypair::derive is one thread per item for its hashes (keypair_scalars_job) and a program for pk (program.hpp:compile_keypair).
// Word w of the nw words of an item: item-major [count][nw][8] (the host calls) or struct-of-arrays [nw][count][8] (the *_device calls).
AFX_HD size_t sym_word(u32 count, u32 nw, u32 item_major, u32 w, u32 item) {
    return (item_major ? (size_t)item * nw + w : (size_t)w * count + item) * 8;
}

// Plaintext::from(&[u8; 30]): M1 = the first candidate 2i || data || j (j = 0..63, i = 0..127) that decompresses, h = SHA-512(data),
// M2 = from_uniform_bytes(h), m3 = h mod l.  Variable time in the number of candidates, as the reference's loop.  status 1 (all-zero
// words) when no candidate decodes, where the reference panics.
AFX_HD void encode_job(const uint8_t* data /*[count][30]*/, u32* pt, uint8_t* status, u32 count, u32 item_major, u32 item) {
    enc32 base;      // 0 || data || 0
    for (int w = 0; w < 8; w++) {
        u32 v = 0;
        for (int b = 0; b < 4; b++) { const int k = 4 * w + b - 1; if (k >= 0 && k < 30) v |= (u32)data[(size_t)item * 30 + k] << (8 * b); }
        base.w[w] = v;
    }
    u32 enc[8], found = 0;
    ge p;
    for (u32 k = 0; k < 64 * 128; k++) {
        for (int w = 0; w < 8; w++) enc[w] = base.w[w];
        enc[0] |= 2u * (k & 127u); enc[7] |= (k >> 7) << 24;
        if (ge_decompress(p, enc)) { found = 1; break; }
    }
    const digest64 h = sha512_30(base);
    u32 m2[8];
    ge_compress(m2, ge_from_uniform(h.w));
    const sc m3 = sc_reduce512(h.w);
    const u32 m = 0u - found;
    u32 m3w[8];
    for (int i = 0; i < 8; i++) { enc[i] &= m; m2[i] &= m; m3w[i] = m3.v[i] & m; }
    store8(pt + sym_word(count, 3, item_major, 0, item), enc);
    store8(pt + sym_word(count, 3, item_major, 1, item), m2);
    store8(pt + sym_word(count, 3, item_major, 2, item), m3w);
    status[item] = (uint8_t)(found ^ 1u);
}

// k * P for a secret k over P's [1P..8P] table (warp-transposed, scan-and-mask reads): 64 signed radix-16 digits, every digit added,
// so neither the instruction stream nor the address stream depends on k.  The digits stay in registers.
AFX_NI ge ct_ladder(const u32* tab, sc k) {
    u32 rec[8];
    sc_recode16(rec, k);
    gc acc = gc_identity();
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 63; i >= 0; i--) {
        if (i != 63) gc_dbl4(acc);
        u32 word = rec[0];
        for (int j = 1; j < 8; j++) word = (i >> 3) == j ? rec[j] : word;     // public index: selects, not a local-memory array
        pniels e = pniels_scan_select_t(tab, ((int)(word << (28 - 4 * (i & 7)))) >> 28);
        GE_LADDER_ADD(acc, e);
    }
    return gc_to_ge(acc);
}

// a0 + a1*m3 (a subroutine: its unrolled limb products would otherwise share the registers of decrypt_job's live points)
AFX_NI sc decrypt_u(const u32* kp, sc m3) { return sc_muladd(load_sc(kp + 16), m3, load_sc(kp + 8)); }

// Keypair::decrypt: M1' = E2 - a*E1, data' = compress(M1')[1..31], h = SHA-512(data'), M2' = from_uniform_bytes(h), m3' = h mod l;
// accept iff (a0 + a1*m3')*M2' == E1.  kp = a, a0, a1 (canonical).  tabs: warp-transposed ladder tables, one per item, used by both
// ladders.  Outputs (data [count][30], the Plaintext words when pt != null) are all-zero and status is 1 when E1 or E2 does not
// decode or the check fails (CredentialError::UndecryptableAttribute).
AFX_HD void decrypt_job(const u32* ct, const u32* kp, u32* tabs, uint8_t* data, u32* pt, uint8_t* status, u32 count, u32 item_major, u32 item) {
    // The outputs are written as soon as they exist and cleared if the check fails, so that nothing but `ok` and the pointers stays
    // live across the ladders (the calls would otherwise spill it).
    u32* tab = tabs + (size_t)(item / 32) * ATAB_BLOCK_WORDS + (item % 32) * 4;
    u32 w[8];
    load8(w, ct + sym_word(count, 2, item_major, 0, item));
    ge p;
    u32 ok = ge_decompress(p, w);
    store_table8(nullptr, p, tab);
    const ge aE1 = ct_ladder(tab, load_sc(kp));
    load8(w, ct + sym_word(count, 2, item_major, 1, item));
    ok &= ge_decompress(p, w);
    const enc32 m1 = ge_compress_v(ge_sub(p, aE1));
    uint8_t* d = data + (size_t)item * 30;
    for (int k = 0; k < 30; k++) d[k] = (uint8_t)(m1.w[(k + 1) >> 2] >> (8 * ((k + 1) & 3)));
    if (pt) store8(pt + sym_word(count, 3, item_major, 0, item), m1.w);
    const digest64 h = sha512_30(m1);
    p = ge_from_uniform(h.w);
    const sc m3 = sc_reduce512(h.w);
    if (pt) {
        ge_compress(w, p);
        store8(pt + sym_word(count, 3, item_major, 1, item), w);
        store8(pt + sym_word(count, 3, item_major, 2, item), m3.v);
    }
    store_table8(nullptr, p, tab);
    const ge E1 = ct_ladder(tab, decrypt_u(kp, m3));
    u32 e1[8];
    ge_compress(w, E1);
    load8(e1, ct + sym_word(count, 2, item_major, 0, item));
    u32 x = 0;
    for (int i = 0; i < 8; i++) x |= w[i] ^ e1[i];
    ok &= (u32)(x == 0);
    if (!ok) {     // the verdict is public
        for (int k = 0; k < 30; k++) d[k] = 0;
        for (int i = 0; i < 8; i++) w[i] = 0;
        if (pt) for (u32 k = 0; k < 3; k++) store8(pt + sym_word(count, 3, item_major, k, item), w);
    }
    status[item] = (uint8_t)(ok ^ 1u);
}

// The scalars of Keypair::derive (symmetric.rs:197-215): a = SHA-512(master secret), a0 = SHA-512(a), a1 = SHA-512(a0), each reduced
// wide mod l.  ms = [count][64] master secrets; rows = the struct-of-arrays rows [3][count][8] a, a0, a1, the fields of
// program.hpp:compile_keypair, whose comb computes pk.  No branch and no address depends on the master secret.
AFX_HD void keypair_scalars_job(const u32* ms, u32* rows, u32 count, u32 item) {
    msg64 m;
    load8(m.w, ms + (size_t)item * 16);
    load8(m.w + 8, ms + (size_t)item * 16 + 8);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (u32 k = 0; k < 3; k++) {
        const digest64 h = sha512_words(m, k == 0 ? 16u : 8u);
        const sc s = sc_reduce512(h.w);
        store8(rows + ((size_t)k * count + item) * 8, s.v);
        for (int i = 0; i < 8; i++) { m.w[i] = s.v[i]; m.w[8 + i] = 0; }
    }
}

// ---- mixed-shape verify calls: device-side bucketing of a pass of records of several shapes ------------------------------------
// A pass is `count` consecutive records as the caller concatenated them, record i being rec_words[ids[i]] words long.  Each shape's
// records are copied into its own item-major bucket (the *_wire layout), in record order, so that the shape's verify program runs on
// the bucket as it is.  The host scans the ids anyway (to validate them and count each shape); it records the running counts and
// the running word offset every BUCKET_TILE records, which leaves the device a rank and an offset within one tile per record.
constexpr u32 BUCKET_TILE = 256;
struct BucketArgs {
    const u32* records;      // the pass's records as received
    u32* fields;             // the buckets: shape s's bucket starts at word base_word[s]
    const uint8_t* ids;      // [count] shape id of every record
    const u32* rec_words;    // [n_shapes] record length in words (n_fields * 8)
    const u64* base_word;    // [n_shapes]
    const u32* vbase;        // [n_shapes] first index of shape s's bucket in the bucket-order verdict array
    const u32* tile_rank;    // [tiles][n_shapes] records of shape s in the pass before the tile
    const u64* tile_src;     // [tiles] word offset of the tile's first record in `records`
    u32* slot;               // [count] out: the record's index in the bucket-order verdict array
    u32 count, n_shapes;
};

// Record i: its index in the bucket-order verdict array, its word offset in the pass (src) and in the buckets (dst).  The rank
// within its shape counts the earlier records of the tile with the same id, so the bucket keeps the record order.  tile_ids are
// the ids of i's tile, rec_words the record lengths (the kernel passes its shared-memory copies).
AFX_HD u32 bucket_locate(const BucketArgs& a, const uint8_t* tile_ids, const u32* rec_words, u32 i, u64& src, u64& dst) {
    const u32 t = i / BUCKET_TILE, j_end = i % BUCKET_TILE, s = tile_ids[j_end];
    u32 rank = a.tile_rank[(size_t)t * a.n_shapes + s];
    u64 off = a.tile_src[t];
    for (u32 j = 0; j < j_end; j++) {
        const u32 sj = tile_ids[j];
        rank += sj == s;
        off += rec_words[sj];
    }
    src = off;
    dst = a.base_word[s] + (u64)rank * rec_words[s];
    return a.vbase[s] + rank;
}

// Copy one record's words in 16-byte quads, lane `lane` of `nlanes` taking every nlanes-th quad (a warp moves 512 contiguous bytes per step).
AFX_HD void bucket_copy(const u32* src, u32* dst, u32 words, u32 lane, u32 nlanes) {
    u32 q[4];
    for (u32 k = 4 * lane; k < words; k += 4 * nlanes) { load4(q, src + k); store4(dst + k, q); }
}

// ---- mixed-shape prover calls: the inverse of the bucketing, for the prover outputs -------------------------------------------
// Each shape's prover program writes its output records item-major into its own region (out_base[s]), in bucket order.  Every record
// goes back to its position in the pass, and its status byte with it.  The rank comes from the slot k_bucket_records wrote; the host
// records the running output word offset every BUCKET_TILE records, as it does for the inputs.
struct UnbucketArgs {
    const u32* outputs;             // the provers' output regions: shape s's starts at word out_base[s]
    u32* records;                   // out: the pass's output records in record order
    const uint8_t* ids;             // [count] shape id of every record
    const u32* out_words;           // [n_shapes] output record length in words
    const u64* out_base;            // [n_shapes]
    const u32* vbase;               // [n_shapes] first index of shape s in the bucket-order status array
    const u64* tile_dst;            // [tiles] word offset of the tile's first output record in `records`
    const u32* slot;                // [count] the record's index in the bucket-order status array (k_bucket_records)
    const uint8_t* bucket_status;   // [count] status in bucket order
    uint8_t* status;                // [count] out: status in record order
    u32 count, n_shapes;
};

// Record i: its status byte, its word offset in the output regions (src) and in the pass's output (dst).  tile_ids are the ids of
// i's tile, out_words the output record lengths (the kernel passes its shared-memory copies).
AFX_HD uint8_t unbucket_locate(const UnbucketArgs& a, const uint8_t* tile_ids, const u32* out_words, u32 i, u64& src, u64& dst) {
    const u32 t = i / BUCKET_TILE, j_end = i % BUCKET_TILE, s = tile_ids[j_end], slot = a.slot[i];
    u64 off = a.tile_dst[t];
    for (u32 j = 0; j < j_end; j++) off += out_words[tile_ids[j]];
    dst = off;
    src = a.out_base[s] + (u64)(slot - a.vbase[s]) * out_words[s];
    return a.bucket_status[slot];
}

}  // namespace afx
