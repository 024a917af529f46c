// ristretto255 / extended twisted Edwards (a = -1) group operations for sm_100a.
//
// Replaces the RistrettoPoint / CompressedRistretto operations aeonflux uses from curve25519-dalek:
// compress()/decompress() (/root/reference/src/nizk/presentation.rs:373-412, encryption.rs:172-185,
// issuance.rs:162-189), +/-/neg (presentation.rs:342-351, encryption.rs:183-185), and the point side of every
// scalar multiplication.  Outputs are compared with the reference only as compressed bytes, so any correct group
// algorithm gives identical bytes (SURVEY A.2).
#pragma once
#include "fe.cuh"

namespace afx {

struct ge { fe X, Y, Z, T; };            // extended coordinates, x = X/Z, y = Y/Z, xy = T/Z
struct pniels { fe YpX, YmX, Z, T2d; };  // projective Niels form of a variable point (128 B)
struct aniels { fe ypx, ymx, xy2d; };    // affine Niels form of a per-issuer constant point (96 B)

AFX_HD ge ge_identity() { ge r; r.X = fe_zero(); r.Y = fe_one(); r.Z = fe_one(); r.T = fe_zero(); return r; }
AFX_HD ge ge_neg(const ge& p) { ge r; r.X = fe_neg(p.X); r.Y = p.Y; r.Z = p.Z; r.T = fe_neg(p.T); return r; }
AFX_HD pniels pniels_identity() { pniels n; n.YpX = fe_one(); n.YmX = fe_one(); n.Z = fe_one(); n.T2d = fe_zero(); return n; }
AFX_HD aniels aniels_identity() { aniels n; n.ypx = fe_one(); n.ymx = fe_one(); n.xy2d = fe_zero(); return n; }

AFX_HD pniels ge_to_pniels(const ge& p) {
    pniels n; n.YpX = fe_add(p.Y, p.X); n.YmX = fe_sub(p.Y, p.X); n.Z = p.Z; n.T2d = fe_mul(p.T, FE_D2()); return n;
}
// conditional negation (branch-free): -(YpX, YmX, Z, T2d) = (YmX, YpX, Z, -T2d)
AFX_HD pniels pniels_cneg(const pniels& n, u32 neg) {
    pniels r; r.YpX = fe_select(n.YpX, n.YmX, neg); r.YmX = fe_select(n.YmX, n.YpX, neg); r.Z = n.Z; r.T2d = fe_cneg(n.T2d, neg); return r;
}
AFX_HD aniels aniels_cneg(const aniels& n, u32 neg) {
    aniels r; r.ypx = fe_select(n.ypx, n.ymx, neg); r.ymx = fe_select(n.ymx, n.ypx, neg); r.xy2d = fe_cneg(n.xy2d, neg); return r;
}

// p + n, 8M.  need_T = false skips the T output (valid when a doubling follows).
AFX_HD ge ge_add_pn_inl(const ge& p, const pniels& n, bool need_T = true) {
    fe PP = fe_mul(fe_add(p.Y, p.X), n.YpX);
    fe MM = fe_mul(fe_sub(p.Y, p.X), n.YmX);
    fe TT = fe_mul(p.T, n.T2d);
    fe ZZ = fe_mul(p.Z, n.Z);
    fe ZZ2 = fe_add(ZZ, ZZ);
    fe E = fe_sub(PP, MM), H = fe_add(PP, MM), G = fe_add(ZZ2, TT), F = fe_sub(ZZ2, TT);
    ge r; r.X = fe_mul(E, F); r.Y = fe_mul(G, H); r.Z = fe_mul(F, G);
    if (need_T) r.T = fe_mul(E, H); else r.T = fe_zero();
    return r;
}
AFX_NI ge ge_add_pn(ge p, pniels n, bool need_T = true) { return ge_add_pn_inl(p, n, need_T); }
// p + n for an affine Niels constant, 7M
AFX_HD ge ge_madd_inl(const ge& p, const aniels& n, bool need_T = true) {
    fe PP = fe_mul(fe_add(p.Y, p.X), n.ypx);
    fe MM = fe_mul(fe_sub(p.Y, p.X), n.ymx);
    fe TT = fe_mul(p.T, n.xy2d);
    fe ZZ2 = fe_add(p.Z, p.Z);
    fe E = fe_sub(PP, MM), H = fe_add(PP, MM), G = fe_add(ZZ2, TT), F = fe_sub(ZZ2, TT);
    ge r; r.X = fe_mul(E, F); r.Y = fe_mul(G, H); r.Z = fe_mul(F, G);
    if (need_T) r.T = fe_mul(E, H); else r.T = fe_zero();
    return r;
}
AFX_NI ge ge_madd(ge p, aniels n, bool need_T = true) { return ge_madd_inl(p, n, need_T); }
// 2p, 4S + 3M (+1M when T is needed).  Reads X, Y, Z only.
AFX_HD ge ge_dbl_inl(const ge& p, bool need_T = true) {
    fe XX = fe_sq(p.X), YY = fe_sq(p.Y), ZZ = fe_sq(p.Z);
    fe ZZ2 = fe_add(ZZ, ZZ);
    fe S = fe_sq(fe_add(p.X, p.Y));
    fe H = fe_add(YY, XX), G = fe_sub(YY, XX);
    fe E = fe_sub(S, H), F = fe_sub(ZZ2, G);
    ge r; r.X = fe_mul(E, F); r.Y = fe_mul(H, G); r.Z = fe_mul(G, F);
    if (need_T) r.T = fe_mul(E, H); else r.T = fe_zero();
    return r;
}
AFX_NI ge ge_dbl(ge p, bool need_T = true) { return ge_dbl_inl(p, need_T); }
// Ladder accumulator in "completed" coordinates (E, F, G, H): X = E*F, Y = G*H, Z = F*G, T = E*H.  Every ladder
// operation starts by forming only the products it reads -- a doubling X, Y, Z (3M), an addition X, Y, Z, T (4M) -- so
// T is never computed for a point that is doubled next: doubling 4S + 3M, add 4M + 4M, mixed add 4M + 3M, with no
// data-dependent choice anywhere (the rolled 4-doubling loop body is uniform).  One multiply fewer per doubling than
// carrying (X, Y, Z, T) through the rolled loop, where ptxas computes T in every iteration and selects.
struct gc { fe E, F, G, H; };
AFX_HD gc gc_identity() { gc r; r.E = fe_zero(); r.F = fe_one(); r.G = fe_one(); r.H = fe_one(); return r; }
AFX_HD ge gc_to_ge(const gc& c) {
    ge r; r.X = fe_mul(c.E, c.F); r.Y = fe_mul(c.G, c.H); r.Z = fe_mul(c.F, c.G); r.T = fe_mul(c.E, c.H); return r;
}
AFX_HD gc gc_dbl_inl(const gc& c) {
    fe X = fe_mul(c.E, c.F), Y = fe_mul(c.G, c.H), Z = fe_mul(c.F, c.G);
    fe XX = fe_sq(X), YY = fe_sq(Y), ZZ = fe_sq(Z);
    fe ZZ2 = fe_add(ZZ, ZZ);
    fe S = fe_sq(fe_add(X, Y));
    gc r; r.H = fe_add(YY, XX); r.G = fe_sub(YY, XX); r.E = fe_sub(S, r.H); r.F = fe_sub(ZZ2, r.G);
    return r;
}
AFX_HD gc gc_add_pn_inl(const gc& c, const pniels& n) {
    fe X = fe_mul(c.E, c.F), Y = fe_mul(c.G, c.H);
    fe PP = fe_mul(fe_add(Y, X), n.YpX);
    fe MM = fe_mul(fe_sub(Y, X), n.YmX);
    fe TT = fe_mul(fe_mul(c.E, c.H), n.T2d);
    fe ZZ = fe_mul(fe_mul(c.F, c.G), n.Z);
    fe ZZ2 = fe_add(ZZ, ZZ);
    gc r; r.E = fe_sub(PP, MM); r.H = fe_add(PP, MM); r.G = fe_add(ZZ2, TT); r.F = fe_sub(ZZ2, TT);
    return r;
}
AFX_HD gc gc_madd_inl(const gc& c, const aniels& n) {
    fe X = fe_mul(c.E, c.F), Y = fe_mul(c.G, c.H);
    fe PP = fe_mul(fe_add(Y, X), n.ypx);
    fe MM = fe_mul(fe_sub(Y, X), n.ymx);
    fe TT = fe_mul(fe_mul(c.E, c.H), n.xy2d);
    fe Z = fe_mul(c.F, c.G);
    fe ZZ2 = fe_add(Z, Z);
    gc r; r.E = fe_sub(PP, MM); r.H = fe_add(PP, MM); r.G = fe_add(ZZ2, TT); r.F = fe_sub(ZZ2, TT);
    return r;
}
// Ladder-loop forms.  On the device the window body is inlined into the (rolled) ladder loop, so the accumulator never
// crosses a call boundary (no argument/return register shuffles: 23.7 -> 23.0 ms for k_ladders on B200).
AFX_HD void gc_dbl4(gc& acc) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1   // rolled: unrolling by 2 / 4 costs 1 % / 6 % (instruction fetch), profiles/README.md
#endif
    for (int j = 0; j < 4; j++) acc = gc_dbl_inl(acc);
}
#define GE_LADDER_ADD(acc, e) acc = gc_add_pn_inl(acc, e)
#define GE_LADDER_MADD(acc, e) acc = gc_madd_inl(acc, e)
AFX_HD ge ge_add(const ge& p, const ge& q) { return ge_add_pn(p, ge_to_pniels(q)); }
AFX_HD ge ge_sub(const ge& p, const ge& q) { return ge_add_pn(p, pniels_cneg(ge_to_pniels(q), 1)); }

// CompressedRistretto::decompress (SURVEY A.2).  w = the 32 encoding bytes as 8 little-endian words.
// Returns 1 and the point, or 0 (and the identity) for a non-canonical / negative / off-group encoding.
struct enc32 { u32 w[8]; };
struct ge_ok { ge p; u32 ok; };
AFX_NI ge_ok ge_decompress_v(enc32 e) {
    const u32* w = e.w;
    ge p;
    fe s = fe_from_bytes_words(w);
    fe sc = fe_canonical(s);
    u32 canonical = 1;
    for (int i = 0; i < 8; i++) canonical &= (sc.v[i] == w[i]);   // also rejects bit 255 set
    u32 ok = canonical & ((w[0] & 1u) ^ 1u);
    fe one = fe_one();
    fe ss = fe_sq(s);
    fe u1 = fe_sub(one, ss), u2 = fe_add(one, ss);
    fe u2s = fe_sq(u2);
    fe v = fe_sub(fe_neg(fe_mul(FE_D(), fe_sq(u1))), u2s);
    fe I;
    ok &= fe_invsqrt(I, fe_mul(v, u2s));
    fe Dx = fe_mul(I, u2);
    fe Dy = fe_mul(fe_mul(I, Dx), v);
    fe x = fe_abs(fe_mul(fe_add(s, s), Dx));
    fe y = fe_mul(u1, Dy);
    fe t = fe_mul(x, y);
    ok &= (fe_is_negative(t) ^ 1u) & (fe_is_zero(y) ^ 1u);
    ge id = ge_identity();
    p.X = fe_select(id.X, x, ok); p.Y = fe_select(id.Y, y, ok); p.Z = one; p.T = fe_select(id.T, t, ok);
    ge_ok o; o.p = p; o.ok = ok;
    return o;
}
AFX_HD u32 ge_decompress(ge& p, const u32* w) {
    enc32 e; for (int i = 0; i < 8; i++) e.w[i] = w[i];
    ge_ok o = ge_decompress_v(e); p = o.p; return o.ok;
}

// RistrettoPoint::compress (SURVEY A.2) -> 8 little-endian words.
AFX_NI enc32 ge_compress_v(ge p) {
    fe u1 = fe_mul(fe_add(p.Z, p.Y), fe_sub(p.Z, p.Y));
    fe u2 = fe_mul(p.X, p.Y);
    fe inv;
    fe_invsqrt(inv, fe_mul(u1, fe_sq(u2)));
    fe i1 = fe_mul(inv, u1), i2 = fe_mul(inv, u2);
    fe z_inv = fe_mul(i1, fe_mul(i2, p.T));
    u32 rotate = fe_is_negative(fe_mul(p.T, z_inv));
    fe X = fe_select(p.X, fe_mul(p.Y, FE_SQRT_M1()), rotate);
    fe Y = fe_select(p.Y, fe_mul(p.X, FE_SQRT_M1()), rotate);
    fe den_inv = fe_select(i2, fe_mul(i1, FE_INVSQRT_A_MINUS_D()), rotate);
    Y = fe_cneg(Y, fe_is_negative(fe_mul(X, z_inv)));
    fe s = fe_abs(fe_mul(den_inv, fe_sub(p.Z, Y)));
    enc32 e; fe_to_bytes_words(e.w, s);
    return e;
}
AFX_HD void ge_compress(u32* out, const ge& p) { enc32 e = ge_compress_v(p); for (int i = 0; i < 8; i++) out[i] = e.w[i]; }

// Encoding of a DOUBLED point, in batches (curve25519-dalek RistrettoPoint::double_and_compress_batch).  For 2Q the square
// root the encoding needs is a rational function of Q's coordinates, so a batch of doubled points shares one field inversion
// (Montgomery's trick) where compress() pays an inverse square root per point.  Per point: dac_begin, then dac_den into the
// batch's running product, then dac_finish with inv = 1 / dac_den.  eg * fh = 0 exactly when 2Q is 4-torsion, whose
// encoding is the identity's (32 zero bytes): such a factor is replaced by 1 so that it does not zero the whole product.
struct dac_state { fe e, f, g, h, eg, fh; };
AFX_NI dac_state dac_begin(ge q) {       // 4S + 4M
    fe XX = fe_sq(q.X), YY = fe_sq(q.Y), ZZ = fe_sq(q.Z), dTT = fe_mul(FE_D(), fe_sq(q.T));
    dac_state s;
    s.e = fe_mul(fe_add(q.X, q.X), q.Y); s.f = fe_add(ZZ, dTT); s.g = fe_add(YY, XX); s.h = fe_sub(ZZ, dTT);
    s.eg = fe_mul(s.e, s.g); s.fh = fe_mul(s.f, s.h);
    return s;
}
// eg * fh, or 1 when it is zero (zero = 1 then)
AFX_HD fe dac_den(const dac_state& s, u32& zero) {
    fe x = fe_mul(s.eg, s.fh);
    zero = fe_is_zero(x);
    return fe_select(x, fe_one(), zero);
}
// 8 encoding words of 2Q from inv = 1 / dac_den: 8M, all selects, no branch
AFX_NI enc32 dac_finish(dac_state s, fe inv, u32 zero) {
    fe z_inv = fe_mul(s.eg, inv), t_inv = fe_mul(s.fh, inv);
    u32 rotate = fe_is_negative(fe_mul(s.eg, z_inv));
    fe e = fe_select(s.e, s.g, rotate);
    fe g = fe_select(s.g, fe_neg(s.e), rotate);
    fe h = fe_select(s.h, fe_mul(s.f, FE_SQRT_M1()), rotate);
    fe magic = fe_select(FE_INVSQRT_A_MINUS_D(), FE_SQRT_M1(), rotate);
    g = fe_cneg(g, fe_is_negative(fe_mul(fe_mul(h, e), z_inv)));
    fe s_ = fe_abs(fe_mul(fe_sub(h, g), fe_mul(magic, fe_mul(g, t_inv))));
    s_ = fe_select(s_, fe_zero(), zero);
    enc32 out; fe_to_bytes_words(out.w, s_);
    return out;
}

// Elligator map (RFC 9496 4.3.4 MAP; dalek elligator_ristretto_flavor), SURVEY A.2
AFX_NI ge ge_elligator(fe r0) {
    fe one = fe_one();
    fe r = fe_mul(FE_SQRT_M1(), fe_sq(r0));
    fe Ns = fe_mul(fe_add(r, one), FE_ONE_MINUS_D_SQ());
    fe c = fe_neg(one);
    fe Dn = fe_mul(fe_sub(c, fe_mul(FE_D(), r)), fe_add(r, FE_D()));
    fe s;
    u32 sq = fe_sqrt_ratio_i(s, Ns, Dn);
    fe s_prime = fe_neg(fe_abs(fe_mul(s, r0)));
    s = fe_select(s_prime, s, sq);
    c = fe_select(r, c, sq);
    fe Nt = fe_sub(fe_mul(fe_mul(c, fe_sub(r, one)), FE_D_MINUS_ONE_SQ()), Dn);
    fe s2 = fe_sq(s);
    fe W0 = fe_mul(fe_add(s, s), Dn), W1 = fe_mul(Nt, FE_SQRT_AD_MINUS_ONE()), W2 = fe_sub(one, s2), W3 = fe_add(one, s2);
    ge p; p.X = fe_mul(W0, W3); p.Y = fe_mul(W2, W1); p.Z = fe_mul(W1, W3); p.T = fe_mul(W0, W2);
    return p;
}
// RistrettoPoint::from_uniform_bytes: 64 bytes = 16 words
AFX_HD ge ge_from_uniform(const u32* w) {
    return ge_add(ge_elligator(fe_from_bytes_words(w)), ge_elligator(fe_from_bytes_words(w + 8)));
}

// [1P .. 8P] in projective Niels form: the per-point table every fixed-window ladder here uses (3 dbl + 4 add).
// Entries are handed to `emit(index, entry)` as they are produced so that at most three points are live at a time.
template <typename Emit>
AFX_HD void ge_table8(const ge& p, Emit emit) {
    pniels n1 = ge_to_pniels(p); emit(0, n1);
    ge p2 = ge_dbl(p); emit(1, ge_to_pniels(p2));
    ge p3 = ge_add_pn(p2, n1); emit(2, ge_to_pniels(p3));
    ge p4 = ge_dbl(p2); emit(3, ge_to_pniels(p4));
    emit(4, ge_to_pniels(ge_add_pn(p4, n1)));
    ge p6 = ge_dbl(p3); emit(5, ge_to_pniels(p6));
    emit(6, ge_to_pniels(ge_add_pn(p6, n1)));
    emit(7, ge_to_pniels(ge_dbl(p4)));
}

}  // namespace afx
