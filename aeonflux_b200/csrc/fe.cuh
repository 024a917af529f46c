// GF(2^255-19) for sm_100a: 8 x 32-bit saturated limbs, lazily reduced mod 2^256-38.
//
// Replaces curve25519-dalek's FieldElement under every point operation of aeonflux's hot path
// (call sites: /root/reference/src/nizk/presentation.rs:342-351,373-412; encryption.rs:172-185;
// issuance.rs:162-189).  Not a port of dalek's 5x51 / 10x25.5 limb code: the layout is chosen for the
// B200 integer pipe -- one 32x32->64 product is one IMAD.WIDE.U32 and carries ride the .X/.CC chain, so a
// multiply is 64 + 8 wide products ("M = 72 limb-products", SURVEY 8d) and a square 36 + 8.
//
// Invariant: every fe holds an integer in [0, 2^256) congruent to the field element; canonical
// reduction happens only in fe_tobytes / comparisons.  2^256 = 38 (mod p).
//
// Every function is __host__ __device__: the host bodies are plain C used only by the test-only
// emulation harness (tests/hostemu); the device bodies are PTX carry chains.  Both compute exactly the
// same limbs.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define AFX_HD __host__ __device__ __forceinline__
#define AFX_D __device__ __forceinline__
// Point-level operations are real subroutines on the device (ptxas keeps their by-value struct arguments in registers):
// this keeps each kernel's code to tens of KB instead of megabytes of inlined multiplies.
#define AFX_NI __host__ __device__ __noinline__
// Keeps the warps of a CTA within one ladder step of each other so that they share instruction-cache lines.
#define AFX_STEP_SYNC() __syncthreads()
#else
#define AFX_STEP_SYNC() do { } while (0)
#define AFX_HD inline
#define AFX_NI inline
#ifndef AFX_STEP_SYNC
#define AFX_STEP_SYNC() do { } while (0)
#endif
#endif

namespace afx {

typedef uint32_t u32;
typedef uint64_t u64;
typedef uint16_t u16;

struct fe { u32 v[8]; };

AFX_HD fe fe_zero() { fe r; for (int i = 0; i < 8; i++) r.v[i] = 0; return r; }
AFX_HD fe fe_one() { fe r = fe_zero(); r.v[0] = 1; return r; }
AFX_HD fe fe_from_words(u32 a0, u32 a1, u32 a2, u32 a3, u32 a4, u32 a5, u32 a6, u32 a7) {
    fe r; r.v[0] = a0; r.v[1] = a1; r.v[2] = a2; r.v[3] = a3; r.v[4] = a4; r.v[5] = a5; r.v[6] = a6; r.v[7] = a7; return r;
}

// ---- constants (little-endian 32-bit words), SURVEY A.1 ---------------------------------------
#define AFX_FE_CONST(name, a0, a1, a2, a3, a4, a5, a6, a7) \
    AFX_HD fe name() { return fe_from_words(a0##u, a1##u, a2##u, a3##u, a4##u, a5##u, a6##u, a7##u); }
AFX_FE_CONST(FE_D, 0x135978a3, 0x75eb4dca, 0x4141d8ab, 0x00700a4d, 0x7779e898, 0x8cc74079, 0x2b6ffe73, 0x52036cee)
AFX_FE_CONST(FE_D2, 0x26b2f159, 0xebd69b94, 0x8283b156, 0x00e0149a, 0xeef3d130, 0x198e80f2, 0x56dffce7, 0x2406d9dc)
AFX_FE_CONST(FE_SQRT_M1, 0x4a0ea0b0, 0xc4ee1b27, 0xad2fe478, 0x2f431806, 0x3dfbd7a7, 0x2b4d0099, 0x4fc1df0b, 0x2b832480)
AFX_FE_CONST(FE_INVSQRT_A_MINUS_D, 0x805d40ea, 0x99c8fdaa, 0x5a4172be, 0x9d2f1617, 0xfe01d840, 0x16c27b91, 0xcfaffca2, 0x786c8905)
AFX_FE_CONST(FE_SQRT_AD_MINUS_ONE, 0x497b2e1b, 0x7e97f6a0, 0x1b7854bd, 0xaf9d8e0c, 0x31f5d1fd, 0x0f3cfcc9, 0x2b8348ac, 0x376931bf)
AFX_FE_CONST(FE_ONE_MINUS_D_SQ, 0x945fc176, 0xe27c09c1, 0xcd5e350f, 0x2c81a138, 0xbe70dfe4, 0x9994abdd, 0xb2b3e0d7, 0x029072a8)
AFX_FE_CONST(FE_D_MINUS_ONE_SQ, 0x44ed4d20, 0x31ad5aaa, 0xb01e1999, 0xd29e4a2c, 0x529b4eeb, 0x4cdcd32f, 0xf66c2241, 0x5968b37a)

// ---- add / sub / neg ---------------------------------------------------------------------------
AFX_HD fe fe_add(const fe& a, const fe& b) {
    fe r;
#if defined(__CUDA_ARCH__)
    u32 c;
    asm("add.cc.u32 %0, %9, %17;\n\t addc.cc.u32 %1, %10, %18;\n\t addc.cc.u32 %2, %11, %19;\n\t addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t addc.cc.u32 %5, %14, %22;\n\t addc.cc.u32 %6, %15, %23;\n\t addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7]), "=&r"(c)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
    u32 k = c * 38u;
    asm("add.cc.u32 %0, %0, %9;\n\t addc.cc.u32 %1, %1, 0;\n\t addc.cc.u32 %2, %2, 0;\n\t addc.cc.u32 %3, %3, 0;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t addc.cc.u32 %5, %5, 0;\n\t addc.cc.u32 %6, %6, 0;\n\t addc.cc.u32 %7, %7, 0;\n\t"
        "addc.u32 %8, 0, 0;"
        : "+&r"(r.v[0]), "+&r"(r.v[1]), "+&r"(r.v[2]), "+&r"(r.v[3]), "+&r"(r.v[4]), "+&r"(r.v[5]), "+&r"(r.v[6]), "+&r"(r.v[7]), "=&r"(c)
        : "r"(k));
    r.v[0] += c * 38u;  // a second wrap leaves a tiny value: no further carry possible
#else
    u64 c = 0;
    for (int i = 0; i < 8; i++) { c += (u64)a.v[i] + b.v[i]; r.v[i] = (u32)c; c >>= 32; }
    u64 k = c * 38; c = k;
    for (int i = 0; i < 8; i++) { c += r.v[i]; r.v[i] = (u32)c; c >>= 32; }
    r.v[0] += (u32)c * 38u;
#endif
    return r;
}

AFX_HD fe fe_sub(const fe& a, const fe& b) {
    fe r;
#if defined(__CUDA_ARCH__)
    u32 bw;
    asm("sub.cc.u32 %0, %9, %17;\n\t subc.cc.u32 %1, %10, %18;\n\t subc.cc.u32 %2, %11, %19;\n\t subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t subc.cc.u32 %5, %14, %22;\n\t subc.cc.u32 %6, %15, %23;\n\t subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7]), "=&r"(bw)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
    u32 k = bw & 38u;  // bw is 0 or 0xffffffff
    asm("sub.cc.u32 %0, %0, %9;\n\t subc.cc.u32 %1, %1, 0;\n\t subc.cc.u32 %2, %2, 0;\n\t subc.cc.u32 %3, %3, 0;\n\t"
        "subc.cc.u32 %4, %4, 0;\n\t subc.cc.u32 %5, %5, 0;\n\t subc.cc.u32 %6, %6, 0;\n\t subc.cc.u32 %7, %7, 0;\n\t"
        "subc.u32 %8, 0, 0;"
        : "+&r"(r.v[0]), "+&r"(r.v[1]), "+&r"(r.v[2]), "+&r"(r.v[3]), "+&r"(r.v[4]), "+&r"(r.v[5]), "+&r"(r.v[6]), "+&r"(r.v[7]), "=&r"(bw)
        : "r"(k));
    r.v[0] -= bw & 38u;  // a second wrap leaves a value close to 2^256: no further borrow possible
#else
    int64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (int64_t)a.v[i] - b.v[i]; r.v[i] = (u32)c; c >>= 32; }
    int64_t k = c ? 38 : 0; c = -k;
    for (int i = 0; i < 8; i++) { c += r.v[i]; r.v[i] = (u32)c; c >>= 32; }
    if (c) r.v[0] -= 38u;
#endif
    return r;
}

AFX_HD fe fe_neg(const fe& a) { return fe_sub(fe_zero(), a); }

// ---- multiply ----------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
// acc[S .. S+7] += (a[J0], a[J0+2], a[J0+4], a[J0+6]) * b, products pair-aligned at S, S+2, ...; carry into acc[S+8].
template <int S, int J0>
AFX_D void fe_row_chain(u32* acc, const u32* a, u32 b) {
    if (S + 8 < 16) {
        asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
            "madc.lo.cc.u32 %2, %10, %13, %2;\n\t madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
            "madc.lo.cc.u32 %4, %11, %13, %4;\n\t madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
            "madc.lo.cc.u32 %6, %12, %13, %6;\n\t madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
            "addc.u32 %8, %8, 0;"
            : "+&r"(acc[S]), "+&r"(acc[S + 1]), "+&r"(acc[S + 2]), "+&r"(acc[S + 3]), "+&r"(acc[S + 4]), "+&r"(acc[S + 5]), "+&r"(acc[S + 6]),
              "+&r"(acc[S + 7]), "+&r"(acc[(S + 8) & 15])
            : "r"(a[J0]), "r"(a[J0 + 2]), "r"(a[J0 + 4]), "r"(a[J0 + 6]), "r"(b));
    } else {
        asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
            "madc.lo.cc.u32 %2, %9, %12, %2;\n\t madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
            "madc.lo.cc.u32 %4, %10, %12, %4;\n\t madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
            "madc.lo.cc.u32 %6, %11, %12, %6;\n\t madc.hi.u32 %7, %11, %12, %7;"
            : "+&r"(acc[S]), "+&r"(acc[S + 1]), "+&r"(acc[S + 2]), "+&r"(acc[S + 3]), "+&r"(acc[S + 4]), "+&r"(acc[S + 5]), "+&r"(acc[S + 6]),
              "+&r"(acc[S + 7])
            : "r"(a[J0]), "r"(a[J0 + 2]), "r"(a[J0 + 4]), "r"(a[J0 + 6]), "r"(b));
    }
}
template <int I>
AFX_D void fe_row(u32* E, u32* O, const u32* a, u32 b) {
    if (I % 2 == 0) { fe_row_chain<I, 0>(E, a, b); fe_row_chain<I + 1, 1>(O, a, b); }
    else            { fe_row_chain<I, 0>(O, a, b); fe_row_chain<I + 1, 1>(E, a, b); }
}
// r = t[0..7] + 38 * t[8..15], folded into [0, 2^256)
AFX_D fe fe_fold512(const u32* t) {
    u32 A[9];
#pragma unroll
    for (int i = 0; i < 8; i++) A[i] = t[i];
    A[8] = 0;
    const u32 c38 = 38u;
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+&r"(A[0]), "+&r"(A[1]), "+&r"(A[2]), "+&r"(A[3]), "+&r"(A[4]), "+&r"(A[5]), "+&r"(A[6]), "+&r"(A[7]), "+&r"(A[8])
        : "r"(t[8]), "r"(t[10]), "r"(t[12]), "r"(t[14]), "r"(c38));
    asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %12, %2;\n\t madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
        "madc.lo.cc.u32 %4, %10, %12, %4;\n\t madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
        "madc.lo.cc.u32 %6, %11, %12, %6;\n\t madc.hi.u32 %7, %11, %12, %7;"
        : "+&r"(A[1]), "+&r"(A[2]), "+&r"(A[3]), "+&r"(A[4]), "+&r"(A[5]), "+&r"(A[6]), "+&r"(A[7]), "+&r"(A[8])
        : "r"(t[9]), "r"(t[11]), "r"(t[13]), "r"(t[15]), "r"(c38));
    // A[8] <= 38: fold it, then the (rare) final carry
    u32 top = A[8] * 38u, cy;
    fe r;
    asm("add.cc.u32 %0, %9, %17;\n\t addc.cc.u32 %1, %10, 0;\n\t addc.cc.u32 %2, %11, 0;\n\t addc.cc.u32 %3, %12, 0;\n\t"
        "addc.cc.u32 %4, %13, 0;\n\t addc.cc.u32 %5, %14, 0;\n\t addc.cc.u32 %6, %15, 0;\n\t addc.cc.u32 %7, %16, 0;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7]), "=&r"(cy)
        : "r"(A[0]), "r"(A[1]), "r"(A[2]), "r"(A[3]), "r"(A[4]), "r"(A[5]), "r"(A[6]), "r"(A[7]), "r"(top));
    r.v[0] += cy * 38u;
    return r;
}
#else
inline fe fe_fold512(const u32* t) {
    u64 A[9];
    for (int i = 0; i < 8; i++) A[i] = t[i];
    A[8] = 0;
    u64 c = 0;
    for (int i = 0; i < 8; i++) { c += A[i] + (u64)t[8 + i] * 38u; A[i] = (u32)c; c >>= 32; }
    A[8] = c;
    u64 top = A[8] * 38u;
    fe r; c = top;
    for (int i = 0; i < 8; i++) { c += A[i]; r.v[i] = (u32)c; c >>= 32; }
    r.v[0] += (u32)c * 38u;
    return r;
}
#endif

AFX_HD fe fe_mul(const fe& x, const fe& y) {
#if defined(__CUDA_ARCH__)
    u32 E[16], O[16];
#pragma unroll
    for (int i = 0; i < 16; i++) { E[i] = 0; O[i] = 0; }
    fe_row<0>(E, O, x.v, y.v[0]); fe_row<1>(E, O, x.v, y.v[1]); fe_row<2>(E, O, x.v, y.v[2]); fe_row<3>(E, O, x.v, y.v[3]);
    fe_row<4>(E, O, x.v, y.v[4]); fe_row<5>(E, O, x.v, y.v[5]); fe_row<6>(E, O, x.v, y.v[6]); fe_row<7>(E, O, x.v, y.v[7]);
    u32 t[16];
    asm("add.cc.u32 %0, %16, %32;\n\t addc.cc.u32 %1, %17, %33;\n\t addc.cc.u32 %2, %18, %34;\n\t addc.cc.u32 %3, %19, %35;\n\t"
        "addc.cc.u32 %4, %20, %36;\n\t addc.cc.u32 %5, %21, %37;\n\t addc.cc.u32 %6, %22, %38;\n\t addc.cc.u32 %7, %23, %39;\n\t"
        "addc.cc.u32 %8, %24, %40;\n\t addc.cc.u32 %9, %25, %41;\n\t addc.cc.u32 %10, %26, %42;\n\t addc.cc.u32 %11, %27, %43;\n\t"
        "addc.cc.u32 %12, %28, %44;\n\t addc.cc.u32 %13, %29, %45;\n\t addc.cc.u32 %14, %30, %46;\n\t addc.u32 %15, %31, %47;"
        : "=&r"(t[0]), "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(t[8]), "=&r"(t[9]), "=&r"(t[10]),
          "=&r"(t[11]), "=&r"(t[12]), "=&r"(t[13]), "=&r"(t[14]), "=&r"(t[15])
        : "r"(E[0]), "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]), "r"(E[10]), "r"(E[11]),
          "r"(E[12]), "r"(E[13]), "r"(E[14]), "r"(E[15]), "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]),
          "r"(O[8]), "r"(O[9]), "r"(O[10]), "r"(O[11]), "r"(O[12]), "r"(O[13]), "r"(O[14]), "r"(O[15]));
    return fe_fold512(t);
#else
    u32 t[16];
    u64 acc[16];
    for (int i = 0; i < 16; i++) acc[i] = 0;
    for (int i = 0; i < 8; i++) {
        u64 c = 0;
        for (int j = 0; j < 8; j++) { c += acc[i + j] + (u64)x.v[j] * y.v[i]; acc[i + j] = (u32)c; c >>= 32; }
        acc[i + 8] = c;
    }
    for (int i = 0; i < 16; i++) t[i] = (u32)acc[i];
    return fe_fold512(t);
#endif
}

AFX_HD fe fe_sq(const fe& x) {
#if defined(__CUDA_ARCH__)
    // cross products a_i*a_j (i<j) into pair-aligned accumulators E (i+j even) and O (i+j odd)
    const u32* a = x.v;
    u32 E[16], O[16];
#pragma unroll
    for (int i = 0; i < 16; i++) { E[i] = 0; O[i] = 0; }
    // row 0: O <- a0*(a1,a3,a5,a7) at 1,3,5,7 ; E <- a0*(a2,a4,a6) at 2,4,6
    asm("mul.lo.u32 %0, %9, %13;\n\t mul.hi.u32 %1, %9, %13;\n\t mul.lo.u32 %2, %10, %13;\n\t mul.hi.u32 %3, %10, %13;\n\t"
        "mul.lo.u32 %4, %11, %13;\n\t mul.hi.u32 %5, %11, %13;\n\t mul.lo.u32 %6, %12, %13;\n\t mul.hi.u32 %7, %12, %13;\n\t mov.u32 %8, 0;"
        : "=&r"(O[1]), "=&r"(O[2]), "=&r"(O[3]), "=&r"(O[4]), "=&r"(O[5]), "=&r"(O[6]), "=&r"(O[7]), "=&r"(O[8]), "=&r"(O[9])
        : "r"(a[1]), "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(a[0]));
    asm("mul.lo.u32 %0, %6, %9;\n\t mul.hi.u32 %1, %6, %9;\n\t mul.lo.u32 %2, %7, %9;\n\t mul.hi.u32 %3, %7, %9;\n\t"
        "mul.lo.u32 %4, %8, %9;\n\t mul.hi.u32 %5, %8, %9;"
        : "=&r"(E[2]), "=&r"(E[3]), "=&r"(E[4]), "=&r"(E[5]), "=&r"(E[6]), "=&r"(E[7])
        : "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(a[0]));
    // row 1: O <- a1*(a2,a4,a6) at 3,5,7 ; E <- a1*(a3,a5,a7) at 4,6,8
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t madc.hi.cc.u32 %1, %7, %10, %1;\n\t madc.lo.cc.u32 %2, %8, %10, %2;\n\t madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t madc.hi.cc.u32 %5, %9, %10, %5;\n\t addc.u32 %6, %6, 0;"
        : "+&r"(O[3]), "+&r"(O[4]), "+&r"(O[5]), "+&r"(O[6]), "+&r"(O[7]), "+&r"(O[8]), "+&r"(O[9])
        : "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(a[1]));
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t madc.hi.cc.u32 %1, %7, %10, %1;\n\t madc.lo.cc.u32 %2, %8, %10, %2;\n\t madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t madc.hi.cc.u32 %5, %9, %10, %5;\n\t addc.u32 %6, %6, 0;"
        : "+&r"(E[4]), "+&r"(E[5]), "+&r"(E[6]), "+&r"(E[7]), "+&r"(E[8]), "+&r"(E[9]), "+&r"(E[10])
        : "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(a[1]));
    // row 2: O <- a2*(a3,a5,a7) at 5,7,9 ; E <- a2*(a4,a6) at 6,8
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t madc.hi.cc.u32 %1, %7, %10, %1;\n\t madc.lo.cc.u32 %2, %8, %10, %2;\n\t madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t madc.hi.cc.u32 %5, %9, %10, %5;\n\t addc.u32 %6, %6, 0;"
        : "+&r"(O[5]), "+&r"(O[6]), "+&r"(O[7]), "+&r"(O[8]), "+&r"(O[9]), "+&r"(O[10]), "+&r"(O[11])
        : "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(a[2]));
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+&r"(E[6]), "+&r"(E[7]), "+&r"(E[8]), "+&r"(E[9]), "+&r"(E[10])
        : "r"(a[4]), "r"(a[6]), "r"(a[2]));
    // row 3: O <- a3*(a4,a6) at 7,9 ; E <- a3*(a5,a7) at 8,10
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+&r"(O[7]), "+&r"(O[8]), "+&r"(O[9]), "+&r"(O[10]), "+&r"(O[11])
        : "r"(a[4]), "r"(a[6]), "r"(a[3]));
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+&r"(E[8]), "+&r"(E[9]), "+&r"(E[10]), "+&r"(E[11]), "+&r"(E[12])
        : "r"(a[5]), "r"(a[7]), "r"(a[3]));
    // row 4: O <- a4*(a5,a7) at 9,11 ; E <- a4*a6 at 10
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t madc.hi.cc.u32 %1, %5, %7, %1;\n\t madc.lo.cc.u32 %2, %6, %7, %2;\n\t madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+&r"(O[9]), "+&r"(O[10]), "+&r"(O[11]), "+&r"(O[12]), "+&r"(O[13])
        : "r"(a[5]), "r"(a[7]), "r"(a[4]));
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t madc.hi.cc.u32 %1, %3, %4, %1;\n\t addc.u32 %2, %2, 0;"
        : "+&r"(E[10]), "+&r"(E[11]), "+&r"(E[12]) : "r"(a[6]), "r"(a[4]));
    // row 5: O <- a5*a6 at 11 ; E <- a5*a7 at 12
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t madc.hi.cc.u32 %1, %3, %4, %1;\n\t addc.u32 %2, %2, 0;"
        : "+&r"(O[11]), "+&r"(O[12]), "+&r"(O[13]) : "r"(a[6]), "r"(a[5]));
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t madc.hi.cc.u32 %1, %3, %4, %1;\n\t addc.u32 %2, %2, 0;"
        : "+&r"(E[12]), "+&r"(E[13]), "+&r"(E[14]) : "r"(a[7]), "r"(a[5]));
    // row 6: O <- a6*a7 at 13
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t madc.hi.cc.u32 %1, %3, %4, %1;\n\t addc.u32 %2, %2, 0;"
        : "+&r"(O[13]), "+&r"(O[14]), "+&r"(O[15]) : "r"(a[7]), "r"(a[6]));
    // t = 2*(E + O)  (word 0 of the cross sum is zero)
    u32 t[16];
    asm("add.cc.u32 %0, %15, %30;\n\t addc.cc.u32 %1, %16, %31;\n\t addc.cc.u32 %2, %17, %32;\n\t addc.cc.u32 %3, %18, %33;\n\t"
        "addc.cc.u32 %4, %19, %34;\n\t addc.cc.u32 %5, %20, %35;\n\t addc.cc.u32 %6, %21, %36;\n\t addc.cc.u32 %7, %22, %37;\n\t"
        "addc.cc.u32 %8, %23, %38;\n\t addc.cc.u32 %9, %24, %39;\n\t addc.cc.u32 %10, %25, %40;\n\t addc.cc.u32 %11, %26, %41;\n\t"
        "addc.cc.u32 %12, %27, %42;\n\t addc.cc.u32 %13, %28, %43;\n\t addc.u32 %14, %29, %44;"
        : "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(t[8]), "=&r"(t[9]), "=&r"(t[10]), "=&r"(t[11]),
          "=&r"(t[12]), "=&r"(t[13]), "=&r"(t[14]), "=&r"(t[15])
        : "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]), "r"(E[10]), "r"(E[11]), "r"(E[12]),
          "r"(E[13]), "r"(E[14]), "r"(E[15]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]), "r"(O[9]),
          "r"(O[10]), "r"(O[11]), "r"(O[12]), "r"(O[13]), "r"(O[14]), "r"(O[15]));
    t[0] = 0;
    asm("add.cc.u32 %0, %0, %0;\n\t addc.cc.u32 %1, %1, %1;\n\t addc.cc.u32 %2, %2, %2;\n\t addc.cc.u32 %3, %3, %3;\n\t"
        "addc.cc.u32 %4, %4, %4;\n\t addc.cc.u32 %5, %5, %5;\n\t addc.cc.u32 %6, %6, %6;\n\t addc.cc.u32 %7, %7, %7;\n\t"
        "addc.cc.u32 %8, %8, %8;\n\t addc.cc.u32 %9, %9, %9;\n\t addc.cc.u32 %10, %10, %10;\n\t addc.cc.u32 %11, %11, %11;\n\t"
        "addc.cc.u32 %12, %12, %12;\n\t addc.cc.u32 %13, %13, %13;\n\t addc.u32 %14, %14, %14;"
        : "+&r"(t[1]), "+&r"(t[2]), "+&r"(t[3]), "+&r"(t[4]), "+&r"(t[5]), "+&r"(t[6]), "+&r"(t[7]), "+&r"(t[8]), "+&r"(t[9]), "+&r"(t[10]), "+&r"(t[11]),
          "+&r"(t[12]), "+&r"(t[13]), "+&r"(t[14]), "+&r"(t[15]));
    // + squares a_i^2 at words (2i, 2i+1)
    asm("mad.lo.cc.u32 %0, %16, %16, %0;\n\t madc.hi.cc.u32 %1, %16, %16, %1;\n\t madc.lo.cc.u32 %2, %17, %17, %2;\n\t madc.hi.cc.u32 %3, %17, %17, %3;\n\t"
        "madc.lo.cc.u32 %4, %18, %18, %4;\n\t madc.hi.cc.u32 %5, %18, %18, %5;\n\t madc.lo.cc.u32 %6, %19, %19, %6;\n\t madc.hi.cc.u32 %7, %19, %19, %7;\n\t"
        "madc.lo.cc.u32 %8, %20, %20, %8;\n\t madc.hi.cc.u32 %9, %20, %20, %9;\n\t madc.lo.cc.u32 %10, %21, %21, %10;\n\t madc.hi.cc.u32 %11, %21, %21, %11;\n\t"
        "madc.lo.cc.u32 %12, %22, %22, %12;\n\t madc.hi.cc.u32 %13, %22, %22, %13;\n\t madc.lo.cc.u32 %14, %23, %23, %14;\n\t madc.hi.u32 %15, %23, %23, %15;"
        : "+&r"(t[0]), "+&r"(t[1]), "+&r"(t[2]), "+&r"(t[3]), "+&r"(t[4]), "+&r"(t[5]), "+&r"(t[6]), "+&r"(t[7]), "+&r"(t[8]), "+&r"(t[9]), "+&r"(t[10]),
          "+&r"(t[11]), "+&r"(t[12]), "+&r"(t[13]), "+&r"(t[14]), "+&r"(t[15])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
    return fe_fold512(t);
#else
    return fe_mul(x, x);
#endif
}

AFX_NI fe fe_sqn(fe x, int n) {
    for (int i = 0; i < n; i++) x = fe_sq(x);
    return x;
}

// ---- canonical form ------------------------------------------------------------------------------
// Reduce to the unique representative in [0, p).
AFX_HD fe fe_canonical(const fe& a) {
    // v' = (v mod 2^255) + 19 * (v >> 255)  <  2^255 + 19
    u32 hi = a.v[7] >> 31;
    fe r = a;
    r.v[7] &= 0x7fffffffu;
    u64 c = (u64)hi * 19u;
    for (int i = 0; i < 8; i++) { c += r.v[i]; r.v[i] = (u32)c; c >>= 32; }
    // subtract p if r >= p  (r + 19 >= 2^255)
    u32 t[8];
    c = 19;
    for (int i = 0; i < 8; i++) { c += r.v[i]; t[i] = (u32)c; c >>= 32; }
    u32 ge = t[7] >> 31;  // r + 19 carried into bit 255  <=>  r >= p
    t[7] &= 0x7fffffffu;
    u32 m = 0u - ge;
    for (int i = 0; i < 8; i++) r.v[i] = (t[i] & m) | (r.v[i] & ~m);
    return r;
}
AFX_HD u32 fe_is_negative(const fe& a) { return fe_canonical(a).v[0] & 1u; }
AFX_HD u32 fe_is_zero(const fe& a) {
    fe c = fe_canonical(a); u32 x = 0;
    for (int i = 0; i < 8; i++) x |= c.v[i];
    return x == 0;
}
AFX_HD u32 fe_equal(const fe& a, const fe& b) { return fe_is_zero(fe_sub(a, b)); }
AFX_HD fe fe_select(const fe& a, const fe& b, u32 take_b) {  // branch-free
    u32 m = 0u - (take_b & 1u); fe r;
    for (int i = 0; i < 8; i++) r.v[i] = (b.v[i] & m) | (a.v[i] & ~m);
    return r;
}
AFX_HD fe fe_cneg(const fe& a, u32 neg) { return fe_select(a, fe_neg(a), neg); }
AFX_HD fe fe_abs(const fe& a) { return fe_cneg(a, fe_is_negative(a)); }

// bytes <-> fe.  from_bytes ignores bit 255 (dalek FieldElement::from_bytes, SURVEY A.1).
AFX_HD fe fe_from_bytes_words(const u32* w) { fe r; for (int i = 0; i < 8; i++) r.v[i] = w[i]; r.v[7] &= 0x7fffffffu; return r; }
AFX_HD void fe_to_bytes_words(u32* w, const fe& a) { fe c = fe_canonical(a); for (int i = 0; i < 8; i++) w[i] = c.v[i]; }

// ---- addition chains -------------------------------------------------------------------------------
// The common head of the two chains below: x^(2^250 - 1) and x^11.  249 squarings + 10 multiplies.
struct fe_pow250 { fe a250, x11; };
AFX_HD fe_pow250 fe_pow22501(const fe& x) {
    fe x2 = fe_sq(x);                       // 2
    fe x9 = fe_mul(fe_sqn(x2, 2), x);       // 9
    fe x11 = fe_mul(x9, x2);                // 11
    fe x31 = fe_mul(fe_sq(x11), x9);        // 2^5 - 1
    fe a10 = fe_mul(fe_sqn(x31, 5), x31);   // 2^10 - 1
    fe a20 = fe_mul(fe_sqn(a10, 10), a10);  // 2^20 - 1
    fe a40 = fe_mul(fe_sqn(a20, 20), a20);  // 2^40 - 1
    fe a50 = fe_mul(fe_sqn(a40, 10), a10);  // 2^50 - 1
    fe a100 = fe_mul(fe_sqn(a50, 50), a50); // 2^100 - 1
    fe a200 = fe_mul(fe_sqn(a100, 100), a100); // 2^200 - 1
    fe_pow250 r; r.a250 = fe_mul(fe_sqn(a200, 50), a50); r.x11 = x11;   // 2^250 - 1
    return r;
}
// x^(2^252 - 3) = x^((p-5)/8): 251 squarings + 11 multiplies, fully in registers.
AFX_NI fe fe_pow_p58(fe x) { return fe_mul(fe_sqn(fe_pow22501(x).a250, 2), x); }
// x^(p-2) = x^(2^255 - 21) = 1/x (0 for x = 0): 254 squarings + 11 multiplies.
AFX_NI fe fe_invert(fe x) { fe_pow250 t = fe_pow22501(x); return fe_mul(fe_sqn(t.a250, 5), t.x11); }

// sqrt_ratio_i(u, v) (SURVEY A.1): returns was_square, r = the non-negative root of u/v or of i*u/v.
struct fe_ok { fe r; u32 ok; };
AFX_NI fe_ok fe_sqrt_ratio_i_v(fe u, fe v) {
    fe r;
    fe v3 = fe_mul(fe_sq(v), v);
    fe v7 = fe_mul(fe_sq(v3), v);
    r = fe_mul(fe_mul(u, v3), fe_pow_p58(fe_mul(u, v7)));
    fe check = fe_mul(v, fe_sq(r));
    fe mu = fe_neg(u);
    u32 correct = fe_equal(check, u);
    u32 flipped = fe_equal(check, mu);
    u32 flipped_i = fe_equal(check, fe_mul(mu, FE_SQRT_M1()));
    r = fe_select(r, fe_mul(r, FE_SQRT_M1()), flipped | flipped_i);
    fe_ok o; o.r = fe_abs(r); o.ok = correct | flipped;
    return o;
}
AFX_HD u32 fe_sqrt_ratio_i(fe& r, const fe& u, const fe& v) { fe_ok o = fe_sqrt_ratio_i_v(u, v); r = o.r; return o.ok; }
// invsqrt(v) = sqrt_ratio_i(1, v), specialised (saves 3 multiplies)
AFX_NI fe_ok fe_invsqrt_v(fe v) {
    fe r;
    fe v3 = fe_mul(fe_sq(v), v);
    fe v7 = fe_mul(fe_sq(v3), v);
    r = fe_mul(v3, fe_pow_p58(v7));
    fe check = fe_mul(v, fe_sq(r));
    fe one = fe_one();
    fe mone = fe_neg(one);
    u32 correct = fe_equal(check, one);
    u32 flipped = fe_equal(check, mone);
    u32 flipped_i = fe_equal(check, fe_neg(FE_SQRT_M1()));
    r = fe_select(r, fe_mul(r, FE_SQRT_M1()), flipped | flipped_i);
    fe_ok o; o.r = fe_abs(r); o.ok = correct | flipped;
    return o;
}
AFX_HD u32 fe_invsqrt(fe& r, const fe& v) { fe_ok o = fe_invsqrt_v(v); r = o.r; return o.ok; }

}  // namespace afx
