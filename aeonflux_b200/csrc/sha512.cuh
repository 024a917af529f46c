// SHA-512 (FIPS 180-4) of messages that fit one padded block: the 30 data bytes of an attribute, which Plaintext::from
// (symmetric.rs:135-143) and Keypair::decrypt (symmetric.rs:273-289) hash, and the 64-byte master secret and 32-byte scalars that
// Keypair::derive (symmetric.rs:197-215) hashes.
#pragma once
#include "ge.cuh"

namespace afx {

AFX_HD u64 rotr64(u64 x, int n) { return (x >> n) | (x << (64 - n)); }
AFX_HD u32 bswap32(u32 x) { return (x >> 24) | ((x >> 8) & 0xff00u) | ((x << 8) & 0xff0000u) | (x << 24); }

struct digest64 { u32 w[16]; };     // the 64 digest bytes as little-endian words (the form sc_reduce512 and ge_from_uniform take)
// The compression function over the one padded block W (16 big-endian words: message, 0x80, zeros, 128-bit bit length), from the
// initial hash value.  The message builders below are its only callers.
AFX_HD digest64 sha512_block(u64 W[16]) {
    const u64 K[80] = {
        0x428a2f98d728ae22ull, 0x7137449123ef65cdull, 0xb5c0fbcfec4d3b2full, 0xe9b5dba58189dbbcull, 0x3956c25bf348b538ull,
        0x59f111f1b605d019ull, 0x923f82a4af194f9bull, 0xab1c5ed5da6d8118ull, 0xd807aa98a3030242ull, 0x12835b0145706fbeull,
        0x243185be4ee4b28cull, 0x550c7dc3d5ffb4e2ull, 0x72be5d74f27b896full, 0x80deb1fe3b1696b1ull, 0x9bdc06a725c71235ull,
        0xc19bf174cf692694ull, 0xe49b69c19ef14ad2ull, 0xefbe4786384f25e3ull, 0x0fc19dc68b8cd5b5ull, 0x240ca1cc77ac9c65ull,
        0x2de92c6f592b0275ull, 0x4a7484aa6ea6e483ull, 0x5cb0a9dcbd41fbd4ull, 0x76f988da831153b5ull, 0x983e5152ee66dfabull,
        0xa831c66d2db43210ull, 0xb00327c898fb213full, 0xbf597fc7beef0ee4ull, 0xc6e00bf33da88fc2ull, 0xd5a79147930aa725ull,
        0x06ca6351e003826full, 0x142929670a0e6e70ull, 0x27b70a8546d22ffcull, 0x2e1b21385c26c926ull, 0x4d2c6dfc5ac42aedull,
        0x53380d139d95b3dfull, 0x650a73548baf63deull, 0x766a0abb3c77b2a8ull, 0x81c2c92e47edaee6ull, 0x92722c851482353bull,
        0xa2bfe8a14cf10364ull, 0xa81a664bbc423001ull, 0xc24b8b70d0f89791ull, 0xc76c51a30654be30ull, 0xd192e819d6ef5218ull,
        0xd69906245565a910ull, 0xf40e35855771202aull, 0x106aa07032bbd1b8ull, 0x19a4c116b8d2d0c8ull, 0x1e376c085141ab53ull,
        0x2748774cdf8eeb99ull, 0x34b0bcb5e19b48a8ull, 0x391c0cb3c5c95a63ull, 0x4ed8aa4ae3418acbull, 0x5b9cca4f7763e373ull,
        0x682e6ff3d6b2b8a3ull, 0x748f82ee5defb2fcull, 0x78a5636f43172f60ull, 0x84c87814a1f0ab72ull, 0x8cc702081a6439ecull,
        0x90befffa23631e28ull, 0xa4506cebde82bde9ull, 0xbef9a3f7b2c67915ull, 0xc67178f2e372532bull, 0xca273eceea26619cull,
        0xd186b8c721c0c207ull, 0xeada7dd6cde0eb1eull, 0xf57d4f7fee6ed178ull, 0x06f067aa72176fbaull, 0x0a637dc5a2c898a6ull,
        0x113f9804bef90daeull, 0x1b710b35131c471bull, 0x28db77f523047d84ull, 0x32caab7b40c72493ull, 0x3c9ebe0a15c9bebcull,
        0x431d67c49c100d4cull, 0x4cc5d4becb3e42b6ull, 0x597f299cfc657e2aull, 0x5fcb6fab3ad6faecull, 0x6c44198c4a475817ull};
    u64 H[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    u64 a = H[0], b = H[1], c = H[2], d = H[3], e = H[4], f = H[5], g = H[6], h = H[7];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int t = 0; t < 80; t++) {
        u64 w;
        if (t < 16) w = W[t];
        else {   // message schedule in a 16-word ring
            const u64 w15 = W[(t - 15) & 15], w2 = W[(t - 2) & 15];
            const u64 s0 = rotr64(w15, 1) ^ rotr64(w15, 8) ^ (w15 >> 7), s1 = rotr64(w2, 19) ^ rotr64(w2, 61) ^ (w2 >> 6);
            w = W[t & 15] + s0 + W[(t - 7) & 15] + s1;
            W[t & 15] = w;
        }
        const u64 S1 = rotr64(e, 14) ^ rotr64(e, 18) ^ rotr64(e, 41), ch = (e & f) ^ (~e & g);
        const u64 t1 = h + S1 + ch + K[t] + w;
        const u64 S0 = rotr64(a, 28) ^ rotr64(a, 34) ^ rotr64(a, 39), maj = (a & b) ^ (a & c) ^ (b & c);
        h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + S0 + maj;
    }
    H[0] += a; H[1] += b; H[2] += c; H[3] += d; H[4] += e; H[5] += f; H[6] += g; H[7] += h;
    digest64 out;
    for (int i = 0; i < 8; i++) {     // big-endian digest bytes -> little-endian words
        out.w[2 * i] = bswap32((u32)(H[i] >> 32));
        out.w[2 * i + 1] = bswap32((u32)H[i]);
    }
    return out;
}

// The message is bytes 1..30 of the 32-byte string msg: where the data sits in its candidate group encodings 2i || data || j
// (encoding.rs:56-70) and in the compressed M1 a decryption recovers (encoding.rs:75-82).  Passing the words keeps the message
// in registers.
AFX_NI digest64 sha512_30(enc32 msg) {
    const u32 len = 30;
    u64 W[16];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int t = 0; t < 16; t++) {
        u64 w = 0;
        for (int b = 0; b < 8; b++) {
            const u32 i = 8u * (u32)t + (u32)b;
            const u64 byte = i < len ? (msg.w[(i + 1) >> 2] >> (8 * ((i + 1) & 3))) & 0xffu : i == len ? 0x80u : 0u;
            w = (w << 8) | byte;
        }
        W[t] = w;
    }
    W[15] |= (u64)len * 8u;
    return sha512_block(W);
}

struct msg64 { u32 w[16]; };        // up to 64 message bytes as little-endian words
// The message is the first 4 * nw bytes of m, nw = 16 (a master secret) or 8 (a scalar's 32 bytes).  nw is public: it selects where
// the padding starts, never a message byte.  Passing the words keeps the message in registers.
AFX_NI digest64 sha512_words(msg64 m, u32 nw) {
    u64 W[16];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int t = 0; t < 16; t++) {
        const u32 k = 2u * (u32)t;
        const u64 word = ((u64)bswap32(m.w[k & 15]) << 32) | bswap32(m.w[(k + 1) & 15]);
        W[t] = k < nw ? word : k == nw ? 0x8000000000000000ull : 0u;
    }
    W[15] |= (u64)nw * 32u;
    return sha512_block(W);
}

}  // namespace afx
