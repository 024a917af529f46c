/* TEST-ONLY: the C oracle's Plaintext::from, Keypair::encrypt and Keypair::decrypt (symmetric.rs:135-143,252-261,273-289) over a
 * batch on all host cores, for the large-batch checks of tests/test_symmetric.py and the CPU rate of tools/bench_symmetric.py.
 * It compiles the oracle (oracle/c/afx_oracle.c) unchanged and adds batch drivers around its primitives. */
#include "../../oracle/c/afx_oracle.c"

typedef struct { int op; const uint8_t* kp; const uint8_t* in; uint8_t* out; uint8_t* out2; uint8_t* status; uint64_t lo, hi; } sym_job;

static int sym_decrypt1(const uint8_t* kp, const uint8_t* c, uint8_t data[30], uint8_t pt[96]) {
    ge E1, E2, t, M1, M2; uint8_t enc[32], h[64], m3[32], u[32], chk[32];
    if (!ge_decompress(&E1, c) || !ge_decompress(&E2, c + 32)) return 0;
    ge_scalarmult_ct(&t, &E1, kp); ge_sub(&M1, &E2, &t);
    ge_compress(enc, &M1); memcpy(data, enc + 1, 30);
    sha512(h, data, 30); ge_from_uniform(&M2, h); sc_from_wide(m3, h);
    sc_muladd(u, kp + 64, m3, kp + 32);
    ge_scalarmult_ct(&t, &M2, u); ge_compress(chk, &t);
    if (memcmp(chk, c, 32) != 0) return 0;
    memcpy(pt, enc, 32); ge_compress(pt + 32, &M2); memcpy(pt + 64, m3, 32);
    return 1;
}

static void* sym_worker(void* arg) {
    sym_job* j = (sym_job*)arg;
    for (uint64_t i = j->lo; i < j->hi; i++) {
        int ok = 1;
        if (j->op == 0) {               /* data [count][30] -> plaintexts [count][3][32] */
            plaintext p; uint8_t* o = j->out + 96 * i;
            plaintext_from30(&p, j->in + 30 * i);
            ge_compress(o, &p.M1); ge_compress(o + 32, &p.M2); memcpy(o + 64, p.m3, 32);
        } else if (j->op == 1) {        /* plaintexts [count][3][32] -> ciphertexts [count][2][32] */
            const uint8_t* w = j->in + 96 * i; uint8_t* o = j->out + 64 * i; ge M1, M2, E1, E2; uint8_t u[32], au[32];
            ok = ge_decompress(&M1, w) && ge_decompress(&M2, w + 32) && sc_is_canonical(w + 64);
            if (ok) {
                sc_muladd(u, j->kp + 64, w + 64, j->kp + 32); sc_mul(au, j->kp, u);
                ge_scalarmult_ct(&E1, &M2, u); ge_scalarmult_ct(&E2, &M2, au); ge_add(&E2, &E2, &M1);
                ge_compress(o, &E1); ge_compress(o + 32, &E2);
            } else memset(o, 0, 64);
        } else {                        /* ciphertexts [count][2][32] -> data [count][30], plaintexts [count][3][32] (nullable) */
            uint8_t pt[96] = {0}, d[30] = {0};
            ok = sym_decrypt1(j->kp, j->in + 64 * i, d, pt);
            if (!ok) { memset(d, 0, 30); memset(pt, 0, 96); }
            memcpy(j->out + 30 * i, d, 30);
            if (j->out2) memcpy(j->out2 + 96 * i, pt, 96);
        }
        j->status[i] = (uint8_t)!ok;
    }
    return NULL;
}

/* op 0 encode, 1 encrypt, 2 decrypt; kp = a || a0 || a1 (ops 1, 2).  Returns the wall-clock seconds of the batch. */
API double afxs_run(int op, const uint8_t* kp, const uint8_t* in, uint64_t count, int threads, uint8_t* out, uint8_t* out2, uint8_t* status) {
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    sym_job js[256]; pthread_t th[256];
    double t0 = now_s();
    for (int t = 0; t < threads; t++) {
        sym_job j = {op, kp, in, out, out2, status, count * (uint64_t)t / (uint64_t)threads, count * (uint64_t)(t + 1) / (uint64_t)threads};
        js[t] = j;
    }
    for (int t = 1; t < threads; t++) pthread_create(&th[t], NULL, sym_worker, &js[t]);
    sym_worker(&js[0]);
    for (int t = 1; t < threads; t++) pthread_join(th[t], NULL);
    return now_s() - t0;
}
