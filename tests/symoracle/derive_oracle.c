/* TEST-ONLY: the C oracle's Keypair::derive (symmetric.rs:197-215) over a batch on all host cores, for the full-size check of
 * tests/test_keypairs.py and the CPU rate of tools/bench_symmetric.py.  It compiles the oracle (oracle/c/afx_oracle.c) unchanged and
 * adds a batch driver around its keypair_derive. */
#include "../../oracle/c/afx_oracle.c"

typedef struct { const afxo_issuer* is; const uint8_t* ms; uint8_t* out; uint64_t lo, hi; } derive_job;

static void* derive_worker(void* arg) {
    derive_job* j = (derive_job*)arg;
    for (uint64_t i = j->lo; i < j->hi; i++) {      /* master secrets [count][64] -> keypairs [count][128] = a || a0 || a1 || pk */
        sym_keypair k; uint8_t* o = j->out + 128 * i;
        keypair_derive(&k, j->is, j->ms + 64 * i);
        memcpy(o, k.a, 32); memcpy(o + 32, k.a0, 32); memcpy(o + 64, k.a1, 32); ge_compress(o + 96, &k.pk);
        memset(&k, 0, sizeof k);
    }
    return NULL;
}

/* keypairs [count][128] from master secrets [count][64] under the system parameters sp (the issuer's public key ipub only completes
 * the oracle's issuer).  Returns the wall-clock seconds of the batch, or -1 if sp / ipub do not parse. */
API double afxd_derive(const uint8_t* sp, size_t sp_len, const uint8_t* ipub, const uint8_t* ms, uint64_t count, int threads, uint8_t* keypairs) {
    afxo_issuer* is = afxo_issuer_new(sp, sp_len, ipub, NULL, 0);
    if (!is) return -1;
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    derive_job js[256]; pthread_t th[256];
    double t0 = now_s();
    for (int t = 0; t < threads; t++) {
        derive_job j = {is, ms, keypairs, count * (uint64_t)t / (uint64_t)threads, count * (uint64_t)(t + 1) / (uint64_t)threads};
        js[t] = j;
    }
    for (int t = 1; t < threads; t++) pthread_create(&th[t], NULL, derive_worker, &js[t]);
    derive_worker(&js[0]);
    for (int t = 1; t < threads; t++) pthread_join(th[t], NULL);
    double secs = now_s() - t0;
    afxo_issuer_free(is);
    return secs;
}
