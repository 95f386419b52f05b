/*
 * u64_inverse_oracle.c -- CPU oracle of the u64 inverse transform and negacyclic product (agx_ref_inv_dev,
 * agx_ref_polymul_dev).  TEST INFRASTRUCTURE ONLY: built into a temporary directory by tests/test_u64_inverse.py and
 * profiles/bench_u64_inv.py, never linked into the product.  No reference counterpart (the reference has only the
 * forward); pinned by tests/test_u64_inverse.py against the big-int definitions of oracle/oracle.py.
 */
#include <stddef.h>
#include <stdint.h>

typedef unsigned __int128 u128;

static uint64_t mulmod(uint64_t a, uint64_t b, uint64_t q) { return (uint64_t)(((u128)a * b) % q); }

/* Gentleman-Sande inverse of one frame, in place: bit-reversed in (any 64-bit words, reduced first), natural out in
 * [0,q); stage with h groups reads iroots[h + i] (iroots[k] = psi^-bitrev(k), ntt.cpp:298-300 order); then * n^-1. */
static void inv_one(uint32_t N, uint64_t *x, uint64_t q, const uint64_t *iroots) {
    for (uint32_t j = 0; j < N; j++) x[j] %= q;
    uint32_t t = 1;
    for (uint32_t h = N >> 1; h >= 1; h >>= 1, t <<= 1)
        for (uint32_t i = 0; i < h; i++) {
            const uint64_t w = iroots[h + i];
            uint64_t *p = x + (size_t)2 * i * t;
            for (uint32_t j = 0; j < t; j++) {
                const uint64_t u = p[j], v = p[j + t];
                p[j] = (uint64_t)(((u128)u + v) % q);
                p[j + t] = mulmod((uint64_t)(((u128)u + q - v) % q), w, q);
            }
        }
    uint64_t ninv = 1;                                      /* n^-1 = ((q+1)/2)^log2 n */
    for (uint32_t m = 1; m < N; m <<= 1) ninv = mulmod(ninv, (q + 1) / 2, q);
    for (uint32_t j = 0; j < N; j++) x[j] = mulmod(x[j], ninv, q);
}

void orc_inv_u64(uint32_t N, uint64_t *data, uint64_t q, const uint64_t *iroots, size_t numFrames, int threads) {
    (void)threads;
#pragma omp parallel for schedule(static) num_threads(threads > 0 ? threads : 1)
    for (long long b = 0; b < (long long)numFrames; b++) inv_one(N, data + (size_t)b * N, q, iroots);
}

/* c = a * b mod (X^N + 1, q), exact: c[k] = sum_{i+j=k} a_i b_j - sum_{i+j=k+N} a_i b_j, every term reduced */
void orc_polymul_schoolbook_u64(uint32_t N, uint64_t q, const uint64_t *a, const uint64_t *b, uint64_t *c) {
    for (uint32_t k = 0; k < N; k++) {
        uint64_t pos = 0, neg = 0;
        for (uint32_t i = 0; i <= k; i++) pos = (uint64_t)(((u128)pos + mulmod(a[i] % q, b[k - i] % q, q)) % q);
        for (uint32_t i = k + 1; i < N; i++) neg = (uint64_t)(((u128)neg + mulmod(a[i] % q, b[N + k - i] % q, q)) % q);
        c[k] = (uint64_t)(((u128)pos + q - neg) % q);
    }
}
