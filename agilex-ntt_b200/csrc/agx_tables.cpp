// agx_tables.cpp -- see agx_tables.h
#include "agx_tables.h"

namespace agx {

uint64_t mulmod_u64(uint64_t a, uint64_t b, uint64_t q) {
    return (uint64_t)(((unsigned __int128)a * b) % q);
}

uint64_t powmod_u64(uint64_t a, uint64_t e, uint64_t q) {
    uint64_t r = 1 % q;
    a %= q;
    for (; e; e >>= 1) {
        if (e & 1) r = mulmod_u64(r, a, q);
        a = mulmod_u64(a, a, q);
    }
    return r;
}

bool is_prime_u64(uint64_t q) {
    if (q < 2) return false;
    for (uint64_t p : {2ull, 3ull, 5ull, 7ull, 11ull, 13ull, 17ull, 19ull, 23ull, 29ull, 31ull, 37ull}) {
        if (q == p) return true;
        if (q % p == 0) return false;
    }
    uint64_t d = q - 1;
    int s = 0;
    while (!(d & 1)) { d >>= 1; s++; }
    for (uint64_t a : {2ull, 3ull, 5ull, 7ull, 11ull, 13ull, 17ull, 19ull, 23ull, 29ull, 31ull, 37ull}) {
        uint64_t x = powmod_u64(a, d, q);
        if (x == 1 || x == q - 1) continue;
        bool composite = true;
        for (int r = 1; r < s && composite; r++) {
            x = mulmod_u64(x, x, q);
            if (x == q - 1) composite = false;
        }
        if (composite) return false;
    }
    return true;
}

uint32_t bit_reverse(uint32_t x, uint32_t bits) {
    uint32_t r = 0;
    for (uint32_t i = 0; i < bits; i++, x >>= 1) r = (r << 1) | (x & 1);
    return r;
}

uint32_t minimal_psi(uint32_t n, uint32_t q) {
    return q >= (1u << 30) ? 0u : (uint32_t)minimal_psi_u64(n, q);
}

uint64_t minimal_psi_u64(uint32_t n, uint64_t q) {
    if (n < 2 || (n & (n - 1)) || q < 3 || q >= (1ull << 62) || (q - 1) % (2ull * n) || !is_prime_u64(q)) return 0;
    const uint64_t e = (q - 1) / (2ull * n);
    uint64_t g = 0;
    for (uint64_t x = 2; x < q && !g; x++) {
        const uint64_t c = powmod_u64(x, e, q);
        if (powmod_u64(c, n, q) == q - 1) g = c;   // order exactly 2n (n is a power of two)
    }
    if (!g) return 0;
    // the primitive 2n-th roots are the odd powers of g; keep the smallest
    const uint64_t g2 = mulmod_u64(g, g, q);
    uint64_t cur = g, best = g;
    for (uint32_t k = 0; k < n; k++) {
        if (cur < best) best = cur;
        cur = mulmod_u64(cur, g2, q);
    }
    return best;
}

}  // namespace agx
