// agx_tables.h -- host-side parameter validation and per-limb scalars for libagxntt.
//
// The "step before the path" of the reference: main.cpp:46-55 fills the twiddle / precon / modulus buffers on the
// host and ntt_input_kernel broadcasts them (ntt.cpp:544-571).  Here the library derives them from (n, q): the host
// finds psi = the minimal primitive 2n-th root (SURVEY.md App. A) and the scalar inverses; the n-entry tables
// (roots[k] = psi^bitrev(k) in the order ntt.cpp:298-300 consumes, Shoup companions floor(w * 2^32 / q), inverse
// tables, n^-1 folding) are computed on the device by gen_tables_kernel (agx_ntt_kernels.cuh).
// Independent of oracle/ (the tests cross-check the two).
#pragma once
#include <cstdint>
#include <vector>

namespace agx {

uint64_t mulmod_u64(uint64_t a, uint64_t b, uint64_t q);
uint64_t powmod_u64(uint64_t a, uint64_t e, uint64_t q);
bool is_prime_u64(uint64_t q);
uint32_t bit_reverse(uint32_t x, uint32_t bits);

// 0 when q is not a usable NTT prime for n (not prime, >= 2^30, q != 1 mod 2n)
uint32_t minimal_psi(uint32_t n, uint32_t q);
// the same for the u64 path: 0 unless q is prime, 3 <= q < 2^62 and q = 1 (mod 2n)
uint64_t minimal_psi_u64(uint32_t n, uint64_t q);

}  // namespace agx
