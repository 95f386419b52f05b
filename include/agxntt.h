/*
 * agxntt.h -- C ABI of the B200-native Agilex-NTT hot path (libagxntt.so).
 *
 * Drop-in boundary for joekurina/Agilex-NTT's kernel API (reference = /root/reference):
 *
 *   reference interface                                        replaced by
 *   ---------------------------------------------------------  -------------------------------------------
 *   ntt_input_kernel(in, in2, modulus, twiddles, precons,      agx_ref_input()      include/kernel/ntt.h:35-41,
 *                    numFrames, q)                                                   src/kernel/ntt.cpp:508-607
 *   fwd_ntt_kernel<id>(q)                                      agx_ref_fwd()        include/kernel/ntt.h:32-33,
 *                                                                                    src/kernel/ntt.cpp:86-506
 *   ntt_output_kernel(out, numFrames, q)                       agx_ref_output()     include/kernel/ntt.h:43-45,
 *                                                                                    src/kernel/ntt.cpp:610-640
 *   sycl::queue::wait()   (src/main.cpp:74)                    agx_wait()
 *   compile-time FPGA_NTT_SIZE / modulus buffer                agx_parms + agx_create()   (the reference has no
 *   (ntt.h:7-23, main.cpp:34)                                  parameter struct; SURVEY.md s.8(b))
 *   caller-filled twiddle / precon buffers                     agx_create_tables() (caller's psi), agx_set_tables()
 *   (ntt.h:38-39, main.cpp:36-37,46-55, ntt.cpp:122-141)       (caller's tables in the reference's order)
 *
 * and the batched u32 entry points BASELINE.json's north_star adds (no reference counterpart):
 *   agx_ntt_fwd / agx_ntt_inv / agx_polymul on device pointers, *_host variants on host pointers.
 *
 * Conventions
 *   - Plain C: pointers and sizes only.  Every function returns 0 (AGX_OK), a negative AGX_E_* code, or a
 *     positive cudaError_t value.  Nothing throws or aborts across this boundary.  There is NO CPU fallback:
 *     without a CUDA device agx_create() fails with the cudaError_t.
 *   - Transform definition (matches ntt.cpp, SURVEY.md App. A): forward is negacyclic Cooley-Tukey, natural
 *     order in, BIT-REVERSED order out, outputs fully reduced to [0,q); inverse is Gentleman-Sande,
 *     bit-reversed in, natural out, n^-1 folded in.  psi = the minimal primitive 2n-th root of unity mod q unless the
 *     caller supplies its own root (agx_create_tables) or its own tables (agx_set_tables).
 *   - Batched layout: uint32_t data[B][L][n] (B polynomials x L RNS limbs), row-major, in place.
 *     Inputs must be < 2q for the u32 entry points (uniform-mod-q data is < q).  Device pointers must be 16-byte
 *     aligned (anything from cudaMalloc is).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device-pointer calls only
 *     enqueue; completion follows normal stream semantics.  *_host calls return after the results are in
 *     host memory.
 *   - A context is bound to one device and is not thread-safe; use one context per host thread / GPU.  Every call
 *     makes the context's device current for its own duration and restores the caller's current device on return.
 */
#ifndef AGXNTT_H
#define AGXNTT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGX_OK 0
#define AGX_E_INVALID (-1)     /* bad argument (null pointer, n not a supported power of two, bad prime ...) */
#define AGX_E_UNSUPPORTED (-2) /* valid request this build cannot serve */
#define AGX_E_NOMEM (-3)       /* host allocation failed */
#define AGX_E_STATE (-4)       /* reference-shaped calls used out of protocol */

typedef struct agx_ctx agx_ctx;

/* Run-time replacement for the reference's compile-time configuration (FPGA_NTT_SIZE ntt.h:7-23, one modulus
 * buffer main.cpp:34).  n = 2^logn in [8, 32768]; every q[i] prime, < 2^30, q = 1 (mod 2n).  The tuned
 * register-resident kernels cover n in {1024, 2048, 4096}; other sizes run a generic shared-memory kernel. */
typedef struct {
    uint32_t n;
    uint32_t logn;
    uint32_t nlimbs;
    const uint32_t *q; /* [nlimbs] */
} agx_parms;

/* parms == NULL creates a table-less context usable only with the agx_ref_* calls. */
int agx_create(agx_ctx **out, const agx_parms *parms, int device);
int agx_destroy(agx_ctx *ctx);

/* The reference's contract is "the caller hands in the roots" (include/kernel/ntt.h:38-39; main.cpp:36-37,46-55 fill
 * the buffers, ntt.cpp:122-141 receives them).  Two ways to do that on the u32 entry points:
 *
 * agx_create_tables: like agx_create, with the caller's primitive 2n-th root per limb, psi[nlimbs] (NULL = the
 *   minimal root, i.e. agx_create).  AGX_E_INVALID unless psi[i]^n = -1 (mod q[i]).  The library derives the forward
 *   and inverse tables from it on the device.
 *
 * agx_set_tables: replaces one limb's forward (inverse == 0) or inverse (inverse != 0) table by the caller's, given in
 *   the reference's order (ntt.cpp:298-300: entry m + i is the twiddle of group i in the stage with m groups, i.e.
 *   roots[k] = psi^bitrev(k) resp. psi^-bitrev(k); entry 0 is unused) as HOST arrays of n words.  precons[k] =
 *   floor(roots[k] * 2^32 / q) -- the 32-bit counterpart of the reference's barrettTwiddleFactors buffer -- or NULL to
 *   have them computed.  The table is checked on the device (roots[1]^2 = -1, roots[2k]^2 = roots[k], roots[2k+1] =
 *   roots[2k] * roots[1], entries < q, precons exact) and re-laid-out for the kernels (the inverse one with n^-1
 *   folded in); AGX_E_INVALID, with the previous table still in place, when it is not consistent.  A caller that
 *   replaces the forward table replaces the inverse one too (the library does not derive one from the other). */
int agx_create_tables(agx_ctx **out, const agx_parms *parms, const uint32_t *psi, int device);
int agx_set_tables(agx_ctx *ctx, uint32_t limb, int inverse, const uint32_t *roots, const uint32_t *precons);

/* Introspection (parity tests compare these with the oracle's tables). roots/precons in the reference's table
 * order, ntt.cpp:298-300: entry k = psi^bitrev(k) and floor(entry * 2^32 / q); inverse != 0 -> psi^-1. */
int agx_get_psi(const agx_ctx *ctx, uint32_t limb, uint32_t *psi);
int agx_get_tables(const agx_ctx *ctx, uint32_t limb, int inverse, uint32_t *roots, uint32_t *precons);

/* ---- batched u32 transforms on DEVICE pointers, in place, asynchronous on `stream` ---- */
int agx_ntt_fwd(agx_ctx *ctx, uint32_t *d_data, size_t B, void *stream);
int agx_ntt_inv(agx_ctx *ctx, uint32_t *d_data, size_t B, void *stream);
/* c = a * b mod (X^n + 1, q_limb) = INTT(NTT(a) .* NTT(b)).  c may alias a and/or b, and a may equal b (squaring), at
 * every size.  n = 1024: forward(a), forward(b), pointwise product and inverse run in ONE launch (3 streams of HBM
 * traffic); n = 2048 and 4096: three launches (c = NTT(a); c = NTT(b) .* c; c = INTT(c) -- 7 streams, no scratch
 * memory; the product is bound by the integer-multiply pipe, not by that traffic: DESIGN.md s.4); other sizes: the
 * transforms of that size (n >= 8192: shared-memory-resident register passes; n <= 512: the generic kernel) around a
 * pointwise launch, with a stream-ordered scratch buffer unless a == b. */
int agx_polymul(agx_ctx *ctx, uint32_t *d_c, const uint32_t *d_a, const uint32_t *d_b, size_t B, void *stream);
/* The product with one operand already in evaluation form -- the shape of an RLWE encryption or key switch, where the
 * key is transformed once and multiplied many times (SURVEY.md s.8(f) rank 4; no reference counterpart):
 * c = INTT(NTT(a) .* b_hat), b_hat = agx_ntt_fwd(b) (reduced, bit-reversed order as the forward transform leaves it).
 * Two launches at n = 1024, 2048, 4096 (c = NTT(a) .* b_hat inside the forward kernel; c = INTT(c): 5 streams of HBM
 * traffic, two transforms' worth of multiplies instead of agx_polymul's three); the generic transforms around a
 * pointwise launch at other sizes.  c may alias a and/or b_hat (aliasing b_hat at the generic sizes costs a scratch
 * copy).  Equals agx_polymul(c, a, b) bit for bit. */
int agx_polymul_by_spectrum(agx_ctx *ctx, uint32_t *d_c, const uint32_t *d_a, const uint32_t *d_b_hat, size_t B,
                            void *stream);

/* ---- limb-wise element-wise arithmetic on [B][L][n] DEVICE data (the operations callers run around the transforms,
 * e.g. spectrum multiply-accumulate between agx_ntt_fwd and agx_ntt_inv; SURVEY.md s.8(f) rank 4; no reference
 * counterpart).  Operands must be reduced (< q_limb); results are in [0, q_limb).  d_c may alias d_a and/or d_b. ---- */
#define AGX_EW_ADD 0 /* c = a + b     */
#define AGX_EW_SUB 1 /* c = a - b     */
#define AGX_EW_MUL 2 /* c = a * b     */
#define AGX_EW_MAC 3 /* c = c + a * b */
int agx_elementwise(agx_ctx *ctx, int op, uint32_t *d_c, const uint32_t *d_a, const uint32_t *d_b, size_t B,
                    void *stream);

/* ---- coefficient-order adapter: permutes every n-coefficient row of [B][L][n] DEVICE data by bit reversal, in place
 * (an involution).  The transforms keep the reference's orders (ntt.cpp:292-300: natural in, bit-reversed out; the
 * inverse takes bit-reversed input); callers holding natural-order spectra convert with this call.  No reference
 * counterpart. ---- */
int agx_bitrev(agx_ctx *ctx, uint32_t *d_data, size_t B, void *stream);

/* ---- the same on HOST pointers: chunked H2D / kernel / D2H pipeline over the context's own streams.
 * Pinned memory (agx_host_alloc, cudaHostAlloc, cudaHostRegister) is copied directly; pageable memory is staged
 * through internal pinned buffers.  h_out may equal h_in. ---- */
int agx_ntt_fwd_host(agx_ctx *ctx, const uint32_t *h_in, uint32_t *h_out, size_t B);
int agx_ntt_inv_host(agx_ctx *ctx, const uint32_t *h_in, uint32_t *h_out, size_t B);
int agx_polymul_host(agx_ctx *ctx, uint32_t *h_c, const uint32_t *h_a, const uint32_t *h_b, size_t B);
int agx_polymul_by_spectrum_host(agx_ctx *ctx, uint32_t *h_c, const uint32_t *h_a, const uint32_t *h_b_hat, size_t B);
int agx_host_alloc(void **p, size_t bytes);
int agx_host_free(void *p);

/* ---- synthetic inputs and checksums on the device (SURVEY.md s.8(d)) ----
 * element g of [B][L][n], counted from polynomial `first_poly`, = splitmix64(seed + g) mod q_limb.
 * checksum = sum_i splitmix64((first_index + i) * 0xD6E8FEB86659FD93 + data[i]) mod 2^64 (shard sums add up). */
int agx_fill_synthetic(agx_ctx *ctx, uint32_t *d_data, size_t B, uint64_t seed, size_t first_poly, void *stream);
int agx_checksum(agx_ctx *ctx, const uint32_t *d_data, size_t count, size_t first_index, uint64_t *h_sum,
                 void *stream);

/* ---- reference-shaped u64 forward pipeline (host pointers; mirrors main.cpp:60-74) ----
 * N in {2^2 .. 2^15} (the reference builds 32, 1024, 8192, 16384, 32768: ntt.h:11-20).  Arithmetic is the
 * reference's u64 Harvey butterfly including wrap-around mod 2^64 for tables that are not Shoup pairs -- and for
 * moduli of 62 bits and more, whose lazy range [0,4q) no longer fits 64 bits (the reference wraps identically; parity
 * is pinned on 50-, 60-, 62- and 63-bit primes against the reference's own code).
 * The three calls only record/enqueue, in any order (the reference's three kernels run concurrently); the work
 * runs once all three were made; agx_wait() blocks until `out` is filled (= q.wait()).  `in`, `in2` hold
 * numFrames*N words (frame b: low half from in[b*N..], high half from in2[b*N + N/2..], ntt.cpp:582-591);
 * twiddles/precon_twiddles hold N words, modulus 1 word.  Host buffers must stay valid until agx_wait(). */
int agx_ref_input(agx_ctx *ctx, uint32_t N, const uint64_t *in, const uint64_t *in2, const uint64_t *modulus,
                  const uint64_t *twiddles, const uint64_t *precon_twiddles, uint32_t numFrames);
int agx_ref_fwd(agx_ctx *ctx, uint32_t compute_unit_id);
int agx_ref_output(agx_ctx *ctx, uint64_t *out, int32_t numFrames);
int agx_wait(agx_ctx *ctx);

/* The same transform on DEVICE pointers, asynchronous on `stream` (what the three calls above run per chunk; exposes
 * the kernels' rate without PCIe): frame b reads d_in[b*N .. b*N + N/2) and d_in2[b*N + N/2 .. (b+1)*N)
 * (ntt.cpp:582-591) and writes d_out[b*N .. (b+1)*N) (ntt.cpp:626-633).  d_twiddles / d_precon_twiddles: N words each
 * on the device.  All five device pointers must be 16-byte aligned (AGX_E_INVALID otherwise; cudaMalloc'd buffers are).
 * d_out may be the same buffer as d_in AND d_in2 (in place) but must not overlap just one of them.
 * Any 64-bit modulus: the arithmetic is the reference's, mod 2^64 (ntt.cpp:147-148, 331-369), so results are the
 * reference's for every modulus it accepts; they are the NTT when q < 2^62 (lazy range [0,4q) inside 64 bits). */
int agx_ref_fwd_dev(agx_ctx *ctx, uint32_t N, const uint64_t *d_in, const uint64_t *d_in2, uint64_t *d_out,
                    uint64_t modulus, const uint64_t *d_twiddles, const uint64_t *d_precon_twiddles, uint32_t numFrames,
                    void *stream);

/* ---- u64 inverse transform and negacyclic product on DEVICE pointers (no reference counterpart: the reference has
 * only the forward, SURVEY.md s.0).  Conventions of agx_ref_fwd_dev: frames [numFrames][N], N in {2^2 .. 2^15}, every
 * device pointer 16-byte aligned, asynchronous on `stream`, the caller's tables in the reference's order (ntt.cpp:298-300)
 * and not checked per call.  Unlike the forward, the modulus must be odd and 3 <= q < 2^62 (AGX_E_INVALID otherwise):
 * there is no reference behaviour to reproduce above 2^62, and the lazy range [0,4q) must fit 64 bits.
 * numFrames == 0 returns AGX_OK and launches nothing.  The results are the inverse NTT / the product exactly when the
 * tables are the Shoup pairs of psi (d_twiddles, d_precon_twiddles: agx_ref_fwd_dev's) and of psi^-1:
 * d_inv_twiddles[k] = psi^-bitrev(k) mod q, d_inv_precon_twiddles[k] = floor(d_inv_twiddles[k] * 2^64 / q)
 * (the forward table's order built from psi^-1; entry 0 unused).
 * Launches counted by agx_launch_count, out of place (N = 32768 in parentheses; an in-place forward there takes the
 * multi-launch pass kernels, see agx_ref_fwd_dev): agx_ref_inv_dev 1 (2), agx_ref_polymul_by_spectrum_dev 2 (3),
 * agx_ref_polymul_dev 3 (4). */

/* x = INTT(X): bit-reversed in (inputs < 2q), natural out in [0,q), n^-1 folded in (Gentleman-Sande, the mirror of
 * ntt.cpp:146-159, 292-300).  d_out == d_in (in place) or disjoint. */
int agx_ref_inv_dev(agx_ctx *ctx, uint32_t N, const uint64_t *d_in, uint64_t *d_out, uint64_t modulus,
                    const uint64_t *d_inv_twiddles, const uint64_t *d_inv_precon_twiddles, uint32_t numFrames,
                    void *stream);
/* c = a * b mod (X^N + 1, q) per frame = INTT(NTT(a) .* NTT(b)); operands reduced (< q), results in [0,q).  c may alias
 * a and/or b, and a may equal b (squaring); any other overlap is not allowed.  NTT(b) goes to a stream-ordered scratch
 * buffer (cudaMallocAsync on `stream`) unless a == b. */
int agx_ref_polymul_dev(agx_ctx *ctx, uint32_t N, uint64_t *d_c, const uint64_t *d_a, const uint64_t *d_b,
                        uint64_t modulus, const uint64_t *d_twiddles, const uint64_t *d_precon_twiddles,
                        const uint64_t *d_inv_twiddles, const uint64_t *d_inv_precon_twiddles, uint32_t numFrames,
                        void *stream);
/* c = INTT(NTT(a) .* b_hat) with b_hat = agx_ref_fwd_dev(b) (reduced, bit-reversed order): the product when one operand
 * is kept in evaluation form.  c may alias a and/or b_hat (c == b_hat costs a stream-ordered scratch buffer for NTT(a)).
 * Equals agx_ref_polymul_dev(c, a, b) bit for bit. */
int agx_ref_polymul_by_spectrum_dev(agx_ctx *ctx, uint32_t N, uint64_t *d_c, const uint64_t *d_a,
                                    const uint64_t *d_b_hat, uint64_t modulus, const uint64_t *d_twiddles,
                                    const uint64_t *d_precon_twiddles, const uint64_t *d_inv_twiddles,
                                    const uint64_t *d_inv_precon_twiddles, uint32_t numFrames, void *stream);

/* ---- u64 RNS batches: L primes of 50-62 bits, [B][L][n] DEVICE data (no reference counterpart; the u64 counterpart of
 * agx_create / agx_ntt_fwd / agx_ntt_inv / agx_polymul / agx_polymul_by_spectrum / agx_elementwise, SURVEY.md s.8(f)).
 * Conventions of the u32 batched entry points (device pointers, in place, asynchronous on `stream`, 16-byte aligned
 * pointers, uint64_t data[B][L][n] row-major: frame f = b * L + l is limb l of polynomial b) with the arithmetic of
 * agx_ref_fwd_dev / agx_ref_inv_dev.  A context holds either a u32 or a u64 parameter set: a u64 call on a u32 context
 * and the reverse give AGX_E_INVALID; the agx_ref_* calls work on every context.
 *
 * agx_create64: n = 2^logn in [4, 32768]; 1 <= nlimbs <= 64; every q[i] prime with 3 <= q < 2^62 and q = 1 (mod 2n).
 *   psi[nlimbs] is the caller's primitive 2n-th root per limb (AGX_E_INVALID unless psi[i]^n = -1 mod q[i]), NULL = the
 *   minimal one.  Anything else gives AGX_E_INVALID and no context.  The tables are built on the device at create time.
 * agx_get_tables64: one limb's table as HOST arrays of n words, in the reference's order (ntt.cpp:298-300): roots[k] =
 *   psi^bitrev(k) (inverse != 0: psi^-bitrev(k)), precons[k] = floor(roots[k] * 2^64 / q), entry 0 = 1 -- exactly the
 *   tables agx_ref_fwd_dev / agx_ref_inv_dev take.
 * Inputs: the forward accepts words < 4q, the inverse < 2q; product and element-wise operands must be reduced (< q).
 * Results are in [0,q).  For every limb, agx_ntt64_fwd, agx_ntt64_inv, agx_polymul64 and agx_polymul64_by_spectrum equal
 * bit for bit agx_ref_fwd_dev, agx_ref_inv_dev, agx_ref_polymul_dev and agx_ref_polymul_by_spectrum_dev on that limb's
 * frames with the tables of agx_get_tables64; agx_polymul64_by_spectrum(c, a, agx_ntt64_fwd(b)) = agx_polymul64(c, a, b).
 * c may alias a and/or b (b_hat), and a may equal b.  NTT(b) of the product takes a stream-ordered scratch buffer unless
 * a == b; so does NTT(a) of the by-spectrum product when c == b_hat.
 * B == 0 returns AGX_OK and launches nothing; B * nlimbs > 2^31 - 1 gives AGX_E_INVALID.
 * Launches (agx_launch_count), every limb in each: agx_ntt64_fwd 1, agx_ntt64_inv 1, agx_polymul64 3,
 * agx_polymul64_by_spectrum 2, agx_elementwise64 1; at n = 32768 the inverse adds one (its last stage streams over the
 * batch), so 1, 2, 4, 3, 1.  The forward at n = 32768 runs two CTAs per frame as a 2-CTA cluster, in place included. ---- */
typedef struct {
    uint32_t n;
    uint32_t logn;
    uint32_t nlimbs;
    const uint64_t *q; /* [nlimbs] */
} agx_parms64;

int agx_create64(agx_ctx **out, const agx_parms64 *parms, const uint64_t *psi, int device);
int agx_get_psi64(const agx_ctx *ctx, uint32_t limb, uint64_t *psi);
int agx_get_tables64(const agx_ctx *ctx, uint32_t limb, int inverse, uint64_t *roots, uint64_t *precons);
int agx_ntt64_fwd(agx_ctx *ctx, uint64_t *d_data, size_t B, void *stream);
int agx_ntt64_inv(agx_ctx *ctx, uint64_t *d_data, size_t B, void *stream);
int agx_polymul64(agx_ctx *ctx, uint64_t *d_c, const uint64_t *d_a, const uint64_t *d_b, size_t B, void *stream);
int agx_polymul64_by_spectrum(agx_ctx *ctx, uint64_t *d_c, const uint64_t *d_a, const uint64_t *d_b_hat, size_t B,
                              void *stream);
/* op = AGX_EW_*, modulo each limb's prime */
int agx_elementwise64(agx_ctx *ctx, int op, uint64_t *d_c, const uint64_t *d_a, const uint64_t *d_b, size_t B,
                      void *stream);

/* ---- u64 RNS rescale: division by the last prime with rounding, L limbs -> L - 1 (the step that brings a product back
 * down the modulus chain; no reference counterpart).  Primes q_0 .. q_{L-1}, L >= 2, Q = prod q_l, q_L' = q_{L-1},
 * Q' = Q / q_L', h = floor(q_L' / 2).  For each polynomial and coefficient j, X in [0, Q) is the CRT value of its L
 * residues, and the result is
 *     Y = floor((X + h) / q_L') mod Q'   (round half up of X / q_L'),
 * given as its residues mod q_0 .. q_{L-2}; since Q / q_L' = Q', it is the same residue vector whether X is read in
 * [0, Q) or centred.  In RNS form, with u = (x_{L-1} + h) mod q_L':  y_i = (x_i - (u - h)) * q_L'^-1 mod q_i, i < L - 1.
 *
 * d_in [B][L][n] -> d_out [B][L-1][n] over the context's first L - 1 primes.  ntt_form == 0: coefficient form (natural
 * order) in and out; ntt_form != 0: evaluation form as agx_ntt64_fwd leaves it (bit-reversed), in and out -- the result
 * is then agx_ntt64_fwd, over the first L - 1 primes, of the coefficient-form rescale of agx_ntt64_inv(d_in).
 * Input words must be reduced (< q_l); results are in [0, q_i); d_in is not modified.
 * AGX_E_INVALID, launching nothing, for: a u32 context; L < 2; a context whose last prime equals an earlier one; a null
 * pointer with B > 0; a pointer not 16-byte aligned; B * L > 2^31 - 1; byte ranges of d_in (B * L * n words) and d_out
 * (B * (L - 1) * n words) that overlap (in place is refused: compacting the stride from L to L - 1 would let one
 * polynomial's CTAs overwrite input another polynomial has not read yet).  B == 0 returns AGX_OK and launches nothing.
 * The evaluation form takes a stream-ordered scratch buffer of B * n words (cudaMallocAsync on `stream`).
 * Launches (agx_launch_count): coefficient form 1; evaluation form 2 (the inverse of limb L - 1; the forward of every
 * other limb with the rescale fused into its load and its store), 3 at n = 32768, where the inverse's last stage streams.
 *
 * The output belongs to the level below: run the other calls on it with a context created over q_0 .. q_{L-2} (with
 * psi[0 .. L-2] when the roots were the caller's).  That context's tables are the full context's first L - 1 limbs, bit
 * for bit, so a chain of levels is a chain of such contexts. ---- */
int agx_rescale64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, int ntt_form, void *stream);

/* ---- u64 RNS basis conversion: the two steps of hybrid key switching around the product with the key (no reference
 * counterpart).  Primes q_0 .. q_{L-1}; for a set of them with product S, X in [0, S) is the CRT value of a
 * coefficient's residues over that set and h_S = (S - 1) / 2 (every prime is odd).  Both calls are exact: mixed-radix
 * conversion in integer arithmetic, bit for bit the stated big-int definitions (not the approximate "fast base
 * conversion", which is off by a multiple of S).  Conventions are agx_rescale64's: device pointers 16-byte aligned,
 * asynchronous on `stream`; inputs reduced (< q), results in [0, q); d_in is not modified; ntt_form == 0: coefficient
 * form (natural order) in and out; ntt_form != 0: spectra as agx_ntt64_fwd leaves them, in and out, the result then being
 * agx_ntt64_fwd of the coefficient-form result of agx_ntt64_inv(d_in), each over its own primes.  The evaluation form
 * takes a stream-ordered scratch buffer of B * m * n words (cudaMallocAsync on `stream`; m = k or count below).
 * Per call, the constants that depend on the source set (h mod q_i, P^-1 mod q_i) are computed on the host from a copy
 * of the pairwise table built at agx_create64 and passed as a kernel parameter: no per-call upload.
 *
 * ModDown: d_in [B][L][n] -> d_out [B][L-k][n].  P = q_{L-k} .. q_{L-1} (the last k primes), Q' = q_0 .. q_{L-k-1}:
 *     Y = floor((X + h_P) / P) mod Q',   X in [0, Q) the CRT value of the L residues,
 * given as its residues over q_0 .. q_{L-k-1}.  k = 1 is agx_rescale64, and is served by it (same kernels, launches).
 * The output belongs to a context over q_0 .. q_{L-k-1} (that context's tables are this one's first L - k limbs).
 * AGX_E_INVALID, launching nothing, for: a u32 context; a null pointer with B > 0; a pointer not 16-byte aligned;
 * B * L > 2^31 - 1; k = 0 or k >= L; two equal primes among the last k, or one of them equal to one of the first L - k;
 * byte ranges of d_in (B * L * n words) and d_out (B * (L - k) * n words) that overlap (in place is refused, as for the
 * rescale: the strides differ).  AGX_E_UNSUPPORTED for k > 16 (AGX_BASIS_MAX_SRC): a coefficient's k digits are kept in
 * registers.  B == 0 returns AGX_OK and launches nothing.
 * Launches (agx_launch_count), k >= 2: coefficient form 1; evaluation form 3 (the inverse of the last k limbs; the
 * mixed-radix digits; the forward of the other limbs with the conversion fused into its load and its store), 4 at
 * n = 32768, where the inverse's last stage streams.  k = 1: the rescale's (1; 2, 3 at n = 32768).
 */
#define AGX_BASIS_MAX_SRC 16
int agx_moddown64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, uint32_t k, int ntt_form, void *stream);

/* ModUp: d_in [B][count][n] over the primes q_first .. q_{first+count-1} (product S) -> d_out [B][L][n] over all L:
 *     X_c = ((X + h_S) mod S) - h_S,   the centred lift of the source residues, given mod every q_i;
 * the source limbs first .. first + count - 1 of d_out equal d_in's limbs.  A key-switch digit over part of the basis
 * thus reaches the whole extended basis Q u P.
 * AGX_E_INVALID, launching nothing, for: a u32 context; a null pointer with B > 0; a pointer not 16-byte aligned;
 * B * L > 2^31 - 1; count = 0, count >= L or first + count > L; two equal source primes, or a target prime equal to a
 * source prime; overlapping byte ranges of d_in (B * count * n words) and d_out (B * L * n words).
 * AGX_E_UNSUPPORTED for count > 16.  B == 0 returns AGX_OK and launches nothing.
 * Launches: coefficient form 1; evaluation form 3 (the inverse of the source limbs; the digits; the forward of the
 * target limbs), 4 at n = 32768; count = 1 needs no digits kernel: 2, 3 at n = 32768.  The evaluation form also copies
 * the source spectra into their output limbs (one pitched device-to-device cudaMemcpy2DAsync, not a launch). ---- */
int agx_modup64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, uint32_t first, uint32_t count,
                int ntt_form, void *stream);

/* ---- u64 RNS Galois automorphisms: the permutation half of a rotation or conjugation (no reference counterpart).  For
 * a Galois element g, odd with 1 <= g < 2n,
 *     sigma_g: a(X) -> a(X^g) mod X^n + 1,
 * the same map on every limb.  d_in [B][L][n] -> d_out [G][B][L][n]: output t, itself an ordinary [B][L][n] batch, is
 * sigma_{galois[t]}(d_in).  galois is a host array of G elements; with G > 1 the input is read once for all G outputs
 * (the hoisted rotations of key switching: one ModUp, then every rotation of the extended digit).  A slot rotation by
 * r steps is g = 5^r mod 2n (r < 0: the inverse of 5^-r), the conjugation g = 2n - 1.
 *   ntt_form == 0, coefficient form (natural order): coefficient i moves to i * g mod 2n; from position m >= n it goes to
 *     m - n negated (X^n = -1), where the negation of x is q_l - x for x != 0 and 0 for x = 0.  As a gather:
 *     out[j] = in[u] for u < n, -in[u - n] for u >= n, with u = j * g^-1 mod 2n.
 *   ntt_form != 0, evaluation form (bit-reversed, as agx_ntt64_fwd leaves it: entry k = a(psi^(2 br(k) + 1))): a pure
 *     permutation, no sign,
 *     out[k] = in[br(((g * (2 br(k) + 1)) mod 2n - 1) / 2)],
 *     equal to agx_ntt64_fwd(sigma_g(agx_ntt64_inv(d_in))) for every primitive 2n-th root, the caller's ones included.
 * Conventions are agx_rescale64's: device pointers 16-byte aligned, asynchronous on `stream`; inputs reduced (< q_l),
 * results in [0, q_l); d_in is not modified.  No scratch memory, no host <-> device copies; the inverses g^-1 mod 2n are
 * passed by value as a kernel parameter.
 * AGX_E_INVALID, launching nothing, for: a u32 context; a null device pointer with B > 0; a null galois with G > 0; a
 * pointer not 16-byte aligned; G * B * L > 2^31 - 1; byte ranges of d_in (B * L * n words) and d_out (G * B * L * n
 * words) that overlap (in place is refused); any element that is even, 0 or >= 2n.  AGX_E_UNSUPPORTED for G > 64
 * (AGX_AUTOMORPH_MAX; the elements are then not read).  B == 0 or G == 0 returns AGX_OK and launches nothing.
 * Launches: 1 per call, in both forms, at every n and every G. ---- */
#define AGX_AUTOMORPH_MAX 64
int agx_automorph64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint32_t *galois, uint32_t G,
                    int ntt_form, void *stream);

/* ---- u64 RNS hybrid key switching in one call (no reference counterpart): the relinearisation of a product, or the
 * key-switch half of a rotation (agx_automorph64, then this).  ctx is a u64 context over Q_l u P, special primes last:
 * L = l + 1 + k primes q_0 .. q_l, p_0 .. p_{k-1}.
 *   d_in  [B][l+1][n] over Q_l, the context's first L - k primes.
 *   Digits: digit j is limbs j*alpha .. min((j+1)*alpha, l+1) - 1 of d_in; dnum = ceil((l+1) / alpha).  alpha >= l + 1
 *     means one digit, so a caller may keep alpha fixed as l drops below it.
 *   d_ksk [>= dnum][2][key_limbs][n], in evaluation form as agx_ntt64_fwd leaves it under this context's roots (the key
 *     is in evaluation form in both forms of the call); the caller guarantees dnum digits.  key_limbs >= L, and context
 *     limb i <= l reads key row i, context limb l + 1 + t (special prime p_t) reads key row key_limbs - k + t.  So
 *     key_limbs = L is a key over exactly this basis, and key_limbs = L_top + k is one key over Q_top u P, generated
 *     once and used unchanged at every level l <= L_top - 1.
 *   d_out [2][B][l+1][n], for c = 0, 1:
 *     out_c = ModDown_P( sum_j ModUp_j(digit_j) (.) ksk[j][c] ),
 *   ModUp_j = agx_modup64(first = j*alpha, count = the digit's size), ModDown_P = agx_moddown64(k), (.) the product of
 *   each limb with its key row: element-wise in evaluation form, the negacyclic product in coefficient form.  Every
 *   step is exact: the result equals, bit for bit, that sequence of public calls with the key rows sliced out of d_ksk
 *   and replicated over the batch.  The output belongs to the context over Q_l.
 *   ntt_form != 0: d_in and d_out are spectra; ntt_form == 0: both in natural coefficient order, d_out then being
 *   agx_ntt64_inv (over Q_l) of the evaluation form applied to agx_ntt64_fwd(d_in).
 * Conventions are agx_moddown64's: device pointers 16-byte aligned, asynchronous on `stream`; inputs reduced, results in
 * [0, q); d_in and d_ksk are not modified.  Scratch: one stream-ordered buffer (cudaMallocFromPoolAsync on `stream`)
 * of (dnum + 2) * B * L * n words, plus B * min(alpha, l+1) * n when dnum > 1, plus what the ModUps and the ModDown take
 * (see above) while they run.  The buffer comes from a memory pool the context creates at its first key switch and
 * keeps until agx_destroy: the pool holds on to the largest scratch a call has used, so later calls do not map it
 * again (the device's default pool returns freed memory at every synchronisation, and mapping gigabytes per call
 * doubled the time of a call at the sizes measured in DESIGN.md).  The digits' constants come from the host copy of the pairwise table: no per-call upload,
 * no host synchronisation.  With dnum > 1 each digit is first gathered into the scratch by one pitched
 * cudaMemcpy2DAsync (not a launch).
 * AGX_E_INVALID, launching nothing, for: a u32 context; a null pointer with B > 0; a pointer not 16-byte aligned;
 * k = 0 or k >= L; alpha = 0; key_limbs < L; two equal primes anywhere in the context; 2 * B * L or dnum * B * L above
 * 2^31 - 1; d_out (2 * B * (l+1) * n words) overlapping d_in (B * (l+1) * n words) or the dnum digits of d_ksk that are
 * read (dnum * 2 * key_limbs * n words).  AGX_E_UNSUPPORTED for min(alpha, l+1) > 16 or k > 16 (AGX_BASIS_MAX_SRC).
 * B == 0 returns AGX_OK and launches nothing.
 * Launches (agx_launch_count): evaluation form sum_j up_j + 1 + down, with up_j the ModUp's launches for digit j (3; 2
 * for a one-prime digit; one more each at n = 32768) and down the ModDown's (3, or 2 for k = 1; one more at n = 32768):
 * 3 * dnum + 4 for digits of two or more primes and k >= 2, 4 * dnum + 5 at n = 32768.  Coefficient form
 * dnum + 4 (one ModUp per digit; the forward of every extended digit; the inner product; the inverse of the two
 * products; the ModDown), dnum + 5 at n = 32768. ---- */
int agx_keyswitch64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint64_t *d_ksk,
                    uint32_t key_limbs, uint32_t alpha, uint32_t k, int ntt_form, void *stream);

/* ---- u64 RNS hoisted rotations in one call (no reference counterpart): G rotations or conjugations of the same
 * ciphertexts, each with its own key, with one ModUp of c1 for all G.  ctx, alpha, k, key_limbs and the key layout are
 * agx_keyswitch64's (dnum = ceil((l+1) / alpha) digits, the row map that lets one top-level key serve every level).
 *   d_in  [2][B][l+1][n]: ciphertexts (c0, c1) over Q_l (the layout agx_keyswitch64 writes, so outputs can be fed back).
 *   galois: a host array of G elements, agx_automorph64's rules (odd, in [1, 2n), G <= AGX_AUTOMORPH_MAX).
 *   d_rk: a host array of G device pointers; key t, [>= dnum][2][key_limbs][n] in evaluation form, switches
 *     sigma_{galois[t]}(s) back to s.  Two elements may share a key pointer; one key_limbs serves all G keys.
 *   d_out [G][2][B][l+1][n], output t being, bit for bit and in both forms, the plain recipe of public calls:
 *     out[t] = ( sigma_t(c0) + KS_t(sigma_t(c1))[0],  KS_t(sigma_t(c1))[1] ),
 *   with sigma_t = agx_automorph64 with galois[t], KS_t = agx_keyswitch64 with key t and the sum agx_elementwise64's add.
 *   The call runs the ModUp of c1's digits once, then for every t the key inner product over the permuted extended
 *   digits with sigma_t(c0) folded in as P * sigma_t(c0) (which ModDown returns exactly), then one ModDown of all 2 G B
 *   polynomials.
 * Conventions are agx_keyswitch64's: device pointers 16-byte aligned, asynchronous on `stream`, inputs reduced, results
 * in [0, q); d_in and the keys are not modified.  Scratch: one buffer from the context's key-switch pool (see
 * agx_keyswitch64) of (dnum + 2 G) * B * L * n words, plus B * min(alpha, l+1) * n when dnum > 1, plus B * (l+1) * n in
 * coefficient form; the ModDown's scratch (evaluation form: 2 G B k n words) comes from the same pool; the ModUps take
 * their own (agx_modup64).  The elements' inverses and the key pointers are passed by value as a kernel parameter.
 * AGX_E_INVALID, launching nothing, for: a u32 context; with B > 0 a null d_out, d_in or d_rk[t]; with G > 0 a null
 * galois or d_rk; a pointer not 16-byte aligned; k = 0 or k >= L; alpha = 0; key_limbs < L; two equal primes anywhere in
 * the context; an element that is even, 0 or >= 2n; 2 * G * B * L or dnum * B * L above 2^31 - 1; d_out (2 G B (l+1) n
 * words) overlapping d_in (2 B (l+1) n words) or the dnum * 2 * key_limbs * n words read from any key.
 * AGX_E_UNSUPPORTED for G > 64 (the elements and keys are then not read), min(alpha, l+1) > 16 or k > 16.
 * B == 0 or G == 0 returns AGX_OK and launches nothing.
 * Launches (agx_launch_count), independent of G: evaluation form sum_j up_j + 1 + down with agx_keyswitch64's up_j and
 * down: 3 * dnum + 4 for digits of two or more primes and k >= 2, 4 * dnum + 5 at n = 32768 (one fewer per one-prime
 * digit, and one fewer for k = 1).  Coefficient form dnum + 5 (one ModUp per digit; the forward of the extended digits;
 * the forward of c0; the inner products; the inverse of A; the ModDown), dnum + 6 at n = 32768. ---- */
int agx_rotate64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint32_t *galois, uint32_t G,
                 const uint64_t *const *d_rk, uint32_t key_limbs, uint32_t alpha, uint32_t k, int ntt_form, void *stream);

/* ---- u64 RNS hoisted linear transforms in one call (no reference counterpart): M plaintext-weighted sums of G
 * rotations of the same ciphertexts, out[m] = sum_t d_{m,t} (.) rot_t(ct), with one ModUp of c1 for all G and one
 * ModDown per output (double hoisting: the baby steps of a baby-step/giant-step matrix-vector product, CoeffToSlot /
 * SlotToCoeff factors, slot sums).  ctx, alpha, k, key_limbs, the key layout and galois are agx_rotate64's.
 *   d_in  [2][B][l+1][n]: ciphertexts (c0, c1) over Q_l, agx_rotate64's layout.
 *   d_rk: a host array of G device pointers, key t switching sigma_t(s) to s; d_rk[t] may be NULL only when
 *     galois[t] == 1: that term is the identity, with no key switch.
 *   d_diag: a host array of M * G device pointers; entry m * G + t is the diagonal d_{m,t}, [L][n] over all L primes of
 *     the context (Q_l u P), in evaluation form as agx_ntt64_fwd leaves it (in both forms of the call), shared by the
 *     whole batch.  NULL is a zero diagonal and is skipped; entries may share a pointer.  A diagonal encoded over Q_l
 *     reaches Q_l u P with agx_modup64.
 *   d_out [M][2][B][l+1][n], for every m and c = 0, 1:
 *     A_t[c]    = sum_j sigma_t(ModUp_j(digit_j(c1))) (.) rk_t[j][c] + [c = 0] P sigma_t(c0)   (agx_rotate64's, over Q_l u P)
 *     A_t       = (P c0, P c1)                                        when galois[t] == 1 and d_rk[t] == NULL
 *     out[m][c] = ModDown_P( sum_t d_{m,t} (.) A_t[c] ),
 *   P x being 0 on the special primes and (P mod q_i) x on limb i of Q_l.  So out[m] = sum_t d_{m,t} sigma_t(c0) +
 *   ModDown(sum_t d_{m,t} KS_t): one rounding per output.  Every step is exact, so the result equals, bit for bit, that
 *   sequence of public calls (modup of each digit, automorph, elementwise products and sums, one moddown of 2 M B); it is
 *   NOT bit-equal to sum_t d_{m,t} (.) agx_rotate64(...)[t], which rounds G times.  An output whose diagonals are all
 *   NULL is the zero ciphertext, and it is written.  ntt_form != 0: d_in and d_out are spectra; ntt_form == 0: both in
 *   natural coefficient order, d_out then being agx_ntt64_inv (over Q_l) of the evaluation-form result applied to
 *   agx_ntt64_fwd(d_in).  Keys and diagonals are in evaluation form either way.
 * Conventions are agx_rotate64's: device pointers 16-byte aligned, asynchronous on `stream`, inputs reduced, results in
 * [0, q); d_in, keys and diagonals are not modified.  Scratch: one buffer from the context's key-switch pool (see
 * agx_keyswitch64) of (dnum + 2 M) * B * L * n words, plus B * min(alpha, l+1) * n when dnum > 1, plus 2 B (l+1) n in
 * coefficient form; the ModDown's scratch comes from the same pool; the ModUps take their own.  No [G] buffer: the
 * A_t are formed in registers and never stored.  Elements, key and diagonal pointers travel by value as a kernel
 * parameter; terms whose M diagonals are all NULL are dropped before the launch.
 * AGX_E_INVALID, launching nothing, for agx_rotate64's cases (a u32 context; with B > 0 a null d_out or d_in; with
 * G > 0 a null galois or d_rk; a pointer not 16-byte aligned; k = 0 or k >= L; alpha = 0; key_limbs < L; two equal
 * primes; an even element, 0 or >= 2n) and for: with B > 0 a NULL key with g != 1; G == 0 with M > 0; M > 0 with a null
 * d_diag; 2 M B L or dnum B L above 2^31 - 1; with B, M > 0, d_out (2 M B (l+1) n words) overlapping d_in
 * (2 B (l+1) n), the dnum * 2 * key_limbs * n words read from any key, or any non-NULL diagonal (L n words).
 * AGX_E_UNSUPPORTED for G > 64, M > AGX_LINTRANS_MAX_OUT or M * G > AGX_LINTRANS_MAX_TERMS (the elements, keys and
 * diagonals are then not read), min(alpha, l+1) > 16 or k > 16.  B == 0 or M == 0 returns AGX_OK and launches nothing.
 * Launches (agx_launch_count), independent of G and M and equal to agx_rotate64's: evaluation form 3 * dnum + 4 for
 * digits of two or more primes and k >= 2, 4 * dnum + 5 at n = 32768 (one fewer per one-prime digit, and one fewer for
 * k = 1).  Coefficient form dnum + 5 (one ModUp per digit; the forward of the extended digits; the forward of c0 and c1;
 * the inner sums; the inverse of the sums; the ModDown), dnum + 6 at n = 32768. ---- */
#define AGX_LINTRANS_MAX_OUT 16    /* M */
#define AGX_LINTRANS_MAX_TERMS 256 /* M * G: the diagonal pointers travel by value as a kernel parameter (< 4 KB) */
int agx_lintrans64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint32_t *galois, uint32_t G,
                   const uint64_t *const *d_rk, uint32_t key_limbs, const uint64_t *const *d_diag, uint32_t M,
                   uint32_t alpha, uint32_t k, int ntt_form, void *stream);

/* ---- u64 RNS ciphertext multiplication in one call (no reference counterpart): the tensor product of two
 * ciphertexts, its relinearisation and, optionally, the rescale by q_l.  ctx, alpha, k, key_limbs and the key layout are
 * agx_keyswitch64's: ctx is Q_l u P with the k special primes last, dnum = ceil((l+1) / min(alpha, l+1)).
 *   d_a, d_b [2][B][l+1][n]: ciphertexts (a0, a1) and (b0, b1) over Q_l, agx_keyswitch64's output layout.  d_a == d_b
 *     squares; both are only read, so any overlap between them is harmless.
 *   d_rlk [>= dnum][2][key_limbs][n]: the relinearisation key, i.e. agx_keyswitch64's key for s' = s^2, in evaluation
 *     form; its row map lets one key over Q_top u P serve every level.
 *   For c = 0, 1, every product per limb (element-wise in evaluation form):
 *     D_0 = a0 b0,  D_1 = a0 b1 + a1 b0,  D_2 = a1 b1                                  over Q_l
 *     A_c = sum_j ModUp_j(digit_j(D_2)) (.) rlk[j][c]  +  P D_c                         over Q_l u P,
 *   P D_c being (P mod q_i) D_c on limb i <= l and 0 on the special primes.
 *   rescale == 0: d_out [2][B][l+1][n], out_c = ModDown_P(A_c) = D_c + agx_keyswitch64(D_2)[c] (the fold: ModDown of
 *     X + P C is ModDown(X) + C exactly).  Bit for bit the recipe of public calls: the tensor, agx_keyswitch64 of D_2,
 *     then agx_elementwise64 adds.
 *   rescale != 0: d_out [2][B][l][n] over Q_{l-1}, belonging to the context over q_0 .. q_{l-1}:
 *     out_c = floor((X_c + h) / (q_l P)) mod Q_{l-1},  X_c in [0, Q_l P) the CRT value of A_c, h = (q_l P - 1) / 2,
 *     i.e. agx_moddown64 with k + 1 of A_c: bit for bit the recipe of public calls ending in one agx_moddown64(k + 1)
 *     of the 2 B polynomials.  It rounds once, and it also equals agx_rescale64 of the rescale == 0 output bit for
 *     bit (so the two differ by 0, within any bound of 1): h = h_P + P h_q with h_P = (P - 1) / 2 and
 *     h_q = (q_l - 1) / 2, and floor((floor((X + h_P) / P) + h_q) / q_l) = floor((X + h) / (q_l P)) (nested floor
 *     division); the reduction mod Q_l between the steps changes nothing mod Q_{l-1}.  The call saves the rescale's
 *     pass, not a rounding.
 *   ntt_form != 0: d_a, d_b and d_out are spectra; ntt_form == 0: all three in natural coefficient order, d_out then
 *   being the inverse of the evaluation-form result on the spectra of d_a and d_b.  The key is in evaluation form
 *   either way.
 * Conventions are agx_keyswitch64's: device pointers 16-byte aligned, asynchronous on `stream`, inputs reduced, results
 * in [0, q); d_a, d_b and the key are not modified.  Scratch: one buffer from the context's key-switch pool (see
 * agx_keyswitch64) of (dnum + 2) * B * L * n + B * (l+1) * n words, plus B * min(alpha, l+1) * n when dnum > 1, plus
 * 4 B (l+1) n in coefficient form (2 B (l+1) n when squaring); the ModDown's scratch comes from the same pool; the
 * ModUps take their own.  D_0 and D_1 are formed in registers and never stored.
 * AGX_E_INVALID, launching nothing, for agx_keyswitch64's cases (a u32 context; with B > 0 a null d_out, d_a, d_b or
 * d_rlk; a pointer not 16-byte aligned; k = 0 or k >= L; alpha = 0; key_limbs < L; two equal primes) and for: rescale
 * != 0 with l + 1 < 2; 2 B L or dnum B L above 2^31 - 1; with B > 0, d_out (2 B (l+1) n words, 2 B l n with rescale)
 * overlapping d_a or d_b (2 B (l+1) n each) or the dnum * 2 * key_limbs * n key words read.
 * AGX_E_UNSUPPORTED for min(alpha, l+1) > 16, k > 16, or rescale != 0 with k + 1 > 16.  B == 0 returns AGX_OK and
 * launches nothing.
 * Launches (agx_launch_count), independent of B: evaluation form 3 * dnum + 5 (the product D_2 = a1 b1; three per
 * digit's ModUp; the inner sums; the ModDown's three), 4 * dnum + 6 at n = 32768; one fewer per one-prime digit, and
 * one fewer for k = 1 without rescale (the ModDown is then agx_rescale64's two).  Coefficient form 3 * dnum + 6 (the
 * forwards of a and b; as above; the inverse of the sums; the coefficient-form ModDown's one), 4 * dnum + 7 at
 * n = 32768, one fewer when squaring (d_a == d_b: one forward) and one fewer per one-prime digit. ---- */
int agx_mulrelin64(agx_ctx *ctx, uint64_t *d_out, const uint64_t *d_a, const uint64_t *d_b, size_t B,
                   const uint64_t *d_rlk, uint32_t key_limbs, uint32_t alpha, uint32_t k, int rescale, int ntt_form,
                   void *stream);

/* ---- u64 RNS CKKS encoding and decoding (no reference counterpart): complex slot vectors to plaintexts and back.
 * n = 2^logn, S = n / 2 slots, zeta = exp(i pi / n).  Slot j of a real polynomial m is m(zeta^(5^j mod 2n)), j < S, so
 * agx_automorph64 with g = 5^r (a rotation by r steps) maps the slot vector z to out_j = z_(j+r mod S), and g = 2n - 1
 * conjugates every slot.  Encoding is the inverse with real coefficients: m_i = (2 / n) sum_j Re(z_j zeta^(-i 5^j)).
 * Both calls run the special FFT of length S in FP64 on the device (the HEAAN form: stage twiddles zeta^((5^j mod 8h)
 * (2n / 8h)) for half-length h), one CTA per polynomial with its S complex words in shared memory; at n = 32768 a 2-CTA
 * cluster per polynomial (the encode's first and the decode's last stage cross the halves).
 *   d_slots [B][S][2] doubles (re, im): a contiguous complex128 (B, S).  Residues [B][limbs][n] over the context's first
 *   `limbs` primes, 1 <= limbs <= L.  With limbs = L on a Q_l u P context the encode writes what agx_lintrans64 takes as
 *   a diagonal (ntt_form = 1); with limbs = l + 1 a plaintext over Q_l.
 * agx_encode64: m~ = the FP64 inverse special FFT of z (its 1 / S folded into the scale, exactly: scale / S is kept
 *   normal by the refusal below), c_i = rint(fl(scale
 *   m~_i)) rounding half to even, an integer of any magnitude a double holds, and out[b][l][i] = c_i mod q_l in [0, q_l).
 *   The residue is exact at every magnitude: |c| < 2^63 through a 64-bit integer, above that c = M 2^e with M < 2^53 and
 *   (M mod q) times 2^e mod q, the sign applied last (scales above 2^64, e.g. q_l q_(l-1), are normal).  Error against
 *   the exact m: |c_i - scale m_i| <= 1/2 + scale ||z||_inf * 5 * log2(n) * 2^-53 (DESIGN.md s.4).  Slot values are not
 *   checked: a non-finite slot gives unspecified residues.  ntt_form != 0: the output equals, bit for bit,
 *   agx_ntt64_fwd over limbs 0 .. limbs - 1 of the coefficient-form output.
 * agx_decode64: X_i the CRT value of in[b][0 .. limbs-1][i] over Q = q_0 ... q_(limbs-1), X_c = ((X + h) mod Q) - h with
 *   h = (Q - 1) / 2 (agx_modup64's centred lift), m_i = X_c / scale in FP64, z = the FP64 forward special FFT of m.
 *   ntt_form != 0: d_in is a spectrum, decoded as agx_ntt64_inv of it.  The CRT step is exact mixed-radix digits
 *   (Garner, O(limbs^2) per coefficient: decoding normally happens at low levels), the centring done on the digits
 *   (no cancellation), then Horner in double from the top digit and one division: |m_i - X_c / scale| <=
 *   (2 limbs + 1) 2^-53 |X_c / scale|; |X_c| / scale >= 2^1024 gives +-inf.  The FFT adds at most
 *   5 log2(n) 2^-53 S ||m||_inf per slot.  d_in is not modified.
 * Conventions are agx_rescale64's: device pointers 16-byte aligned, asynchronous on `stream`; residues reduced.
 * AGX_E_INVALID, launching nothing, for: a u32 context; a null pointer with B > 0; a pointer not 16-byte aligned;
 * limbs = 0 or limbs > L; a scale that is not finite or is <= 0 (for the encode, below 2^-1022 * S); B * limbs >
 * 2^31 - 1; byte ranges of the slots
 * (B * n words) and the residues (B * limbs * n words) that overlap; for the decode, two equal primes among the first
 * limbs.  B == 0 returns AGX_OK and launches nothing.
 * Launches (agx_launch_count), independent of B, of the scale and of whether the call is the context's first: encode 1
 * in coefficient form, 2 in evaluation form (the forward over the output limbs, in place); decode 2 in coefficient form
 * (the CRT step, the FFT), 3 in evaluation form (the inverse into scratch first), 4 at n = 32768 where the inverse
 * streams its last stage.  n = 32768 adds no launch of its own (the clusters).
 * Scratch: the decode takes B * n doubles, plus B * limbs * n words in evaluation form, from the context's key-switch
 * pool (agx_keyswitch64).  The S twiddles (complex128, 256 KB at n = 32768) are computed on the host in long double at
 * the context's first encode or decode, uploaded by one synchronous cudaMemcpy followed by cudaDeviceSynchronize (a
 * pageable upload may still be in flight when cudaMemcpy returns, and a non-blocking stream is not ordered after it),
 * and kept until agx_destroy. ---- */
int agx_encode64(agx_ctx *ctx, uint64_t *d_out, const double *d_slots, size_t B, double scale, uint32_t limbs,
                 int ntt_form, void *stream);
int agx_decode64(agx_ctx *ctx, double *d_slots, const uint64_t *d_in, size_t B, double scale, uint32_t limbs,
                 int ntt_form, void *stream);

/* ---- diagnostics ---- */
const char *agx_error_string(int code);
/* kernels this library launched on ctx since creation (bench.py's gpu_launches claim) */
int agx_launch_count(const agx_ctx *ctx, uint64_t *count);
/* name of the kernel variant serving (n): "ntt2p<LOGN,LE>" or "generic" */
int agx_variant(const agx_ctx *ctx, char *buf, size_t buflen);
/* The measured integer roofline of this GPU: the butterfly's instruction stream alone (no memory operations), one CTA
 * of `threads_per_sm` (128..1024, multiple of 128) threads per SM, timed in SM clocks.  kind 0: the u32 Harvey/Shoup
 * butterfly of the batched kernels; kind 1: the u64 butterfly of the reference-shaped path (ntt.cpp:331-369); kind 2 / 3:
 * kind 0 with one / two extra non-multiply instructions per butterfly (the issue-slot load of a real kernel); kinds 4-6:
 * further variants of the stream used by profiles/diag_issue_pressure.py (see csrc/agx_diag.cuh).
 * *per_clk_per_sm = butterflies retired per clock per SM; *sm_mhz (may be NULL) = the clock the run implied. */
int agx_measure_butterfly_peak(agx_ctx *ctx, int kind, int threads_per_sm, double *per_clk_per_sm, double *sm_mhz);

#ifdef __cplusplus
}
#endif
#endif /* AGXNTT_H */
