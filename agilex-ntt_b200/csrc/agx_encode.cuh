// CKKS encoding and decoding on the u64 RNS path (agx_encode64 / agx_decode64): complex slot vectors to RNS
// plaintexts and back.  Included by agx_api.cu after agx_ntt_kernels.cuh, whose u64 helpers it uses.
//
// n = 2^logn, S = n / 2 slots, zeta = exp(i pi / n), slot j of a real polynomial m is m(zeta^(5^j mod 2n)).  The
// special FFT of length S (the HEAAN / Lattigo form) maps between the slots and v_i = m_i + i m_(i+S):
//   inverse (encode): for h = S/2 .. 1, every block of 2h, j < h:  (u, v) <- (u + v, (u - v) conj(w[h + j]));
//                     then bit reversal and the factor 1 / S;
//   forward (decode): bit reversal, then for h = 1 .. S/2:         (u, v) <- (u + v w[h + j], u - v w[h + j]).
// w[h + j] = zeta^((5^j mod 8h) * (2n / 8h)), the stage-ordered table of S words (entry 0 unused) that the context
// builds on the host in long double at its first encode or decode call.
//
// Geometry: one CTA per polynomial holds its S complex words in shared memory (128 KB at n = 16384).  At n = 32768
// (256 KB) a polynomial runs on a 2-CTA cluster, each CTA holding one half: the encode's first stage (h = S/2, which
// pairs the two halves) is computed from global memory by both CTAs, CTA r keeping output half r; the decode's last
// stage reads the partner's half through distributed shared memory.  Everything between is local to a CTA.
#pragma once

namespace agx {

constexpr uint32_t kEncodeMaxLocal = 8192;   // complex words one CTA holds: S at n <= 16384, S / 2 at n = 32768
constexpr uint32_t kDecodeCrtThreads = 128;

__host__ __device__ __forceinline__ uint32_t slot_threads(uint32_t logn) {
    const uint32_t half = 1u << (logn >= 15 ? 13 : logn - 1);     // complex words per CTA
    return half / 2 < 32 ? 32 : (half / 2 > 512 ? 512 : half / 2);
}

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cmul_conj(double2 a, double2 b) {   // a * conj(b)
    return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csubd(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }

__device__ __forceinline__ double2 ld_dsmem_d2(uint32_t saddr, uint32_t rank) {
    uint32_t a;
    double x, y;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(saddr), "r"(rank));
    asm volatile("ld.shared::cluster.v2.f64 {%0, %1}, [%2];" : "=d"(x), "=d"(y) : "r"(a));
    return make_double2(x, y);
}

__device__ __forceinline__ void encode_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// c mod q for an integer-valued double c of any magnitude (exact): |c| < 2^63 through a 64-bit integer; above, c =
// M 2^e with M < 2^53, and M mod q is multiplied by 2^64 (reduce128) e / 64 times and by 2^(e mod 64) once.  The sign
// is applied last.  A non-finite c gives an unspecified residue (the loop is bounded all the same).
__device__ __forceinline__ uint64_t encode_residue(double c, uint64_t q, uint64_t one_p, const RnsLimb64 *lc) {
    const double a = fabs(c);
    uint64_t r;
    if (a < 9223372036854775808.0) {
        r = ref_csub_u64(ref_shoup_u64((uint64_t)__double2ll_rz(a), 1, one_p, q), q);
    } else {
        int E;
        const double f = frexp(a, &E);                             // a = f 2^E, f in [0.5, 1)
        const uint64_t M = (uint64_t)__double2ull_rz(ldexp(f, 53));
        int e = min(max(E - 53, 0), 1024);
        r = ref_csub_u64(ref_shoup_u64(M, 1, one_p, q), q);
        const LazyRed64 lr = lazy_red64(lc);
        while (e > 0) {
            const int s = min(e, 64);
            const uint64_t hi = s == 64 ? r : r >> (64 - s), lo = s == 64 ? 0 : r << s;
            r = reduce128(lo, hi, lr);
            e -= s;
        }
    }
    return (c < 0 && r) ? q - r : r;
}

// agx_encode64: slots [B][S] complex -> residues [B][limbs][n], coefficient form.  CL = 2 at n = 32768.
// c_i = rint(fl(sc * Re(v_i))), c_(i+S) = rint(fl(sc * Im(v_i))) with sc = scale / S (exact: S is a power of two), v
// the inverse special FFT before its 1 / S.  Thread t takes output index i and writes c_i and c_(i+S) to every limb,
// consecutive threads consecutive i; the coefficients never reach memory as doubles.
template <int CL>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(512) encode64_kernel(uint64_t *__restrict__ out, const double2 *__restrict__ slots,
                                                       const double2 *__restrict__ tw,
                                                       const BasisLimb64 *__restrict__ bl,
                                                       const RnsLimb64 *__restrict__ lc, uint32_t logn, uint32_t limbs,
                                                       double sc) {
    extern __shared__ __align__(16) double2 sv[];
    const uint32_t n = 1u << logn, S = n >> 1, part = S / CL, lgp = logn - 1 - (CL == 2 ? 1 : 0);
    const uint32_t rank = CL == 2 ? blockIdx.x & 1 : 0, poly = CL == 2 ? blockIdx.x >> 1 : blockIdx.x;
    const double2 *z = slots + (size_t)poly * S;
    uint32_t hstart = S >> 1;
    if (CL == 2) {                                                 // first stage h = S/2 from global, half `rank` kept
        const uint32_t h = S >> 1;
        for (uint32_t k = threadIdx.x; k < part; k += blockDim.x) {
            const double2 u = z[k], v = z[k + h];
            sv[k] = rank == 0 ? cadd(u, v) : cmul_conj(csubd(u, v), tw[h + k]);
        }
        hstart = h >> 1;
    } else {
        for (uint32_t k = threadIdx.x; k < part; k += blockDim.x) sv[k] = z[k];
    }
    __syncthreads();
    for (uint32_t h = hstart; h >= 1; h >>= 1) {
        for (uint32_t b = threadIdx.x; b < part / 2; b += blockDim.x) {
            const uint32_t j = b & (h - 1), i = ((b - j) << 1) + j;
            const double2 u = sv[i], v = sv[i + h];
            sv[i] = cadd(u, v);
            sv[i + h] = cmul_conj(csubd(u, v), tw[h + j]);
        }
        __syncthreads();
    }
    if (CL == 2) encode_cluster_sync();                            // both halves are final
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(sv);
    uint64_t *dst = out + (size_t)poly * limbs * n;
    for (uint32_t t = threadIdx.x; t < part; t += blockDim.x) {
        const uint32_t i = rank * part + t;                         // output index
        double2 v;
        if (CL == 2) v = ld_dsmem_d2(sbase + (__brev(i >> 1) >> (32 - lgp)) * 16, i & 1);
        else v = sv[__brev(i) >> (32 - lgp)];
        const double c0 = rint(sc * v.x), c1 = rint(sc * v.y);
        for (uint32_t l = 0; l < limbs; l++) {
            const uint64_t q = __ldg(&bl[l].q), one_p = __ldg(&bl[l].one_p);
            uint64_t *row = dst + ((size_t)l << logn);
            row[i] = encode_residue(c0, q, one_p, lc + l);
            row[i + S] = encode_residue(c1, q, one_p, lc + l);
        }
    }
    if (CL == 2) encode_cluster_sync();                            // no partner still reads this CTA's shared memory
}

// The per-call constants of the CRT step, passed by value (< 1 KB).
struct DecodeCall64 {
    uint32_t logn, limbs, L;
    int se;                               // scale = sm 2^se, sm in [0.5, 1)
    double sm;
    uint64_t hd[kBasisMaxLimbs];          // mixed-radix digits of h = (Q - 1) / 2 over q_0 .. q_(limbs-1)
};

// agx_decode64, step 1: residues [B][limbs][n] (coefficient form) -> m [B][n] doubles, one thread per coefficient.
// Garner in place over the limbs (d_t <- (d_t - d_j) q_j^-1 mod q_t for j < t, the running digits in shared memory,
// [limb][thread]), centring by comparing the digits with those of h from the top, the complement (Q - 1 - X) + 1 when X
// > h, then Horner in double from the top digit (rescaled by 2^-512 whenever the sum passes 2^512, so no intermediate
// overflows) and one division by the scale.  O(limbs^2) per coefficient.
__global__ void __launch_bounds__(kDecodeCrtThreads) decode64_crt_kernel(double *__restrict__ m,
                                                                         const uint64_t *__restrict__ in,
                                                                         const BasisLimb64 *__restrict__ bl,
                                                                         const BasisPair64 *__restrict__ pr,
                                                                         const __grid_constant__ DecodeCall64 cp,
                                                                         size_t total) {
    extern __shared__ uint64_t dg[];                                // [limbs][blockDim.x]
    const uint32_t logn = cp.logn, limbs = cp.limbs, T = blockDim.x;
    uint64_t *d = dg + threadIdx.x;
    for (size_t x = (size_t)blockIdx.x * T + threadIdx.x; x < total; x += (size_t)gridDim.x * T) {
        const size_t b = x >> logn, i = x & ((1u << logn) - 1);
        const uint64_t *src = in + ((b * limbs) << logn) + i;
        for (uint32_t t = 0; t < limbs; t++) {
            const uint64_t p = __ldg(&bl[t].q), big = __ldg(&bl[t].big);
            uint64_t v = src[(size_t)t << logn];
            const BasisPair64 *row = pr + (size_t)t * cp.L;
            for (uint32_t j = 0; j < t; j++)
                v = ref_shoup_u64(v + big - d[j * T], __ldg(&row[j].inv), __ldg(&row[j].inv_p), p);
            d[t * T] = ref_csub_u64(ref_csub_u64(v, p << 1), p);  // reduced input: v < q; else < 2q from the product
        }
        int cmp = 0;                                               // sign of X - h
        for (int t = (int)limbs - 1; t >= 0 && cmp == 0; t--) {
            const uint64_t v = d[t * T];
            cmp = v > cp.hd[t] ? 1 : (v < cp.hd[t] ? -1 : 0);
        }
        const bool neg = cmp > 0;
        if (neg) {                                                 // |X_c| = Q - X = (Q - 1 - X) + 1, digit by digit
            uint64_t carry = 1;
            for (uint32_t t = 0; t < limbs; t++) {
                const uint64_t p = __ldg(&bl[t].q);
                uint64_t v = p - 1 - d[t * T] + carry;
                carry = v == p;
                d[t * T] = carry ? 0 : v;
            }
        }
        double acc = 0.0, f = 1.0;                                 // |X_c| = acc 2^E, digits scaled by f = 2^-E
        int E = 0;
        for (int t = (int)limbs - 1; t >= 0; t--) {
            acc = acc * (double)__ldg(&bl[t].q) + (double)d[t * T] * f;
            if (acc >= 0x1p512) { acc *= 0x1p-512; f *= 0x1p-512; E += 512; }
        }
        const double r = ldexp(acc / cp.sm, E - cp.se);
        m[x] = neg ? -r : r;
    }
}

// agx_decode64, step 2: m [B][n] -> slots [B][S], the forward special FFT.  CL = 2 at n = 32768: CTA r loads the
// bit-reversed half r (the inputs i = 2 i' + r), runs the stages h = 1 .. S/4 locally, and the last stage (h = S/2)
// reads the partner's half through distributed shared memory; CTA r writes slots [r S/2, (r + 1) S/2).
template <int CL>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(512) decode64_fft_kernel(double2 *__restrict__ slots, const double *__restrict__ m,
                                                           const double2 *__restrict__ tw, uint32_t logn) {
    extern __shared__ __align__(16) double2 sv[];
    const uint32_t n = 1u << logn, S = n >> 1, part = S / CL, lgp = logn - 1 - (CL == 2 ? 1 : 0);
    const uint32_t rank = CL == 2 ? blockIdx.x & 1 : 0, poly = CL == 2 ? blockIdx.x >> 1 : blockIdx.x;
    const double *src = m + (size_t)poly * n;
    for (uint32_t t = threadIdx.x; t < part; t += blockDim.x) {
        const uint32_t i = CL == 2 ? 2 * t + rank : t;
        const uint32_t k = __brev(t) >> (32 - lgp);
        sv[k] = make_double2(src[i], src[i + S]);
    }
    __syncthreads();
    for (uint32_t h = 1; h < part; h <<= 1) {
        for (uint32_t b = threadIdx.x; b < part / 2; b += blockDim.x) {
            const uint32_t j = b & (h - 1), i = ((b - j) << 1) + j;
            const double2 u = sv[i], v = cmul(sv[i + h], tw[h + j]);
            sv[i] = cadd(u, v);
            sv[i + h] = csubd(u, v);
        }
        __syncthreads();
    }
    double2 *dst = slots + (size_t)poly * S;
    if (CL == 2) {
        encode_cluster_sync();                                     // both halves are through their local stages
        const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(sv), h = S >> 1;
        for (uint32_t k = threadIdx.x; k < part; k += blockDim.x) {
            const double2 a = rank == 0 ? sv[k] : ld_dsmem_d2(sbase + k * 16, 0);
            const double2 b = rank == 0 ? ld_dsmem_d2(sbase + k * 16, 1) : sv[k];
            const double2 v = cmul(b, tw[h + k]);
            dst[rank * h + k] = rank == 0 ? cadd(a, v) : csubd(a, v);
        }
        encode_cluster_sync();                                     // no partner still reads this CTA's shared memory
    } else {
        for (uint32_t k = threadIdx.x; k < part; k += blockDim.x) dst[k] = sv[k];
    }
}

}  // namespace agx
