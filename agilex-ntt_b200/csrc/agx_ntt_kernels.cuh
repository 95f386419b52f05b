// agx_ntt_kernels.cuh -- register-resident two-pass negacyclic NTT kernels for sm_100a.
//
// Replaces the reference's loader + compute + drain single_tasks (ntt_input_kernel ntt.cpp:508-607,
// fwd_ntt_kernel ntt.cpp:86-506, ntt_output_kernel ntt.cpp:610-640) with ONE kernel per direction: a CTA of
// TPP = n/E threads owns one polynomial (one (batch, limb) row of the [B][L][n] array), each thread keeps
// E = 2^LE coefficients in registers and the log2(n) butterfly stages run as two register-resident passes with
// a single shared-memory transpose between them:
//
//   forward  pass A: thread t holds x[t + TPP*k]   -> stages 0..LE-1     (twiddles identical for all threads)
//            transpose through a padded smem image (STS.32 columns -> LDS.128 rows, both conflict-free)
//            pass B: thread T holds x[E*T .. E*T+E) -> stages LE..logn-1 (per-thread twiddles, coalesced 16-B loads
//                                                      from a table stored in kernel order)
//            final reduction to [0,q); rows into hardware-swizzled smem tiles, written back by TMA tensor stores
//            (or, without a tensor-map encoder, staged through the padded image and coalesced 16-B stores).
//   inverse  is the mirror image (Gentleman-Sande), n^-1 folded into the twiddles of the last four stages (kInvFold).
//   polymul  n = 1024: forward(a), parked in smem, forward(b), pointwise Barrett, inverse -- one launch;
//            n >= 2048: three launches (NTT(a); NTT(b) .* it; INTT), see agx_api.cu.
// Also here: the generic any-n kernel, the limb-wise element-wise ops, the bit-reversal adapter, the reference-shaped
// u64 pass kernels, the device-side table generator, synthetic data and checksum.
//
// The FPGA's X/X2/Xm double-buffer and reorder muxes (ntt.cpp:90-98, 160-289, 397-496) exist to dodge BRAM port
// conflicts and have no arithmetic effect (SURVEY.md s.0); they have no counterpart here.
//
// Twiddle table (per limb, per direction) `tw[n]` of (w, w') pairs:
//   entries [1, E)      : natural order, entry k = psi^bitrev(k)  (ntt.cpp:298-300 indexing, roots[m + i])
//   entries [2^s, 2^s+1): for stages s >= LE the 2^s entries of the stage are permuted so that thread T's
//                         c = 2^(s-LT) twiddles are reached by coalesced loads:
//                         natural 2^s + T*c + kk  ->  2^s + ((kk>>1)*TPP + T)*2 + (kk&1)   (c >= 2)
//   inverse table: entry 0 = (n^-1, .), entry 1 = (psi^-bitrev(1) * n^-1, .)
#pragma once
#include <cuda.h>   // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "agx_arith.cuh"

namespace agx {

struct KParams {
    const uint2 *tw_fwd;     // [L][n] kernel order
    const uint2 *tw_inv;     // [L][n] kernel order
    const uint2 *twc_fwd;    // [L][n] column-pass copy: stage j < LE twiddles at the offsets the row pass uses
    const uint2 *twc_inv;
    const LimbConst *lc;     // [L]
    uint32_t L;
    LimbConst c0;                // limb 0's constants by value: kernel parameters live in the constant bank, so the
                                 // butterfly's q / 2q / -q / -2q / 0 operands cost no register-file read when L == 1
};

// Per-limb constants of a polynomial: kernels instantiated with CL = true (single-limb batches) read them from the
// parameter block, i.e. as constant-bank operands; CL = false loads the limb's entry of the table in global memory.
#define AGX_LIMB_CONSTS(CL, p, limb)            \
    LimbConst limb_consts_;                     \
    if constexpr (!(CL)) limb_consts_ = (p).lc[limb]; \
    const LimbConst &c = (CL) ? (p).c0 : limb_consts_

template <int LOGN, int LE>
struct Geo {
    static constexpr int N = 1 << LOGN;
    static constexpr int E = 1 << LE;            // coefficients per thread
    static constexpr int LT = LOGN - LE;
    static constexpr int TPP = 1 << LT;          // threads per polynomial
    static constexpr int CPR = E / 4;            // 16-byte chunks of data per smem row
    static constexpr int PITCH4 = CPR + 1;       // row pitch in 16-byte chunks: one chunk of padding per row
    static constexpr int PITCH = 4 * PITCH4;     // ... in words
    static constexpr int SMEM_CHUNKS = TPP * PITCH4;
    static_assert(LT >= 5 && LT <= LE, "need 32 <= TPP <= E");
};

// kernel-order position of the twiddle for (stage s >= LE, thread T, local index kk)
template <int LOGN, int LE>
__host__ __device__ constexpr uint32_t tw_pos(int s, uint32_t T, uint32_t kk) {
    constexpr int LT = LOGN - LE;
    constexpr uint32_t TPP = 1u << LT;
    const uint32_t c = 1u << (s - LT);
    return c == 1 ? (1u << s) + T : (1u << s) + ((kk >> 1) * TPP + T) * 2 + (kk & 1);
}

// L2 prefetch of the polynomial a CTA slot will work on about half a wave later.  The CTA that owns it then finds its 16 KB in
// L2 (~250 clk) instead of paying a loaded-HBM round trip (~1.8 us measured as the load wait in the phase trace).
#ifndef AGX_PREFETCH_DIST
#define AGX_PREFETCH_DIST (4 * 148)   // half a wave of n = 4096 CTAs ahead: 0.3-0.4 % better than a full wave in two A/B runs
#endif
template <int LOGN, int TPP>
__device__ __forceinline__ void prefetch_ahead(const uint32_t *g_this, uint32_t poly, uint32_t T, uint32_t tid) {
    constexpr int LINES = (4 << LOGN) / 128;                 // 128-byte lines per polynomial
    if (AGX_PREFETCH_DIST > 0 && poly + AGX_PREFETCH_DIST < T) {
        const char *nxt = reinterpret_cast<const char *>(g_this) + (size_t)AGX_PREFETCH_DIST * (4u << LOGN);
#pragma unroll
        for (int i = 0; i < (LINES + TPP - 1) / TPP; i++)
            if (i * TPP + tid < LINES) asm volatile("prefetch.global.L2 [%0];" ::"l"(nxt + (size_t)(i * TPP + tid) * 128));
    }
}


// Streaming accesses to the polynomial rows: read once / written once per launch, so they must not displace the
// twiddle table from L1 (AGX_STREAM_POLICY 0: ld/st.global.cs; 1: L1::no_allocate loads; experiments in profiles/).
#ifndef AGX_STREAM_POLICY
#define AGX_STREAM_POLICY 0
#endif
__device__ __forceinline__ uint32_t ld_stream(const uint32_t *p) {
#if AGX_STREAM_POLICY == 1
    uint32_t v;
    asm volatile("ld.global.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
#else
    return __ldcs(p);
#endif
}
__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
#if AGX_STREAM_POLICY == 1
    uint4 v;
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
#else
    return __ldcs(p);
#endif
}
// Result stores (AGX_STORE_POLICY 0: st.global.cs streaming; 1: default write-back; 2: .cg; 3: .wt; experiments in profiles/)
#ifndef AGX_STORE_POLICY
#define AGX_STORE_POLICY 0
#endif
template <typename V>
__device__ __forceinline__ void st_stream(V *p, V v) {
#if AGX_STORE_POLICY == 1
    *p = v;
#elif AGX_STORE_POLICY == 2
    __stcg(p, v);
#elif AGX_STORE_POLICY == 3
    __stwt(p, v);
#else
    __stcs(p, v);
#endif
}
__device__ __forceinline__ uint2 ld_twiddle(const uint2 *p) {
#if AGX_STREAM_POLICY == 1
    uint2 v;
    asm volatile("ld.global.nc.L1::evict_last.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
#else
    return __ldg(p);
#endif
}
__device__ __forceinline__ uint4 ld_twiddle(const uint4 *p) {
#if AGX_STREAM_POLICY == 1
    uint4 v;
    asm volatile("ld.global.nc.L1::evict_last.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
#else
    return __ldg(p);
#endif
}

template <int TPP>
__device__ __forceinline__ void poly_sync() {
    if constexpr (TPP == 32) __syncwarp(); else __syncthreads();
}

// ---------------------------------------------------------------------------------------------- smem transposes

// Shared-memory image of one polynomial: TPP rows of E words, each row padded by 16 bytes (pitch 4E+16 bytes).
// With that pitch every access pattern of the kernels is conflict-free AND a compile-time offset from a per-thread
// base, so no address arithmetic is left in the unrolled code:
//   columns (STS.32/LDS.32): element tid + TPP*k -> row*PITCH + col, lanes on consecutive words;
//   rows (LDS.128/STS.128):  thread T, chunk c -> T*PITCH4 + c; eight consecutive T start 16 bytes apart mod 128;
//   copy in/out (LDS.128/STS.128): chunk index i*TPP + tid -> consecutive chunks of one row per quarter-warp.
// (An earlier XOR swizzle was also conflict-free but cost one LOP3 per access.)
template <int LOGN, int LE>
__device__ __forceinline__ constexpr uint32_t col_off(int k) {
    using G = Geo<LOGN, LE>;
    const int ebase = G::TPP * k;
    return (ebase >> LE) * G::PITCH + (ebase & (G::E - 1));
}

template <int LOGN, int LE>
__device__ __forceinline__ void sts_columns(uint32_t *sw, const uint32_t (&x)[1 << LE], uint32_t tid) {
#pragma unroll
    for (int k = 0; k < (1 << LE); k++) sw[tid + col_off<LOGN, LE>(k)] = x[k];
}

template <int LOGN, int LE>
__device__ __forceinline__ void lds_columns(const uint32_t *sw, uint32_t (&x)[1 << LE], uint32_t tid) {
#pragma unroll
    for (int k = 0; k < (1 << LE); k++) x[k] = sw[tid + col_off<LOGN, LE>(k)];
}

template <int LOGN, int LE>
__device__ __forceinline__ void lds_row(const uint4 *sm, uint32_t (&x)[1 << LE], uint32_t tid) {
    using G = Geo<LOGN, LE>;
    const uint4 *r = sm + tid * G::PITCH4;
#pragma unroll
    for (int c = 0; c < G::CPR; c++) {
        const uint4 v = r[c];
        x[4 * c + 0] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
    }
}

template <int LOGN, int LE>
__device__ __forceinline__ void sts_row(uint4 *sm, const uint32_t (&x)[1 << LE], uint32_t tid) {
    using G = Geo<LOGN, LE>;
    uint4 *r = sm + tid * G::PITCH4;
#pragma unroll
    for (int c = 0; c < G::CPR; c++) r[c] = make_uint4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
}

// coalesced 16-byte copies between the padded smem image and the polynomial's row in global memory
template <int LOGN, int LE>
__device__ __forceinline__ void smem_to_global(const uint4 *sm, uint32_t *g, uint32_t tid) {
    using G = Geo<LOGN, LE>;
    uint4 *g4 = reinterpret_cast<uint4 *>(g) + tid;
    const uint4 *s = sm + (tid / G::CPR) * G::PITCH4 + (tid % G::CPR);
#pragma unroll
    for (int i = 0; i < G::N / 4 / G::TPP; i++)      // chunk i*TPP + tid: row advances by TPP/CPR per step
        st_stream(g4 + i * G::TPP, s[i * (G::TPP / G::CPR) * G::PITCH4]);
}

template <int LOGN, int LE>
__device__ __forceinline__ void global_to_smem(uint4 *sm, const uint32_t *g, uint32_t tid) {
    using G = Geo<LOGN, LE>;
    const uint4 *g4 = reinterpret_cast<const uint4 *>(g) + tid;
    uint4 *s = sm + (tid / G::CPR) * G::PITCH4 + (tid % G::CPR);
    uint4 v[G::N / 4 / G::TPP];
#pragma unroll
    for (int i = 0; i < G::N / 4 / G::TPP; i++) v[i] = ld_stream(g4 + i * G::TPP);
#pragma unroll
    for (int i = 0; i < G::N / 4 / G::TPP; i++) s[i * (G::TPP / G::CPR) * G::PITCH4] = v[i];
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Inverse-kernel input.  Shipped (AGX_INV_INPUT = 3): cp.async (LDGSTS.128: L2 -> shared memory without passing registers
// or allocating in L1), and each warp stages exactly the rows its own threads will read (warp w: rows 32w .. 32w+31,
// 8 KB contiguous in global memory), so a __syncwarp replaces the CTA barrier: inverse 0.4983 -> 0.4943 ms in one call
// (profiles/r02_experiments.md).  A/B values: 0 = LDG.128 -> registers -> STS.128 (global_to_smem above) + CTA barrier
// (round 1), 1 = cp.async + CTA barrier (0.4979-0.4983), 2 = warp-local rows with LDG/STS (0.5011).
#ifndef AGX_INV_INPUT
#define AGX_INV_INPUT 3
#endif
template <int LOGN, int LE>
__device__ __forceinline__ void inv_stage_input(uint4 *sm, const uint32_t *g, uint32_t tid) {
    using G = Geo<LOGN, LE>;
    constexpr int NCH = G::N / 4 / G::TPP;               // 16-byte chunks per thread
    constexpr bool WARP_LOCAL = (AGX_INV_INPUT & 2) != 0 && G::TPP > 32;
    constexpr bool ASYNC = (AGX_INV_INPUT & 1) != 0;
    // thread's chunk i is polynomial chunk c0 + i*STEP (row c / CPR, column c % CPR of the image); STEP is a multiple of
    // CPR, so source and destination are a per-thread base plus a compile-time offset
    constexpr int STEP = WARP_LOCAL ? 32 : G::TPP;
    static_assert(STEP % G::CPR == 0, "a step must cover whole image rows");
    const uint32_t c0 = WARP_LOCAL ? (tid >> 5) * (32 * NCH) + (tid & 31) : tid;
    const uint4 *src = reinterpret_cast<const uint4 *>(g) + c0;
    uint4 *dst = sm + (c0 / G::CPR) * G::PITCH4 + (c0 % G::CPR);
    if constexpr (ASYNC) {
        const uint32_t d32 = smem_u32(dst);
#pragma unroll
        for (int i = 0; i < NCH; i++)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d32 + i * (STEP / G::CPR) * G::PITCH4 * 16), "l"(src + i * STEP)
                         : "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
    } else {
        uint4 v[NCH];
#pragma unroll
        for (int i = 0; i < NCH; i++) v[i] = ld_stream(src + i * STEP);
#pragma unroll
        for (int i = 0; i < NCH; i++) dst[i * (STEP / G::CPR) * G::PITCH4] = v[i];
    }
    if constexpr (WARP_LOCAL) __syncwarp(); else poly_sync<G::TPP>();
}

// ---------------------------------------------------------------------------------- results by TMA tensor store
// Forward results leave the SM as E/32 asynchronous tensor stores issued by ONE thread instead of 16 x (LDS.128 +
// STG.128) per thread.  Every thread writes its row into DENSE shared-memory tiles -- one per 32-word half of the rows,
// TPP rows x 128 bytes each -- in the TMA engine's 128-byte swizzle (16-byte chunk index XOR (row & 7): conflict-free
// STS.128 at a pitch of 128 bytes); after a proxy fence and a barrier one thread issues cp.async.bulk.tensor (3-D map
// over the destination batch: {32 words, E/32 halves, T*TPP rows}, box {32, 1, TPP}) and waits only until the tiles have
// been READ.  The tiles must start on a 1024-byte boundary (the swizzle is a function of address bits 7..9).
// Measured and not kept (profiles/r01_experiments.md): the same tiles for the transpose as well, tensor LOADS for the
// inverse kernel's input, tensor stores for its output.

__device__ __forceinline__ void mbar_init(uint64_t *b, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *b, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "AGX_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra AGX_DONE;\n"
        "bra AGX_WAIT;\n"
        "AGX_DONE:\n"
        "}" ::"r"(smem_u32(b)), "r"(parity) : "memory");
}

template <int LOGN, int LE>
struct Swz {
    using G = Geo<LOGN, LE>;
    static constexpr int HALVES = G::E / 32;
    static constexpr int HALF_BYTES = G::TPP * 128;
    static constexpr int HALF_WORDS = G::TPP * 32;
    static constexpr int BYTES = HALVES * HALF_BYTES;    // = 4n
};

template <int LOGN, int LE>
__device__ __forceinline__ void sts_row_swz(uint4 *sm, const uint32_t (&x)[1 << LE], uint32_t tid) {
    using S = Swz<LOGN, LE>;
    char *base = reinterpret_cast<char *>(sm) + tid * 128;
    const uint32_t swz = (tid & 7) << 4;
#pragma unroll
    for (int cc = 0; cc < 8; cc++) {
        char *at = base + ((cc << 4) ^ swz);
#pragma unroll
        for (int h = 0; h < S::HALVES; h++) {
            const int j = 4 * (8 * h + cc);
            *reinterpret_cast<uint4 *>(at + h * S::HALF_BYTES) = make_uint4(x[j], x[j + 1], x[j + 2], x[j + 3]);
        }
    }
}

// one thread: the CTA's polynomial, shared-memory tiles -> global, asynchronously; returns when the tiles have been read
template <int LOGN, int LE>
__device__ __forceinline__ void tma_store_poly(const uint4 *sm, const CUtensorMap *map, uint32_t poly) {
    using G = Geo<LOGN, LE>;
    using S = Swz<LOGN, LE>;
#pragma unroll
    for (int h = 0; h < S::HALVES; h++)
        asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map),
                     "r"(smem_u32(reinterpret_cast<const char *>(sm) + h * S::HALF_BYTES)), "r"(0), "r"(h), "r"(poly * G::TPP)
                     : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory must outlive the engine's reads
}

// minimum resident CTAs per SM requested from ptxas (sets the register cap): 64 coefficients/thread -> 512 threads
// per SM (128 registers each), 32 coefficients/thread -> 768 threads (85 registers).
#ifndef AGX_THREADS_E64
#define AGX_THREADS_E64 512
#endif
#ifndef AGX_MINB
#define AGX_MINB(LOGN, LE) ((1 << (LE)) >= 64 ? (AGX_THREADS_E64 >> ((LOGN) - (LE))) : (768 >> ((LOGN) - (LE))))
#endif
// A/B knob: an explicit register cap for the 64-coefficient kernels instead of a minimum CTA count
// (-DAGX_MAXNREG_E64=112 -> 9 CTAs of 64 threads per SM)
#ifdef AGX_MAXNREG_E64
#define AGX_KERNEL_BOUNDS(LOGN, LE) __launch_bounds__(1 << ((LOGN) - (LE))) __maxnreg__((1 << (LE)) >= 64 ? AGX_MAXNREG_E64 : 80)
#else
#define AGX_KERNEL_BOUNDS(LOGN, LE) __launch_bounds__(1 << ((LOGN) - (LE)), AGX_MINB(LOGN, LE))
#endif

// ------------------------------------------------------------------------------ looped two-pass kernels
// The fully unrolled passes above are ~47 KB of SASS per kernel; with 16 warps per SM each at a different point
// of that straight-line code the instruction caches thrash (ncu: stall_no_instruction 2.7 per issue, the top
// stall).  Both passes of a transform apply the SAME register pairing pattern to x[0..E): stage j pairs
// x[k] with x[k + (E/2 >> j)].  Only the twiddle addressing differs, and that is affine in three per-pass
// values (sbase, tstride, toff).  So the kernels below run ONE copy of the stage code inside a 2-trip loop,
// which halves the code footprint and lets it stay resident in the SM's instruction cache.
//   pass over columns (uniform twiddles): sbase = 0,  tstride = 1,   toff = 0
//   pass over rows (per-thread twiddles): sbase = LT, tstride = TPP, toff = tid
//   twiddle (local stage j >= 1, group g) lives at uint4 index (1 << (sbase+j-1)) + (g>>1)*tstride + toff,
//   twiddle (j = 0) at uint2 index (1 << sbase) + toff.
// When LT < LE (n = 2048) the row pass has only LE-1... LT stages: local stage 0 is skipped there (j0 = LE-LT).

// Per-pass twiddle base pointers.  Every twiddle load of the shared stage code is `base + compile-time offset`:
//   row pass   : table = tw (kernel order), b4 = (uint4*)tw + tid,  b2 = tw + (1<<LT) + tid
//   column pass: table = twc (the same offsets, populated only where a thread with tid = 0 would look), b4, b2 alike
// so the loop body contains no address arithmetic (an earlier version computed base + h*stride at run time, which
// ptxas turned into IMAD.WIDE -- on the pipe this kernel is bound by).
struct PassAddr {
    const uint4 *b4;
    const uint2 *b2;
    const uint4 *b4b;    // inverse only: the "already scaled" twiddle variant (see kInvFold); == b4 in the row pass
};

template <int LOGN, int LE>
__device__ __forceinline__ PassAddr pass_addr(const uint2 *__restrict__ table, uint32_t toff, uint32_t variant_b = 0u) {
    const uint4 *b4 = reinterpret_cast<const uint4 *>(table) + toff;
    return PassAddr{b4, table + (1u << (LOGN - LE)) + toff, b4 + variant_b};
}

// Inverse transform, where n^-1 goes.  Every stage multiplies only its difference outputs, so n^-1 cannot ride on one
// stage's twiddles alone.  It is folded into the column pass (the last LE stages) like this: local stage kInvFold
// stores ALL its twiddles pre-multiplied by n^-1, which scales every coefficient whose register index has bit
// half(kInvFold) set.  In the later stages J < kInvFold a pair whose index has any of the bits half(J+1..kInvFold) set
// is already scaled and takes the unscaled twiddle (variant B, stored one 16-byte slot after variant A in the column
// table); a pair with none of them set is still unscaled: its sum stays so, its difference takes the scaled twiddle
// (variant A).  Only the E / 2^(kInvFold+1) last-stage pairs that were sums all the way need the two explicit scaling
// multiplies.  The row pass runs the same stage code with b4b == b4 (both variants are the plain twiddle).
#ifndef AGX_INV_FOLD
#define AGX_INV_FOLD 3
#endif
constexpr int kInvFold = AGX_INV_FOLD;
template <int LE>
__host__ __device__ constexpr int inv_fold_mask(int J) {   // index bits that mark a pair as already scaled at local stage J
    int m = 0;
    for (int jj = J + 1; jj <= kInvFold; jj++) m += (1 << LE) >> (jj + 1);
    return J < kInvFold ? m : 0;
}

// AGX_TW_INTERLEAVE: the two twiddles of a 16-byte table slot are stored word-interleaved, (w0, w1, w0', w1') instead of
// (w0, w0', w1, w1').  A 16-byte load fills four consecutive registers, and the register file has two banks by register
// parity: with (w, w') in an even/odd pair one of the butterfly's two multiplies y*w, hi(y*w') always reads both of its
// operands from y's bank; interleaved, both words of a twiddle share a parity and ptxas can keep y in the other bank.
#ifndef AGX_TW_INTERLEAVE
#define AGX_TW_INTERLEAVE 1
#endif
template <int LOGN, int LE, int J>
__device__ __forceinline__ void load_tw_generic(uint2 (&w)[1 << J], const PassAddr &a) {
    constexpr int LT = LOGN - LE, TPP = 1 << LT;
    if constexpr (J == 0) {
        w[0] = ld_twiddle(a.b2);
    } else {
#pragma unroll
        for (int h = 0; h < (1 << (J - 1)); h++) {
            const uint4 v = ld_twiddle(a.b4 + ((1 << (LT + J - 1)) + h * TPP));
#if AGX_TW_INTERLEAVE
            w[2 * h] = make_uint2(v.x, v.z);
            w[2 * h + 1] = make_uint2(v.y, v.w);
#else
            w[2 * h] = make_uint2(v.x, v.y);
            w[2 * h + 1] = make_uint2(v.z, v.w);
#endif
        }
    }
}

template <int LOGN, int LE, int J>
__device__ __forceinline__ void ct_stage(uint32_t (&x)[1 << LE], const PassAddr &a, const LimbConst &c) {
    constexpr int half = (1 << LE) >> (J + 1);
    uint2 w[1 << J];
    load_tw_generic<LOGN, LE, J>(w, a);
#pragma unroll
    for (int g = 0; g < (1 << J); g++)
#pragma unroll
        for (int i = 0; i < half; i++) ct_bfly(x[g * 2 * half + i], x[g * 2 * half + i + half], w[g], c);
}

template <int LOGN, int LE, int J>
__device__ __forceinline__ void gs_stage(uint32_t (&x)[1 << LE], const PassAddr &a, const LimbConst &c) {
    constexpr int half = (1 << LE) >> (J + 1);
    constexpr int mask = J >= 1 ? inv_fold_mask<LE>(J) : 0;
    uint2 w[1 << J];
    load_tw_generic<LOGN, LE, J>(w, a);
    if constexpr (mask != 0) {
        uint2 wb[1 << J];
        PassAddr ab = a;
        ab.b4 = a.b4b;
        load_tw_generic<LOGN, LE, J>(wb, ab);
#pragma unroll
        for (int g = 0; g < (1 << J); g++)
#pragma unroll
            for (int i = 0; i < half; i++)
                gs_bfly(x[g * 2 * half + i], x[g * 2 * half + i + half], (i & mask) ? wb[g] : w[g], c);
    } else {
#pragma unroll
        for (int g = 0; g < (1 << J); g++)
#pragma unroll
            for (int i = 0; i < half; i++) gs_bfly(x[g * 2 * half + i], x[g * 2 * half + i + half], w[g], c);
    }
}

template <int LOGN, int LE, int J>
__device__ __forceinline__ void ct_stages_from(uint32_t (&x)[1 << LE], const PassAddr &a, const LimbConst &c) {
    ct_stage<LOGN, LE, J>(x, a, c);
    if constexpr (J + 1 < LE) ct_stages_from<LOGN, LE, J + 1>(x, a, c);
}

template <int LOGN, int LE, int J>
__device__ __forceinline__ void gs_stages_down_to1(uint32_t (&x)[1 << LE], const PassAddr &a, const LimbConst &c) {
    gs_stage<LOGN, LE, J>(x, a, c);
    if constexpr (J > 1) gs_stages_down_to1<LOGN, LE, J - 1>(x, a, c);
}

// Last inverse stage (global stage 0).  With the n^-1 folding described at kInvFold only the pairs whose index has none
// of the fold bits set are still unscaled and take the two scaling multiplies (tw[0] = (n^-1, .), tw[1] =
// (iroot1 * n^-1, .)); all others arrive scaled and take the plain butterfly with the unscaled twiddle twc[TPP] = iroot1.
// Saves (E/2)(1 - 2^-kInvFold) Shoup multiplies per thread against scaling every last-stage pair.
template <int LOGN, int LE>
__device__ __forceinline__ void inv_last_stage(uint32_t (&x)[1 << LE], const uint2 *__restrict__ tw,
                                               const uint2 *__restrict__ twc, const LimbConst &c) {
    using G = Geo<LOGN, LE>;
    const uint2 wn = __ldg(tw), w1n = __ldg(tw + 1), w1 = __ldg(twc + G::TPP);
    constexpr int mask = inv_fold_mask<LE>(0);
#pragma unroll
    for (int j = 0; j < G::E / 2; j++) {
        if ((j & mask) == 0) gs_bfly_last(x[j], x[j + G::E / 2], wn, w1n, c);
        else gs_bfly_last_prescaled(x[j], x[j + G::E / 2], w1, c);
    }
}

// dst may equal src (in place: agx_ntt_fwd).  MUL: the three-launch polynomial product's middle step -- the spectrum
// is multiplied pointwise by `mul` (the other operand's spectrum, same layout; may equal dst) before it is stored,
// and left in [0,2q), which is what the inverse kernel accepts.
// TMA: results leave through tma_store_rows (dst is then described by `tmap`); otherwise through the padded staging
// image and coalesced 16-byte stores.
template <int LOGN, int LE, bool MUL, bool CL, bool TMA = false>
__global__ void AGX_KERNEL_BOUNDS(LOGN, LE)
ntt_fwd_loop_kernel(uint32_t *dst, const uint32_t *src, const uint32_t *mul, KParams p, uint32_t T,
                    const __grid_constant__ CUtensorMap tmap) {
    using G = Geo<LOGN, LE>;
    __shared__ __align__(1024) uint4 sm[G::SMEM_CHUNKS];
    const uint32_t tid = threadIdx.x;
    const uint32_t poly = blockIdx.x;
    const uint32_t limb = p.L == 1 ? 0 : poly % p.L;
    AGX_LIMB_CONSTS(CL, p, limb);
    const uint2 *tw = p.tw_fwd + (size_t)limb * G::N;
    const uint2 *twc = p.twc_fwd + (size_t)limb * G::N;
    const uint32_t *gs = src + (size_t)poly * G::N;
    uint32_t *g = dst + (size_t)poly * G::N;

    uint32_t x[G::E];
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
        PassAddr a;
        if (pass == 0) {                             // column pass: x[k] = poly[tid + TPP*k], stages 0..LE-1
            a = pass_addr<LOGN, LE>(twc, 0u);
#pragma unroll
            for (int k = 0; k < G::E; k++) x[k] = ld_stream(gs + tid + G::TPP * k);
            prefetch_ahead<LOGN, G::TPP>(gs, poly, T, tid);
        } else {                                     // row pass: x[j] = poly[E*tid + j], stages LE..logn-1
            a = pass_addr<LOGN, LE>(tw, tid);
            lds_row<LOGN, LE>(sm, x, tid);
        }
        if (G::LT == LE || pass == 0) ct_stage<LOGN, LE, 0>(x, a, c);
        ct_stages_from<LOGN, LE, 1>(x, a, c);
        if (pass == 0) {
            sts_columns<LOGN, LE>(reinterpret_cast<uint32_t *>(sm), x, tid);
            poly_sync<G::TPP>();
        }
    }
#pragma unroll
    for (int j = 0; j < G::E; j++) x[j] = reduce4q(x[j], c);
    if constexpr (MUL) {
        poly_sync<G::TPP>();                         // every thread has read its row of the transpose buffer
        global_to_smem<LOGN, LE>(sm, mul + (size_t)poly * G::N, tid);
        poly_sync<G::TPP>();
#pragma unroll
        for (int cc = 0; cc < G::CPR; cc++) {
            const uint4 mv = sm[tid * G::PITCH4 + cc];
            x[4 * cc + 0] = csub(barrett_mul_lazy(mv.x, x[4 * cc + 0], c), c.neg2q);
            x[4 * cc + 1] = csub(barrett_mul_lazy(mv.y, x[4 * cc + 1], c), c.neg2q);
            x[4 * cc + 2] = csub(barrett_mul_lazy(mv.z, x[4 * cc + 2], c), c.neg2q);
            x[4 * cc + 3] = csub(barrett_mul_lazy(mv.w, x[4 * cc + 3], c), c.neg2q);
        }
    }
    if constexpr (TMA) {
        poly_sync<G::TPP>();                         // the dense tiles overlap other threads' rows of the padded image
        sts_row_swz<LOGN, LE>(sm, x, tid);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the TMA engine
        poly_sync<G::TPP>();
        if (tid == 0) tma_store_poly<LOGN, LE>(sm, &tmap, poly);
    } else {
        sts_row<LOGN, LE>(sm, x, tid);               // own row only: no barrier needed before
        poly_sync<G::TPP>();
        smem_to_global<LOGN, LE>(sm, g, tid);
    }
}

template <int LOGN, int LE, bool CL>
__global__ void AGX_KERNEL_BOUNDS(LOGN, LE)
ntt_inv_loop_kernel(uint32_t *__restrict__ data, KParams p, uint32_t T) {
    using G = Geo<LOGN, LE>;
    __shared__ uint4 sm[G::SMEM_CHUNKS];
    const uint32_t tid = threadIdx.x;
    const uint32_t poly = blockIdx.x;
    const uint32_t limb = p.L == 1 ? 0 : poly % p.L;
    AGX_LIMB_CONSTS(CL, p, limb);
    const uint2 *tw = p.tw_inv + (size_t)limb * G::N;
    const uint2 *twc = p.twc_inv + (size_t)limb * G::N;
    uint32_t *g = data + (size_t)poly * G::N;

    uint32_t x[G::E];
#if AGX_INV_INPUT == 0
    global_to_smem<LOGN, LE>(sm, g, tid);
    prefetch_ahead<LOGN, G::TPP>(g, poly, T, tid);
    poly_sync<G::TPP>();
#else
    prefetch_ahead<LOGN, G::TPP>(g, poly, T, tid);
    inv_stage_input<LOGN, LE>(sm, g, tid);
#endif
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
        PassAddr a;
        if (pass == 0) {                             // row pass: stages logn-1 .. LE
            a = pass_addr<LOGN, LE>(tw, tid);
            lds_row<LOGN, LE>(sm, x, tid);
        } else {                                     // column pass: stages LE-1 .. 1 (stage 0 below)
            a = pass_addr<LOGN, LE>(twc, 0u, 1u);
            lds_columns<LOGN, LE>(reinterpret_cast<const uint32_t *>(sm), x, tid);
        }
        gs_stages_down_to1<LOGN, LE, LE - 1>(x, a, c);
        if (pass == 0) {
            if (G::LT == LE) gs_stage<LOGN, LE, 0>(x, a, c);
            sts_row<LOGN, LE>(sm, x, tid);
            poly_sync<G::TPP>();
        }
    }
    inv_last_stage<LOGN, LE>(x, tw, twc, c);
#pragma unroll
    for (int k = 0; k < G::E; k++) st_stream(g + tid + G::TPP * k, x[k]);
}

// Fused negacyclic product c = a * b mod (X^n + 1, q): forward(a), forward(b), pointwise, inverse in ONE launch
// (BASELINE.json config 4).  The forward stage code runs 4 times (2 operands x 2 passes) and the inverse stage code
// twice, each from a single copy; NTT(a) waits in a second shared-memory buffer (own row per thread) while b is
// transformed.  HBM traffic: 3 * n * 4 bytes per product.
template <int LOGN, int LE, bool CL>
__global__ void __launch_bounds__(1 << (LOGN - LE), AGX_MINB(LOGN, LE))
polymul_loop_kernel(uint32_t *out, const uint32_t *a, const uint32_t *b, KParams p) {   // out may alias a and/or b
    using G = Geo<LOGN, LE>;
    __shared__ uint4 sm[G::SMEM_CHUNKS];
    __shared__ uint4 park[G::SMEM_CHUNKS];
    const uint32_t tid = threadIdx.x;
    const uint32_t poly = blockIdx.x;
    const uint32_t limb = p.L == 1 ? 0 : poly % p.L;
    AGX_LIMB_CONSTS(CL, p, limb);
    const uint2 *twf = p.tw_fwd + (size_t)limb * G::N, *twfc = p.twc_fwd + (size_t)limb * G::N;
    const uint2 *twi = p.tw_inv + (size_t)limb * G::N, *twic = p.twc_inv + (size_t)limb * G::N;
    const size_t off = (size_t)poly * G::N;

    uint32_t x[G::E];
#pragma unroll 1
    for (int opnd = 0; opnd < 2; opnd++) {
        const uint32_t *src = (opnd == 0 ? a : b) + off;
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {
            PassAddr ad;
            if (pass == 0) {
                ad = pass_addr<LOGN, LE>(twfc, 0u);
#pragma unroll
                for (int k = 0; k < G::E; k++) x[k] = ld_stream(src + tid + G::TPP * k);
            } else {
                ad = pass_addr<LOGN, LE>(twf, tid);
                lds_row<LOGN, LE>(sm, x, tid);
            }
            if (G::LT == LE || pass == 0) ct_stage<LOGN, LE, 0>(x, ad, c);
            ct_stages_from<LOGN, LE, 1>(x, ad, c);
            if (pass == 0) {
                poly_sync<G::TPP>();                 // all rows of the previous operand have been read
                sts_columns<LOGN, LE>(reinterpret_cast<uint32_t *>(sm), x, tid);
                poly_sync<G::TPP>();
            }
        }
#pragma unroll
        for (int j = 0; j < G::E; j++) x[j] = reduce4q(x[j], c);
        if (opnd == 0) sts_row<LOGN, LE>(park, x, tid);   // NTT(a): written and later read by this thread only
    }
#pragma unroll
    for (int cc = 0; cc < G::CPR; cc++) {            // pointwise: NTT(a) .* NTT(b), lazily reduced to [0,2q)
        const uint4 av = park[tid * G::PITCH4 + cc];
        x[4 * cc + 0] = csub(barrett_mul_lazy(av.x, x[4 * cc + 0], c), c.neg2q);
        x[4 * cc + 1] = csub(barrett_mul_lazy(av.y, x[4 * cc + 1], c), c.neg2q);
        x[4 * cc + 2] = csub(barrett_mul_lazy(av.z, x[4 * cc + 2], c), c.neg2q);
        x[4 * cc + 3] = csub(barrett_mul_lazy(av.w, x[4 * cc + 3], c), c.neg2q);
    }
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
        PassAddr ad;
        if (pass == 0) {
            ad = pass_addr<LOGN, LE>(twi, tid);
        } else {
            ad = pass_addr<LOGN, LE>(twic, 0u, 1u);
            lds_columns<LOGN, LE>(reinterpret_cast<const uint32_t *>(sm), x, tid);
        }
        gs_stages_down_to1<LOGN, LE, LE - 1>(x, ad, c);
        if (pass == 0) {
            if (G::LT == LE) gs_stage<LOGN, LE, 0>(x, ad, c);
            sts_row<LOGN, LE>(sm, x, tid);           // own row of `sm`: last read by this thread (lds_row of b)
            poly_sync<G::TPP>();
        }
    }
    inv_last_stage<LOGN, LE>(x, twi, twic, c);
#pragma unroll
    for (int k = 0; k < G::E; k++) st_stream(out + off + tid + G::TPP * k, x[k]);
}

// ---------------------------------------------------------------------------------- generic (any n) u32 kernels
// One CTA per polynomial, whole polynomial in dynamic shared memory, radix-2 stages with a barrier between
// them.  Serves sizes outside {1024, 2048, 4096}; natural-order tables (ntt.cpp:298-300 indexing).
template <bool INVERSE>
__global__ void __launch_bounds__(256) ntt_generic_kernel(uint32_t *__restrict__ data, const uint2 *__restrict__ tw_nat,
                                                          const LimbConst *__restrict__ lc, uint32_t L, uint32_t logn) {
    extern __shared__ uint32_t s[];
    const uint32_t n = 1u << logn;
    const uint32_t poly = blockIdx.x, limb = poly % L;
    const LimbConst c = lc[limb];
    const uint2 *tw = tw_nat + (size_t)limb * n;
    uint32_t *g = data + (size_t)poly * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s[i] = g[i];
    __syncthreads();
    if (!INVERSE) {
        uint32_t tlog = logn - 1;
        for (uint32_t m = 1; m < n; m <<= 1, tlog--) {
            for (uint32_t bf = threadIdx.x; bf < n / 2; bf += blockDim.x) {
                const uint32_t i = bf >> tlog, j = bf & ((1u << tlog) - 1);   // ntt.cpp:292-297
                const uint32_t a0 = (i << (tlog + 1)) + j;
                uint32_t x = s[a0], y = s[a0 + (1u << tlog)];
                ct_bfly(x, y, tw[m + i], c);
                s[a0] = x; s[a0 + (1u << tlog)] = y;
            }
            __syncthreads();
        }
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) g[i] = reduce4q(s[i], c);
    } else {
        uint32_t tlog = 0;
        for (uint32_t h = n >> 1; h >= 1; h >>= 1, tlog++) {
            for (uint32_t bf = threadIdx.x; bf < n / 2; bf += blockDim.x) {
                const uint32_t i = bf >> tlog, j = bf & ((1u << tlog) - 1);
                const uint32_t a0 = (i << (tlog + 1)) + j;
                uint32_t u = s[a0], v = s[a0 + (1u << tlog)];
                gs_bfly(u, v, tw[h + i], c);
                s[a0] = u; s[a0 + (1u << tlog)] = v;
            }
            __syncthreads();
        }
        const uint2 wn = tw[0];   // natural inverse table keeps (n^-1, .) in the unused entry 0
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) g[i] = csub(shoup_mul(s[i], wn, c.negq), c.negq);
    }
}

// ------------------------------------------------------------------- large sizes (n = 8192, 16384, 32768), u32
// Above the two-pass kernels' reach a polynomial (32-128 KB) no longer fits the register files of one CTA's threads, but it
// fits ONE CTA's shared memory, so it is still read from HBM once and written once.  The log2 n stages (ntt.cpp:146-159 loop
// nest, :292-300 twiddle index m + i) run as passes of up to four stages on 16 coefficients per (virtual) thread -- the
// scheme of the u64 frame kernel below, with the u32 butterflies of agx_arith.cuh and natural-order tables:
//   pass 0 works on index bits [logn-4, logn), the next ones on the four bits below, ... (the last of those may be partial:
//   it then holds bits [4,8) and runs only the stages of the bits not yet done), a final pass on bits 3..0.
// Pass p is described by (lo, jf, sf): element k of virtual thread vt = (t_hi, t_lo) is index (t_hi << (lo+4)) + t_lo + (k << lo),
// local stages jf..3 are global stages sf.., stage j pairs x[g*2h+i] with x[g*2h+i+h], h = 8 >> j, under twiddle
// tw[2^(sf+j-jf) + (t_hi << j) + g].  The inverse runs the same passes backwards with Gentleman-Sande butterflies on the same
// indices of the inverse table and multiplies by n^-1 (entry 0 of that table) on the way out.
// Image in shared memory: one word of padding per 32 (A(idx) = idx + idx/32): conflict-free when lanes walk along
// consecutive indices (lo >= 5) and when every lane reads its own 16 consecutive words (lo = 0).
__device__ __forceinline__ uint32_t big_img(uint32_t idx) { return idx + (idx >> 5); }

template <bool INVERSE, int JF>
__device__ __forceinline__ void big_pass16(uint32_t (&x)[16], const uint2 *__restrict__ tw, uint32_t sf, uint32_t t_hi,
                                           const LimbConst &c) {
#pragma unroll
    for (int jj = JF; jj < 4; jj++) {
        const int j = INVERSE ? 3 + JF - jj : jj;              // forward JF..3, inverse 3..JF
        const int h = 8 >> j;
        const uint32_t tbase = (1u << (sf + j - JF)) + (t_hi << j);
        uint2 w[8];
        if (j == 0) {
            w[0] = __ldg(tw + tbase);
        } else {                                             // 2^j consecutive entries from a 2^j-aligned index: 16-byte pairs
            const uint4 *t4 = reinterpret_cast<const uint4 *>(tw + tbase);
#pragma unroll
            for (int g2 = 0; g2 < (1 << j) / 2; g2++) {
                const uint4 v = __ldg(t4 + g2);
                w[2 * g2] = make_uint2(v.x, v.y);
                w[2 * g2 + 1] = make_uint2(v.z, v.w);
            }
        }
#pragma unroll
        for (int g = 0; g < (1 << j); g++)
#pragma unroll
            for (int i = 0; i < h; i++) {
                if (INVERSE) gs_bfly(x[g * 2 * h + i], x[g * 2 * h + i + h], w[g], c);
                else ct_bfly(x[g * 2 * h + i], x[g * 2 * h + i + h], w[g], c);
            }
    }
}

template <bool INVERSE>
__device__ __forceinline__ void big_pass16_jf(uint32_t (&x)[16], const uint2 *__restrict__ tw, uint32_t jf, uint32_t sf,
                                              uint32_t t_hi, const LimbConst &c) {
    if (jf == 0) big_pass16<INVERSE, 0>(x, tw, sf, t_hi, c);
    else if (jf == 1) big_pass16<INVERSE, 1>(x, tw, sf, t_hi, c);
    else if (jf == 2) big_pass16<INVERSE, 2>(x, tw, sf, t_hi, c);
    else big_pass16<INVERSE, 3>(x, tw, sf, t_hi, c);
}

// LOGN is a template parameter so that every pass's bit position, stride and stage count is a compile-time constant (image
// accesses are base + immediate, the pass loop unrolls into exactly the passes a size runs), as in ref_u64_frame_kernel.
template <bool INVERSE, int LOGN>
__global__ void __launch_bounds__(1024, 1) ntt_big_kernel(uint32_t *data, const uint2 *__restrict__ tw_nat,
                                                           const LimbConst *__restrict__ lc, uint32_t L) {
    extern __shared__ uint32_t bimg[];
    constexpr uint32_t logn = LOGN;
    constexpr uint32_t n = 1u << logn, vthreads = n >> 4;
    const uint32_t tid = threadIdx.x, NT = blockDim.x;
    const uint32_t poly = blockIdx.x, limb = poly % L;
    const LimbConst c = lc[limb];
    const uint2 *tw = tw_nat + (size_t)limb * n;
    uint32_t *g = data + (size_t)poly * n;
    constexpr int np = 2 + (int)((logn - 8 + 3) / 4);          // pass 0, the passes on the bits between, the final pass
    uint32_t x[16];

#pragma unroll
    for (int pp = 0; pp < np; pp++) {
        const int p = INVERSE ? np - 1 - pp : pp;
        uint32_t lo, jf, sf;
        if (p == 0) { lo = logn - 4; jf = 0; sf = 0; }
        else if (p == np - 1) { lo = 0; jf = 0; sf = logn - 4; }
        else {
            const uint32_t rem = logn - 8 - 4 * (uint32_t)(p - 1);
            lo = rem >= 4 ? rem : 4; jf = rem >= 4 ? 0 : 4 - rem; sf = 4 + 4 * (uint32_t)(p - 1);
        }
        // the first pass of either direction reads global memory, the last one writes it: pass 0 by coalesced 4-byte
        // accesses (lanes on consecutive indices), the final pass by four 16-byte accesses of a thread's own 64 bytes
        const bool from_global = pp == 0, to_global = pp == np - 1;
        // Image address of element k: A(idx0 + (k << lo)) = A(idx0) + k * stride + fix(k), all of it a per-thread base plus
        // uniform or compile-time terms: lo >= 5: k << lo is a multiple of 32, stride = 2^lo + 2^(lo-5), fix = 0;
        // lo == 4 (idx0 % 256 < 16): stride = 16, fix = k >> 1;  lo == 0 (idx0 % 16 == 0): stride = 1, fix = 0.
        const uint32_t stride = lo >= 5 ? (1u << lo) + (1u << (lo - 5)) : (1u << lo);
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint32_t *sp = bimg + big_img(idx0);
            if (from_global && INVERSE) {                      // final pass first: lo == 0
                const uint4 *g4 = reinterpret_cast<const uint4 *>(g + idx0);
#pragma unroll
                for (int k4 = 0; k4 < 4; k4++) {
                    const uint4 v = g4[k4];
                    x[4 * k4] = v.x; x[4 * k4 + 1] = v.y; x[4 * k4 + 2] = v.z; x[4 * k4 + 3] = v.w;
                }
            } else if (from_global) {
                const uint32_t *gp = g + idx0;
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = __ldcs(gp + ((uint32_t)k << lo));
            } else if (lo == 4) {
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = sp[16 * k + (k >> 1)];
            } else {
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = sp[k * stride];
            }
            big_pass16_jf<INVERSE>(x, tw, jf, sf, t_hi, c);
            if (!INVERSE && p == np - 1) {                     // ntt.cpp:377-393
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = reduce4q(x[k], c);
            }
            if (to_global && INVERSE) {                        // pass 0 last: scale by n^-1, coalesced 4-byte stores
                const uint2 wn = __ldg(tw);                    // the inverse table keeps (n^-1, .) in its unused entry 0
                uint32_t *gp = g + idx0;
#pragma unroll
                for (int k = 0; k < 16; k++) __stcs(gp + ((uint32_t)k << lo), csub(shoup_mul(x[k], wn, c.negq), c.negq));
            } else if (to_global) {                            // final pass last: lo == 0
                uint4 *g4 = reinterpret_cast<uint4 *>(g + idx0);
#pragma unroll
                for (int k4 = 0; k4 < 4; k4++) g4[k4] = make_uint4(x[4 * k4], x[4 * k4 + 1], x[4 * k4 + 2], x[4 * k4 + 3]);
            } else if (lo == 4) {
#pragma unroll
                for (int k = 0; k < 16; k++) sp[16 * k + (k >> 1)] = x[k];
            } else {
#pragma unroll
                for (int k = 0; k < 16; k++) sp[k * stride] = x[k];
            }
        }
        __syncthreads();
    }
}

template <int DUMMY = 0>
__global__ void __launch_bounds__(256) pointwise_generic_kernel(uint32_t *a, const uint32_t *b,   // a may equal b (squaring)
                                                                const LimbConst *__restrict__ lc, uint32_t L,
                                                                uint32_t logn, size_t total) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const LimbConst c = lc[(i >> logn) % L];
    a[i] = csub(barrett_mul_lazy(a[i], b[i], c), c.neg2q);   // [0,2q): valid inverse input
}

// ------------------------------------------------------------------- limb-wise (RNS) element-wise arithmetic
// The operations a caller performs around the transforms on [B][L][n] data (SURVEY.md s.8(f) rank 4): add, subtract,
// multiply and multiply-accumulate modulo each limb's prime, e.g. on spectra between agx_ntt_fwd and agx_ntt_inv.
// Pure streaming kernels: 16-byte vector accesses, grid-stride, 3 (add/sub/mul) or 4 (mac) u32 streams of HBM traffic.
enum EwOp { EW_ADD = 0, EW_SUB = 1, EW_MUL = 2, EW_MAC = 3 };

template <int OP>
__device__ __forceinline__ uint32_t ew_apply(uint32_t cv, uint32_t av, uint32_t bv, const LimbConst &c) {
    if (OP == EW_ADD) return csub(av + bv, c.negq);
    if (OP == EW_SUB) return csub(av + c.q - bv, c.negq);
    const uint32_t m = csub(csub(barrett_mul_lazy(av, bv, c), c.neg2q), c.negq);
    if (OP == EW_MUL) return m;
    return csub(cv + m, c.negq);
}

template <int OP>
__global__ void __launch_bounds__(256) elementwise_kernel(uint4 *c4, const uint4 *a4, const uint4 *b4,
                                                          const LimbConst *__restrict__ lc, uint32_t L, uint32_t logn,
                                                          size_t total4) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (size_t)gridDim.x * blockDim.x) {
        const LimbConst c = lc[((i * 4) >> logn) % L];
        const uint4 a = a4[i], b = b4[i];
        uint4 r = make_uint4(0, 0, 0, 0);
        if (OP == EW_MAC) r = c4[i];
        r.x = ew_apply<OP>(r.x, a.x, b.x, c);
        r.y = ew_apply<OP>(r.y, a.y, b.y, c);
        r.z = ew_apply<OP>(r.z, a.z, b.z, c);
        r.w = ew_apply<OP>(r.w, a.w, b.w, c);
        c4[i] = r;
    }
}

// ------------------------------------------------------------------------- reference-shaped u64 forward kernel
// Arithmetic of fwd_ntt_kernel (ntt.cpp:146-159, 292-300, 331-332, 344-363, 368-369, 377-393), including
// wrap-around mod 2^64 when the tables are not Shoup pairs (main.cpp:49-55 feeds such data).  One CTA per frame
// (ntt.cpp:579-595 frame layout: low half from `in`, high half from `in2`); work array in dynamic smem when
// N*8 bytes fits, else in the output buffer itself.
// ref_fwd_u64_body is this kernel's body for the per-limb variant (ref_fwd_u64_rns_kernel).  ref_fwd_u64_kernel keeps its
// own copy: routed through the shared body it compiles to different SASS, and the single-modulus kernels stay as they were.
// TWIN: ref_fwd_u64_rescale_kernel (the rescale's fused forward below N = 1024) is a copy of this body with a prologue and
// an epilogue; a fix here belongs there too.
// TWIN: ref_fwd_u64_basis_kernel (ModUp / ModDown's fused forward below N = 1024) is another such copy; a fix here
// belongs there too.
__device__ __forceinline__ void ref_fwd_u64_body(const uint64_t *__restrict__ in, const uint64_t *__restrict__ in2,
                                                 uint64_t *__restrict__ out, const uint64_t *__restrict__ roots,
                                                 const uint64_t *__restrict__ precons, uint64_t q, uint32_t logn, int use_smem,
                                                 uint32_t frame) {
    extern __shared__ uint64_t s64[];
    const uint32_t N = 1u << logn;
    const size_t base = (size_t)frame * N;
    uint64_t *X = use_smem ? s64 : out + base;
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) X[i] = i < N / 2 ? in[base + i] : in2[base + i];
    __syncthreads();
    const uint64_t twice = q << 1;
    uint32_t tlog = logn - 1;
    for (uint32_t m = 1; m < N; m <<= 1, tlog--) {
        const bool last = (m == N / 2);
        for (uint32_t bf = threadIdx.x; bf < N / 2; bf += blockDim.x) {
            const uint32_t i = bf >> tlog, j = bf & ((1u << tlog) - 1);
            const uint32_t a0 = (i << (tlog + 1)) + j, a1 = a0 + (1u << tlog);
            const uint64_t W = roots[m + i], Wp = precons[m + i];
            uint64_t tx = X[a0];
            if (tx >= twice) tx -= twice;
            const uint64_t a = X[a1];
            const uint64_t c1 = __umul64hi(a, Wp);
            const uint64_t Q = W * a - c1 * q;
            uint64_t o0 = tx + Q, o1 = tx + twice - Q;
            if (last) {
                if (o0 >= twice) o0 -= twice;
                if (o0 >= q) o0 -= q;
                if (o1 >= twice) o1 -= twice;
                if (o1 >= q) o1 -= q;
            }
            X[a0] = o0; X[a1] = o1;
        }
        __syncthreads();
    }
    if (use_smem)
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) out[base + i] = X[i];
}

// TWIN: ref_fwd_u64_body is a copy of this kernel for the per-limb (RNS) variants; a fix here belongs there too (this copy is
// kept apart so that the single-modulus kernel keeps its SASS).
__global__ void __launch_bounds__(1024) ref_fwd_u64_kernel(const uint64_t *__restrict__ in, const uint64_t *__restrict__ in2,
                                                           uint64_t *__restrict__ out, const uint64_t *__restrict__ roots,
                                                           const uint64_t *__restrict__ precons, uint64_t q, uint32_t logn,
                                                           int use_smem) {
    extern __shared__ uint64_t s64[];
    const uint32_t N = 1u << logn;
    const size_t base = (size_t)blockIdx.x * N;
    uint64_t *X = use_smem ? s64 : out + base;
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) X[i] = i < N / 2 ? in[base + i] : in2[base + i];
    __syncthreads();
    const uint64_t twice = q << 1;
    uint32_t tlog = logn - 1;
    for (uint32_t m = 1; m < N; m <<= 1, tlog--) {
        const bool last = (m == N / 2);
        for (uint32_t bf = threadIdx.x; bf < N / 2; bf += blockDim.x) {
            const uint32_t i = bf >> tlog, j = bf & ((1u << tlog) - 1);
            const uint32_t a0 = (i << (tlog + 1)) + j, a1 = a0 + (1u << tlog);
            const uint64_t W = roots[m + i], Wp = precons[m + i];
            uint64_t tx = X[a0];
            if (tx >= twice) tx -= twice;
            const uint64_t a = X[a1];
            const uint64_t c1 = __umul64hi(a, Wp);
            const uint64_t Q = W * a - c1 * q;
            uint64_t o0 = tx + Q, o1 = tx + twice - Q;
            if (last) {
                if (o0 >= twice) o0 -= twice;
                if (o0 >= q) o0 -= q;
                if (o1 >= twice) o1 -= twice;
                if (o1 >= q) o1 -= q;
            }
            X[a0] = o0; X[a1] = o1;
        }
        __syncthreads();
    }
    if (use_smem)
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) out[base + i] = X[i];
}

// ------------------------------------------------------------------------------------ coefficient-order adapter
// The transforms keep the reference's orders (ntt.cpp: natural in, bit-reversed out; the inverse the other way round).
// Callers that hold or want spectra in natural order (textbook / NTL-style code) permute with this kernel: row i of
// each n-coefficient polynomial moves to bitrev(i).  An involution; in place; one CTA per polynomial, through shared
// memory so that both the global reads and the global writes are coalesced 16-byte accesses.
__global__ void __launch_bounds__(256) bitrev_rows_kernel(uint32_t *__restrict__ data, uint32_t logn) {
    extern __shared__ uint32_t s[];
    const uint32_t n = 1u << logn;
    uint32_t *g = data + ((size_t)blockIdx.x << logn);
    for (uint32_t i = threadIdx.x * 4; i < n; i += blockDim.x * 4) {
        const uint4 v = *reinterpret_cast<const uint4 *>(g + i);
        s[__brev(i) >> (32 - logn)] = v.x;
        s[__brev(i + 1) >> (32 - logn)] = v.y;
        s[__brev(i + 2) >> (32 - logn)] = v.z;
        s[__brev(i + 3) >> (32 - logn)] = v.w;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x * 4; i < n; i += blockDim.x * 4)
        *reinterpret_cast<uint4 *>(g + i) = make_uint4(s[i], s[i + 1], s[i + 2], s[i + 3]);
}

// ------------------------------------------------------------- reference-shaped u64 forward: register-radix passes
// The reference's native sizes (ntt.h:11-20: 1024, 8192, 16384, 32768) as a sequence of launches over a chunk of
// frames that stays resident in L2: every pass keeps 2^LS coefficients of one butterfly network in registers and
// runs LS stages on them (ntt.cpp:146-159 loop nest, :292-300 twiddle index m + i, :331-369 butterfly), so a frame
// makes logN/4 round trips instead of logN through shared memory, and N = 32768 (256 KB, more than an SM's shared
// memory) needs no special case.  Arithmetic is the u64 butterfly of ref_fwd_u64_kernel, mod 2^64 exactly.
//   strided passes : thread holds p = p_hi * 2^(logN-s0) + k * 2^(logN-s0-LS) + p_lo, k < 2^LS; consecutive threads
//                    take consecutive p_lo (coalesced 8-byte accesses); twiddles are uniform over p_lo.
//   last pass      : the final 4 stages act on 16 consecutive coefficients (128 B) per thread; a warp stages its
//                    512 consecutive coefficients through a private padded shared-memory tile so that global
//                    accesses stay coalesced; includes the final reduction to [0,q) (ntt.cpp:377-393).
// A/B knobs of the 64-bit butterfly and its twiddle loads (profiles/r02_experiments.md).  AGX_U64_VECTW: 0 = 8-byte twiddle
// loads everywhere, 1 = 16-byte pairs in the frame kernel's 512-thread instantiation only (N >= 16384: +2-6 %; the smaller
// CTAs lose up to 7 % to the 32 bytes of spills the pairs cost at 128 registers), 2 = pairs everywhere.
#ifndef AGX_U64_NEGQ
#define AGX_U64_NEGQ 1
#endif
#ifndef AGX_U64_VECTW
#define AGX_U64_VECTW 1
#endif
// AGX_U64_BORROW: the x-correction (ntt.cpp:331-332) decided by the borrow of the 64-bit subtraction it needs anyway
// instead of a separate 64-bit compare: two ISETP less per butterfly, and fewer of the remaining adds placed on the multiply
// pipe by ptxas -- the isolated butterfly stream goes from 3.00-3.05 to 3.36-3.38 butterflies/clk/SM, the frame kernel gains
// 4 % (profiles/r02_u64_borrow_ab.txt).
#ifndef AGX_U64_BORROW
#define AGX_U64_BORROW 1
#endif
__device__ __forceinline__ uint64_t ref_csub_u64(uint64_t x, uint64_t m) {
#if AGX_U64_BORROW
    const uint32_t x0 = (uint32_t)x, x1 = (uint32_t)(x >> 32);
    uint32_t d0, d1, b;
    asm("{\n\t"
        "sub.cc.u32 %0, %3, %5;\n\t"
        "subc.cc.u32 %1, %4, %6;\n\t"
        "subc.u32 %2, 0, 0;\n\t"
        "}" : "=r"(d0), "=r"(d1), "=r"(b) : "r"(x0), "r"(x1), "r"((uint32_t)m), "r"((uint32_t)(m >> 32)));
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(b ? x0 : d0), "r"(b ? x1 : d1));
    return r;
#else
    return x >= m ? x - m : x;
#endif
}

__device__ __forceinline__ void ref_bfly_u64(uint64_t &x, uint64_t &y, uint64_t W, uint64_t Wp, uint64_t q, uint64_t twice) {
    const uint64_t tx = ref_csub_u64(x, twice);   // ntt.cpp:331-332
    const uint64_t c1 = __umul64hi(y, Wp);        // ntt.cpp:344-358
#if AGX_U64_NEGQ
    uint64_t negq;                                // -q through an opaque (pure, hence hoisted and shared) instruction:
    asm("neg.s64 %0, %1;" : "=l"(negq) : "l"(q)); // left as 0 - q the compiler folds the sum below back into a difference
    const uint64_t Q = W * y + c1 * negq;         // ntt.cpp:363  W*y - c1*q mod 2^64; written as a sum the second product
                                                  // accumulates onto the first (ptxas otherwise negates c1 per butterfly:
                                                  // 25.5 instead of 27.5 SASS instructions, profiles/r02_experiments.md)
#else
    const uint64_t Q = W * y - c1 * q;            // ntt.cpp:363
#endif
    x = tx + Q;                                   // ntt.cpp:368
    y = tx + twice - Q;                           // ntt.cpp:369
}

// The 2^j twiddles (and precons) a thread needs at local stage j of a register pass are consecutive table entries starting
// at an index that is a multiple of 2^j (ntt.cpp:298-300: m + i with m = 2^s >= 2^j groups and i = (group of the pass) << j),
// so for j >= 1 they come in as 16-byte pairs: half the load instructions of one LDG.64 per entry.  The tables must be
// 16-byte aligned (cudaMalloc'd ones are; agx_ref_fwd_dev checks the caller's).
template <int CNT, bool VEC>
__device__ __forceinline__ void ref_load_tw_u64(uint64_t (&W)[CNT], uint64_t (&Wp)[CNT], const uint64_t *__restrict__ roots,
                                                const uint64_t *__restrict__ precons, uint32_t tbase) {
    if constexpr (CNT == 1 || !VEC) {
#pragma unroll
        for (int g = 0; g < CNT; g++) {
            W[g] = __ldg(roots + tbase + g);
            Wp[g] = __ldg(precons + tbase + g);
        }
    } else {
        const ulonglong2 *r2 = reinterpret_cast<const ulonglong2 *>(roots + tbase);
        const ulonglong2 *p2 = reinterpret_cast<const ulonglong2 *>(precons + tbase);
#pragma unroll
        for (int g2 = 0; g2 < CNT / 2; g2++) {
            const ulonglong2 a = __ldg(r2 + g2), b = __ldg(p2 + g2);
            W[2 * g2] = a.x; W[2 * g2 + 1] = a.y;
            Wp[2 * g2] = b.x; Wp[2 * g2 + 1] = b.y;
        }
    }
}

// one stage of a register pass over E = 2^LS coefficients: local stage J pairs x[g*2h + i] with x[g*2h + i + h], h = E >> (J+1)
template <int LS, int J, bool VEC>
__device__ __forceinline__ void ref_stage_u64(uint64_t (&x)[1 << LS], const uint64_t *__restrict__ roots,
                                              const uint64_t *__restrict__ precons, uint32_t tbase, uint64_t q, uint64_t twice) {
    constexpr int half = (1 << LS) >> (J + 1);
    uint64_t W[1 << J], Wp[1 << J];
    ref_load_tw_u64<(1 << J), VEC>(W, Wp, roots, precons, tbase);
#pragma unroll
    for (int g = 0; g < (1 << J); g++)
#pragma unroll
        for (int i = 0; i < half; i++) ref_bfly_u64(x[g * 2 * half + i], x[g * 2 * half + i + half], W[g], Wp[g], q, twice);
}

template <int LS, int J = 0>
__device__ __forceinline__ void ref_stages_u64(uint64_t (&x)[1 << LS], const uint64_t *__restrict__ roots,
                                               const uint64_t *__restrict__ precons, uint32_t s0, uint32_t p_hi, uint64_t q) {
    // roots[m + i]: m = 2^s groups, i = p >> (logN - s)
    ref_stage_u64<LS, J, (AGX_U64_VECTW >= 2)>(x, roots, precons, (1u << (s0 + J)) + (p_hi << J), q, q << 1);
    if constexpr (J + 1 < LS) ref_stages_u64<LS, J + 1>(x, roots, precons, s0, p_hi, q);
}

template <int LS>
__global__ void __launch_bounds__(256) ref_u64_strided_pass_kernel(const uint64_t *src, const uint64_t *src2, uint64_t *dst,
                                                                   const uint64_t *__restrict__ roots,
                                                                   const uint64_t *__restrict__ precons, uint64_t q,
                                                                   uint32_t logn, uint32_t s0, uint32_t frames) {
    constexpr int E = 1 << LS;
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t frame = gid >> (logn - LS), tidx = gid & ((1u << (logn - LS)) - 1);
    if (frame >= frames) return;
    const uint32_t lo_bits = logn - s0 - LS;
    const uint32_t p_lo = tidx & ((1u << lo_bits) - 1), p_hi = tidx >> lo_bits;
    const uint32_t pos = (p_hi << (logn - s0)) + p_lo;                    // position of element k = 0 inside the frame
    const size_t base = ((size_t)frame << logn) + pos;
    uint64_t x[E];
#pragma unroll
    for (int k = 0; k < E; k++) {                                         // high half of a frame comes from src2 (ntt.cpp:587-589)
        const uint64_t *s = ((pos + ((uint32_t)k << lo_bits)) >> (logn - 1)) ? src2 : src;
        x[k] = s[base + ((size_t)k << lo_bits)];
    }
    ref_stages_u64<LS>(x, roots, precons, s0, p_hi, q);
#pragma unroll
    for (int k = 0; k < E; k++) dst[base + ((size_t)k << lo_bits)] = x[k];
}

__global__ void __launch_bounds__(128) ref_u64_last_pass_kernel(uint64_t *data, const uint64_t *__restrict__ roots,
                                                                const uint64_t *__restrict__ precons, uint64_t q,
                                                                uint32_t logn, uint32_t frames) {
    constexpr int LS = 4, E = 16, PITCH4 = 9;                 // 8 chunks of 16 bytes per thread row + 1 of padding
    __shared__ uint4 tile[4][32 * PITCH4];
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t frame = gid >> (logn - LS), tidx = gid & ((1u << (logn - LS)) - 1);
    if (frame >= frames) return;                              // whole warps: a frame has N/16 >= 64 threads
    uint4 *t = tile[wib];
    uint4 *g4 = reinterpret_cast<uint4 *>(data + ((size_t)(gid - lane) << LS));   // the warp's 512 coefficients
#pragma unroll
    for (int i = 0; i < 8; i++) {                             // chunk c = i*32 + lane: row c/8, column c%8
        const uint32_t c = i * 32 + lane;
        t[(c >> 3) * PITCH4 + (c & 7)] = g4[c];
    }
    __syncwarp();
    uint64_t x[E];
#pragma unroll
    for (int c = 0; c < 8; c++) {
        const uint4 v = t[lane * PITCH4 + c];
        x[2 * c] = (uint64_t)v.x | ((uint64_t)v.y << 32);
        x[2 * c + 1] = (uint64_t)v.z | ((uint64_t)v.w << 32);
    }
    ref_stages_u64<LS>(x, roots, precons, logn - LS, tidx, q);
    const uint64_t twice = q << 1;
#pragma unroll
    for (int k = 0; k < E; k++) {                             // ntt.cpp:377-393
        x[k] = ref_csub_u64(ref_csub_u64(x[k], twice), q);
    }
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 8; c++)
        t[lane * PITCH4 + c] = make_uint4((uint32_t)x[2 * c], (uint32_t)(x[2 * c] >> 32), (uint32_t)x[2 * c + 1],
                                          (uint32_t)(x[2 * c + 1] >> 32));
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t c = i * 32 + lane;
        g4[c] = t[(c >> 3) * PITCH4 + (c & 7)];
    }
}

// ---------------------------------------------------------------- reference-shaped u64 forward: one launch per round
// The whole frame lives in ONE CTA's shared memory (N <= 16384: 128 KB + padding; a B200 SM offers 227 KB), so a frame is
// read from HBM once and written once instead of making logN/4 round trips: loader, compute unit and drain of the
// reference (ntt.cpp:508-607, 86-506, 610-640) in one kernel.  N = 32768 (256 KB) takes two CTAs per frame: stage 0
// pairs x[i] with x[i + N/2] (ntt.cpp:292-300 with m = 1), after which the halves are independent 16384-point
// sub-transforms; each CTA reads both halves, keeps its own output of stage 0 and carries on alone (costs one extra
// stage of arithmetic in 15, no exchange between CTAs).
// 512 threads per SM at <= 128 registers (the 64-bit butterfly with its twiddle pairs in flight does not fit 64, measured:
// 570 bytes of spills), so the 1024 "virtual threads" of a 16384-point frame are two rounds of a 512-thread CTA.
// Every "virtual thread" keeps 16 coefficients in registers per pass (index bits [lo, lo+4) vary inside the thread) and
// runs up to 4 stages on them; passes go from the top index bits down to bit 4 -- the last of those may be partial --
// and a final pass works on bits 3..0, i.e. on 16 consecutive coefficients.  Image in shared memory: a row of 16
// coefficients every 17 words of 8 bytes (A(idx) = idx + idx/16), which makes every pass's 64-bit accesses
// conflict-free: lanes walk along a row when lo >= 4, and down the rows at a 136-byte pitch when lo = 0.
// Arithmetic: ref_bfly_u64 (ntt.cpp:331-369 mod 2^64, any tables), final reduction ntt.cpp:377-393.
template <bool VEC, int JFIRST, int J = JFIRST>
__device__ __forceinline__ void ref_pass16_u64(uint64_t (&x)[16], const uint64_t *__restrict__ roots,
                                               const uint64_t *__restrict__ precons, uint32_t s_first, uint32_t t_hi, uint64_t q,
                                               uint64_t twice) {
    // local stage J (JFIRST..3) is global stage s_first + (J - JFIRST); pairs x[g*2h + i], x[g*2h + i + h], h = 8 >> J;
    // twiddle index m + i of ntt.cpp:298-300 = 2^s + (t_hi << J) + g  (s_first >= JFIRST in every caller, so the index of
    // g = 0 is a multiple of 2^J as ref_load_tw_u64 needs)
    ref_stage_u64<4, J, VEC>(x, roots, precons, (1u << (s_first + J - JFIRST)) + (t_hi << J), q, twice);
    if constexpr (J < 3) ref_pass16_u64<VEC, JFIRST, J + 1>(x, roots, precons, s_first, t_hi, q, twice);
}

// ref_u64_frame_kernel (below) as the body of its per-limb variants (ref_u64_rns_frame_kernel, ...); the single-modulus
// kernel keeps its own copy, as ref_fwd_u64_kernel does.  PAIR: the two CTAs of a split frame form a 2-CTA
// cluster and each waits on the cluster barrier before its final global stores, so that neither overwrites a half its
// partner has not read yet (pass 0 is the only phase that reads global memory): in place is then safe at N = 32768.
// TWIN: ref_u64_rescale_fwd_kernel (the rescale's fused forward) is a copy of this body with a prologue in pass 0 and an
// epilogue in the final store; a fix here belongs there too.
// TWIN: ref_u64_basis_fwd_kernel (ModUp / ModDown's fused forward) is another such copy; a fix here belongs there too.
template <int NT, bool PAIR = false>
__device__ __forceinline__ void ref_u64_frame_body(const uint64_t *in, const uint64_t *in2, uint64_t *out,
                                                   const uint64_t *__restrict__ roots, const uint64_t *__restrict__ precons,
                                                   uint64_t q, uint32_t logn, uint32_t split, uint32_t frame, uint32_t half_id) {
    // split = 0: one CTA per frame, logn <= 14.  split = 1: two CTAs per frame (logn = 15), CTA parity = which half.
    extern __shared__ uint64_t img[];
    constexpr bool VEC = AGX_U64_VECTW >= 2 || (AGX_U64_VECTW == 1 && NT >= 512);   // 16-byte twiddle pairs
    const uint32_t tid = threadIdx.x;
    // log2 of the coefficients this CTA owns: always log2(NT) + 5 (a CTA is N/32 threads, agx_api.cu ref_launch), so it is a
    // compile-time constant and with it every pass's bit position, stride and stage count: shared-memory accesses become
    // base + immediate and the pass loop unrolls into exactly the passes this size runs
    constexpr uint32_t lg = (NT == 512 ? 14u : NT == 256 ? 13u : NT == 128 ? 12u : NT == 64 ? 11u : 10u);
    constexpr uint32_t M = 1u << lg, vthreads = M >> 4;
    if (logn - split != lg) return;                                // launch contract (never taken)
    const uint64_t twice = q << 1;
    const size_t fbase = (size_t)frame << logn;
    const uint64_t *lo_src = in + fbase, *hi_src = in2 + fbase;    // low / high half of the frame (ntt.cpp:587-589)
    uint64_t x[16];

    // ---- pass 0: stages (split ..) on index bits [lg-4, lg), coefficients straight from global memory
    {
        constexpr uint32_t lo = lg - 4;
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            if (split) {
                // stage 0 of the 32768-point frame, this CTA keeping only its half (ntt.cpp:331-369 with roots[1])
                const uint64_t W = __ldg(roots + 1), Wp = __ldg(precons + 1);
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    uint64_t a = lo_src[i], b = hi_src[M + i];
                    ref_bfly_u64(a, b, W, Wp, q, twice);
                    x[k] = half_id ? b : a;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    x[k] = (k < 8 ? lo_src : hi_src)[i];
                }
            }
            // this CTA's sub-transform: stage s of it is global stage s + split, group offset half_id << s
            // (roots index = 2^(s+split) + (half_id << s) + local group)
            ref_pass16_u64<VEC, 0>(x, roots, precons, split, half_id, q, twice);
            uint64_t *s = img + vt + (vt >> 4);
            constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
    }
    if constexpr (PAIR) asm volatile("barrier.cluster.arrive.aligned;" ::: "memory");   // this CTA's global reads are done
    __syncthreads();
    // ---- middle passes: index bits from lg-5 down to 4, four at a time (the last one may cover fewer)
    uint32_t s_done = 4;                                           // stages of the sub-transform finished so far
#pragma unroll
    for (int rem = (int)lg - 8; rem > 0; rem -= 4) {
        const uint32_t lo = rem >= 4 ? (uint32_t)rem : 4u;
        const uint32_t jfirst = rem >= 4 ? 0u : (uint32_t)(4 - rem);
        const uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint64_t *s = img + idx0 + (idx0 >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            // twiddle index: 2^(s+split) + ((half_id << s) + group) with group = (t_hi << j) + g at local stage j
            const uint32_t sg = s_done + split;                    // global stage of the first active local stage
            const uint32_t th = t_hi + (half_id << (s_done - jfirst));   // the CTA's half as the top bit of the group index
            if (jfirst == 0) ref_pass16_u64<VEC, 0>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 1) ref_pass16_u64<VEC, 1>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 2) ref_pass16_u64<VEC, 2>(x, roots, precons, sg, th, q, twice);
            else ref_pass16_u64<VEC, 3>(x, roots, precons, sg, th, q, twice);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
        s_done += 4 - jfirst;
        __syncthreads();
    }
    // ---- final pass: bits 3..0 (16 consecutive coefficients), reduction to [0,q) (ntt.cpp:377-393)
#pragma unroll 1
    for (uint32_t vt = tid; vt < vthreads; vt += NT) {
        uint64_t *s = img + vt * 17;
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = s[k];
        ref_pass16_u64<VEC, 0>(x, roots, precons, s_done + split, vt + (half_id << s_done), q, twice);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            s[k] = ref_csub_u64(ref_csub_u64(x[k], twice), q);
        }
    }
    __syncthreads();
    if constexpr (PAIR) asm volatile("barrier.cluster.wait.aligned;" ::: "memory");     // ... and the partner's too
    uint64_t *dst = out + fbase + (size_t)half_id * M;
    for (uint32_t i = tid; i < M; i += NT) dst[i] = img[i + (i >> 4)];
}

// TWIN: ref_u64_frame_body is a copy of this kernel for the per-limb (RNS) variants; a fix here belongs there too (this copy is
// kept apart so that the single-modulus kernel keeps its SASS).
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_frame_kernel(const uint64_t *in, const uint64_t *in2,   // may alias each other and out
                                                              uint64_t *out, const uint64_t *__restrict__ roots,
                                                              const uint64_t *__restrict__ precons, uint64_t q, uint32_t logn,
                                                              uint32_t split) {
    // split = 0: one CTA per frame, logn <= 14.  split = 1: two CTAs per frame (logn = 15), CTA parity = which half.
    extern __shared__ uint64_t img[];
    constexpr bool VEC = AGX_U64_VECTW >= 2 || (AGX_U64_VECTW == 1 && NT >= 512);   // 16-byte twiddle pairs
    const uint32_t tid = threadIdx.x;
    const uint32_t frame = split ? blockIdx.x >> 1 : blockIdx.x, half_id = split ? blockIdx.x & 1u : 0u;
    // log2 of the coefficients this CTA owns: always log2(NT) + 5 (a CTA is N/32 threads, agx_api.cu ref_launch), so it is a
    // compile-time constant and with it every pass's bit position, stride and stage count: shared-memory accesses become
    // base + immediate and the pass loop unrolls into exactly the passes this size runs
    constexpr uint32_t lg = (NT == 512 ? 14u : NT == 256 ? 13u : NT == 128 ? 12u : NT == 64 ? 11u : 10u);
    constexpr uint32_t M = 1u << lg, vthreads = M >> 4;
    if (logn - split != lg) return;                                // launch contract (never taken)
    const uint64_t twice = q << 1;
    const size_t fbase = (size_t)frame << logn;
    const uint64_t *lo_src = in + fbase, *hi_src = in2 + fbase;    // low / high half of the frame (ntt.cpp:587-589)
    uint64_t x[16];

    // ---- pass 0: stages (split ..) on index bits [lg-4, lg), coefficients straight from global memory
    {
        constexpr uint32_t lo = lg - 4;
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            if (split) {
                // stage 0 of the 32768-point frame, this CTA keeping only its half (ntt.cpp:331-369 with roots[1])
                const uint64_t W = __ldg(roots + 1), Wp = __ldg(precons + 1);
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    uint64_t a = lo_src[i], b = hi_src[M + i];
                    ref_bfly_u64(a, b, W, Wp, q, twice);
                    x[k] = half_id ? b : a;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    x[k] = (k < 8 ? lo_src : hi_src)[i];
                }
            }
            // this CTA's sub-transform: stage s of it is global stage s + split, group offset half_id << s
            // (roots index = 2^(s+split) + (half_id << s) + local group)
            ref_pass16_u64<VEC, 0>(x, roots, precons, split, half_id, q, twice);
            uint64_t *s = img + vt + (vt >> 4);
            constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
    }
    __syncthreads();
    // ---- middle passes: index bits from lg-5 down to 4, four at a time (the last one may cover fewer)
    uint32_t s_done = 4;                                           // stages of the sub-transform finished so far
#pragma unroll
    for (int rem = (int)lg - 8; rem > 0; rem -= 4) {
        const uint32_t lo = rem >= 4 ? (uint32_t)rem : 4u;
        const uint32_t jfirst = rem >= 4 ? 0u : (uint32_t)(4 - rem);
        const uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint64_t *s = img + idx0 + (idx0 >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            // twiddle index: 2^(s+split) + ((half_id << s) + group) with group = (t_hi << j) + g at local stage j
            const uint32_t sg = s_done + split;                    // global stage of the first active local stage
            const uint32_t th = t_hi + (half_id << (s_done - jfirst));   // the CTA's half as the top bit of the group index
            if (jfirst == 0) ref_pass16_u64<VEC, 0>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 1) ref_pass16_u64<VEC, 1>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 2) ref_pass16_u64<VEC, 2>(x, roots, precons, sg, th, q, twice);
            else ref_pass16_u64<VEC, 3>(x, roots, precons, sg, th, q, twice);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
        s_done += 4 - jfirst;
        __syncthreads();
    }
    // ---- final pass: bits 3..0 (16 consecutive coefficients), reduction to [0,q) (ntt.cpp:377-393)
#pragma unroll 1
    for (uint32_t vt = tid; vt < vthreads; vt += NT) {
        uint64_t *s = img + vt * 17;
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = s[k];
        ref_pass16_u64<VEC, 0>(x, roots, precons, s_done + split, vt + (half_id << s_done), q, twice);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            s[k] = ref_csub_u64(ref_csub_u64(x[k], twice), q);
        }
    }
    __syncthreads();
    uint64_t *dst = out + fbase + (size_t)half_id * M;
    for (uint32_t i = tid; i < M; i += NT) dst[i] = img[i + (i >> 4)];
}

// ------------------------------------------------------------------- u64 inverse transform and negacyclic product
// No reference counterpart (the reference has only the forward, SURVEY.md s.0).  The mirror of the forward above:
// Gentleman-Sande stages h = N/2 .. 1 (h groups, group j reads iroots[h + j] -- the table order of ntt.cpp:298-300 built
// from psi^-1, so stage h has the shape of the forward's stage m = h), Harvey-lazy on [0,2q):
//   u' = u + v  (one conditional subtraction of 2q),   v' = Shoup(u - v + 2q, w)  (< 2q for any input below 2^64)
// and n^-1 folded into the last stage (h = 1): u' = Shoup(u + v, n^-1), v' = Shoup(u - v + 2q, iroots[1] * n^-1), then
// the reduction to [0,q).  The lazy range [0,4q) must fit 64 bits: q < 2^62 (agx_ref_inv_dev refuses larger moduli).
// Optional fused operand `mul` (nullptr = none): the load phase replaces x[i] by x[i] * mul[i] mod q (Barrett, HAC 14.42
// with b = 2: k = bitlen(q), mu = floor(2^2k / q) < 2^63; the remainder is < 3q, so two conditional subtractions), which
// makes the pointwise product of agx_ref_polymul_dev part of the inverse's load.
struct RefInvConst {
    uint64_t q, ninv, ninv_p;      // n^-1 mod q and floor(n^-1 * 2^64 / q)
    uint64_t mu;                   // floor(2^(2k) / q)
    uint64_t recip;                // floor(2^(63+k) / q) < 2^64 (ref_inv_fold)
    uint32_t k;                    // bit length of q, 2 <= k <= 62
};

__device__ __forceinline__ uint64_t ref_shoup_u64(uint64_t y, uint64_t W, uint64_t Wp, uint64_t q) {
    const uint64_t c1 = __umul64hi(y, Wp);
#if AGX_U64_NEGQ
    uint64_t negq;                                // see ref_bfly_u64
    asm("neg.s64 %0, %1;" : "=l"(negq) : "l"(q));
    return W * y + c1 * negq;                     // W*y - c1*q mod 2^64, in [0,2q)
#else
    return W * y - c1 * q;
#endif
}

__device__ __forceinline__ void ref_gs_bfly_u64(uint64_t &x, uint64_t &y, uint64_t W, uint64_t Wp, uint64_t q, uint64_t twice) {
    const uint64_t d = x + twice - y;
    x = ref_csub_u64(x + y, twice);
    y = ref_shoup_u64(d, W, Wp, q);
}

// the last stage with n^-1 folded in, and the reduction to [0,q); f = (iroots[1] * n^-1, its Shoup companion)
__device__ __forceinline__ void ref_gs_last_bfly_u64(uint64_t &x, uint64_t &y, const RefInvConst &p, ulonglong2 f) {
    const uint64_t d = x + (p.q << 1) - y;
    x = ref_csub_u64(ref_shoup_u64(x + y, p.ninv, p.ninv_p, p.q), p.q);
    y = ref_csub_u64(ref_shoup_u64(d, f.x, f.y, p.q), p.q);
}

// (iroots[1] * n^-1 mod q, floor(that * 2^64 / q)): the table is the caller's and on the device, so this is computed here,
// once per CTA (a blocking read on the host would break the call's asynchrony).  The companion without a 128-bit division
// (a bit-serial loop of microseconds, which a whole CTA would wait for): w * recip >> (k-1) is floor(w * 2^64 / q) - e with
// e in [0,2], so the remainder w * 2^64 - estimate * q lies in [0,3q) and is its own low 64 bits; each q it holds past the
// first is one more unit of the quotient.
__device__ __forceinline__ uint64_t ref_shoup_companion(uint64_t w, const RefInvConst &p) {   // floor(w * 2^64 / q), w < q
    const uint32_t s = p.k - 1;
    uint64_t wp = (__umul64hi(w, p.recip) << (64 - s)) | ((w * p.recip) >> s);
    uint64_t r = 0 - wp * p.q;
#pragma unroll
    for (int i = 0; i < 2; i++)
        if (r >= p.q) { r -= p.q; wp++; }
    return wp;
}

__device__ __forceinline__ ulonglong2 ref_inv_fold(const uint64_t *__restrict__ roots, const RefInvConst &p) {
    const uint64_t w = ref_csub_u64(ref_shoup_u64(__ldg(roots + 1), p.ninv, p.ninv_p, p.q), p.q);
    return make_ulonglong2(w, ref_shoup_companion(w, p));
}

// a * b mod q exactly, a, b < q (HAC 14.42, b = 2, computed from the low 64 bits of the remainder)
__device__ __forceinline__ uint64_t ref_mulmod_u64(uint64_t a, uint64_t b, const RefInvConst &p) {
    const uint64_t lo = a * b, hi = __umul64hi(a, b);
    const uint64_t q1 = (hi << (65 - p.k)) | (lo >> (p.k - 1));                        // x >> (k-1)  < 2^(k+1)
    const uint64_t q3 = (__umul64hi(q1, p.mu) << (63 - p.k)) | ((q1 * p.mu) >> (p.k + 1));   // q1 * mu >> (k+1)
    uint64_t r = lo - q3 * p.q;                                                         // x - q3*q in [0,3q)
    r = ref_csub_u64(r, p.q);
    return ref_csub_u64(r, p.q);
}

// GS stage J of a register pass over 2^LS coefficients: pairs x[g*2h + i], x[g*2h + i + h], h = 2^LS >> (J+1)
template <int LS, int J, bool VEC>
__device__ __forceinline__ void ref_istage_u64(uint64_t (&x)[1 << LS], const uint64_t *__restrict__ roots,
                                               const uint64_t *__restrict__ precons, uint32_t tbase, uint64_t q, uint64_t twice) {
    constexpr int half = (1 << LS) >> (J + 1);
    uint64_t W[1 << J], Wp[1 << J];
    ref_load_tw_u64<(1 << J), VEC>(W, Wp, roots, precons, tbase);
#pragma unroll
    for (int g = 0; g < (1 << J); g++)
#pragma unroll
        for (int i = 0; i < half; i++) ref_gs_bfly_u64(x[g * 2 * half + i], x[g * 2 * half + i + half], W[g], Wp[g], q, twice);
}

// ref_pass16_u64 run backwards: local stages J = 3 .. JLO, local stage J being stage s_first + (J - JFIRST) of the
// forward numbering (h = 2^that groups), twiddle index h + (t_hi << J) + g
template <bool VEC, int JFIRST, int JLO = JFIRST, int J = 3>
__device__ __forceinline__ void ref_ipass16_u64(uint64_t (&x)[16], const uint64_t *__restrict__ roots,
                                                const uint64_t *__restrict__ precons, uint32_t s_first, uint32_t t_hi, uint64_t q,
                                                uint64_t twice) {
    ref_istage_u64<4, J, VEC>(x, roots, precons, (1u << (s_first + J - JFIRST)) + (t_hi << J), q, twice);
    if constexpr (J > JLO) ref_ipass16_u64<VEC, JFIRST, JLO, J - 1>(x, roots, precons, s_first, t_hi, q, twice);
}

// ref_u64_frame_kernel's geometry (NT = N/32 threads, lg = log2(NT) + 5 coefficients per CTA, the 17-word-per-16 image,
// 16-coefficient register passes) with the passes in the opposite order: the frame is loaded into the image with coalesced
// reads (times `mul` when given), the first pass works on index bits 3..0, the middle passes move upward, and the last
// pass on the top four bits writes global memory at (k << lo) + vt, coalesced.  logn = lg: one CTA per frame, n^-1 folded
// into the last pass, results in [0,q).  logn = lg + 1 (N = 32768, split): two CTAs per frame, each running the first 14
// stages of its own half (the half is the top bit of every group index, as the forward's half_id); no stage before the
// last couples the halves, so each CTA reads and writes only its own half (in place is safe) and leaves it in [0,2q) for
// ref_u64_inv_last_stage_kernel.
// ref_u64_inv_frame_body is that kernel for its per-limb variant (ref_u64_rns_inv_frame_kernel); the single-modulus kernel
// keeps its own copy, as ref_fwd_u64_kernel does.  K supplies the modulus constants (RefInvOne, RefInvLimb).
//
// Where the inverse kernels take their modulus constants from.  One modulus (agx_ref_*): the kernel parameters, and the
// folded last-stage twiddle computed from the caller's table.
struct RefInvOne {
    RefInvConst p;
    const uint64_t *roots;
    __device__ __forceinline__ uint64_t q() const { return p.q; }
    __device__ __forceinline__ RefInvConst consts() const { return p; }
    __device__ __forceinline__ ulonglong2 fold() const { return ref_inv_fold(roots, p); }
};

template <int NT>
__host__ __device__ constexpr uint32_t ref_frame_lg() { return NT == 512 ? 14u : NT == 256 ? 13u : NT == 128 ? 12u : NT == 64 ? 11u : 10u; }

template <int NT, class K>
__device__ __forceinline__ void ref_u64_inv_frame_body(const uint64_t *in, const uint64_t *mul, uint64_t *out,
                                                       const uint64_t *__restrict__ roots, const uint64_t *__restrict__ precons,
                                                       const K &kc, uint32_t logn, uint32_t frame, uint32_t half_id) {
    extern __shared__ uint64_t img[];
    __shared__ ulonglong2 fold;
    constexpr bool VEC = AGX_U64_VECTW >= 2 || (AGX_U64_VECTW == 1 && NT >= 512);
    constexpr uint32_t lg = ref_frame_lg<NT>();
    constexpr uint32_t M = 1u << lg, vthreads = M >> 4;
    const uint32_t tid = threadIdx.x, split = logn - lg;
    if (split > 1) return;                                         // launch contract (never taken)
    const uint64_t q = kc.q(), twice = q << 1;
    const size_t base = ((size_t)frame << logn) + (size_t)half_id * M;
    if (!split && tid == 0) fold = kc.fold();                      // read after the barrier that ends the load

    uint64_t x[16];
    // ---- load (and the fused pointwise product): 16 coalesced reads in flight per thread, the forward's pass-0 pattern
    {
        constexpr uint32_t lo = lg - 4;
        constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = in[base + (k << lo) + vt];
            if (mul) {
                const RefInvConst p = kc.consts();
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = ref_mulmod_u64(x[k], mul[base + (k << lo) + vt], p);
            }
            uint64_t *s = img + vt + (vt >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
    }
    __syncthreads();
    // ---- first pass: bits 3..0, stages h = N/2 .. N/16 of this CTA's sub-transform
#pragma unroll 1
    for (uint32_t vt = tid; vt < vthreads; vt += NT) {
        uint64_t *s = img + vt * 17;
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = s[k];
        ref_ipass16_u64<VEC, 0>(x, roots, precons, lg - 4 + split, vt + (half_id << (lg - 4)), q, twice);
#pragma unroll
        for (int k = 0; k < 16; k++) s[k] = x[k];
    }
    __syncthreads();
    // ---- middle passes: the forward's windows (lo, jfirst) from the lowest up; the lowest may be partial
#pragma unroll
    for (int rem = ((int)lg - 9) % 4 + 1; rem <= (int)lg - 8; rem += 4) {
        const uint32_t lo = rem >= 4 ? (uint32_t)rem : 4u;
        const uint32_t jfirst = rem >= 4 ? 0u : (uint32_t)(4 - rem);
        const uint32_t stride = (1u << lo) + (1u << (lo - 4));
        const uint32_t s_first = lg - 4 - lo + jfirst;             // sub-transform stage of local stage jfirst
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint64_t *s = img + idx0 + (idx0 >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            const uint32_t sg = s_first + split, th = t_hi + (half_id << (s_first - jfirst));
            if (jfirst == 0) ref_ipass16_u64<VEC, 0>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 1) ref_ipass16_u64<VEC, 1>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 2) ref_ipass16_u64<VEC, 2>(x, roots, precons, sg, th, q, twice);
            else ref_ipass16_u64<VEC, 3>(x, roots, precons, sg, th, q, twice);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
        __syncthreads();
    }
    // ---- last pass: the top four bits, straight to global memory
    {
        constexpr uint32_t lo = lg - 4;
        constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
        uint64_t *dst = out + base;
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint64_t *s = img + vt + (vt >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            if (split) {
                ref_ipass16_u64<VEC, 0>(x, roots, precons, 1, half_id, q, twice);
            } else {
                ref_ipass16_u64<VEC, 0, 1>(x, roots, precons, 0, 0, q, twice);
                const ulonglong2 f = fold;
                const RefInvConst p = kc.consts();
#pragma unroll
                for (int i = 0; i < 8; i++) ref_gs_last_bfly_u64(x[i], x[i + 8], p, f);
            }
#pragma unroll
            for (int k = 0; k < 16; k++) dst[(k << lo) + vt] = x[k];
        }
    }
}

// TWIN: ref_u64_inv_frame_body is a copy of this kernel for the per-limb (RNS) variants; a fix here belongs there too (this copy is
// kept apart so that the single-modulus kernel keeps its SASS).
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_inv_frame_kernel(const uint64_t *in, const uint64_t *mul,   // may alias out
                                                                  uint64_t *out, const uint64_t *__restrict__ roots,
                                                                  const uint64_t *__restrict__ precons, RefInvConst p,
                                                                  uint32_t logn) {
    extern __shared__ uint64_t img[];
    __shared__ ulonglong2 fold;
    constexpr bool VEC = AGX_U64_VECTW >= 2 || (AGX_U64_VECTW == 1 && NT >= 512);
    constexpr uint32_t lg = (NT == 512 ? 14u : NT == 256 ? 13u : NT == 128 ? 12u : NT == 64 ? 11u : 10u);
    constexpr uint32_t M = 1u << lg, vthreads = M >> 4;
    const uint32_t tid = threadIdx.x, split = logn - lg;
    if (split > 1) return;                                         // launch contract (never taken)
    const uint32_t frame = split ? blockIdx.x >> 1 : blockIdx.x, half_id = split ? blockIdx.x & 1u : 0u;
    const uint64_t q = p.q, twice = q << 1;
    const size_t base = ((size_t)frame << logn) + (size_t)half_id * M;
    if (!split && tid == 0) fold = ref_inv_fold(roots, p);         // read after the barrier that ends the load

    uint64_t x[16];
    // ---- load (and the fused pointwise product): 16 coalesced reads in flight per thread, the forward's pass-0 pattern
    {
        constexpr uint32_t lo = lg - 4;
        constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = in[base + (k << lo) + vt];
            if (mul) {
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = ref_mulmod_u64(x[k], mul[base + (k << lo) + vt], p);
            }
            uint64_t *s = img + vt + (vt >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
    }
    __syncthreads();
    // ---- first pass: bits 3..0, stages h = N/2 .. N/16 of this CTA's sub-transform
#pragma unroll 1
    for (uint32_t vt = tid; vt < vthreads; vt += NT) {
        uint64_t *s = img + vt * 17;
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = s[k];
        ref_ipass16_u64<VEC, 0>(x, roots, precons, lg - 4 + split, vt + (half_id << (lg - 4)), q, twice);
#pragma unroll
        for (int k = 0; k < 16; k++) s[k] = x[k];
    }
    __syncthreads();
    // ---- middle passes: the forward's windows (lo, jfirst) from the lowest up; the lowest may be partial
#pragma unroll
    for (int rem = ((int)lg - 9) % 4 + 1; rem <= (int)lg - 8; rem += 4) {
        const uint32_t lo = rem >= 4 ? (uint32_t)rem : 4u;
        const uint32_t jfirst = rem >= 4 ? 0u : (uint32_t)(4 - rem);
        const uint32_t stride = (1u << lo) + (1u << (lo - 4));
        const uint32_t s_first = lg - 4 - lo + jfirst;             // sub-transform stage of local stage jfirst
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint64_t *s = img + idx0 + (idx0 >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            const uint32_t sg = s_first + split, th = t_hi + (half_id << (s_first - jfirst));
            if (jfirst == 0) ref_ipass16_u64<VEC, 0>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 1) ref_ipass16_u64<VEC, 1>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 2) ref_ipass16_u64<VEC, 2>(x, roots, precons, sg, th, q, twice);
            else ref_ipass16_u64<VEC, 3>(x, roots, precons, sg, th, q, twice);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
        __syncthreads();
    }
    // ---- last pass: the top four bits, straight to global memory
    {
        constexpr uint32_t lo = lg - 4;
        constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
        uint64_t *dst = out + base;
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint64_t *s = img + vt + (vt >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            if (split) {
                ref_ipass16_u64<VEC, 0>(x, roots, precons, 1, half_id, q, twice);
            } else {
                ref_ipass16_u64<VEC, 0, 1>(x, roots, precons, 0, 0, q, twice);
                const ulonglong2 f = fold;
#pragma unroll
                for (int i = 0; i < 8; i++) ref_gs_last_bfly_u64(x[i], x[i + 8], p, f);
            }
#pragma unroll
            for (int k = 0; k < 16; k++) dst[(k << lo) + vt] = x[k];
        }
    }
}

// N = 32768: the last stage (h = 1, pairs i and i + N/2) with n^-1 folded in and the reduction to [0,q), over frames
// whose halves ref_u64_inv_frame_kernel left in [0,2q).  Grid-stride, two pairs per thread and step (16-byte accesses).
__global__ void __launch_bounds__(256) ref_u64_inv_last_stage_kernel(uint64_t *data, const uint64_t *__restrict__ roots,
                                                                     RefInvConst p, uint32_t logn, size_t frames) {
    __shared__ ulonglong2 fold;
    if (threadIdx.x == 0) fold = ref_inv_fold(roots, p);
    __syncthreads();
    const ulonglong2 f = fold;
    const uint32_t hlog = logn - 2;                                // 2-pair units per half frame
    const size_t units = frames << hlog;
    for (size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x; u < units; u += (size_t)gridDim.x * blockDim.x) {
        const size_t i = ((u >> hlog) << logn) + ((u & ((1u << hlog) - 1)) << 1);
        ulonglong2 *lo = reinterpret_cast<ulonglong2 *>(data + i), *hi = reinterpret_cast<ulonglong2 *>(data + i + (1u << (logn - 1)));
        const ulonglong2 a = *lo, b = *hi;
        uint64_t u0 = a.x, u1 = a.y, v0 = b.x, v1 = b.y;
        ref_gs_last_bfly_u64(u0, v0, p, f);
        ref_gs_last_bfly_u64(u1, v1, p, f);
        *lo = make_ulonglong2(u0, u1);
        *hi = make_ulonglong2(v0, v1);
    }
}

// N < 1024: plain radix-2 GS, one CTA per frame, the frame in shared memory (in the manner of ref_fwd_u64_kernel)
template <class K>
__device__ __forceinline__ void ref_inv_u64_body(const uint64_t *in, const uint64_t *mul, uint64_t *out,
                                                 const uint64_t *__restrict__ roots, const uint64_t *__restrict__ precons,
                                                 const K &kc, uint32_t logn, uint32_t frame) {
    __shared__ uint64_t X[512];
    __shared__ ulonglong2 fold;
    const uint32_t N = 1u << logn;
    const size_t base = (size_t)frame * N;
    const RefInvConst p = kc.consts();
    const uint64_t q = p.q, twice = q << 1;
    if (threadIdx.x == 0) fold = kc.fold();
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x)
        X[i] = mul ? ref_mulmod_u64(in[base + i], mul[base + i], p) : in[base + i];
    __syncthreads();
    for (uint32_t h = N >> 1, tlog = 0; h >= 1; h >>= 1, tlog++) {        // butterfly distance 2^tlog
        for (uint32_t bf = threadIdx.x; bf < N / 2; bf += blockDim.x) {
            const uint32_t j = bf >> tlog, a0 = (j << (tlog + 1)) + (bf & ((1u << tlog) - 1)), a1 = a0 + (1u << tlog);
            uint64_t u = X[a0], v = X[a1];
            if (h == 1) ref_gs_last_bfly_u64(u, v, p, fold);
            else ref_gs_bfly_u64(u, v, __ldg(roots + h + j), __ldg(precons + h + j), q, twice);
            X[a0] = u; X[a1] = v;
        }
        __syncthreads();
    }
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) out[base + i] = X[i];
}

__global__ void __launch_bounds__(256) ref_inv_u64_kernel(const uint64_t *in, const uint64_t *mul, uint64_t *out,
                                                          const uint64_t *__restrict__ roots, const uint64_t *__restrict__ precons,
                                                          RefInvConst p, uint32_t logn) {
    ref_inv_u64_body(in, mul, out, roots, precons, RefInvOne{p, roots}, logn, blockIdx.x);
}

// ------------------------------------------------------------------------ u64 RNS batches ([B][L][N], agx_create64)
// The kernels above over L primes at once: frame f = b * L + l is limb l = f % L of polynomial b.  Each CTA derives its
// limb from its frame, offsets the library's tables ([L][N] words per table, the reference's order) by limb * N and reads
// its modulus constants from a per-limb array built at create time -- including the inverse's folded last-stage twiddle
// iroots[1] * n^-1, which the single-modulus kernels derive per CTA from the caller's table.  Arithmetic and geometry are
// the single-modulus kernels' (the same bodies), so every limb's result equals the single-modulus call's bit for bit.
struct RnsLimb64 {
    RefInvConst p;          // q, n^-1 and its companion, Barrett mu / k, reciprocal floor(2^(63+k) / q)
    ulonglong2 fold;        // iroots[1] * n^-1 mod q and floor(that * 2^64 / q)
    uint64_t psi, psi_inv;  // table bases (gen_tables64_kernel)
};

// The inverse's constants from one limb's entry: q is loaded once, the rest where it is used (the frame kernels run at
// the 128-register cap, so nothing is held in registers across the passes that the passes do not need).
struct RefInvLimb {
    const RnsLimb64 *lc;
    uint64_t q_;
    __device__ __forceinline__ uint64_t q() const { return q_; }
    __device__ __forceinline__ RefInvConst consts() const {
        RefInvConst p;
        p.q = q_;
        p.ninv = __ldg(&lc->p.ninv);
        p.ninv_p = __ldg(&lc->p.ninv_p);
        p.mu = __ldg(&lc->p.mu);
        p.recip = __ldg(&lc->p.recip);
        p.k = __ldg(&lc->p.k);
        return p;
    }
    __device__ __forceinline__ ulonglong2 fold() const { return __ldg(&lc->fold); }
};

// forward, N >= 1024 except N = 32768: one CTA per frame
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_rns_frame_kernel(const uint64_t *in, uint64_t *out,   // in may be out
                                                                  const uint64_t *__restrict__ roots,
                                                                  const uint64_t *__restrict__ precons,
                                                                  const RnsLimb64 *__restrict__ lc, uint32_t L, uint32_t logn) {
    const uint32_t frame = blockIdx.x, limb = frame % L;
    const size_t toff = (size_t)limb << logn;
    ref_u64_frame_body<NT>(in, in, out, roots + toff, precons + toff, __ldg(&lc[limb].p.q), logn, 0, frame, 0);
}

// forward, N = 32768: the two CTAs of a frame as a 2-CTA cluster (ref_u64_frame_body<PAIR>), in place or not
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(512, 1)
    ref_u64_rns_frame_pair_kernel(const uint64_t *in, uint64_t *out, const uint64_t *__restrict__ roots,
                                  const uint64_t *__restrict__ precons, const RnsLimb64 *__restrict__ lc, uint32_t L) {
    constexpr uint32_t logn = 15;
    const uint32_t frame = blockIdx.x >> 1, limb = frame % L;
    const size_t toff = (size_t)limb << logn;
    ref_u64_frame_body<512, true>(in, in, out, roots + toff, precons + toff, __ldg(&lc[limb].p.q), logn, 1, frame,
                                  blockIdx.x & 1u);
}

// inverse, N >= 1024 (two CTAs per frame and ref_u64_rns_inv_last_stage_kernel at N = 32768)
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_rns_inv_frame_kernel(const uint64_t *in, const uint64_t *mul,   // may alias out
                                                                      uint64_t *out, const uint64_t *__restrict__ roots,
                                                                      const uint64_t *__restrict__ precons,
                                                                      const RnsLimb64 *__restrict__ lc, uint32_t L,
                                                                      uint32_t logn) {
    const uint32_t split = logn - ref_frame_lg<NT>();
    const uint32_t frame = split ? blockIdx.x >> 1 : blockIdx.x, limb = frame % L;
    const size_t toff = (size_t)limb << logn;
    ref_u64_inv_frame_body<NT>(in, mul, out, roots + toff, precons + toff, RefInvLimb{lc + limb, __ldg(&lc[limb].p.q)}, logn,
                               frame, split ? blockIdx.x & 1u : 0u);
}

// N = 32768: the last inverse stage (ref_u64_inv_last_stage_kernel), each 2-pair unit with its own frame's limb
__global__ void __launch_bounds__(256) ref_u64_rns_inv_last_stage_kernel(uint64_t *data, const RnsLimb64 *__restrict__ lc,
                                                                         uint32_t L, uint32_t logn, size_t frames) {
    const uint32_t hlog = logn - 2;                                // 2-pair units per half frame
    const size_t units = frames << hlog;
    for (size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x; u < units; u += (size_t)gridDim.x * blockDim.x) {
        const RnsLimb64 *c = lc + (uint32_t)((u >> hlog) % L);
        const RefInvConst p = RefInvLimb{c, __ldg(&c->p.q)}.consts();
        const ulonglong2 f = __ldg(&c->fold);
        const size_t i = ((u >> hlog) << logn) + ((u & ((1u << hlog) - 1)) << 1);
        ulonglong2 *lo = reinterpret_cast<ulonglong2 *>(data + i), *hi = reinterpret_cast<ulonglong2 *>(data + i + (1u << (logn - 1)));
        const ulonglong2 a = *lo, b = *hi;
        uint64_t u0 = a.x, u1 = a.y, v0 = b.x, v1 = b.y;
        ref_gs_last_bfly_u64(u0, v0, p, f);
        ref_gs_last_bfly_u64(u1, v1, p, f);
        *lo = make_ulonglong2(u0, u1);
        *hi = make_ulonglong2(v0, v1);
    }
}

// N < 1024: the radix-2 kernels, one CTA per frame
__global__ void __launch_bounds__(1024) ref_fwd_u64_rns_kernel(const uint64_t *__restrict__ in, uint64_t *__restrict__ out,
                                                               const uint64_t *__restrict__ roots,
                                                               const uint64_t *__restrict__ precons,
                                                               const RnsLimb64 *__restrict__ lc, uint32_t L, uint32_t logn) {
    const uint32_t frame = blockIdx.x, limb = frame % L;
    const size_t toff = (size_t)limb << logn;
    ref_fwd_u64_body(in, in, out, roots + toff, precons + toff, __ldg(&lc[limb].p.q), logn, 1, frame);
}

__global__ void __launch_bounds__(256) ref_inv_u64_rns_kernel(const uint64_t *in, const uint64_t *mul, uint64_t *out,
                                                              const uint64_t *__restrict__ roots,
                                                              const uint64_t *__restrict__ precons,
                                                              const RnsLimb64 *__restrict__ lc, uint32_t L, uint32_t logn) {
    const uint32_t frame = blockIdx.x, limb = frame % L;
    const size_t toff = (size_t)limb << logn;
    ref_inv_u64_body(in, mul, out, roots + toff, precons + toff, RefInvLimb{lc + limb, __ldg(&lc[limb].p.q)}, logn, frame);
}

// c = a + b | a - b | a * b | c + a * b modulo each limb's prime over [B][L][N] words (operands < q, results in [0,q)),
// two words per 16-byte access (N >= 4, so an access never straddles two limbs); grid-stride
template <int OP>
__global__ void __launch_bounds__(256) elementwise64_kernel(ulonglong2 *c2, const ulonglong2 *a2, const ulonglong2 *b2,
                                                            const RnsLimb64 *__restrict__ lc, uint32_t L, uint32_t logn,
                                                            size_t total2) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total2; i += (size_t)gridDim.x * blockDim.x) {
        const RnsLimb64 *l = lc + (uint32_t)(((i << 1) >> logn) % L);
        const uint64_t q = __ldg(&l->p.q);
        const ulonglong2 a = a2[i], b = b2[i];
        uint64_t r[2];
        const uint64_t av[2] = {a.x, a.y}, bv[2] = {b.x, b.y};
        if constexpr (OP == EW_ADD) {
#pragma unroll
            for (int j = 0; j < 2; j++) r[j] = ref_csub_u64(av[j] + bv[j], q);
        } else if constexpr (OP == EW_SUB) {
#pragma unroll
            for (int j = 0; j < 2; j++) r[j] = ref_csub_u64(av[j] + q - bv[j], q);
        } else {
            const RefInvConst p = RefInvLimb{l, q}.consts();
#pragma unroll
            for (int j = 0; j < 2; j++) r[j] = ref_mulmod_u64(av[j], bv[j], p);
            if constexpr (OP == EW_MAC) {
                const ulonglong2 c = c2[i];
                r[0] = ref_csub_u64(r[0] + c.x, q);
                r[1] = ref_csub_u64(r[1] + c.y, q);
            }
        }
        c2[i] = make_ulonglong2(r[0], r[1]);
    }
}

// The library's u64 tables: one thread per (direction, limb, k), w = base^bitrev(k) mod q (base = psi forward, psi^-1
// inverse) by square-and-multiply with the exact Barrett product, and its Shoup companion floor(w * 2^64 / q) by the
// reciprocal estimate and correction of ref_inv_fold (a 128-bit division compiles to a bit-serial loop).  The order is
// the reference's (ntt.cpp:298-300), which the kernels above read directly.  tab: [4][L][n] = forward roots, forward
// companions, inverse roots, inverse companions.
__global__ void __launch_bounds__(256) gen_tables64_kernel(uint64_t *__restrict__ tab, const RnsLimb64 *__restrict__ lc,
                                                           uint32_t L, uint32_t logn) {
    const uint32_t n = 1u << logn;
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= 2u * L * n) return;
    const uint32_t k = gid & (n - 1), limb = (gid >> logn) % L;
    const bool inverse = gid >= L * n;
    const RefInvConst p = lc[limb].p;
    const uint32_t e = __brev(k) >> (32 - logn);
    uint64_t w = 1, b = inverse ? lc[limb].psi_inv : lc[limb].psi;
    for (uint32_t i = 0; i < logn; i++) {
        if ((e >> i) & 1) w = ref_mulmod_u64(w, b, p);
        b = ref_mulmod_u64(b, b, p);
    }
    const uint64_t wp = ref_shoup_companion(w, p);
    const size_t at = (size_t)(inverse ? 2 : 0) * L * n + (size_t)limb * n + k;
    tab[at] = w;
    tab[at + (size_t)L * n] = wp;
}

// ------------------------------------------------------------------ u64 RNS rescale ([B][L][N] -> [B][L-1][N])
// Division by the last prime q_L' = q_{L-1} with rounding (agx_rescale64): with h = floor(q_L' / 2) and, per coefficient,
// u = (x_{L-1} + h) mod q_L', every other limb i < L - 1 becomes
//   y_i = (x_i - (u - h)) * q_L'^-1  mod q_i,
// the residues of round-half-up(X / q_L') for the CRT value X of the L residues.  u < q_L' may exceed q_i (the primes
// come in any order): it is reduced by a Shoup product with 1, whose companion floor(2^64 / q_i) brings ANY 64-bit word
// into [0, 2q_i) -- unlike the exact Barrett product (ref_mulmod_u64), which needs its argument below 2^(2k_i) and so
// would fail for a small q_i beside a 62-bit q_L'.  Per-limb constants, built at create time (agx_create64, L >= 2) in
// an array of their own; q_L' and h are the same for every limb and go in as kernel parameters.
struct RescaleLimb64 {
    uint64_t q;              // q_i
    uint64_t one_p;          // floor(2^64 / q_i): Shoup companion of 1
    uint64_t h;              // h mod q_i
    uint64_t qinv, qinv_p;   // q_L'^-1 mod q_i and floor(qinv * 2^64 / q_i)
};

// The forward's input from a word t < q_L' of limb L - 1 in coefficient form: u = (t + h) mod q_L', returned as a word
// congruent to u - h (mod q_i) in (q_i, 4q_i), the forward transform's input range.  twice_minus_h = 2q_i - (h mod q_i).
__device__ __forceinline__ uint64_t rescale_lift_u64(uint64_t t, uint64_t qlast, uint64_t h, uint64_t one_p, uint64_t q,
                                                     uint64_t twice_minus_h) {
    return ref_shoup_u64(ref_csub_u64(t + h, qlast), 1, one_p, q) + twice_minus_h;
}

// (x - r) * q_L'^-1 mod q_i in [0, q_i), for x < 2q_i and r < 2q_i   (x + 2q_i - r < 4q_i < 2^64; Shoup gives [0, 2q_i))
__device__ __forceinline__ uint64_t rescale_finish_u64(uint64_t x, uint64_t r, uint64_t q, uint64_t qinv, uint64_t qinv_p) {
    return ref_csub_u64(ref_shoup_u64(x + (q << 1) - r, qinv, qinv_p, q), q);
}

// Coefficient form: grid-stride over the 16-byte pairs of one limb row of every polynomial.  A thread loads its pair of
// x_{L-1} once, forms u, and then walks the L - 1 output limbs: B*L*n words read, B*(L-1)*n written, nothing else.
__global__ void __launch_bounds__(256) rescale64_coeff_kernel(ulonglong2 *__restrict__ out2, const ulonglong2 *__restrict__ in2,
                                                              const RescaleLimb64 *__restrict__ rc, uint64_t qlast, uint64_t h,
                                                              uint32_t L, uint32_t logn, size_t pairs) {
    const uint32_t hlog = logn - 1;                                // pairs per row
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < pairs; p += (size_t)gridDim.x * blockDim.x) {
        const size_t b = p >> hlog, j = p & ((1u << hlog) - 1);
        const ulonglong2 *row = in2 + ((b * L) << hlog) + j;
        ulonglong2 *dst = out2 + ((b * (L - 1)) << hlog) + j;
        const ulonglong2 xl = row[(size_t)(L - 1) << hlog];
        const uint64_t u0 = ref_csub_u64(xl.x + h, qlast), u1 = ref_csub_u64(xl.y + h, qlast);
        for (uint32_t i = 0; i < L - 1; i++) {
            const RescaleLimb64 *c = rc + i;
            const uint64_t q = __ldg(&c->q), one_p = __ldg(&c->one_p), qh = q - __ldg(&c->h);
            const uint64_t qinv = __ldg(&c->qinv), qinv_p = __ldg(&c->qinv_p);
            const ulonglong2 x = row[(size_t)i << hlog];
            // r = (u mod q_i) + q_i - (h mod q_i), in (0, 2q_i)
            const uint64_t r0 = ref_csub_u64(ref_shoup_u64(u0, 1, one_p, q), q) + qh;
            const uint64_t r1 = ref_csub_u64(ref_shoup_u64(u1, 1, one_p, q), q) + qh;
            dst[(size_t)i << hlog] = make_ulonglong2(rescale_finish_u64(x.x, r0, q, qinv, qinv_p),
                                                     rescale_finish_u64(x.y, r1, q, qinv, qinv_p));
        }
    }
}

// Evaluation form, step 1: the inverse transform of limb L - 1 of every polynomial into the contiguous scratch [B][n]
// (ref_u64_inv_frame_body / ref_inv_u64_body on pointers already offset to the polynomial's last limb and to its scratch
// row, frame 0).  roots / precons: the inverse table of limb L - 1; last = lc + L - 1.  At N = 32768 the halves are left
// in [0,2q) for ref_u64_rns_inv_last_stage_kernel, run on the scratch as a 1-limb batch of that limb.
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_rescale_inv_frame_kernel(const uint64_t *in, uint64_t *scratch,
                                                                          const uint64_t *__restrict__ roots,
                                                                          const uint64_t *__restrict__ precons,
                                                                          const RnsLimb64 *__restrict__ last, uint32_t L,
                                                                          uint32_t logn) {
    const uint32_t split = logn - ref_frame_lg<NT>();
    const size_t b = split ? blockIdx.x >> 1 : blockIdx.x;
    ref_u64_inv_frame_body<NT>(in + ((b * L + L - 1) << logn), nullptr, scratch + (b << logn), roots, precons,
                               RefInvLimb{last, __ldg(&last->p.q)}, logn, 0, split ? blockIdx.x & 1u : 0u);
}

__global__ void __launch_bounds__(256) ref_inv_u64_rescale_kernel(const uint64_t *in, uint64_t *scratch,
                                                                  const uint64_t *__restrict__ roots,
                                                                  const uint64_t *__restrict__ precons,
                                                                  const RnsLimb64 *__restrict__ last, uint32_t L, uint32_t logn) {
    const size_t b = blockIdx.x;
    ref_inv_u64_body(in + ((b * L + L - 1) << logn), nullptr, scratch + (b << logn), roots, precons,
                     RefInvLimb{last, __ldg(&last->p.q)}, logn, 0);
}

// Evaluation form, step 2: the forward transform of r_i = (u - h) mod q_i under limb i's tables, with its input computed
// on the fly from the scratch row of polynomial b and its output merged with the caller's spectrum in the store:
//   out[b][i] = (x_hat_i - NTT_i(r_i)) * q_L'^-1  mod q_i.
// Frame f < B * (L - 1) is limb i = f mod (L - 1) of polynomial b = f / (L - 1).  roots / precons: the library's forward
// tables, offset here by i * N.
// TWIN: a copy of ref_u64_frame_body (split = 1 at N = 32768: two CTAs per frame, each reading both halves of the
// scratch row for stage 0) with that prologue in pass 0 and that epilogue in the final store; a fix to the transform
// belongs in both.  The output is a separate buffer from both inputs, so the split frame needs no cluster barrier.
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_rescale_fwd_kernel(const uint64_t *in, const uint64_t *scratch,
                                                                    uint64_t *out, const uint64_t *__restrict__ roots,
                                                                    const uint64_t *__restrict__ precons,
                                                                    const RescaleLimb64 *__restrict__ rc, uint64_t qlast,
                                                                    uint64_t h, uint32_t L, uint32_t logn) {
    extern __shared__ uint64_t img[];
    constexpr bool VEC = AGX_U64_VECTW >= 2 || (AGX_U64_VECTW == 1 && NT >= 512);   // 16-byte twiddle pairs
    const uint32_t tid = threadIdx.x;
    constexpr uint32_t lg = ref_frame_lg<NT>();
    constexpr uint32_t M = 1u << lg, vthreads = M >> 4;
    const uint32_t split = logn - lg;
    if (split > 1) return;                                         // launch contract (never taken)
    const uint32_t frame = split ? blockIdx.x >> 1 : blockIdx.x, half_id = split ? blockIdx.x & 1u : 0u;
    const uint32_t limb = frame % (L - 1), b = frame / (L - 1);
    roots += (size_t)limb << logn;
    precons += (size_t)limb << logn;
    const RescaleLimb64 *c = rc + limb;
    const uint64_t q = __ldg(&c->q), twice = q << 1;
    const uint64_t *src = scratch + ((size_t)b << logn);           // both halves of the frame come from the scratch row
    {
        // the epilogue's operand x_hat_i towards L2 while the transform runs: read only after the last pass, it would
        // otherwise cost an HBM round trip at a point where this CTA has nothing else to overlap with it
        const uint64_t *xin = in + (((size_t)b * L + limb) << logn) + (size_t)half_id * M;
        for (uint32_t l = tid; l < M / 16; l += NT) asm volatile("prefetch.global.L2 [%0];" ::"l"(xin + 16 * l));
    }
    uint64_t x[16];

    // ---- pass 0: stages (split ..) on index bits [lg-4, lg), coefficients from the scratch row through the prologue
    {
        constexpr uint32_t lo = lg - 4;
        const uint64_t one_p = __ldg(&c->one_p), th = twice - __ldg(&c->h);
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            if (split) {
                // stage 0 of the 32768-point frame, this CTA keeping only its half (ntt.cpp:331-369 with roots[1])
                const uint64_t W = __ldg(roots + 1), Wp = __ldg(precons + 1);
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    uint64_t a = rescale_lift_u64(src[i], qlast, h, one_p, q, th);
                    uint64_t bb = rescale_lift_u64(src[M + i], qlast, h, one_p, q, th);
                    ref_bfly_u64(a, bb, W, Wp, q, twice);
                    x[k] = half_id ? bb : a;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    x[k] = rescale_lift_u64(src[i], qlast, h, one_p, q, th);
                }
            }
            // this CTA's sub-transform: stage s of it is global stage s + split, group offset half_id << s
            // (roots index = 2^(s+split) + (half_id << s) + local group)
            ref_pass16_u64<VEC, 0>(x, roots, precons, split, half_id, q, twice);
            uint64_t *s = img + vt + (vt >> 4);
            constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
    }
    __syncthreads();
    // ---- middle passes: index bits from lg-5 down to 4, four at a time (the last one may cover fewer)
    uint32_t s_done = 4;                                           // stages of the sub-transform finished so far
#pragma unroll
    for (int rem = (int)lg - 8; rem > 0; rem -= 4) {
        const uint32_t lo = rem >= 4 ? (uint32_t)rem : 4u;
        const uint32_t jfirst = rem >= 4 ? 0u : (uint32_t)(4 - rem);
        const uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint64_t *s = img + idx0 + (idx0 >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            // twiddle index: 2^(s+split) + ((half_id << s) + group) with group = (t_hi << j) + g at local stage j
            const uint32_t sg = s_done + split;                    // global stage of the first active local stage
            const uint32_t th = t_hi + (half_id << (s_done - jfirst));   // the CTA's half as the top bit of the group index
            if (jfirst == 0) ref_pass16_u64<VEC, 0>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 1) ref_pass16_u64<VEC, 1>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 2) ref_pass16_u64<VEC, 2>(x, roots, precons, sg, th, q, twice);
            else ref_pass16_u64<VEC, 3>(x, roots, precons, sg, th, q, twice);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
        s_done += 4 - jfirst;
        __syncthreads();
    }
    // ---- final pass: bits 3..0 (16 consecutive coefficients), reduction to [0,q) (ntt.cpp:377-393)
#pragma unroll 1
    for (uint32_t vt = tid; vt < vthreads; vt += NT) {
        uint64_t *s = img + vt * 17;
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = s[k];
        ref_pass16_u64<VEC, 0>(x, roots, precons, s_done + split, vt + (half_id << s_done), q, twice);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            s[k] = ref_csub_u64(ref_csub_u64(x[k], twice), q);
        }
    }
    __syncthreads();
    // ---- epilogue: merge with the caller's spectrum of limb i and scale by q_L'^-1; 16 reads of x_hat_i in flight per
    // thread (M = 32 * NT: two rounds)
    const uint64_t qinv = __ldg(&c->qinv), qinv_p = __ldg(&c->qinv_p);
    const uint64_t *xin = in + (((size_t)b * L + limb) << logn) + (size_t)half_id * M;
    uint64_t *dst = out + ((size_t)frame << logn) + (size_t)half_id * M;
#pragma unroll 1
    for (uint32_t i0 = tid; i0 < M; i0 += 16 * NT) {
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = xin[i0 + k * NT];
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const uint32_t i = i0 + k * NT;
            dst[i] = rescale_finish_u64(x[k], img[i + (i >> 4)], q, qinv, qinv_p);
        }
    }
}

// N < 1024: the same on the radix-2 forward.  TWIN: a copy of ref_fwd_u64_body (shared-memory work array) with the
// rescale's prologue on the load and its epilogue on the store; a fix to the transform belongs in both.
__global__ void __launch_bounds__(1024) ref_fwd_u64_rescale_kernel(const uint64_t *__restrict__ in,
                                                                   const uint64_t *__restrict__ scratch,
                                                                   uint64_t *__restrict__ out, const uint64_t *__restrict__ roots,
                                                                   const uint64_t *__restrict__ precons,
                                                                   const RescaleLimb64 *__restrict__ rc, uint64_t qlast,
                                                                   uint64_t h, uint32_t L, uint32_t logn) {
    extern __shared__ uint64_t s64[];
    const uint32_t N = 1u << logn;
    const uint32_t frame = blockIdx.x, limb = frame % (L - 1), b = frame / (L - 1);
    roots += (size_t)limb << logn;
    precons += (size_t)limb << logn;
    const RescaleLimb64 *c = rc + limb;
    const uint64_t q = __ldg(&c->q), twice = q << 1;
    uint64_t *X = s64;
    {
        const uint64_t *src = scratch + ((size_t)b << logn);
        const uint64_t one_p = __ldg(&c->one_p), th = twice - __ldg(&c->h);
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x)
            X[i] = rescale_lift_u64(src[i], qlast, h, one_p, q, th);
    }
    __syncthreads();
    uint32_t tlog = logn - 1;
    for (uint32_t m = 1; m < N; m <<= 1, tlog--) {
        const bool last = (m == N / 2);
        for (uint32_t bf = threadIdx.x; bf < N / 2; bf += blockDim.x) {
            const uint32_t i = bf >> tlog, j = bf & ((1u << tlog) - 1);
            const uint32_t a0 = (i << (tlog + 1)) + j, a1 = a0 + (1u << tlog);
            const uint64_t W = roots[m + i], Wp = precons[m + i];
            uint64_t tx = X[a0];
            if (tx >= twice) tx -= twice;
            const uint64_t a = X[a1];
            const uint64_t c1 = __umul64hi(a, Wp);
            const uint64_t Q = W * a - c1 * q;
            uint64_t o0 = tx + Q, o1 = tx + twice - Q;
            if (last) {
                if (o0 >= twice) o0 -= twice;
                if (o0 >= q) o0 -= q;
                if (o1 >= twice) o1 -= twice;
                if (o1 >= q) o1 -= q;
            }
            X[a0] = o0; X[a1] = o1;
        }
        __syncthreads();
    }
    const uint64_t qinv = __ldg(&c->qinv), qinv_p = __ldg(&c->qinv_p);
    const uint64_t *xin = in + (((size_t)b * L + limb) << logn);
    uint64_t *dst = out + ((size_t)frame << logn);
    for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) dst[i] = rescale_finish_u64(xin[i], X[i], q, qinv, qinv_p);
}

// ------------------------------------------------------- u64 RNS basis conversion (ModUp / ModDown over [B][L][N])
// Exact conversions between sub-bases of the context's primes by mixed-radix conversion (MRC), no floating point.  For m
// source primes p_0 .. p_{m-1} (contiguous limbs s0 .. s0 + m - 1, product S) and h = (S - 1) / 2, per coefficient:
//   1. y_t = (x_t + h) mod p_t;
//   2. digits d_0 = y_0, d_t = (..((y_t - d_0) p_0^-1 - d_1) p_1^-1 .. - d_{t-1}) p_{t-1}^-1 mod p_t, so that
//      V = (X + h) mod S = sum_t d_t prod_{j<t} p_j exactly (m(m-1)/2 Shoup products);
//   3. per target prime q_i, Horner: T_i = V mod q_i = (..(d_{m-1} p_{m-2} + d_{m-2}) p_{m-3} + ..) p_0 + d_0 mod q_i
//      (m - 1 Shoup products, and one more with 1 that reduces the sum);
//   4. ModUp: out_i = T_i - h mod q_i, the centred lift of the source residues.  ModDown (sources = the last k limbs,
//      S = P): out_i = (x_i + h - T_i) P^-1 mod q_i = floor((X + h) / P) mod q_i.
// A Shoup product accepts any 64-bit word and returns [0, 2q), so Horner adds the digits (< p_t < 2^62) unreduced: the
// sum stays below 2q_i + 2^62 < 2^64.  In step 2, d_j < 2^62 may exceed p_t: it is subtracted from y + big_t, big_t the
// largest multiple of p_t not above 2^63 (> 2^62 > d_j), and the sum, below 2p_t + 2^63 < 2^64, goes into the product.
constexpr uint32_t kBasisMaxSrc = 16;        // m <= 16: a coefficient's digits stay in registers (agx_modup64 / moddown64)
constexpr uint32_t kBasisMaxLimbs = 64;      // agx_create64's limit on L

struct BasisLimb64 {
    uint64_t q;              // q_i
    uint64_t one_p;          // floor(2^64 / q_i): Shoup companion of 1
    uint64_t big;            // q_i * floor(2^63 / q_i)
};

// entry [i][j] of the L x L array that follows the L BasisLimb64 entries: constants modulo q_i of prime q_j
struct BasisPair64 {
    uint64_t w, w_p;         // q_j mod q_i and floor(w * 2^64 / q_i)
    uint64_t inv, inv_p;     // q_j^-1 mod q_i and its companion (0 when q_j = q_i)
};

// The per-call constants, passed by value as a kernel parameter (at most ~1.5 KB): nothing is uploaded per call.
struct BasisCall64 {
    uint32_t L, logn;
    uint32_t s0, m;          // source limbs s0 .. s0 + m - 1
    uint32_t ntgt;           // target limbs: t < s0 is limb t, t >= s0 is limb t + m
    uint32_t lift;           // 1: the forward's scratch rows hold y_0 - h ... (m = 1, no digits kernel): add h first
    uint64_t h[kBasisMaxLimbs];                           // h mod q_i
    uint64_t pinv[kBasisMaxLimbs], pinv_p[kBasisMaxLimbs]; // ModDown: P^-1 mod q_i and its companion
};

__device__ __forceinline__ uint32_t basis_target_limb(const BasisCall64 &cp, uint32_t t) { return t < cp.s0 ? t : t + cp.m; }

// steps 1 and 2 on W lanes: d[t][w] = x_t (reduced) in, digit t out, for t < m
template <int W>
__device__ __forceinline__ void basis_digits_u64(uint64_t (&d)[kBasisMaxSrc][W], const BasisLimb64 *__restrict__ bl,
                                                 const BasisPair64 *__restrict__ pr, const BasisCall64 &cp) {
#pragma unroll
    for (uint32_t t = 0; t < kBasisMaxSrc; t++) {
        if (t < cp.m) {
            const uint32_t lt = cp.s0 + t;
            const uint64_t p = __ldg(&bl[lt].q), big = __ldg(&bl[lt].big), h = cp.h[lt];
#pragma unroll
            for (int w = 0; w < W; w++) d[t][w] = ref_csub_u64(d[t][w] + h, p);
#pragma unroll
            for (uint32_t j = 0; j < t; j++) {
                const BasisPair64 *c = pr + (size_t)lt * cp.L + cp.s0 + j;
                const uint64_t v = __ldg(&c->inv), vp = __ldg(&c->inv_p);
#pragma unroll
                for (int w = 0; w < W; w++) d[t][w] = ref_shoup_u64(d[t][w] + big - d[j][w], v, vp, p);
            }
#pragma unroll
            for (int w = 0; w < W; w++) d[t][w] = ref_csub_u64(d[t][w], p);
        }
    }
}

// step 3 on W lanes for target limb i: T_i in [0, 2q_i)
template <int W>
__device__ __forceinline__ void basis_horner_u64(uint64_t (&T)[W], const uint64_t (&d)[kBasisMaxSrc][W],
                                                 const BasisPair64 *__restrict__ row, uint64_t q, uint64_t one_p,
                                                 const BasisCall64 &cp) {
#pragma unroll
    for (int w = 0; w < W; w++) T[w] = 0;
#pragma unroll
    for (int t = kBasisMaxSrc - 1; t >= 0; t--) {
        if ((uint32_t)t < cp.m) {
            if ((uint32_t)t + 1 < cp.m) {
                const uint64_t v = __ldg(&row[cp.s0 + t].w), vp = __ldg(&row[cp.s0 + t].w_p);
#pragma unroll
                for (int w = 0; w < W; w++) T[w] = ref_shoup_u64(T[w], v, vp, q);
            }
#pragma unroll
            for (int w = 0; w < W; w++) T[w] += d[t][w];
        }
    }
#pragma unroll
    for (int w = 0; w < W; w++) T[w] = ref_shoup_u64(T[w], 1, one_p, q);
}

// Coefficient form, one launch: grid-stride over the 16-byte pairs of one limb row of every polynomial.  A thread reads
// its m source pairs once, forms the digits, then walks the target limbs.  DOWN: in [B][L][n] -> out [B][L-m][n];
// else in [B][m][n] -> out [B][L][n], the source words written through to limbs s0 .. s0 + m - 1.
template <bool DOWN>
__global__ void __launch_bounds__(256) basis64_coeff_kernel(ulonglong2 *__restrict__ out2, const ulonglong2 *__restrict__ in2,
                                                            const BasisLimb64 *__restrict__ bl,
                                                            const BasisPair64 *__restrict__ pr, const __grid_constant__ BasisCall64 cp,
                                                            size_t pairs) {
    const uint32_t hlog = cp.logn - 1;                             // pairs per row
    const uint32_t inL = DOWN ? cp.L : cp.m, outL = DOWN ? cp.L - cp.m : cp.L, src0 = DOWN ? cp.s0 : 0;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < pairs; p += (size_t)gridDim.x * blockDim.x) {
        const size_t b = p >> hlog, j = p & ((1u << hlog) - 1);
        const ulonglong2 *row = in2 + ((b * inL) << hlog) + j;
        ulonglong2 *dst = out2 + ((b * outL) << hlog) + j;
        uint64_t d[kBasisMaxSrc][2];
#pragma unroll
        for (uint32_t t = 0; t < kBasisMaxSrc; t++) {
            if (t < cp.m) {
                const ulonglong2 x = row[(size_t)(src0 + t) << hlog];
                d[t][0] = x.x;
                d[t][1] = x.y;
                if (!DOWN) dst[(size_t)(cp.s0 + t) << hlog] = x;
            }
        }
        basis_digits_u64<2>(d, bl, pr, cp);
        for (uint32_t t = 0; t < cp.ntgt; t++) {
            const uint32_t i = basis_target_limb(cp, t);
            const uint64_t q = __ldg(&bl[i].q), one_p = __ldg(&bl[i].one_p);
            uint64_t T[2];
            basis_horner_u64<2>(T, d, pr + (size_t)i * cp.L, q, one_p, cp);
            const uint64_t h = cp.h[i];
            if (DOWN) {
                const ulonglong2 x = row[(size_t)i << hlog];
                const uint64_t xh0 = x.x + h + (q << 1), xh1 = x.y + h + (q << 1);   // < 4q_i; T < 2q_i
                dst[(size_t)i << hlog] = make_ulonglong2(
                    ref_csub_u64(ref_shoup_u64(xh0 - T[0], cp.pinv[i], cp.pinv_p[i], q), q),
                    ref_csub_u64(ref_shoup_u64(xh1 - T[1], cp.pinv[i], cp.pinv_p[i], q), q));
            } else {
                dst[(size_t)i << hlog] = make_ulonglong2(ref_csub_u64(ref_csub_u64(T[0], q) + q - h, q),
                                                         ref_csub_u64(ref_csub_u64(T[1], q) + q - h, q));
            }
        }
    }
}

// Evaluation form, step 2 (m >= 2): the scratch [B][m][n] of source residues in coefficient form becomes, in place, the
// m rows of mixed-radix digits of (X + h) mod S.  Grid-stride over 16-byte pairs.
__global__ void __launch_bounds__(256) basis64_digits_kernel(ulonglong2 *scr2, const BasisLimb64 *__restrict__ bl,
                                                             const BasisPair64 *__restrict__ pr, const __grid_constant__ BasisCall64 cp,
                                                             size_t pairs) {
    const uint32_t hlog = cp.logn - 1;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < pairs; p += (size_t)gridDim.x * blockDim.x) {
        const size_t b = p >> hlog, j = p & ((1u << hlog) - 1);
        ulonglong2 *row = scr2 + ((b * cp.m) << hlog) + j;
        uint64_t d[kBasisMaxSrc][2];
#pragma unroll
        for (uint32_t t = 0; t < kBasisMaxSrc; t++) {
            if (t < cp.m) {
                const ulonglong2 x = row[(size_t)t << hlog];
                d[t][0] = x.x;
                d[t][1] = x.y;
            }
        }
        basis_digits_u64<2>(d, bl, pr, cp);
#pragma unroll
        for (uint32_t t = 0; t < kBasisMaxSrc; t++)
            if (t < cp.m) row[(size_t)t << hlog] = make_ulonglong2(d[t][0], d[t][1]);
    }
}

// Evaluation form, step 1 of ModDown: the inverse of the last k limbs of every polynomial into the contiguous scratch
// [B][k][n] -- ref_u64_rescale_inv_frame_kernel / ref_inv_u64_rescale_kernel from "the last limb" to "the last k limbs":
// frame f is limb L - k + f mod k of polynomial f / k.  At N = 32768 the halves are left in [0,2q) for
// ref_u64_rns_inv_last_stage_kernel, run on the scratch as a k-limb batch of those limbs.
template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_basis_inv_frame_kernel(const uint64_t *in, uint64_t *scratch,
                                                                        const uint64_t *__restrict__ roots,
                                                                        const uint64_t *__restrict__ precons,
                                                                        const RnsLimb64 *__restrict__ lc, uint32_t L,
                                                                        uint32_t k, uint32_t logn) {
    const uint32_t split = logn - ref_frame_lg<NT>();
    const size_t f = split ? blockIdx.x >> 1 : blockIdx.x, b = f / k;
    const uint32_t limb = L - k + (uint32_t)(f % k);
    const size_t toff = (size_t)limb << logn;
    ref_u64_inv_frame_body<NT>(in + ((b * L + limb) << logn), nullptr, scratch + (f << logn), roots + toff, precons + toff,
                               RefInvLimb{lc + limb, __ldg(&lc[limb].p.q)}, logn, 0, split ? blockIdx.x & 1u : 0u);
}

__global__ void __launch_bounds__(256) ref_inv_u64_basis_kernel(const uint64_t *in, uint64_t *scratch,
                                                                const uint64_t *__restrict__ roots,
                                                                const uint64_t *__restrict__ precons,
                                                                const RnsLimb64 *__restrict__ lc, uint32_t L, uint32_t k,
                                                                uint32_t logn) {
    const size_t f = blockIdx.x, b = f / k;
    const uint32_t limb = L - k + (uint32_t)(f % k);
    const size_t toff = (size_t)limb << logn;
    ref_inv_u64_body(in + ((b * L + limb) << logn), nullptr, scratch + (f << logn), roots + toff, precons + toff,
                     RefInvLimb{lc + limb, __ldg(&lc[limb].p.q)}, logn, 0);
}

// The forward's input at coefficient j from the m scratch rows src[t * n + j] of one polynomial: T_i - h mod q_i as a
// word in (0, 4q_i), the forward transform's input range.  Rows hold the digits (m >= 2), or y_0 - h when cp.lift.
__device__ __forceinline__ uint64_t basis_lift_u64(const uint64_t *src, uint32_t j, const BasisLimb64 *__restrict__ bl,
                                                   const BasisPair64 *__restrict__ row, const BasisCall64 &cp, uint64_t q,
                                                   uint64_t one_p, uint64_t twice_minus_h) {
    const uint32_t n = 1u << cp.logn;
    uint64_t T = src[(size_t)(cp.m - 1) * n + j];
    if (cp.lift) T = ref_csub_u64(T + cp.h[cp.s0], __ldg(&bl[cp.s0].q));
    for (int t = (int)cp.m - 2; t >= 0; t--)
        T = ref_shoup_u64(T, __ldg(&row[cp.s0 + t].w), __ldg(&row[cp.s0 + t].w_p), q) + src[(size_t)t * n + j];
    return ref_shoup_u64(T, 1, one_p, q) + twice_minus_h;
}

// Evaluation form, step 3: the forward transform of T_i - h under target limb i's tables, its input computed on the fly
// from the digit rows of polynomial b.  Frame f < B * ntgt is target t = f mod ntgt of polynomial b = f / ntgt.
// DOWN: out[b][i] = (x_hat_i - NTT_i(T_i - h)) * P^-1 mod q_i, merged with the caller's spectrum in the store;
// else: out[b][i] = NTT_i(T_i - h), out being [B][L][n].
// TWIN: a copy of ref_u64_frame_body (split = 1 at N = 32768: two CTAs per frame, each reading both halves of the
// scratch rows for stage 0) with that prologue in pass 0 and that epilogue in the final store, as
// ref_u64_rescale_fwd_kernel is; a fix to the transform belongs in all three.
template <int NT, bool DOWN>
__global__ void __launch_bounds__(NT, 512 / NT) ref_u64_basis_fwd_kernel(const uint64_t *in, const uint64_t *scratch,
                                                                  uint64_t *out, const uint64_t *__restrict__ roots,
                                                                  const uint64_t *__restrict__ precons,
                                                                  const BasisLimb64 *__restrict__ bl,
                                                                  const BasisPair64 *__restrict__ pr, const __grid_constant__ BasisCall64 cp) {
    extern __shared__ uint64_t img[];
    constexpr bool VEC = AGX_U64_VECTW >= 2 || (AGX_U64_VECTW == 1 && NT >= 512);   // 16-byte twiddle pairs
    const uint32_t tid = threadIdx.x, logn = cp.logn;
    constexpr uint32_t lg = ref_frame_lg<NT>();
    constexpr uint32_t M = 1u << lg, vthreads = M >> 4;
    const uint32_t split = logn - lg;
    if (split > 1) return;                                         // launch contract (never taken)
    const uint32_t frame = split ? blockIdx.x >> 1 : blockIdx.x, half_id = split ? blockIdx.x & 1u : 0u;
    const uint32_t b = frame / cp.ntgt, limb = basis_target_limb(cp, frame % cp.ntgt);
    roots += (size_t)limb << logn;
    precons += (size_t)limb << logn;
    const BasisPair64 *row = pr + (size_t)limb * cp.L;
    const uint64_t q = __ldg(&bl[limb].q), twice = q << 1;
    const uint64_t *src = scratch + (((size_t)b * cp.m) << logn);  // both halves of the frame come from the scratch rows
    if (DOWN) {
        // the epilogue's operand x_hat_i towards L2 while the transform runs (as in ref_u64_rescale_fwd_kernel)
        const uint64_t *xin = in + (((size_t)b * cp.L + limb) << logn) + (size_t)half_id * M;
        for (uint32_t l = tid; l < M / 16; l += NT) asm volatile("prefetch.global.L2 [%0];" ::"l"(xin + 16 * l));
    }
    uint64_t x[16];

    // ---- pass 0: stages (split ..) on index bits [lg-4, lg), coefficients from the scratch rows through the prologue
    {
        constexpr uint32_t lo = lg - 4;
        const uint64_t one_p = __ldg(&bl[limb].one_p), th = twice - cp.h[limb];
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            if (NT == 512 && split) {                               // only NT = 512 runs N = 32768
                // stage 0 of the 32768-point frame, this CTA keeping only its half (ntt.cpp:331-369 with roots[1])
                const uint64_t W = __ldg(roots + 1), Wp = __ldg(precons + 1);
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    const uint32_t i = (k << lo) + vt;
                    uint64_t a = basis_lift_u64(src, i, bl, row, cp, q, one_p, th);
                    uint64_t bb = basis_lift_u64(src, M + i, bl, row, cp, q, one_p, th);
                    ref_bfly_u64(a, bb, W, Wp, q, twice);
                    x[k] = half_id ? bb : a;
                }
            } else {
                // basis_lift_u64 on 16 coefficients at once: each Horner step's constants are loaded once
                const uint32_t n = 1u << logn;
                const uint64_t *top = src + (size_t)(cp.m - 1) * n + vt;
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = top[k << lo];
                if (cp.lift) {
                    const uint64_t hs = cp.h[cp.s0], ps = __ldg(&bl[cp.s0].q);
#pragma unroll
                    for (int k = 0; k < 16; k++) x[k] = ref_csub_u64(x[k] + hs, ps);
                }
#pragma unroll 1
                for (int t = (int)cp.m - 2; t >= 0; t--) {
                    const uint64_t w = __ldg(&row[cp.s0 + t].w), wp = __ldg(&row[cp.s0 + t].w_p);
                    const uint64_t *dt = src + (size_t)t * n + vt;
#pragma unroll
                    for (int k = 0; k < 16; k++) x[k] = ref_shoup_u64(x[k], w, wp, q) + dt[k << lo];
                }
#pragma unroll
                for (int k = 0; k < 16; k++) x[k] = ref_shoup_u64(x[k], 1, one_p, q) + th;
            }
            // this CTA's sub-transform: stage s of it is global stage s + split, group offset half_id << s
            // (roots index = 2^(s+split) + (half_id << s) + local group)
            ref_pass16_u64<VEC, 0>(x, roots, precons, split, half_id, q, twice);
            uint64_t *s = img + vt + (vt >> 4);
            constexpr uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
    }
    __syncthreads();
    // ---- middle passes: index bits from lg-5 down to 4, four at a time (the last one may cover fewer)
    uint32_t s_done = 4;                                           // stages of the sub-transform finished so far
#pragma unroll
    for (int rem = (int)lg - 8; rem > 0; rem -= 4) {
        const uint32_t lo = rem >= 4 ? (uint32_t)rem : 4u;
        const uint32_t jfirst = rem >= 4 ? 0u : (uint32_t)(4 - rem);
        const uint32_t stride = (1u << lo) + (1u << (lo - 4));
#pragma unroll 1
        for (uint32_t vt = tid; vt < vthreads; vt += NT) {
            const uint32_t t_lo = vt & ((1u << lo) - 1), t_hi = vt >> lo;
            const uint32_t idx0 = (t_hi << (lo + 4)) + t_lo;
            uint64_t *s = img + idx0 + (idx0 >> 4);
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = s[k * stride];
            // twiddle index: 2^(s+split) + ((half_id << s) + group) with group = (t_hi << j) + g at local stage j
            const uint32_t sg = s_done + split;                    // global stage of the first active local stage
            const uint32_t th = t_hi + (half_id << (s_done - jfirst));   // the CTA's half as the top bit of the group index
            if (jfirst == 0) ref_pass16_u64<VEC, 0>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 1) ref_pass16_u64<VEC, 1>(x, roots, precons, sg, th, q, twice);
            else if (jfirst == 2) ref_pass16_u64<VEC, 2>(x, roots, precons, sg, th, q, twice);
            else ref_pass16_u64<VEC, 3>(x, roots, precons, sg, th, q, twice);
#pragma unroll
            for (int k = 0; k < 16; k++) s[k * stride] = x[k];
        }
        s_done += 4 - jfirst;
        __syncthreads();
    }
    // ---- final pass: bits 3..0 (16 consecutive coefficients), reduction to [0,q) (ntt.cpp:377-393)
#pragma unroll 1
    for (uint32_t vt = tid; vt < vthreads; vt += NT) {
        uint64_t *s = img + vt * 17;
#pragma unroll
        for (int k = 0; k < 16; k++) x[k] = s[k];
        ref_pass16_u64<VEC, 0>(x, roots, precons, s_done + split, vt + (half_id << s_done), q, twice);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            s[k] = ref_csub_u64(ref_csub_u64(x[k], twice), q);
        }
    }
    __syncthreads();
    // ---- epilogue.  DOWN: merge with the caller's spectrum of limb i and scale by P^-1, 16 reads of x_hat_i in flight
    // per thread (M = 32 * NT: two rounds).  Else: store into output limb i.
    if (DOWN) {
        const uint64_t pinv = cp.pinv[limb], pinv_p = cp.pinv_p[limb];
        const uint64_t *xin = in + (((size_t)b * cp.L + limb) << logn) + (size_t)half_id * M;
        uint64_t *dst = out + ((size_t)frame << logn) + (size_t)half_id * M;
#pragma unroll 1
        for (uint32_t i0 = tid; i0 < M; i0 += 16 * NT) {
#pragma unroll
            for (int k = 0; k < 16; k++) x[k] = xin[i0 + k * NT];
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const uint32_t i = i0 + k * NT;
                dst[i] = rescale_finish_u64(x[k], img[i + (i >> 4)], q, pinv, pinv_p);
            }
        }
    } else {
        uint64_t *dst = out + (((size_t)b * cp.L + limb) << logn) + (size_t)half_id * M;
        for (uint32_t i = tid; i < M; i += NT) dst[i] = img[i + (i >> 4)];
    }
}

// N < 1024: the same on the radix-2 forward.  TWIN: a copy of ref_fwd_u64_body (shared-memory work array) with the
// basis conversion's prologue on the load and its epilogue on the store, as ref_fwd_u64_rescale_kernel is; a fix to the
// transform belongs in all three.
template <bool DOWN>
__global__ void __launch_bounds__(1024) ref_fwd_u64_basis_kernel(const uint64_t *__restrict__ in,
                                                                 const uint64_t *__restrict__ scratch,
                                                                 uint64_t *__restrict__ out, const uint64_t *__restrict__ roots,
                                                                 const uint64_t *__restrict__ precons,
                                                                 const BasisLimb64 *__restrict__ bl,
                                                                 const BasisPair64 *__restrict__ pr, const __grid_constant__ BasisCall64 cp) {
    extern __shared__ uint64_t s64[];
    const uint32_t logn = cp.logn, N = 1u << logn;
    const uint32_t frame = blockIdx.x, b = frame / cp.ntgt, limb = basis_target_limb(cp, frame % cp.ntgt);
    roots += (size_t)limb << logn;
    precons += (size_t)limb << logn;
    const uint64_t q = __ldg(&bl[limb].q), twice = q << 1;
    uint64_t *X = s64;
    {
        const uint64_t *src = scratch + (((size_t)b * cp.m) << logn);
        const BasisPair64 *row = pr + (size_t)limb * cp.L;
        const uint64_t one_p = __ldg(&bl[limb].one_p), th = twice - cp.h[limb];
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) X[i] = basis_lift_u64(src, i, bl, row, cp, q, one_p, th);
    }
    __syncthreads();
    uint32_t tlog = logn - 1;
    for (uint32_t m = 1; m < N; m <<= 1, tlog--) {
        const bool last = (m == N / 2);
        for (uint32_t bf = threadIdx.x; bf < N / 2; bf += blockDim.x) {
            const uint32_t i = bf >> tlog, j = bf & ((1u << tlog) - 1);
            const uint32_t a0 = (i << (tlog + 1)) + j, a1 = a0 + (1u << tlog);
            const uint64_t W = roots[m + i], Wp = precons[m + i];
            uint64_t tx = X[a0];
            if (tx >= twice) tx -= twice;
            const uint64_t a = X[a1];
            const uint64_t c1 = __umul64hi(a, Wp);
            const uint64_t Q = W * a - c1 * q;
            uint64_t o0 = tx + Q, o1 = tx + twice - Q;
            if (last) {
                if (o0 >= twice) o0 -= twice;
                if (o0 >= q) o0 -= q;
                if (o1 >= twice) o1 -= twice;
                if (o1 >= q) o1 -= q;
            }
            X[a0] = o0; X[a1] = o1;
        }
        __syncthreads();
    }
    if (DOWN) {
        const uint64_t pinv = cp.pinv[limb], pinv_p = cp.pinv_p[limb];
        const uint64_t *xin = in + (((size_t)b * cp.L + limb) << logn);
        uint64_t *dst = out + ((size_t)frame << logn);
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) dst[i] = rescale_finish_u64(xin[i], X[i], q, pinv, pinv_p);
    } else {
        uint64_t *dst = out + (((size_t)b * cp.L + limb) << logn);
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) dst[i] = X[i];
    }
}

// ------------------------------------------------------------ u64 RNS Galois automorphisms ([B][L][N] -> [G][B][L][N])
// sigma_g: a(X) -> a(X^g) mod X^n + 1, g odd in [1, 2n).  Both kernels work with gi = g^-1 mod 2n, the only per-element
// value they need:
//   coefficient form: out[j] = in[u] if u < n, else -in[u - n] mod q_l, with u = j * gi mod 2n (coefficient i goes to
//     i * g mod 2n, and X^n = -1);
//   evaluation form (entry k = a(psi^(2 br(k) + 1))): out[k] = in[pi_g(k)], pi_g(k) = br((g (2 br(k) + 1) mod 2n - 1) / 2),
//     a permutation with no sign and the same on every limb.  pi_gi is its inverse, so out[pi_gi(j)] = in[j].
// pi maps every aligned block of 2^m entries onto an aligned block of 2^m entries (an odd factor keeps the low bits of
// 2 br(k) + 1 among the low bits, and br swaps low and high), and pi(j + 1) = pi(j) ^ 1 for even j (the top bit of
// br(j), i.e. a summand n of 2 br(j) + 1, times odd g is again n mod 2n).  So a 16-byte input pair is a 16-byte output
// pair, swapped when pi(j) is odd, and a warp's 32 pairs land in one aligned 512-byte block of each output.
constexpr uint32_t kAutomorphMax = 64;       // elements per call (agx_automorph64)
constexpr uint32_t kAutomorphThreads = 512;  // coefficient form: threads per CTA
constexpr uint32_t kAutomorphPart = 8192;    // coefficient form, n <= 8192: words one CTA stages (64 KB)
constexpr uint32_t kAutomorphRows = 256;     // coefficient form: most rows per CTA (n <= 32; the rows' q follow them)

// The per-call constants, passed by value (272 bytes): nothing is uploaded per call.
struct AutomorphCall64 {
    uint32_t R;                      // rows B * L of the input; output t is rows [t * R, (t + 1) * R)
    uint32_t L, logn, G;
    uint32_t gi[kAutomorphMax];      // g_t^-1 mod 2n
};

__device__ __forceinline__ uint64_t automorph_neg_u64(uint64_t x, uint64_t q) { return x ? q - x : 0; }

// Evaluation form, one launch: grid-stride over the 16-byte pairs of the input, each read once and written to all G
// outputs at pi_gi.
__global__ void __launch_bounds__(256) automorph64_ntt_kernel(ulonglong2 *__restrict__ out2, const ulonglong2 *__restrict__ in2,
                                                              const __grid_constant__ AutomorphCall64 cp, size_t pairs) {
    const uint32_t hlog = cp.logn - 1, sh = 32 - cp.logn, m2n = (2u << cp.logn) - 1;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < pairs; p += (size_t)gridDim.x * blockDim.x) {
        const ulonglong2 x = in2[p];
        const uint32_t h = (uint32_t)p & ((1u << hlog) - 1);       // pair within the row: words j = 2h, 2h + 1
        const size_t row = p - h;
        const uint32_t e = ((__brev(2 * h) >> sh) << 1) | 1;       // 2 br(j) + 1
        for (uint32_t t = 0; t < cp.G; t++) {
            const uint32_t d = __brev(((cp.gi[t] * e) & m2n) >> 1) >> sh;   // pi_gi(j); word j + 1 goes to d ^ 1
            out2[t * pairs + row + (d >> 1)] = (d & 1) ? make_ulonglong2(x.y, x.x) : x;
        }
    }
}

// Coefficient form, n <= 16384, one launch: a CTA stages `rpc` whole rows (at most kAutomorphPart words, or one row of
// 16384 words: 128 KB) and their q in shared memory, then writes its rows of every output coalesced.  The gather reads shared memory at the odd stride gi,
// so a half-warp's 8-byte reads hit 16 distinct bank pairs; the wrap mod n subtracts a multiple of 16 words.
__global__ void __launch_bounds__(kAutomorphThreads, 3) automorph64_coeff_kernel(uint64_t *__restrict__ out, const uint64_t *__restrict__ in,
                                                                                const RnsLimb64 *__restrict__ lc,
                                                                                const __grid_constant__ AutomorphCall64 cp,
                                                                                uint32_t rpc) {
    extern __shared__ __align__(16) uint64_t srow[];              // [rpc][n] words, then [rpc] q
    const uint32_t logn = cp.logn, n = 1u << logn, m2n = 2 * n - 1;
    const uint32_t r0 = blockIdx.x * rpc, rows = min(rpc, cp.R - r0), words = rows << logn;
    uint64_t *sq = srow + ((size_t)rpc << logn);
    const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(in + ((size_t)r0 << logn));
#pragma unroll 4
    for (uint32_t i = threadIdx.x; i < words / 2; i += kAutomorphThreads) reinterpret_cast<ulonglong2 *>(srow)[i] = src[i];
    for (uint32_t r = threadIdx.x; r < rows; r += kAutomorphThreads) sq[r] = __ldg(&lc[(r0 + r) % cp.L].p.q);
    __syncthreads();
    for (uint32_t t = 0; t < cp.G; t++) {
        const uint32_t gi = cp.gi[t];
        uint64_t *dst = out + (((size_t)t * cp.R + r0) << logn);
#pragma unroll 4
        for (uint32_t w = threadIdx.x; w < words; w += kAutomorphThreads) {
            const uint32_t j = w & (n - 1), u = (j * gi) & m2n;
            const uint64_t x = srow[(w - j) | (u & (n - 1))];
            dst[w] = (u & n) ? automorph_neg_u64(x, sq[w >> logn]) : x;
        }
    }
}

// a word of CTA `rank`'s shared memory in this cluster, at the shared::cta address `saddr` of the same variable here
__device__ __forceinline__ uint64_t ld_dsmem_u64(uint32_t saddr, uint32_t rank) {
    uint32_t a;
    uint64_t v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(saddr), "r"(rank));
    asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(a));
    return v;
}

__device__ __forceinline__ void automorph_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Coefficient form, n = 32768, one launch: a row over a cluster of CL CTAs (a row of 256 KB fits no CTA).  CTA `rank`
// stages words [rank * part, (rank + 1) * part) of the row and writes the same words of every output, gathering through
// distributed shared memory.  The second cluster barrier keeps every CTA resident until all partners have finished
// reading it.
template <int CL>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(kAutomorphThreads, 3)
    automorph64_coeff_cluster_kernel(uint64_t *__restrict__ out, const uint64_t *__restrict__ in,
                                     const RnsLimb64 *__restrict__ lc, const __grid_constant__ AutomorphCall64 cp) {
    constexpr uint32_t part = 32768 / CL;
    extern __shared__ __align__(16) uint64_t srow[];              // this CTA's part of the row
    const uint32_t logn = cp.logn, n = 1u << logn, m2n = 2 * n - 1;
    const uint32_t rank = blockIdx.x % CL, row = blockIdx.x / CL;
    const size_t base = ((size_t)row << logn) + rank * part;
    const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(in + base);
#pragma unroll 8
    for (uint32_t i = threadIdx.x; i < part / 2; i += kAutomorphThreads) reinterpret_cast<ulonglong2 *>(srow)[i] = src[i];
    const uint64_t q = __ldg(&lc[row % cp.L].p.q);
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(srow);
    automorph_cluster_sync();                                      // every part of the row is staged
    for (uint32_t t = 0; t < cp.G; t++) {
        const uint32_t gi = cp.gi[t];
        uint64_t *dst = out + (size_t)t * cp.R * n + base;
#pragma unroll 4
        for (uint32_t w = threadIdx.x; w < part; w += kAutomorphThreads) {
            const uint32_t u = ((rank * part + w) * gi) & m2n, v = u & (n - 1);
            const uint64_t x = ld_dsmem_u64(sbase + (v % part) * 8, v / part);
            dst[w] = (u & n) ? automorph_neg_u64(x, q) : x;
        }
    }
    automorph_cluster_sync();                                      // no partner still reads this CTA's shared memory
}

// ------------------------------------------------------------- u64 RNS key switching: the key inner product
// agx_keyswitch64's one kernel of its own.  In: the dnum extended digits U[dnum][B][L][n] (ModUp's outputs, evaluation
// form) and the key ksk[>= dnum][2][key_limbs][n]; out: A[2][B][L][n],
//   A_c[b][i] = sum_j U_j[b][i] * ksk[j][c][row(i)]  mod q_i,   row(i) = i (i < l + 1), i + key_limbs - L (special primes).
// A work item is one 16-byte pair of one limb row over a slice of the batch: its thread loads the key pairs of up to DC
// digits into registers once and then walks the slice, so the key is read once per slice, not once per polynomial.
// Each product is below q^2 < 2^124 and is added unreduced into a 128-bit sum: DC <= 8 products and a carried partial
// sum (< q) stay below 2^128.  The sum x = hi * 2^64 + lo is then reduced exactly over its whole range by two Shoup
// products, hi * (2^64 mod q) and lo * 1, each of which takes any 64-bit word into [0, 2q).  With dnum > DC the digits
// run in chunks of DC, each chunk's reduced sum stored in A and carried into the next.
constexpr uint32_t kKeySwitchChunk = 8;      // most digits a thread holds key words for at once

// The constants of limb q that reduce a 128-bit lazy sum: floor(2^64 / q), 2^64 mod q and its Shoup companion.
struct LazyRed64 {
    uint64_t q, one_p, r64, r64_p;
};

__device__ __forceinline__ LazyRed64 lazy_red64(const RnsLimb64 *l) {
    LazyRed64 r;
    r.q = __ldg(&l->p.q);
    const RefInvConst p = RefInvLimb{l, r.q}.consts();
    r.one_p = ref_shoup_companion(1, p);
    r.r64 = 0 - r.one_p * r.q;
    r.r64_p = ref_shoup_companion(r.r64, p);
    return r;
}

// hi * 2^64 + lo += a * b
__device__ __forceinline__ void mac128(uint64_t &lo, uint64_t &hi, uint64_t a, uint64_t b) {
    const uint64_t pl = a * b, ph = __umul64hi(a, b);
    lo += pl;
    hi += ph + (lo < pl);
}

// (hi * 2^64 + lo) mod q, exact for every 128-bit value
__device__ __forceinline__ uint64_t reduce128(uint64_t lo, uint64_t hi, const LazyRed64 &r) {
    const uint64_t s = ref_shoup_u64(hi, r.r64, r.r64_p, r.q) + ref_shoup_u64(lo, 1, r.one_p, r.q);
    return ref_csub_u64(ref_csub_u64(s, r.q << 1), r.q);           // s < 4q
}

struct KeySwitchCall64 {
    uint32_t L, logn;
    uint32_t ell1;           // l + 1: the limbs of Q_l, which read key rows 0 .. l
    uint32_t key_off;        // key_limbs - L: special prime i >= l + 1 reads key row i + key_off
    uint32_t key_limbs, dnum;
    uint32_t B, slice;       // polynomials, and polynomials per work item
};

template <int DC>
__global__ void __launch_bounds__(256) keyswitch64_inner_kernel(ulonglong2 *__restrict__ acc2,
                                                                const ulonglong2 *__restrict__ u2,
                                                                const ulonglong2 *__restrict__ k2,
                                                                const RnsLimb64 *__restrict__ lc,
                                                                const KeySwitchCall64 cp, size_t items) {
    const uint32_t hlog = cp.logn - 1;
    const size_t row2 = (size_t)1 << hlog;                         // pairs per limb row
    const size_t poly2 = (size_t)cp.L << hlog;                     // pairs per polynomial
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < items; w += (size_t)gridDim.x * blockDim.x) {
        const size_t j = w & (row2 - 1), r = w >> hlog;
        const uint32_t i = (uint32_t)(r % cp.L);
        const uint32_t b0 = (uint32_t)(r / cp.L) * cp.slice, b1 = min(cp.B, b0 + cp.slice);
        const LazyRed64 red = lazy_red64(lc + i);
        const size_t krow = i < cp.ell1 ? i : i + cp.key_off;
        const ulonglong2 *ukey = k2 + (krow << hlog) + j;
        const ulonglong2 *ubase = u2 + ((size_t)i << hlog) + j;
        ulonglong2 *abase = acc2 + ((size_t)i << hlog) + j;
        const size_t keyc = (size_t)cp.key_limbs << hlog, digit = (size_t)cp.B * poly2, comp = digit;
        for (uint32_t d0 = 0; d0 < cp.dnum; d0 += DC) {
            ulonglong2 kv[DC][2];
#pragma unroll
            for (int t = 0; t < DC; t++)
                if (d0 + t < cp.dnum) {
                    kv[t][0] = __ldg(ukey + (2 * (size_t)(d0 + t)) * keyc);
                    kv[t][1] = __ldg(ukey + (2 * (size_t)(d0 + t) + 1) * keyc);
                }
            for (uint32_t b = b0; b < b1; b++) {
                uint64_t lo[2][2] = {}, hi[2][2] = {};             // [component][word]
                if (d0) {
                    const ulonglong2 a0 = abase[b * poly2], a1 = abase[comp + b * poly2];
                    lo[0][0] = a0.x; lo[0][1] = a0.y; lo[1][0] = a1.x; lo[1][1] = a1.y;
                }
#pragma unroll
                for (int t = 0; t < DC; t++)
                    if (d0 + t < cp.dnum) {
                        const ulonglong2 x = __ldg(ubase + (d0 + t) * digit + b * poly2);
                        const uint64_t xv[2] = {x.x, x.y};
#pragma unroll
                        for (int c = 0; c < 2; c++) {
                            const uint64_t kw[2] = {kv[t][c].x, kv[t][c].y};
#pragma unroll
                            for (int v = 0; v < 2; v++) mac128(lo[c][v], hi[c][v], xv[v], kw[v]);
                        }
                    }
                uint64_t y[2][2];
#pragma unroll
                for (int c = 0; c < 2; c++)
#pragma unroll
                    for (int v = 0; v < 2; v++) y[c][v] = reduce128(lo[c][v], hi[c][v], red);
                abase[b * poly2] = make_ulonglong2(y[0][0], y[0][1]);
                abase[comp + b * poly2] = make_ulonglong2(y[1][0], y[1][1]);
            }
        }
    }
}

// P mod q_i for a limb i of Q_l, P the product of the special primes q_{l+1} .. q_{L-1}, from the pairwise table
__device__ __forceinline__ uint64_t p_mod_q(const BasisPair64 *__restrict__ bp, uint32_t i, uint32_t ell1, uint32_t L,
                                            uint64_t q) {
    const BasisPair64 *row = bp + (size_t)i * L;
    uint64_t pm = 1;
    for (uint32_t s = ell1; s < L; s++) pm = ref_csub_u64(ref_shoup_u64(pm, __ldg(&row[s].w), __ldg(&row[s].w_p), q), q);
    return pm;
}

// automorph64_ntt_kernel's permutation in evaluation form: the entry that word `word` of a row comes from under element
// `g` (out[k] = in[pi_g(k)]), or where it goes under g^-1.  sh = 32 - log n, m2n = 2n - 1.
__device__ __forceinline__ uint32_t eval_perm(uint32_t g, uint32_t word, uint32_t sh, uint32_t m2n) {
    const uint32_t e = ((__brev(word) >> sh) << 1) | 1;            // 2 br(word) + 1
    return __brev(((g * e) & m2n) >> 1) >> sh;
}

// ------------------------------------------------------------- u64 RNS hoisted rotations: the G key inner products
// agx_rotate64's one kernel of its own.  In: the dnum extended digits U[dnum][B][L][n] of c1 (ModUp's outputs), the
// spectrum c0h[B][l+1][n] of c0 and G keys rk_t[>= dnum][2][key_limbs][n], all in evaluation form; out: A[G][2][B][L][n],
//   A_t[c][b][i][k] = sum_j U_j[b][i][pi_t(k)] * rk_t[j][c][row(i)][k]  +  [c = 0, i <= l] (P mod q_i) c0h[b][i][pi_t(k)]
// mod q_i, with row(i) keyswitch64_inner_kernel's and pi_t automorph64_ntt_kernel's permutation for g_t (out[k] =
// in[pi_g(k)], i.e. input entry j lands at pi_{g^-1}(j), which is how this kernel, like that one, uses it).  ModDown of
// A_t is sigma_t(c0) + KS_t(sigma_t(c1)): floor((X + P C + h_P) / P) = C + floor((X + h_P) / P), and P C = 0 mod p_t.
// A work item is one 16-byte pair j of one input limb row, for one element t, over a slice of the batch.  Its thread
// loads key t's words at the pair's destination pi_{g^-1}(j) into registers once, then walks the slice.  Items run in
// the order (slice and limb row, 32-pair block of the input, t, pair): the G warps that read one 512-byte block of U
// and of c0h follow one another, so each block comes from HBM once and its G - 1 re-reads from L2.  The permutation
// maps that block onto one aligned block of every key and output, and keeps pairs together (swapped when the
// destination word is odd), so every warp access covers whole 512-byte blocks.
// The 128-bit lazy sum and its reduction are keyswitch64_inner_kernel's.  The first chunk holds DC <= 8 products and
// the c0 product, a later one DC products and the carried sum (< q): at most 9 * 2^124 < 2^128.
struct RotateCall64 {
    KeySwitchCall64 ks;                          // slice: polynomials per work item
    uint32_t G;
    uint32_t gi[kAutomorphMax];                  // g_t^-1 mod 2n
    const ulonglong2 *rk[kAutomorphMax];         // key t
};

template <int DC>
__global__ void __launch_bounds__(256) rotate64_inner_kernel(ulonglong2 *__restrict__ acc2,
                                                             const ulonglong2 *__restrict__ u2,
                                                             const ulonglong2 *__restrict__ c02,
                                                             const RnsLimb64 *__restrict__ lc,
                                                             const BasisPair64 *__restrict__ bp,
                                                             const __grid_constant__ RotateCall64 cp, size_t items) {
    const KeySwitchCall64 &ks = cp.ks;
    const uint32_t hlog = ks.logn - 1, sh = 32 - ks.logn, m2n = (2u << ks.logn) - 1;
    const uint32_t lb = min(hlog, 5u);                             // log2 of the pairs in a block
    const size_t row2 = (size_t)1 << hlog;
    const size_t poly2 = (size_t)ks.L << hlog;
    const size_t digit = (size_t)ks.B * poly2, comp = digit, keyc = (size_t)ks.key_limbs << hlog;
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < items; w += (size_t)gridDim.x * blockDim.x) {
        const size_t blk = w >> lb, rest = blk / cp.G;             // rest: (row r, block of the row)
        const uint32_t t = (uint32_t)(blk - rest * cp.G);
        const size_t r = rest >> (hlog - lb);
        const uint32_t j = (uint32_t)(((rest << lb) & (row2 - 1)) | (w & ((1u << lb) - 1)));   // input pair
        const uint32_t i = (uint32_t)(r % ks.L);
        const uint32_t b0 = (uint32_t)(r / ks.L) * ks.slice, b1 = min(ks.B, b0 + ks.slice);
        const uint32_t d = eval_perm(cp.gi[t], 2 * j, sh, m2n);   // word 2j goes to d, word 2j + 1 to d ^ 1
        const bool swap = d & 1;
        const size_t o = d >> 1;                                   // the destination pair
        const LazyRed64 red = lazy_red64(lc + i);
        const bool has_c0 = i < ks.ell1;
        const uint64_t pm = has_c0 ? p_mod_q(bp, i, ks.ell1, ks.L, red.q) : 1;   // P mod q_i
        const size_t krow = has_c0 ? i : i + ks.key_off;
        const ulonglong2 *ukey = cp.rk[t] + (krow << hlog) + o;
        const ulonglong2 *ubase = u2 + ((size_t)i << hlog) + j;
        const ulonglong2 *cbase = c02 + ((size_t)i << hlog) + j;   // c0h row b * (l + 1) + i
        ulonglong2 *abase = acc2 + (size_t)t * 2 * digit + ((size_t)i << hlog) + o;
        for (uint32_t d0 = 0; d0 < ks.dnum; d0 += DC) {
            ulonglong2 kv[DC][2];
#pragma unroll
            for (int u = 0; u < DC; u++)
                if (d0 + u < ks.dnum) {
                    kv[u][0] = __ldg(ukey + (2 * (size_t)(d0 + u)) * keyc);
                    kv[u][1] = __ldg(ukey + (2 * (size_t)(d0 + u) + 1) * keyc);
                }
            for (uint32_t b = b0; b < b1; b++) {
                uint64_t lo[2][2] = {}, hi[2][2] = {};             // [component][word]
                if (d0) {
                    const ulonglong2 a0 = abase[b * poly2], a1 = abase[comp + b * poly2];
                    lo[0][0] = a0.x; lo[0][1] = a0.y; lo[1][0] = a1.x; lo[1][1] = a1.y;
                } else if (has_c0) {
                    const ulonglong2 x = __ldg(cbase + (size_t)b * ks.ell1 * row2);
                    const uint64_t xv[2] = {swap ? x.y : x.x, swap ? x.x : x.y};
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        lo[0][v] = xv[v] * pm;
                        hi[0][v] = __umul64hi(xv[v], pm);
                    }
                }
#pragma unroll
                for (int u = 0; u < DC; u++)
                    if (d0 + u < ks.dnum) {
                        const ulonglong2 x = __ldg(ubase + (d0 + u) * digit + b * poly2);
                        const uint64_t xv[2] = {swap ? x.y : x.x, swap ? x.x : x.y};
#pragma unroll
                        for (int c = 0; c < 2; c++) {
                            const uint64_t kw[2] = {kv[u][c].x, kv[u][c].y};
#pragma unroll
                            for (int v = 0; v < 2; v++) mac128(lo[c][v], hi[c][v], xv[v], kw[v]);
                        }
                    }
                uint64_t y[2][2];
#pragma unroll
                for (int c = 0; c < 2; c++)
#pragma unroll
                    for (int v = 0; v < 2; v++) y[c][v] = reduce128(lo[c][v], hi[c][v], red);
                abase[b * poly2] = make_ulonglong2(y[0][0], y[0][1]);
                abase[comp + b * poly2] = make_ulonglong2(y[1][0], y[1][1]);
            }
        }
    }
}

// ------------------------------------------------------------- u64 RNS hoisted linear transforms: sum_t d_t (.) A_t
// agx_lintrans64's one kernel of its own.  In: agx_rotate64's U[dnum][B][L][n] and keys, the ciphertexts'
// spectra ct[2][B][l+1][n] (c0, then c1), and M x G diagonals d_{m,t}[L][n] over Q_l u P; all in evaluation form.
// Out: Acc[M][2][B][L][n],
//   Acc[m][c][b][i][o] = sum_t d_{m,t}[i][o] * A_t[c][b][i][o]  mod q_i,
// A_t being rotate64_inner_kernel's output t (the key inner product over the permuted digits plus P sigma_t(c0)), or
// (P c0, P c1) for a keyless term (g = 1).  ModDown of Acc[m] is then sum_t d_{m,t} sigma_t(c0) + ModDown(sum_t d_{m,t}
// KS_t) by the same fold as agx_rotate64's.  A work item owns one output pair o of one limb row of one polynomial and
// gathers: for each term t it reads key t's words at o and U and ct at the source pair pi_t(o) (out[k] =
// in[pi_g(k)], automorph64_ntt_kernel's map; the pair is swapped when pi_t(2o) is odd), forms A_t in registers, and
// adds d_{m,t} * A_t into each of the M accumulators.  So no A_t reaches memory, and keys and digits are read once per
// (element, term) however large M is.  pi_t maps an aligned 32-pair block onto an aligned block and keeps pairs
// together, so every warp gather covers whole 512-byte blocks.  Items run limb-major, (limb, polynomial, pair): the B
// polynomials of one limb follow one another and share that limb's key and diagonal rows (2 G dnum + M G rows of
// n / 2 pairs), which therefore come from HBM once per call and from L2 for the other polynomials, while the rows being
// gathered (U, c0, c1 of a few polynomials) are small enough to serve their G re-reads from L2 too.
// A_t's lazy sum is rotate64_inner_kernel's chunking (DC <= 8 products plus the c0 product or the carried sum).  The
// accumulators are kept reduced: each d * A_t (< q^2 < 2^124) is added to one (< q) and the 128-bit sum reduced at
// once, so a thread holds MC x 4 words, MC = 4 or 16 (the most outputs of its instantiation).  Terms whose diagonals
// are all zero are dropped on the host; a NULL d_{m,t} is skipped.
constexpr uint32_t kLintransMaxOut = 16;      // outputs per call (agx_lintrans64)
constexpr uint32_t kLintransMaxTerms = 256;   // diagonals per call: M * G

struct LintransCall64 {
    KeySwitchCall64 ks;                          // slice unused
    uint32_t G, M;                               // terms kept, outputs
    uint32_t g[kAutomorphMax];                   // term t's Galois element
    const ulonglong2 *rk[kAutomorphMax];         // key t; nullptr: a keyless identity term
    const ulonglong2 *diag[kLintransMaxTerms];   // d_{m,t} at [m * G + t]; nullptr: zero
};

template <int DC, int MC>
__global__ void __launch_bounds__(256) lintrans64_inner_kernel(ulonglong2 *__restrict__ acc2,
                                                               const ulonglong2 *__restrict__ u2,
                                                               const ulonglong2 *__restrict__ ct2,
                                                               const RnsLimb64 *__restrict__ lc,
                                                               const BasisPair64 *__restrict__ bp,
                                                               const __grid_constant__ LintransCall64 cp, size_t items) {
    const KeySwitchCall64 &ks = cp.ks;
    const uint32_t hlog = ks.logn - 1, sh = 32 - ks.logn, m2n = (2u << ks.logn) - 1;
    const size_t row2 = (size_t)1 << hlog;
    const size_t poly2 = (size_t)ks.L << hlog;
    const size_t digit = (size_t)ks.B * poly2, keyc = (size_t)ks.key_limbs << hlog;
    const size_t c1off = (size_t)ks.B * ks.ell1 * row2;            // c1 after c0 in ct
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < items; w += (size_t)gridDim.x * blockDim.x) {
        const size_t r = w >> hlog;                                // (limb i, polynomial b), limb-major
        const uint32_t o = (uint32_t)(w & (row2 - 1));             // output pair
        const uint32_t i = (uint32_t)(r / ks.B), b = (uint32_t)(r - (size_t)i * ks.B);
        const LazyRed64 red = lazy_red64(lc + i);
        const bool has_c0 = i < ks.ell1;
        const uint64_t pm = has_c0 ? p_mod_q(bp, i, ks.ell1, ks.L, red.q) : 0;   // P mod q_i; P = 0 mod p_t
        const size_t krow = has_c0 ? i : i + ks.key_off;
        const ulonglong2 *ubase = u2 + (size_t)b * poly2 + ((size_t)i << hlog);
        const ulonglong2 *cbase = ct2 + ((size_t)b * ks.ell1 + i) * row2;
        const size_t dof = ((size_t)i << hlog) + o;                // the output pair in a diagonal
        uint64_t acc[MC][2][2] = {};                               // [output][component][word], reduced
        for (uint32_t t = 0; t < cp.G; t++) {
            const ulonglong2 *rk = cp.rk[t];
            if (!rk && !has_c0) continue;                          // (P c0, P c1) is zero on the special primes
            const uint32_t s = eval_perm(cp.g[t], 2 * o, sh, m2n);   // word 2o comes from s, word 2o + 1 from s ^ 1
            const bool swap = s & 1;
            const size_t src = s >> 1;
            uint64_t a[2][2];                                      // A_t at the output pair: [component][word]
            if (!rk) {
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    const ulonglong2 x = __ldg(cbase + c * c1off + src);
                    const uint64_t xv[2] = {swap ? x.y : x.x, swap ? x.x : x.y};
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        uint64_t lo = 0, hi = 0;
                        mac128(lo, hi, xv[v], pm);
                        a[c][v] = reduce128(lo, hi, red);
                    }
                }
            } else {
                const ulonglong2 *ukey = rk + (krow << hlog) + o;
                for (uint32_t d0 = 0; d0 < ks.dnum; d0 += DC) {
                    uint64_t lo[2][2] = {}, hi[2][2] = {};
                    if (d0) {
#pragma unroll
                        for (int c = 0; c < 2; c++)
#pragma unroll
                            for (int v = 0; v < 2; v++) lo[c][v] = a[c][v];
                    } else if (has_c0) {
                        const ulonglong2 x = __ldg(cbase + src);
                        mac128(lo[0][0], hi[0][0], swap ? x.y : x.x, pm);
                        mac128(lo[0][1], hi[0][1], swap ? x.x : x.y, pm);
                    }
#pragma unroll
                    for (int u = 0; u < DC; u++)
                        if (d0 + u < ks.dnum) {
                            const ulonglong2 x = __ldg(ubase + (d0 + u) * digit + src);
                            const uint64_t xv[2] = {swap ? x.y : x.x, swap ? x.x : x.y};
#pragma unroll
                            for (int c = 0; c < 2; c++) {
                                const ulonglong2 kv = __ldg(ukey + (2 * (size_t)(d0 + u) + c) * keyc);
                                mac128(lo[c][0], hi[c][0], xv[0], kv.x);
                                mac128(lo[c][1], hi[c][1], xv[1], kv.y);
                            }
                        }
#pragma unroll
                    for (int c = 0; c < 2; c++)
#pragma unroll
                        for (int v = 0; v < 2; v++) a[c][v] = reduce128(lo[c][v], hi[c][v], red);
                }
            }
#pragma unroll
            for (int m = 0; m < MC; m++) {
                const ulonglong2 *dg = m < (int)cp.M ? cp.diag[m * cp.G + t] : nullptr;
                if (!dg) continue;
                const ulonglong2 dv = __ldg(dg + dof);
                const uint64_t dw[2] = {dv.x, dv.y};
#pragma unroll
                for (int c = 0; c < 2; c++)
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        uint64_t lo = acc[m][c][v], hi = 0;
                        mac128(lo, hi, dw[v], a[c][v]);
                        acc[m][c][v] = reduce128(lo, hi, red);
                    }
            }
        }
        ulonglong2 *abase = acc2 + (size_t)b * poly2 + ((size_t)i << hlog) + o;
#pragma unroll
        for (int m = 0; m < MC; m++)
            if (m < (int)cp.M)
#pragma unroll
                for (int c = 0; c < 2; c++) abase[(2 * (size_t)m + c) * digit] = make_ulonglong2(acc[m][c][0], acc[m][c][1]);
    }
}

// ------------------------------------------------------------- u64 RNS ciphertext multiplication: tensor + relinearisation
// agx_mulrelin64's one kernel of its own.  In: the dnum extended digits U[dnum][B][L][n] of D_2 = a1 b1 (ModUp's
// outputs), the spectra a[2][B][l+1][n] and b[2][B][l+1][n] of the two ciphertexts (a == b when squaring) and the
// relinearisation key rlk[>= dnum][2][key_limbs][n], all in evaluation form; out: A[2][B][L][n],
//   A_c[b][i] = sum_j U_j[b][i] * rlk[j][c][row(i)]  +  [i <= l] (P mod q_i) D_c[b][i]   mod q_i,
//   D_0 = a0 b0,  D_1 = a0 b1 + a1 b0   (per limb, mod q_i),
// row(i) being keyswitch64_inner_kernel's.  ModDown_P of A_c is D_c + KS(D_2)[c] by rotate64_inner_kernel's fold, and
// ModDown over q_l P (the last k + 1 primes) is the product rescaled with one rounding.  The walk is
// keyswitch64_inner_kernel's: key words of up to DC digits in registers, one slice of the batch per work item.  D_0 and
// D_1 are formed in registers from the four input pairs and reduced to [0, q), so (P mod q_i) D_c is one product
// below 2^120 and the first chunk holds DC + 1 <= 9 products: below 2^128.  No D_c reaches memory.
template <int DC>
__global__ void __launch_bounds__(256) mulrelin64_inner_kernel(ulonglong2 *__restrict__ acc2,
                                                               const ulonglong2 *__restrict__ u2,
                                                               const ulonglong2 *__restrict__ a2,
                                                               const ulonglong2 *__restrict__ b2,
                                                               const ulonglong2 *__restrict__ k2,
                                                               const RnsLimb64 *__restrict__ lc,
                                                               const BasisPair64 *__restrict__ bp,
                                                               const KeySwitchCall64 cp, size_t items) {
    const uint32_t hlog = cp.logn - 1;
    const size_t row2 = (size_t)1 << hlog;                         // pairs per limb row
    const size_t poly2 = (size_t)cp.L << hlog;                     // pairs per polynomial over Q_l u P
    const size_t ct2 = (size_t)cp.ell1 << hlog;                    // pairs per polynomial over Q_l
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < items; w += (size_t)gridDim.x * blockDim.x) {
        const size_t j = w & (row2 - 1), r = w >> hlog;
        const uint32_t i = (uint32_t)(r % cp.L);
        const uint32_t b0 = (uint32_t)(r / cp.L) * cp.slice, b1 = min(cp.B, b0 + cp.slice);
        const LazyRed64 red = lazy_red64(lc + i);
        const bool has_d = i < cp.ell1;                            // P D_c = 0 mod the special primes
        const uint64_t pm = has_d ? p_mod_q(bp, i, cp.ell1, cp.L, red.q) : 0;   // P mod q_i
        const size_t krow = has_d ? i : i + cp.key_off;
        const ulonglong2 *ukey = k2 + (krow << hlog) + j;
        const ulonglong2 *ubase = u2 + ((size_t)i << hlog) + j;
        const ulonglong2 *xa = a2 + ((size_t)i << hlog) + j, *xb = b2 + ((size_t)i << hlog) + j;
        ulonglong2 *abase = acc2 + ((size_t)i << hlog) + j;
        const size_t keyc = (size_t)cp.key_limbs << hlog, digit = (size_t)cp.B * poly2, comp = digit;
        const size_t ctc = (size_t)cp.B * ct2;                     // c1 after c0 in a and b
        for (uint32_t d0 = 0; d0 < cp.dnum; d0 += DC) {
            ulonglong2 kv[DC][2];
#pragma unroll
            for (int t = 0; t < DC; t++)
                if (d0 + t < cp.dnum) {
                    kv[t][0] = __ldg(ukey + (2 * (size_t)(d0 + t)) * keyc);
                    kv[t][1] = __ldg(ukey + (2 * (size_t)(d0 + t) + 1) * keyc);
                }
            for (uint32_t b = b0; b < b1; b++) {
                uint64_t lo[2][2] = {}, hi[2][2] = {};             // [component][word]
                if (d0) {
                    const ulonglong2 a0 = abase[b * poly2], a1 = abase[comp + b * poly2];
                    lo[0][0] = a0.x; lo[0][1] = a0.y; lo[1][0] = a1.x; lo[1][1] = a1.y;
                } else if (has_d) {
                    const ulonglong2 x0 = __ldg(xa + b * ct2), x1 = __ldg(xa + ctc + b * ct2);
                    const ulonglong2 y0 = __ldg(xb + b * ct2), y1 = __ldg(xb + ctc + b * ct2);
                    const uint64_t av0[2] = {x0.x, x0.y}, av1[2] = {x1.x, x1.y};
                    const uint64_t bv0[2] = {y0.x, y0.y}, bv1[2] = {y1.x, y1.y};
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        uint64_t l0 = 0, h0 = 0, l1 = 0, h1 = 0;
                        mac128(l0, h0, av0[v], bv0[v]);
                        mac128(l1, h1, av0[v], bv1[v]);
                        mac128(l1, h1, av1[v], bv0[v]);
                        const uint64_t dc[2] = {reduce128(l0, h0, red), reduce128(l1, h1, red)};
#pragma unroll
                        for (int c = 0; c < 2; c++) {
                            lo[c][v] = dc[c] * pm;
                            hi[c][v] = __umul64hi(dc[c], pm);
                        }
                    }
                }
#pragma unroll
                for (int t = 0; t < DC; t++)
                    if (d0 + t < cp.dnum) {
                        const ulonglong2 x = __ldg(ubase + (d0 + t) * digit + b * poly2);
                        const uint64_t xv[2] = {x.x, x.y};
#pragma unroll
                        for (int c = 0; c < 2; c++) {
                            const uint64_t kw[2] = {kv[t][c].x, kv[t][c].y};
#pragma unroll
                            for (int v = 0; v < 2; v++) mac128(lo[c][v], hi[c][v], xv[v], kw[v]);
                        }
                    }
                uint64_t y[2][2];
#pragma unroll
                for (int c = 0; c < 2; c++)
#pragma unroll
                    for (int v = 0; v < 2; v++) y[c][v] = reduce128(lo[c][v], hi[c][v], red);
                abase[b * poly2] = make_ulonglong2(y[0][0], y[0][1]);
                abase[comp + b * poly2] = make_ulonglong2(y[1][0], y[1][1]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------- twiddle tables on device
// The step before the path: the reference fills its root / precon buffers on the host (main.cpp:46-55) and the loader
// broadcasts them (ntt.cpp:544-571).  Here one thread per (limb, direction, k) computes
//   w = base^bitrev(k) mod q   (base = psi forward, psi^-1 inverse; the table order ntt.cpp:298-300 consumes),
//   w' = floor(w * 2^32 / q)   (Shoup companion),
// and writes it to the natural-order table (introspection, generic kernel), to its kernel-order slot (tw_pos) and, for
// k < E, to the column pass's slot.  Inverse kernel-order entries 0 and 1 carry n^-1 (see ntt_inv_loop_kernel).
struct LimbGen {
    uint32_t q, psi, psi_inv, n_inv;
};

__device__ __forceinline__ uint32_t mulmod_dev(uint32_t a, uint32_t b, uint32_t q) {
    return (uint32_t)(((uint64_t)a * b) % q);
}

// Places entry k (value r = base^bitrev(k)) of one limb's table into every layout the kernels read:
// natural order, kernel order (tw_pos) and -- for k < E -- the column pass's slots; inverse tables get n^-1 folded in.
// le == 0: generic sizes, kernel order == natural order and no column tables.
struct TableSet {
    uint2 *nat, *tw, *twc;      // one limb, one direction
};

__device__ __forceinline__ uint2 shoup_pair(uint32_t w, uint32_t q) { return make_uint2(w, (uint32_t)(((uint64_t)w << 32) / q)); }

// entry `pos` of a kernel-order table; `vec4`: the slot is fetched by the kernels' 16-byte loads (see AGX_TW_INTERLEAVE)
__device__ __forceinline__ void store_tw(uint2 *tab, uint32_t pos, uint2 v, bool vec4) {
#if AGX_TW_INTERLEAVE
    if (vec4) {
        uint32_t *w = reinterpret_cast<uint32_t *>(tab) + (pos >> 1) * 4 + (pos & 1);
        w[0] = v.x;
        w[2] = v.y;
        return;
    }
#endif
    tab[pos] = v;
}

__device__ __forceinline__ void place_table_entry(const TableSet &t, uint32_t k, uint32_t r, bool inverse, uint32_t q,
                                                  uint32_t n_inv, uint32_t logn, int le) {
    const uint2 natural = shoup_pair(r, q);
    t.nat[k] = natural;
    uint32_t w = r;
    if (inverse && k == 0) w = n_inv;                                    // unused slot carries n^-1
    if (inverse && k == 1 && le) w = mulmod_dev(r, n_inv, q);            // last GS stage folds n^-1 (two-pass kernels)
    uint32_t pos = k;
    if (le && k >= (1u << le)) {
        const int s = 31 - __clz(k), lt = (int)logn - le;
        const uint32_t c = 1u << (s - lt), rr = k - (1u << s), tpp = 1u << lt;
        const uint32_t T = rr / c, kk = rr % c;
        pos = c == 1 ? (1u << s) + T : (1u << s) + ((kk >> 1) * tpp + T) * 2 + (kk & 1);   // = tw_pos<LOGN,LE>(s, T, kk)
    }
    store_tw(t.tw, pos, shoup_pair(w, q), le && pos >= (2u << ((int)logn - le)));   // stages read by 16-byte loads
    if (le && k >= 1 && k < (1u << le)) {   // column pass: local stage j, group gq sits where the row pass of thread 0 looks
        const int j = 31 - __clz(k), lt = (int)logn - le;
        const uint32_t gq = k - (1u << j), tpp = 1u << lt;
        const uint32_t cpos = j == 0 ? tpp : 2 * ((1u << (lt + j - 1)) + (gq >> 1) * tpp) + (gq & 1);
        uint2 cval = natural;
        if (inverse && j >= 1 && j <= kInvFold) cval = shoup_pair(mulmod_dev(r, n_inv, q), q);   // variant A carries n^-1
        store_tw(t.twc, cpos, cval, j >= 1);
        if (inverse && j >= 1) store_tw(t.twc, cpos + 2, natural, true);  // variant B: one 16-byte slot further
    }
}

// Tables from psi: one thread per (direction, limb, k).
__global__ void __launch_bounds__(256) gen_tables_kernel(uint2 *__restrict__ nat_fwd, uint2 *__restrict__ nat_inv,
                                                         uint2 *__restrict__ tw_fwd, uint2 *__restrict__ tw_inv,
                                                         uint2 *__restrict__ twc_fwd, uint2 *__restrict__ twc_inv,
                                                         const LimbGen *__restrict__ lg, uint32_t L, uint32_t logn, int le) {
    const uint32_t n = 1u << logn;
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= 2u * L * n) return;
    const uint32_t k = gid & (n - 1), limb = (gid >> logn) % L;
    const bool inverse = gid >= L * n;
    const LimbGen g = lg[limb];
    const uint32_t e = __brev(k) >> (32 - logn);
    uint32_t r = 1, b = inverse ? g.psi_inv : g.psi;
    for (uint32_t i = 0; i < logn; i++) {
        if ((e >> i) & 1) r = mulmod_dev(r, b, g.q);
        b = mulmod_dev(b, b, g.q);
    }
    const size_t base = (size_t)limb * n;
    const TableSet t{(inverse ? nat_inv : nat_fwd) + base, (inverse ? tw_inv : tw_fwd) + base,
                     le ? (inverse ? twc_inv : twc_fwd) + base : nullptr};
    place_table_entry(t, k, r, inverse, g.q, g.n_inv, logn, le);
}

// Tables handed in by the caller in the reference's order (ntt.cpp:298-300: entry m + i = twiddle of group i in the
// stage with m groups; include/kernel/ntt.h:35-41, main.cpp:36-37,46-55 hand such buffers to the loader): checked for
// consistency and re-laid-out for the kernels.  One thread per k.  A table is consistent when, with I = roots[1],
//   I^2 = -1,  roots[2k]^2 = roots[k],  roots[2k+1] = roots[2k] * I   (k >= 1),  every entry < q,
// which is equivalent to roots[k] = psi^bitrev(k) for the primitive 2n-th root psi = roots[n/2]; precons (optional)
// must be the Shoup companions floor(roots[k] * 2^32 / q).  Violations are counted in *bad.
__global__ void __launch_bounds__(256) relayout_tables_kernel(TableSet t, const uint32_t *__restrict__ roots,
                                                              const uint32_t *__restrict__ precons, bool inverse, uint32_t q,
                                                              uint32_t n_inv, uint32_t logn, int le, unsigned *bad) {
    const uint32_t n = 1u << logn;
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t r = k ? roots[k] : 1u;
    bool ok = r < q && r != 0;
    if (ok && k >= 1) {
        if (precons && precons[k] != shoup_pair(r, q).y) ok = false;
        const uint32_t I = roots[1];
        if (k == 1 && mulmod_dev(I, I, q) != q - 1) ok = false;
        if (2 * k < n) {
            const uint32_t e = roots[2 * k], o = roots[2 * k + 1];
            if (e >= q || o >= q || mulmod_dev(e, e, q) != r || mulmod_dev(e, I % q, q) != o) ok = false;
        }
    }
    if (!ok) { atomicAdd(bad, 1u); return; }
    place_table_entry(t, k, r, inverse, q, n_inv, logn, le);
}

// ---------------------------------------------------------------------------------- synthetic data + checksum
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    uint64_t z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256) fill_synthetic_kernel(uint32_t *__restrict__ data, size_t total, uint32_t logn,
                                                             uint32_t L, const LimbConst *__restrict__ lc, uint64_t seed,
                                                             uint64_t first_elem) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t q = lc[((first_elem + i) >> logn) % L].q;
        data[i] = (uint32_t)(splitmix64(seed + first_elem + i) % q);
    }
}

__global__ void __launch_bounds__(256) checksum_kernel(const uint32_t *__restrict__ data, size_t count, uint64_t first_index,
                                                       unsigned long long *__restrict__ sum) {
    uint64_t acc = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
        acc += splitmix64((first_index + i) * 0xD6E8FEB86659FD93ULL + data[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(sum, (unsigned long long)acc);
}

}  // namespace agx
