// agx_api.cu -- the C ABI of include/agxntt.h over the sm_100a kernels.  No torch types, no CPU fallback.
#include "../../include/agxntt.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "agx_ntt_kernels.cuh"
#include "agx_encode.cuh"
#include "agx_diag.cuh"
// Build-time option, OFF in the shipped library: the radix-16 three-pass kernels for n = 4096 (16 coefficients per thread,
// 40 warps per SM).  Bit-exact, measured 6-9 % slower than the two-pass kernels (profiles/r02_experiments.md), kept out of
// the product tree; a variant library with them is built by `make -C experiments r16` and selected with AGX_KERNEL=r16.
#ifndef AGX_WITH_R16
#define AGX_WITH_R16 0
#endif
#if AGX_WITH_R16
#include "agx_ntt_r16.cuh"
#endif
#include "agx_tables.h"
#include "agx_copycrew.h"

using namespace agx;

#define CK(call)                                   \
    do {                                           \
        cudaError_t e__ = (call);                  \
        if (e__ != cudaSuccess) return (int)e__;   \
    } while (0)

namespace {

constexpr int kSlots = 3;                          // host pipeline depth (H2D / kernel / D2H in flight)
constexpr size_t kChunkBytes = 32u << 20;          // per-slot chunk of the host pipeline when the SM count is unknown

struct HostPipe {
    cudaStream_t stream[kSlots] = {};
    cudaEvent_t done[kSlots] = {};
    uint32_t *d_a[kSlots] = {}, *d_b[kSlots] = {};
    uint32_t *p_in[kSlots] = {}, *p_in2[kSlots] = {}, *p_out[kSlots] = {};   // pinned staging (pageable callers)
    size_t cap = 0;                                // bytes per device / staging buffer
    bool have_b = false, have_stage = false;
};

constexpr size_t kRefChunkBytes = 16u << 20;       // frame data per slot of the reference-shaped pipeline when the SM count is unknown

struct RefState {
    bool have_in = false, have_fwd = false, have_out = false, busy = false;
    uint32_t N = 0, frames = 0;
    const uint64_t *in = nullptr, *in2 = nullptr, *mod = nullptr, *tw = nullptr, *pre = nullptr;
    uint64_t *out = nullptr;
    int32_t out_frames = 0;
    // device side: tables, and per slot one input and one output chunk (H2D / kernel / D2H of different slots overlap)
    uint64_t *d_tw = nullptr, *d_pre = nullptr;
    uint64_t *d_in[kSlots] = {}, *d_out[kSlots] = {};
    uint64_t *p_in[kSlots] = {}, *p_out[kSlots] = {};      // pinned staging for pageable callers
    size_t cap_chunk = 0, cap_tab = 0;
    bool have_stage_in = false, have_stage_out = false;
    cudaStream_t stream[kSlots] = {};
    cudaEvent_t done[kSlots] = {}, tables = nullptr;
};

}  // namespace

struct agx_ctx {
    int device = 0;
    int sms = 148;
    bool has_parms = false;
    uint32_t n = 0, logn = 0, L = 0;
    int le = 0;                                    // 0 = generic kernel
    std::vector<uint32_t> q, psi, n_inv;
    uint2 *d_nat_fwd = nullptr, *d_nat_inv = nullptr;      // natural order, ntt.cpp:298-300 (agx_get_tables)
    uint2 *d_tw_fwd = nullptr, *d_tw_inv = nullptr;        // kernel order (natural, with n^-1 in inverse entry 0, when le == 0)
    uint2 *d_twc_fwd = nullptr, *d_twc_inv = nullptr;      // column-pass tables (two-pass kernels only)
    LimbConst *d_lc = nullptr;
    LimbConst lc0 = {};                                    // limb 0, passed by value in the kernel parameters
    bool r16 = false;                                      // AGX_WITH_R16 builds only
    bool big = false;                                      // n >= 8192 (u32): ntt_big_kernel instead of the radix-2 kernel
#if AGX_WITH_R16
    uint2 *d_tw16_fwd = nullptr, *d_tw16_inv = nullptr, *d_u16_fwd = nullptr, *d_u16_inv = nullptr;
    uint2 u16_fwd0[kR16UInv] = {}, u16_inv0[kR16UInv] = {};   // limb 0's uniform twiddles, passed by value
#endif
    unsigned long long *d_sum = nullptr;
    uint64_t launches = 0;
    // TMA tensor maps over result buffers (forward kernels store through cp.async.bulk.tensor): the encoder entry
    // point of the driver, and the maps of the most recently used (pointer, polynomial count) pairs
    void *encode_tiled = nullptr;
    struct MapSlot { const void *ptr = nullptr; size_t T = 0; int kind = 0; CUtensorMap map; };
    MapSlot maps[8];
    unsigned map_next = 0;
    // u64 parameter set (agx_create64); a context holds either this or the u32 one
    bool has_parms64 = false;
    std::vector<uint64_t> q64, psi64;
    uint64_t *d_tab64 = nullptr;                           // [4][L][n]: roots, companions; forward then inverse
    RnsLimb64 *d_lc64 = nullptr;                           // per-limb modulus constants
    RescaleLimb64 *d_rs64 = nullptr;                       // [L-1] rescale constants (L >= 2, q_{L-1} unlike the others)
    uint64_t rs_qlast = 0, rs_h = 0;                       // q_{L-1} and floor(q_{L-1} / 2)
    BasisLimb64 *d_bl64 = nullptr;                         // [L] limbs, then [L][L] BasisPair64 (ModUp / ModDown)
    BasisPair64 *d_bp64 = nullptr;                         // points into d_bl64's allocation
    // agx_keyswitch64's scratch (gigabytes at real batch sizes): a pool of this context that keeps its memory between
    // calls, so that a call does not map it afresh, as the device's default pool would after every synchronisation
    cudaMemPool_t ks_pool = nullptr;
    double2 *d_slot_tw = nullptr;                          // agx_encode64 / agx_decode64: the special FFT's S twiddles
    std::vector<BasisLimb64> bl64;                         // host copies of both
    std::vector<BasisPair64> bp64;
    HostPipe pipe;
    RefState ref;
    CopyCrew *crew_in = nullptr, *crew_out = nullptr;      // created with the first pageable call
};

namespace {

int select_le(uint32_t logn) {
    switch (logn) {
        case 12: return 6;
        case 11: return 6;
        case 10: return 5;
        default: return 0;
    }
}

// Every entry point makes the context's device current for its own duration and puts the caller's current device
// back on return (a library call must not retarget the caller's later CUDA / torch work).
class DeviceGuard {
    int prev_ = -1;
    cudaError_t err_ = cudaSuccess;
public:
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev_) != cudaSuccess) { cudaGetLastError(); prev_ = -1; }
        if (prev_ != device) err_ = cudaSetDevice(device); else prev_ = -1;
    }
    ~DeviceGuard() { if (prev_ >= 0) cudaSetDevice(prev_); }
    int error() const { return (int)err_; }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};
#define AGX_ON_DEVICE(c)                    \
    DeviceGuard guard__((c)->device);       \
    if (guard__.error()) return guard__.error()

int refresh_r16(agx_ctx *c);

// Per-limb scalars on the host (psi search, inverses, Barrett constants); the n-entry tables themselves are
// computed on the device by gen_tables_kernel.
int build_tables(agx_ctx *c, const uint32_t *psi_in) {
    const uint32_t n = c->n, L = c->L;
    const size_t entries = (size_t)L * n;
    std::vector<LimbConst> lc(L);
    std::vector<LimbGen> lg(L);
    for (uint32_t l = 0; l < L; l++) {
        const uint32_t q = c->q[l];
        uint32_t psi = minimal_psi(n, q);                                 // also validates q (prime, < 2^30, = 1 mod 2n)
        if (!psi) return AGX_E_INVALID;
        if (psi_in) {                                                     // the caller's root: must be a primitive 2n-th root
            psi = psi_in[l];
            if (psi == 0 || psi >= q || powmod_u64(psi, n, q) != q - 1) return AGX_E_INVALID;
        }
        c->psi[l] = psi;
        lg[l] = LimbGen{q, psi, (uint32_t)powmod_u64(psi, q - 2, q), (uint32_t)powmod_u64(n, q - 2, q)};
        int k = 0;
        while ((1ull << k) <= q) k++;                                   // bit length of q
        LimbConst &x = lc[l];
        x.q = q; x.twoq = 2 * q; x.negq = 0u - q; x.neg2q = 0u - 2 * q;
        const uint64_t mu = (uint64_t)((((unsigned __int128)1) << (2 * k)) / q);
        x.bar_mu = (uint32_t)(mu << (31 - k));
        x.bar_sh = (uint32_t)(k - 1);
        x.psi = psi; x.zero = 0;
        c->n_inv[l] = lg[l].n_inv;
    }
    c->lc0 = lc[0];
    CK(cudaMalloc(&c->d_nat_fwd, entries * sizeof(uint2)));
    CK(cudaMalloc(&c->d_nat_inv, entries * sizeof(uint2)));
    CK(cudaMalloc(&c->d_lc, lc.size() * sizeof(LimbConst)));
    CK(cudaMalloc(&c->d_sum, sizeof(unsigned long long)));
    CK(cudaMalloc(&c->d_tw_fwd, entries * sizeof(uint2)));   // generic sizes: natural order with n^-1 in inverse entry 0
    CK(cudaMalloc(&c->d_tw_inv, entries * sizeof(uint2)));
    if (c->le) {
        CK(cudaMalloc(&c->d_twc_fwd, entries * sizeof(uint2)));
        CK(cudaMalloc(&c->d_twc_inv, entries * sizeof(uint2)));
        CK(cudaMemset(c->d_twc_fwd, 0, entries * sizeof(uint2)));
        CK(cudaMemset(c->d_twc_inv, 0, entries * sizeof(uint2)));
    }
    CK(cudaMemcpy(c->d_lc, lc.data(), lc.size() * sizeof(LimbConst), cudaMemcpyHostToDevice));
    LimbGen *d_lg = nullptr;
    CK(cudaMalloc(&d_lg, lg.size() * sizeof(LimbGen)));
    cudaError_t e = cudaMemcpy(d_lg, lg.data(), lg.size() * sizeof(LimbGen), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        const unsigned total = 2u * L * n;
        gen_tables_kernel<<<(total + 255) / 256, 256>>>(c->d_nat_fwd, c->d_nat_inv, c->d_tw_fwd, c->d_tw_inv, c->d_twc_fwd,
                                                        c->d_twc_inv, d_lg, L, c->logn, c->le);
        c->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    cudaFree(d_lg);
    if (e != cudaSuccess) return (int)e;
#if AGX_WITH_R16
    if (c->r16) {
        CK(cudaMalloc(&c->d_tw16_fwd, entries * sizeof(uint2)));
        CK(cudaMalloc(&c->d_tw16_inv, entries * sizeof(uint2)));
        CK(cudaMalloc(&c->d_u16_fwd, (size_t)L * kR16UFwd * sizeof(uint2)));
        CK(cudaMalloc(&c->d_u16_inv, (size_t)L * kR16UInv * sizeof(uint2)));
        return refresh_r16(c);
    }
#endif
    return AGX_OK;
}

KParams kparams(const agx_ctx *c) {
    return KParams{c->d_tw_fwd, c->d_tw_inv, c->d_twc_fwd, c->d_twc_inv, c->d_lc, c->L, c->lc0};
}

enum Op { OP_FWD, OP_INV, OP_MUL, OP_MULSPEC };   // OP_MULSPEC: b is already a spectrum (agx_polymul_by_spectrum)

#ifndef AGX_TMA_STORE
#define AGX_TMA_STORE 1
#endif
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Tensor map over `T` result rows-of-polynomials at `ptr`: {32 words, E/32 halves, T * TPP rows}, box {32, 1, TPP},
// 128-byte swizzle (tma_store_rows).  nullptr when the driver offers no encoder or the shape is out of range: the
// caller then uses the staging-image kernel.
const CUtensorMap *result_map(agx_ctx *c, void *ptr, size_t T, uint32_t E, uint32_t TPP) {
    if (!AGX_TMA_STORE || !c->encode_tiled || (reinterpret_cast<uintptr_t>(ptr) & 15) || T * TPP > 0x7fffffffull) return nullptr;   // box coordinates are signed 32-bit
    for (auto &m : c->maps)
        if (m.ptr == ptr && m.T == T && m.kind == 0) return &m.map;
    agx_ctx::MapSlot &m = c->maps[c->map_next++ % 8];
    const cuuint64_t gdim[3] = {32, E / 32, (cuuint64_t)T * TPP};
    const cuuint64_t gstr[2] = {128, (cuuint64_t)E * 4};
    const cuuint32_t box[3] = {32, 1, TPP}, estr[3] = {1, 1, 1};
    const CUresult r = reinterpret_cast<EncodeTiledFn>(c->encode_tiled)(
        &m.map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { m.ptr = nullptr; return nullptr; }
    m.ptr = ptr; m.T = T; m.kind = 0;
    return &m.map;
}

#if AGX_WITH_R16
// Tensor map of the radix-16 kernels: the batch as rows of 32 words, {32, T * n/32}, box {32, n/32} = one polynomial
// as a dense 128-byte-swizzled tile; serves the forward kernel's store and the inverse kernel's load.
const CUtensorMap *tile_map(agx_ctx *c, const void *ptr, size_t T, uint32_t n) {
    const uint32_t rows = n / 32;
    if (!c->encode_tiled || (reinterpret_cast<uintptr_t>(ptr) & 15) || T * rows > 0x7fffffffull || rows > 256) return nullptr;
    for (auto &m : c->maps)
        if (m.ptr == ptr && m.T == T && m.kind == 1) return &m.map;
    agx_ctx::MapSlot &m = c->maps[c->map_next++ % 8];
    const cuuint64_t gdim[2] = {32, (cuuint64_t)T * rows};
    const cuuint64_t gstr[1] = {128};
    const cuuint32_t box[2] = {32, rows}, estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<EncodeTiledFn>(c->encode_tiled)(
        &m.map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void *>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { m.ptr = nullptr; return nullptr; }
    m.ptr = ptr; m.T = T; m.kind = 1;
    return &m.map;
}

// (Re)derives what the radix-16 kernels read from the context's natural-order tables: the kernel-order copies and
// the uniform twiddles of the first forward / last inverse pass (entries k < 16, the inverse ones with n^-1 folded in).
int refresh_r16(agx_ctx *c) {
    if (!c->r16) return AGX_OK;
    const uint32_t n = c->n, L = c->L, entries = L * n;
    r16_relayout_kernel<<<(entries + 255) / 256, 256>>>(c->d_tw16_fwd, c->d_nat_fwd, c->logn, entries);
    r16_relayout_kernel<<<(entries + 255) / 256, 256>>>(c->d_tw16_inv, c->d_nat_inv, c->logn, entries);
    c->launches += 2;
    CK(cudaGetLastError());
    std::vector<uint2> uf((size_t)L * kR16UFwd), ui((size_t)L * kR16UInv), nat(16);
    for (uint32_t l = 0; l < L; l++) {
        const uint64_t q = c->q[l], s = c->n_inv[l];
        auto pair = [&](uint64_t w) { return make_uint2((uint32_t)w, (uint32_t)((w << 32) / q)); };
        CK(cudaMemcpy(nat.data(), c->d_nat_fwd + (size_t)l * n, 16 * sizeof(uint2), cudaMemcpyDeviceToHost));
        for (int k = 0; k < 16; k++) uf[(size_t)l * kR16UFwd + k] = nat[k];
        CK(cudaMemcpy(nat.data(), c->d_nat_inv + (size_t)l * n, 16 * sizeof(uint2), cudaMemcpyDeviceToHost));
        uint2 *u = ui.data() + (size_t)l * kR16UInv;
        for (int g = 0; g < 8; g++) u[g] = pair(mulmod_u64(nat[8 + g].x, s, q));
        for (int g = 0; g < 4; g++) { u[8 + g] = pair(mulmod_u64(nat[4 + g].x, s, q)); u[12 + g] = nat[4 + g]; }
        for (int g = 0; g < 2; g++) { u[16 + g] = pair(mulmod_u64(nat[2 + g].x, s, q)); u[18 + g] = nat[2 + g]; }
        u[20] = nat[1]; u[21] = pair(s); u[22] = pair(mulmod_u64(nat[1].x, s, q)); u[23] = make_uint2(0, 0);
    }
    CK(cudaMemcpy(c->d_u16_fwd, uf.data(), uf.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_u16_inv, ui.data(), ui.size() * sizeof(uint2), cudaMemcpyHostToDevice));
    for (int k = 0; k < kR16UInv; k++) { c->u16_fwd0[k] = k < kR16UFwd ? uf[k] : make_uint2(0, 0); c->u16_inv0[k] = ui[k]; }
    return AGX_OK;
}

R16Params r16params(const agx_ctx *c, bool inverse) {
    R16Params p{c->d_tw16_fwd, c->d_tw16_inv, c->d_u16_fwd, c->d_u16_inv, c->d_lc, c->L, c->lc0, {}};
    for (int k = 0; k < kR16UInv; k++) p.u[k] = inverse ? c->u16_inv0[k] : c->u16_fwd0[k];
    return p;
}
#else
int refresh_r16(agx_ctx *) { return AGX_OK; }
#endif

template <int LOGN, int LE, bool CL>
int launch_fast(agx_ctx *c, Op op, uint32_t *out, const uint32_t *a, const uint32_t *b, size_t T, cudaStream_t s) {
    using G = Geo<LOGN, LE>;
    const KParams p = kparams(c);
    const dim3 grid((unsigned)T), block(G::TPP);
    const uint32_t Tu = (uint32_t)T;
    static const CUtensorMap no_map = {};          // kernels instantiated without the TMA store ignore their map
#define AGX_FWD(dst, src)                                                                                              \
    do {                                                                                                               \
        if (const CUtensorMap *tm = result_map(c, dst, T, G::E, G::TPP))                                               \
            ntt_fwd_loop_kernel<LOGN, LE, false, CL, true><<<grid, block, 0, s>>>(dst, src, nullptr, p, Tu, *tm);      \
        else                                                                                                           \
            ntt_fwd_loop_kernel<LOGN, LE, false, CL, false><<<grid, block, 0, s>>>(dst, src, nullptr, p, Tu, no_map);  \
    } while (0)
#define AGX_INV(dst) ntt_inv_loop_kernel<LOGN, LE, CL><<<grid, block, 0, s>>>(dst, p, Tu)
    if (op == OP_FWD) {
        AGX_FWD(out, out);
        c->launches++;
    } else if (op == OP_INV) {
        AGX_INV(out);
        c->launches++;
    } else if (op == OP_MULSPEC) {
        // b is NTT(b) already: out = NTT(a) .* b (forward kernel with the pointwise epilogue, lazily reduced); out = INTT(out)
        if (const CUtensorMap *tm = result_map(c, out, T, G::E, G::TPP))
            ntt_fwd_loop_kernel<LOGN, LE, true, CL, true><<<grid, block, 0, s>>>(out, a, b, p, Tu, *tm);
        else
            ntt_fwd_loop_kernel<LOGN, LE, true, CL, false><<<grid, block, 0, s>>>(out, a, b, p, Tu, no_map);
        AGX_INV(out);
        c->launches += 2;
    } else if constexpr (LOGN <= 10) {
        // n = 1024: forward(a), forward(b), pointwise, inverse fused in one launch (its 28 KB of code fits the
        // instruction cache; at n >= 2048 the fused kernel is 57-60 KB and runs 30 % slower than the split below)
        polymul_loop_kernel<LOGN, LE, CL><<<grid, block, 0, s>>>(out, a, b, p);
        c->launches++;
    } else {
        // three launches, no scratch buffer: out = NTT(a); out = NTT(b) .* out; out = INTT(out)
        if (out == b && out != a) { const uint32_t *t = a; a = b; b = t; }     // the product commutes
        AGX_FWD(out, a);
        if (a == b) {                                                          // squaring: out already holds NTT(b)
            const size_t total = T * G::N;
            pointwise_generic_kernel<0><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(out, out, c->d_lc, c->L, LOGN, total);
        } else {
            if (const CUtensorMap *tm = result_map(c, out, T, G::E, G::TPP))
                ntt_fwd_loop_kernel<LOGN, LE, true, CL, true><<<grid, block, 0, s>>>(out, b, out, p, Tu, *tm);
            else
                ntt_fwd_loop_kernel<LOGN, LE, true, CL, false><<<grid, block, 0, s>>>(out, b, out, p, Tu, no_map);
        }
        AGX_INV(out);
        c->launches += 3;
    }
#undef AGX_FWD
#undef AGX_INV
    return (int)cudaGetLastError();
}

// one transform per (polynomial, limb) row of `d`, in place, at a size outside {1024, 2048, 4096}: n >= 8192 through the
// register-radix passes of ntt_big_kernel, smaller sizes (and AGX_GENERIC_ONLY=1) through the radix-2 kernel
void launch_generic_ntt(agx_ctx *c, bool inverse, uint32_t *d, size_t T, cudaStream_t s) {
    const uint2 *tw = inverse ? c->d_tw_inv : c->d_tw_fwd;
    if (c->big) {
        const size_t smem = ((size_t)c->n + c->n / 32) * 4;
        const unsigned threads = c->logn <= 14 ? 512 : 1024;   // two CTAs per SM cover each other's barriers where they fit
#define AGX_BIG(LOGN)                                                                                 \
    do {                                                                                              \
        if (inverse) ntt_big_kernel<true, LOGN><<<(unsigned)T, threads, smem, s>>>(d, tw, c->d_lc, c->L);  \
        else ntt_big_kernel<false, LOGN><<<(unsigned)T, threads, smem, s>>>(d, tw, c->d_lc, c->L);         \
    } while (0)
        if (c->logn == 13) AGX_BIG(13); else if (c->logn == 14) AGX_BIG(14); else AGX_BIG(15);
#undef AGX_BIG
    } else {
        const size_t smem = (size_t)c->n * 4;
        const unsigned threads = c->n / 2 < 256 ? (c->n / 2 < 32 ? 32 : c->n / 2) : 256;
        if (inverse) ntt_generic_kernel<true><<<(unsigned)T, threads, smem, s>>>(d, tw, c->d_lc, c->L, c->logn);
        else ntt_generic_kernel<false><<<(unsigned)T, threads, smem, s>>>(d, tw, c->d_lc, c->L, c->logn);
    }
    c->launches++;
}

int launch_generic(agx_ctx *c, Op op, uint32_t *out, const uint32_t *a, const uint32_t *b, size_t T, cudaStream_t s) {
    if (op == OP_FWD) {
        launch_generic_ntt(c, false, out, T, s);
    } else if (op == OP_INV) {
        launch_generic_ntt(c, true, out, T, s);
    } else if (op == OP_MULSPEC) {
        // generic sizes, b already a spectrum: out <- NTT(a); out <- INTT(out .* b).  When out is b's buffer the spectrum
        // is moved to a stream-ordered scratch buffer first.
        const size_t bytes = T * c->n * 4, total = T * c->n;
        uint32_t *tmp = nullptr;
        cudaError_t e = cudaSuccess;
        if (out == b) {
            e = cudaMallocAsync(&tmp, bytes, s);
            if (e == cudaSuccess) e = cudaMemcpyAsync(tmp, b, bytes, cudaMemcpyDeviceToDevice, s);
            b = tmp;
        }
        if (e == cudaSuccess && out != a) e = cudaMemcpyAsync(out, a, bytes, cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess) {
            launch_generic_ntt(c, false, out, T, s);
            pointwise_generic_kernel<0><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(out, b, c->d_lc, c->L, c->logn, total);
            c->launches++;
            launch_generic_ntt(c, true, out, T, s);
            e = cudaGetLastError();
        }
        if (tmp) { const cudaError_t ef = cudaFreeAsync(tmp, s); if (e == cudaSuccess) e = ef; }
        return (int)e;
    } else {
        // generic sizes: out <- NTT(a), tmp <- NTT(b) in a stream-ordered scratch buffer, out <- INTT(out .* tmp).
        // Every aliasing case of the fast path is served: the product commutes (out == b), squaring needs no scratch.
        if (out == b && out != a) { const uint32_t *t = a; a = b; b = t; }
        const size_t bytes = T * c->n * 4, total = T * c->n;
        uint32_t *tmp = nullptr;
        cudaError_t e = cudaSuccess;
        if (out != a) e = cudaMemcpyAsync(out, a, bytes, cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess && a != b) {
            e = cudaMallocAsync(&tmp, bytes, s);
            if (e == cudaSuccess) e = cudaMemcpyAsync(tmp, b, bytes, cudaMemcpyDeviceToDevice, s);
        }
        if (e == cudaSuccess) {
            launch_generic_ntt(c, false, out, T, s);
            if (tmp) launch_generic_ntt(c, false, tmp, T, s);
            pointwise_generic_kernel<0><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(out, tmp ? tmp : out, c->d_lc, c->L, c->logn, total);
            c->launches++;
            launch_generic_ntt(c, true, out, T, s);
            e = cudaGetLastError();
        }
        if (tmp) { const cudaError_t ef = cudaFreeAsync(tmp, s); if (e == cudaSuccess) e = ef; }   // freed on every path
        return (int)e;
    }
    return (int)cudaGetLastError();
}

#if AGX_WITH_R16
// n = 4096 through the radix-16 three-pass kernels; false when a tensor map cannot be encoded for these buffers (the
// caller then takes the two-pass kernels, which serve every case)
template <bool CL>
bool launch_r16(agx_ctx *c, Op op, uint32_t *out, const uint32_t *a, const uint32_t *b, size_t T, cudaStream_t s, int *rc) {
    using G = R16<12>;
    const CUtensorMap *tm = tile_map(c, out, T, G::N);
    if (!tm) return false;
    const dim3 grid((unsigned)T), block(G::TPP);
    const uint32_t Tu = (uint32_t)T;
    if (op == OP_FWD) {
        r16_fwd_kernel<12, false, CL><<<grid, block, 0, s>>>(out, out, nullptr, r16params(c, false), Tu, *tm);
        c->launches++;
    } else if (op == OP_INV) {
        r16_inv_kernel<12, CL><<<grid, block, 0, s>>>(out, r16params(c, true), Tu, *tm);
        c->launches++;
    } else {
        // three launches, no scratch buffer: out = NTT(a); out = NTT(b) .* out; out = INTT(out)
        if (out == b && out != a) { const uint32_t *t = a; a = b; b = t; }     // the product commutes
        r16_fwd_kernel<12, false, CL><<<grid, block, 0, s>>>(out, a, nullptr, r16params(c, false), Tu, *tm);
        if (a == b) {
            const size_t total = T * G::N;
            pointwise_generic_kernel<0><<<(unsigned)((total + 255) / 256), 256, 0, s>>>(out, out, c->d_lc, c->L, 12, total);
        } else {
            r16_fwd_kernel<12, true, CL><<<grid, block, 0, s>>>(out, b, out, r16params(c, false), Tu, *tm);
        }
        r16_inv_kernel<12, CL><<<grid, block, 0, s>>>(out, r16params(c, true), Tu, *tm);
        c->launches += 3;
    }
    *rc = (int)cudaGetLastError();
    return true;
}
#endif

int launch(agx_ctx *c, Op op, uint32_t *out, const uint32_t *a, const uint32_t *b, size_t B, cudaStream_t s) {
    const size_t T = B * c->L;
    if (T == 0) return AGX_OK;
    if (T > 0x7fffffffull) return AGX_E_INVALID;
#if AGX_WITH_R16
    if (c->r16 && op != OP_MULSPEC) {
        int rc = 0;
        if (c->L == 1 ? launch_r16<true>(c, op, out, a, b, T, s, &rc) : launch_r16<false>(c, op, out, a, b, T, s, &rc)) return rc;
    }
#endif
    switch (c->le ? c->logn : 0) {
        // single-limb batches run the instantiation whose modulus constants are constant-bank operands
        case 12: return c->L == 1 ? launch_fast<12, 6, true>(c, op, out, a, b, T, s) : launch_fast<12, 6, false>(c, op, out, a, b, T, s);
        case 11: return c->L == 1 ? launch_fast<11, 6, true>(c, op, out, a, b, T, s) : launch_fast<11, 6, false>(c, op, out, a, b, T, s);
        case 10: return c->L == 1 ? launch_fast<10, 5, true>(c, op, out, a, b, T, s) : launch_fast<10, 5, false>(c, op, out, a, b, T, s);
        default: return launch_generic(c, op, out, a, b, T, s);
    }
}

int check_dev_call(agx_ctx *c, const void *p, size_t B) {
    if (!c || !c->has_parms) return AGX_E_INVALID;
    if (B && !p) return AGX_E_INVALID;
    if (reinterpret_cast<uintptr_t>(p) & 15) return AGX_E_INVALID;   // 16-byte vector accesses and tensor copies
    return AGX_OK;
}

// ------------------------------------------------------------------------------------------- host pipeline

bool is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Pageable callers: results are staged in pinned chunks and copied to the caller's buffer by a helper thread (with its own
// CopyCrew), so that the copy-out of chunk i runs beside the staging-in of chunk i+1 on the calling thread.  Chunks are
// drained strictly in order.
class OutDrainer {
    struct Item { void *dst; const void *src; size_t bytes; cudaEvent_t ev; };
    Item items_[kSlots] = {};
    std::atomic<size_t> issued_{0}, drained_{0};
    std::atomic<int> err_{0};
    std::atomic<bool> stop_{false};
    std::thread th_;
    bool inline_ = false;
    int device_;
    CopyCrew *crew_;
    void run() {
        cudaSetDevice(device_);
        for (size_t i = 0;; i++) {
            while (issued_.load(std::memory_order_acquire) <= i) {
                if (stop_.load(std::memory_order_acquire)) return;
                std::this_thread::yield();
            }
            const Item it = items_[i % kSlots];
            const cudaError_t e = cudaEventSynchronize(it.ev);
            if (e != cudaSuccess) err_.store((int)e);
            else if (crew_) crew_->copy(it.dst, it.src, it.bytes);
            else memcpy(it.dst, it.src, it.bytes);
            drained_.store(i + 1, std::memory_order_release);
        }
    }
public:
    explicit OutDrainer(int device, CopyCrew *crew = nullptr) : device_(device), crew_(crew) {}
    ~OutDrainer() { finish(); }
    // before chunk i reuses its slot's staging buffers: chunk i - kSlots must have been copied out
    void wait_slot_free(size_t i) {
        if (i < (size_t)kSlots) return;
        while (drained_.load(std::memory_order_acquire) < i - kSlots + 1) std::this_thread::yield();
    }
    void submit(size_t i, void *dst, const void *src, size_t bytes, cudaEvent_t ev) {
        if (!th_.joinable() && !inline_) {
            try { th_ = std::thread(&OutDrainer::run, this); } catch (...) { inline_ = true; }   // nothing throws across the C ABI
        }
        if (inline_) {                                   // no helper thread to be had: drain on the calling thread
            const cudaError_t e = cudaEventSynchronize(ev);
            if (e != cudaSuccess) err_.store((int)e);
            else if (crew_) crew_->copy(dst, src, bytes);
            else memcpy(dst, src, bytes);
            issued_.store(i + 1, std::memory_order_release);
            drained_.store(i + 1, std::memory_order_release);
            return;
        }
        items_[i % kSlots] = Item{dst, src, bytes, ev};
        issued_.store(i + 1, std::memory_order_release);
    }
    int finish() {
        if (th_.joinable()) {
            while (drained_.load(std::memory_order_acquire) < issued_.load(std::memory_order_acquire)) std::this_thread::yield();
            stop_.store(true, std::memory_order_release);
            th_.join();
        }
        return err_.load();
    }
};

int ensure_crews(agx_ctx *c) {
    try {                                              // thread creation can fail; nothing may throw across the C ABI
        if (!c->crew_in) c->crew_in = new CopyCrew();
        if (!c->crew_out) c->crew_out = new CopyCrew();
    } catch (...) {
        return AGX_E_NOMEM;
    }
    return AGX_OK;
}

int pipe_prepare(agx_ctx *c, bool need_b, bool need_stage) {
    HostPipe &P = c->pipe;
    if (!P.stream[0]) {
        for (int i = 0; i < kSlots; i++) {
            CK(cudaStreamCreateWithFlags(&P.stream[i], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&P.done[i], cudaEventDisableTiming));
        }
        const size_t poly_bytes = (size_t)c->L * c->n * 4;
        // two waves of transform CTAs per chunk (a wave is SMs x 128 KiB of rows at n = 4096 and 2048): a chunk's kernel takes
        // whole waves' time, and that time is added to the copy engines' period (profiles/pipeline_timeline.py); 37 MiB on a
        // B200 against the former 32: 1.408-1.412 -> 1.416-1.419 M pairs/s end to end in one call
        size_t chunk_bytes = c->sms > 0 ? (size_t)c->sms << 18 : kChunkBytes;
        if (const char *e = getenv("AGX_HOST_CHUNK_MB")) {            // tuning knob for the host pipeline
            const long mb = atol(e);
            if (mb >= 1 && mb <= 1024) chunk_bytes = (size_t)mb << 20;
        }
        size_t polys = chunk_bytes / poly_bytes;
        if (polys == 0) polys = 1;
        P.cap = polys * poly_bytes;
        for (int i = 0; i < kSlots; i++) CK(cudaMalloc(&P.d_a[i], P.cap));
    }
    if (need_b && !P.have_b) {
        for (int i = 0; i < kSlots; i++) CK(cudaMalloc(&P.d_b[i], P.cap));
        P.have_b = true;
    }
    if (need_stage && !P.have_stage) {
        for (int i = 0; i < kSlots; i++) {
            CK(cudaHostAlloc(&P.p_in[i], P.cap, cudaHostAllocDefault));
            CK(cudaHostAlloc(&P.p_in2[i], P.cap, cudaHostAllocDefault));
            CK(cudaHostAlloc(&P.p_out[i], P.cap, cudaHostAllocDefault));
        }
        P.have_stage = true;
    }
    return AGX_OK;
}

// Chunked pipeline: slot i%3 carries H2D -> kernel -> D2H on its own stream, so the copy engines and the SMs
// overlap across slots (the GPU analogue of the reference's concurrently running loader/compute/drain kernels).
int run_host(agx_ctx *c, Op op, const uint32_t *h_a, const uint32_t *h_b, uint32_t *h_out, size_t B) {
    if (!c || !c->has_parms) return AGX_E_INVALID;
    if (B == 0) return AGX_OK;
    const bool two = op == OP_MUL || op == OP_MULSPEC;
    if (!h_a || !h_out || (two && !h_b)) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    const bool pin_a = is_pinned(h_a), pin_b = !two || is_pinned(h_b), pin_o = is_pinned(h_out);
    int rc = pipe_prepare(c, two, !(pin_a && pin_b && pin_o));
    if (rc) return rc;
    HostPipe &P = c->pipe;
    const size_t poly_words = (size_t)c->L * c->n, poly_bytes = poly_words * 4;
    const size_t chunk_polys = P.cap / poly_bytes;
    if (!(pin_a && pin_b && pin_o) && (rc = ensure_crews(c)) != AGX_OK) return rc;
    OutDrainer drain(c->device, c->crew_out);
    // One way out: whatever fails, no copy may still be touching the caller's memory when this function returns.
    auto finish = [&](int code) {
        for (int k = 0; k < kSlots; k++) {
            const cudaError_t e = cudaStreamSynchronize(P.stream[k]);
            if (!code && e != cudaSuccess) code = (int)e;
        }
        const int d = drain.finish();
        return code ? code : d;
    };
#define STEP(call) do { const cudaError_t e__ = (call); if (e__ != cudaSuccess) return finish((int)e__); } while (0)
    size_t done = 0;
    for (size_t i = 0; done < B; i++) {
        const int sl = (int)(i % kSlots);
        const size_t cnt = B - done < chunk_polys ? B - done : chunk_polys, bytes = cnt * poly_bytes;
        const size_t off = done * poly_words;
        if (i >= (size_t)kSlots) {                       // slot reuse: its previous chunk must have drained
            if (!pin_o) drain.wait_slot_free(i);
            else if (!pin_a || !pin_b) STEP(cudaEventSynchronize(P.done[sl]));
        }
        const uint32_t *src_a = h_a + off;
        if (!pin_a) { c->crew_in->copy(P.p_in[sl], src_a, bytes); src_a = P.p_in[sl]; }
        STEP(cudaMemcpyAsync(P.d_a[sl], src_a, bytes, cudaMemcpyHostToDevice, P.stream[sl]));
        if (two) {
            const uint32_t *src_b = h_b + off;
            if (!pin_b) { c->crew_in->copy(P.p_in2[sl], src_b, bytes); src_b = P.p_in2[sl]; }
            STEP(cudaMemcpyAsync(P.d_b[sl], src_b, bytes, cudaMemcpyHostToDevice, P.stream[sl]));
        }
        rc = launch(c, op, P.d_a[sl], P.d_a[sl], P.d_b[sl], cnt, P.stream[sl]);
        if (rc) return finish(rc);
        uint32_t *dst = h_out + off;
        STEP(cudaMemcpyAsync(pin_o ? dst : P.p_out[sl], P.d_a[sl], bytes, cudaMemcpyDeviceToHost, P.stream[sl]));
        STEP(cudaEventRecord(P.done[sl], P.stream[sl]));
        if (!pin_o) drain.submit(i, dst, P.p_out[sl], bytes, P.done[sl]);
        done += cnt;
    }
#undef STEP
    return finish(AGX_OK);
}

void pipe_destroy(HostPipe &P) {
    for (int i = 0; i < kSlots; i++) {
        if (P.stream[i]) cudaStreamDestroy(P.stream[i]);
        if (P.done[i]) cudaEventDestroy(P.done[i]);
        cudaFree(P.d_a[i]); cudaFree(P.d_b[i]);
        if (P.p_in[i]) cudaFreeHost(P.p_in[i]);
        if (P.p_in2[i]) cudaFreeHost(P.p_in2[i]);
        if (P.p_out[i]) cudaFreeHost(P.p_out[i]);
    }
    P = HostPipe{};
}

// ------------------------------------------------------------------------------- reference-shaped u64 kernels

// The forward transform of `frames` frames resident on the device (frame b: low half from in[b*N ..), high half from
// in2[b*N + N/2 ..), ntt.cpp:582-591; out must not alias the inputs unless in == in2 == out).
int ref_launch(agx_ctx *c, uint32_t logn, const uint64_t *d_in, const uint64_t *d_in2, uint64_t *d_out, const uint64_t *d_tw,
               const uint64_t *d_pre, uint64_t modulus, size_t frames, cudaStream_t st) {
    const uint32_t N = 1u << logn;
    const size_t frame_bytes = (size_t)N * 8;
    static const bool naive = getenv("AGX_REF_NAIVE") != nullptr;   // A/B knobs: one-CTA-per-frame radix-2 kernel,
    static const bool passes_only = getenv("AGX_REF_PASSES") != nullptr;   // ... the multi-launch pass kernels
    // One launch, frame resident in shared memory (two CTAs per frame at N = 32768, which is unsafe in place: the CTA of
    // one half would overwrite what the other has not read yet).  Splitting N = 16384 the same way -- two independent
    // 8192-point halves per SM instead of one 136 KB CTA, which cover each other's barriers and load phases -- measured
    // +5 % on a 1 GiB batch and -5 % on a 16 MiB chunk (less than a wave of CTAs either way), so it is done for batches of
    // at least two waves of whole-frame CTAs when the output is a separate buffer (AGX_REF_SPLIT14=0 / 1: never / always).
    const bool in_place = d_out == d_in || d_out == d_in2;
    static const char *split14_env = getenv("AGX_REF_SPLIT14");
    const bool split14 = logn == 14 && !in_place &&
                         (split14_env ? split14_env[0] == '1' : frames >= (size_t)2 * (size_t)c->sms);
    if (logn >= 10 && !naive && !passes_only && !(logn == 15 && in_place)) {
        const uint32_t split = (logn == 15 || split14) ? 1u : 0u, lg = logn - split;
        const size_t smem = ((size_t)17 << (lg - 4)) * 8;
        const unsigned grid = (unsigned)(frames << split);
        // N/32 threads per CTA, two virtual threads each (512 at N = 16384, the largest frame an SM holds): below that
        // several independent CTAs share an SM and cover each other's barriers and load phases
        switch (lg) {
            case 14: ref_u64_frame_kernel<512><<<grid, 512, smem, st>>>(d_in, d_in2, d_out, d_tw, d_pre, modulus, logn, split); break;
            case 13: ref_u64_frame_kernel<256><<<grid, 256, smem, st>>>(d_in, d_in2, d_out, d_tw, d_pre, modulus, logn, split); break;
            case 12: ref_u64_frame_kernel<128><<<grid, 128, smem, st>>>(d_in, d_in2, d_out, d_tw, d_pre, modulus, logn, split); break;
            case 11: ref_u64_frame_kernel<64><<<grid, 64, smem, st>>>(d_in, d_in2, d_out, d_tw, d_pre, modulus, logn, split); break;
            default: ref_u64_frame_kernel<32><<<grid, 32, smem, st>>>(d_in, d_in2, d_out, d_tw, d_pre, modulus, logn, split); break;
        }
        c->launches++;
        return (int)cudaGetLastError();
    }
    if (logn >= 10 && !naive) {
        // register-radix passes over the L2-resident chunk: logN - 4 strided stages in groups of <= 4, then the
        // last 4 stages on contiguous 16-coefficient runs (with the final reduction)
        uint32_t s0 = 0, left = logn - 4, passes = (logn - 4 + 3) / 4;   // 11 -> 4,4,3; 10 -> 4,3,3; 9 -> 3,3,3; 6 -> 3,3
        const uint64_t *src = d_in, *src2 = d_in2;
        for (; passes; passes--) {
            const uint32_t ls = (left + passes - 1) / passes;
            const unsigned blocks = (unsigned)((frames << (logn - ls)) + 255) / 256;
            if (ls == 4) ref_u64_strided_pass_kernel<4><<<blocks, 256, 0, st>>>(src, src2, d_out, d_tw, d_pre, modulus, logn, s0, (uint32_t)frames);
            else         ref_u64_strided_pass_kernel<3><<<blocks, 256, 0, st>>>(src, src2, d_out, d_tw, d_pre, modulus, logn, s0, (uint32_t)frames);
            c->launches++;
            src = src2 = d_out;
            s0 += ls; left -= ls;
        }
        ref_u64_last_pass_kernel<<<(unsigned)((frames << (logn - 4)) + 127) / 128, 128, 0, st>>>(d_out, d_tw, d_pre, modulus, logn, (uint32_t)frames);
        c->launches++;
    } else {
        const int use_smem = frame_bytes <= (128u << 10);
        const unsigned threads = N / 2 < 1024 ? (N / 2 < 32 ? 32 : N / 2) : 1024;
        ref_fwd_u64_kernel<<<(unsigned)frames, threads, use_smem ? frame_bytes : 0, st>>>(d_in, d_in2, d_out, d_tw, d_pre, modulus, logn, use_smem);
        c->launches++;
    }
    return (int)cudaGetLastError();
}

// The inverse transform of `frames` frames [frames][N] (bit-reversed in, natural out, results in [0,q)), with the
// pointwise product by d_mul fused into its load when d_mul is not null.  d_out may equal d_in and/or d_mul.
// Odd modulus, 3 <= q < 2^62 (checked by the callers).
// The inverse's constants of an odd modulus 3 <= q < 2^62 at size 2^logn.
RefInvConst ref_inv_const(uint64_t q, uint32_t logn) {
    typedef unsigned __int128 u128;
    RefInvConst p{};
    p.q = q;
    uint64_t half = (q + 1) / 2, ninv = 1;                         // n^-1 = ((q+1)/2)^logn mod q
    for (uint32_t i = 0; i < logn; i++) ninv = (uint64_t)((u128)ninv * half % q);
    p.ninv = ninv;
    p.ninv_p = (uint64_t)(((u128)ninv << 64) / q);
    p.k = 64 - (uint32_t)__builtin_clzll(q);
    p.mu = (uint64_t)(((u128)1 << (2 * p.k)) / q);
    p.recip = (uint64_t)(((u128)1 << (63 + p.k)) / q);
    return p;
}

int ref_inv_launch(agx_ctx *c, uint32_t logn, const uint64_t *d_in, const uint64_t *d_mul, uint64_t *d_out,
                   const uint64_t *d_itw, const uint64_t *d_ipre, uint64_t q, size_t frames, cudaStream_t st) {
    const RefInvConst p = ref_inv_const(q, logn);
    if (logn >= 10) {
        // one CTA per frame up to N = 16384; two per frame and a streaming last stage at N = 32768
        const uint32_t split = logn == 15 ? 1u : 0u, lg = logn - split;
        const size_t smem = ((size_t)17 << (lg - 4)) * 8;
        const unsigned grid = (unsigned)(frames << split);
        switch (lg) {
            case 14: ref_u64_inv_frame_kernel<512><<<grid, 512, smem, st>>>(d_in, d_mul, d_out, d_itw, d_ipre, p, logn); break;
            case 13: ref_u64_inv_frame_kernel<256><<<grid, 256, smem, st>>>(d_in, d_mul, d_out, d_itw, d_ipre, p, logn); break;
            case 12: ref_u64_inv_frame_kernel<128><<<grid, 128, smem, st>>>(d_in, d_mul, d_out, d_itw, d_ipre, p, logn); break;
            case 11: ref_u64_inv_frame_kernel<64><<<grid, 64, smem, st>>>(d_in, d_mul, d_out, d_itw, d_ipre, p, logn); break;
            default: ref_u64_inv_frame_kernel<32><<<grid, 32, smem, st>>>(d_in, d_mul, d_out, d_itw, d_ipre, p, logn); break;
        }
        c->launches++;
        if (split) {
            const size_t units = frames << (logn - 2);
            const unsigned blocks = (unsigned)std::min<size_t>((units + 255) / 256, (size_t)c->sms * 8);
            ref_u64_inv_last_stage_kernel<<<blocks, 256, 0, st>>>(d_out, d_itw, p, logn, frames);
            c->launches++;
        }
    } else {
        const uint32_t N = 1u << logn;
        const unsigned threads = N / 2 < 32 ? 32 : N / 2;
        ref_inv_u64_kernel<<<(unsigned)frames, threads, 0, st>>>(d_in, d_mul, d_out, d_itw, d_ipre, p, logn);
        c->launches++;
    }
    return (int)cudaGetLastError();
}

// Argument checks shared by the u64 inverse and product entry points: AGX_OK, or AGX_E_INVALID with *logn untouched.
int ref_inv_check(agx_ctx *c, uint32_t N, std::initializer_list<const void *> ptrs, uint64_t modulus, uint32_t *logn) {
    if (!c || N < 4 || N > 32768 || (N & (N - 1))) return AGX_E_INVALID;
    // odd, and the lazy range [0,4q) inside 64 bits; q = 1 has no Barrett constants
    if (!(modulus & 1) || modulus >= (1ull << 62) || modulus < 3) return AGX_E_INVALID;
    for (const void *p : ptrs)                                    // frames and tables are read by 16-byte accesses
        if (!p || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    uint32_t l = 0;
    while ((1u << l) < N) l++;
    *logn = l;
    return AGX_OK;
}

// ------------------------------------------------------------------------------------- u64 RNS batches

// The library's tables of the u64 parameter set: forward roots, forward companions, inverse roots, inverse companions.
const uint64_t *tab64(const agx_ctx *c, int which) { return c->d_tab64 + (size_t)which * c->L * c->n; }

// Forward transform of T frames [T][n], in -> out (in == out or disjoint): one launch.  The frames are a
// [T / count][count][n] batch over the context's limbs first .. first + count - 1 (the whole context: first = 0,
// count = L).  N = 32768 runs the 2-CTA cluster kernel, which is safe in place.
int rns_fwd_launch(agx_ctx *c, const uint64_t *in, uint64_t *out, size_t T, cudaStream_t st, uint32_t first,
                   uint32_t count) {
    const uint32_t logn = c->logn, L = count;
    const size_t toff = (size_t)first << logn;
    const uint64_t *tw = tab64(c, 0) + toff, *pre = tab64(c, 1) + toff;
    const RnsLimb64 *lc = c->d_lc64 + first;
    const unsigned grid = (unsigned)T;
    const size_t smem = logn >= 10 ? ((size_t)17 << (std::min(logn, 14u) - 4)) * 8 : 0;
    switch (logn) {
        case 15: ref_u64_rns_frame_pair_kernel<<<2 * grid, 512, smem, st>>>(in, out, tw, pre, lc, L); break;
        case 14: ref_u64_rns_frame_kernel<512><<<grid, 512, smem, st>>>(in, out, tw, pre, lc, L, logn); break;
        case 13: ref_u64_rns_frame_kernel<256><<<grid, 256, smem, st>>>(in, out, tw, pre, lc, L, logn); break;
        case 12: ref_u64_rns_frame_kernel<128><<<grid, 128, smem, st>>>(in, out, tw, pre, lc, L, logn); break;
        case 11: ref_u64_rns_frame_kernel<64><<<grid, 64, smem, st>>>(in, out, tw, pre, lc, L, logn); break;
        case 10: ref_u64_rns_frame_kernel<32><<<grid, 32, smem, st>>>(in, out, tw, pre, lc, L, logn); break;
        default: {
            const uint32_t N = 1u << logn;
            ref_fwd_u64_rns_kernel<<<grid, N / 2 < 32 ? 32 : N / 2, (size_t)N * 8, st>>>(in, out, tw, pre, lc, L, logn);
        }
    }
    c->launches++;
    return (int)cudaGetLastError();
}

// Inverse of T frames, times d_mul on load when not null (ref_inv_launch's geometry): one launch, two at N = 32768.
// The frames are a [T / count][count][n] batch over the context's limbs first .. first + count - 1 (the whole context:
// first = 0, count = L).
int rns_inv_launch(agx_ctx *c, const uint64_t *in, const uint64_t *mul, uint64_t *out, size_t T, cudaStream_t st,
                   uint32_t first, uint32_t count) {
    const uint32_t logn = c->logn, L = count;
    const size_t toff = (size_t)first << logn;
    const uint64_t *itw = tab64(c, 2) + toff, *ipre = tab64(c, 3) + toff;
    const RnsLimb64 *lc = c->d_lc64 + first;
    if (logn >= 10) {
        const uint32_t split = logn == 15 ? 1u : 0u, lg = logn - split;
        const size_t smem = ((size_t)17 << (lg - 4)) * 8;
        const unsigned grid = (unsigned)(T << split);
        switch (lg) {
            case 14: ref_u64_rns_inv_frame_kernel<512><<<grid, 512, smem, st>>>(in, mul, out, itw, ipre, lc, L, logn); break;
            case 13: ref_u64_rns_inv_frame_kernel<256><<<grid, 256, smem, st>>>(in, mul, out, itw, ipre, lc, L, logn); break;
            case 12: ref_u64_rns_inv_frame_kernel<128><<<grid, 128, smem, st>>>(in, mul, out, itw, ipre, lc, L, logn); break;
            case 11: ref_u64_rns_inv_frame_kernel<64><<<grid, 64, smem, st>>>(in, mul, out, itw, ipre, lc, L, logn); break;
            default: ref_u64_rns_inv_frame_kernel<32><<<grid, 32, smem, st>>>(in, mul, out, itw, ipre, lc, L, logn); break;
        }
        c->launches++;
        if (split) {
            const size_t units = T << (logn - 2);
            const unsigned blocks = (unsigned)std::min<size_t>((units + 255) / 256, (size_t)c->sms * 8);
            ref_u64_rns_inv_last_stage_kernel<<<blocks, 256, 0, st>>>(out, lc, L, logn, T);
            c->launches++;
        }
    } else {
        const uint32_t N = 1u << logn;
        ref_inv_u64_rns_kernel<<<(unsigned)T, N / 2 < 32 ? 32 : N / 2, 0, st>>>(in, mul, out, itw, ipre, lc, L, logn);
        c->launches++;
    }
    return (int)cudaGetLastError();
}

// Argument checks of the u64 batched calls: a u64 context, 16-byte aligned operands, B * L frames within a grid.
// *T = B * L.
int check_dev_call64(const agx_ctx *c, std::initializer_list<const void *> ptrs, size_t B, size_t *T) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : ptrs)
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    if (B > 0x7fffffffull / c->L) return AGX_E_INVALID;
    *T = B * c->L;
    return AGX_OK;
}

// ------------------------------------------------------------------------------- reference-shaped u64 pipeline

// Reference-shaped round: loader + compute unit + drain (ntt.cpp:508-607, 86-506, 610-640) as a chunked three-slot
// pipeline.  Frame b takes its low half from in[b*N ..) and its high half from in2[b*N + N/2 ..) (ntt.cpp:582-591), so
// only those halves cross PCIe (one contiguous copy when in2 == in, two pitched copies otherwise).  Pinned caller
// buffers (the host mirror's sycl::buffer allocates pinned memory) are copied directly and the whole round is
// asynchronous until agx_wait(); pageable buffers are staged through pinned chunks inside this call.
int ref_flush(agx_ctx *c) {
    RefState &R = c->ref;
    if (!(R.have_in && R.have_fwd && R.have_out)) return AGX_OK;     // still waiting for the other calls
    R.have_in = R.have_fwd = R.have_out = false;
    if (R.out_frames < 0 || (uint32_t)R.out_frames != R.frames) return AGX_E_INVALID;
    if (R.frames == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    if (!R.stream[0]) {
        for (int i = 0; i < kSlots; i++) {
            CK(cudaStreamCreateWithFlags(&R.stream[i], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&R.done[i], cudaEventDisableTiming));
        }
        CK(cudaEventCreateWithFlags(&R.tables, cudaEventDisableTiming));
    }
    const size_t N = R.N, frame_bytes = N * 8, half_bytes = N * 4;
    // Chunk = whole waves of frame CTAs (a wave is SMs x 128 KiB of frames at every N the frame kernel serves: N/32 threads
    // per CTA, 512 per SM; half as many frames at N = 32768): a chunk's kernel takes a wave's time whether the wave is full or
    // not, and that time is added to the copy engines' period (profiles/pipeline_timeline.py).  Two waves for rounds of half a
    // GiB and more, where fill and drain matter less: 43.0 -> 44.7 GB/s each way on 1 GiB rounds against the former 16 MiB
    // (profiles/r02_u64_chunk_sweep.jsonl).
    size_t ref_chunk_bytes = c->sms > 0 ? (size_t)c->sms << 17 : kRefChunkBytes;
    if ((size_t)R.frames * frame_bytes >= ((size_t)512 << 20)) ref_chunk_bytes *= 2;
    if (const char *e = getenv("AGX_REF_CHUNK_KB")) {               // tuning knob, like AGX_HOST_CHUNK_MB
        const long kb = atol(e);
        if (kb >= 64 && kb <= (1 << 20)) ref_chunk_bytes = (size_t)kb << 10;
    }
    size_t chunk_frames = ref_chunk_bytes / frame_bytes;
    if (chunk_frames == 0) chunk_frames = 1;
    if (chunk_frames > R.frames) chunk_frames = R.frames;
    const size_t chunk_bytes = chunk_frames * frame_bytes;
    if (chunk_bytes > R.cap_chunk) {
        for (int i = 0; i < kSlots; i++) {
            cudaFree(R.d_in[i]); cudaFree(R.d_out[i]);
            if (R.p_in[i]) cudaFreeHost(R.p_in[i]);
            if (R.p_out[i]) cudaFreeHost(R.p_out[i]);
            R.d_in[i] = R.d_out[i] = R.p_in[i] = R.p_out[i] = nullptr;
        }
        R.cap_chunk = 0; R.have_stage_in = R.have_stage_out = false;
        for (int i = 0; i < kSlots; i++) { CK(cudaMalloc(&R.d_in[i], chunk_bytes)); CK(cudaMalloc(&R.d_out[i], chunk_bytes)); }
        R.cap_chunk = chunk_bytes;
    }
    if (frame_bytes > R.cap_tab) {
        cudaFree(R.d_tw); cudaFree(R.d_pre);
        R.d_tw = R.d_pre = nullptr; R.cap_tab = 0;
        CK(cudaMalloc(&R.d_tw, frame_bytes)); CK(cudaMalloc(&R.d_pre, frame_bytes));
        R.cap_tab = frame_bytes;
    }
    const bool same = R.in2 == R.in;
    const bool pin_in = is_pinned(R.in) && (same || is_pinned(R.in2)), pin_out = is_pinned(R.out);
    if (!pin_in && !R.have_stage_in) {
        for (int i = 0; i < kSlots; i++) CK(cudaHostAlloc(&R.p_in[i], R.cap_chunk, cudaHostAllocDefault));
        R.have_stage_in = true;
    }
    if (!pin_out && !R.have_stage_out) {
        for (int i = 0; i < kSlots; i++) CK(cudaHostAlloc(&R.p_out[i], R.cap_chunk, cudaHostAllocDefault));
        R.have_stage_out = true;
    }
    const uint64_t modulus = R.mod[0];
    if (!pin_in || !pin_out) { const int rc = ensure_crews(c); if (rc) return rc; }
    OutDrainer drain(c->device, c->crew_out);
    // From here on copies touch the caller's buffers.  On any failure: drain every stream and the helper thread before
    // returning, so that nothing is in flight behind the caller's back; on success the round stays asynchronous and
    // agx_wait() completes it (R.busy).
    auto fail = [&](int code) {
        for (int k = 0; k < kSlots; k++) cudaStreamSynchronize(R.stream[k]);
        drain.finish();
        R.busy = false;
        return code;
    };
#define STEP(call) do { const cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail((int)e__); } while (0)
    R.busy = true;
    // tables: once per round (ntt.cpp:119-144 receives them once per mini-batch), the other slots wait for them
    STEP(cudaMemcpyAsync(R.d_tw, R.tw, frame_bytes, cudaMemcpyHostToDevice, R.stream[0]));
    STEP(cudaMemcpyAsync(R.d_pre, R.pre, frame_bytes, cudaMemcpyHostToDevice, R.stream[0]));
    STEP(cudaEventRecord(R.tables, R.stream[0]));
    for (int i = 1; i < kSlots; i++) STEP(cudaStreamWaitEvent(R.stream[i], R.tables, 0));
    uint32_t logn = 0;
    while ((1u << logn) < R.N) logn++;
    size_t done = 0;
    for (size_t i = 0; done < R.frames; i++) {
        const int sl = (int)(i % kSlots);
        cudaStream_t st = R.stream[sl];
        const size_t cnt = R.frames - done < chunk_frames ? R.frames - done : chunk_frames, bytes = cnt * frame_bytes;
        const size_t off = done * N;
        if (i >= (size_t)kSlots) {                                   // staging buffers of this slot are about to be reused
            if (!pin_out) drain.wait_slot_free(i);
            else if (!pin_in) STEP(cudaEventSynchronize(R.done[sl]));
        }
        if (pin_in) {
            if (same) {
                STEP(cudaMemcpyAsync(R.d_in[sl], R.in + off, bytes, cudaMemcpyHostToDevice, st));
            } else {
                STEP(cudaMemcpy2DAsync(R.d_in[sl], frame_bytes, R.in + off, frame_bytes, half_bytes, cnt, cudaMemcpyHostToDevice, st));
                STEP(cudaMemcpy2DAsync(R.d_in[sl] + N / 2, frame_bytes, R.in2 + off + N / 2, frame_bytes, half_bytes, cnt,
                                       cudaMemcpyHostToDevice, st));
            }
        } else {
            if (same) {
                c->crew_in->copy(R.p_in[sl], R.in + off, bytes);
            } else {                                                 // ntt.cpp:582-591: low half from in, high half from in2
                const size_t parts = std::min<size_t>((size_t)c->crew_in->threads(), std::max<size_t>(1, bytes >> 20));
                const size_t per = (cnt + parts - 1) / parts;
                uint64_t *stage = R.p_in[sl];
                const uint64_t *in = R.in, *in2 = R.in2;
                c->crew_in->run(parts, [&](size_t part) {
                    for (size_t f = part * per; f < std::min(cnt, (part + 1) * per); f++) {
                        memcpy(stage + f * N, in + off + f * N, half_bytes);
                        memcpy(stage + f * N + N / 2, in2 + off + f * N + N / 2, half_bytes);
                    }
                });
            }
            STEP(cudaMemcpyAsync(R.d_in[sl], R.p_in[sl], bytes, cudaMemcpyHostToDevice, st));
        }
        const int rc = ref_launch(c, logn, R.d_in[sl], R.d_in[sl], R.d_out[sl], R.d_tw, R.d_pre, modulus, cnt, st);
        if (rc) return fail(rc);
        uint64_t *dst = R.out + off;
        STEP(cudaMemcpyAsync(pin_out ? dst : R.p_out[sl], R.d_out[sl], bytes, cudaMemcpyDeviceToHost, st));
        STEP(cudaEventRecord(R.done[sl], st));
        if (!pin_out) drain.submit(i, dst, R.p_out[sl], bytes, R.done[sl]);
        done += cnt;
    }
#undef STEP
    const int rc = drain.finish();                                   // pageable results are complete on return
    return rc ? fail(rc) : AGX_OK;
}

// A context without a parameter set on `device`, which the caller has made current: the driver's tensor-map encoder, and
// the dynamic shared-memory opt-in of every kernel that takes more than 48 KB.
int ctx_new(agx_ctx **out, int device) {
    CK(cudaFree(0));
    agx_ctx *c = new (std::nothrow) agx_ctx();
    if (!c) return AGX_E_NOMEM;
    c->device = device;
    cudaDeviceGetAttribute(&c->sms, cudaDevAttrMultiProcessorCount, device);
    {
        cudaDriverEntryPointQueryResult qres;
        void *fn = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            c->encode_tiled = fn;
        else
            cudaGetLastError();
        if (getenv("AGX_NO_TMA")) c->encode_tiled = nullptr;   // force the staging-image kernels (tests cover both)
    }
    // kernels that take more than 48 KB of dynamic shared memory opt in per device (function attributes are
    // per-context state, so this is repeated for every context rather than cached in a process-wide flag)
    {
        cudaError_t e = cudaFuncSetAttribute(ntt_generic_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 << 10);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ntt_generic_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 << 10);
#define AGX_BIG_SMEM(LOGN)                                                                                                              \
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ntt_big_kernel<false, LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, 33 * 1024 * 4); \
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ntt_big_kernel<true, LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, 33 * 1024 * 4);
        AGX_BIG_SMEM(13) AGX_BIG_SMEM(14) AGX_BIG_SMEM(15)
#undef AGX_BIG_SMEM
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_fwd_u64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 << 10);
        const int frame_smem = 17 * 1024 * 8;                          // N = 16384 image: 136 KB
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_frame_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_frame_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_inv_frame_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_inv_frame_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(bitrev_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 << 10);
        if (e != cudaSuccess) { delete c; return (int)e; }
    }
    *out = c;
    return AGX_OK;
}

// ModUp / ModDown (agx_modup64 / agx_moddown64).  The source limbs s0 .. s0 + m - 1 must each differ from every other
// prime of the context: then S is invertible modulo every target and the MRC's p_j^-1 mod p_t exist.
static_assert(kBasisMaxSrc == AGX_BASIS_MAX_SRC, "the header states the kernels' bound");

bool basis_sources_distinct(const agx_ctx *c, uint32_t s0, uint32_t m) {
    for (uint32_t t = s0; t < s0 + m; t++)
        for (uint32_t j = 0; j < c->L; j++)
            if (j != t && c->q64[j] == c->q64[t]) return false;
    return true;
}

// The per-call constants from the host copy of the pairwise array: h = (S - 1) / 2 mod q_i = (S - 1) * 2^-1 mod q_i for
// every limb (S odd), and for ModDown S^-1 mod q_i with its companion for every target.
BasisCall64 basis_call(const agx_ctx *c, uint32_t s0, uint32_t m, bool down) {
    typedef unsigned __int128 u128;
    BasisCall64 cp{};
    cp.L = c->L; cp.logn = c->logn; cp.s0 = s0; cp.m = m;
    cp.ntgt = c->L - m;
    cp.lift = !down && m == 1;
    for (uint32_t i = 0; i < c->L; i++) {
        const uint64_t q = c->bl64[i].q;
        const BasisPair64 *row = c->bp64.data() + (size_t)i * c->L;
        uint64_t Smod = 1 % q, Sinv = 1 % q;
        for (uint32_t t = s0; t < s0 + m; t++) {
            Smod = mulmod_u64(Smod, row[t].w, q);
            Sinv = mulmod_u64(Sinv, row[t].inv, q);
        }
        cp.h[i] = mulmod_u64((Smod + q - 1) % q, (q + 1) / 2, q);
        if (down && (i < s0 || i >= s0 + m)) {
            cp.pinv[i] = Sinv;
            cp.pinv_p[i] = (uint64_t)(((u128)Sinv << 64) / q);
        }
    }
    return cp;
}

// Stream-ordered scratch: from `pool` when not null, else from the device's default pool.
int scratch_alloc(uint64_t **p, size_t words, cudaMemPool_t pool, cudaStream_t st) {
    void **v = reinterpret_cast<void **>(p);
    const size_t bytes = words * sizeof(uint64_t);
    return (int)(pool ? cudaMallocFromPoolAsync(v, bytes, pool, st) : cudaMallocAsync(v, bytes, st));
}

// The launches of both calls once the arguments are checked (B > 0).  in: [B][L][n] (down) or [B][m][n];
// out: [B][L-m][n] (down) or [B][L][n].  The evaluation form's scratch comes from `pool` (see scratch_alloc).
int basis_launch(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, uint32_t s0, uint32_t m, bool down,
                 int ntt_form, cudaStream_t st, cudaMemPool_t pool = nullptr) {
    const uint32_t logn = c->logn, L = c->L, N = c->n;
    const BasisCall64 cp = basis_call(c, s0, m, down);
    const BasisLimb64 *bl = c->d_bl64;
    const BasisPair64 *bp = c->d_bp64;
    const size_t pairs = B * N / 2;
    const unsigned pblocks = (unsigned)std::min<size_t>((pairs + 255) / 256, (size_t)c->sms * 16);
    if (!ntt_form) {
        auto *o2 = reinterpret_cast<ulonglong2 *>(d_out);
        auto *i2 = reinterpret_cast<const ulonglong2 *>(d_in);
        if (down) basis64_coeff_kernel<true><<<pblocks, 256, 0, st>>>(o2, i2, bl, bp, cp, pairs);
        else basis64_coeff_kernel<false><<<pblocks, 256, 0, st>>>(o2, i2, bl, bp, cp, pairs);
        c->launches++;
        return (int)cudaGetLastError();
    }
    int rc = AGX_OK;
    if (!down)                                                     // the source spectra are the output's source limbs
        rc = (int)cudaMemcpy2DAsync(d_out + ((size_t)s0 << logn), (size_t)L * N * sizeof(uint64_t), d_in,
                                    (size_t)m * N * sizeof(uint64_t), (size_t)m * N * sizeof(uint64_t), B,
                                    cudaMemcpyDeviceToDevice, st);
    // scratch[b][t] = INTT(source limb t of polynomial b), then its digits in place; then the fused forward
    uint64_t *tmp = nullptr;
    if (!rc) rc = scratch_alloc(&tmp, B * m * N, pool, st);
    if (!rc) {
        if (!down) {
            rc = rns_inv_launch(c, d_in, nullptr, tmp, B * m, st, s0, m);
        } else {
            const uint64_t *itw = tab64(c, 2), *ipre = tab64(c, 3);
            const RnsLimb64 *lc = c->d_lc64;
            if (logn >= 10) {
                const uint32_t split = logn == 15 ? 1u : 0u, lg = logn - split;
                const size_t smem = ((size_t)17 << (lg - 4)) * 8;
                const unsigned grid = (unsigned)((B * m) << split);
                switch (lg) {
                    case 14: ref_u64_basis_inv_frame_kernel<512><<<grid, 512, smem, st>>>(d_in, tmp, itw, ipre, lc, L, m, logn); break;
                    case 13: ref_u64_basis_inv_frame_kernel<256><<<grid, 256, smem, st>>>(d_in, tmp, itw, ipre, lc, L, m, logn); break;
                    case 12: ref_u64_basis_inv_frame_kernel<128><<<grid, 128, smem, st>>>(d_in, tmp, itw, ipre, lc, L, m, logn); break;
                    case 11: ref_u64_basis_inv_frame_kernel<64><<<grid, 64, smem, st>>>(d_in, tmp, itw, ipre, lc, L, m, logn); break;
                    default: ref_u64_basis_inv_frame_kernel<32><<<grid, 32, smem, st>>>(d_in, tmp, itw, ipre, lc, L, m, logn); break;
                }
                c->launches++;
                if (split) {                                       // the scratch as a batch of B polynomials over the m limbs
                    const size_t units = (B * m) << (logn - 2);
                    const unsigned blocks = (unsigned)std::min<size_t>((units + 255) / 256, (size_t)c->sms * 8);
                    ref_u64_rns_inv_last_stage_kernel<<<blocks, 256, 0, st>>>(tmp, lc + s0, m, logn, B * m);
                    c->launches++;
                }
            } else {
                ref_inv_u64_basis_kernel<<<(unsigned)(B * m), N / 2 < 32 ? 32 : N / 2, 0, st>>>(d_in, tmp, itw, ipre, lc, L, m, logn);
                c->launches++;
            }
            rc = (int)cudaGetLastError();
        }
    }
    if (!rc && m >= 2) {
        basis64_digits_kernel<<<pblocks, 256, 0, st>>>(reinterpret_cast<ulonglong2 *>(tmp), bl, bp, cp, pairs);
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc) {
        const uint64_t *tw = tab64(c, 0), *pre = tab64(c, 1);
        const unsigned frames = (unsigned)(B * cp.ntgt);
        if (logn >= 10) {
            const uint32_t split = logn == 15 ? 1u : 0u, lg = logn - split;
            const size_t smem = ((size_t)17 << (lg - 4)) * 8;
            const unsigned grid = frames << split;
#define AGX_BASIS_FWD(NT)                                                                                                \
    (down ? ref_u64_basis_fwd_kernel<NT, true><<<grid, NT, smem, st>>>(d_in, tmp, d_out, tw, pre, bl, bp, cp)            \
          : ref_u64_basis_fwd_kernel<NT, false><<<grid, NT, smem, st>>>(d_in, tmp, d_out, tw, pre, bl, bp, cp))
            switch (lg) {
                case 14: AGX_BASIS_FWD(512); break;
                case 13: AGX_BASIS_FWD(256); break;
                case 12: AGX_BASIS_FWD(128); break;
                case 11: AGX_BASIS_FWD(64); break;
                default: AGX_BASIS_FWD(32); break;
            }
#undef AGX_BASIS_FWD
        } else {
            const unsigned nt = N / 2 < 32 ? 32 : N / 2;
            if (down) ref_fwd_u64_basis_kernel<true><<<frames, nt, (size_t)N * 8, st>>>(d_in, tmp, d_out, tw, pre, bl, bp, cp);
            else ref_fwd_u64_basis_kernel<false><<<frames, nt, (size_t)N * 8, st>>>(d_in, tmp, d_out, tw, pre, bl, bp, cp);
        }
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (tmp) { const int rf = (int)cudaFreeAsync(tmp, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

// byte ranges [p, p + words) overlap
bool ranges_overlap(const void *a, size_t wa, const void *b, size_t wb) {
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(a), a1 = a0 + wa * sizeof(uint64_t);
    const uintptr_t b0 = reinterpret_cast<uintptr_t>(b), b1 = b0 + wb * sizeof(uint64_t);
    return a0 < b1 && b0 < a1;
}

// Galois elements of agx_automorph64 and agx_rotate64: false unless every g_t is odd and in [1, 2n); gi[t] = g_t^-1 mod 2n.
bool galois_inverses(const agx_ctx *c, const uint32_t *galois, uint32_t G, uint32_t *gi) {
    const uint32_t m2n = 2 * c->n - 1;
    for (uint32_t t = 0; t < G; t++) {
        const uint32_t g = galois[t];
        if (!(g & 1) || g > m2n) return false;
        uint32_t x = g;                                    // g^-1 mod 2^32 by Newton: each step doubles the correct bits
        for (int i = 0; i < 5; i++) x *= 2 - g * x;
        gi[t] = x & m2n;
    }
    return true;
}

// The key-switch scratch pool of the context (agx_keyswitch64, agx_rotate64): gigabytes at real batch sizes, kept
// between calls so that a call does not map it afresh, as the device's default pool would after every synchronisation.
int ks_pool_ready(agx_ctx *c) {
    if (c->ks_pool) return AGX_OK;
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = c->device;
    int rc = (int)cudaMemPoolCreate(&c->ks_pool, &props);
    uint64_t keep = UINT64_MAX;                                    // never trimmed at synchronisation: freed at agx_destroy
    if (!rc) rc = (int)cudaMemPoolSetAttribute(c->ks_pool, cudaMemPoolAttrReleaseThreshold, &keep);
    if (rc) { if (c->ks_pool) cudaMemPoolDestroy(c->ks_pool); c->ks_pool = nullptr; }
    return rc;
}

// ModUp of the dnum gadget digits of d_in[B][l+1][n] (digit j: limbs j*m .. min((j+1)*m, l+1) - 1) into
// U[dnum][B][L][n].  With dnum > 1 each digit is first gathered into dig[B][m][n] by one pitched copy, since ModUp
// reads its source limbs contiguously.
int ks_modup_digits(agx_ctx *c, uint64_t *U, uint64_t *dig, const uint64_t *d_in, size_t B, uint32_t ell1, uint32_t m,
                    uint32_t dnum, int ntt_form, cudaStream_t st) {
    const size_t N = c->n, T = B * c->L;
    int rc = AGX_OK;
    for (uint32_t j = 0; !rc && j < dnum; j++) {
        const uint32_t first = j * m, cnt = std::min(m, ell1 - first);
        const uint64_t *src = d_in;
        if (dnum > 1) {
            rc = (int)cudaMemcpy2DAsync(dig, cnt * N * sizeof(uint64_t), d_in + first * N, ell1 * N * sizeof(uint64_t),
                                        cnt * N * sizeof(uint64_t), B, cudaMemcpyDeviceToDevice, st);
            src = dig;
        }
        if (!rc) rc = agx_modup64(c, U + j * T * N, src, B, first, cnt, ntt_form, st);
    }
    return rc;
}

// The key-switch parameters of agx_keyswitch64 and agx_rotate64 against a u64 context over Q_l u P: 0 < k < L,
// alpha > 0, key_limbs >= L, and no two equal primes (every prime is a digit's source or one of P's).
bool ks_params_valid(const agx_ctx *c, uint32_t key_limbs, uint32_t alpha, uint32_t k) {
    const uint32_t L = c->L;
    if (k == 0 || k >= L || alpha == 0 || key_limbs < L) return false;
    for (uint32_t i = 0; i < L; i++)
        for (uint32_t j = 0; j < i; j++)
            if (c->q64[i] == c->q64[j]) return false;
    return true;
}

// Slices of the batch for the key inner products: enough work items to fill the GPU, each reading its key words once
// for its slice.  per_slice: work items per slice.  Returns polynomials per slice.
uint32_t ks_slice(const agx_ctx *c, size_t B, size_t per_slice) {
    const size_t want = (size_t)c->sms * 1024;
    const size_t S = std::min<size_t>(B, std::max<size_t>(1, (want + per_slice - 1) / per_slice));
    return (uint32_t)((B + S - 1) / S);
}


// The special FFT's twiddles (agx_encode64 / agx_decode64), at the context's first encode or decode: entry h + j, for
// h = 1 .. S/2 and j < h, is zeta^((5^j mod 8h) (2n / 8h)), computed in long double and rounded to double, uploaded by
// one synchronous copy followed by a device synchronisation, and kept until agx_destroy.  The kernels' shared-memory limits are raised at the same time.
int slots_ready(agx_ctx *c) {
    if (c->d_slot_tw) return AGX_OK;
    const uint32_t n = c->n, S = n / 2;
    std::vector<double2> w(S, make_double2(0.0, 0.0));
    const long double pi = 3.141592653589793238462643383279502884L;
    for (uint32_t h = 1; h < S; h <<= 1) {
        const uint32_t lenq = 8 * h;
        uint32_t r = 1;                                            // 5^j mod lenq
        for (uint32_t j = 0; j < h; j++) {
            const long double a = pi * (long double)(r * (2 * n / lenq)) / (long double)n;
            w[h + j] = make_double2((double)cosl(a), (double)sinl(a));
            r = r * 5 % lenq;
        }
    }
    const int fft_smem = kEncodeMaxLocal * sizeof(double2), crt_smem = kBasisMaxLimbs * kDecodeCrtThreads * 8;
    cudaError_t e = cudaFuncSetAttribute(encode64_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, fft_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(encode64_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, fft_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(decode64_fft_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, fft_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(decode64_fft_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, fft_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(decode64_crt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, crt_smem);
    double2 *d = nullptr;
    if (e == cudaSuccess) e = cudaMalloc(&d, S * sizeof(double2));
    if (e == cudaSuccess) e = cudaMemcpy(d, w.data(), S * sizeof(double2), cudaMemcpyHostToDevice);
    // a pageable upload may still be in flight when cudaMemcpy returns, and only the legacy stream is ordered after
    // it: the caller's stream (a non-blocking one included) must find the table written
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { cudaFree(d); return (int)e; }
    c->d_slot_tw = d;
    return AGX_OK;
}

// The slot kernels of agx_encode64 / agx_decode64: one CTA per polynomial, a 2-CTA cluster at n = 32768.
void slot_fft_launch(agx_ctx *c, bool encode, void *out, const void *in, size_t B, uint32_t limbs, double sc,
                     cudaStream_t st) {
    const uint32_t logn = c->logn, th = slot_threads(logn);
    const bool pair = logn == 15;
    const unsigned grid = (unsigned)(pair ? 2 * B : B);
    const size_t smem = (size_t)(pair ? kEncodeMaxLocal : c->n / 2) * sizeof(double2);
    auto *o64 = static_cast<uint64_t *>(out);
    auto *z = static_cast<const double2 *>(in);
    auto *zo = static_cast<double2 *>(out);
    auto *m = static_cast<const double *>(in);
    if (encode && pair) encode64_kernel<2><<<grid, th, smem, st>>>(o64, z, c->d_slot_tw, c->d_bl64, c->d_lc64, logn, limbs, sc);
    else if (encode) encode64_kernel<1><<<grid, th, smem, st>>>(o64, z, c->d_slot_tw, c->d_bl64, c->d_lc64, logn, limbs, sc);
    else if (pair) decode64_fft_kernel<2><<<grid, th, smem, st>>>(zo, m, c->d_slot_tw, logn);
    else decode64_fft_kernel<1><<<grid, th, smem, st>>>(zo, m, c->d_slot_tw, logn);
    c->launches++;
}
}  // namespace

// ================================================================================================== C ABI

extern "C" {

int agx_create(agx_ctx **out, const agx_parms *parms, int device) { return agx_create_tables(out, parms, nullptr, device); }

int agx_create_tables(agx_ctx **out, const agx_parms *parms, const uint32_t *psi, int device) {
    if (!out) return AGX_E_INVALID;
    *out = nullptr;
    if (psi && !parms) return AGX_E_INVALID;
    DeviceGuard guard__(device);
    if (guard__.error()) return guard__.error();
    agx_ctx *c = nullptr;
    if (const int rc = ctx_new(&c, device)) return rc;
    if (const char *e = getenv("AGX_CARVEOUT")) {      // A/B knob: shared-memory carve-out (percent) of the n = 4096 kernels
        const int pct = atoi(e);
        cudaFuncSetAttribute(ntt_fwd_loop_kernel<12, 6, false, true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
        cudaFuncSetAttribute(ntt_fwd_loop_kernel<12, 6, false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
        cudaFuncSetAttribute(ntt_inv_loop_kernel<12, 6, true>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
        cudaFuncSetAttribute(ntt_inv_loop_kernel<12, 6, false>, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    }
    if (parms) {
        if (!parms->q || parms->nlimbs == 0 || parms->nlimbs > 64 || parms->logn < 3 || parms->logn > 15 ||
            parms->n != (1u << parms->logn)) { delete c; return AGX_E_INVALID; }
        c->has_parms = true;
        c->n = parms->n; c->logn = parms->logn; c->L = parms->nlimbs;
        c->le = select_le(c->logn);
        c->big = c->le == 0 && c->logn >= 13 && getenv("AGX_GENERIC_ONLY") == nullptr;   // A/B and test knob: the radix-2 kernel
#if AGX_WITH_R16
        {   // n = 4096: radix-16 three-pass kernels (they need the TMA tensor-map encoder), selected with AGX_KERNEL=r16
            const char *k = getenv("AGX_KERNEL");
            c->r16 = c->logn == 12 && c->encode_tiled && k && strcmp(k, "r16") == 0;
        }
#endif
        c->q.assign(parms->q, parms->q + parms->nlimbs);
        c->psi.resize(c->L);
        c->n_inv.resize(c->L);
        int rc = build_tables(c, psi);
        if (rc) { agx_destroy(c); return rc; }
    }
    *out = c;
    return AGX_OK;
}

int agx_destroy(agx_ctx *c) {
    if (!c) return AGX_OK;
    {
        DeviceGuard guard__(c->device);
        cudaDeviceSynchronize();
        pipe_destroy(c->pipe);
        delete c->crew_in; delete c->crew_out;
        RefState &R = c->ref;
        for (int i = 0; i < kSlots; i++) {
            cudaFree(R.d_in[i]); cudaFree(R.d_out[i]);
            if (R.p_in[i]) cudaFreeHost(R.p_in[i]);
            if (R.p_out[i]) cudaFreeHost(R.p_out[i]);
            if (R.stream[i]) cudaStreamDestroy(R.stream[i]);
            if (R.done[i]) cudaEventDestroy(R.done[i]);
        }
        if (R.tables) cudaEventDestroy(R.tables);
        cudaFree(R.d_tw); cudaFree(R.d_pre);
        cudaFree(c->d_tw_fwd); cudaFree(c->d_tw_inv); cudaFree(c->d_nat_fwd); cudaFree(c->d_nat_inv);
        cudaFree(c->d_twc_fwd); cudaFree(c->d_twc_inv);
        cudaFree(c->d_lc); cudaFree(c->d_sum);
        cudaFree(c->d_tab64); cudaFree(c->d_lc64); cudaFree(c->d_rs64); cudaFree(c->d_bl64);
        if (c->ks_pool) cudaMemPoolDestroy(c->ks_pool);
        cudaFree(c->d_slot_tw);
#if AGX_WITH_R16
        cudaFree(c->d_tw16_fwd); cudaFree(c->d_tw16_inv); cudaFree(c->d_u16_fwd); cudaFree(c->d_u16_inv);
#endif
    }
    delete c;
    return AGX_OK;
}

int agx_get_psi(const agx_ctx *c, uint32_t limb, uint32_t *psi) {
    if (!c || !c->has_parms || limb >= c->L || !psi) return AGX_E_INVALID;
    *psi = c->psi[limb];
    return AGX_OK;
}

int agx_get_tables(const agx_ctx *c, uint32_t limb, int inverse, uint32_t *roots, uint32_t *precons) {
    if (!c || !c->has_parms || limb >= c->L || !roots || !precons) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    std::vector<uint2> t(c->n);
    CK(cudaMemcpy(t.data(), (inverse ? c->d_nat_inv : c->d_nat_fwd) + (size_t)limb * c->n, (size_t)c->n * sizeof(uint2),
                  cudaMemcpyDeviceToHost));
    for (uint32_t k = 0; k < c->n; k++) { roots[k] = t[k].x; precons[k] = t[k].y; }
    return AGX_OK;
}

int agx_set_tables(agx_ctx *c, uint32_t limb, int inverse, const uint32_t *roots, const uint32_t *precons) {
    if (!c || !c->has_parms || limb >= c->L || !roots) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    const uint32_t n = c->n;
    const size_t base = (size_t)limb * n;
    // the new tables are built beside the live ones and swapped in only when the caller's table proved consistent
    uint32_t *d_in = nullptr;
    uint2 *d_new = nullptr;
    unsigned *d_bad = nullptr;
    const size_t sets = c->le ? 3 : 2;
    cudaError_t e = cudaMalloc(&d_in, (size_t)n * 8);
    if (e == cudaSuccess) e = cudaMalloc(&d_new, sets * n * sizeof(uint2));
    if (e == cudaSuccess) e = cudaMalloc(&d_bad, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(d_bad, 0, sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(d_new, 0, sets * n * sizeof(uint2));
    if (e == cudaSuccess) e = cudaMemcpy(d_in, roots, (size_t)n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && precons) e = cudaMemcpy(d_in + n, precons, (size_t)n * 4, cudaMemcpyHostToDevice);
    unsigned bad = 1;
    if (e == cudaSuccess) {
        const TableSet t{d_new, d_new + n, c->le ? d_new + 2 * (size_t)n : nullptr};
        relayout_tables_kernel<<<(n + 255) / 256, 256>>>(t, d_in, precons ? d_in + n : nullptr, inverse != 0, c->q[limb],
                                                         c->n_inv[limb], c->logn, c->le, d_bad);
        c->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpy(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost);
    }
    if (e == cudaSuccess && bad == 0) {
        const size_t bytes = (size_t)n * sizeof(uint2);
        e = cudaMemcpy((inverse ? c->d_nat_inv : c->d_nat_fwd) + base, d_new, bytes, cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess) e = cudaMemcpy((inverse ? c->d_tw_inv : c->d_tw_fwd) + base, d_new + n, bytes, cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess && c->le)
            e = cudaMemcpy((inverse ? c->d_twc_inv : c->d_twc_fwd) + base, d_new + 2 * (size_t)n, bytes, cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess && !inverse) {                               // psi = roots[n/2] (bitrev(n/2) = 1)
            c->psi[limb] = roots[n / 2];
            if (limb == 0) c->lc0.psi = roots[n / 2];
        }
    }
    cudaFree(d_in); cudaFree(d_new); cudaFree(d_bad);
    if (e != cudaSuccess) return (int)e;
    if (bad) return AGX_E_INVALID;
    return refresh_r16(c);
}

int agx_ntt_fwd(agx_ctx *c, uint32_t *d, size_t B, void *stream) {
    int rc = check_dev_call(c, d, B);
    if (rc) return rc;
    AGX_ON_DEVICE(c);
    return launch(c, OP_FWD, d, d, nullptr, B, (cudaStream_t)stream);
}

int agx_ntt_inv(agx_ctx *c, uint32_t *d, size_t B, void *stream) {
    int rc = check_dev_call(c, d, B);
    if (rc) return rc;
    AGX_ON_DEVICE(c);
    return launch(c, OP_INV, d, d, nullptr, B, (cudaStream_t)stream);
}

int agx_polymul(agx_ctx *c, uint32_t *dc, const uint32_t *da, const uint32_t *db, size_t B, void *stream) {
    int rc = check_dev_call(c, dc, B);
    if (rc) return rc;
    if (B && (!da || !db)) return AGX_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(db)) & 15) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    return launch(c, OP_MUL, dc, da, db, B, (cudaStream_t)stream);
}

int agx_polymul_by_spectrum(agx_ctx *c, uint32_t *dc, const uint32_t *da, const uint32_t *db_hat, size_t B, void *stream) {
    int rc = check_dev_call(c, dc, B);
    if (rc) return rc;
    if (B && (!da || !db_hat)) return AGX_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(db_hat)) & 15) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    return launch(c, OP_MULSPEC, dc, da, db_hat, B, (cudaStream_t)stream);
}

int agx_elementwise(agx_ctx *c, int op, uint32_t *dc, const uint32_t *da, const uint32_t *db, size_t B, void *stream) {
    int rc = check_dev_call(c, dc, B);
    if (rc) return rc;
    if (op < 0 || op > 3) return AGX_E_INVALID;
    if (B == 0) return AGX_OK;
    if (!da || !db) return AGX_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(da) | reinterpret_cast<uintptr_t>(db)) & 15) return AGX_E_INVALID;   // read as uint4
    AGX_ON_DEVICE(c);
    const size_t total4 = B * c->L * c->n / 4;
    size_t blocks = (total4 + 255) / 256;
    if (blocks > (size_t)c->sms * 16) blocks = (size_t)c->sms * 16;
    cudaStream_t s = (cudaStream_t)stream;
    uint4 *c4 = reinterpret_cast<uint4 *>(dc);
    const uint4 *a4 = reinterpret_cast<const uint4 *>(da), *b4 = reinterpret_cast<const uint4 *>(db);
    switch (op) {
        case EW_ADD: elementwise_kernel<EW_ADD><<<(unsigned)blocks, 256, 0, s>>>(c4, a4, b4, c->d_lc, c->L, c->logn, total4); break;
        case EW_SUB: elementwise_kernel<EW_SUB><<<(unsigned)blocks, 256, 0, s>>>(c4, a4, b4, c->d_lc, c->L, c->logn, total4); break;
        case EW_MUL: elementwise_kernel<EW_MUL><<<(unsigned)blocks, 256, 0, s>>>(c4, a4, b4, c->d_lc, c->L, c->logn, total4); break;
        default:     elementwise_kernel<EW_MAC><<<(unsigned)blocks, 256, 0, s>>>(c4, a4, b4, c->d_lc, c->L, c->logn, total4); break;
    }
    c->launches++;
    return (int)cudaGetLastError();
}

int agx_bitrev(agx_ctx *c, uint32_t *d, size_t B, void *stream) {
    int rc = check_dev_call(c, d, B);
    if (rc || B == 0) return rc;
    const size_t T = B * c->L;
    if (T > 0x7fffffffull) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    const unsigned threads = c->n / 4 < 256 ? (c->n / 4 < 32 ? 32 : c->n / 4) : 256;
    bitrev_rows_kernel<<<(unsigned)T, threads, (size_t)c->n * 4, (cudaStream_t)stream>>>(d, c->logn);
    c->launches++;
    return (int)cudaGetLastError();
}

int agx_ntt_fwd_host(agx_ctx *c, const uint32_t *h_in, uint32_t *h_out, size_t B) {
    return run_host(c, OP_FWD, h_in, nullptr, h_out, B);
}
int agx_ntt_inv_host(agx_ctx *c, const uint32_t *h_in, uint32_t *h_out, size_t B) {
    return run_host(c, OP_INV, h_in, nullptr, h_out, B);
}
int agx_polymul_host(agx_ctx *c, uint32_t *h_c, const uint32_t *h_a, const uint32_t *h_b, size_t B) {
    return run_host(c, OP_MUL, h_a, h_b, h_c, B);
}

int agx_polymul_by_spectrum_host(agx_ctx *c, uint32_t *h_c, const uint32_t *h_a, const uint32_t *h_b_hat, size_t B) {
    return run_host(c, OP_MULSPEC, h_a, h_b_hat, h_c, B);
}

int agx_host_alloc(void **p, size_t bytes) {
    if (!p) return AGX_E_INVALID;
    CK(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
    return AGX_OK;
}
int agx_host_free(void *p) {
    CK(cudaFreeHost(p));
    return AGX_OK;
}

int agx_fill_synthetic(agx_ctx *c, uint32_t *d, size_t B, uint64_t seed, size_t first_poly, void *stream) {
    int rc = check_dev_call(c, d, B);
    if (rc || B == 0) return rc;
    AGX_ON_DEVICE(c);
    const size_t total = B * c->L * c->n;
    size_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    fill_synthetic_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        d, total, c->logn, c->L, c->d_lc, seed, (uint64_t)first_poly * c->L * c->n);
    c->launches++;
    return (int)cudaGetLastError();
}

int agx_checksum(agx_ctx *c, const uint32_t *d, size_t count, size_t first_index, uint64_t *h_sum, void *stream) {
    if (!c || !c->has_parms || !h_sum || (count && !d)) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    cudaStream_t s = (cudaStream_t)stream;
    CK(cudaMemsetAsync(c->d_sum, 0, sizeof(unsigned long long), s));
    if (count) {
        size_t blocks = (count + 255) / 256;
        if (blocks > 148 * 16) blocks = 148 * 16;
        checksum_kernel<<<(unsigned)blocks, 256, 0, s>>>(d, count, first_index, c->d_sum);
        c->launches++;
        CK(cudaGetLastError());
    }
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, c->d_sum, sizeof v, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *h_sum = v;
    return AGX_OK;
}

int agx_ref_input(agx_ctx *c, uint32_t N, const uint64_t *in, const uint64_t *in2, const uint64_t *modulus,
                  const uint64_t *twiddles, const uint64_t *precon_twiddles, uint32_t numFrames) {
    if (!c || !in || !in2 || !modulus || !twiddles || !precon_twiddles) return AGX_E_INVALID;
    if (N < 4 || N > 32768 || (N & (N - 1))) return AGX_E_INVALID;
    RefState &R = c->ref;
    if (R.have_in || R.busy) return AGX_E_STATE;
    R.N = N; R.frames = numFrames; R.in = in; R.in2 = in2; R.mod = modulus; R.tw = twiddles; R.pre = precon_twiddles;
    R.have_in = true;
    return ref_flush(c);
}

int agx_ref_fwd(agx_ctx *c, uint32_t compute_unit_id) {
    if (!c) return AGX_E_INVALID;
    if (compute_unit_id != 0) return AGX_E_UNSUPPORTED;   // the reference instantiates only <0> (ntt.cpp:648)
    if (c->ref.have_fwd || c->ref.busy) return AGX_E_STATE;
    c->ref.have_fwd = true;
    return ref_flush(c);
}

int agx_ref_output(agx_ctx *c, uint64_t *out, int32_t numFrames) {
    if (!c || !out) return AGX_E_INVALID;
    if (c->ref.have_out || c->ref.busy) return AGX_E_STATE;
    c->ref.out = out; c->ref.out_frames = numFrames; c->ref.have_out = true;
    return ref_flush(c);
}

int agx_wait(agx_ctx *c) {
    if (!c) return AGX_E_INVALID;
    RefState &R = c->ref;
    if (R.have_in || R.have_fwd || R.have_out) {
        // a partial round can never complete (the reference would hang on its pipes): report and reset
        R.have_in = R.have_fwd = R.have_out = false;
        return AGX_E_STATE;
    }
    if (R.busy) {
        AGX_ON_DEVICE(c);
        R.busy = false;
        int rc = AGX_OK;
        for (int i = 0; i < kSlots; i++) {                // every stream, even after a failure on an earlier one
            const cudaError_t e = cudaStreamSynchronize(R.stream[i]);
            if (!rc && e != cudaSuccess) rc = (int)e;
        }
        return rc;
    }
    return AGX_OK;
}

int agx_ref_fwd_dev(agx_ctx *c, uint32_t N, const uint64_t *d_in, const uint64_t *d_in2, uint64_t *d_out, uint64_t modulus,
                    const uint64_t *d_twiddles, const uint64_t *d_precon_twiddles, uint32_t numFrames, void *stream) {
    if (!c || !d_in || !d_in2 || !d_out || !d_twiddles || !d_precon_twiddles) return AGX_E_INVALID;
    if (N < 4 || N > 32768 || (N & (N - 1))) return AGX_E_INVALID;
    if ((reinterpret_cast<uintptr_t>(d_in) | reinterpret_cast<uintptr_t>(d_in2) | reinterpret_cast<uintptr_t>(d_out) |
         reinterpret_cast<uintptr_t>(d_twiddles) | reinterpret_cast<uintptr_t>(d_precon_twiddles)) & 15)
        return AGX_E_INVALID;                          // frames and tables are read by 16-byte accesses
    // the passes work in place in d_out after the first one, so an input that overlaps it is only safe when it IS it
    if ((d_in != d_out || d_in2 != d_out) && (d_in == d_out || d_in2 == d_out)) return AGX_E_INVALID;
    if (numFrames == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    uint32_t logn = 0;
    while ((1u << logn) < N) logn++;
    return ref_launch(c, logn, d_in, d_in2, d_out, d_twiddles, d_precon_twiddles, modulus, numFrames, (cudaStream_t)stream);
}

int agx_ref_inv_dev(agx_ctx *c, uint32_t N, const uint64_t *d_in, uint64_t *d_out, uint64_t modulus,
                    const uint64_t *d_inv_twiddles, const uint64_t *d_inv_precon_twiddles, uint32_t numFrames, void *stream) {
    uint32_t logn = 0;
    if (ref_inv_check(c, N, {d_in, d_out, d_inv_twiddles, d_inv_precon_twiddles}, modulus, &logn)) return AGX_E_INVALID;
    if (numFrames == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    return ref_inv_launch(c, logn, d_in, nullptr, d_out, d_inv_twiddles, d_inv_precon_twiddles, modulus, numFrames,
                          (cudaStream_t)stream);
}

int agx_ref_polymul_dev(agx_ctx *c, uint32_t N, uint64_t *d_c, const uint64_t *d_a, const uint64_t *d_b, uint64_t modulus,
                        const uint64_t *d_twiddles, const uint64_t *d_precon_twiddles, const uint64_t *d_inv_twiddles,
                        const uint64_t *d_inv_precon_twiddles, uint32_t numFrames, void *stream) {
    uint32_t logn = 0;
    if (ref_inv_check(c, N, {d_c, d_a, d_b, d_twiddles, d_precon_twiddles, d_inv_twiddles, d_inv_precon_twiddles}, modulus,
                      &logn))
        return AGX_E_INVALID;
    if (numFrames == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    if (d_c == d_b && d_c != d_a) std::swap(d_a, d_b);             // the product commutes: c == a from here on
    // c = NTT(a); scratch = NTT(b) unless squaring; c = INTT(c .* (scratch or c))
    uint64_t *tmp = nullptr;
    int rc = ref_launch(c, logn, d_a, d_a, d_c, d_twiddles, d_precon_twiddles, modulus, numFrames, st);
    if (!rc && d_a != d_b) {
        rc = (int)cudaMallocAsync(&tmp, (size_t)numFrames * N * 8, st);
        if (!rc) rc = ref_launch(c, logn, d_b, d_b, tmp, d_twiddles, d_precon_twiddles, modulus, numFrames, st);
    }
    if (!rc) rc = ref_inv_launch(c, logn, d_c, tmp ? tmp : d_c, d_c, d_inv_twiddles, d_inv_precon_twiddles, modulus, numFrames, st);
    if (tmp) { const int rf = (int)cudaFreeAsync(tmp, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

int agx_ref_polymul_by_spectrum_dev(agx_ctx *c, uint32_t N, uint64_t *d_c, const uint64_t *d_a, const uint64_t *d_b_hat,
                                    uint64_t modulus, const uint64_t *d_twiddles, const uint64_t *d_precon_twiddles,
                                    const uint64_t *d_inv_twiddles, const uint64_t *d_inv_precon_twiddles, uint32_t numFrames,
                                    void *stream) {
    uint32_t logn = 0;
    if (ref_inv_check(c, N, {d_c, d_a, d_b_hat, d_twiddles, d_precon_twiddles, d_inv_twiddles, d_inv_precon_twiddles},
                      modulus, &logn))
        return AGX_E_INVALID;
    if (numFrames == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    // NTT(a) goes to c unless c holds b_hat, which the inverse still has to read: then to a scratch buffer
    uint64_t *tmp = nullptr, *spec = d_c;
    int rc = AGX_OK;
    if (d_c == d_b_hat) {
        rc = (int)cudaMallocAsync(&tmp, (size_t)numFrames * N * 8, st);
        spec = tmp;
    }
    if (!rc) rc = ref_launch(c, logn, d_a, d_a, spec, d_twiddles, d_precon_twiddles, modulus, numFrames, st);
    if (!rc) rc = ref_inv_launch(c, logn, spec, d_b_hat, d_c, d_inv_twiddles, d_inv_precon_twiddles, modulus, numFrames, st);
    if (tmp) { const int rf = (int)cudaFreeAsync(tmp, st); if (!rc) rc = rf; }
    return rc;
}

// ------------------------------------------------------------------------------------------------ u64 RNS batches

int agx_create64(agx_ctx **out, const agx_parms64 *parms, const uint64_t *psi, int device) {
    typedef unsigned __int128 u128;
    if (!out) return AGX_E_INVALID;
    *out = nullptr;
    if (!parms || !parms->q || parms->nlimbs == 0 || parms->nlimbs > 64 || parms->logn < 2 || parms->logn > 15 ||
        parms->n != (1u << parms->logn))
        return AGX_E_INVALID;
    const uint32_t n = parms->n, logn = parms->logn, L = parms->nlimbs;
    std::vector<RnsLimb64> lc(L);
    for (uint32_t l = 0; l < L; l++) {
        const uint64_t q = parms->q[l];
        uint64_t root = minimal_psi_u64(n, q);                         // also validates q (prime, < 2^62, = 1 mod 2n)
        if (!root) return AGX_E_INVALID;
        if (psi) {                                                     // the caller's root: must be a primitive 2n-th root
            root = psi[l];
            if (root == 0 || root >= q || powmod_u64(root, n, q) != q - 1) return AGX_E_INVALID;
        }
        RnsLimb64 &x = lc[l];
        x.p = ref_inv_const(q, logn);
        x.psi = root;
        x.psi_inv = powmod_u64(root, q - 2, q);
        // iroots[1] = psi^-bitrev(1) = psi^-(n/2), with n^-1 folded in (what ref_inv_fold computes from a caller's table)
        const uint64_t w = mulmod_u64(powmod_u64(x.psi_inv, n / 2, q), x.p.ninv, q);
        x.fold = make_ulonglong2(w, (uint64_t)(((u128)w << 64) / q));
    }
    DeviceGuard guard__(device);
    if (guard__.error()) return guard__.error();
    agx_ctx *c = nullptr;
    if (const int rc = ctx_new(&c, device)) return rc;
    c->has_parms64 = true;
    c->n = n; c->logn = logn; c->L = L;
    c->q64.assign(parms->q, parms->q + L);
    for (const RnsLimb64 &x : lc) c->psi64.push_back(x.psi);
    const int frame_smem = 17 * 1024 * 8;                              // N = 16384 image: 136 KB
    cudaError_t e = cudaFuncSetAttribute(ref_u64_rns_frame_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rns_frame_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rns_frame_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rns_inv_frame_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rns_inv_frame_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rescale_fwd_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rescale_fwd_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rescale_inv_frame_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_rescale_inv_frame_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_basis_fwd_kernel<512, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_basis_fwd_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_basis_fwd_kernel<512, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_basis_fwd_kernel<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_basis_inv_frame_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ref_u64_basis_inv_frame_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, frame_smem / 2);
    const int automorph_smem = (16384 + 1) * 8;                        // one n = 16384 row and its q: 128 KB
    if (e == cudaSuccess) e = cudaFuncSetAttribute(automorph64_coeff_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, automorph_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(automorph64_coeff_cluster_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8);
    const size_t entries = (size_t)L * n;
    if (e == cudaSuccess) e = cudaMalloc(&c->d_tab64, 4 * entries * sizeof(uint64_t));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_lc64, L * sizeof(RnsLimb64));
    if (e == cudaSuccess) e = cudaMemcpy(c->d_lc64, lc.data(), L * sizeof(RnsLimb64), cudaMemcpyHostToDevice);
    // the rescale's constants (agx_rescale64): for each i < L - 1, q_{L-1}^-1 mod q_i and its Shoup companion, h mod q_i
    // and floor(2^64 / q_i); none when L = 1 or when q_{L-1} repeats an earlier prime (then it has no inverse)
    const uint64_t qlast = parms->q[L - 1];
    bool rescalable = L >= 2;
    for (uint32_t i = 0; i + 1 < L; i++) rescalable = rescalable && parms->q[i] != qlast;
    if (e == cudaSuccess && rescalable) {
        std::vector<RescaleLimb64> rs(L - 1);
        c->rs_qlast = qlast;
        c->rs_h = qlast / 2;
        for (uint32_t i = 0; i + 1 < L; i++) {
            const uint64_t q = parms->q[i];
            RescaleLimb64 &r = rs[i];
            r.q = q;
            r.one_p = (uint64_t)(((u128)1 << 64) / q);
            r.h = c->rs_h % q;
            r.qinv = powmod_u64(qlast % q, q - 2, q);
            r.qinv_p = (uint64_t)(((u128)r.qinv << 64) / q);
        }
        e = cudaMalloc(&c->d_rs64, (L - 1) * sizeof(RescaleLimb64));
        if (e == cudaSuccess) e = cudaMemcpy(c->d_rs64, rs.data(), (L - 1) * sizeof(RescaleLimb64), cudaMemcpyHostToDevice);
    }
    // the basis conversions' constants (agx_modup64 / agx_moddown64): per limb q_i, floor(2^64 / q_i) and the largest
    // multiple of q_i not above 2^63; per pair (i, j) q_j mod q_i and q_j^-1 mod q_i with their Shoup companions (the
    // inverse is 0 where q_j = q_i: the calls refuse such source sets).  Kept on the host too, for the per-call constants.
    if (e == cudaSuccess) {
        c->bl64.resize(L);
        c->bp64.resize((size_t)L * L);
        for (uint32_t i = 0; i < L; i++) {
            const uint64_t q = parms->q[i];
            c->bl64[i] = BasisLimb64{q, (uint64_t)(((u128)1 << 64) / q), q * ((1ull << 63) / q)};
            for (uint32_t j = 0; j < L; j++) {
                const uint64_t w = parms->q[j] % q, inv = w ? powmod_u64(w, q - 2, q) : 0;
                c->bp64[(size_t)i * L + j] = BasisPair64{w, (uint64_t)(((u128)w << 64) / q), inv, (uint64_t)(((u128)inv << 64) / q)};
            }
        }
        const size_t lb = L * sizeof(BasisLimb64), pb = (size_t)L * L * sizeof(BasisPair64);
        e = cudaMalloc(&c->d_bl64, lb + pb);
        if (e == cudaSuccess) {
            c->d_bp64 = reinterpret_cast<BasisPair64 *>(reinterpret_cast<char *>(c->d_bl64) + lb);
            e = cudaMemcpy(c->d_bl64, c->bl64.data(), lb, cudaMemcpyHostToDevice);
        }
        if (e == cudaSuccess) e = cudaMemcpy(c->d_bp64, c->bp64.data(), pb, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) {
        const size_t total = 2 * entries;
        gen_tables64_kernel<<<(unsigned)((total + 255) / 256), 256>>>(c->d_tab64, c->d_lc64, L, logn);
        c->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    if (e != cudaSuccess) { agx_destroy(c); return (int)e; }
    *out = c;
    return AGX_OK;
}

int agx_get_psi64(const agx_ctx *c, uint32_t limb, uint64_t *psi) {
    if (!c || !c->has_parms64 || limb >= c->L || !psi) return AGX_E_INVALID;
    *psi = c->psi64[limb];
    return AGX_OK;
}

int agx_get_tables64(const agx_ctx *c, uint32_t limb, int inverse, uint64_t *roots, uint64_t *precons) {
    if (!c || !c->has_parms64 || limb >= c->L || !roots || !precons) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    const size_t bytes = (size_t)c->n * sizeof(uint64_t), off = (size_t)limb * c->n;
    CK(cudaMemcpy(roots, tab64(c, inverse ? 2 : 0) + off, bytes, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(precons, tab64(c, inverse ? 3 : 1) + off, bytes, cudaMemcpyDeviceToHost));
    return AGX_OK;
}

int agx_ntt64_fwd(agx_ctx *c, uint64_t *d, size_t B, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {d}, B, &T)) return rc;
    if (T == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    return rns_fwd_launch(c, d, d, T, (cudaStream_t)stream, 0, c->L);
}

int agx_ntt64_inv(agx_ctx *c, uint64_t *d, size_t B, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {d}, B, &T)) return rc;
    if (T == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    return rns_inv_launch(c, d, nullptr, d, T, (cudaStream_t)stream, 0, c->L);
}

int agx_polymul64(agx_ctx *c, uint64_t *dc, const uint64_t *da, const uint64_t *db, size_t B, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {dc, da, db}, B, &T)) return rc;
    if (T == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    if (dc == db && dc != da) std::swap(da, db);                   // the product commutes: c == a from here on
    // c = NTT(a); scratch = NTT(b) unless squaring; c = INTT(c .* (scratch or c))  (agx_ref_polymul_dev's sequence)
    uint64_t *tmp = nullptr;
    int rc = rns_fwd_launch(c, da, dc, T, st, 0, c->L);
    if (!rc && da != db) {
        rc = (int)cudaMallocAsync(&tmp, T * c->n * sizeof(uint64_t), st);
        if (!rc) rc = rns_fwd_launch(c, db, tmp, T, st, 0, c->L);
    }
    if (!rc) rc = rns_inv_launch(c, dc, tmp ? tmp : dc, dc, T, st, 0, c->L);
    if (tmp) { const int rf = (int)cudaFreeAsync(tmp, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

int agx_polymul64_by_spectrum(agx_ctx *c, uint64_t *dc, const uint64_t *da, const uint64_t *db_hat, size_t B, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {dc, da, db_hat}, B, &T)) return rc;
    if (T == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    // NTT(a) goes to c unless c holds b_hat, which the inverse still has to read: then to a scratch buffer
    uint64_t *tmp = nullptr, *spec = dc;
    int rc = AGX_OK;
    if (dc == db_hat) {
        rc = (int)cudaMallocAsync(&tmp, T * c->n * sizeof(uint64_t), st);
        spec = tmp;
    }
    if (!rc) rc = rns_fwd_launch(c, da, spec, T, st, 0, c->L);
    if (!rc) rc = rns_inv_launch(c, spec, db_hat, dc, T, st, 0, c->L);
    if (tmp) { const int rf = (int)cudaFreeAsync(tmp, st); if (!rc) rc = rf; }
    return rc;
}

int agx_elementwise64(agx_ctx *c, int op, uint64_t *dc, const uint64_t *da, const uint64_t *db, size_t B, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {dc, da, db}, B, &T)) return rc;
    if (op < 0 || op > 3) return AGX_E_INVALID;
    if (T == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const size_t total2 = T * c->n / 2;
    const unsigned blocks = (unsigned)std::min<size_t>((total2 + 255) / 256, (size_t)c->sms * 16);
    const cudaStream_t s = (cudaStream_t)stream;
    ulonglong2 *c2 = reinterpret_cast<ulonglong2 *>(dc);
    const ulonglong2 *a2 = reinterpret_cast<const ulonglong2 *>(da), *b2 = reinterpret_cast<const ulonglong2 *>(db);
    switch (op) {
        case EW_ADD: elementwise64_kernel<EW_ADD><<<blocks, 256, 0, s>>>(c2, a2, b2, c->d_lc64, c->L, c->logn, total2); break;
        case EW_SUB: elementwise64_kernel<EW_SUB><<<blocks, 256, 0, s>>>(c2, a2, b2, c->d_lc64, c->L, c->logn, total2); break;
        case EW_MUL: elementwise64_kernel<EW_MUL><<<blocks, 256, 0, s>>>(c2, a2, b2, c->d_lc64, c->L, c->logn, total2); break;
        default:     elementwise64_kernel<EW_MAC><<<blocks, 256, 0, s>>>(c2, a2, b2, c->d_lc64, c->L, c->logn, total2); break;
    }
    c->launches++;
    return (int)cudaGetLastError();
}

// The launches of agx_rescale64 once the arguments are checked (B > 0); the evaluation form's scratch comes from `pool`
// (see scratch_alloc).
static int rescale_launch(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, int ntt_form, cudaStream_t st,
                          cudaMemPool_t pool) {
    const uint32_t logn = c->logn, L = c->L, N = c->n;
    const size_t T = B * L;
    if (!ntt_form) {
        const size_t pairs = B * N / 2;
        const unsigned blocks = (unsigned)std::min<size_t>((pairs + 255) / 256, (size_t)c->sms * 16);
        rescale64_coeff_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<ulonglong2 *>(d_out),
                                                       reinterpret_cast<const ulonglong2 *>(d_in), c->d_rs64, c->rs_qlast,
                                                       c->rs_h, L, logn, pairs);
        c->launches++;
        return (int)cudaGetLastError();
    }
    // evaluation form: scratch[b] = INTT_{L-1}(x_hat[b][L-1]); out[b][i] = (x_hat[b][i] - NTT_i(r_i(scratch[b]))) / q_{L-1}
    uint64_t *tmp = nullptr;
    int rc = scratch_alloc(&tmp, B * N, pool, st);
    if (!rc) {
        const RnsLimb64 *last = c->d_lc64 + (L - 1);
        const size_t toff = (size_t)(L - 1) * N;
        const uint64_t *itw = tab64(c, 2) + toff, *ipre = tab64(c, 3) + toff;
        if (logn >= 10) {
            const uint32_t split = logn == 15 ? 1u : 0u, lg = logn - split;
            const size_t smem = ((size_t)17 << (lg - 4)) * 8;
            const unsigned grid = (unsigned)(B << split);
            switch (lg) {
                case 14: ref_u64_rescale_inv_frame_kernel<512><<<grid, 512, smem, st>>>(d_in, tmp, itw, ipre, last, L, logn); break;
                case 13: ref_u64_rescale_inv_frame_kernel<256><<<grid, 256, smem, st>>>(d_in, tmp, itw, ipre, last, L, logn); break;
                case 12: ref_u64_rescale_inv_frame_kernel<128><<<grid, 128, smem, st>>>(d_in, tmp, itw, ipre, last, L, logn); break;
                case 11: ref_u64_rescale_inv_frame_kernel<64><<<grid, 64, smem, st>>>(d_in, tmp, itw, ipre, last, L, logn); break;
                default: ref_u64_rescale_inv_frame_kernel<32><<<grid, 32, smem, st>>>(d_in, tmp, itw, ipre, last, L, logn); break;
            }
            c->launches++;
            if (split) {                                           // the scratch as a batch of B frames of limb L - 1
                const size_t units = B << (logn - 2);
                const unsigned blocks = (unsigned)std::min<size_t>((units + 255) / 256, (size_t)c->sms * 8);
                ref_u64_rns_inv_last_stage_kernel<<<blocks, 256, 0, st>>>(tmp, last, 1, logn, B);
                c->launches++;
            }
        } else {
            ref_inv_u64_rescale_kernel<<<(unsigned)B, N / 2 < 32 ? 32 : N / 2, 0, st>>>(d_in, tmp, itw, ipre, last, L, logn);
            c->launches++;
        }
        rc = (int)cudaGetLastError();
    }
    if (!rc) {
        const uint64_t *tw = tab64(c, 0), *pre = tab64(c, 1);
        const RescaleLimb64 *rs = c->d_rs64;
        const uint64_t ql = c->rs_qlast, h = c->rs_h;
        const unsigned frames = (unsigned)(T - B);                 // B * (L - 1)
        if (logn >= 10) {
            const uint32_t split = logn == 15 ? 1u : 0u, lg = logn - split;
            const size_t smem = ((size_t)17 << (lg - 4)) * 8;
            const unsigned grid = frames << split;
            switch (lg) {
                case 14: ref_u64_rescale_fwd_kernel<512><<<grid, 512, smem, st>>>(d_in, tmp, d_out, tw, pre, rs, ql, h, L, logn); break;
                case 13: ref_u64_rescale_fwd_kernel<256><<<grid, 256, smem, st>>>(d_in, tmp, d_out, tw, pre, rs, ql, h, L, logn); break;
                case 12: ref_u64_rescale_fwd_kernel<128><<<grid, 128, smem, st>>>(d_in, tmp, d_out, tw, pre, rs, ql, h, L, logn); break;
                case 11: ref_u64_rescale_fwd_kernel<64><<<grid, 64, smem, st>>>(d_in, tmp, d_out, tw, pre, rs, ql, h, L, logn); break;
                default: ref_u64_rescale_fwd_kernel<32><<<grid, 32, smem, st>>>(d_in, tmp, d_out, tw, pre, rs, ql, h, L, logn); break;
            }
        } else {
            ref_fwd_u64_rescale_kernel<<<frames, N / 2 < 32 ? 32 : N / 2, (size_t)N * 8, st>>>(d_in, tmp, d_out, tw, pre, rs,
                                                                                            ql, h, L, logn);
        }
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (tmp) { const int rf = (int)cudaFreeAsync(tmp, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

int agx_rescale64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, int ntt_form, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {d_out, d_in}, B, &T)) return rc;
    if (c->L < 2 || !c->d_rs64) return AGX_E_INVALID;
    // in place is refused: the compaction from stride L to L - 1 lets one polynomial's CTAs overwrite input that
    // another polynomial's CTAs have not read yet
    const uintptr_t i0 = reinterpret_cast<uintptr_t>(d_in), i1 = i0 + T * c->n * sizeof(uint64_t);
    const uintptr_t o0 = reinterpret_cast<uintptr_t>(d_out), o1 = o0 + (T - B) * c->n * sizeof(uint64_t);
    if (B && i0 < o1 && o0 < i1) return AGX_E_INVALID;
    if (B == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    return rescale_launch(c, d_out, d_in, B, ntt_form, (cudaStream_t)stream, nullptr);
}

int agx_moddown64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, uint32_t k, int ntt_form, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {d_out, d_in}, B, &T)) return rc;
    const uint32_t L = c->L;
    if (k == 0 || k >= L || !basis_sources_distinct(c, L - k, k)) return AGX_E_INVALID;
    if (B && ranges_overlap(d_in, T * c->n, d_out, B * (L - k) * c->n)) return AGX_E_INVALID;
    if (k > kBasisMaxSrc) return AGX_E_UNSUPPORTED;
    if (B == 0) return AGX_OK;
    if (k == 1) return agx_rescale64(c, d_out, d_in, B, ntt_form, stream);   // the same division: its own kernels
    AGX_ON_DEVICE(c);
    return basis_launch(c, d_out, d_in, B, L - k, k, true, ntt_form, (cudaStream_t)stream);
}

// agx_moddown64's launches once the arguments are checked (B > 0), with the scratch from `pool` (see scratch_alloc).
static int moddown_launch(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, uint32_t k, int ntt_form,
                          cudaStream_t st, cudaMemPool_t pool) {
    if (k == 1) return rescale_launch(c, d_out, d_in, B, ntt_form, st, pool);
    return basis_launch(c, d_out, d_in, B, c->L - k, k, true, ntt_form, st, pool);
}

int agx_modup64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, uint32_t first, uint32_t count,
                int ntt_form, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {d_out, d_in}, B, &T)) return rc;
    const uint32_t L = c->L;
    if (count == 0 || count >= L || first > L - count || !basis_sources_distinct(c, first, count)) return AGX_E_INVALID;
    if (B && ranges_overlap(d_in, B * count * c->n, d_out, T * c->n)) return AGX_E_INVALID;
    if (count > kBasisMaxSrc) return AGX_E_UNSUPPORTED;
    if (B == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    return basis_launch(c, d_out, d_in, B, first, count, false, ntt_form, (cudaStream_t)stream);
}

static_assert(kAutomorphMax == AGX_AUTOMORPH_MAX, "the header states the call's bound");

int agx_automorph64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint32_t *galois, uint32_t G,
                    int ntt_form, void *stream) {
    size_t T = 0;
    if (const int rc = check_dev_call64(c, {d_out, d_in}, B, &T)) return rc;
    if (G && !galois) return AGX_E_INVALID;
    if (T && (size_t)G > 0x7fffffffull / T) return AGX_E_INVALID;
    if (T && G && ranges_overlap(d_in, T * c->n, d_out, G * T * c->n)) return AGX_E_INVALID;
    if (G > kAutomorphMax) return AGX_E_UNSUPPORTED;
    AutomorphCall64 cp{};
    cp.R = (uint32_t)T; cp.L = c->L; cp.logn = c->logn; cp.G = G;
    if (!galois_inverses(c, galois, G, cp.gi)) return AGX_E_INVALID;
    if (B == 0 || G == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    const uint32_t logn = c->logn;
    if (ntt_form) {
        const size_t pairs = T * c->n / 2;
        const unsigned blocks = (unsigned)std::min<size_t>((pairs + 255) / 256, (size_t)c->sms * 16);
        automorph64_ntt_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<ulonglong2 *>(d_out),
                                                       reinterpret_cast<const ulonglong2 *>(d_in), cp, pairs);
    } else if (logn <= 14) {
        const uint32_t rpc = (uint32_t)std::min<size_t>(std::min(kAutomorphRows, std::max(kAutomorphPart >> logn, 1u)), T);
        const size_t smem = ((size_t)rpc * (c->n + 1)) * 8;
        automorph64_coeff_kernel<<<(unsigned)((T + rpc - 1) / rpc), kAutomorphThreads, smem, st>>>(d_out, d_in, c->d_lc64, cp, rpc);
    } else {
        automorph64_coeff_cluster_kernel<2><<<(unsigned)(2 * T), kAutomorphThreads, 16384 * 8, st>>>(d_out, d_in, c->d_lc64, cp);
    }
    c->launches++;
    return (int)cudaGetLastError();
}

int agx_keyswitch64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint64_t *d_ksk,
                    uint32_t key_limbs, uint32_t alpha, uint32_t k, int ntt_form, void *stream) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : {(const void *)d_out, (const void *)d_in, (const void *)d_ksk})
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    const uint32_t L = c->L;
    if (!ks_params_valid(c, key_limbs, alpha, k)) return AGX_E_INVALID;
    const uint32_t ell1 = L - k, m = std::min(alpha, ell1), dnum = (ell1 + m - 1) / m;
    if (B > 0x7fffffffull / (2ull * L) || B > 0x7fffffffull / ((size_t)dnum * L)) return AGX_E_INVALID;
    const size_t N = c->n;
    if (B && (ranges_overlap(d_out, 2 * B * ell1 * N, d_in, B * ell1 * N) ||
              ranges_overlap(d_out, 2 * B * ell1 * N, d_ksk, (size_t)dnum * 2 * key_limbs * N)))
        return AGX_E_INVALID;
    if (m > kBasisMaxSrc || k > kBasisMaxSrc) return AGX_E_UNSUPPORTED;
    if (B == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t T = B * L;
    // scratch: U [dnum][B][L][n] (the extended digits), A [2][B][L][n] (the inner products), and with dnum > 1 one
    // digit [B][m][n] gathered out of d_in for ModUp, which reads its source limbs contiguously
    int rc = ks_pool_ready(c);
    if (rc) return rc;
    uint64_t *U = nullptr;
    rc = (int)cudaMallocFromPoolAsync(reinterpret_cast<void **>(&U),
                                      ((dnum + 2) * T + (dnum > 1 ? B * m : 0)) * N * sizeof(uint64_t), c->ks_pool, st);
    uint64_t *A = rc ? nullptr : U + dnum * T * N, *dig = rc ? nullptr : A + 2 * T * N;
    if (!rc) rc = ks_modup_digits(c, U, dig, d_in, B, ell1, m, dnum, ntt_form, st);
    if (!rc && !ntt_form) rc = rns_fwd_launch(c, U, U, dnum * T, st, 0, L);   // the products are per limb in evaluation form
    if (!rc) {
        KeySwitchCall64 cp{};
        cp.L = L; cp.logn = c->logn; cp.ell1 = ell1; cp.key_off = key_limbs - L; cp.key_limbs = key_limbs;
        cp.dnum = dnum; cp.B = (uint32_t)B;
        const size_t per_slice = (size_t)L * N / 2;
        cp.slice = ks_slice(c, B, per_slice);
        const size_t items = ((B + cp.slice - 1) / cp.slice) * per_slice;
        const unsigned blocks = (unsigned)std::min<size_t>((items + 255) / 256, (size_t)c->sms * 8);
        auto *a2 = reinterpret_cast<ulonglong2 *>(A);
        const auto *u2 = reinterpret_cast<const ulonglong2 *>(U), *k2 = reinterpret_cast<const ulonglong2 *>(d_ksk);
        if (dnum == 1) keyswitch64_inner_kernel<1><<<blocks, 256, 0, st>>>(a2, u2, k2, c->d_lc64, cp, items);
        else if (dnum == 2) keyswitch64_inner_kernel<2><<<blocks, 256, 0, st>>>(a2, u2, k2, c->d_lc64, cp, items);
        else if (dnum <= 4) keyswitch64_inner_kernel<4><<<blocks, 256, 0, st>>>(a2, u2, k2, c->d_lc64, cp, items);
        else keyswitch64_inner_kernel<kKeySwitchChunk><<<blocks, 256, 0, st>>>(a2, u2, k2, c->d_lc64, cp, items);
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc && !ntt_form) rc = rns_inv_launch(c, A, nullptr, A, 2 * T, st, 0, L);
    if (!rc) rc = agx_moddown64(c, d_out, A, 2 * B, k, ntt_form, stream);   // both components as one batch of 2B
    if (U) { const int rf = (int)cudaFreeAsync(U, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

int agx_rotate64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint32_t *galois, uint32_t G,
                 const uint64_t *const *d_rk, uint32_t key_limbs, uint32_t alpha, uint32_t k, int ntt_form, void *stream) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : {(const void *)d_out, (const void *)d_in})
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    if (G && (!galois || !d_rk)) return AGX_E_INVALID;
    const uint32_t L = c->L;
    if (!ks_params_valid(c, key_limbs, alpha, k)) return AGX_E_INVALID;
    const uint32_t ell1 = L - k, m = std::min(alpha, ell1), dnum = (ell1 + m - 1) / m;
    if (B > 0x7fffffffull / ((size_t)dnum * L) || (B && G > 0x7fffffffull / (2ull * L * B))) return AGX_E_INVALID;
    const size_t N = c->n;
    const size_t in_w = 2 * B * ell1 * N, out_w = (size_t)G * in_w, key_w = (size_t)dnum * 2 * key_limbs * N;
    if (B && G && ranges_overlap(d_out, out_w, d_in, in_w)) return AGX_E_INVALID;
    if (G > kAutomorphMax) return AGX_E_UNSUPPORTED;               // elements and keys are not read
    RotateCall64 cp{};
    if (!galois_inverses(c, galois, G, cp.gi)) return AGX_E_INVALID;
    for (uint32_t t = 0; t < G; t++) {
        const uint64_t *rk = d_rk[t];
        if ((B && !rk) || (reinterpret_cast<uintptr_t>(rk) & 15)) return AGX_E_INVALID;
        if (B && ranges_overlap(d_out, out_w, rk, key_w)) return AGX_E_INVALID;
        cp.rk[t] = reinterpret_cast<const ulonglong2 *>(rk);
    }
    if (m > kBasisMaxSrc || k > kBasisMaxSrc) return AGX_E_UNSUPPORTED;
    if (B == 0 || G == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t T = B * L;
    // scratch: U [dnum][B][L][n] (c1's extended digits), A [G][2][B][L][n] (the inner products), with dnum > 1 one digit
    // [B][m][n] gathered for ModUp, and in coefficient form c0's spectrum [B][l+1][n]
    int rc = ks_pool_ready(c);
    if (rc) return rc;
    uint64_t *U = nullptr;
    const size_t words = (dnum + 2 * (size_t)G) * T + (dnum > 1 ? B * m : 0) + (ntt_form ? 0 : B * ell1);
    rc = (int)cudaMallocFromPoolAsync(reinterpret_cast<void **>(&U), words * N * sizeof(uint64_t), c->ks_pool, st);
    uint64_t *A = rc ? nullptr : U + dnum * T * N, *dig = rc ? nullptr : A + 2 * G * T * N;
    uint64_t *c0h = rc ? nullptr : dig + (dnum > 1 ? B * m * N : 0);
    const uint64_t *c1 = d_in + B * ell1 * N;
    if (!rc) rc = ks_modup_digits(c, U, dig, c1, B, ell1, m, dnum, ntt_form, st);
    if (!rc && !ntt_form) rc = rns_fwd_launch(c, U, U, dnum * T, st, 0, L);   // the products are per limb in evaluation form
    if (!rc && !ntt_form) rc = rns_fwd_launch(c, d_in, c0h, B * ell1, st, 0, ell1);
    if (!rc) {
        KeySwitchCall64 &ks = cp.ks;
        ks.L = L; ks.logn = c->logn; ks.ell1 = ell1; ks.key_off = key_limbs - L; ks.key_limbs = key_limbs;
        ks.dnum = dnum; ks.B = (uint32_t)B;
        cp.G = G;
        const size_t per_slice = (size_t)G * L * N / 2;
        ks.slice = ks_slice(c, B, per_slice);
        const size_t items = ((B + ks.slice - 1) / ks.slice) * per_slice;
        const unsigned blocks = (unsigned)std::min<size_t>((items + 255) / 256, (size_t)c->sms * 8);
        auto *a2 = reinterpret_cast<ulonglong2 *>(A);
        const auto *u2 = reinterpret_cast<const ulonglong2 *>(U);
        const auto *c02 = reinterpret_cast<const ulonglong2 *>(ntt_form ? d_in : c0h);
        const BasisPair64 *bp = c->d_bp64;
        if (dnum == 1) rotate64_inner_kernel<1><<<blocks, 256, 0, st>>>(a2, u2, c02, c->d_lc64, bp, cp, items);
        else if (dnum == 2) rotate64_inner_kernel<2><<<blocks, 256, 0, st>>>(a2, u2, c02, c->d_lc64, bp, cp, items);
        else if (dnum <= 4) rotate64_inner_kernel<4><<<blocks, 256, 0, st>>>(a2, u2, c02, c->d_lc64, bp, cp, items);
        else rotate64_inner_kernel<kKeySwitchChunk><<<blocks, 256, 0, st>>>(a2, u2, c02, c->d_lc64, bp, cp, items);
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc && !ntt_form) rc = rns_inv_launch(c, A, nullptr, A, 2 * G * T, st, 0, L);
    // every output's two components as one batch of 2 G B, with its scratch from the pool too
    if (!rc) rc = moddown_launch(c, d_out, A, 2 * G * B, k, ntt_form, st, c->ks_pool);
    if (U) { const int rf = (int)cudaFreeAsync(U, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

static_assert(kLintransMaxOut == AGX_LINTRANS_MAX_OUT && kLintransMaxTerms == AGX_LINTRANS_MAX_TERMS,
              "the header states the call's bounds");

int agx_lintrans64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_in, size_t B, const uint32_t *galois, uint32_t G,
                   const uint64_t *const *d_rk, uint32_t key_limbs, const uint64_t *const *d_diag, uint32_t M,
                   uint32_t alpha, uint32_t k, int ntt_form, void *stream) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : {(const void *)d_out, (const void *)d_in})
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    if (G && (!galois || !d_rk)) return AGX_E_INVALID;
    if (M && (!G || !d_diag)) return AGX_E_INVALID;
    const uint32_t L = c->L;
    if (!ks_params_valid(c, key_limbs, alpha, k)) return AGX_E_INVALID;
    const uint32_t ell1 = L - k, m = std::min(alpha, ell1), dnum = (ell1 + m - 1) / m;
    if (B > 0x7fffffffull / ((size_t)dnum * L) || (B && M > 0x7fffffffull / (2ull * L * B))) return AGX_E_INVALID;
    const size_t N = c->n;
    const size_t in_w = 2 * B * ell1 * N, out_w = (size_t)M * in_w, key_w = (size_t)dnum * 2 * key_limbs * N;
    const bool work = B && M;
    if (work && ranges_overlap(d_out, out_w, d_in, in_w)) return AGX_E_INVALID;
    if (G > kAutomorphMax || M > kLintransMaxOut || (size_t)M * G > kLintransMaxTerms) return AGX_E_UNSUPPORTED;
    LintransCall64 cp{};
    uint32_t gi[kAutomorphMax];                                    // unused: the kernel gathers with g itself
    if (!galois_inverses(c, galois, G, gi)) return AGX_E_INVALID;
    for (uint32_t t = 0; t < G; t++) {
        const uint64_t *rk = d_rk[t];
        if ((B && !rk && galois[t] != 1) || (reinterpret_cast<uintptr_t>(rk) & 15)) return AGX_E_INVALID;
        if (work && rk && ranges_overlap(d_out, out_w, rk, key_w)) return AGX_E_INVALID;
    }
    uint32_t keep[kAutomorphMax];                                  // the terms with a non-zero diagonal: the others add nothing
    for (uint32_t t = 0; t < G; t++) {
        bool used = false;
        for (uint32_t j = 0; j < M; j++) {
            const uint64_t *d = d_diag[(size_t)j * G + t];
            if (reinterpret_cast<uintptr_t>(d) & 15) return AGX_E_INVALID;
            if (work && d && ranges_overlap(d_out, out_w, d, (size_t)L * N)) return AGX_E_INVALID;
            used |= d != nullptr;
        }
        if (used) keep[cp.G++] = t;
    }
    if (m > kBasisMaxSrc || k > kBasisMaxSrc) return AGX_E_UNSUPPORTED;
    if (!work) return AGX_OK;
    for (uint32_t u = 0; u < cp.G; u++) {
        const uint32_t t = keep[u];
        cp.g[u] = galois[t];
        cp.rk[u] = reinterpret_cast<const ulonglong2 *>(d_rk[t]);
        for (uint32_t j = 0; j < M; j++) cp.diag[j * cp.G + u] = reinterpret_cast<const ulonglong2 *>(d_diag[(size_t)j * G + t]);
    }
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t T = B * L;
    // scratch: U [dnum][B][L][n] (c1's extended digits), Acc [M][2][B][L][n] (the sums), with dnum > 1 one digit
    // [B][m][n] gathered for ModUp, and in coefficient form the spectra of c0 and c1 [2][B][l+1][n]
    int rc = ks_pool_ready(c);
    if (rc) return rc;
    uint64_t *U = nullptr;
    const size_t words = (dnum + 2 * (size_t)M) * T + (dnum > 1 ? B * m : 0) + (ntt_form ? 0 : 2 * B * ell1);
    rc = (int)cudaMallocFromPoolAsync(reinterpret_cast<void **>(&U), words * N * sizeof(uint64_t), c->ks_pool, st);
    uint64_t *Acc = rc ? nullptr : U + dnum * T * N, *dig = rc ? nullptr : Acc + 2 * M * T * N;
    uint64_t *cth = rc ? nullptr : dig + (dnum > 1 ? B * m * N : 0);
    if (!rc) rc = ks_modup_digits(c, U, dig, d_in + B * ell1 * N, B, ell1, m, dnum, ntt_form, st);
    if (!rc && !ntt_form) rc = rns_fwd_launch(c, U, U, dnum * T, st, 0, L);   // the products are per limb in evaluation form
    if (!rc && !ntt_form) rc = rns_fwd_launch(c, d_in, cth, 2 * B * ell1, st, 0, ell1);   // c0 and c1 in one launch
    if (!rc) {
        KeySwitchCall64 &ks = cp.ks;
        ks.L = L; ks.logn = c->logn; ks.ell1 = ell1; ks.key_off = key_limbs - L; ks.key_limbs = key_limbs;
        ks.dnum = dnum; ks.B = (uint32_t)B;
        cp.M = M;
        const size_t items = T * N / 2;
        const unsigned blocks = (unsigned)std::min<size_t>((items + 255) / 256, (size_t)c->sms * 8);
        auto *a2 = reinterpret_cast<ulonglong2 *>(Acc);
        const auto *u2 = reinterpret_cast<const ulonglong2 *>(U);
        const auto *c2 = reinterpret_cast<const ulonglong2 *>(ntt_form ? d_in : cth);
        const RnsLimb64 *lc = c->d_lc64;
        const BasisPair64 *bp = c->d_bp64;
#define AGX_LINTRANS(DC)                                                                               \
    (M <= 4 ? lintrans64_inner_kernel<DC, 4><<<blocks, 256, 0, st>>>(a2, u2, c2, lc, bp, cp, items)    \
            : lintrans64_inner_kernel<DC, 16><<<blocks, 256, 0, st>>>(a2, u2, c2, lc, bp, cp, items))
        if (dnum == 1) AGX_LINTRANS(1);
        else if (dnum == 2) AGX_LINTRANS(2);
        else if (dnum <= 4) AGX_LINTRANS(4);
        else AGX_LINTRANS(kKeySwitchChunk);
#undef AGX_LINTRANS
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc && !ntt_form) rc = rns_inv_launch(c, Acc, nullptr, Acc, 2 * M * T, st, 0, L);
    // every output's two components as one batch of 2 M B, with its scratch from the pool too
    if (!rc) rc = moddown_launch(c, d_out, Acc, 2 * M * B, k, ntt_form, st, c->ks_pool);
    if (U) { const int rf = (int)cudaFreeAsync(U, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

int agx_mulrelin64(agx_ctx *c, uint64_t *d_out, const uint64_t *d_a, const uint64_t *d_b, size_t B,
                   const uint64_t *d_rlk, uint32_t key_limbs, uint32_t alpha, uint32_t k, int rescale, int ntt_form,
                   void *stream) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : {(const void *)d_out, (const void *)d_a, (const void *)d_b, (const void *)d_rlk})
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    const uint32_t L = c->L;
    if (!ks_params_valid(c, key_limbs, alpha, k)) return AGX_E_INVALID;
    const uint32_t ell1 = L - k, m = std::min(alpha, ell1), dnum = (ell1 + m - 1) / m;
    if (rescale && ell1 < 2) return AGX_E_INVALID;
    if (B > 0x7fffffffull / (2ull * L) || B > 0x7fffffffull / ((size_t)dnum * L)) return AGX_E_INVALID;
    const uint32_t kd = rescale ? k + 1 : k;                       // the last kd primes are divided out: P or q_l P
    const size_t N = c->n;
    const size_t in_w = 2 * B * ell1 * N, out_w = 2 * B * (L - kd) * N, key_w = (size_t)dnum * 2 * key_limbs * N;
    if (B && (ranges_overlap(d_out, out_w, d_a, in_w) || ranges_overlap(d_out, out_w, d_b, in_w) ||
              ranges_overlap(d_out, out_w, d_rlk, key_w)))
        return AGX_E_INVALID;
    if (m > kBasisMaxSrc || kd > kBasisMaxSrc) return AGX_E_UNSUPPORTED;
    if (B == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t T = B * L, Tq = B * ell1;
    const bool square = d_a == d_b;
    // scratch: U [dnum][B][L][n] (D_2's extended digits), Acc [2][B][L][n] (the sums), D_2's spectrum [B][l+1][n], with
    // dnum > 1 one digit [B][m][n] gathered for ModUp, and in coefficient form the spectra of a and b [2][B][l+1][n]
    // (one of them when squaring)
    int rc = ks_pool_ready(c);
    if (rc) return rc;
    uint64_t *U = nullptr;
    const size_t words = (dnum + 2) * T + Tq + (dnum > 1 ? B * m : 0) + (ntt_form ? 0 : (square ? 2 : 4) * Tq);
    rc = (int)cudaMallocFromPoolAsync(reinterpret_cast<void **>(&U), words * N * sizeof(uint64_t), c->ks_pool, st);
    uint64_t *Acc = rc ? nullptr : U + dnum * T * N, *d2 = rc ? nullptr : Acc + 2 * T * N;
    uint64_t *dig = rc ? nullptr : d2 + Tq * N, *ah = rc ? nullptr : dig + (dnum > 1 ? B * m * N : 0);
    uint64_t *bh = rc || square ? ah : ah + 2 * Tq * N;
    if (!rc && !ntt_form) rc = rns_fwd_launch(c, d_a, ah, 2 * Tq, st, 0, ell1);
    if (!rc && !ntt_form && !square) rc = rns_fwd_launch(c, d_b, bh, 2 * Tq, st, 0, ell1);
    const uint64_t *sa = ntt_form ? d_a : ah, *sb = ntt_form ? d_b : bh;
    if (!rc) {                                                     // D_2's spectrum a1 b1 over Q_l, for ModUp
        const size_t total2 = Tq * N / 2;
        const unsigned blocks = (unsigned)std::min<size_t>((total2 + 255) / 256, (size_t)c->sms * 16);
        elementwise64_kernel<EW_MUL><<<blocks, 256, 0, st>>>(reinterpret_cast<ulonglong2 *>(d2),
                                                             reinterpret_cast<const ulonglong2 *>(sa + Tq * N),
                                                             reinterpret_cast<const ulonglong2 *>(sb + Tq * N),
                                                             c->d_lc64, ell1, c->logn, total2);
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc) rc = ks_modup_digits(c, U, dig, d2, B, ell1, m, dnum, 1, st);
    if (!rc) {
        KeySwitchCall64 cp{};
        cp.L = L; cp.logn = c->logn; cp.ell1 = ell1; cp.key_off = key_limbs - L; cp.key_limbs = key_limbs;
        cp.dnum = dnum; cp.B = (uint32_t)B;
        const size_t per_slice = (size_t)L * N / 2;
        cp.slice = ks_slice(c, B, per_slice);
        const size_t items = ((B + cp.slice - 1) / cp.slice) * per_slice;
        const unsigned blocks = (unsigned)std::min<size_t>((items + 255) / 256, (size_t)c->sms * 8);
        auto *acc2 = reinterpret_cast<ulonglong2 *>(Acc);
        const auto *u2 = reinterpret_cast<const ulonglong2 *>(U), *k2 = reinterpret_cast<const ulonglong2 *>(d_rlk);
        const auto *a2 = reinterpret_cast<const ulonglong2 *>(sa), *b2 = reinterpret_cast<const ulonglong2 *>(sb);
        const RnsLimb64 *lc = c->d_lc64;
        const BasisPair64 *bp = c->d_bp64;
        if (dnum == 1) mulrelin64_inner_kernel<1><<<blocks, 256, 0, st>>>(acc2, u2, a2, b2, k2, lc, bp, cp, items);
        else if (dnum == 2) mulrelin64_inner_kernel<2><<<blocks, 256, 0, st>>>(acc2, u2, a2, b2, k2, lc, bp, cp, items);
        else if (dnum <= 4) mulrelin64_inner_kernel<4><<<blocks, 256, 0, st>>>(acc2, u2, a2, b2, k2, lc, bp, cp, items);
        else mulrelin64_inner_kernel<kKeySwitchChunk><<<blocks, 256, 0, st>>>(acc2, u2, a2, b2, k2, lc, bp, cp, items);
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc && !ntt_form) rc = rns_inv_launch(c, Acc, nullptr, Acc, 2 * T, st, 0, L);
    // both components as one batch of 2 B over the last k primes, or the last k + 1 for the rescale
    if (!rc) rc = moddown_launch(c, d_out, Acc, 2 * B, kd, ntt_form, st, c->ks_pool);
    if (U) { const int rf = (int)cudaFreeAsync(U, st); if (!rc) rc = rf; }   // freed on every path
    return rc;
}

int agx_encode64(agx_ctx *c, uint64_t *d_out, const double *d_slots, size_t B, double scale, uint32_t limbs,
                 int ntt_form, void *stream) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : {(const void *)d_out, (const void *)d_slots})
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    // scale / S must stay normal for the fold of 1 / S into it to be exact
    if (limbs == 0 || limbs > c->L || !std::isfinite(scale) || !(scale >= std::ldexp(1.0, -1022) * (c->n / 2)))
        return AGX_E_INVALID;
    if (B > 0x7fffffffull / limbs) return AGX_E_INVALID;
    const size_t N = c->n;
    if (B && ranges_overlap(d_out, B * limbs * N, d_slots, B * N)) return AGX_E_INVALID;
    if (B == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    int rc = slots_ready(c);
    if (rc) return rc;
    slot_fft_launch(c, true, d_out, d_slots, B, limbs, scale / (double)(N / 2), st);   // 1 / S folded in: exact (normal)
    rc = (int)cudaGetLastError();
    if (!rc && ntt_form) rc = rns_fwd_launch(c, d_out, d_out, B * limbs, st, 0, limbs);
    return rc;
}

int agx_decode64(agx_ctx *c, double *d_slots, const uint64_t *d_in, size_t B, double scale, uint32_t limbs,
                 int ntt_form, void *stream) {
    if (!c || !c->has_parms64) return AGX_E_INVALID;
    for (const void *p : {(const void *)d_slots, (const void *)d_in})
        if ((B && !p) || (reinterpret_cast<uintptr_t>(p) & 15)) return AGX_E_INVALID;
    if (limbs == 0 || limbs > c->L || !(scale > 0) || !std::isfinite(scale)) return AGX_E_INVALID;
    if (B > 0x7fffffffull / limbs) return AGX_E_INVALID;
    for (uint32_t i = 0; i < limbs; i++)
        for (uint32_t j = 0; j < i; j++)
            if (c->q64[i] == c->q64[j]) return AGX_E_INVALID;
    const size_t N = c->n;
    if (B && ranges_overlap(d_slots, B * N, d_in, B * limbs * N)) return AGX_E_INVALID;
    if (B == 0) return AGX_OK;
    AGX_ON_DEVICE(c);
    const cudaStream_t st = (cudaStream_t)stream;
    int rc = slots_ready(c);
    if (!rc) rc = ks_pool_ready(c);
    if (rc) return rc;
    // the CRT constants: scale = sm 2^se, and the mixed-radix digits of h = (Q - 1) / 2, whose residues are (q_t - 1) / 2
    DecodeCall64 cp{};
    cp.logn = c->logn; cp.limbs = limbs; cp.L = c->L;
    cp.sm = frexp(scale, &cp.se);
    for (uint32_t t = 0; t < limbs; t++) {
        const uint64_t q = c->q64[t];
        uint64_t v = (q - 1) / 2;
        for (uint32_t j = 0; j < t; j++)
            v = mulmod_u64((v + q - cp.hd[j] % q) % q, c->bp64[(size_t)t * c->L + j].inv, q);
        cp.hd[t] = v;
    }
    // scratch: m [B][n] doubles, and in evaluation form the coefficient-form residues [B][limbs][n]
    uint64_t *tmp = nullptr;
    rc = scratch_alloc(&tmp, B * N + (ntt_form ? B * limbs * N : 0), c->ks_pool, st);
    if (rc) return rc;
    double *m = reinterpret_cast<double *>(tmp);
    const uint64_t *src = d_in;
    if (ntt_form) {
        rc = rns_inv_launch(c, d_in, nullptr, tmp + B * N, B * limbs, st, 0, limbs);
        src = tmp + B * N;
    }
    if (!rc) {
        const size_t total = B * N;
        const unsigned blocks = (unsigned)std::min<size_t>((total + kDecodeCrtThreads - 1) / kDecodeCrtThreads,
                                                           (size_t)c->sms * 16);
        decode64_crt_kernel<<<blocks, kDecodeCrtThreads, (size_t)limbs * kDecodeCrtThreads * 8, st>>>(
            m, src, c->d_bl64, c->d_bp64, cp, total);
        c->launches++;
        rc = (int)cudaGetLastError();
    }
    if (!rc) {
        slot_fft_launch(c, false, d_slots, m, B, limbs, 0.0, st);
        rc = (int)cudaGetLastError();
    }
    const int rf = (int)cudaFreeAsync(tmp, st);                  // freed on every path
    return rc ? rc : rf;
}

int agx_measure_butterfly_peak(agx_ctx *c, int kind, int threads_per_sm, double *per_clk_per_sm, double *sm_mhz) {
    if (!c || !per_clk_per_sm || kind < 0 || kind > 6) return AGX_E_INVALID;
    if (threads_per_sm < 128 || threads_per_sm > 1024 || threads_per_sm % 128) return AGX_E_INVALID;
    AGX_ON_DEVICE(c);
    uint32_t *d_out = nullptr;
    long long *d_cyc = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    const int sms = c->sms;
    const uint32_t q = 1053818881u;
    const LimbConst lc{q, 2 * q, 0u - q, 0u - 2 * q, 0, 29, 0, 0};
    const uint64_t q64 = 1152921504606584833ull;
    cudaError_t e = cudaMalloc(&d_out, sizeof(uint32_t) * sms * 1024);
    if (e == cudaSuccess) e = cudaMalloc(&d_cyc, sizeof(long long) * sms);
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    float ms = 0;
    std::vector<long long> cyc(sms);
    if (e == cudaSuccess) {
        for (int rep = 0; rep < 2; rep++) {                // first launch warms the clocks and the instruction cache
            if (rep == 1) cudaEventRecord(e0, 0);
            const uint2 wc = make_uint2(12345u | 1u, 12345u * 3u + 5u);
#define AGX_DIAG(K) diag_bfly_kernel<K><<<sms, threads_per_sm>>>(d_out, d_cyc, 12345u, lc, q64, wc)
            switch (kind) {
                case 0: AGX_DIAG(0); break;
                case 1: AGX_DIAG(1); break;
                case 2: AGX_DIAG(2); break;
                case 3: AGX_DIAG(3); break;
                case 4: AGX_DIAG(4); break;
                case 5: AGX_DIAG(5); break;
                default: AGX_DIAG(6); break;
            }
#undef AGX_DIAG
            c->launches++;
        }
        cudaEventRecord(e1, 0);
        e = cudaEventSynchronize(e1);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        if (e == cudaSuccess) e = cudaMemcpy(cyc.data(), d_cyc, sizeof(long long) * sms, cudaMemcpyDeviceToHost);
    }
    if (e == cudaSuccess) {
        std::sort(cyc.begin(), cyc.end());
        const double med = (double)cyc[sms / 2];
        *per_clk_per_sm = (double)kDiagIters * kDiagUnroll * kDiagChains * threads_per_sm / med;
        if (sm_mhz) *sm_mhz = ms > 0 ? med / (ms * 1e3) : 0.0;
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(d_out); cudaFree(d_cyc);
    return (int)e;
}

const char *agx_error_string(int code) {
    switch (code) {
        case AGX_OK: return "ok";
        case AGX_E_INVALID: return "invalid argument";
        case AGX_E_UNSUPPORTED: return "unsupported request";
        case AGX_E_NOMEM: return "host allocation failed";
        case AGX_E_STATE: return "reference-shaped calls out of protocol";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int agx_launch_count(const agx_ctx *c, uint64_t *count) {
    if (!c || !count) return AGX_E_INVALID;
    *count = c->launches;
    return AGX_OK;
}

int agx_variant(const agx_ctx *c, char *buf, size_t buflen) {
    if (!c || !buf || !buflen) return AGX_E_INVALID;
    if (c->has_parms64) snprintf(buf, buflen, "u64_rns<%u>", c->logn);
    else if (!c->has_parms) snprintf(buf, buflen, "ref_u64");
    else if (c->r16) snprintf(buf, buflen, "ntt_r16<%u>", c->logn);
    else if (c->le) snprintf(buf, buflen, "ntt2p<%u,%d>", c->logn, c->le);
    else if (c->big) snprintf(buf, buflen, "ntt_big<%u>", c->logn);
    else snprintf(buf, buflen, "generic");
    return AGX_OK;
}

}  // extern "C"
