"""u64 RNS hoisted rotations in one call (agx_rotate64, Context64.rotate).

Definition, for a context over Q_l u P (the k special primes last), ciphertexts ct = (c0, c1) over Q_l, G Galois
elements and G keys in agx_keyswitch64's layout, key t switching sigma_t(s) to s:
    out[t] = ( sigma_t(c0) + KS_t(sigma_t(c1))[0] ,  KS_t(sigma_t(c1))[1] ),
sigma_t being agx_automorph64 with galois[t] and KS_t agx_keyswitch64 with key t: the plain recipe of public calls.

The call computes it with one ModUp of c1 for all G, the automorphism applied to the extended digits, and sigma_t(c0)
folded into the inner product as P * sigma_t(c0), which ModDown returns exactly.  The CPU tests pin a big-integer
oracle of the definition (built from the key-switch and automorphism oracles) as a rotation that decrypts within the key
switch's bound, check that the hoisted route equals it on big integers, pin the fold identity including its boundary
values, and check the new kernels' resources.  The GPU tests compare the call with the plain recipe bit for bit in both
forms and cover digit shapes, one key set at several levels, element and key variety, batches, an end-to-end rotation,
refusals, launch counts, unchanged inputs and side-stream ordering."""
import ctypes as C
import random
import re
from math import prod

import numpy as np
import pytest

import test_u64_automorph as AM
import test_u64_keyswitch as KS
from oracle import oracle as O

gpu = pytest.mark.gpu
SIZES = KS.SIZES
PRIMES, QS, PS, Q17, P17 = KS.PRIMES, KS.QS, KS.PS, KS.Q17, KS.P17


# ---- big ints: the oracle
def rotate_oracle(ct, gs, kcoefs, primes, k, alpha):
    """ct [2][B][l+1][N] in coefficient form over primes[:l+1]; kcoefs[t] key t in coefficient form (as
    keyswitch_oracle takes it) -> [G][2][B][l+1][N]: the plain recipe on the oracles of its parts."""
    qs = primes[:len(primes) - k]
    q = np.array(qs, dtype=object).reshape(1, -1, 1)
    out = []
    for g, kc in zip(gs, kcoefs):
        r0, r1 = AM.automorph_coeff(ct[0], g, qs), AM.automorph_coeff(ct[1], g, qs)
        ks = KS.keyswitch_oracle(r1, kc, primes, k, alpha)
        out.append(np.stack([((r0.astype(object) + ks[0].astype(object)) % q).astype(np.uint64), ks[1]]))
    return np.stack(out)


def hoisted_bigint(ct, gs, kcoefs, primes, k, alpha):
    """The call's route on big integers: the centred lift of each digit of c1 (not rotated), sigma_t of the lifted
    integers, the negacyclic products with key t summed mod QP, plus P * sigma_t(c0) (c0's CRT value in [0, Q)), then
    floor((X + h_P) / P) mod Q."""
    L = len(primes)
    ell1 = L - k
    Q, P, QP = prod(primes[:ell1]), prod(primes[ell1:]), prod(primes)
    _, B, _, N = ct.shape
    out = np.empty((len(gs), 2, B, ell1, N), dtype=np.uint64)
    for t, (g, kc) in enumerate(zip(gs, kcoefs)):
        rows = KS.key_rows(L, k, kc.shape[2])
        keys = [[[KS.crt([kc[j, c, rows[i], x] for i in range(L)], primes) for x in range(N)] for c in (0, 1)]
                for j in range(len(KS.digits_of(ell1, alpha)))]
        for b in range(B):
            acc = [[0] * N, [0] * N]
            for j, (f, cnt) in enumerate(KS.digits_of(ell1, alpha)):
                src = primes[f:f + cnt]
                S = prod(src)
                h = (S - 1) // 2
                U = AM.automorph_ints([(KS.crt(ct[1, b, f:f + cnt, x], src) + h) % S - h for x in range(N)], g)
                for c in (0, 1):
                    acc[c] = [(u + v) % QP for u, v in zip(acc[c], KS.negacyclic(U, keys[j][c]))]
            C0 = AM.automorph_ints([KS.crt(ct[0, b, :, x], primes[:ell1]) for x in range(N)], g)
            acc[0] = [(X + P * c0) % QP for X, c0 in zip(acc[0], C0)]
            for c in (0, 1):
                Y = [((X + (P - 1) // 2) // P) % Q for X in acc[c]]
                for i, q in enumerate(primes[:ell1]):
                    out[t, c, b, i] = [y % q for y in Y]
    return out


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("N,qs,ps,alpha", [(8, QS[:3], PS, 1), (16, QS, PS, 2), (32, QS[:4], PS[:1], 3)])
def test_oracle_is_a_rotation(N, qs, ps, alpha):
    """With gadget keys for sigma_t(s), the oracle's out[t] decrypts under s to sigma_t(c0 + c1 s) within the key
    switch's bound, and the call's hoisted route gives the same words."""
    rng = random.Random(N * 3 + alpha)
    primes, k = qs + ps, len(ps)
    gs = [1, AM.galois_element(N, 1), 2 * N - 1]
    s = KS.ternary(rng, N)
    ebound = 6
    kcs = [KS.gadget_key_coeff(primes, k, alpha, len(qs), s, AM.automorph_ints(s, g), ebound, rng) for g in gs]
    ct = np.stack([KS.rand_res(2, qs, N, rng) for _ in (0, 1)])
    out = rotate_oracle(ct, gs, kcs, primes, k, alpha)
    assert (hoisted_bigint(ct, gs, kcs, primes, k, alpha) == out).all()
    Q = prod(qs)
    bound = KS.ks_bound(qs, ps, alpha, N, ebound)
    assert bound < Q >> 40
    for b in range(2):
        m = [(KS.crt(ct[0, b, :, x], qs) + v) % Q
             for x, v in enumerate(KS.negacyclic([KS.crt(ct[1, b, :, x], qs) for x in range(N)], s))]
        for t, g in enumerate(gs):
            c0 = [KS.crt(out[t, 0, b, :, x], qs) for x in range(N)]
            c1 = [KS.crt(out[t, 1, b, :, x], qs) for x in range(N)]
            r = [(u + v - w) % Q for u, v, w in zip(c0, KS.negacyclic(c1, s), AM.automorph_ints(m, g))]
            assert max(min(v, Q - v) for v in r) <= bound, (b, g)


@pytest.mark.parametrize("ps", [PS, PS[:1], [PRIMES[62][5], PRIMES[60][5], PRIMES[50][5]]])
def test_fold_identity(ps):
    """floor((X + P C + h_P) / P) = C + floor((X + h_P) / P) for every integer C >= 0 and X >= 0, so ModDown of
    X + P C mod QP is ModDown(X) + C mod Q whenever X + P C < QP (the special primes see P C = 0); pinned on seeded
    values and on the boundaries where X + h_P crosses a multiple of P."""
    qs = QS
    Q, P = prod(qs), prod(ps)
    QP, hP = Q * P, (P - 1) // 2
    rng = random.Random(len(ps))
    Xs = [0, 1, hP - 1, hP, hP + 1, P - hP - 1, P - hP, P - 1, P, P + hP, QP - P * Q // 2, QP - 1 - P * (Q - 1)]
    Xs += [m * P - hP + d for m in (1, 2, Q // 3) for d in (-1, 0, 1)]
    Xs += [rng.randrange(QP) for _ in range(200)]
    Cs = [0, 1, Q - 1, Q // 2] + [rng.randrange(Q) for _ in range(20)]
    down = lambda X: ((X % QP + hP) // P) % Q
    for X in Xs:
        for Cv in Cs:
            assert (X + P * Cv + hP) // P == Cv + (X + hP) // P
            assert down(X + P * Cv) == (down(X) + Cv) % Q
    # in RNS: the special primes' residues do not change, so the ModDown's conversion of them does not either
    for X in Xs[:20]:
        for p in ps:
            assert (X + P * Cs[-1]) % p == X % p


def test_rotate_kernels_use_no_local_memory():
    """Every instantiation of the rotations' inner product (1, 2, 4 and 8 digits per chunk) is in the sm_100a code and
    runs without local memory or stack."""
    usage = KS._cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*rotate64_inner\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    assert sorted(re.search(r"ILi(\d+)E", n).group(1) for n, *_ in found) == ["1", "2", "4", "8"]
    for name, reg, stack, local in found:
        assert int(local) == 0 and int(stack) == 0, name


# ------------------------------------------------------------------------------------------ on a GPU

dev, host, data, empty, rand_key, caller_roots = KS.dev, KS.host, KS.data, KS.empty, KS.rand_key, KS.caller_roots


@pytest.fixture(scope="module")
def A():
    import agilex_ntt_b200 as A
    return A


_CTX = {}


@pytest.fixture(scope="module")
def ctx(A):
    """Context64 per (N, primes, roots), kept for the module."""
    def get(N, primes, psis=None):
        key = (N, tuple(primes), tuple(psis) if psis else None)
        if key not in _CTX:
            _CTX[key] = A.Context64(N, primes, psi=psis)
        return _CTX[key]
    yield get
    for c in _CTX.values():
        c.close()
    _CTX.clear()


def elements(N, G):
    """G = 1: a rotation by one step; G = 3: g = 1, a rotation by -3 and the conjugation; G = 8: automorph's eight."""
    return {1: [AM.galois_element(N, 1)], 3: [1, AM.galois_element(N, -3), 2 * N - 1]}.get(G) or AM.eight_elements(N)


def ciphertexts(B, qs, N, seed):
    return data(2 * B, qs, N, seed).reshape(2, B, len(qs), N)


def plain(ctx, c, ct, gs, rks, alpha, k, form, psis=None):
    """The definition from public calls: automorph of (c0, c1), keyswitch of sigma(c1) with key t, add sigma(c0)."""
    B, ell1, N = ct.shape[1], ct.shape[2], ct.shape[3]
    cq = ctx(N, c.primes[:ell1], psis[:ell1] if psis else None)
    out = empty(len(gs), 2, B, ell1, N)
    for t, g in enumerate(gs):
        r = empty(2, B, ell1, N)
        cq.automorph(r.view(2 * B, ell1, N), ct.reshape(2 * B, ell1, N), g, ntt_form=form)
        c.keyswitch(out[t], r[1], rks[t], alpha, k, ntt_form=form)
        cq.elementwise("add", out[t, 0], out[t, 0], r[0])
    return out


def call(c, ct, gs, rks, alpha, k, form, stream=None):
    out = empty(len(gs), 2, ct.shape[1], ct.shape[2], c.n)
    return c.rotate(out, ct, gs, rks, alpha, k, ntt_form=form, stream=stream)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_vs_plain_recipe(ctx, N, form):
    """Three digits (2, 2 and 1 primes), k = 2, keys with two extra rows, G = 1, 3 and 8 (with g = 1 and 2n - 1)."""
    import torch
    primes = QS + PS
    c = ctx(N, primes)
    key_primes = QS + [PRIMES[50][10], PRIMES[50][11]] + PS
    ct = dev(ciphertexts(2, QS, N, 3 + N))
    for G in (1, 3, 8):
        gs = elements(N, G)
        rks = [dev(rand_key(3, key_primes, N, 100 * t + N)) for t in range(G)]
        got = call(c, ct, gs, rks, 2, 2, form)
        torch.cuda.synchronize()
        assert torch.equal(got, plain(ctx, c, ct, gs, rks, 2, 2, form)), G


@gpu
@pytest.mark.parametrize("N", (16,))
def test_vs_oracle(ctx, N):
    """Coefficient form at small n against the big-integer oracle, evaluation form against its transform."""
    qs, ps, alpha, k = QS, PS, 2, 2
    primes = qs + ps
    c = ctx(N, primes)
    rng = random.Random(N)
    gs = elements(N, 3)
    kcs = [np.stack([KS.rand_res(2, primes, N, rng) for _ in range(3)]) for _ in gs]
    rks = [dev(KS.rns_fwd(kc, primes)) for kc in kcs]
    ct = ciphertexts(2, qs, N, 17)
    want = rotate_oracle(ct, gs, kcs, primes, k, alpha)
    assert (host(call(c, dev(ct), gs, rks, alpha, k, False)) == want).all()
    got = call(c, dev(KS.rns_fwd(ct, qs)), gs, rks, alpha, k, True)
    assert (host(got) == KS.rns_fwd(want, qs)).all()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 32768))
def test_caller_roots(ctx, N):
    import torch
    primes = QS + PS
    psis = caller_roots(N, primes)
    c = ctx(N, primes, psis)
    gs = elements(N, 3)
    rks = [dev(rand_key(3, primes, N, 21 + N + t)) for t in range(3)]
    ct = dev(ciphertexts(2, QS, N, 23 + N))
    for form in (False, True):
        got = call(c, ct, gs, rks, 2, 2, form)
        torch.cuda.synchronize()
        assert torch.equal(got, plain(ctx, c, ct, gs, rks, 2, 2, form, psis)), form


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (32, 4096))
@pytest.mark.parametrize("shape", ("alpha1_dnum17", "one_digit", "alpha_above", "partial_last", "k1"))
def test_digit_shapes(ctx, N, form, shape):
    """alpha = 1 with l + 1 = 17 (17 digits: the lazy sums fold, the c0 term in the first chunk only), one digit,
    alpha > l + 1, a partial last digit (5 = 3 + 2), and k = 1 (the ModDown is the rescale)."""
    import torch
    qs, ps, alpha = {"alpha1_dnum17": (Q17, P17, 1), "one_digit": (QS, PS, 5), "alpha_above": (QS, PS, 40),
                     "partial_last": (QS, PS, 3), "k1": (QS, PS[:1], 2)}[shape]
    primes = qs + ps
    c = ctx(N, primes)
    dnum = len(KS.digits_of(len(qs), alpha))
    gs = elements(N, 3)
    rks = [dev(rand_key(dnum, primes, N, 31 + N + t)) for t in range(3)]
    ct = dev(ciphertexts(3, qs, N, 37 + N))
    got = call(c, ct, gs, rks, alpha, len(ps), form)
    torch.cuda.synchronize()
    assert torch.equal(got, plain(ctx, c, ct, gs, rks, alpha, len(ps), form))


@gpu
def test_one_key_set_at_three_levels(ctx):
    """One key set over Q_top u P (key_limbs = 7 + 2), alpha = 3, used unchanged at l + 1 = 7, 5 and 2."""
    import torch
    N = 1024
    qtop = QS + [PRIMES[62][3], PRIMES[50][3]]
    key_primes = qtop + PS
    gs = elements(N, 3)
    rks = [dev(rand_key(3, key_primes, N, 41 + t)) for t in range(3)]
    for ell1 in (7, 5, 2):
        qs = qtop[:ell1]
        c = ctx(N, qs + PS)
        ct = dev(ciphertexts(2, qs, N, 43 + ell1))
        for form in (False, True):
            got = call(c, ct, gs, rks, 3, 2, form)
            torch.cuda.synchronize()
            assert torch.equal(got, plain(ctx, c, ct, gs, rks, 3, 2, form)), (ell1, form)


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_element_and_key_variety(ctx, form):
    """G = 64 elements with 64 distinct keys, and two elements sharing one key tensor."""
    import torch
    N = 1024
    primes = QS + PS
    c = ctx(N, primes)
    ct = dev(ciphertexts(2, QS, N, 47))
    gs = [AM.galois_element(N, r) for r in range(-31, 32)] + [2 * N - 1]
    assert len(set(gs)) == 64
    rks = [dev(rand_key(3, primes, N, 500 + t)) for t in range(64)]
    got = call(c, ct, gs, rks, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(got, plain(ctx, c, ct, gs, rks, 2, 2, form))
    shared = [rks[0], rks[0], rks[1]]
    gs3 = elements(N, 3)
    got = call(c, ct, gs3, shared, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(got, plain(ctx, c, ct, gs3, shared, 2, 2, form))


@gpu
@pytest.mark.parametrize("N", (512, 16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """More polynomials than two waves of every transform geometry and than one slice of the inner product."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = -(-(2 * sms + 5) // len(QS))
    c = ctx(N, QS + PS)
    gs = elements(N, 3)
    rks = [dev(rand_key(3, QS + PS, N, 61 + t)) for t in range(3)]
    ct = dev(ciphertexts(B, QS, N, 67 + N))
    for form in (False, True):
        got = call(c, ct, gs, rks, 2, 2, form)
        assert torch.equal(got, plain(ctx, c, ct, gs, rks, 2, 2, form)), form
        del got
        torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_batch_is_single_calls(ctx, form):
    import torch
    N = 2048
    c = ctx(N, QS + PS)
    gs = elements(N, 8)
    rks = [dev(rand_key(3, QS + PS, N, 71 + t)) for t in range(8)]
    ct = dev(ciphertexts(5, QS, N, 73))
    got = call(c, ct, gs, rks, 2, 2, form)
    for b in range(5):
        one = call(c, ct[:, b:b + 1].contiguous(), gs, rks, 2, 2, form)
        torch.cuda.synchronize()
        assert torch.equal(got[:, :, b:b + 1], one), b


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_rotation_end_to_end(A, ctx, form):
    """Encrypt m under s, rotate by 1 and -3 steps and conjugate in one call with gadget keys for sigma_g(s), and decrypt
    each output under s to sigma_g(m) within the key switch's bound plus |e|."""
    import torch
    N = 1024
    qs, alpha, k = QS, 3, len(PS)
    Q = prod(qs)
    gs = [A.galois_element(N, 1), A.galois_element(N, -3), 2 * N - 1]
    rng = random.Random(83)
    s = KS.ternary(rng, N)
    ebound = 8
    key_primes = qs + PS
    ctop = ctx(N, key_primes)
    rks = [KS.gadget_key_gpu(ctop, key_primes, k, alpha, len(qs), s, AM.automorph_ints(s, g), ebound, rng) for g in gs]
    cq = ctx(N, qs)
    m, e = KS.small(rng, N, 1000), KS.small(rng, N, ebound)
    res = lambda v: dev(np.array([[x % q for x in v] for q in qs], dtype=np.uint64).reshape(1, len(qs), N))
    a = dev(data(1, qs, N, 89))
    c0 = empty(1, len(qs), N)
    cq.polymul(c0, a, res(s))
    cq.elementwise("sub", c0, res([x + y for x, y in zip(m, e)]), c0)
    ct = torch.stack([c0, a]).contiguous()
    if form:
        cq.fwd(ct.view(2, len(qs), N))
    out = call(ctx(N, key_primes), ct, gs, rks, alpha, k, form)
    if form:
        cq.inv(out.view(2 * len(gs), len(qs), N))
    got = host(out)
    bound = KS.ks_bound(qs, PS, alpha, N, ebound) + ebound
    assert bound < Q >> 40
    for t, g in enumerate(gs):
        c0v = [KS.crt(got[t, 0, 0, :, x], qs) for x in range(N)]
        c1v = [KS.crt(got[t, 1, 0, :, x], qs) for x in range(N)]
        r = [(u + v - w) % Q for u, v, w in zip(c0v, KS.negacyclic(c1v, s), AM.automorph_ints(m, g))]
        assert max(min(v, Q - v) for v in r) <= bound, g


def _u32(*gs):
    return (C.c_uint32 * max(len(gs), 1))(*gs)


def _ptrs(*ps):
    return (C.c_void_p * max(len(ps), 1))(*ps)


@gpu
def test_refusals_and_empty_calls(A, ctx):
    import torch
    N = 1024
    lib = A.lib()
    primes = QS + PS
    L, ell1 = len(primes), len(QS)
    c, c19 = ctx(N, primes), ctx(N, Q17 + P17)
    x = dev(ciphertexts(2, QS, N, 3))
    rk0, rk1 = dev(rand_key(3, primes, N, 4)), dev(rand_key(3, primes, N, 5))
    xs, k0s, k1s = x.clone(), rk0.clone(), rk1.clone()
    o = empty(2, 2, 2, ell1, N)
    pi, po, p0, p1 = x.data_ptr(), o.data_ptr(), rk0.data_ptr(), rk1.data_ptr()
    big = torch.zeros(40 * L * N, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    dup = A.Context64(N, [QS[0], QS[1], QS[0], PS[0]])
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    ctxs = (c, c19, dup)
    g2, r2 = _u32(3, 5), _ptrs(p0, p1)
    kw = 3 * 2 * L * N                                                         # words read from each key
    cw = 2 * 2 * ell1 * N                                                      # words of the two ciphertexts
    try:
        for form in (0, 1):
            invalid = [
                (c32._h, po, pi, 2, g2, 2, r2, L, 2, 2),                               # u32 context
                (c._h, None, pi, 2, g2, 2, r2, L, 2, 2), (c._h, po, None, 2, g2, 2, r2, L, 2, 2),
                (c._h, po, pi, 2, None, 2, r2, L, 2, 2), (c._h, po, pi, 2, g2, 2, None, L, 2, 2),
                (c._h, po, pi, 2, g2, 2, _ptrs(p0, None), L, 2, 2),                     # null key with B > 0
                (c._h, po + 8, pi, 1, g2, 2, r2, L, 2, 2), (c._h, po, pi + 8, 1, g2, 2, r2, L, 2, 2),
                (c._h, po, pi, 1, g2, 2, _ptrs(p0, p1 + 8), L, 2, 2),                   # misaligned key
                (c._h, po, pi, 2, g2, 2, r2, L, 2, 0), (c._h, po, pi, 2, g2, 2, r2, L, 2, L),   # k = 0, k = L
                (c._h, po, pi, 2, g2, 2, r2, L, 0, 2),                                 # alpha = 0
                (c._h, po, pi, 2, g2, 2, r2, L - 1, 2, 2),                             # key_limbs < L
                (dup._h, po, pi, 2, g2, 2, r2, 4, 1, 1),                               # two equal primes
                (c._h, po, pi, 2, _u32(3, 4), 2, r2, L, 2, 2), (c._h, po, pi, 2, _u32(0, 3), 2, r2, L, 2, 2),
                (c._h, po, pi, 2, _u32(3, 2 * N), 2, r2, L, 2, 2), (c._h, po, pi, 2, _u32(0xffffffff, 3), 2, r2, L, 2, 2),
                (c._h, po, pi, 0x7fffffff // (4 * L) + 1, g2, 2, r2, L, 9, 2),         # 2 G B L > 2^31 - 1 (dnum = 1)
                (c._h, po, pi, 0x7fffffff // (5 * L) + 1, _u32(3), 1, _ptrs(p0), L, 1, 2),   # dnum B L > 2^31 - 1
                (c._h, pi, pi, 2, g2, 2, r2, L, 2, 2),                                 # out on in
                (c._h, bp + 8 * (cw - 2), bp, 2, g2, 2, r2, L, 2, 2),                  # in's last 16 bytes are out's first
                (c._h, bp, bp + 8 * (2 * cw - 2), 2, g2, 2, r2, L, 2, 2),              # out's last 16 bytes are in's first
                (c._h, bp + 8 * (kw - 2), pi, 2, g2, 2, _ptrs(p0, bp), L, 2, 2),       # out starts in key 1's last digit
                (c._h, bp, pi, 2, g2, 2, _ptrs(bp + 8 * (2 * cw - 2), p1), L, 2, 2),   # key 0 starts in out
            ]
            for h, o_, i_, B, gp, G, rp, kl, al, kk in invalid:
                l0 = [t.launch_count() for t in ctxs]
                assert lib.agx_rotate64(h, o_, i_, B, gp, G, rp, kl, al, kk, form, None) == -1, (form, B, G, kl, al, kk)
                assert [t.launch_count() for t in ctxs] == l0
            l0 = c.launch_count()
            g65 = _u32(*([2] * 65))                                                # even: refused if they were read
            assert lib.agx_rotate64(c._h, bp + 8 * 2 * kw, pi, 2, g65, 65, _ptrs(*([None] * 65)), L, 2, 2, form, None) == -2
            for al, kk in ((17, 2), (16, 17)):                                     # 17 digit primes; k = 17
                l19 = c19.launch_count()
                assert lib.agx_rotate64(c19._h, bp, bp + 8 * 40 * N, 1, _u32(3), 1, _ptrs(p0), 19, al, kk, form,
                                        None) == -2, (al, kk)
                assert c19.launch_count() == l19
            for o_, i_, rp in ((None, None, _ptrs(None, None)), (po, pi, r2), (bp, bp + 16, _ptrs(bp, bp))):   # B == 0
                assert lib.agx_rotate64(c._h, o_, i_, 0, g2, 2, rp, L, 2, 2, form, None) == 0
            assert lib.agx_rotate64(c._h, po, pi, 2, None, 0, None, L, 2, 2, form, None) == 0             # G == 0
            assert lib.agx_rotate64(c._h, pi, pi, 2, None, 0, None, L, 2, 2, form, None) == 0
            assert c.launch_count() == l0
            # adjacent, not overlapping: allowed; a key digit that is not read may overlap
            assert lib.agx_rotate64(c._h, bp + 8 * kw, pi, 2, g2, 2, _ptrs(bp, bp), L, 2, 2, form, None) == 0
            assert lib.agx_rotate64(c._h, bp + 8 * 2 * L * N, pi, 2, g2, 2, _ptrs(bp, p1), L, 9, 2, form, None) == 0
        bad = [
            lambda: c.rotate(empty(2, 2, 1, ell1, N), x, [3, 5], [rk0, rk1], 2, 2),          # out batch
            lambda: c.rotate(empty(2, 2, 2, ell1, N), x, 3, [rk0], 2, 2),                     # one element, G outputs
            lambda: c.rotate(empty(2, 2, ell1, N), x, [3], [rk0], 2, 2),                      # a sequence, no G axis
            lambda: c.rotate(o, x, [3, 5], [rk0], 2, 2),                                      # fewer keys than elements
            lambda: c.rotate(o, x, [3, 5], [rk0, rk1[:2]], 2, 2),                             # fewer key digits
            lambda: c.rotate(o, x, [3, 5], [rk0, rk1[:, :, :L - 1].contiguous()], 2, 2),      # key_limbs < L
            lambda: c.rotate(o, x, [3, 5], [rk0, torch.cat([rk1, rk1], 2)], 2, 2),             # unequal key_limbs
            lambda: c.rotate(o, x[0], [3, 5], [rk0, rk1], 2, 2),                              # not a ciphertext
            lambda: c.rotate(o, x, [3, 5], [rk0, rk1], 0, 2),                                 # alpha = 0
            lambda: c.rotate(o, x, [3, 5], [rk0, rk1], 2, 0),                                 # k = 0
            lambda: c.rotate(o, x.cpu(), [3, 5], [rk0, rk1], 2, 2),                           # host tensor
            lambda: c.rotate(o, x, [3, 5], [rk0, rk1.cpu()], 2, 2),
            lambda: c.rotate(o, x, [3, 2**32 + 5], [rk0, rk1], 2, 2),                         # not 32-bit
            lambda: c.rotate(o, x, [-1, 5], [rk0, rk1], 2, 2),
        ]
        for fn in bad:
            with pytest.raises(ValueError):
                fn()
        with pytest.raises(A.AgxError) as e:
            c.rotate(o, x, [3, 4], [rk0, rk1], 2, 2)                                          # even element
        assert e.value.code == -1
        torch.cuda.synchronize()
        assert torch.equal(x, xs) and torch.equal(rk0, k0s) and torch.equal(rk1, k1s)
    finally:
        for t in (dup, c32):
            t.close()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_inputs_unchanged(ctx, form):
    import torch
    N = 4096
    c = ctx(N, QS + PS)
    gs = elements(N, 3)
    rks = [dev(rand_key(3, QS + PS, N, 91 + t)) for t in range(3)]
    ct = dev(ciphertexts(4, QS, N, 93))
    snap, ksnap = ct.clone(), [r.clone() for r in rks]
    call(c, ct, gs, rks, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(ct, snap) and all(torch.equal(r, s) for r, s in zip(rks, ksnap))


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    """The header's counts, the same for G = 1 and G = 8."""
    import torch
    x = int(N == 32768)
    c, c1 = ctx(N, QS + PS), ctx(N, QS + PS[:1])
    ct = dev(ciphertexts(2, QS, N, 99))
    key = dev(rand_key(5, QS + PS, N, 97))

    def launches(cx, G, alpha, k, form, rk=key):
        l0 = cx.launch_count()
        call(cx, ct, elements(N, G), [rk] * G, alpha, k, form)
        torch.cuda.synchronize()
        return cx.launch_count() - l0

    k1 = key[:, :, :len(QS) + 1].contiguous()
    for G in (1, 8):
        # alpha = 2: digits of 2, 2 and 1 primes (ModUps 3 + 3 + 2, one more each at N = 32768); inner 1; ModDown 3 (4)
        assert launches(c, G, 2, 2, True) == 8 + 3 * x + 1 + 3 + x
        assert launches(c, G, 2, 2, False) == 3 + 5 + x                      # dnum + 5
        # alpha = 5: one digit: 3 * dnum + 4 (4 * dnum + 5 at N = 32768)
        assert launches(c, G, 5, 2, True) == 7 + 2 * x
        assert launches(c, G, 5, 2, False) == 6 + x
        # k = 1: the ModDown is the rescale (2; 3 at N = 32768)
        assert launches(c1, G, 5, 1, True, k1) == 3 + x + 1 + 2 + x
        assert launches(c1, G, 5, 1, False, k1) == 6 + x


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    c = ctx(N, QS + PS)
    gs = elements(N, 8)
    keys = [rand_key(3, QS + PS, N, 101 + t) for t in range(8)]
    x = ciphertexts(4, QS, N, 103)
    want = plain(ctx, c, dev(x), gs, [dev(k) for k in keys], 2, 2, form)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_x = dev(x)
        ct = torch.empty_like(d_x)
        ct.copy_(d_x)                                                   # torch work the call must follow
        rks = []
        for k in keys:
            d_k = dev(k)
            rk = torch.empty_like(d_k)
            rk.copy_(d_k)
            rks.append(rk)
        out = empty(8, 2, 4, len(QS), N)
    c.rotate(out, ct, gs, rks, 2, 2, ntt_form=form, stream=s)
    s.synchronize()
    assert torch.equal(out, want)
