"""u64 RNS hoisted linear transforms in one call (agx_lintrans64, Context64.lintrans).

Definition, for a context over Q_l u P (the k special primes last), ciphertexts ct = (c0, c1) over Q_l, G Galois
elements with keys in agx_rotate64's layout (key t switching sigma_t(s) to s, or none for g = 1) and M x G diagonals
d_{m,t} over Q_l u P (or none, a zero diagonal):
    A_t[c]    = sum_j sigma_t(ModUp_j(digit_j(c1))) (.) rk_t[j][c] + [c = 0] P sigma_t(c0)
    A_t       = (P c0, P c1)                                    for a keyless g = 1
    out[m][c] = ModDown_P( sum_t d_{m,t} (.) A_t[c] ).
By the fold identity (test_u64_rotate.py) that is sum_t d_{m,t} sigma_t(c0) + ModDown(sum_t d_{m,t} KS_t): one
rounding per output where summing agx_rotate64's outputs rounds G times.

The CPU tests pin a big-integer oracle of the definition, check that with identity diagonals it is rotate_oracle and that
the keyless identity term returns the input, that it decrypts within the double-hoisting bound, and the new kernels'
resources.  The GPU tests compare the call with the recipe composed from public calls bit for bit in both forms, cover
digit shapes, term and output counts, NULL and shared pointers, check the identity cases against agx_rotate64 and the
input, run a 2 x 4 baby-step/giant-step product end to end, and cover refusals, launch counts, unchanged inputs and
side-stream ordering."""
import ctypes as C
import random
import re
from math import prod

import numpy as np
import pytest

import test_u64_automorph as AM
import test_u64_keyswitch as KS
import test_u64_rotate as RT
from oracle import oracle as O

gpu = pytest.mark.gpu
SIZES = KS.SIZES
PRIMES, QS, PS, Q17, P17 = KS.PRIMES, KS.QS, KS.PS, KS.Q17, KS.P17


# ---- big ints: the oracle
def lintrans_oracle(ct, gs, kcoefs, dcoefs, primes, k, alpha):
    """ct [2][B][l+1][N] in coefficient form over primes[:l+1]; kcoefs[t] key t in coefficient form (as
    keyswitch_oracle takes it) or None (g = 1, no key); dcoefs[m][t] the diagonal [L][N] in coefficient form over all
    primes, or None -> [M][2][B][l+1][N].  Centred digit lifts, sigma_t on the integers, negacyclic products with the
    keys mod QP, plus P sigma_t(c0), times d_{m,t}, summed, then floor((X + h_P) / P) mod Q."""
    L = len(primes)
    ell1 = L - k
    qs = primes[:ell1]
    Q, P, QP = prod(qs), prod(primes[ell1:]), prod(primes)
    hP = (P - 1) // 2
    _, B, _, N = ct.shape
    digits = KS.digits_of(ell1, alpha)
    keys = []
    for kc in kcoefs:
        if kc is None:
            keys.append(None)
            continue
        rows = KS.key_rows(L, k, kc.shape[2])
        keys.append([[[KS.crt([kc[j, c, rows[i], x] for i in range(L)], primes) for x in range(N)] for c in (0, 1)]
                     for j in range(len(digits))])
    D = [[None if d is None else [KS.crt(d[:, x], primes) for x in range(N)] for d in row] for row in dcoefs]
    out = np.empty((len(dcoefs), 2, B, ell1, N), dtype=np.uint64)
    for b in range(B):
        C0 = [KS.crt(ct[0, b, :, x], qs) for x in range(N)]
        C1 = [KS.crt(ct[1, b, :, x], qs) for x in range(N)]
        Us = []
        for f, cnt in digits:
            src = primes[f:f + cnt]
            S = prod(src)
            Us.append([(KS.crt(ct[1, b, f:f + cnt, x], src) + (S - 1) // 2) % S - (S - 1) // 2 for x in range(N)])
        A = []
        for g, key in zip(gs, keys):
            if key is None:
                assert g == 1
                A.append([[P * v % QP for v in C0], [P * v % QP for v in C1]])
                continue
            acc = [[0] * N, [0] * N]
            for j, U in enumerate(Us):
                sU = AM.automorph_ints(U, g)
                for c in (0, 1):
                    acc[c] = [(u + v) % QP for u, v in zip(acc[c], KS.negacyclic(sU, key[j][c]))]
            acc[0] = [(X + P * v) % QP for X, v in zip(acc[0], AM.automorph_ints(C0, g))]
            A.append(acc)
        for m, row in enumerate(D):
            for c in (0, 1):
                X = [0] * N
                for d, At in zip(row, A):
                    if d is not None:
                        X = [(u + v) % QP for u, v in zip(X, KS.negacyclic(d, At[c]))]
                Y = [((x + hP) // P) % Q for x in X]
                for i, q in enumerate(qs):
                    out[m, c, b, i] = [y % q for y in Y]
    return out


def residues(v, primes):
    """[L][N] residues of integer coefficients v"""
    return np.array([[x % q for x in v] for q in primes], dtype=np.uint64)


def lintrans_bound(ks_bound, N, dnorms):
    """The double-hoisting decryption bound of one output: sum_t N |d_t| (ks_bound - (N+1)/2) + (N+1)/2."""
    return sum(N * dn * (ks_bound - (N + 1) // 2) for dn in dnorms) + (N + 1) // 2


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("N,qs,ps,alpha", [(8, QS[:3], PS, 1), (16, QS, PS, 2), (32, QS[:4], PS[:1], 3)])
def test_oracle_identity_diagonals_are_rotations(N, qs, ps, alpha):
    """M = G with d_{m,t} = 1 iff m == t (None otherwise) is rotate_oracle, word for word; G = M = 1 with g = 1, no key
    and d = 1 returns the input."""
    rng = random.Random(N * 5 + alpha)
    primes, k = qs + ps, len(ps)
    gs = [1, AM.galois_element(N, 1), 2 * N - 1]
    kcs = [np.stack([KS.rand_res(2, primes, N, rng) for _ in KS.digits_of(len(qs), alpha)]) for _ in gs]
    ct = np.stack([KS.rand_res(2, qs, N, rng) for _ in (0, 1)])
    one = residues([1] + [0] * (N - 1), primes)
    diags = [[one if m == t else None for t in range(len(gs))] for m in range(len(gs))]
    assert (lintrans_oracle(ct, gs, kcs, diags, primes, k, alpha) == RT.rotate_oracle(ct, gs, kcs, primes, k, alpha)).all()
    assert (lintrans_oracle(ct, [1], [None], [[one]], primes, k, alpha)[0] == ct).all()


@pytest.mark.parametrize("N,qs,ps,alpha", [(8, QS[:3], PS, 1), (16, QS, PS, 2), (32, QS[:4], PS[:1], 3)])
def test_oracle_decrypts_within_the_double_hoisting_bound(N, qs, ps, alpha):
    """With gadget keys for sigma_t(s) (t = 0 keyless, g = 1) and diagonals of small coefficients, out[m] decrypts under
    s to sum_t d_{m,t} sigma_t(mu), mu = c0 + c1 s the input's phase, with error at most
        sum_t N |d_{m,t}| (ks_bound - (N+1)/2) + (N+1)/2.
    Derivation: A_t[0] + A_t[1] s = P sigma_t(mu) + E_t (mod QP), with |E_t| <= N |e| sum_j D_j / 2 < P (ks_bound -
    (N+1)/2) the gadget sum's error (E_t = 0 for the keyless term).  So X_0 + X_1 s = P sum_t d_t sigma_t(mu) +
    sum_t d_t E_t, and |d_t E_t| <= N |d_t| |E_t|.  ModDown divides by P and rounds each of X_0, X_1 once: that adds
    e_0 + e_1 s with |e_c| <= 1/2, at most (N+1)/2 for ternary s.  Single hoisting pays that rounding once per term."""
    rng = random.Random(N * 11 + alpha)
    primes, k = qs + ps, len(ps)
    Q = prod(qs)
    gs = [1, AM.galois_element(N, 1), AM.galois_element(N, -2), 2 * N - 1]
    s = KS.ternary(rng, N)
    ebound = 6
    kcs = [None] + [KS.gadget_key_coeff(primes, k, alpha, len(qs), s, AM.automorph_ints(s, g), ebound, rng)
                    for g in gs[1:]]
    dints = [[KS.small(rng, N, 3) for _ in gs], [KS.small(rng, N, 2) if t % 2 else None for t in range(len(gs))]]
    diags = [[None if d is None else residues(d, primes) for d in row] for row in dints]
    ct = np.stack([KS.rand_res(1, qs, N, rng) for _ in (0, 1)])
    out = lintrans_oracle(ct, gs, kcs, diags, primes, k, alpha)
    mu = [(KS.crt(ct[0, 0, :, x], qs) + v) % Q for x, v in enumerate(KS.negacyclic([KS.crt(ct[1, 0, :, x], qs)
                                                                                       for x in range(N)], s))]
    ksb = KS.ks_bound(qs, ps, alpha, N, ebound)
    for m, row in enumerate(dints):
        want = [0] * N
        for d, g in zip(row, gs):
            if d is not None:
                want = [u + v for u, v in zip(want, KS.negacyclic(d, AM.automorph_ints(mu, g)))]
        c0 = [KS.crt(out[m, 0, 0, :, x], qs) for x in range(N)]
        c1 = [KS.crt(out[m, 1, 0, :, x], qs) for x in range(N)]
        r = [(u + v - w) % Q for u, v, w in zip(c0, KS.negacyclic(c1, s), want)]
        bound = lintrans_bound(ksb, N, [max(map(abs, d)) for d in row if d is not None])
        assert bound < Q >> 40
        assert max(min(v, Q - v) for v in r) <= bound, m


def test_lintrans_kernels_use_no_local_memory():
    """Every instantiation of the linear transform's inner sums (1, 2, 4 and 8 digits per chunk, for up to 4 and up to
    16 outputs) is in the sm_100a code and runs without local memory or stack."""
    usage = KS._cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*lintrans64_inner\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    got = sorted(re.search(r"ILi(\d+)ELi(\d+)E", n).groups() for n, *_ in found)
    assert got == sorted((dc, mc) for dc in ("1", "2", "4", "8") for mc in ("4", "16"))
    for name, reg, stack, local in found:
        assert int(local) == 0 and int(stack) == 0, name


# ------------------------------------------------------------------------------------------ on a GPU

dev, host, data, empty, rand_key, caller_roots = KS.dev, KS.host, KS.data, KS.empty, KS.rand_key, KS.caller_roots
ciphertexts, elements = RT.ciphertexts, RT.elements


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


def recipe(ctx, c, ct, gs, rks, diags, alpha, k, form, psis=None):
    """The definition from public calls, in evaluation form: modup of each digit of c1, automorph of the extended digits
    over Q_l u P and of c0 over Q_l, elementwise mul / mac with the key rows sliced by the row map and replicated over
    B, the P sigma(c0) fold as a mac with (P mod q_i) rows zero on P, mac with the diagonals replicated over B, then one
    moddown of 2 M B.  Coefficient form: the same between a forward and an inverse over Q_l."""
    import torch
    L, N, B = c.L, c.n, ct.shape[1]
    ell1 = L - k
    cq = ctx(N, c.primes[:ell1], psis[:ell1] if psis else None)
    if not form:
        ct = ct.clone()
        cq.fwd(ct.view(2 * B, ell1, N))
    P = prod(c.primes[ell1:])
    pm = dev(np.array([[P % q if i < ell1 else 0] * N for i, q in enumerate(c.primes)], dtype=np.uint64))
    pm = pm.expand(B, L, N).contiguous()
    pad = lambda x: torch.cat([x, torch.zeros(B, k, N, dtype=x.dtype, device=x.device)], 1)
    Us = []
    for f, cnt in KS.digits_of(ell1, alpha):
        U = empty(B, L, N)
        c.modup(U, ct[1, :, f:f + cnt].contiguous(), f, cnt, ntt_form=True)
        Us.append(U)
    M = len(diags)
    acc = torch.zeros(M, 2, B, L, N, dtype=torch.int64, device="cuda")
    for t, (g, rk) in enumerate(zip(gs, rks)):
        At = [empty(B, L, N), empty(B, L, N)]
        if rk is None:
            for cc in (0, 1):
                c.elementwise("mul", At[cc], pad(ct[cc]), pm)
        else:
            kr = torch.cat([rk[:, :, :ell1], rk[:, :, rk.shape[2] - k:]], dim=2)
            for j, U in enumerate(Us):
                sU = empty(B, L, N)
                c.automorph(sU, U, g)
                for cc in (0, 1):
                    c.elementwise("mul" if j == 0 else "mac", At[cc], sU, kr[j, cc].expand(B, L, N).contiguous())
            s0 = empty(B, ell1, N)
            cq.automorph(s0, ct[0], g)
            c.elementwise("mac", At[0], pad(s0), pm)
        for m, row in enumerate(diags):
            if row[t] is not None:
                dd = row[t].expand(B, L, N).contiguous()
                for cc in (0, 1):
                    c.elementwise("mac", acc[m, cc], At[cc], dd)
    out = empty(M, 2, B, ell1, N)
    c.moddown(out.view(2 * M * B, ell1, N), acc.view(2 * M * B, L, N), k)
    if not form:
        cq.inv(out.view(2 * M * B, ell1, N))
    return out


def call(c, ct, gs, rks, diags, alpha, k, form, stream=None):
    out = empty(len(diags), 2, ct.shape[1], ct.shape[2], c.n)
    return c.lintrans(out, ct, gs, rks, diags, alpha, k, ntt_form=form, stream=stream)


def rand_diag(primes, N, seed):
    return dev(data(1, primes, N, seed)[0])


def check(ctx, c, ct, gs, rks, diags, alpha, k, form, psis=None):
    import torch
    got = call(c, ct, gs, rks, diags, alpha, k, form)
    torch.cuda.synchronize()
    assert torch.equal(got, recipe(ctx, c, ct, gs, rks, diags, alpha, k, form, psis))


def pattern(N, primes, G, M, seed):
    """M x G diagonals: distinct random ones, a NULL, a pointer shared between two entries, and an all-NULL last row
    when M > 1."""
    diags = [[rand_diag(primes, N, seed + 37 * m + t) for t in range(G)] for m in range(M)]
    if G > 1:
        diags[0][1] = None
    if M > 1:
        diags[-1] = [None] * G
        diags[0][0] = diags[M - 2][G - 1]
    return diags


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_vs_composed_recipe(ctx, N, form):
    """Three digits (2, 2 and 1 primes), k = 2, keys with two extra rows; G = 3 (g = 1 keyless, a rotation by -3 and the
    conjugation) with M = 4, and G = 8 (g = 1 with a key) with M = 1."""
    primes = QS + PS
    c = ctx(N, primes)
    key_primes = QS + [PRIMES[50][10], PRIMES[50][11]] + PS
    ct = dev(ciphertexts(2, QS, N, 3 + N))
    gs = elements(N, 3)
    rks = [None] + [dev(rand_key(3, key_primes, N, 100 * t + N)) for t in (1, 2)]
    check(ctx, c, ct, gs, rks, pattern(N, primes, 3, 4, N), 2, 2, form)
    gs = elements(N, 8)
    rks = [dev(rand_key(3, key_primes, N, 200 * t + N)) for t in range(8)]
    check(ctx, c, ct, gs, rks, pattern(N, primes, 8, 1, 7 * N), 2, 2, form)


@gpu
def test_vs_oracle(ctx):
    """Coefficient form at N = 16 against the big-integer oracle, evaluation form against its transform."""
    N, qs, ps, alpha, k = 16, QS, PS, 2, 2
    primes = qs + ps
    c = ctx(N, primes)
    rng = random.Random(N)
    gs = elements(N, 3)
    kcs = [None] + [np.stack([KS.rand_res(2, primes, N, rng) for _ in range(3)]) for _ in gs[1:]]
    rks = [None if kc is None else dev(KS.rns_fwd(kc, primes)) for kc in kcs]
    dcs = [[KS.rand_res(1, primes, N, rng)[0] for _ in gs] for _ in range(2)]
    dcs[1][0] = None
    diags = [[None if d is None else dev(KS.rns_fwd(d, primes)) for d in row] for row in dcs]
    ct = ciphertexts(2, qs, N, 17)
    want = lintrans_oracle(ct, gs, kcs, dcs, primes, k, alpha)
    assert (host(call(c, dev(ct), gs, rks, diags, alpha, k, False)) == want).all()
    got = call(c, dev(KS.rns_fwd(ct, qs)), gs, rks, diags, alpha, k, True)
    assert (host(got) == KS.rns_fwd(want, qs)).all()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 32768))
def test_caller_roots(ctx, N):
    primes = QS + PS
    psis = caller_roots(N, primes)
    c = ctx(N, primes, psis)
    gs = elements(N, 3)
    rks = [None] + [dev(rand_key(3, primes, N, 21 + N + t)) for t in (1, 2)]
    ct = dev(ciphertexts(2, QS, N, 23 + N))
    diags = pattern(N, primes, 3, 2, 5 * N)
    for form in (False, True):
        check(ctx, c, ct, gs, rks, diags, 2, 2, form, psis)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (32, 4096))
@pytest.mark.parametrize("shape", ("alpha1_dnum17", "one_digit", "partial_last", "k1"))
def test_digit_shapes(ctx, N, form, shape):
    """alpha = 1 with l + 1 = 17 (17 digits: A_t's lazy sum folds), one digit, a partial last digit (5 = 3 + 2), and
    k = 1 (the ModDown is the rescale)."""
    qs, ps, alpha = {"alpha1_dnum17": (Q17, P17, 1), "one_digit": (QS, PS, 5), "partial_last": (QS, PS, 3),
                     "k1": (QS, PS[:1], 2)}[shape]
    primes = qs + ps
    c = ctx(N, primes)
    dnum = len(KS.digits_of(len(qs), alpha))
    gs = elements(N, 3)
    rks = [None] + [dev(rand_key(dnum, primes, N, 31 + N + t)) for t in (1, 2)]
    ct = dev(ciphertexts(3, qs, N, 37 + N))
    check(ctx, c, ct, gs, rks, pattern(N, primes, 3, 2, 3 * N), alpha, len(ps), form)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("G,M", ((64, 4), (16, 16), (1, 16), (64, 1)))
def test_term_and_output_counts(ctx, form, G, M):
    """M * G = 256 with 64 distinct keys, and with 16 outputs (the larger instantiation) in a sparse layout; one term
    for 16 outputs; 64 terms for one.  Shared key pointers and a keyless g = 1 term in every case but G = 1."""
    N = 256
    primes = QS + PS
    c = ctx(N, primes)
    ct = dev(ciphertexts(2, QS, N, 47 + G))
    steps = range(-31, 32) if G == 64 else range(G)                       # step 0 is g = 1
    gs = [AM.galois_element(N, r) for r in steps] + ([2 * N - 1] if G == 64 else [])
    assert len(set(gs)) == G
    rks = [dev(rand_key(3, primes, N, 500 + t)) for t in range(G)]
    if G > 1:
        rks[gs.index(1)] = None
        rks[-1] = rks[-2]
    rng = random.Random(G * M)
    diags = [[rand_diag(primes, N, 900 + 64 * m + t) if rng.random() < (0.3 if M == 16 else 1.0) else None
              for t in range(G)] for m in range(M)]
    if M > 1:
        diags[1] = [None] * G
        diags[0][0] = diags[2][G - 1] = rand_diag(primes, N, 7)           # one tensor for two entries
    check(ctx, c, ct, gs, rks, diags, 2, 2, form)


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_identity_diagonals_are_rotate(A, ctx, form):
    """M = G with d_{m,t} = 1 iff m == t equals agx_rotate64's G outputs bit for bit; G = M = 1 with g = 1, no key and
    d = 1 returns d_in."""
    import torch
    N = 2048
    primes = QS + PS
    c = ctx(N, primes)
    gs = elements(N, 8)
    rks = [dev(rand_key(3, primes, N, 71 + t)) for t in range(8)]
    ct = dev(ciphertexts(3, QS, N, 73))
    ones = torch.ones(len(primes), N, dtype=torch.int64, device="cuda")
    diags = [[ones if m == t else None for t in range(8)] for m in range(8)]
    got = call(c, ct, gs, rks, diags, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(got, RT.call(c, ct, gs, rks, 2, 2, form))
    got = call(c, ct, [1], [None], [[ones]], 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(got[0], ct)


@gpu
@pytest.mark.parametrize("N", (512, 16384))
def test_batches_above_two_waves(ctx, N):
    """More polynomials than two waves of every transform geometry."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = -(-(2 * sms + 5) // len(QS))
    primes = QS + PS
    c = ctx(N, primes)
    gs = elements(N, 3)
    rks = [None] + [dev(rand_key(3, primes, N, 61 + t)) for t in (1, 2)]
    ct = dev(ciphertexts(B, QS, N, 67 + N))
    diags = pattern(N, primes, 3, 2, 11 * N)
    for form in (False, True):
        check(ctx, c, ct, gs, rks, diags, 2, 2, form)
        torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_bsgs_end_to_end(A, ctx, form):
    """A 2 x 4 baby-step/giant-step product: encrypt mu under s, one lintrans call with the baby steps sigma_{5^i},
    i = 0..3 (i = 0 keyless) and M = 2 giant-step inner sums y_j = sum_i d_{j,i} sigma_{5^i}(ct), then
    y_0 + rotate(y_1, 5^4).  It decrypts to sum_j sigma_{5^{4j}}(sum_i d_{j,i} sigma_{5^i}(mu)) within the double-hoisting
    bound of both sums plus one key switch."""
    import torch
    N = 256
    qs, alpha, k = QS, 3, len(PS)
    primes = qs + PS
    Q = prod(qs)
    baby = [A.galois_element(N, i) for i in range(4)]
    giant = A.galois_element(N, 4)
    rng = random.Random(97)
    s = KS.ternary(rng, N)
    ebound = 8
    c = ctx(N, primes)
    key = lambda g: KS.gadget_key_gpu(c, primes, k, alpha, len(qs), s, AM.automorph_ints(s, g), ebound, rng)
    rks = [None] + [key(g) for g in baby[1:]]
    rk_giant = key(giant)
    cq = ctx(N, qs)
    m, e = KS.small(rng, N, 1000), KS.small(rng, N, ebound)
    res = lambda v, ps: dev(residues(v, ps))
    a = dev(data(1, qs, N, 89))
    c0 = empty(1, len(qs), N)
    cq.polymul(c0, a, res(s, qs).view(1, len(qs), N))
    cq.elementwise("sub", c0, res([x + y for x, y in zip(m, e)], qs).view(1, len(qs), N), c0)
    ct = torch.stack([c0, a]).contiguous()
    dints = [[KS.small(rng, N, 3) for _ in baby] for _ in range(2)]
    diags = []
    for row in dints:
        diags.append([])
        for d in row:
            dd = res(d, primes)
            c.fwd(dd.view(1, len(primes), N))
            diags[-1].append(dd)
    if form:
        cq.fwd(ct.view(2, len(qs), N))
    y = call(c, ct, baby, rks, diags, alpha, k, form)
    r1 = empty(2, 1, len(qs), N)
    c.rotate(r1, y[1], giant, [rk_giant], alpha, k, ntt_form=form)
    cq.elementwise("add", y[0].view(2, len(qs), N), y[0].view(2, len(qs), N), r1.view(2, len(qs), N))
    if form:
        cq.inv(y[0].view(2, len(qs), N))
    got = host(y[0])
    mu = [x + v for x, v in zip(m, e)]
    want = [0] * N
    for j, row in enumerate(dints):
        inner = [0] * N
        for d, g in zip(row, baby):
            inner = [u + v for u, v in zip(inner, KS.negacyclic(d, AM.automorph_ints(mu, g)))]
        want = [u + v for u, v in zip(want, AM.automorph_ints(inner, pow(giant, j, 2 * N)))]
    ksb = KS.ks_bound(qs, PS, alpha, N, ebound)
    bound = sum(lintrans_bound(ksb, N, [max(map(abs, d)) for d in row]) for row in dints) + ksb
    assert bound < Q >> 40
    c0v = [KS.crt(got[0, 0, :, x], qs) for x in range(N)]
    c1v = [KS.crt(got[1, 0, :, x], qs) for x in range(N)]
    r = [(u + v - w) % Q for u, v, w in zip(c0v, KS.negacyclic(c1v, s), want)]
    assert max(min(v, Q - v) for v in r) <= bound


_u32, _ptrs = RT._u32, RT._ptrs


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
    d0, d1 = rand_diag(primes, N, 6), rand_diag(primes, N, 7)
    snaps = [t.clone() for t in (x, rk0, rk1, d0, d1)]
    o = torch.full((2, 2, 2, ell1, N), 12345, dtype=torch.int64, device="cuda")
    osnap = o.clone()
    pi, po, p0, p1, q0, q1 = x.data_ptr(), o.data_ptr(), rk0.data_ptr(), rk1.data_ptr(), d0.data_ptr(), d1.data_ptr()
    big = torch.zeros(40 * L * N, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    dup = A.Context64(N, [QS[0], QS[1], QS[0], PS[0]])
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    ctxs = (c, c19, dup)
    g2, r2, D = _u32(3, 5), _ptrs(p0, p1), _ptrs(q0, q1, None, q1)            # M = 2, G = 2
    kw = 3 * 2 * L * N                                                         # words read from each key
    cw = 2 * 2 * ell1 * N                                                      # words of the two ciphertexts
    ow = 2 * cw                                                                # words of the two outputs
    try:
        for form in (0, 1):
            invalid = [
                (c32._h, po, pi, 2, g2, 2, r2, L, D, 2, 2, 2),                          # u32 context
                (c._h, None, pi, 2, g2, 2, r2, L, D, 2, 2, 2), (c._h, po, None, 2, g2, 2, r2, L, D, 2, 2, 2),
                (c._h, po, pi, 2, None, 2, r2, L, D, 2, 2, 2), (c._h, po, pi, 2, g2, 2, None, L, D, 2, 2, 2),
                (c._h, po, pi, 2, g2, 2, r2, L, None, 2, 2, 2),                         # null diagonal array
                (c._h, po, pi, 2, None, 0, None, L, D, 2, 2, 2),                        # G == 0 with M > 0
                (c._h, po, pi, 2, g2, 2, _ptrs(p0, None), L, D, 2, 2, 2),               # null key with g != 1
                (c._h, po, pi, 2, _u32(1, 3), 2, _ptrs(p0, None), L, D, 2, 2, 2),
                (c._h, po + 8, pi, 1, g2, 2, r2, L, D, 2, 2, 2), (c._h, po, pi + 8, 1, g2, 2, r2, L, D, 2, 2, 2),
                (c._h, po, pi, 1, g2, 2, _ptrs(p0, p1 + 8), L, D, 2, 2, 2),             # misaligned key
                (c._h, po, pi, 1, g2, 2, r2, L, _ptrs(q0, q1, None, q1 + 8), 2, 2, 2),  # misaligned diagonal
                (c._h, po, pi, 2, g2, 2, r2, L, D, 2, 2, 0), (c._h, po, pi, 2, g2, 2, r2, L, D, 2, 2, L),   # k = 0, L
                (c._h, po, pi, 2, g2, 2, r2, L, D, 2, 0, 2),                            # alpha = 0
                (c._h, po, pi, 2, g2, 2, r2, L - 1, D, 2, 2, 2),                        # key_limbs < L
                (dup._h, po, pi, 2, g2, 2, r2, 4, D, 2, 1, 1),                          # two equal primes
                (c._h, po, pi, 2, _u32(3, 4), 2, r2, L, D, 2, 2, 2), (c._h, po, pi, 2, _u32(0, 3), 2, r2, L, D, 2, 2, 2),
                (c._h, po, pi, 2, _u32(3, 2 * N), 2, r2, L, D, 2, 2, 2),
                (c._h, po, pi, 0x7fffffff // (4 * L) + 1, g2, 2, r2, L, D, 2, 9, 2),    # 2 M B L > 2^31 - 1 (dnum = 1)
                (c._h, po, pi, 0x7fffffff // (5 * L) + 1, _u32(3), 1, _ptrs(p0), L, _ptrs(q0), 1, 1, 2),   # dnum B L
                (c._h, pi, pi, 2, g2, 2, r2, L, D, 2, 2, 2),                            # out on in
                (c._h, bp + 8 * (cw - 2), bp, 2, g2, 2, r2, L, D, 2, 2, 2),             # in's last 16 bytes are out's first
                (c._h, bp, bp + 8 * (ow - 2), 2, g2, 2, r2, L, D, 2, 2, 2),             # out's last 16 bytes are in's first
                (c._h, bp + 8 * (kw - 2), pi, 2, g2, 2, _ptrs(p0, bp), L, D, 2, 2, 2),  # out starts in key 1's last digit
                (c._h, bp, pi, 2, g2, 2, _ptrs(bp + 8 * (ow - 2), p1), L, D, 2, 2, 2),  # key 0 starts in out
                (c._h, bp + 8 * (L * N - 2), pi, 2, g2, 2, r2, L, _ptrs(q0, bp, None, q1), 2, 2, 2),   # out on diagonal
                (c._h, bp, pi, 2, g2, 2, r2, L, _ptrs(q0, q1, None, bp + 8 * (ow - 2)), 2, 2, 2),     # diagonal in out
            ]
            for h, o_, i_, B, gp, G, rp, kl, dp, M, al, kk in invalid:
                l0 = [t.launch_count() for t in ctxs]
                assert lib.agx_lintrans64(h, o_, i_, B, gp, G, rp, kl, dp, M, al, kk, form, None) == -1, \
                    (form, B, G, M, kl, al, kk)
                assert [t.launch_count() for t in ctxs] == l0
            l0 = c.launch_count()
            nul = lambda n: _ptrs(*([None] * n))                                   # refused if they were read
            for G, M in ((65, 1), (1, 17), (52, 5)):                               # G > 64, M > 16, M G > 256
                gz = _u32(*([2] * G))
                assert lib.agx_lintrans64(c._h, po, pi, 2, gz, G, nul(G), L, nul(G * M), M, 2, 2, form, None) == -2
            for al, kk in ((17, 2), (16, 17)):                                     # 17 digit primes; k = 17
                l19 = c19.launch_count()
                assert lib.agx_lintrans64(c19._h, bp, bp + 8 * 40 * N, 1, _u32(3), 1, _ptrs(p0), 19, _ptrs(q0), 1,
                                          al, kk, form, None) == -2, (al, kk)
                assert c19.launch_count() == l19
            for o_, i_, rp in ((None, None, _ptrs(None, None)), (po, pi, r2), (bp, bp + 16, _ptrs(bp, bp))):   # B == 0
                assert lib.agx_lintrans64(c._h, o_, i_, 0, g2, 2, rp, L, D, 2, 2, 2, form, None) == 0
            assert lib.agx_lintrans64(c._h, po, pi, 2, g2, 2, r2, L, None, 0, 2, 2, form, None) == 0       # M == 0
            assert lib.agx_lintrans64(c._h, pi, pi, 2, None, 0, None, L, None, 0, 2, 2, form, None) == 0
            assert c.launch_count() == l0
            torch.cuda.synchronize()
            assert torch.equal(o, osnap)
            # adjacent, not overlapping: allowed; a NULL diagonal's address and an unread key digit may overlap
            assert lib.agx_lintrans64(c._h, bp + 8 * kw, pi, 2, g2, 2, _ptrs(bp, bp), L, _ptrs(q0, bp + 8 * (kw - L * N)),
                                      1, 2, 2, form, None) == 0
            assert lib.agx_lintrans64(c._h, bp + 8 * 2 * L * N, pi, 2, g2, 2, _ptrs(bp, p1), L, D, 2, 9, 2, form,
                                      None) == 0
        ones = torch.ones(L, N, dtype=torch.int64, device="cuda")
        bad = [
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1], [[d0, d1]], 2, 2),                 # out has M = 2
            lambda: c.lintrans(o[:, :, :1], x, [3, 5], [rk0, rk1], [[d0, d1]] * 2, 2, 2),    # out batch
            lambda: c.lintrans(o, x, [3, 5], [rk0], [[d0, d1]] * 2, 2, 2),                   # fewer keys than elements
            lambda: c.lintrans(o, x, [3, 5], [rk0, None], [[d0, d1]] * 2, 2, 2),             # no key for g != 1
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1], [[d0], [d0]], 2, 2),                # a short row of diagonals
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1], [[d0, d1[:ell1].contiguous()]] * 2, 2, 2),   # diagonal over Q_l
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1[:2]], [[d0, d1]] * 2, 2, 2),          # fewer key digits
            lambda: c.lintrans(o, x, [3, 5], [rk0, torch.cat([rk1, rk1], 2)], [[d0, d1]] * 2, 2, 2),   # key_limbs
            lambda: c.lintrans(o, x[0], [3, 5], [rk0, rk1], [[d0, d1]] * 2, 2, 2),           # not a ciphertext
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1], [[d0, d1]] * 2, 0, 2),              # alpha = 0
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1], [[d0, d1]] * 2, 2, 0),              # k = 0
            lambda: c.lintrans(o, x, [3, 5], [rk0, rk1], [[d0, d1.cpu()]] * 2, 2, 2),        # host tensor
            lambda: c.lintrans(o, x, [3, 2**32 + 5], [rk0, rk1], [[d0, d1]] * 2, 2, 2),      # not 32-bit
        ]
        for fn in bad:
            with pytest.raises(ValueError):
                fn()
        with pytest.raises(A.AgxError) as e:
            c.lintrans(o, x, [3, 4], [rk0, rk1], [[d0, ones]] * 2, 2, 2)                     # even element
        assert e.value.code == -1
        torch.cuda.synchronize()
        assert torch.equal(o, osnap)
        assert all(torch.equal(t, s) for t, s in zip((x, rk0, rk1, d0, d1), snaps))
    finally:
        for t in (dup, c32):
            t.close()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_inputs_unchanged(ctx, form):
    import torch
    N = 4096
    primes = QS + PS
    c = ctx(N, primes)
    gs = elements(N, 3)
    rks = [None] + [dev(rand_key(3, primes, N, 91 + t)) for t in (1, 2)]
    ct = dev(ciphertexts(4, QS, N, 93))
    diags = pattern(N, primes, 3, 3, 95)
    flat = [d for row in diags for d in row if d is not None]
    snap, ksnap, dsnap = ct.clone(), [r.clone() for r in rks[1:]], [d.clone() for d in flat]
    call(c, ct, gs, rks, diags, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(ct, snap) and all(torch.equal(r, s) for r, s in zip(rks[1:], ksnap))
    assert all(torch.equal(d, s) for d, s in zip(flat, dsnap))


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    """The header's counts (agx_rotate64's), the same for (G, M) = (1, 1), (3, 4) with a keyless term and (8, 16)."""
    import torch
    x = int(N == 32768)
    primes = QS + PS
    c, c1 = ctx(N, primes), ctx(N, QS + PS[:1])
    ct = dev(ciphertexts(2, QS, N, 99))
    key = dev(rand_key(5, primes, N, 97))
    dg = rand_diag(primes, N, 98)

    def launches(cx, G, M, alpha, k, form, rk=key):
        gs = elements(N, G)
        rks = [None if g == 1 and t == 0 else rk for t, g in enumerate(gs)]
        l0 = cx.launch_count()
        call(cx, ct, gs, rks, [[dg if cx is c else dg[:cx.L].contiguous()] * G] * M, alpha, k, form)
        torch.cuda.synchronize()
        return cx.launch_count() - l0

    k1 = key[:, :, :len(QS) + 1].contiguous()
    for G, M in ((1, 1), (3, 4), (8, 16)):
        # alpha = 2: digits of 2, 2 and 1 primes (ModUps 3 + 3 + 2, one more each at N = 32768); inner 1; ModDown 3 (4)
        assert launches(c, G, M, 2, 2, True) == 8 + 3 * x + 1 + 3 + x
        assert launches(c, G, M, 2, 2, False) == 3 + 5 + x                  # dnum + 5
        # alpha = 5: one digit: 3 * dnum + 4 (4 * dnum + 5 at N = 32768)
        assert launches(c, G, M, 5, 2, True) == 7 + 2 * x
        assert launches(c, G, M, 5, 2, False) == 6 + x
        # k = 1: the ModDown is the rescale (2; 3 at N = 32768)
        assert launches(c1, G, M, 5, 1, True, k1) == 3 + x + 1 + 2 + x
        assert launches(c1, G, M, 5, 1, False, k1) == 6 + x


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    primes = QS + PS
    c = ctx(N, primes)
    gs = elements(N, 8)
    keys = [rand_key(3, primes, N, 101 + t) for t in range(8)]
    dgs = [data(1, primes, N, 150 + t)[0] for t in range(8)]
    x = ciphertexts(4, QS, N, 103)
    want = recipe(ctx, c, dev(x), gs, [dev(k) for k in keys], [[dev(d) for d in dgs]] * 2, 2, 2, form)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        copies = []
        for h in [x] + keys + dgs:
            d_h = dev(h)
            t = torch.empty_like(d_h)
            t.copy_(d_h)                                                # torch work the call must follow
            copies.append(t)
        ct, rks, diags = copies[0], copies[1:9], [copies[9:]] * 2
        out = empty(2, 2, 4, len(QS), N)
    c.lintrans(out, ct, gs, rks, diags, 2, 2, ntt_form=form, stream=s)
    s.synchronize()
    assert torch.equal(out, want)
