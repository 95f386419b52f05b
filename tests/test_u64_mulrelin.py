"""u64 RNS ciphertext multiplication in one call (agx_mulrelin64, Context64.mulrelin).

Definition, for a context over Q_l u P (the k special primes last), ciphertexts a = (a0, a1) and b = (b0, b1) over Q_l
and a relinearisation key rlk in agx_keyswitch64's layout (its key for s' = s^2):
    D_0 = a0 b0,  D_1 = a0 b1 + a1 b0,  D_2 = a1 b1                                  over Q_l
    A_c = sum_j ModUp_j(digit_j(D_2)) (.) rlk[j][c]  +  P D_c                         over Q_l u P
    rescale = 0: out_c = ModDown_P(A_c) = D_c + KS(D_2)[c]                            over Q_l
    rescale = 1: out_c = floor((X_c + h) / (q_l P)) mod Q_{l-1}, X_c the CRT value of A_c, h = (q_l P - 1) / 2.

The CPU tests pin a big-integer oracle of that definition: with rescale = 0 it is the tensor plus the key-switch
oracle of D_2, with rescale = 1 it is that result rescaled by q_l, and encrypted products decrypt within the bounds
derived below; a further test checks the new kernels' resources.  The GPU tests compare the call with the oracle
and, bit for bit in both forms, with the recipe composed from public calls, and cover squaring, digit shapes, one key at
several levels, batches, an encrypted level chain, refusals, launch counts, unchanged inputs and side-stream ordering.

Decryption bounds (s ternary, the key's errors |e_j| <= E, digit j's primes multiplying to D_j, phases phi_a = a0 +
a1 s and phi_b over the integers, Phi = phi_a phi_b negacyclic).  Write K = sum_j U_j e_j, |U_j| <= D_j / 2, so
|K| <= N E sum_j D_j / 2.  The gadget key gives X_0 + X_1 s = P Phi + K (mod Q P) coefficient-wise.
- rescale = 0: the key switch's derivation applies unchanged to D_2, and D_0 + D_1 s + D_2 s^2 = Phi (mod Q), so
  out_0 + out_1 s - Phi is centred mod Q within |K| / P + (N + 1) / 2 (agx_keyswitch64's bound, KS.ks_bound).
- rescale = 1: out_c = (X_c + h - r_c) / (q P) with 0 <= r_c < q P, and h (1 + s) - r_0 - r_1 s is at most
  (N + 1) / 2 * q P in absolute value.  So q (out_0 + out_1 s) - Phi = K / P + q R (mod Q) with |R| <= (N + 1) / 2: the
  product over q_l within |K| / (q_l P) + (N + 1) / 2: one rounding term, where bounding the key switch and a rescale
  after it separately would add two.

The fused rescale rounds once, yet it equals agx_rescale64 of the rescale = 0 result bit for bit: with h_P = (P - 1) / 2
and h_q = (q_l - 1) / 2, h = h_P + P h_q, and floor((floor((X + h_P) / P) + h_q) / q_l) = floor((X + h) / (q_l P)) for
every X >= 0 (nested floor division); the reduction mod Q between the two steps changes nothing mod Q_{l-1}."""
import random
import re
from math import prod

import numpy as np
import pytest

import test_u64_keyswitch as KS
from oracle import oracle as O

gpu = pytest.mark.gpu
SIZES = KS.SIZES
PRIMES, QS, PS, Q17, P17 = KS.PRIMES, KS.QS, KS.PS, KS.Q17, KS.P17


# ---- big ints: the oracle
def centred(v, Q):
    v %= Q
    return v - Q if v > Q // 2 else v


def ints(x, qs):
    """[l+1][N] residues -> N CRT values in [0, Q)"""
    return [KS.crt(x[:, i], qs) for i in range(x.shape[1])]


def tensor_ints(a, b, qs, bb):
    """D_0, D_1, D_2 of ciphertexts a[:, bb], b[:, bb] as CRT values mod Q"""
    Q = prod(qs)
    A0, A1, B0, B1 = ints(a[0, bb], qs), ints(a[1, bb], qs), ints(b[0, bb], qs), ints(b[1, bb], qs)
    d1 = [u + v for u, v in zip(KS.negacyclic(A0, B1), KS.negacyclic(A1, B0))]
    return [[v % Q for v in d] for d in (KS.negacyclic(A0, B0), d1, KS.negacyclic(A1, B1))]


def residues(vals, qs):
    return np.array([[v % q for v in vals] for q in qs], dtype=np.uint64)


def mulrelin_oracle(a, b, kc, primes, k, alpha, rescale):
    """a, b [2][B][l+1][N] in coefficient form over primes[:l+1]; kc the key in coefficient form (as keyswitch_oracle
    takes it) -> [2][B][l+1][N], or [2][B][l][N] with rescale.  Big integers mod QP throughout: the tensor, the centred
    lift of each digit of D_2, the negacyclic products with the key summed, plus P D_c, then floor((X + h) / P') with
    P' = P, or q_l P with rescale."""
    L = len(primes)
    ell1 = L - k
    qs = primes[:ell1]
    P, QP = prod(primes[ell1:]), prod(primes)
    Pd = P * qs[-1] if rescale else P
    qo = qs[:-1] if rescale else qs
    Qo = prod(qo)
    rows = KS.key_rows(L, k, kc.shape[2])
    digits = KS.digits_of(ell1, alpha)
    N, B = a.shape[3], a.shape[1]
    keys = [[[KS.crt([kc[j, c, rows[i], x] for i in range(L)], primes) for x in range(N)] for c in (0, 1)]
            for j in range(len(digits))]
    out = np.empty((2, B, len(qo), N), dtype=np.uint64)
    for bb in range(B):
        D = tensor_ints(a, b, qs, bb)
        acc = [[P * d % QP for d in D[0]], [P * d % QP for d in D[1]]]
        for j, (f, cnt) in enumerate(digits):
            S = prod(primes[f:f + cnt])
            h = (S - 1) // 2
            U = [(d + h) % S - h for d in D[2]]                           # the digit's residues are D_2 mod S
            for c in (0, 1):
                acc[c] = [(u + v) % QP for u, v in zip(acc[c], KS.negacyclic(U, keys[j][c]))]
        for c in (0, 1):
            out[c, bb] = residues([((X + (Pd - 1) // 2) // Pd) % Qo for X in acc[c]], qo)
    return out


def encrypt(rng, s, m, qs, ebound):
    """(c0, c1) = (-a s + m + e, a) mod each prime: [2][1][l+1][N]"""
    N = len(s)
    a = [rng.randrange(prod(qs)) for _ in range(N)]
    e = KS.small(rng, N, ebound)
    c0 = [-u + v + w for u, v, w in zip(KS.negacyclic(a, s), m, e)]
    return np.stack([residues(c0, qs), residues(a, qs)]).reshape(2, 1, len(qs), N)


def phase(ct, s, qs):
    """c0 + c1 s over the integers, centred mod Q"""
    Q = prod(qs)
    c0, c1 = ints(ct[0, 0], qs), ints(ct[1, 0], qs)
    return [centred(u + v, Q) for u, v in zip(c0, KS.negacyclic(c1, s))]


def relin_noise(qs, ps, alpha, N, ebound):
    """|K| / P rounded up: the key's part of the bounds (module docstring)"""
    return N * ebound * sum(prod(qs[f:f + c]) // 2 for f, c in KS.digits_of(len(qs), alpha)) // prod(ps) + 1


def check_product(out, pa, pb, s, qs, ps, alpha, ebound, rescale):
    """out [2][1][.][N] decrypts to pa pb (rescale 0) or pa pb / q_l (rescale 1) within the module docstring's bound"""
    N, Q = len(s), prod(qs)
    Phi = KS.negacyclic(pa, pb)
    assert max(abs(v) for v in Phi) < Q >> 40
    if not rescale:
        bound = KS.ks_bound(qs, ps, alpha, N, ebound)
        got = phase(out, s, qs)
        err = [centred(g - v, Q) for g, v in zip(got, Phi)]
        assert max(abs(v) for v in err) <= bound
        return got
    ql = qs[-1]
    bound = relin_noise(qs, ps, alpha, N, ebound) + ql * ((N + 1) // 2)     # on q_l times the decryption
    got = phase(out, s, qs[:-1])
    err = [centred(ql * g - v, Q) for g, v in zip(got, Phi)]
    assert max(abs(v) for v in err) <= bound
    assert bound < Q >> 40
    return got


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("N,qs,ps,alpha", [(8, QS[:3], PS, 1), (16, QS, PS, 2), (16, QS[:4], PS[:1], 3),
                                           (8, QS[:2], PS, 5)])
def test_oracle_is_tensor_plus_keyswitch(N, qs, ps, alpha):
    """rescale = 0: the oracle is D_c + keyswitch_oracle(D_2)[c]; rescale = 1: it is that divided by q_l and rounded
    (floor((Y + h_q) / q_l) mod Q_{l-1}, Y the CRT value in [0, Q)), exactly: the two roundings compose into one."""
    rng = random.Random(N * 11 + alpha + len(qs))
    primes, k = qs + ps, len(ps)
    kc = np.stack([KS.rand_res(2, primes, N, rng) for _ in KS.digits_of(len(qs), alpha)])
    a = np.stack([KS.rand_res(2, qs, N, rng) for _ in (0, 1)], 1)
    b = np.stack([KS.rand_res(2, qs, N, rng) for _ in (0, 1)], 1)
    out0 = mulrelin_oracle(a, b, kc, primes, k, alpha, False)
    out1 = mulrelin_oracle(a, b, kc, primes, k, alpha, True)
    Q, ql = prod(qs), qs[-1]
    Qr = Q // ql
    d2 = np.stack([residues(tensor_ints(a, b, qs, bb)[2], qs) for bb in range(2)])
    ks = KS.keyswitch_oracle(d2, kc, primes, k, alpha)
    for bb in range(2):
        D = tensor_ints(a, b, qs, bb)
        for c in (0, 1):
            want = [(d + KS.crt(ks[c, bb, :, x], qs)) % Q for x, d in enumerate(D[c])]
            assert (out0[c, bb] == residues(want, qs)).all()
            twice = [((y + (ql - 1) // 2) // ql) % Qr for y in want]
            assert (out1[c, bb] == residues(twice, qs[:-1])).all()
    # squaring is the product with itself
    assert (mulrelin_oracle(a, a, kc, primes, k, alpha, True) ==
            mulrelin_oracle(a, a.copy(), kc, primes, k, alpha, True)).all()


@pytest.mark.parametrize("N,qs,ps,alpha", [(16, QS, PS, 2), (8, QS[:3], PS, 1), (16, QS[:4], PS[:1], 4)])
def test_oracle_decrypts_to_the_product(N, qs, ps, alpha):
    """With a gadget key for s^2, encrypted m1, m2 multiply to m1 m2 (rescale 0) and to m1 m2 / q_l (rescale 1)
    within the module docstring's bounds; the rescaled bound has one rounding term (N + 1) / 2."""
    rng = random.Random(N * 5 + alpha)
    primes, k = qs + ps, len(ps)
    s = KS.ternary(rng, N)
    ebound = 6
    kc = KS.gadget_key_coeff(primes, k, alpha, len(qs), s, KS.negacyclic(s, s), ebound, rng)
    m1 = [rng.randint(-(1 << 45), 1 << 45) for _ in range(N)]
    m2 = [rng.randint(-(1 << 45), 1 << 45) for _ in range(N)]
    c1, c2 = encrypt(rng, s, m1, qs, ebound), encrypt(rng, s, m2, qs, ebound)
    p1, p2 = phase(c1, s, qs), phase(c2, s, qs)
    for rescale in (False, True):
        out = mulrelin_oracle(c1, c2, kc, primes, k, alpha, rescale)
        check_product(out, p1, p2, s, qs, ps, alpha, ebound, rescale)
    # a key for a wrong s' leaves an error of the size of Q
    bad = KS.gadget_key_coeff(primes, k, alpha, len(qs), s, [x + 1 for x in KS.negacyclic(s, s)], ebound, rng)
    out = mulrelin_oracle(c1, c2, bad, primes, k, alpha, False)
    Phi = KS.negacyclic(p1, p2)
    assert max(abs(centred(g - v, prod(qs))) for g, v in zip(phase(out, s, qs), Phi)) > prod(qs) >> 20


def test_mulrelin_kernels_use_no_local_memory():
    """Every instantiation of the multiplication's inner product (1, 2, 4 and 8 digits per chunk) is in the sm_100a
    code and runs without local memory or stack."""
    usage = KS._cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*mulrelin64_inner\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
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


def ciphertexts(B, qs, N, seed):
    return data(2 * B, qs, N, seed).reshape(2, B, len(qs), N)


def tensor(cq, a, b, form):
    """D [3][B][l+1][n] from public calls: element-wise products in evaluation form, negacyclic products otherwise"""
    D = empty(3, *a.shape[1:])
    if form:
        cq.elementwise("mul", D[0], a[0], b[0])
        cq.elementwise("mul", D[1], a[0], b[1])
        cq.elementwise("mac", D[1], a[1], b[0])
        cq.elementwise("mul", D[2], a[1], b[1])
    else:
        t = empty(*a.shape[1:])
        cq.polymul(D[0], a[0], b[0])
        cq.polymul(D[1], a[0], b[1])
        cq.polymul(t, a[1], b[0])
        cq.elementwise("add", D[1], D[1], t)
        cq.polymul(D[2], a[1], b[1])
    return D


def fold_sums(c, D, rlk, alpha, k):
    """A_c [2][B][L][n] in evaluation form from public calls: modup of each digit of D_2, element-wise products with the
    key rows (sliced and replicated) summed, plus (P mod q_i) D_c on Q_l padded with zeros on P"""
    import torch
    L, N, B = c.L, c.n, D.shape[1]
    ell1 = L - k
    kr = torch.cat([rlk[:, :, :ell1], rlk[:, :, rlk.shape[2] - k:]], dim=2)
    P = prod(c.primes[ell1:])
    pm = torch.tensor([P % q if i < ell1 else 0 for i, q in enumerate(c.primes)], dtype=torch.int64,
                      device="cuda").view(1, L, 1).expand(B, L, N).contiguous()
    acc = empty(2, B, L, N)
    for j, (f, cnt) in enumerate(KS.digits_of(ell1, alpha)):
        U = empty(B, L, N)
        c.modup(U, D[2, :, f:f + cnt].contiguous(), f, cnt, ntt_form=True)
        for cc in (0, 1):
            c.elementwise("mul" if j == 0 else "mac", acc[cc], U, kr[j, cc].expand(B, L, N).contiguous())
    for cc in (0, 1):
        padded = torch.cat([D[cc], torch.zeros(B, k, N, dtype=D.dtype, device=D.device)], 1)
        c.elementwise("mac", acc[cc], padded, pm)
    return acc


def recipe(ctx, c, a, b, rlk, alpha, k, rescale, form, psis=None):
    """The definition from public calls.  rescale 0: the tensor, keyswitch of D_2 and two adds, all in the call's form.
    rescale 1: the tensor in evaluation form, fold_sums, and one moddown by the last k + 1 primes in the call's form."""
    import torch
    B, ell1, N = a.shape[1], a.shape[2], a.shape[3]
    cq = ctx(N, c.primes[:ell1], psis[:ell1] if psis else None)
    if not rescale:
        D = tensor(cq, a, b, form)
        out = c.keyswitch(empty(2, B, ell1, N), D[2], rlk, alpha, k, ntt_form=form)
        for cc in (0, 1):
            cq.elementwise("add", out[cc], out[cc], D[cc])
        return out
    if form:
        ah, bh = a, b
    else:
        ah, bh = a.clone(), b.clone()
        cq.fwd(ah.view(2 * B, ell1, N))
        cq.fwd(bh.view(2 * B, ell1, N))
    acc = fold_sums(c, tensor(cq, ah, bh, True), rlk, alpha, k)
    if not form:
        c.inv(acc.view(2 * B, c.L, N))
    out = empty(2, B, ell1 - 1, N)
    c.moddown(out.view(2 * B, ell1 - 1, N), acc.view(2 * B, c.L, N), k + 1, ntt_form=form)
    torch.cuda.synchronize()
    return out


def call(c, a, b, rlk, alpha, k, rescale, form, stream=None):
    ell1 = c.L - k
    out = empty(2, a.shape[1], ell1 - 1 if rescale else ell1, c.n)
    return c.mulrelin(out, a, b, rlk, alpha, k, rescale=rescale, ntt_form=form, stream=stream)


@gpu
@pytest.mark.parametrize("roots", ("minimal", "caller"))
@pytest.mark.parametrize("N,alpha,k", [(8, 2, 2), (16, 3, 1), (32, 9, 2)])
def test_vs_oracle(ctx, N, alpha, k, roots):
    """Coefficient form against the big-integer oracle, evaluation form against its transform, both rescale values."""
    qs = QS
    primes = qs + PS[:k]
    psis = caller_roots(N, primes) if roots == "caller" else None
    c = ctx(N, primes, psis)
    rng = random.Random(N + alpha)
    dnum = len(KS.digits_of(len(qs), alpha))
    kc = np.stack([KS.rand_res(2, primes, N, rng) for _ in range(dnum)])
    rlk = dev(KS.rns_fwd(kc, primes, psis))
    a, b = ciphertexts(2, qs, N, 7 + N), ciphertexts(2, qs, N, 11 + N)
    for rescale in (False, True):
        want = mulrelin_oracle(a, b, kc, primes, k, alpha, rescale)
        assert (host(call(c, dev(a), dev(b), rlk, alpha, k, rescale, False)) == want).all(), rescale
        qo = qs[:-1] if rescale else qs
        got = call(c, dev(KS.rns_fwd(a, qs, psis)), dev(KS.rns_fwd(b, qs, psis)), rlk, alpha, k, rescale, True)
        assert (host(got) == KS.rns_fwd(want, qo, psis[:len(qo)] if psis else None)).all(), rescale


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_vs_composed_recipe(ctx, N, form):
    """Three digits (2, 2 and 1 primes), k = 2, a key with two extra rows; with and without rescale."""
    import torch
    primes = QS + PS
    c = ctx(N, primes)
    rlk = dev(rand_key(3, QS + [PRIMES[50][10], PRIMES[50][11]] + PS, N, 5 + N))
    a, b = dev(ciphertexts(2, QS, N, 13 + N)), dev(ciphertexts(2, QS, N, 17 + N))
    for rescale in (False, True):
        got = call(c, a, b, rlk, 2, 2, rescale, form)
        torch.cuda.synchronize()
        assert torch.equal(got, recipe(ctx, c, a, b, rlk, 2, 2, rescale, form)), rescale


@gpu
@pytest.mark.parametrize("N", (32, 1024, 32768))
def test_caller_roots(ctx, N):
    import torch
    primes = QS + PS
    psis = caller_roots(N, primes)
    c = ctx(N, primes, psis)
    rlk = dev(rand_key(3, primes, N, 19 + N))
    a, b = dev(ciphertexts(2, QS, N, 23 + N)), dev(ciphertexts(2, QS, N, 29 + N))
    for form in (False, True):
        for rescale in (False, True):
            got = call(c, a, b, rlk, 2, 2, rescale, form)
            torch.cuda.synchronize()
            assert torch.equal(got, recipe(ctx, c, a, b, rlk, 2, 2, rescale, form, psis)), (form, rescale)


@gpu
@pytest.mark.parametrize("N", (32, 4096, 32768))
def test_rescale_equals_rescale_of_product(ctx, N):
    """The fused rescale equals agx_rescale64 applied to the unrescaled product, bit for bit, in both forms (module
    docstring: the two roundings compose into one); k = 2 and k = 1."""
    import torch
    for ps in (PS, PS[:1]):
        primes = QS + ps
        c, cq = ctx(N, primes), ctx(N, QS)
        rlk = dev(rand_key(3, primes, N, 31))
        a, b = dev(ciphertexts(3, QS, N, 37)), dev(ciphertexts(3, QS, N, 41))
        for form in (False, True):
            once = call(c, a, b, rlk, 2, len(ps), True, form)
            full = call(c, a, b, rlk, 2, len(ps), False, form)
            twice = empty(2, 3, len(QS) - 1, N)
            cq.rescale(twice.view(6, len(QS) - 1, N), full.view(6, len(QS), N), ntt_form=form)
            torch.cuda.synchronize()
            assert torch.equal(once, twice), (len(ps), form)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (32, 16384))
def test_squaring(ctx, N, form):
    """d_a == d_b equals the call with b a separate copy (the coefficient form then forwards once)."""
    import torch
    c = ctx(N, QS + PS)
    rlk = dev(rand_key(3, QS + PS, N, 43))
    a = dev(ciphertexts(3, QS, N, 47 + N))
    for rescale in (False, True):
        got = call(c, a, a, rlk, 2, 2, rescale, form)
        want = call(c, a, a.clone(), rlk, 2, 2, rescale, form)
        torch.cuda.synchronize()
        assert torch.equal(got, want), rescale
        assert torch.equal(got, recipe(ctx, c, a, a, rlk, 2, 2, rescale, form)), rescale


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (32, 4096))
@pytest.mark.parametrize("shape", ("alpha1_dnum17", "one_digit", "partial_last", "k1"))
def test_digit_shapes(ctx, N, form, shape):
    """alpha = 1 with l + 1 = 17 (17 digits: the lazy sums fold, the P D_c term in the first chunk only), one digit, a
    partial last digit (5 = 3 + 2), and k = 1 (the rescale is then a two-prime ModDown)."""
    import torch
    qs, ps, alpha = {"alpha1_dnum17": (Q17, P17, 1), "one_digit": (QS, PS, 5), "partial_last": (QS, PS, 3),
                     "k1": (QS, PS[:1], 2)}[shape]
    primes = qs + ps
    c = ctx(N, primes)
    dnum = len(KS.digits_of(len(qs), alpha))
    rlk = dev(rand_key(dnum, primes, N, 53 + N))
    a, b = dev(ciphertexts(2, qs, N, 59 + N)), dev(ciphertexts(2, qs, N, 61 + N))
    for rescale in (False, True):
        got = call(c, a, b, rlk, alpha, len(ps), rescale, form)
        torch.cuda.synchronize()
        assert torch.equal(got, recipe(ctx, c, a, b, rlk, alpha, len(ps), rescale, form)), rescale


@gpu
def test_one_key_at_three_levels(ctx):
    """One key over Q_top u P (key_limbs = 7 + 2), alpha = 3, used unchanged at l + 1 = 7, 5 and 2."""
    import torch
    N = 1024
    qtop = QS + [PRIMES[62][3], PRIMES[50][3]]
    rlk = dev(rand_key(3, qtop + PS, N, 67))
    for ell1 in (7, 5, 2):
        qs = qtop[:ell1]
        c = ctx(N, qs + PS)
        a, b = dev(ciphertexts(2, qs, N, 71 + ell1)), dev(ciphertexts(2, qs, N, 73 + ell1))
        for form in (False, True):
            for rescale in (False, True):
                got = call(c, a, b, rlk, 3, 2, rescale, form)
                torch.cuda.synchronize()
                assert torch.equal(got, recipe(ctx, c, a, b, rlk, 3, 2, rescale, form)), (ell1, form, rescale)


@gpu
@pytest.mark.parametrize("N", (512, 16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """More polynomials than two waves of every transform geometry and than one slice of the inner product."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = -(-(2 * sms + 5) // len(QS))
    c = ctx(N, QS + PS)
    rlk = dev(rand_key(3, QS + PS, N, 79))
    a, b = dev(ciphertexts(B, QS, N, 83 + N)), dev(ciphertexts(B, QS, N, 89 + N))
    for form in (False, True):
        for rescale in (False, True):
            got = call(c, a, b, rlk, 2, 2, rescale, form)
            assert torch.equal(got, recipe(ctx, c, a, b, rlk, 2, 2, rescale, form)), (form, rescale)
            del got
            torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_batch_is_single_calls(ctx, form):
    import torch
    N = 2048
    c = ctx(N, QS + PS)
    rlk = dev(rand_key(3, QS + PS, N, 97))
    a, b = dev(ciphertexts(5, QS, N, 101)), dev(ciphertexts(5, QS, N, 103))
    got = call(c, a, b, rlk, 2, 2, True, form)
    for bb in range(5):
        one = call(c, a[:, bb:bb + 1].contiguous(), b[:, bb:bb + 1].contiguous(), rlk, 2, 2, True, form)
        torch.cuda.synchronize()
        assert torch.equal(got[:, bb:bb + 1], one), bb


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_product_end_to_end(ctx, form):
    """Encrypt m1, m2 (coefficients up to 2^45) under s with a gadget key for s^2 over Q_top u P; multiply with rescale
    and decrypt to m1 m2 / q_l within the module docstring's bound; then square that result with the same key one
    level down and decrypt to its phase squared over q_{l-1}.  Also without rescale: m1 m2 within the key switch's
    bound."""
    import torch
    N = 256
    qs, alpha, k = QS, 2, len(PS)
    rng = random.Random(107)
    s = KS.ternary(rng, N)
    ebound = 8
    key_primes = qs + PS
    rlk = KS.gadget_key_gpu(ctx(N, key_primes), key_primes, k, alpha, len(qs), s, KS.negacyclic(s, s), ebound, rng)
    m1 = [rng.randint(-(1 << 45), 1 << 45) for _ in range(N)]
    m2 = [rng.randint(-(1 << 45), 1 << 45) for _ in range(N)]
    c1, c2 = encrypt(rng, s, m1, qs, ebound), encrypt(rng, s, m2, qs, ebound)
    p1, p2 = phase(c1, s, qs), phase(c2, s, qs)
    assert max(abs(u - v) for u, v in zip(p1, m1)) <= ebound

    def mul(qs_, x, y, rescale):
        c = ctx(N, qs_ + PS)
        cq = ctx(N, qs_)
        dx, dy = dev(x), dev(y)
        if form:
            cq.fwd(dx.view(-1, len(qs_), N))
            cq.fwd(dy.view(-1, len(qs_), N))
        out = call(c, dx, dy, rlk, alpha, k, rescale, form)
        if form:
            ctx(N, qs_[:-1] if rescale else qs_).inv(out.view(2, -1, N))
        torch.cuda.synchronize()
        return host(out)

    check_product(mul(qs, c1, c2, False), p1, p2, s, qs, PS, alpha, ebound, False)
    x = mul(qs, c1, c2, True)
    px = check_product(x, p1, p2, s, qs, PS, alpha, ebound, True)
    assert max(abs(v) for v in px) > 1 << 20                      # m1 m2 / q_l is not a rounding residue
    y = mul(qs[:-1], x, x, True)
    check_product(y, px, px, s, qs[:-1], PS, alpha, ebound, True)


@gpu
def test_refusals_and_empty_calls(A, ctx):
    import ctypes as C
    import torch
    N = 1024
    lib = A.lib()
    primes = QS + PS
    L, ell1 = len(primes), len(QS)
    c, c19 = ctx(N, primes), ctx(N, Q17 + P17)
    c1p = ctx(N, QS[:1] + PS)                                              # l + 1 = 1
    x, y = dev(ciphertexts(2, QS, N, 3)), dev(ciphertexts(2, QS, N, 5))
    rk = dev(rand_key(3, primes, N, 4))
    xs, ys, ks = x.clone(), y.clone(), rk.clone()
    o = empty(2, 2, ell1, N)
    pa, pb, po, pk = x.data_ptr(), y.data_ptr(), o.data_ptr(), rk.data_ptr()
    big = torch.zeros(40 * L * N, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    dup = A.Context64(N, [QS[0], QS[1], QS[0], PS[0]])
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    ctxs = (c, c19, c1p, dup)
    kw = 3 * 2 * L * N                                                      # key words read (dnum = 3)
    cw = 2 * 2 * ell1 * N                                                   # words of one input
    ow1 = 2 * 2 * (ell1 - 1) * N                                            # words of a rescaled output
    try:
        for form in (0, 1):
            for rs in (0, 1):
                ow = ow1 if rs else cw
                invalid = [
                    (c32._h, po, pa, pb, 2, pk, L, 2, 2),                             # u32 context
                    (c._h, None, pa, pb, 2, pk, L, 2, 2), (c._h, po, None, pb, 2, pk, L, 2, 2),
                    (c._h, po, pa, None, 2, pk, L, 2, 2), (c._h, po, pa, pb, 2, None, L, 2, 2),
                    (c._h, po + 8, pa, pb, 1, pk, L, 2, 2), (c._h, po, pa + 8, pb, 1, pk, L, 2, 2),
                    (c._h, po, pa, pb + 8, 1, pk, L, 2, 2), (c._h, po, pa, pb, 1, pk + 8, L, 2, 2),
                    (c._h, po, pa, pb, 2, pk, L, 2, 0), (c._h, po, pa, pb, 2, pk, L, 2, L),   # k = 0, k = L
                    (c._h, po, pa, pb, 2, pk, L, 0, 2),                               # alpha = 0
                    (c._h, po, pa, pb, 2, pk, L - 1, 2, 2),                           # key_limbs < L
                    (dup._h, po, pa, pb, 2, pk, 4, 1, 1),                             # two equal primes
                    (c._h, po, pa, pb, 0x7fffffff // (2 * L) + 1, pk, L, 9, 2),       # 2 B L > 2^31 - 1 (dnum = 1)
                    (c._h, po, pa, pb, 0x7fffffff // (5 * L) + 1, pk, L, 1, 2),       # dnum B L > 2^31 - 1
                    (c._h, pa, pa, pb, 2, pk, L, 2, 2), (c._h, pb, pa, pb, 2, pk, L, 2, 2),   # out on an input
                    (c._h, bp + 8 * (cw - 2), bp, pb, 2, pk, L, 2, 2),                # a's last 16 bytes are out's first
                    (c._h, bp, pa, bp + 8 * (ow - 2), 2, pk, L, 2, 2),                # out's last 16 bytes are b's first
                    (c._h, bp + 8 * (kw - 2), pa, pb, 2, bp, L, 2, 2),                # out starts in the key's last digit
                    (c._h, bp, pa, pb, 2, bp + 8 * (ow - 2), L, 2, 2),                # the key starts in out
                ]
                if rs:
                    invalid.append((c1p._h, po, pa, pb, 2, pk, L, 2, 2))              # rescale with l + 1 = 1
                for h, o_, a_, b_, B, k_, kl, al, kk in invalid:
                    l0 = [t.launch_count() for t in ctxs]
                    assert lib.agx_mulrelin64(h, o_, a_, b_, B, k_, kl, al, kk, rs, form, None) == -1, \
                        (form, rs, B, kl, al, kk)
                    assert [t.launch_count() for t in ctxs] == l0
                l0 = c.launch_count()
                for o_, a_, b_, k_ in ((None, None, None, None), (po, pa, pb, pk), (bp, bp + 16, bp, bp)):   # B == 0
                    assert lib.agx_mulrelin64(c._h, o_, a_, b_, 0, k_, L, 2, 2, rs, form, None) == 0
                assert c.launch_count() == l0
                # adjacent, not overlapping: allowed; a and b may be one tensor
                assert lib.agx_mulrelin64(c._h, bp + 8 * kw, pa, pa, 2, bp, L, 2, 2, rs, form, None) == 0
                assert lib.agx_mulrelin64(c._h, bp, bp + 8 * ow, bp + 8 * ow, 2, pk, L, 2, 2, rs, form, None) == 0
        bad = [
            lambda: c.mulrelin(empty(2, 1, ell1, N), x, y, rk, 2, 2),                       # out batch
            lambda: c.mulrelin(o, x, y[:, :1].contiguous(), rk, 2, 2),                      # unequal batches
            lambda: c.mulrelin(o, x, y, rk, 2, 2, rescale=True),                            # out not rescaled
            lambda: c.mulrelin(empty(2, 2, ell1 - 1, N), x, y, rk, 2, 2),                   # out rescaled
            lambda: c.mulrelin(o, x[0], y, rk, 2, 2),                                       # not a ciphertext
            lambda: c.mulrelin(o, x, y, rk[:2], 2, 2),                                      # fewer key digits
            lambda: c.mulrelin(o, x, y, rk[:, :, :L - 1].contiguous(), 2, 2),               # key_limbs < L
            lambda: c.mulrelin(o, x, y, rk, 0, 2),                                          # alpha = 0
            lambda: c.mulrelin(o, x, y, rk, 2, 0),                                          # k = 0
            lambda: c.mulrelin(o, x.cpu(), y, rk, 2, 2),                                    # host tensor
            lambda: c.mulrelin(o, x, y, rk.cpu(), 2, 2),
            lambda: c1p.mulrelin(empty(2, 2, 0, N), x[:, :, :1].contiguous(), x[:, :, :1].contiguous(), rk, 2, 2,
                                 rescale=True),                                             # nothing to rescale
        ]
        for fn in bad:
            with pytest.raises(ValueError):
                fn()
        torch.cuda.synchronize()
        assert torch.equal(x, xs) and torch.equal(y, ys) and torch.equal(rk, ks)
    finally:
        for t in (dup, c32):
            t.close()


@gpu
def test_unsupported(ctx):
    """More than 16 primes in a digit, k > 16, or k + 1 > 16 with rescale: AGX_E_UNSUPPORTED, launching nothing."""
    import agilex_ntt_b200 as A
    N = 32
    lib = A.lib()
    c19 = ctx(N, Q17 + P17)                                                 # L = 19
    big = empty(200 * 19 * N)
    bp = big.data_ptr()
    l0 = c19.launch_count()
    # (alpha, k, rescale): 17 digit primes; k = 16 with rescale (17 primes divided); k = 17 needs L >= 18 + ... a
    # context of 19 primes with k = 17 leaves l + 1 = 2
    for al, kk, rs in ((17, 2, 0), (17, 2, 1), (1, 16, 1), (1, 17, 0), (1, 17, 1)):
        assert lib.agx_mulrelin64(c19._h, bp, bp + 8 * 40 * 19 * N, bp + 8 * 40 * 19 * N, 1, bp + 8 * 80 * 19 * N,
                                  19, al, kk, rs, 1, None) == -2, (al, kk, rs)
    assert lib.agx_mulrelin64(c19._h, bp, bp + 8 * 40 * 19 * N, bp + 8 * 40 * 19 * N, 0, bp + 8 * 80 * 19 * N,
                              19, 1, 15, 1, 1, None) == 0                   # k + 1 = 16 is supported
    assert c19.launch_count() == l0


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_inputs_unchanged(ctx, form):
    import torch
    N = 4096
    c = ctx(N, QS + PS)
    rlk = dev(rand_key(3, QS + PS, N, 109))
    a, b = dev(ciphertexts(4, QS, N, 113)), dev(ciphertexts(4, QS, N, 127))
    snap = (a.clone(), b.clone(), rlk.clone())
    for rescale in (False, True):
        call(c, a, b, rlk, 2, 2, rescale, form)
        call(c, a, a, rlk, 2, 2, rescale, form)
    torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip((a, b, rlk), snap))


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    """The header's counts, the same for B = 1 and B = 6."""
    import torch
    x = int(N == 32768)
    c, c1 = ctx(N, QS + PS), ctx(N, QS + PS[:1])
    key = dev(rand_key(5, QS + PS, N, 131))
    k1 = key[:, :, :len(QS) + 1].contiguous()

    def launches(cx, B, alpha, k, rescale, form, rk=key, square=False):
        a = dev(ciphertexts(B, QS, N, 137))
        b = a if square else dev(ciphertexts(B, QS, N, 139))
        torch.cuda.synchronize()
        l0 = cx.launch_count()
        call(cx, a, b, rk, alpha, k, rescale, form)
        torch.cuda.synchronize()
        return cx.launch_count() - l0

    for B in (1, 6):
        for rs in (False, True):
            # alpha = 2: digits of 2, 2 and 1 primes (ModUps 3 + 3 + 2, one more each at N = 32768); product 1; inner 1;
            # ModDown 3 (4)
            assert launches(c, B, 2, 2, rs, True) == 1 + 8 + 3 * x + 1 + 3 + x
            # coefficient form: two forwards (one when squaring), the same, the inverse of the sums (2 at 32768) and one
            # coefficient-form ModDown
            assert launches(c, B, 2, 2, rs, False) == 2 + 1 + 8 + 3 * x + 1 + 1 + x + 1
            assert launches(c, B, 2, 2, rs, False, square=True) == 1 + 1 + 8 + 3 * x + 1 + 1 + x + 1
            # alpha = 5: one digit: 3 * dnum + 5 (4 * dnum + 6 at N = 32768), 3 * dnum + 6 in coefficient form
            assert launches(c, B, 5, 2, rs, True) == 8 + 2 * x
            assert launches(c, B, 5, 2, rs, False) == 9 + 2 * x
        # k = 1: without rescale the ModDown is the rescale (2; 3 at N = 32768), with it a two-prime ModDown (3; 4)
        assert launches(c1, B, 5, 1, False, True, k1) == 1 + 3 + x + 1 + 2 + x
        assert launches(c1, B, 5, 1, True, True, k1) == 1 + 3 + x + 1 + 3 + x
        assert launches(c1, B, 5, 1, False, False, k1) == 9 + 2 * x


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    c = ctx(N, QS + PS)
    key = rand_key(3, QS + PS, N, 149)
    ha, hb = ciphertexts(4, QS, N, 151), ciphertexts(4, QS, N, 157)
    want = recipe(ctx, c, dev(ha), dev(hb), dev(key), 2, 2, True, form)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        ins = []
        for h in (ha, hb, key):
            d = dev(h)
            t = torch.empty_like(d)
            t.copy_(d)                                                      # torch work the call must follow
            ins.append(t)
        out = empty(2, 4, len(QS) - 1, N)
    c.mulrelin(out, ins[0], ins[1], ins[2], 2, 2, rescale=True, ntt_form=form, stream=s)
    s.synchronize()
    assert torch.equal(out, want)
