"""u64 RNS hybrid key switching in one call (agx_keyswitch64, Context64.keyswitch).

Definition, for a context over Q_l u P (L = l + 1 + k primes, the k special primes last), alpha and a key
ksk[>= dnum][2][key_limbs][n] in evaluation form whose row map sends limb i <= l to row i and special prime t to row
key_limbs - k + t:
    out_c = ModDown_P( sum_j ModUp_j(digit_j) (.) ksk[j][c] ),   c = 0, 1,
digit j being limbs j*alpha .. min((j+1)*alpha, l+1) - 1 of the input, ModUp_j the centred lift of the digit's CRT
value, (.) the product of every limb with its key row and ModDown_P = floor((X + h_P) / P).

The CPU tests pin a big-integer oracle of that definition against the derivation of a gadget key switch (the result
decrypts within N |e| sum_j (D_j / 2) / P + (N + 1) / 2) and, with one digit, against a limb-by-limb ModUp / ModDown
composition; a further test checks the new kernels' resources on the compiled library.  The GPU tests compare the call
with the oracle and with the same recipe composed from public calls (key rows sliced and replicated), bit for bit, in
both forms, and cover digit shapes, one key at several levels, batch sharing, relinearisation, a rotation, refusals,
launch counts and side-stream ordering."""
import os
import random
import re
import shutil
import subprocess
from math import prod

import numpy as np
import pytest

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
SIZES = (4, 32, 512, 1024, 2048, 4096, 8192, 16384, 32768)


def find_primes(bits: int, count: int):
    """The `count` largest primes q < 2^bits of exactly `bits` bits with q = 1 (mod 2^16): usable at every N <= 32768."""
    out, q = [], (1 << bits) - (1 << 16) + 1
    while len(out) < count:
        if O.is_prime(q):
            out.append(q)
        q -= 1 << 16
    return out


PRIMES = {b: find_primes(b, 12) for b in (50, 60, 62)}
# Q_l: 5 mixed primes; P: 2 special primes.  alpha = 2 gives digits of 2, 2 and 1 primes (a partial last digit).
QS = [PRIMES[60][0], PRIMES[50][0], PRIMES[62][0], PRIMES[50][1], PRIMES[60][1]]
PS = [PRIMES[62][1], PRIMES[60][2]]
# 17 Q primes and 2 special primes: alpha = 1 makes 17 digits, more than one 128-bit lazy sum holds
Q17 = [PRIMES[(50, 60, 62)[i % 3]][2 + i // 3] for i in range(17)]
P17 = [PRIMES[62][9], PRIMES[60][9]]


# ---- big ints: the oracle
def crt(res, primes):
    Q = prod(primes)
    X = 0
    for r, q in zip(res, primes):
        m = Q // q
        X += int(r) * m * pow(m, -1, q)
    return X % Q


def negacyclic(a, b):
    """a * b mod X^N + 1 over the integers (lists of Python ints)"""
    N = len(a)
    c = [0] * N
    for i, x in enumerate(a):
        if x:
            for j, y in enumerate(b):
                if i + j < N:
                    c[i + j] += x * y
                else:
                    c[i + j - N] -= x * y
    return c


def digits_of(ell1, alpha):
    m = min(alpha, ell1)
    return [(f, min(m, ell1 - f)) for f in range(0, ell1, m)]


def key_rows(L, k, key_limbs):
    ell1 = L - k
    return list(range(ell1)) + [key_limbs - k + t for t in range(k)]


def keyswitch_oracle(d, kcoef, primes, k, alpha):
    """d [B][l+1][N] over primes[:l+1]; kcoef [D][2][key_limbs][N], the key in coefficient form (row r of the context
    limb it serves reduced mod that limb's prime) -> [2][B][l+1][N].  Works on big integers modulo QP throughout: the
    centred lift of each digit, the key's CRT value, the negacyclic products summed mod QP, then floor((X + h_P) / P)."""
    L = len(primes)
    ell1 = L - k
    Q, P, QP = prod(primes[:ell1]), prod(primes[ell1:]), prod(primes)
    rows = key_rows(L, k, kcoef.shape[2])
    B, N = d.shape[0], d.shape[2]
    out = np.empty((2, B, ell1, N), dtype=np.uint64)
    keys = [[[crt([kcoef[j, c, rows[i], x] for i in range(L)], primes) for x in range(N)] for c in (0, 1)]
            for j in range(len(digits_of(ell1, alpha)))]
    for b in range(B):
        acc = [[0] * N, [0] * N]
        for j, (f, cnt) in enumerate(digits_of(ell1, alpha)):
            src = primes[f:f + cnt]
            S = prod(src)
            h = (S - 1) // 2
            U = [(crt(d[b, f:f + cnt, x], src) + h) % S - h for x in range(N)]
            for c in (0, 1):
                acc[c] = [(u + v) % QP for u, v in zip(acc[c], negacyclic(U, keys[j][c]))]
        for c in (0, 1):
            Y = [((X + (P - 1) // 2) // P) % Q for X in acc[c]]
            for i, q in enumerate(primes[:ell1]):
                out[c, b, i] = [y % q for y in Y]
    return out


def limbwise_one_digit(d, kcoef, primes, k):
    """dnum = 1 by the limb-by-limb route: ModUp of the whole input, the negacyclic product mod each q_i with the key row,
    then ModDown of each coefficient's residues."""
    L = len(primes)
    ell1 = L - k
    Q, P = prod(primes[:ell1]), prod(primes[ell1:])
    rows = key_rows(L, k, kcoef.shape[2])
    B, N = d.shape[0], d.shape[2]
    h = (Q - 1) // 2
    out = np.empty((2, B, ell1, N), dtype=np.uint64)
    for b in range(B):
        Xc = [(crt(d[b, :, x], primes[:ell1]) + h) % Q - h for x in range(N)]
        for c in (0, 1):
            res = [[v % q for v in negacyclic([x % q for x in Xc], [int(w) for w in kcoef[0, c, rows[i]]])]
                   for i, q in enumerate(primes)]
            Y = [((crt([res[i][x] for i in range(L)], primes) + (P - 1) // 2) // P) % Q for x in range(N)]
            for i, q in enumerate(primes[:ell1]):
                out[c, b, i] = [y % q for y in Y]
    return out


def ternary(rng, N):
    return [rng.choice((-1, 0, 1)) for _ in range(N)]


def small(rng, N, bound):
    return [rng.randint(-bound, bound) for _ in range(N)]


def gadget_key_coeff(primes, k, alpha, ell1_key, s, s2, ebound, rng):
    """ksk_j = (-a_j s + e_j + [i in D_j] (P mod q_i) s', a_j) over `primes` (the key's own basis, special primes last,
    digits of Q_top = its first ell1_key primes), in coefficient form: [dnum][2][len(primes)][N]."""
    N, Lk = len(s), len(primes)
    P = prod(primes[Lk - k:])
    digits = digits_of(ell1_key, alpha)
    out = np.empty((len(digits), 2, Lk, N), dtype=np.uint64)
    for j, (f, cnt) in enumerate(digits):
        a = [rng.randrange(1 << 62) for _ in range(N)]
        e = small(rng, N, ebound)
        for i, q in enumerate(primes):
            a_i = [x % q for x in a]
            as_ = negacyclic(a_i, [x % q for x in s])
            g = (P % q) if f <= i < f + cnt else 0
            out[j, 0, i] = [(-u + v + g * w) % q for u, v, w in zip(as_, e, s2)]
            out[j, 1, i] = a_i
    return out


def residual(out, d, s, s2, qs):
    """max |c0 + c1 s - d s'| over the coefficients, centred mod Q (out [2][1][l+1][N], d [1][l+1][N] residues)"""
    Q, N = prod(qs), d.shape[2]
    c0 = [crt(out[0, 0, :, x], qs) for x in range(N)]
    c1 = [crt(out[1, 0, :, x], qs) for x in range(N)]
    dd = [crt(d[0, :, x], qs) for x in range(N)]
    r = [(u + v - w) % Q for u, v, w in zip(c0, negacyclic(c1, s), negacyclic(dd, s2))]
    return max(min(v, Q - v) for v in r)


def ks_bound(qs, ps, alpha, N, ebound):
    P = prod(ps)
    return N * ebound * sum(prod(qs[f:f + c]) // 2 for f, c in digits_of(len(qs), alpha)) // P + (N + 1) // 2 + 1


def rand_res(B, primes, N, rng):
    return np.array([[[rng.randrange(q) for _ in range(N)] for q in primes] for _ in range(B)], dtype=np.uint64)


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("N,qs,ps,alpha", [
    (8, QS[:3], PS, 1), (16, QS, PS, 2), (32, QS[:4], PS[:1] + [PRIMES[62][2]], 3), (64, QS[:2], PS[:1], 5)])
def test_oracle_is_a_key_switch(N, qs, ps, alpha):
    """With a gadget key for s', the oracle's (c0, c1) satisfies c0 + c1 s - d s' = small (mod Q_l) within the bound."""
    rng = random.Random(N * 7 + alpha)
    primes, k = qs + ps, len(ps)
    s, s2 = ternary(rng, N), small(rng, N, 3)
    ebound = 6
    kc = gadget_key_coeff(primes, k, alpha, len(qs), s, s2, ebound, rng)
    d = rand_res(1, qs, N, rng)
    out = keyswitch_oracle(d, kc, primes, k, alpha)
    bound = ks_bound(qs, ps, alpha, N, ebound)
    assert bound < prod(qs) >> 40
    assert residual(out, d, s, s2, qs) <= bound
    # a wrong s' leaves a residual of the size of Q
    assert residual(out, d, s, [x + 1 for x in s2], qs) > prod(qs) >> 20


@pytest.mark.parametrize("N,qs,ps,key_extra", [(8, QS[:3], PS, 0), (16, QS[:2], PS, 2), (32, QS, PS[:1], 1)])
def test_oracle_one_digit_is_modup_then_moddown(N, qs, ps, key_extra):
    """dnum = 1: the oracle equals ModUp of the input, the limb products with the key rows, and ModDown, limb by limb;
    key rows beyond l + 1 and before the special rows are not read."""
    rng = random.Random(N + key_extra)
    primes, k = qs + ps, len(ps)
    rows = key_rows(len(primes), k, len(primes) + key_extra)
    kc = np.zeros((1, 2, len(primes) + key_extra, N), dtype=np.uint64)
    for i, r in enumerate(rows):
        kc[0, :, r] = [[rng.randrange(primes[i]) for _ in range(N)] for _ in (0, 1)]
    d = rand_res(2, qs, N, rng)
    for alpha in (len(qs), len(qs) + 3):
        assert (keyswitch_oracle(d, kc, primes, k, alpha) == limbwise_one_digit(d, kc, primes, k)).all()


def _cuobjdump(*args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import agilex_ntt_b200 as A
    return subprocess.run([exe, *args, A.build.build_lib()], capture_output=True, text=True, check=True).stdout


def test_keyswitch_kernels_use_no_local_memory():
    """Every instantiation of the key inner product (1, 2, 4 and 8 digits per chunk) is in the sm_100a code and runs
    without local memory or stack."""
    usage = _cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*keyswitch\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    assert sorted(re.search(r"ILi(\d+)E", n).group(1) for n, *_ in found) == ["1", "2", "4", "8"]
    for name, reg, stack, local in found:
        assert int(local) == 0 and int(stack) == 0, name


# ------------------------------------------------------------------------------------------ on a GPU

def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(np.uint64)


def data(B, primes, N, seed):
    """[B][L][N] words, limb l uniform below q_l."""
    mods = np.array(primes, dtype=np.uint64).reshape(1, len(primes), 1)
    return O.synthetic_u64(B * len(primes) * N, seed, (1 << 64) - 1).reshape(B, len(primes), N) % mods


def rns_fwd(x, primes, psis=None):
    """per-limb forward of [..][L][N] on the CPU (the C restatement of the reference's forward)"""
    N = x.shape[-1]
    flat = x.reshape(-1, len(primes), N)
    out = np.empty_like(flat)
    for l, q in enumerate(primes):
        tw, pre = O.tables_u64(N, q, psis[l] if psis else None)
        v = np.ascontiguousarray(flat[:, l, :])
        out[:, l, :] = O.ref_fwd_u64(v, v, q, tw, pre, v.shape[0]).reshape(flat.shape[0], N)
    return out.reshape(x.shape)


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


def caller_roots(N, primes):
    return [O.primitive_roots_2n(N, q, 2)[1] for q in primes]        # non-minimal roots


def empty(*shape):
    import torch
    return torch.empty(shape, dtype=torch.int64, device="cuda")


def rand_key(D, key_primes, N, seed):
    """[D][2][key_limbs][N], row r uniform below key_primes[r] (a key is uniform in evaluation form)"""
    return data(2 * D, key_primes, N, seed).reshape(D, 2, len(key_primes), N)


def recipe(c, d_in, ksk, alpha, k, form):
    """The key switch composed from public calls: each digit copied out and extended by modup, the key rows sliced out
    and replicated over the batch, products accumulated by elementwise mul / mac (evaluation form) or
    polymul_by_spectrum and add (coefficient form), then moddown of each component."""
    import torch
    L, N, B = c.L, c.n, d_in.shape[0]
    ell1 = L - k
    kr = torch.cat([ksk[:, :, :ell1], ksk[:, :, ksk.shape[2] - k:]], dim=2)
    acc = [empty(B, L, N), empty(B, L, N)]
    for j, (f, cnt) in enumerate(digits_of(ell1, alpha)):
        U = empty(B, L, N)
        c.modup(U, d_in[:, f:f + cnt].contiguous(), f, cnt, ntt_form=form)
        for cc in (0, 1):
            kk = kr[j, cc].expand(B, L, N).contiguous()
            if form:
                c.elementwise("mul" if j == 0 else "mac", acc[cc], U, kk)
            elif j == 0:
                c.polymul_by_spectrum(acc[cc], U, kk)
            else:
                t = empty(B, L, N)
                c.polymul_by_spectrum(t, U, kk)
                c.elementwise("add", acc[cc], acc[cc], t)
    out = empty(2, B, ell1, N)
    for cc in (0, 1):
        c.moddown(out[cc], acc[cc], k, ntt_form=form)
    return out


def call(c, d_in, ksk, alpha, k, form, stream=None):
    out = empty(2, d_in.shape[0], c.L - k, c.n)
    return c.keyswitch(out, d_in, ksk, alpha, k, ntt_form=form, stream=stream)


@gpu
@pytest.mark.parametrize("roots", ("minimal", "caller"))
@pytest.mark.parametrize("N,alpha,k,key_extra", [(8, 2, 2, 0), (32, 2, 1, 1), (64, 3, 2, 2), (16, 9, 2, 0)])
def test_vs_oracle(ctx, N, alpha, k, key_extra, roots):
    """Both forms against the big-integer oracle at small n, with key rows that the map must skip."""
    import torch
    qs, ps = QS, PS[:k]
    primes = qs + ps
    psis = caller_roots(N, primes) if roots == "caller" else None
    c = ctx(N, primes, psis)
    rng = random.Random(N + alpha + k)
    dnum = len(digits_of(len(qs), alpha))
    key_primes = qs + [PRIMES[50][9 + t] for t in range(key_extra)] + ps
    kc = np.stack([rand_res(2, key_primes, N, rng) for _ in range(dnum + 1)])       # one digit more than read
    kpsis = None
    if psis:
        kpsis = psis[:len(qs)] + [None] * key_extra + psis[len(qs):]
    ksk = dev(rns_fwd(kc, key_primes, kpsis))
    d = data(3, qs, N, 11 + N)
    want = keyswitch_oracle(d, kc, primes, k, alpha)
    got = call(c, dev(d), ksk, alpha, k, False)
    assert (host(got) == want).all()
    qpsis = psis[:len(qs)] if psis else None
    got = call(c, dev(rns_fwd(d, qs, qpsis)), ksk, alpha, k, True)
    torch.cuda.synchronize()
    assert (host(got) == rns_fwd(want, qs, qpsis)).all()


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_vs_composed_recipe(ctx, N, form):
    """Three digits (2, 2 and 1 primes), k = 2, a key with two extra rows: equal to the public-call recipe with the key
    rows sliced and replicated, bit for bit, at every geometry."""
    import torch
    primes = QS + PS
    c = ctx(N, primes)
    key_primes = QS + [PRIMES[50][10], PRIMES[50][11]] + PS
    ksk = dev(rand_key(3, key_primes, N, 5 + N))
    d_in = dev(data(2, QS, N, 7 + N))
    got = call(c, d_in, ksk, 2, 2, form)
    want = recipe(c, d_in, ksk, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(got, want)


@gpu
@pytest.mark.parametrize("N", (32, 1024, 32768))
def test_caller_roots(ctx, N):
    """Under caller roots the call equals the recipe (both forms), and the evaluation form is fwd of the coefficient form
    applied to inv of the input."""
    import torch
    primes = QS + PS
    psis = caller_roots(N, primes)
    c, lower = ctx(N, primes, psis), ctx(N, QS, psis[:len(QS)])
    ksk = dev(rand_key(3, primes, N, 21 + N))
    d_in = dev(data(2, QS, N, 23 + N))
    for form in (False, True):
        assert torch.equal(call(c, d_in, ksk, 2, 2, form), recipe(c, d_in, ksk, 2, 2, form)), form
    spec = call(c, d_in, ksk, 2, 2, True)
    t = d_in.clone()
    lower.inv(t)
    coeff = call(c, t, ksk, 2, 2, False)
    lower.fwd(coeff)
    torch.cuda.synchronize()
    assert torch.equal(spec, coeff)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (32, 4096))
@pytest.mark.parametrize("shape", ("alpha1_dnum17", "one_digit", "alpha_above", "partial_last", "k1"))
def test_digit_shapes(ctx, N, form, shape):
    """alpha = 1 with l + 1 = 17 (17 digits: the lazy sums fold), alpha = l + 1 and alpha > l + 1 (one digit), a partial
    last digit (5 = 3 + 2), and k = 1 (the ModDown is the rescale)."""
    import torch
    qs, ps, alpha = {"alpha1_dnum17": (Q17, P17, 1), "one_digit": (QS, PS, 5), "alpha_above": (QS, PS, 40),
                     "partial_last": (QS, PS, 3), "k1": (QS, PS[:1], 2)}[shape]
    primes = qs + ps
    c = ctx(N, primes)
    dnum = len(digits_of(len(qs), alpha))
    ksk = dev(rand_key(dnum, primes, N, 31 + N))
    d_in = dev(data(3, qs, N, 37 + N))
    got = call(c, d_in, ksk, alpha, len(ps), form)
    torch.cuda.synchronize()
    assert torch.equal(got, recipe(c, d_in, ksk, alpha, len(ps), form))


def gadget_key_gpu(ctx_top, key_primes, k, alpha, ell1_top, s, s2, ebound, rng):
    """The gadget key over Q_top u P, built with the library's products and transformed: [dnum][2][key_limbs][N]."""
    import torch
    N, Lk = ctx_top.n, len(key_primes)
    P = prod(key_primes[Lk - k:])
    res = lambda v: dev(np.array([[x % q for x in v] for q in key_primes], dtype=np.uint64).reshape(1, Lk, N))
    d_s, d_s2 = res(s), res(s2)
    keys = []
    for f, cnt in digits_of(ell1_top, alpha):
        a = dev(data(1, key_primes, N, rng.randrange(1 << 30)))
        k0 = empty(1, Lk, N)
        ctx_top.polymul(k0, a, d_s)
        ctx_top.elementwise("sub", k0, res(small(rng, N, ebound)), k0)
        g = dev(np.array([[(P % q) if f <= i < f + cnt else 0] * N for i, q in enumerate(key_primes)],
                         dtype=np.uint64).reshape(1, Lk, N))
        ctx_top.elementwise("mul", g, g, d_s2)
        ctx_top.elementwise("add", k0, k0, g)
        ctx_top.fwd(k0)
        ctx_top.fwd(a)
        keys.append(torch.stack([k0[0], a[0]]))
    return torch.stack(keys).contiguous()


@gpu
@pytest.mark.parametrize("N", (1024,))
def test_one_key_at_three_levels(ctx, N):
    """One gadget key over Q_top u P (key_limbs = 7 + 2), alpha = 3 fixed, used unchanged at l + 1 = 7, 5 and 2: each
    level equals its own sliced-key recipe in both forms and decrypts within the key switch's bound."""
    import torch
    qtop = QS + [PRIMES[62][3], PRIMES[50][3]]
    key_primes = qtop + PS
    k, alpha = len(PS), 3
    rng = random.Random(5)
    s, s2 = ternary(rng, N), ternary(rng, N)
    ebound = 8
    ksk = gadget_key_gpu(ctx(N, key_primes), key_primes, k, alpha, len(qtop), s, s2, ebound, rng)
    for ell1 in (7, 5, 2):
        qs = qtop[:ell1]
        c = ctx(N, qs + PS)
        d = data(1, qs, N, 40 + ell1)
        d_in = dev(d)
        got = call(c, d_in, ksk, alpha, k, False)
        assert torch.equal(got, recipe(c, d_in, ksk, alpha, k, False)), ell1
        spec = dev(d)
        ctx(N, qs).fwd(spec)
        assert torch.equal(call(c, spec, ksk, alpha, k, True), recipe(c, spec, ksk, alpha, k, True)), ell1
        bound = ks_bound(qs, PS, alpha, N, ebound)
        assert bound < prod(qs) >> 40
        assert residual(host(got), d, s, s2, qs) <= bound, ell1


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_one_key_on_a_batch_is_single_calls(ctx, form):
    import torch
    N = 2048
    c = ctx(N, QS + PS)
    ksk = dev(rand_key(3, QS + PS, N, 51))
    d_in = dev(data(5, QS, N, 53))
    got = call(c, d_in, ksk, 2, 2, form)
    for b in range(5):
        one = call(c, d_in[b:b + 1].contiguous(), ksk, 2, 2, form)
        assert torch.equal(got[:, b:b + 1], one), b


@gpu
@pytest.mark.parametrize("N", (512, 16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """More than two waves of CTAs in every forward geometry (radix-2, frame, split frame) and more polynomials than
    one slice of the inner product: equal to the recipe in both forms."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = -(-(2 * sms + 5) // len(QS))
    c = ctx(N, QS + PS)
    ksk = dev(rand_key(3, QS + PS, N, 61))
    d_in = dev(data(B, QS, N, 67 + N))
    for form in (False, True):
        got = call(c, d_in, ksk, 2, 2, form)
        assert torch.equal(got, recipe(c, d_in, ksk, 2, 2, form)), form
        del got
        torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_relinearisation(ctx, form):
    """The product of two ciphertexts (b_i, a_i), b_i = -a_i s + m_i + e_i, has d2 = a1 a2 on s^2; switching d2 with a
    key for s' = s^2 gives (c0, c1) with c0 + c1 s - d2 s^2 within the key switch's bound, so (d0 + c0, d1 + c1)
    decrypts like (d0, d1, d2)."""
    import torch
    N = 1024
    qs, alpha, k = QS, 2, len(PS)
    rng = random.Random(71)
    s = ternary(rng, N)
    s2 = negacyclic(s, s)                                              # s^2 over the integers (|coefficients| <= N)
    ebound = 8
    key_primes = qs + PS
    ksk = gadget_key_gpu(ctx(N, key_primes), key_primes, k, alpha, len(qs), s, s2, ebound, rng)
    cq, c = ctx(N, qs), ctx(N, key_primes)
    a1, a2 = dev(data(1, qs, N, 73)), dev(data(1, qs, N, 79))
    d2 = empty(1, len(qs), N)
    cq.polymul(d2, a1, a2)
    d = host(d2)
    inp = d2.clone()
    if form:
        cq.fwd(inp)
    got = call(c, inp, ksk, alpha, k, form)
    if form:
        cq.inv(got[0])
        cq.inv(got[1])
    assert residual(host(got), d, s, s2, qs) <= ks_bound(qs, PS, alpha, N, ebound)


@gpu
@pytest.mark.parametrize("step", (1, -3))
def test_rotation_end_to_end(A, ctx, step):
    """A rotation from automorph + keyswitch: (sigma(b), sigma(a)) decrypts under sigma(s); switching sigma(a) with a key
    for s' = sigma(s) gives c0 + c1 s - sigma(a) sigma(s) within the bound, in both forms, and the two forms agree."""
    import torch
    N = 1024
    qs, alpha, k = QS, 3, len(PS)
    g = A.galois_element(N, step)
    rng = random.Random(83 + step)
    s = ternary(rng, N)
    sg = [0] * N
    for i, v in enumerate(s):                                          # sigma_g(s): X^i -> X^(i g) mod X^N + 1
        e = i * g % (2 * N)
        sg[e % N] += v if e < N else -v
    ebound = 8
    key_primes = qs + PS
    ksk = gadget_key_gpu(ctx(N, key_primes), key_primes, k, alpha, len(qs), s, sg, ebound, rng)
    cq, c = ctx(N, qs), ctx(N, key_primes)
    a = dev(data(1, qs, N, 89))
    ra = empty(1, len(qs), N)
    cq.automorph(ra, a, g, ntt_form=False)
    coeff = call(c, ra, ksk, alpha, k, False)
    assert residual(host(coeff), host(ra), s, sg, qs) <= ks_bound(qs, PS, alpha, N, ebound)
    a_hat = a.clone()
    cq.fwd(a_hat)
    ra_hat = empty(1, len(qs), N)
    cq.automorph(ra_hat, a_hat, g, ntt_form=True)
    spec = call(c, ra_hat, ksk, alpha, k, True)
    cq.inv(spec[0])
    cq.inv(spec[1])
    torch.cuda.synchronize()
    assert torch.equal(spec, coeff)


@gpu
def test_refusals_and_empty_batches(A, ctx):
    import torch
    N = 1024
    lib = A.lib()
    primes = QS + PS
    L, ell1 = len(primes), len(QS)
    c, c19 = ctx(N, primes), ctx(N, Q17 + P17)
    x = dev(data(2, QS, N, 3))
    ksk = dev(rand_key(3, primes, N, 4))
    xs, ks = x.clone(), ksk.clone()
    o = empty(2, 2, ell1, N)
    pi, po, pk = x.data_ptr(), o.data_ptr(), ksk.data_ptr()
    big = torch.zeros(16 * L * N, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    dup = A.Context64(N, [QS[0], QS[1], QS[0], PS[0]])                       # equal Q primes: refused here
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    ctxs = (c, c19, dup)
    kw = 3 * 2 * L * N                                                         # words of the three key digits read
    try:
        for form in (0, 1):
            invalid = [
                (c32._h, po, pi, 2, pk, L, 2, 2),                              # u32 context
                (c._h, None, pi, 2, pk, L, 2, 2), (c._h, po, None, 2, pk, L, 2, 2), (c._h, po, pi, 2, None, L, 2, 2),
                (c._h, po + 8, pi, 1, pk, L, 2, 2), (c._h, po, pi + 8, 1, pk, L, 2, 2), (c._h, po, pi, 1, pk + 8, L, 2, 2),
                (c._h, po, pi, 2, pk, L, 2, 0), (c._h, po, pi, 2, pk, L, 2, L),    # k = 0, k = L
                (c._h, po, pi, 2, pk, L, 0, 2),                                # alpha = 0
                (c._h, po, pi, 2, pk, L - 1, 2, 2),                            # key_limbs < L
                (dup._h, po, pi, 2, pk, 4, 1, 1),                              # two equal primes
                (c._h, po, pi, 0x7fffffff // (2 * L) + 1, pk, L, 9, 2),        # 2 * B * L > 2^31 - 1 (dnum = 1)
                (c._h, po, pi, 0x7fffffff // (3 * L) + 1, pk, L, 2, 2),        # dnum * B * L > 2^31 - 1
                (c._h, pi, pi, 2, pk, L, 2, 2),                                # out on in
                (c._h, bp + 8 * (2 * ell1 * N - 2), bp, 2, pk, L, 2, 2),       # in's last 16 bytes are out's first
                (c._h, bp, bp + 8 * (4 * ell1 * N - 2), 2, pk, L, 2, 2),       # out's last 16 bytes are in's first
                (c._h, bp + 8 * (kw - 2), pi, 2, bp, L, 2, 2),                 # out starts in the last key digit read
                (c._h, bp, pi, 2, bp + 8 * (4 * ell1 * N - 2), L, 2, 2),       # the key starts in out
            ]
            for h, o_, i_, B, k_, kl, al, kk in invalid:
                l0 = [t.launch_count() for t in ctxs]
                assert lib.agx_keyswitch64(h, o_, i_, B, k_, kl, al, kk, form, None) == -1, (form, B, kl, al, kk)
                assert [t.launch_count() for t in ctxs] == l0
            for al, kk in ((17, 2), (16, 17)):                                 # 17 digit primes; k = 17
                l0 = c19.launch_count()
                assert lib.agx_keyswitch64(c19._h, bp, bp + 8 * 34 * N, 1, pk, 19, al, kk, form, None) == -2, (al, kk)
                assert c19.launch_count() == l0
            l0 = c.launch_count()
            for o_, i_, k_ in ((None, None, None), (po, pi, pk), (bp, bp + 16, bp)):      # B == 0
                assert lib.agx_keyswitch64(c._h, o_, i_, 0, k_, L, 2, 2, form, None) == 0
            assert c.launch_count() == l0
            # adjacent, not overlapping: allowed; a key digit that is not read may overlap
            assert lib.agx_keyswitch64(c._h, bp + 8 * kw, pi, 2, bp, L, 2, 2, form, None) == 0
            assert lib.agx_keyswitch64(c._h, bp + 8 * 2 * L * N, pi, 2, bp, L, 9, 2, form, None) == 0
        bad = [
            lambda: c.keyswitch(empty(2, 1, ell1, N), x, ksk, 2, 2),           # out batch
            lambda: c.keyswitch(empty(2, 2, ell1 + 1, N), x, ksk, 2, 2),
            lambda: c.keyswitch(o, x, ksk, 0, 2),                              # alpha = 0
            lambda: c.keyswitch(o, x, ksk, 1 << 32, 2),
            lambda: c.keyswitch(o, x, ksk, 2, 0),                              # k = 0
            lambda: c.keyswitch(o, x, ksk[:2], 2, 2),                          # fewer key digits than dnum
            lambda: c.keyswitch(o, x, ksk[:, :, :L - 1].contiguous(), 2, 2),   # key_limbs < L
            lambda: c.keyswitch(o, x, ksk[:, :1].contiguous(), 2, 2),          # one component
            lambda: c.keyswitch(o, x.cpu(), ksk, 2, 2),                        # host tensor
        ]
        for fn in bad:
            with pytest.raises(ValueError):
                fn()
        with pytest.raises(A.AgxError) as e:
            c.keyswitch(ksk.view(-1)[:2 * 2 * ell1 * N].view(2, 2, ell1, N), x, ksk, 2, 2)   # out inside the key
        assert e.value.code == -1
        torch.cuda.synchronize()
        assert torch.equal(x, xs) and torch.equal(ksk, ks)
    finally:
        for t in (dup, c32):
            t.close()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_inputs_unchanged(ctx, form):
    import torch
    N = 4096
    c = ctx(N, QS + PS)
    ksk = dev(rand_key(3, QS + PS, N, 91))
    d_in = dev(data(4, QS, N, 93))
    ks, xs = ksk.clone(), d_in.clone()
    call(c, d_in, ksk, 2, 2, form)
    torch.cuda.synchronize()
    assert torch.equal(d_in, xs) and torch.equal(ksk, ks)


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    import torch
    big = N == 32768
    c, c1 = ctx(N, QS + PS), ctx(N, QS + PS[:1])
    ksk = dev(rand_key(5, QS + PS, N, 97))
    d_in = dev(data(2, QS, N, 99))

    def launches(cx, fn):
        l0 = cx.launch_count()
        fn()
        torch.cuda.synchronize()
        return cx.launch_count() - l0

    x = int(big)
    # alpha = 2: digits of 2, 2, 1 primes (ModUps 3 + 3 + 2, one more each at N = 32768); inner 1; ModDown 3 (4)
    assert launches(c, lambda: call(c, d_in, ksk, 2, 2, True)) == 8 + 3 * x + 1 + 3 + x
    assert launches(c, lambda: call(c, d_in, ksk, 2, 2, False)) == 3 + 4 + x
    # alpha = 5: one digit: 3 + 1 + 3 = 3 * dnum + 4
    assert launches(c, lambda: call(c, d_in, ksk, 5, 2, True)) == 7 + 2 * x
    assert launches(c, lambda: call(c, d_in, ksk, 5, 2, False)) == 5 + x
    # alpha = 1: five one-prime digits (2 each) + 1 + 3
    assert launches(c, lambda: call(c, d_in, ksk, 1, 2, True)) == 10 + 5 * x + 1 + 3 + x
    # k = 1: the ModDown is the rescale (2; 3 at N = 32768)
    k1 = ksk[:, :, :len(QS) + 1].contiguous()
    assert launches(c1, lambda: call(c1, d_in, k1, 5, 1, True)) == 3 + x + 1 + 2 + x
    assert launches(c1, lambda: call(c1, d_in, k1, 5, 1, False)) == 5 + x
    for form in (False, True):
        assert launches(c, lambda: call(c, d_in[:0], ksk, 2, 2, form)) == 0


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    c = ctx(N, QS + PS)
    k = rand_key(3, QS + PS, N, 101)
    x = data(4, QS, N, 103)
    want = recipe(c, dev(x), dev(k), 2, 2, form)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_x, d_k = dev(x), dev(k)
        d_in, ksk = torch.empty_like(d_x), torch.empty_like(d_k)
        d_in.copy_(d_x)                                                 # torch work the call must follow
        ksk.copy_(d_k)
        out = empty(2, 4, len(QS), N)
    c.keyswitch(out, d_in, ksk, 2, 2, ntt_form=form, stream=s)
    s.synchronize()
    assert torch.equal(out, want)
