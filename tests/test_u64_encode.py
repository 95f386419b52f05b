"""u64 RNS CKKS encoding and decoding (agx_encode64 / agx_decode64, Context64.encode / decode).

Conventions: n = 2^logn, S = n / 2 slots, zeta = exp(i pi / n), slot j of a real polynomial m is m(zeta^(5^j mod 2n)),
and encoding is the inverse with real coefficients, m_i = (2 / n) sum_j Re(z_j zeta^(-i 5^j)).  The numpy oracle needs
no special FFT: with w_(5^j) = z_j and w_(-5^j mod 2n) = conj(z_j) on the odd indices of a length-2n array,
m = Re(exp(-i pi i / n) fft(w[1::2]) / n).  Under these conventions agx_automorph64 with g = 5^r maps z to roll(z, -r)
and g = 2n - 1 conjugates every slot; the CPU tests pin both on the oracle, and the GPU tests check them through the
library's own calls, in the clear and encrypted.

Error bounds (DESIGN.md s.4, u = 2^-53, kappa = 5):
- encode: |c_i - scale m_i| <= 1/2 + scale ||z||_inf kappa log2(n) u;
- decode, CRT step: |m_i - X_c / scale| <= (2 limbs + 1) u |X_c / scale|;
- decode, FFT: |z~_j - z_j| <= kappa log2(n) u S ||m||_inf.
The FP64 numpy oracle carries an error of the same form, so the tests comparing against it allow twice kappa; kappa = 5
itself is asserted against a 60-digit mpmath oracle at n <= 256 (test_encode_bound_with_kappa_5,
test_decode_fft_bound_with_kappa_5)."""
import math
import random
import re
from fractions import Fraction
from math import prod

import numpy as np
import pytest

import test_u64_automorph as AM
import test_u64_keyswitch as KS
import test_u64_lintrans as LT
import test_u64_mulrelin as MR

gpu = pytest.mark.gpu
SIZES = KS.SIZES
QS, PS = KS.QS, KS.PS
U = 2.0 ** -53
KAPPA = 5


# ---- the oracle
def rot_group(n):
    return np.array([pow(5, j, 2 * n) for j in range(n // 2)], dtype=np.int64)


def oracle_encode(z, n):
    """z [..][S] complex -> m [..][n] real (float64)"""
    z = np.asarray(z, dtype=np.complex128)
    g = rot_group(n)
    w = np.zeros(z.shape[:-1] + (2 * n,), dtype=np.complex128)
    w[..., g] = z
    w[..., (-g) % (2 * n)] = np.conj(z)
    i = np.arange(n)
    return (np.exp(-1j * np.pi * i / n) * np.fft.fft(w[..., 1::2], axis=-1) / n).real


def oracle_decode(m, n):
    """m [..][n] real -> z [..][S]: m evaluated at zeta^(5^j)"""
    i = np.arange(n)
    vals = n * np.fft.ifft(np.asarray(m, dtype=np.float64) * np.exp(1j * np.pi * i / n), axis=-1)   # m(zeta^(2t+1))
    return vals[..., (rot_group(n) - 1) // 2]


def direct_encode(z, n):
    g = rot_group(n)
    i = np.arange(n).reshape(-1, 1)
    return (2.0 / n) * (np.asarray(z).reshape(1, -1) * np.exp(-1j * np.pi * i * g.reshape(1, -1) / n)).real.sum(1)


def direct_decode(m, n):
    g = rot_group(n)
    i = np.arange(n).reshape(1, -1)
    return (np.asarray(m).reshape(1, -1) * np.exp(1j * np.pi * g.reshape(-1, 1) * i / n)).sum(1)


def encode_ints(z, n, scale):
    """c_i = rint(fl(scale * m_i)) from the oracle's m (Python round: half to even)"""
    return [round(float(scale) * float(x)) for x in oracle_encode(z, n)]


def residue_of(c, q):
    return c % q


def crt_centred(res, primes):
    Q = prod(primes)
    X = KS.crt(res, primes)
    return X - Q if X > (Q - 1) // 2 else X


def rand_slots(rng, B, S, r=1.0):
    return (rng.uniform(-r, r, (B, S)) + 1j * rng.uniform(-r, r, (B, S))).astype(np.complex128)


def enc_tol(scale, z, n, kappa=2 * KAPPA):
    return 0.5 + scale * np.abs(z).max() * kappa * math.log2(n) * U


def dec_tol(m_inf, n, limbs, kappa=2 * KAPPA):
    return (n // 2) * m_inf * U * (kappa * math.log2(n) + math.sqrt(2) * (2 * limbs + 1)) + 1e-300


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("n", (4, 8, 16, 64, 256))
def test_oracle_is_the_definition(n):
    """The numpy-FFT oracle equals the O(n^2) definitions, both directions, and they invert each other."""
    rng = np.random.default_rng(n)
    z = rand_slots(rng, 1, n // 2)[0]
    m = oracle_encode(z, n)
    assert np.abs(m - direct_encode(z, n)).max() < 1e-12
    assert np.abs(oracle_decode(m, n) - z).max() < 1e-12
    mm = rng.normal(size=n)
    assert np.abs(oracle_decode(mm, n) - direct_decode(mm, n)).max() < 1e-9 * n


@pytest.mark.parametrize("n", (4, 16, 64))
def test_oracle_matches_mpmath(n):
    """At 50 digits: m_i = (2/n) sum_j Re(z_j zeta^(-i 5^j)) and z_j = m(zeta^(5^j))."""
    import mpmath
    mpmath.mp.dps = 50
    rng = np.random.default_rng(n + 1)
    z = rand_slots(rng, 1, n // 2)[0]
    m = oracle_encode(z, n)
    zeta = mpmath.exp(1j * mpmath.pi / n)
    g = rot_group(n)
    for i in range(n):
        want = 2 * sum((mpmath.mpc(complex(zj)) * zeta ** (-i * int(gj))).real for zj, gj in zip(z, g)) / n
        assert abs(float(want) - m[i]) < 1e-14
    for j in range(n // 2):
        want = sum(mpmath.mpf(float(x)) * zeta ** (int(g[j]) * i) for i, x in enumerate(m))
        assert abs(complex(want) - z[j]) < 1e-13


@pytest.mark.parametrize("n", (4, 8, 32, 256))
def test_rotation_and_conjugation_act_on_slots(n):
    """On the oracle: sigma_(5^r) (automorph_ints) maps the slots z to roll(z, -r); sigma_(2n-1) to conj(z)."""
    rng = np.random.default_rng(3 * n)
    S = n // 2
    z = rand_slots(rng, 1, S, 100.0)[0]
    m = encode_ints(z, n, 2.0 ** 30)
    for r in (1, -3, S - 1):
        got = oracle_decode(np.array(AM.automorph_ints(m, pow(5, r, 2 * n)), dtype=np.float64), n) / 2.0 ** 30
        assert np.abs(got - np.roll(z, -r)).max() < 1e-4
    got = oracle_decode(np.array(AM.automorph_ints(m, 2 * n - 1), dtype=np.float64), n) / 2.0 ** 30
    assert np.abs(got - np.conj(z)).max() < 1e-4


def test_big_integer_oracles():
    """The double -> residue map (Python round of the float product is half to even) and the centred CRT."""
    primes = KS.find_primes(60, 3)
    Q = prod(primes)
    assert round(2.5) == 2 and round(3.5) == 4 and round(-2.5) == -2
    for c in (0, 1, -1, 2 ** 53 + 2, -(2 ** 63), 2 ** 64, 3 * 2 ** 100, -(2 ** 120) + 2 ** 70):
        assert float(c) == c
        res = [residue_of(c, q) for q in primes]
        assert crt_centred(res, primes) == c
    h = (Q - 1) // 2
    assert crt_centred([h % q for q in primes], primes) == h
    assert crt_centred([(h + 1) % q for q in primes], primes) == h + 1 - Q == -h


def test_encode_kernels_use_no_local_memory():
    """The encode and decode kernels (both cluster shapes of the FFTs) are in the sm_100a code and run without local
    memory or stack."""
    usage = KS._cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*(?:encode64|decode64)\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    names = sorted(re.sub(r"^_ZN3agx\d+", "", n)[:22] for n, *_ in found)
    assert len(found) == 5, names
    for name, reg, stack, local in found:
        assert int(local) == 0 and int(stack) == 0, name


# ------------------------------------------------------------------------------------------ on a GPU

dev, host, data, empty = KS.dev, KS.host, KS.data, KS.empty


@pytest.fixture(scope="module")
def A():
    import agilex_ntt_b200 as A
    return A


_CTX = {}


@pytest.fixture(scope="module")
def ctx(A):
    def get(N, primes, psis=None):
        key = (N, tuple(primes), tuple(psis) if psis else None)
        if key not in _CTX:
            _CTX[key] = A.Context64(N, primes, psi=psis)
        return _CTX[key]
    yield get
    for c in _CTX.values():
        c.close()
    _CTX.clear()


def zdev(z):
    import torch
    return torch.from_numpy(np.ascontiguousarray(z, dtype=np.complex128)).cuda()


def zempty(B, S):
    import torch
    return torch.empty((B, S), dtype=torch.complex128, device="cuda")


def encode(c, z, scale, limbs, form, stream=None):
    out = empty(z.shape[0], limbs, c.n)
    return c.encode(out, z, scale, ntt_form=form, stream=stream)


def decode(c, res, scale, form, stream=None):
    z = zempty(res.shape[0], c.n // 2)
    return c.decode(z, res, scale, ntt_form=form, stream=stream)


def centred_ints(res, primes):
    """[B][limbs][n] residues -> [B][n] centred integers"""
    B, _, n = res.shape
    return [[crt_centred([int(res[b, l, i]) for l in range(len(primes))], primes) for i in range(n)] for b in range(B)]


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_encode_vs_oracle(ctx, N, form):
    """|c_i - scale m_i| within the bound for limbs 1, 3 and L; the evaluation form is fwd of the coefficient form."""
    import torch
    c = ctx(N, QS)
    rng = np.random.default_rng(N)
    B = 3 if N <= 4096 else 2
    z = rand_slots(rng, B, N // 2)
    scale = 2.0 ** 40
    m = oracle_encode(z, N)
    tol = max(enc_tol(scale, z[b], N) for b in range(B))
    for limbs in (1, 3, len(QS)):
        coef = encode(c, zdev(z), scale, limbs, False)
        if form:
            got = encode(c, zdev(z), scale, limbs, True)
            ref = coef.clone()
            ctx(N, QS[:limbs]).fwd(ref)
            torch.cuda.synchronize()
            assert torch.equal(got, ref), limbs
        h = host(coef).astype(np.int64)                             # residues < 2^62
        limb = lambda l: np.where(h[:, l] > QS[l] // 2, h[:, l] - QS[l], h[:, l])
        ci = limb(0)
        assert np.abs(ci.astype(np.float64) - scale * m).max() <= tol, limbs
        for l in range(1, limbs):                                   # every limb holds the same integer
            assert (limb(l) == ci).all(), l


def _exact_cases():
    """(a, scale) with |rint(scale a)| around 2^53, 2^63, 2^64 and 2^100, both signs, exact .5 ties, and products that
    round"""
    out = []
    for T in (2 ** 53 - 1, 2 ** 53, 2 ** 53 + 2, 2 ** 63 - 1024, 2 ** 63, 2 ** 63 + 2048, 2 ** 64 - 4096, 2 ** 64,
              2 ** 64 + 4096, 2 ** 100, 3 * 2 ** 99, 2 ** 100 + 2 ** 48, 2 ** 180):
        for sgn in (1, -1):
            out.append((sgn * T / 2.0 ** 40, 2.0 ** 40))
            out.append((sgn * T / 2.0 ** 200, 2.0 ** 200))
    for a in (0.5, 1.5, 2.5, 3.5, -2.5, 2.0 ** 51 + 0.5, 2.0 ** 51 + 1.5, -(2.0 ** 51 + 0.5), 0.0, 1.0):
        out.append((a, 1.0))
    rng = random.Random(5)
    for _ in range(8):
        out.append((rng.uniform(-1, 1), 2.0 ** rng.uniform(40, 110)))
    return out


@gpu
@pytest.mark.parametrize("N", (32, 32768))
def test_encode_exact_residues(ctx, N):
    """Constant real slots z_j = a encode to the constant polynomial rint(fl(scale a)), every other coefficient 0, the
    residues bit for bit the big-integer ones (|c_0| up to 2^180 over four 60-bit primes)."""
    import torch
    primes = KS.find_primes(60, 4)
    c = ctx(N, primes)
    S = N // 2
    for a, scale in _exact_cases():
        want = round(float(scale) * float(a))
        assert 2 * abs(want) < prod(primes)
        z = zdev(np.full((1, S), complex(a, 0.0)))
        got = host(encode(c, z, scale, len(primes), False))
        assert [int(v) for v in got[0, :, 0]] == [want % q for q in primes], (a, scale)
        assert not got[0, :, 1:].any(), (a, scale)
    torch.cuda.synchronize()


_P64 = []


def primes64():
    if not _P64:
        _P64.extend(KS.find_primes(60, 64))
    return _P64


@gpu
@pytest.mark.parametrize("limbs", (1, 2, 16, 17, 64))
def test_decode_crt_exact(ctx, limbs):
    """A constant polynomial X_c decodes to m_0 = X_c / scale in every slot with imaginary part 0, within
    (2 limbs + 1) 2^-53 of float(Fraction(X_c) / scale); inf where that overflows."""
    N = 32
    primes = primes64()
    c = ctx(N, primes)
    qs = primes[:limbs]
    Q = prod(qs)
    h = (Q - 1) // 2
    rng = random.Random(limbs)
    xs = [0, 1, -1, h, -h, (Q + 1) // 2 - Q] + [rng.randrange(-h, h + 1) for _ in range(10)]
    xs += [rng.randrange(-(2 ** 70), 2 ** 70) % (h + 1) for _ in range(3)]
    res = np.zeros((len(xs), limbs, N), dtype=np.uint64)
    for b, x in enumerate(xs):
        res[b, :, 0] = [x % q for q in qs]
    for scale in (1.0, 2.0 ** 40, 2.0 ** 900, 3.0 * 2.0 ** 500):
        for form in (False, True):
            d = dev(res)
            if form:
                ctx(N, qs).fwd(d)
            got = decode(c, d, scale, form).cpu().numpy()
            for b, x in enumerate(xs):
                assert (got[b] == got[b, 0]).all() and got[b, 0].imag == 0, (b, scale)
                try:
                    want = float(Fraction(x) / Fraction(scale))
                except OverflowError:
                    assert np.isinf(got[b, 0].real) and np.sign(got[b, 0].real) == np.sign(x), (b, scale)
                    continue
                if abs(want) > 1.7e308:                             # rounds to the largest double: allow inf
                    continue
                assert abs(got[b, 0].real - want) <= (2 * limbs + 1) * U * abs(want), (b, scale, form)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_decode_vs_oracle(ctx, N, form):
    """Random big-integer polynomials (uniform residues over 3 primes, scale Q / 2^30) against the oracle on their
    exact m; and decode(encode(z)) = z within the bounds."""
    c = ctx(N, QS)
    qs = QS[:3]
    Q = prod(qs)
    B = 2
    res = data(B, qs, N, 7 + N)
    scale = float(Q >> 30)
    X = centred_ints(res, qs)
    m = np.array([[float(Fraction(x) / Fraction(scale)) for x in row] for row in X])
    d = dev(res)
    if form:
        ctx(N, qs).fwd(d)
    got = decode(c, d, scale, form).cpu().numpy()
    assert np.abs(got - oracle_decode(m, N)).max() <= dec_tol(np.abs(m).max(), N, 3)
    rng = np.random.default_rng(N + 1)
    z = rand_slots(rng, B, N // 2)
    sc = 2.0 ** 45
    back = decode(c, encode(c, zdev(z), sc, len(QS), form), sc, form).cpu().numpy()
    tol = N * enc_tol(sc, z, N) / sc + dec_tol(2.0, N, len(QS))
    assert np.abs(back - z).max() <= tol


@gpu
@pytest.mark.parametrize("N", (1024, 16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """More polynomials than two waves of CTAs: the batch equals the calls one polynomial at a time, both forms."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 2 * sms + 5 if N < 32768 else sms + 3
    c = ctx(N, QS)
    rng = np.random.default_rng(N)
    z = zdev(rand_slots(rng, B, N // 2))
    for form in (False, True):
        res = encode(c, z, 2.0 ** 50, 2, form)
        back = decode(c, res, 2.0 ** 50, form)
        for b in (0, B // 2, B - 1):
            one = encode(c, z[b:b + 1].contiguous(), 2.0 ** 50, 2, form)
            assert torch.equal(res[b:b + 1], one), (form, b)
            assert torch.equal(back[b:b + 1], decode(c, one, 2.0 ** 50, form)), (form, b)
        assert (back - z).abs().max().item() < 1e-6
        del res, back
        torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", SIZES)
def test_rotation_in_the_clear(A, ctx, N, form):
    """decode(automorph(encode(z), galois_element(n, r))) = roll(z, -r) for r = 1, -3, S - 1, and conj(z) for 2n - 1."""
    c = ctx(N, QS[:2])
    S = N // 2
    rng = np.random.default_rng(N + 9)
    z = rand_slots(rng, 2, S)
    sc = 2.0 ** 45
    res = encode(c, zdev(z), sc, 2, form)
    tol = N * enc_tol(sc, z, N) / sc + dec_tol(2.0, N, 2)
    gs = [A.galois_element(N, r) for r in (1, -3, S - 1)] + [2 * N - 1]
    out = empty(len(gs), 2, 2, N)
    c.automorph(out, res, gs, ntt_form=form)
    wants = [np.roll(z, -r, axis=1) for r in (1, -3, S - 1)] + [np.conj(z)]
    for t, want in enumerate(wants):
        got = decode(c, out[t], sc, form).cpu().numpy()
        assert np.abs(got - want).max() <= tol, t


# ---- encrypted: encode, encrypt as test_bsgs_end_to_end does, evaluate, decrypt with polymul and elementwise, decode
DELTA = 2.0 ** 50


def encrypt_dev(cq, s, mres, qs, ebound, rng, seed):
    """(c0, c1) = (-a s + m + e, a) over qs from the library's products: [2][1][l+1][n], coefficient form"""
    import torch
    N = cq.n
    res = lambda v: dev(MR.residues(v, qs)).view(1, len(qs), N)
    a = dev(data(1, qs, N, seed))
    c0 = empty(1, len(qs), N)
    e = KS.small(rng, N, ebound)
    cq.elementwise("add", c0, mres, res(e))
    t = empty(1, len(qs), N)
    cq.polymul(t, a, res(s))
    cq.elementwise("sub", c0, c0, t)
    return torch.stack([c0, a]).contiguous()


def decrypt_dev(cq, ct, s, qs):
    """c0 + c1 s over qs, [1][l+1][n] residues"""
    N = cq.n
    sres = dev(MR.residues(s, qs)).view(1, len(qs), N)
    p = empty(1, len(qs), N)
    cq.polymul(p, ct[1].reshape(1, len(qs), N).contiguous(), sres)
    cq.elementwise("add", p, p, ct[0].reshape(1, len(qs), N).contiguous())
    return p


@gpu
def test_rotation_encrypted(A, ctx):
    """Encrypt encode(z); rotate by 1 and -3 and conjugate in one call; each decrypts and decodes to roll(z, -r) or
    conj(z) within n (key-switch bound + |e| + 1) / Delta."""
    N = 1024
    qs, alpha, k = QS, 1, len(PS)
    rng = random.Random(3)
    s = KS.ternary(rng, N)
    ebound = 8
    key_primes = qs + PS
    ctop = ctx(N, key_primes)
    gs = [A.galois_element(N, 1), A.galois_element(N, -3), 2 * N - 1]
    rks = [KS.gadget_key_gpu(ctop, key_primes, k, alpha, len(qs), s, AM.automorph_ints(s, g), ebound, rng) for g in gs]
    cq = ctx(N, qs)
    z = rand_slots(np.random.default_rng(4), 1, N // 2)
    ct = encrypt_dev(cq, s, encode(cq, zdev(z), DELTA, len(qs), False), qs, ebound, rng, 5)
    out = empty(len(gs), 2, 1, len(qs), N)
    ctop.rotate(out, ct, gs, rks, alpha, k, ntt_form=False)
    tol = N * (KS.ks_bound(qs, PS, alpha, N, ebound) + ebound + 1) / DELTA + dec_tol(2.0, N, len(qs))
    wants = [np.roll(z, -1, axis=1), np.roll(z, 3, axis=1), np.conj(z)]
    for t, want in enumerate(wants):
        got = decode(cq, decrypt_dev(cq, out[t], s, qs), DELTA, False).cpu().numpy()
        assert np.abs(got - want).max() <= tol, t


@gpu
def test_mulrelin_rescale_multiplies_slots(ctx):
    """Encrypt encode(z1), encode(z2) at Delta; mulrelin with rescale decrypts and decodes, at scale Delta^2 / q_l, to
    z1 (.) z2 within the slot image of the rescaled product's bound and of the encryption errors."""
    N = 256
    qs, alpha, k = QS, 1, len(PS)
    rng = random.Random(11)
    s = KS.ternary(rng, N)
    ebound = 8
    key_primes = qs + PS
    c = ctx(N, key_primes)
    rlk = KS.gadget_key_gpu(c, key_primes, k, alpha, len(qs), s, KS.negacyclic(s, s), ebound, rng)
    cq = ctx(N, qs)
    g = np.random.default_rng(12)
    z1, z2 = rand_slots(g, 1, N // 2), rand_slots(g, 1, N // 2)
    ct1 = encrypt_dev(cq, s, encode(cq, zdev(z1), DELTA, len(qs), False), qs, ebound, rng, 13)
    ct2 = encrypt_dev(cq, s, encode(cq, zdev(z2), DELTA, len(qs), False), qs, ebound, rng, 14)
    out = empty(2, 1, len(qs) - 1, N)
    c.mulrelin(out, ct1, ct2, rlk, alpha, k, rescale=True, ntt_form=False)
    ql = qs[-1]
    scale = float(Fraction(int(DELTA) ** 2, ql))
    cr = ctx(N, qs[:-1])
    got = decode(cr, decrypt_dev(cr, out, s, qs[:-1]), scale, False).cpu().numpy()
    # each factor's slots carry n (e + 1) / Delta (the error and the encoding's rounding); the product adds the
    # rescaled relinearisation bound, n (|K| / (q_l P) + (N + 1) / 2) in coefficient units at scale Delta^2 / q_l
    fac = N * (ebound + 1) / DELTA
    tol = 3 * fac * (1 + fac) + N * (MR.relin_noise(qs, PS, alpha, N, ebound) / ql + (N + 1) / 2) / scale
    assert np.abs(got - z1 * z2).max() <= tol + dec_tol(4.0, N, len(qs) - 1)


@gpu
def test_bsgs_matrix_vector_product(A, ctx):
    """INTEGRATION.md's 2 x 4 baby-step/giant-step recipe on a banded S x S matrix A (diagonals 0 .. 7): diagonal
    k = 4 j + i of A, pre-rotated by 4 j, encoded by agx_encode64 over Q_l u P in evaluation form at Delta_d, one
    lintrans call for the baby steps, one rotate for the giant step and an add.  Decrypted and decoded at
    Delta Delta_d: A z within the lintrans bound / (Delta Delta_d) and the encoding errors."""
    import torch
    N = 256
    S = N // 2
    qs, alpha, k = QS, 1, len(PS)
    primes = qs + PS
    rng = random.Random(17)
    s = KS.ternary(rng, N)
    ebound = 8
    c, cq = ctx(N, primes), ctx(N, qs)
    baby = [A.galois_element(N, i) for i in range(4)]
    giant = A.galois_element(N, 4)
    key = lambda g: KS.gadget_key_gpu(c, primes, k, alpha, len(qs), s, AM.automorph_ints(s, g), ebound, rng)
    rks = [None] + [key(g) for g in baby[1:]]
    rk_giant = key(giant)
    g = np.random.default_rng(18)
    Amat = np.zeros((S, S), dtype=np.complex128)
    for kk in range(8):
        for t in range(S):
            Amat[t, (t + kk) % S] = complex(g.uniform(-1, 1), g.uniform(-1, 1))
    diag = lambda kk: np.array([Amat[t, (t + kk) % S] for t in range(S)])
    dd = 2.0 ** 30
    diags = [[encode(c, zdev(np.roll(diag(4 * j + i), 4 * j).reshape(1, S)), dd, len(primes), True)[0]
              for i in range(4)] for j in range(2)]
    z = rand_slots(g, 1, S)
    ct = encrypt_dev(cq, s, encode(cq, zdev(z), DELTA, len(qs), False), qs, ebound, rng, 19)
    y = empty(2, 2, 1, len(qs), N)
    c.lintrans(y, ct, baby, rks, diags, alpha, k, ntt_form=False)
    r1 = empty(2, 1, len(qs), N)
    c.rotate(r1, y[1], giant, [rk_giant], alpha, k, ntt_form=False)
    cq.elementwise("add", y[0].view(2, len(qs), N), y[0].view(2, len(qs), N), r1.view(2, len(qs), N))
    got = decode(cq, decrypt_dev(cq, y[0], s, qs), DELTA * dd, False).cpu().numpy()
    # coefficient norms of the encoded diagonals (centred), for the noise bound
    dn = []
    for row in diags:
        dn.append([])
        for d in row:
            coef = d.clone().view(1, len(primes), N)
            c.inv(coef)
            dn[-1].append(max(abs(v) for v in centred_ints(host(coef), primes)[0]))
    ksb = KS.ks_bound(qs, PS, alpha, N, ebound)
    noise = sum(LT.lintrans_bound(ksb, N, row) for row in dn) + ksb
    # the encrypted message's error (e and the encoding's rounding) times the diagonals, and the diagonals' rounding
    # times the message
    mnorm = math.sqrt(2) * DELTA                                   # |m_i| <= ||z||_inf
    err = noise + 8 * N * max(max(r) for r in dn) * (ebound + 1) + 8 * N * 0.5 * mnorm
    tol = N * err / (DELTA * dd) + dec_tol(16.0, N, len(qs))
    want = (Amat @ z[0]).reshape(1, S)
    assert np.abs(got - want).max() <= tol
    torch.cuda.synchronize()


# ---- call behaviour
@gpu
def test_refusals_and_empty_calls(A, ctx):
    import torch
    from oracle import oracle as O
    N = 1024
    lib = A.lib()
    c = ctx(N, QS)
    L = len(QS)
    dup = A.Context64(N, [QS[0], QS[1], QS[0]])
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    z = zdev(rand_slots(np.random.default_rng(1), 2, N // 2))
    r = dev(data(2, QS, N, 2))
    zs, rs = z.clone(), r.clone()
    pz, pr = z.data_ptr(), r.data_ptr()
    big = torch.zeros(4 * L * N, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    torch.cuda.synchronize()
    ctxs = (c, dup)
    try:
        for form in (0, 1):
            for fn, is_dec in ((lib.agx_encode64, False), (lib.agx_decode64, True)):
                def call(h, o, i, B, scale, limbs):
                    return fn(h, o, i, B, scale, limbs, form, None)
                po, pi = (pz, pr) if is_dec else (pr, pz)
                invalid = [
                    (c32._h, po, pi, 2, 1.0, 2),                                      # u32 context
                    (c._h, None, pi, 2, 1.0, 2), (c._h, po, None, 2, 1.0, 2),         # null pointers
                    (c._h, po + 8, pi, 1, 1.0, 2), (c._h, po, pi + 8, 1, 1.0, 2),     # misaligned
                    (c._h, po, pi, 2, 1.0, 0), (c._h, po, pi, 2, 1.0, L + 1),         # limbs
                    (c._h, po, pi, 2, 0.0, 2), (c._h, po, pi, 2, -1.0, 2),            # scale
                    (c._h, po, pi, 2, float("inf"), 2), (c._h, po, pi, 2, float("nan"), 2),
                    (c._h, po, pi, 0x7fffffff // 2 + 1, 1.0, 2),                      # B limbs > 2^31 - 1
                    (c._h, bp, bp + 8 * (N - 2), 1, 1.0, 2),                          # overlapping ranges
                    (c._h, bp + 8 * (N - 2), bp, 1, 1.0, 2),
                ]
                if is_dec:
                    invalid.append((dup._h, po, pi, 2, 1.0, 3))                       # equal primes
                for h, o_, i_, B, scale, limbs in invalid:
                    l0 = [t.launch_count() for t in ctxs]
                    assert call(h, o_, i_, B, scale, limbs) == -1, (is_dec, form, B, scale, limbs)
                    assert [t.launch_count() for t in ctxs] == l0
                l0 = c.launch_count()
                assert call(c._h, None, None, 0, 1.0, 2) == 0 and call(c._h, bp, bp, 0, 1.0, 2) == 0
                assert c.launch_count() == l0
                # adjacent, not overlapping, is allowed; equal primes beyond `limbs` are no concern of the decode
                assert call(c._h, bp, bp + 8 * (1 if is_dec else 2) * N, 1, 1.0, 2) == 0
                if is_dec:
                    assert call(dup._h, bp, pr, 1, 1.0, 2) == 0
        bad = [
            lambda: c.encode(empty(2, 2, N), z.real.contiguous(), 1.0),              # not complex
            lambda: c.encode(empty(3, 2, N), z, 1.0),                                 # batch
            lambda: c.encode(empty(2, L + 1, N), z, 1.0),                             # limbs > L
            lambda: c.encode(empty(2, 2, N // 2), z, 1.0),
            lambda: c.decode(zempty(2, N // 4), r, 1.0),
            lambda: c.decode(z, r.cpu(), 1.0),
            lambda: c.decode(z.cpu(), r, 1.0),
        ]
        for fn in bad:
            with pytest.raises(ValueError):
                fn()
        with pytest.raises(A.AgxError):
            c.encode(empty(2, 2, N), z, 0.0)
        torch.cuda.synchronize()
        assert torch.equal(z, zs) and torch.equal(r, rs)
    finally:
        dup.close()
        c32.close()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(A, N):
    """The header's counts, the same on a context's first call and later ones, for B = 1 and B = 5."""
    import torch
    x = int(N == 32768)
    z = zdev(rand_slots(np.random.default_rng(N), 5, N // 2))
    for first in (True, False):
        for B in (1, 5):
            for form, enc_n, dec_n in ((False, 1, 2), (True, 2, 3 + x)):
                c = A.Context64(N, QS)
                if not first:
                    decode(c, encode(c, z, 2.0 ** 40, 3, form), 2.0 ** 40, form)
                torch.cuda.synchronize()
                l0 = c.launch_count()
                res = encode(c, z[:B], 2.0 ** 40, 3, form)
                torch.cuda.synchronize()
                assert c.launch_count() - l0 == enc_n, (first, B, form)
                l0 = c.launch_count()
                decode(c, res, 2.0 ** 40, form)
                torch.cuda.synchronize()
                assert c.launch_count() - l0 == dec_n, (first, B, form)
                c.close()


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_inputs_unchanged(ctx, form):
    import torch
    N = 4096
    c = ctx(N, QS)
    z = zdev(rand_slots(np.random.default_rng(5), 4, N // 2))
    zs = z.clone()
    res = encode(c, z, 2.0 ** 40, len(QS), form)
    rs = res.clone()
    decode(c, res, 2.0 ** 40, form)
    torch.cuda.synchronize()
    assert torch.equal(z, zs) and torch.equal(res, rs)


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    c = ctx(N, QS)
    hz = rand_slots(np.random.default_rng(6), 4, N // 2)
    want_res = encode(c, zdev(hz), 2.0 ** 40, 3, form)
    want_z = decode(c, want_res, 2.0 ** 40, form)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        zi = torch.empty_like(want_z)
        zi.copy_(zdev(hz))                                          # torch work the call must follow
        res = empty(4, 3, N)
        zo = zempty(4, N // 2)
    c.encode(res, zi, 2.0 ** 40, ntt_form=form, stream=s)
    c.decode(zo, res, 2.0 ** 40, ntt_form=form, stream=s)
    s.synchronize()
    assert torch.equal(res, want_res) and torch.equal(zo, want_z)


@gpu
@pytest.mark.parametrize("first", ("encode", "decode"))
@pytest.mark.parametrize("N", (1024, 32768))
def test_first_call_on_a_side_stream(A, ctx, N, first):
    """A fresh context's first call (which builds and uploads the twiddle table) issued on a non-blocking torch side
    stream, synchronised on that stream only, equals the same call on a context that has already worked."""
    import torch
    ref = ctx(N, QS)
    hz = rand_slots(np.random.default_rng(N + 21), 3, N // 2)
    want_res = encode(ref, zdev(hz), 2.0 ** 40, 3, True)
    want_z = decode(ref, want_res, 2.0 ** 40, True)
    torch.cuda.synchronize()
    c = A.Context64(N, QS)
    try:
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            if first == "encode":
                zi = torch.empty_like(want_z)
                zi.copy_(zdev(hz))
                res = empty(3, 3, N)
                c.encode(res, zi, 2.0 ** 40, ntt_form=True, stream=s)
                s.synchronize()
                assert torch.equal(res, want_res)
            else:
                ri = torch.empty_like(want_res)
                ri.copy_(want_res)
                zo = zempty(3, N // 2)
                c.decode(zo, ri, 2.0 ** 40, ntt_form=True, stream=s)
                s.synchronize()
                assert torch.equal(zo, want_z)
    finally:
        c.close()


def _exact_m(z, n):
    """m_i = (2/n) sum_j Re(z_j zeta^(-i 5^j)) in 60-digit arithmetic (mpmath), one polynomial"""
    import mpmath
    mpmath.mp.dps = 60
    pw = [mpmath.expjpi(mpmath.mpf(k) / n) for k in range(2 * n)]          # zeta^k
    g = [int(v) for v in rot_group(n)]
    zs = [mpmath.mpc(float(v.real), float(v.imag)) for v in z]
    return [2 * sum((zj * pw[(-i * gj) % (2 * n)]).real for zj, gj in zip(zs, g)) / n for i in range(n)]


@gpu
@pytest.mark.parametrize("N", (4, 16, 64, 256))
def test_encode_bound_with_kappa_5(ctx, N):
    """The stated bound itself, kappa = 5, against m computed in 60-digit arithmetic: |c_i - scale m_i| <= 1/2 +
    scale ||z||_inf 5 log2(n) 2^-53, for several scales (exact residues at limb 0 give c_i)."""
    import mpmath
    c = ctx(N, QS)
    rng = np.random.default_rng(N + 31)
    z = rand_slots(rng, 2, N // 2)
    exact = [_exact_m(z[b], N) for b in range(2)]
    for scale in (2.0 ** 20, 2.0 ** 45, 3.0 * 2.0 ** 50):
        h = host(encode(c, zdev(z), scale, 1, False)).astype(np.int64)
        ci = np.where(h[:, 0] > QS[0] // 2, h[:, 0] - QS[0], h[:, 0])
        for b in range(2):
            bound = 0.5 + scale * np.abs(z[b]).max() * KAPPA * math.log2(N) * U
            err = max(abs(int(ci[b, i]) - mpmath.mpf(scale) * exact[b][i]) for i in range(N))
            assert err <= bound, (scale, b, float(err), bound)


@gpu
@pytest.mark.parametrize("N", (4, 16, 64, 256))
def test_decode_fft_bound_with_kappa_5(ctx, N):
    """The forward FFT's stated bound, kappa = 5, against 60-digit evaluation: integer polynomials below 2^50 at a
    power-of-two scale make m_i = X_i / scale exact, so |z~_j - z_j| <= 5 log2(n) 2^-53 S ||m||_inf is the FFT's alone."""
    import mpmath
    mpmath.mp.dps = 60
    c = ctx(N, QS)
    rng = random.Random(N + 41)
    X = [[rng.randrange(-(2 ** 50), 2 ** 50) for _ in range(N)] for _ in range(2)]
    res = np.array([[[x % q for x in row] for q in QS[:2]] for row in X], dtype=np.uint64)
    scale = 2.0 ** 30
    got = decode(c, dev(res), scale, False).cpu().numpy()
    pw = [mpmath.expjpi(mpmath.mpf(k) / N) for k in range(2 * N)]
    for b in range(2):
        m = [mpmath.mpf(x) / mpmath.mpf(scale) for x in X[b]]
        bound = KAPPA * math.log2(N) * U * (N // 2) * float(max(abs(v) for v in m))
        for j, gj in enumerate(rot_group(N)):
            want = sum(mi * pw[(i * int(gj)) % (2 * N)] for i, mi in enumerate(m))
            assert abs(mpmath.mpc(got[b, j].real, got[b, j].imag) - want) <= bound, (b, j)


@gpu
def test_tiny_scales(A, ctx):
    """The encode refuses scales below 2^-1022 S (scale / S would be subnormal, and folding 1 / S into it would round),
    launching nothing; at 2^-1022 S it runs.  The decode takes any positive finite scale."""
    N = 64
    lib = A.lib()
    c = ctx(N, QS)
    z = zdev(rand_slots(np.random.default_rng(2), 1, N // 2))
    r = empty(1, 2, N)
    edge = 2.0 ** -1022 * (N // 2)
    l0 = c.launch_count()
    for sc in (edge / 2, np.nextafter(edge, 0), 5e-324):
        for form in (0, 1):
            assert lib.agx_encode64(c._h, r.data_ptr(), z.data_ptr(), 1, float(sc), 2, form, None) == -1, sc
    assert c.launch_count() == l0
    assert not host(encode(c, z, edge, 2, False)).any()            # |scale m| < 1/2: every coefficient rounds to 0
    zo = decode(c, encode(c, z, 2.0 ** 40, 2, False), 5e-324, False)   # runs; |X_c| / scale overflows the doubles
    assert not np.isfinite(zo.cpu().numpy()).all()
