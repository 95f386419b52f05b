"""u64 RNS basis conversion (agx_moddown64 / agx_modup64, Context64.moddown / modup): the two steps of hybrid key
switching, in coefficient and in evaluation form.

Definitions, for a set of the context's primes with product S and h_S = (S - 1) / 2:
- ModDown, k special primes last (P = their product, Q' = the others): [B][L][N] -> [B][L-k][N], the residues over Q'
  of Y = floor((X + h_P) / P) mod Q' for the CRT value X in [0, Q) of the L residues.
- ModUp from q_first .. q_{first+count-1}: [B][count][N] -> [B][L][N], every limb the residue of the centred lift
  ((X + h_S) mod S) - h_S of the source residues.

The CPU tests pin a mixed-radix-conversion (MRC) oracle, the four steps the kernels run, against those big-int
definitions, and check on the compiled library that the new kernels use no local memory.  The GPU tests compare the
library with the oracle bit for bit, the evaluation form with the existing calls composed around the coefficient form,
ModDown with k = 1 with the rescale, a ModUp / ModDown round trip, and a whole key switch built from public calls."""
import ctypes as C
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
_u64p = C.POINTER(C.c_uint64)


def find_primes(bits: int, count: int):
    """The `count` largest primes q < 2^bits of exactly `bits` bits with q = 1 (mod 2^16): usable at every N <= 32768."""
    out, q = [], (1 << bits) - (1 << 16) + 1
    while len(out) < count:
        if O.is_prime(q):
            out.append(q)
        q -= 1 << 16
    return out


PRIMES = {b: find_primes(b, 6) for b in (50, 60, 62)}
ASC = [PRIMES[50][0], PRIMES[50][1], PRIMES[60][0], PRIMES[60][1], PRIMES[62][0], PRIMES[62][1]]
DESC = ASC[::-1]
MIXED = [PRIMES[60][2], PRIMES[50][2], PRIMES[62][2], PRIMES[50][3], PRIMES[62][3], PRIMES[60][3]]
SETS = {"ascending": ASC, "descending": DESC, "mixed": MIXED}


# ---- big ints and the MRC oracle
def crt(res, primes):
    Q = prod(primes)
    X = 0
    for r, q in zip(res, primes):
        m = Q // q
        X += int(r) * m * pow(m, -1, q)
    return X % Q


def moddown_bigint(X, primes, k):
    P, Qd = prod(primes[-k:]), prod(primes[:-k])
    return ((X + (P - 1) // 2) // P) % Qd


def modup_bigint(X, src):
    """the centred lift of X in [0, S)"""
    S = prod(src)
    h = (S - 1) // 2
    return (X + h) % S - h


def mrc_lift(y, src, targets):
    """Steps 1-3 on object arrays: y[t] residues mod src[t] -> (X + h) mod S mod each target (a list of arrays)."""
    m = len(src)
    h = (prod(src) - 1) // 2
    d = []
    for t in range(m):
        a = (y[t] + h % src[t]) % src[t]                         # step 1
        for j in range(t):                                       # step 2: the digits
            a = (a - d[j]) * pow(src[j], -1, src[t]) % src[t]
        d.append(a)
    out = []
    for q in targets:                                            # step 3: Horner
        T = d[m - 1]
        for t in range(m - 2, -1, -1):
            T = T * (src[t] % q) + d[t]
        out.append(T % q)
    return out, h


def moddown_mrc(x, primes, k):
    """[B][L][N] -> [B][L-k][N] by the four steps"""
    src, tgt = primes[-k:], primes[:-k]
    xo = x.astype(object)
    T, h = mrc_lift([xo[:, len(tgt) + t, :] for t in range(k)], src, tgt)
    P = prod(src)
    out = np.empty((x.shape[0], len(tgt), x.shape[2]), dtype=np.uint64)
    for i, q in enumerate(tgt):                                  # step 4
        out[:, i, :] = ((xo[:, i, :] + h % q - T[i]) * pow(P, -1, q) % q).astype(np.uint64)
    return out


def modup_mrc(x, primes, first, count):
    """[B][count][N] over primes[first:first+count] -> [B][L][N]"""
    src = primes[first:first + count]
    xo = x.astype(object)
    T, h = mrc_lift([xo[:, t, :] for t in range(count)], src, primes)
    out = np.empty((x.shape[0], len(primes), x.shape[2]), dtype=np.uint64)
    for i, q in enumerate(primes):
        out[:, i, :] = ((T[i] - h) % q).astype(np.uint64)
    out[:, first:first + count, :] = x                           # source limbs copied
    return out


def boundary_values(S, P, rng, m_count=6):
    """X = 0, S - 1, S/2 +- 1, h_S, h_S +- 1, and the rounding boundaries j*P + h_P and j*P + h_P - 1 (P = S for ModUp)."""
    h, hP = (S - 1) // 2, (P - 1) // 2
    Xs = [0, 1, S - 1, S - 2, S // 2 - 1, S // 2, S // 2 + 1, h - 1, h, h + 1]
    for j in [0, 1, S // P - 1, S // P // 2] + [rng.randrange(S // P) for _ in range(m_count)]:
        Xs += [j * P + hP, j * P + hP - 1]
    return [X for X in Xs if 0 <= X < S]


def residues(Xs, primes):
    """[1][L][len(Xs)] residues of the big ints Xs"""
    return np.array([[X % q for X in Xs] for q in primes], dtype=np.uint64).reshape(1, len(primes), len(Xs))


def ranges(L, m):
    """source ranges of m limbs: at the start, in the middle, at the end"""
    return sorted({0, (L - m) // 2, L - m})


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("k", (1, 2, 3, 4, 5))
@pytest.mark.parametrize("name", SETS)
def test_moddown_oracle_is_the_definition(name, k):
    primes = SETS[name]
    rng = random.Random(31 * k + len(name))
    Q, P = prod(primes), prod(primes[-k:])
    Xs = boundary_values(Q, P, rng) + [rng.randrange(Q) for _ in range(2000)]
    got = moddown_mrc(residues(Xs, primes), primes, k)[0]
    for j, X in enumerate(Xs):
        Y = moddown_bigint(X, primes, k)
        assert [int(v) for v in got[:, j]] == [Y % q for q in primes[:-k]], (name, k, X)


@pytest.mark.parametrize("m", (1, 2, 3, 4, 5))
@pytest.mark.parametrize("name", SETS)
def test_modup_oracle_is_the_definition(name, m):
    primes = SETS[name]
    for first in ranges(len(primes), m):
        src = primes[first:first + m]
        rng = random.Random(17 * m + first + len(name))
        S = prod(src)
        Xs = boundary_values(S, S, rng) + [rng.randrange(S) for _ in range(2000)]
        got = modup_mrc(residues(Xs, src), primes, first, m)[0]
        for j, X in enumerate(Xs):
            Xc = modup_bigint(X, src)
            assert [int(v) for v in got[:, j]] == [Xc % q for q in primes], (name, m, first, X)


def _cuobjdump(*args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import agilex_ntt_b200 as A
    return subprocess.run([exe, *args, A.build.build_lib()], capture_output=True, text=True, check=True).stdout


def test_basis_kernels_use_no_local_memory():
    """Every basis-conversion kernel of the library's sm_100a code runs without spills (no local memory, no stack),
    the frame kernels at the 128-register cap, and every expected instantiation is there."""
    usage = _cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*basis\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    names = {n for n, *_ in found}
    assert len([n for n in names if "ref_u64_basis_fwd_kernel" in n]) == 10        # NT = 32 .. 512, both directions
    assert len([n for n in names if "ref_u64_basis_inv_frame_kernel" in n]) == 5
    assert len([n for n in names if "basis64_coeff_kernel" in n]) == 2
    assert len([n for n in names if "ref_fwd_u64_basis_kernel" in n]) == 2
    for k in ("basis64_digits_kernel", "ref_inv_u64_basis_kernel"):
        assert any(k in n for n in names), k
    for name, reg, stack, local in found:
        assert int(local) == 0 and int(stack) == 0, name
        assert int(reg) <= 128, name


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


def with_boundaries(x, primes, Xs):
    """x with the big ints Xs written into the first columns of polynomial 0 (as far as they fit)"""
    bv = residues(Xs, primes)[0]
    k = min(x.shape[2], bv.shape[1])
    x = x.copy()
    x[0, :, :k] = bv[:, :k]
    if bv.shape[1] > k and x.shape[0] > 1:
        r = min(x.shape[2], bv.shape[1] - k)
        x[1, :, :r] = bv[:, k:k + r]
    return x


@pytest.fixture(scope="module")
def orc(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "native", "u64_inverse_oracle.c")
    so = str(tmp_path_factory.mktemp("u64_basis_oracle") / "libu64oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc") or "cc"
    base = [cc, "-O2", "-std=c11", "-fPIC", "-shared", "-o", so, src]
    if subprocess.run(base + ["-fopenmp"], capture_output=True).returncode != 0:
        subprocess.run(base + ["-Wno-unknown-pragmas"], check=True)
    L = C.CDLL(so)
    L.orc_inv_u64.argtypes = [C.c_uint32, _u64p, C.c_uint64, _u64p, C.c_size_t, C.c_int]
    return L


def rns_fwd(x, primes, psis=None):
    """per-limb forward of [B][L][N] (the C restatement of the reference's forward)"""
    N, out = x.shape[-1], np.empty_like(x)
    for l, q in enumerate(primes):
        tw, pre = O.tables_u64(N, q, psis[l] if psis else None)
        v = np.ascontiguousarray(x[:, l, :])
        out[:, l, :] = O.ref_fwd_u64(v, v, q, tw, pre, v.shape[0]).reshape(x.shape[0], N)
    return out


def rns_inv(orc, X, primes, psis=None):
    N, out = X.shape[-1], np.empty_like(X)
    for l, q in enumerate(primes):
        itw, _ = O.tables_u64(N, q, psis[l] if psis else None, inverse=True)
        y = np.ascontiguousarray(X[:, l, :]).copy()
        orc.orc_inv_u64(N, y.ctypes.data_as(_u64p), q, itw.ctypes.data_as(_u64p), y.shape[0],
                        max(1, min(O.max_threads(), 16)))
        out[:, l, :] = y
    return out


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


def empty(B, L, N):
    import torch
    return torch.empty((B, L, N), dtype=torch.int64, device="cuda")


DOWN_CASES = (("mixed", 2), ("ascending", 3), ("descending", 5))
UP_CASES = (("mixed", 0, 2), ("descending", 2, 3), ("ascending", 5, 1), ("mixed", 1, 4))


@gpu
@pytest.mark.parametrize("case", DOWN_CASES)
@pytest.mark.parametrize("N", SIZES)
def test_moddown_coefficient_form_vs_oracle(ctx, N, case):
    name, k = case
    primes = SETS[name]
    c = ctx(N, primes)
    Q, P = prod(primes), prod(primes[-k:])
    x = with_boundaries(data(3, primes, N, 101 + N), primes, boundary_values(Q, P, random.Random(N)))
    d_in = dev(x)
    d_out = empty(3, len(primes) - k, N)
    c.moddown(d_out, d_in, k, ntt_form=False)
    assert (host(d_out) == moddown_mrc(x, primes, k)).all()
    assert (host(d_in) == x).all()                                      # d_in is not modified


@gpu
@pytest.mark.parametrize("case", UP_CASES)
@pytest.mark.parametrize("N", SIZES)
def test_modup_coefficient_form_vs_oracle(ctx, N, case):
    name, first, count = case
    primes = SETS[name]
    src = primes[first:first + count]
    c = ctx(N, primes)
    S = prod(src)
    x = with_boundaries(data(3, src, N, 103 + N), src, boundary_values(S, S, random.Random(N)))
    d_in = dev(x)
    d_out = empty(3, len(primes), N)
    c.modup(d_out, d_in, first, count, ntt_form=False)
    assert (host(d_out) == modup_mrc(x, primes, first, count)).all()
    assert (host(d_in) == x).all()


@gpu
@pytest.mark.parametrize("roots", ("minimal", "caller"))
@pytest.mark.parametrize("case", DOWN_CASES)
@pytest.mark.parametrize("N", SIZES)
def test_moddown_evaluation_form(orc, ctx, N, case, roots):
    """moddown(ntt_form=1)(x_hat) = fwd_{L-k}(moddown(ntt_form=0)(inv_L(x_hat))) through the existing calls and a context
    over the first L - k primes, and = the oracle's per-limb forward of the MRC result."""
    import torch
    name, k = case
    primes = SETS[name]
    L = len(primes)
    psis = caller_roots(N, primes) if roots == "caller" else None
    c, lower = ctx(N, primes, psis), ctx(N, primes[:-k], psis[:-k] if psis else None)
    x_hat = data(2, primes, N, 211 + N)
    d_in = dev(x_hat)
    got = empty(2, L - k, N)
    c.moddown(got, d_in, k, ntt_form=True)
    t = d_in.clone()
    c.inv(t)
    want = empty(2, L - k, N)
    c.moddown(want, t, k, ntt_form=False)
    lower.fwd(want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert (host(d_in) == x_hat).all()
    X = rns_inv(orc, x_hat, primes, psis)
    assert (host(got) == rns_fwd(moddown_mrc(X, primes, k), primes[:-k], psis[:-k] if psis else None)).all()


@gpu
@pytest.mark.parametrize("roots", ("minimal", "caller"))
@pytest.mark.parametrize("case", UP_CASES)
@pytest.mark.parametrize("N", SIZES)
def test_modup_evaluation_form(orc, ctx, N, case, roots):
    """modup(ntt_form=1)(x_hat) = fwd_L(modup(ntt_form=0)(inv_src(x_hat))), its source limbs equal x_hat, and it equals
    the oracle's per-limb forward of the MRC result."""
    import torch
    name, first, count = case
    primes = SETS[name]
    src = primes[first:first + count]
    L = len(primes)
    psis = caller_roots(N, primes) if roots == "caller" else None
    spsis = psis[first:first + count] if psis else None
    c, sc = ctx(N, primes, psis), ctx(N, src, spsis)
    x_hat = data(2, src, N, 223 + N)
    d_in = dev(x_hat)
    got = empty(2, L, N)
    c.modup(got, d_in, first, count, ntt_form=True)
    t = d_in.clone()
    sc.inv(t)
    want = empty(2, L, N)
    c.modup(want, t, first, count, ntt_form=False)
    c.fwd(want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    g = host(got)
    assert (g[:, first:first + count, :] == x_hat).all()
    assert (host(d_in) == x_hat).all()
    X = rns_inv(orc, x_hat, src, spsis)
    assert (g == rns_fwd(modup_mrc(X, primes, first, count), primes, psis)).all()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 32768))
def test_sixteen_sources(ctx, N):
    """The largest supported k and count (16), against the oracle in coefficient form and the composed calls in
    evaluation form; 17 is AGX_E_UNSUPPORTED."""
    import torch
    primes = find_primes(60, 18) + [PRIMES[50][4]]                     # L = 19
    L = len(primes)
    c = ctx(N, primes)
    x = data(2, primes, N, 5 + N)
    d = dev(x)
    out = empty(2, L - 16, N)
    c.moddown(out, d, 16, ntt_form=False)
    assert (host(out) == moddown_mrc(x, primes, 16)).all()
    got = empty(2, L - 16, N)
    e = d.clone()
    c.fwd(e)
    c.moddown(got, e, 16, ntt_form=True)
    ctx(N, primes[:L - 16]).fwd(out)
    torch.cuda.synchronize()
    assert torch.equal(got, out)
    xs = x[:, 2:18, :].copy()
    up = empty(2, L, N)
    c.modup(up, dev(xs), 2, 16, ntt_form=False)
    assert (host(up) == modup_mrc(xs, primes, 2, 16)).all()
    xs_hat = dev(xs)
    ctx(N, primes[2:18]).fwd(xs_hat)
    upe = empty(2, L, N)
    c.modup(upe, xs_hat, 2, 16, ntt_form=True)
    c.fwd(up)
    torch.cuda.synchronize()
    assert torch.equal(upe, up)
    import agilex_ntt_b200 as A
    lib = A.lib()
    l0 = c.launch_count()
    for form in (0, 1):
        assert lib.agx_moddown64(c._h, out.data_ptr(), d.data_ptr(), 2, 17, form, None) == -2
        assert lib.agx_modup64(c._h, up.data_ptr(), d.data_ptr(), 2, 0, 17, form, None) == -2
    assert c.launch_count() == l0


@gpu
@pytest.mark.parametrize("N", (32, 4096, 32768))
def test_moddown_k1_is_the_rescale(ctx, N):
    import torch
    c = ctx(N, MIXED)
    x = dev(data(2, MIXED, N, 41 + N))
    for form in (False, True):
        a, b = empty(2, 5, N), empty(2, 5, N)
        l0 = c.launch_count()
        c.moddown(a, x, 1, ntt_form=form)
        torch.cuda.synchronize()
        l1 = c.launch_count()
        c.rescale(b, x, ntt_form=form)
        torch.cuda.synchronize()
        assert c.launch_count() - l1 == l1 - l0
        assert torch.equal(a, b)


def p_broadcast(primes, Pbig, B, N):
    """[B][L][N] words: P mod q_i everywhere (the constant polynomial P in coefficient form has it at coefficient 0 only;
    as an element-wise factor the broadcast is P times the operand in either form)"""
    return dev(np.broadcast_to(np.array([Pbig % q for q in primes], dtype=np.uint64).reshape(1, -1, 1),
                               (B, len(primes), N)))


@gpu
@pytest.mark.parametrize("N", (32, 2048, 32768))
@pytest.mark.parametrize("k", (2, 3))
def test_round_trip(ctx, N, k):
    """x over the first L - k primes: moddown(P * modup(x)) = x exactly, in both forms."""
    import torch
    primes = MIXED
    L = len(primes)
    c, lower = ctx(N, primes), ctx(N, primes[:-k])
    x = data(2, primes[:-k], N, 61 + N)
    Pb = p_broadcast(primes, prod(primes[-k:]), 2, N)
    for form in (False, True):
        d = dev(x)
        if form:
            lower.fwd(d)
        up = empty(2, L, N)
        c.modup(up, d, 0, L - k, ntt_form=form)
        c.elementwise("mul", up, up, Pb)
        back = empty(2, L - k, N)
        c.moddown(back, up, k, ntt_form=form)
        torch.cuda.synchronize()
        assert torch.equal(back, d), form


def ternary(rng, N):
    return [rng.choice((-1, 0, 1)) for _ in range(N)]


def small(rng, N, bound):
    return [rng.randint(-bound, bound) for _ in range(N)]


def rns_of(coeffs, primes):
    """[1][L][N] residues of a list of integer coefficients"""
    return np.array([[v % q for v in coeffs] for q in primes], dtype=np.uint64).reshape(1, len(primes), len(coeffs))


@gpu
@pytest.mark.parametrize("N", (1024, 8192))
def test_key_switch_end_to_end(ctx, N):
    """Hybrid key switching with one digit, public calls only.  QP = 2 Q-primes and 3 special primes (P > Q).
    ksk = (-a*s + e + P*s', a) over QP; D = modup(d); (c0, c1) = moddown(D * ksk).  Then
    c0 + c1*s - d*s' = D*e/P + r0 + r1*s (mod Q) with |r0|, |r1| <= 1/2, so its centred coefficients are at most
    N * (Q/2) * |e|_inf / P + (N + 1) / 2 -- far below Q.  Coefficient and evaluation form give the same (c0, c1)."""
    import torch
    Qp = [PRIMES[60][4], PRIMES[62][4]]
    Pp = [PRIMES[62][5], PRIMES[60][5], PRIMES[50][5]]
    QP = Qp + Pp
    Q, P = prod(Qp), prod(Pp)
    assert P > Q
    k, L = len(Pp), len(QP)
    cqp, cq = ctx(N, QP), ctx(N, Qp)
    rng = random.Random(N)
    ebound = 8
    s, s2, e = ternary(rng, N), ternary(rng, N), small(rng, N, ebound)
    d_s, d_s2, d_e = (dev(rns_of(v, QP)) for v in (s, s2, e))
    d_a = dev(data(1, QP, N, 77))
    # ksk0 = -a*s + e + P*s' over QP
    as_ = empty(1, L, N)
    cqp.polymul(as_, d_a, d_s)
    ksk0 = empty(1, L, N)
    cqp.elementwise("sub", ksk0, d_e, as_)
    ps2 = empty(1, L, N)
    cqp.elementwise("mul", ps2, d_s2, p_broadcast(QP, P, 1, N))
    cqp.elementwise("add", ksk0, ksk0, ps2)
    ksk1 = d_a
    d = data(1, Qp, N, 79)
    # coefficient form
    D = empty(1, L, N)
    cqp.modup(D, dev(d), 0, len(Qp), ntt_form=False)
    t0, t1 = empty(1, L, N), empty(1, L, N)
    cqp.polymul(t0, D, ksk0)
    cqp.polymul(t1, D, ksk1)
    c0, c1 = empty(1, 2, N), empty(1, 2, N)
    cqp.moddown(c0, t0, k, ntt_form=False)
    cqp.moddown(c1, t1, k, ntt_form=False)
    # evaluation form: spectra all the way, back to coefficients at the end
    d_hat = dev(d)
    cq.fwd(d_hat)
    D_hat = empty(1, L, N)
    cqp.modup(D_hat, d_hat, 0, len(Qp), ntt_form=True)
    k0, k1 = ksk0.clone(), ksk1.clone()
    cqp.fwd(k0)
    cqp.fwd(k1)
    cqp.elementwise("mul", k0, D_hat, k0)
    cqp.elementwise("mul", k1, D_hat, k1)
    e0, e1 = empty(1, 2, N), empty(1, 2, N)
    cqp.moddown(e0, k0, k, ntt_form=True)
    cqp.moddown(e1, k1, k, ntt_form=True)
    cq.inv(e0)
    cq.inv(e1)
    torch.cuda.synchronize()
    assert torch.equal(e0, c0) and torch.equal(e1, c1)
    # c0 + c1*s - d*s' over Q
    sq, s2q = dev(rns_of(s, Qp)), dev(rns_of(s2, Qp))
    r = empty(1, 2, N)
    cq.polymul(r, c1, sq)
    cq.elementwise("add", r, r, c0)
    ds2 = empty(1, 2, N)
    cq.polymul(ds2, dev(d), s2q)
    cq.elementwise("sub", r, r, ds2)
    rh = host(r)[0]
    vals = [crt(rh[:, j], Qp) for j in range(N)]
    worst = max(min(v, Q - v) for v in vals)
    bound = N * (Q // 2) * ebound // P + (N + 1) // 2 + 1
    assert worst <= bound, (worst, bound)
    assert bound < Q >> 60


@gpu
@pytest.mark.parametrize("N", (512, 16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """Frames of more than two waves of CTAs for each forward geometry (radix-2, frame, split frame): the evaluation form
    equals the composed calls on every polynomial; the coefficient form equals the oracle on a sample."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    primes, k, first, count = MIXED, 2, 1, 3
    L = len(primes)
    B = -(-(2 * sms + 5) // (L - k))
    c, lower = ctx(N, primes), ctx(N, primes[:-k])
    sc = ctx(N, primes[first:first + count])
    x = data(B, primes, N, 307 + N)
    d_in = dev(x)
    sample = sorted({0, 1, B // 2, B - 2, B - 1} | set(random.Random(N).sample(range(B), 4)))
    coeff = empty(B, L - k, N)
    c.moddown(coeff, d_in, k, ntt_form=False)
    assert (host(coeff)[sample] == moddown_mrc(x[sample], primes, k)).all()
    got = empty(B, L - k, N)
    c.moddown(got, d_in, k, ntt_form=True)
    t = d_in.clone()
    c.inv(t)
    want = empty(B, L - k, N)
    c.moddown(want, t, k, ntt_form=False)
    lower.fwd(want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    del got, want, t, coeff
    xs = np.ascontiguousarray(x[:, first:first + count, :])
    d_s = dev(xs)
    up = empty(B, L, N)
    c.modup(up, d_s, first, count, ntt_form=False)
    assert (host(up)[sample] == modup_mrc(xs[sample], primes, first, count)).all()
    upe = empty(B, L, N)
    c.modup(upe, d_s, first, count, ntt_form=True)
    ts = d_s.clone()
    sc.inv(ts)
    c.modup(up, ts, first, count, ntt_form=False)
    c.fwd(up)
    torch.cuda.synchronize()
    assert torch.equal(upe, up)


@gpu
def test_refusals_and_empty_batches(A, ctx):
    import torch
    N = 1024
    lib = A.lib()
    c = ctx(N, MIXED)
    L = len(MIXED)
    x = dev(data(2, MIXED, N, 3))
    snap = x.clone()
    o = empty(2, L, N)
    pin, pout = x.data_ptr(), o.data_ptr()
    big = torch.zeros(4 * L * N + 2, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    dup_last = A.Context64(N, [MIXED[2], MIXED[0], MIXED[1], MIXED[2]])       # a special prime repeats a Q prime
    dup_pair = A.Context64(N, [MIXED[0], MIXED[1], MIXED[2], MIXED[2]])       # two equal special primes
    dup_q = A.Context64(N, [MIXED[0], MIXED[0], MIXED[1], MIXED[2]])          # equal Q primes: fine for ModDown k = 2
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    ctxs = (c, dup_last, dup_pair, dup_q)
    try:
        for form in (0, 1):
            down = [
                (c32._h, pout, pin, 2, 2),                                     # u32 context
                (c._h, None, pin, 2, 2), (c._h, pout, None, 2, 2),             # null with B > 0
                (c._h, pout + 8, pin, 1, 2), (c._h, pout, pin + 8, 1, 2),      # 8-byte aligned
                (c._h, pout, pin, 0x7fffffff // L + 1, 2),                     # B * L > 2^31 - 1
                (c._h, pout, pin, 2, 0), (c._h, pout, pin, 2, L),              # k = 0, k = L
                (dup_last._h, pout, pin, 2, 2), (dup_pair._h, pout, pin, 2, 2),
                (dup_last._h, pout, pin, 2, 1),                                # k = 1: the rescale's rule
                (c._h, pin, pin, 2, 2),                                        # in place
                (c._h, bp + 8 * L * N, bp, 2, 2),                              # out starts inside in
                (c._h, bp, bp + 8 * 2 * N, 2, 2),                              # in starts inside out
                (c._h, bp + 8 * (2 * L * N - 2), bp, 2, 2),                    # last 16 bytes of in are out's first
            ]
            for h, po, pi, B, k in down:
                l0 = [t.launch_count() for t in ctxs]
                assert lib.agx_moddown64(h, po, pi, B, k, form, None) == -1, (form, po, pi, B, k)
                assert [t.launch_count() for t in ctxs] == l0
            up = [
                (c32._h, pout, pin, 2, 0, 2),
                (c._h, None, pin, 2, 0, 2), (c._h, pout, None, 2, 0, 2),
                (c._h, pout + 8, pin, 1, 0, 2), (c._h, pout, pin + 8, 1, 0, 2),
                (c._h, pout, pin, 0x7fffffff // L + 1, 0, 2),
                (c._h, pout, pin, 2, 0, 0), (c._h, pout, pin, 2, 0, L),        # count = 0, count = L
                (c._h, pout, pin, 2, L - 1, 2), (c._h, pout, pin, 2, 0xffffffff, 2),   # first + count > L
                (dup_pair._h, pout, pin, 2, 2, 2),                             # equal source primes
                (dup_last._h, pout, pin, 2, 0, 1),                             # a target equals the source
                (dup_q._h, pout, pin, 2, 1, 2),                                # a source equals a target
                (c._h, pin, pin, 2, 0, 2),                                     # in place
                (c._h, bp + 8 * 2 * N, bp, 2, 0, 2),                           # out starts inside in
                (c._h, bp, bp + 8 * 2 * N, 2, 0, 2),                           # in starts inside out
                (c._h, bp + 8 * (2 * 2 * N - 2), bp, 2, 0, 2),
            ]
            for h, po, pi, B, first, count in up:
                l0 = [t.launch_count() for t in ctxs]
                assert lib.agx_modup64(h, po, pi, B, first, count, form, None) == -1, (form, po, pi, B, first, count)
                assert [t.launch_count() for t in ctxs] == l0
            l0 = c.launch_count()
            for po, pi in ((None, None), (pout, pin), (bp, bp + 16)):              # B == 0
                assert lib.agx_moddown64(c._h, po, pi, 0, 2, form, None) == 0
                assert lib.agx_modup64(c._h, po, pi, 0, 0, 2, form, None) == 0
            assert c.launch_count() == l0
            # adjacent, not overlapping: allowed; equal Q primes do not stop a ModDown
            assert lib.agx_moddown64(c._h, bp + 8 * 2 * L * N, bp, 2, 2, form, None) == 0
            assert lib.agx_modup64(c._h, bp + 8 * 2 * 2 * N, bp, 2, 0, 2, form, None) == 0
            assert lib.agx_moddown64(dup_q._h, pout, pin, 2, 2, form, None) == 0
        with pytest.raises(ValueError):
            c.moddown(empty(1, L - 2, N), x, 2)
        with pytest.raises(ValueError):
            c.moddown(empty(2, L - 2, N), x, 0)
        with pytest.raises(ValueError):
            c.modup(empty(2, L, N), x[:, :2], 5, 2)
        with pytest.raises(A.AgxError) as e:
            c.moddown(x.view(-1)[:2 * (L - 2) * N].view(2, L - 2, N), x, 2)    # overlapping views
        assert e.value.code == -1
        torch.cuda.synchronize()
        assert torch.equal(x, snap)
    finally:
        for t in (dup_last, dup_pair, dup_q, c32):
            t.close()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    import torch
    c = ctx(N, MIXED)
    L = len(MIXED)
    d_in = dev(data(2, MIXED, N, 5))
    s3 = dev(data(2, MIXED[:3], N, 6))

    def launches(fn):
        l0 = c.launch_count()
        fn()
        torch.cuda.synchronize()
        return c.launch_count() - l0

    big = N == 32768
    for k in (2, 3):
        assert launches(lambda: c.moddown(empty(2, L - k, N), d_in, k, ntt_form=False)) == 1
        assert launches(lambda: c.moddown(empty(2, L - k, N), d_in, k, ntt_form=True)) == (4 if big else 3)
    assert launches(lambda: c.moddown(empty(2, L - 1, N), d_in, 1, ntt_form=False)) == 1
    assert launches(lambda: c.moddown(empty(2, L - 1, N), d_in, 1, ntt_form=True)) == (3 if big else 2)
    assert launches(lambda: c.modup(empty(2, L, N), s3, 1, 3, ntt_form=False)) == 1
    assert launches(lambda: c.modup(empty(2, L, N), s3, 1, 3, ntt_form=True)) == (4 if big else 3)
    s1 = s3[:, :1].contiguous()
    assert launches(lambda: c.modup(empty(2, L, N), s1, 4, 1, ntt_form=False)) == 1
    assert launches(lambda: c.modup(empty(2, L, N), s1, 4, 1, ntt_form=True)) == (3 if big else 2)
    for form in (False, True):
        assert launches(lambda: c.moddown(empty(0, L - 2, N), d_in[:0], 2, ntt_form=form)) == 0
        assert launches(lambda: c.modup(empty(0, L, N), s3[:0], 0, 3, ntt_form=form)) == 0


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N, k, first, count = 8192, 3, 2, 2
    primes = MIXED
    L = len(primes)
    c, lower, sc = ctx(N, primes), ctx(N, primes[:-k]), ctx(N, primes[first:first + count])
    x = data(4, primes, N, 9)
    xs = np.ascontiguousarray(x[:, first:first + count, :])
    want_down, want_up = moddown_mrc(x, primes, k), modup_mrc(xs, primes, first, count)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_x, d_xs = dev(x), dev(xs)                                     # the copies are ordered on s
        d_in, d_s = torch.empty_like(d_x), torch.empty_like(d_xs)
        d_in.copy_(d_x)                                                 # torch work the calls must follow
        d_s.copy_(d_xs)
        if form:
            c.fwd(d_in, stream=s)
            sc.fwd(d_s, stream=s)
        d_down, d_up = empty(4, L - k, N), empty(4, L, N)
    c.moddown(d_down, d_in, k, ntt_form=form, stream=s)
    c.modup(d_up, d_s, first, count, ntt_form=form, stream=s)
    if form:
        lower.inv(d_down, stream=s)
        c.inv(d_up, stream=s)
    s.synchronize()
    assert (d_down.cpu().numpy().view(np.uint64) == want_down).all()
    assert (d_up.cpu().numpy().view(np.uint64) == want_up).all()
