"""u64 RNS rescale (agx_rescale64 / Context64.rescale): [B][L][N] -> [B][L-1][N], the division by the last prime
q_L' = q_{L-1} with rounding, in coefficient and in evaluation form.

Definition: for the CRT value X in [0, Q) of a coefficient's L residues, the result is the residue vector of
Y = floor((X + h) / q_L') mod Q' over q_0 .. q_{L-2}, with h = floor(q_L' / 2) and Q' = Q / q_L'.  The CPU tests pin the
RNS formula used as the oracle here, y_i = (x_i - (u - h)) * q_L'^-1 mod q_i with u = (x_{L-1} + h) mod q_L', against
that big-int definition, and check on the compiled library that the new kernels use no local memory.  The GPU tests
compare the library with the oracle bit for bit, the evaluation form with the existing calls composed around the
coefficient form, and a chain of two rescales through per-level contexts with big ints."""
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


PRIMES = {b: find_primes(b, 3) for b in (50, 60, 62)}
MIXED = [PRIMES[50][0], PRIMES[60][0], PRIMES[62][0]]                  # ascending: u < q_L' can exceed q_0, q_1
DESC = MIXED[::-1]                                                     # descending: divide by the 50-bit prime
FOUR = [PRIMES[62][1], PRIMES[50][1], PRIMES[60][1], PRIMES[62][2]]    # L = 4
SETS = {"ascending": MIXED, "descending": DESC, "four": FOUR}


# ---- big ints and the RNS oracle
def crt(res, primes):
    Q = prod(primes)
    X = 0
    for r, q in zip(res, primes):
        m = Q // q
        X += int(r) * m * pow(m, -1, q)
    return X % Q


def rescale_bigint(X, primes):
    qL = primes[-1]
    return ((X + qL // 2) // qL) % prod(primes[:-1])


def rescale_rns(x, primes):
    """[B][L][N] residues -> [B][L-1][N]: y_i = (x_i - (u - h)) * q_L'^-1 mod q_i, u = (x_{L-1} + h) mod q_L'."""
    qL, h = primes[-1], primes[-1] // 2
    u = (x[:, -1, :].astype(object) + h) % qL
    out = np.empty((x.shape[0], len(primes) - 1, x.shape[2]), dtype=np.uint64)
    for i, q in enumerate(primes[:-1]):
        out[:, i, :] = ((x[:, i, :].astype(object) - (u - h)) * pow(qL, -1, q) % q).astype(np.uint64)
    return out


def boundary_values(primes, rng, m_count=6):
    """X = 0, Q - 1, values around Q/2, and the rounding boundary m*q_L' + h and m*q_L' + h - 1."""
    Q, qL = prod(primes), primes[-1]
    h = qL // 2
    Xs = [0, 1, Q - 1, Q - 2, Q // 2 - 1, Q // 2, Q // 2 + 1, (Q + 1) // 2, h, h - 1, qL - 1, qL]
    ms = [0, 1, Q // qL - 1, Q // qL // 2] + [rng.randrange(Q // qL) for _ in range(m_count)]
    for m in ms:
        Xs += [m * qL + h, m * qL + h - 1]
    return [X for X in Xs if 0 <= X < Q]


def residues(Xs, primes):
    """[1][L][len(Xs)] residues of the big ints Xs"""
    return np.array([[X % q for X in Xs] for q in primes], dtype=np.uint64).reshape(1, len(primes), len(Xs))


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("name", SETS)
def test_rns_oracle_is_the_definition(name):
    primes = SETS[name]
    rng = random.Random(7 + len(name))
    Q = prod(primes)
    Xs = boundary_values(primes, rng) + [rng.randrange(Q) for _ in range(2000)]
    got = rescale_rns(residues(Xs, primes), primes)[0]
    for j, X in enumerate(Xs):
        Y = rescale_bigint(X, primes)
        assert [int(v) for v in got[:, j]] == [Y % q for q in primes[:-1]], (name, X)
    # centred reading of X gives the same residues (Q / q_L' = Q')
    X = Q - 5
    assert rescale_bigint(X, primes) % primes[0] == ((X - Q + primes[-1] // 2) // primes[-1]) % primes[0]


def _cuobjdump(*args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import agilex_ntt_b200 as A
    return subprocess.run([exe, *args, A.build.build_lib()], capture_output=True, text=True, check=True).stdout


def test_rescale_kernels_use_no_local_memory():
    """Every rescale kernel of the library's sm_100a code, the frame kernels at the 128-register cap included, runs
    without spills: no local memory."""
    usage = _cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*rescale\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    names = {n for n, *_ in found}
    assert len([n for n in names if "ref_u64_rescale_fwd_kernel" in n]) == 5        # NT = 32 .. 512
    assert len([n for n in names if "ref_u64_rescale_inv_frame_kernel" in n]) == 5
    for k in ("rescale64_coeff_kernel", "ref_fwd_u64_rescale_kernel", "ref_inv_u64_rescale_kernel"):
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


@pytest.fixture(scope="module")
def orc(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "native", "u64_inverse_oracle.c")
    so = str(tmp_path_factory.mktemp("u64_rescale_oracle") / "libu64oracle.so")
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


def out_like(x):
    import torch
    return torch.empty((x.shape[0], x.shape[1] - 1, x.shape[2]), dtype=torch.int64, device="cuda")


@gpu
@pytest.mark.parametrize("name", SETS)
@pytest.mark.parametrize("N", SIZES)
def test_coefficient_form_vs_oracle(ctx, N, name):
    """Bit-exact against the RNS oracle, with the constructed boundary values in polynomial 0."""
    primes = SETS[name]
    c = ctx(N, primes)
    L = len(primes)
    flat = data(3, primes, N, 101 + N).transpose(1, 0, 2).reshape(L, 3 * N)   # [L][3N]: polynomial-major columns
    bv = residues(boundary_values(primes, random.Random(N)), primes)[0]
    k = min(flat.shape[1], bv.shape[1])
    flat[:, :k] = bv[:, :k]
    x = np.ascontiguousarray(flat.reshape(L, 3, N).transpose(1, 0, 2))
    d_in = dev(x)
    d_out = out_like(d_in)
    c.rescale(d_out, d_in, ntt_form=False)
    assert (host(d_out) == rescale_rns(x, primes)).all()
    assert (host(d_in) == x).all()                                      # d_in is not modified


@gpu
@pytest.mark.parametrize("case", ("ascending", "descending", "four", "ascending-caller-roots", "four-caller-roots"))
@pytest.mark.parametrize("N", SIZES)
def test_evaluation_form(orc, ctx, N, case):
    """rescale(ntt_form=1)(x_hat) = fwd_{L-1}(rescale(ntt_form=0)(inv_L(x_hat))) through the existing calls and a context
    over the first L - 1 primes, and = the oracle's per-limb forward of the big-int result."""
    import torch
    name = case.split("-")[0]
    primes = SETS[name]
    psis = caller_roots(N, primes) if "caller" in case else None
    c, lower = ctx(N, primes, psis), ctx(N, primes[:-1], psis[:-1] if psis else None)
    x_hat = data(2, primes, N, 211 + N)
    d_in = dev(x_hat)
    got = out_like(d_in)
    c.rescale(got, d_in, ntt_form=True)
    t = d_in.clone()
    c.inv(t)
    want = out_like(d_in)
    c.rescale(want, t, ntt_form=False)
    lower.fwd(want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert (host(d_in) == x_hat).all()
    X = rns_inv(orc, x_hat, primes, psis)
    assert (host(got) == rns_fwd(rescale_rns(X, primes), primes[:-1], psis[:-1] if psis else None)).all()


@gpu
@pytest.mark.parametrize("N", (16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """B * (L - 1) frames of more than two waves of frame CTAs: the evaluation form equals the existing calls composed
    around the coefficient form on every polynomial; the coefficient form equals the oracle on a sample of them."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = -(-(2 * sms + 5) // 3)
    c, lower = ctx(N, FOUR), ctx(N, FOUR[:3])
    x = data(B, FOUR, N, 307 + N)
    d_in = dev(x)
    coeff = out_like(d_in)
    c.rescale(coeff, d_in, ntt_form=False)
    sample = sorted({0, 1, B // 2, B - 2, B - 1} | set(random.Random(N).sample(range(B), 4)))
    assert (host(coeff)[sample] == rescale_rns(x[sample], FOUR)).all()
    got = out_like(d_in)
    c.rescale(got, d_in, ntt_form=True)
    t = d_in.clone()
    c.inv(t)
    want = out_like(d_in)
    c.rescale(want, t, ntt_form=False)
    lower.fwd(want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)


@gpu
@pytest.mark.parametrize("roots", ("minimal", "caller"))
@pytest.mark.parametrize("N", (32, 1024, 32768))
def test_chain_of_levels(A, ctx, N, roots):
    """L = 4 -> 3 -> 2 through per-level contexts equals floor((floor((X + h3) / q3) + h2) / q2) in big ints, in both
    forms; each lower level's tables are the full context's first limbs."""
    import torch
    psis = caller_roots(N, FOUR) if roots == "caller" else None
    lv = [ctx(N, FOUR[:L], psis[:L] if psis else None) for L in (4, 3, 2)]
    for k, low in ((1, lv[1]), (2, lv[2])):
        for l in range(4 - k):
            for inverse in (False, True):
                r, p = low.tables(l, inverse)
                R, P = lv[0].tables(l, inverse)
                assert (r == R).all() and (p == P).all(), (k, l, inverse)
    x = data(2, FOUR, N, 401 + N)
    d = dev(x)
    y = out_like(d)
    lv[0].rescale(y, d, ntt_form=False)
    z = out_like(y)
    lv[1].rescale(z, y, ntt_form=False)
    got = host(z).reshape(2, 2, N)
    q2, q3 = FOUR[2], FOUR[3]
    for b in range(2):
        for j in range(N):
            X = crt(x[b, :, j], FOUR)
            Z = ((X + q3 // 2) // q3 + q2 // 2) // q2
            assert [int(got[b, 0, j]), int(got[b, 1, j])] == [Z % FOUR[0], Z % FOUR[1]], (b, j)
    # the same chain in evaluation form
    e = d.clone()
    lv[0].fwd(e)
    ye = out_like(e)
    lv[0].rescale(ye, e, ntt_form=True)
    ze = out_like(ye)
    lv[1].rescale(ze, ye, ntt_form=True)
    lv[2].inv(ze)
    torch.cuda.synchronize()
    assert torch.equal(ze, z)


@gpu
def test_refusals_and_empty_batches(A, ctx):
    import torch
    N = 1024
    lib = A.lib()
    c = ctx(N, MIXED)
    x = dev(data(2, MIXED, N, 3))
    o = out_like(x)
    snap = x.clone()
    pin, pout = x.data_ptr(), o.data_ptr()
    words_in = 2 * 3 * N
    big = torch.zeros(words_in + 2 * 2 * N + 2, dtype=torch.int64, device="cuda")   # room for overlapping ranges
    bp = big.data_ptr()
    one = ctx(N, [MIXED[0]])
    dup = A.Context64(N, [MIXED[2], MIXED[0], MIXED[2]])                # last prime repeats an earlier one
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    try:
        for form in (0, 1):
            cases = [
                (c32._h, pout, pin, 2),                                 # u32 context
                (one._h, pout, pin, 2),                                 # L = 1
                (dup._h, pout, pin, 2),                                 # q_{L-1} = q_0: no inverse
                (c._h, None, pin, 2), (c._h, pout, None, 2),            # null with B > 0
                (c._h, pout + 8, pin, 1), (c._h, pout, pin + 8, 1),     # 8-byte aligned
                (c._h, pout, pin, 0x7fffffff // 3 + 1),                 # B * L > 2^31 - 1
                (c._h, pin, pin, 2),                                    # in place
                (c._h, bp + 8 * 3 * N, bp, 2),                          # out starts inside in
                (c._h, bp, bp + 8 * 2 * N, 2),                          # in starts inside out
                (c._h, bp + 8 * (words_in - 2), bp, 2),                 # last 16 bytes of in are the first of out
            ]
            for h, po, pi, B in cases:
                l0 = [k.launch_count() for k in (c, one, dup)]
                assert lib.agx_rescale64(h, po, pi, B, form, None) == -1, (form, po, pi, B)
                assert [k.launch_count() for k in (c, one, dup)] == l0
            l0 = c.launch_count()
            assert lib.agx_rescale64(c._h, None, None, 0, form, None) == 0     # B == 0
            assert lib.agx_rescale64(c._h, pout, pin, 0, form, None) == 0
            assert lib.agx_rescale64(c._h, bp, bp + 8 * 2 * N, 0, form, None) == 0
            assert c.launch_count() == l0
            # adjacent, not overlapping: allowed
            assert lib.agx_rescale64(c._h, bp + 8 * words_in, bp, 2, form, None) == 0
        with pytest.raises(ValueError):
            c.rescale(out_like(x)[:1], x)
        with pytest.raises(ValueError):
            c.rescale(x.clone(), x)
        with pytest.raises(A.AgxError) as e:
            c.rescale(x.view(-1)[:2 * 2 * N].view(2, 2, N), x)               # overlapping views
        assert e.value.code == -1
        torch.cuda.synchronize()
        assert torch.equal(x, snap)
    finally:
        dup.close()
        c32.close()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    import torch
    c = ctx(N, MIXED)
    d_in = dev(data(2, MIXED, N, 5))
    d_out = out_like(d_in)

    def launches(fn):
        l0 = c.launch_count()
        fn()
        torch.cuda.synchronize()
        return c.launch_count() - l0

    assert launches(lambda: c.rescale(d_out, d_in, ntt_form=False)) == 1
    assert launches(lambda: c.rescale(d_out, d_in, ntt_form=True)) == (3 if N == 32768 else 2)
    for form in (False, True):
        assert launches(lambda: c.rescale(d_out[:0], d_in[:0], ntt_form=form)) == 0


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    c, lower = ctx(N, MIXED), ctx(N, MIXED[:-1])
    x = data(4, MIXED, N, 9)
    want = rescale_rns(x, MIXED)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_x = dev(x)                                                    # the copy is ordered on s
        d_in = torch.empty_like(d_x)
        d_in.copy_(d_x)                                                 # torch work the rescale must follow
        if form:
            c.fwd(d_in, stream=s)
        d_out = out_like(d_in)
    c.rescale(d_out, d_in, ntt_form=form, stream=s)
    if form:
        lower.inv(d_out, stream=s)
    s.synchronize()
    assert (d_out.cpu().numpy().view(np.uint64) == want).all()
