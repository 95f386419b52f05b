"""u64 RNS Galois automorphisms (agx_automorph64, Context64.automorph): sigma_g: a(X) -> a(X^g) mod X^n + 1 on [B][L][N]
batches, G elements per call, in coefficient and in evaluation form.

The CPU tests pin a numpy oracle of sigma_g against direct polynomial reduction in Python ints, the evaluation-form
index map against the textbook transform, the block property the kernels rely on, and the group laws; they also check
the compiled kernels (no local memory, the cluster attribute and barriers of the large-n instantiations).  The GPU tests
compare the library with the oracle bit for bit, the evaluation form with the existing calls composed around the
coefficient form, and run a whole rotation (automorphism + key switch) from public calls, plain and hoisted."""
import ctypes as C
import functools
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


def galois_element(n, step):
    import agilex_ntt_b200 as A
    return A.galois_element(n, step)


def eight_elements(n):
    """g = 1 (a copy), rotations by 1, -1, 2, -3, 4 and 8, and the conjugation 2n - 1"""
    return [1] + [galois_element(n, r) for r in (1, -1, 2, -3, 4, 8)] + [2 * n - 1]


# ---- the oracle
def automorph_bigint(a, g, q):
    """a(X^g) mod (X^n + 1, q) by building the polynomial of degree (n - 1) g and reducing with X^n = -1"""
    n = len(a)
    c = [0] * ((n - 1) * g + 1)
    for i, v in enumerate(a):
        c[i * g] += int(v)
    for k in range(len(c) - 1, n - 1, -1):
        c[k - n] -= c[k]
        c[k] = 0
    return [v % q for v in c[:n]]


def automorph_coeff(x, g, primes):
    """sigma_g of [..., L, n] words in coefficient form: coefficient i to i*g mod 2n, negated (x ? q - x : 0) above n"""
    n = x.shape[-1]
    idx = np.arange(n, dtype=np.int64) * g % (2 * n)
    pos, neg = idx % n, idx >= n
    q = np.array(primes, dtype=np.uint64).reshape(-1, 1)
    out = np.empty_like(x)
    out[..., pos[~neg]] = x[..., ~neg]
    out[..., pos[neg]] = np.where(x == 0, np.uint64(0), q - x)[..., neg]
    return out


def automorph_ints(a, g):
    """sigma_g of a list of signed integer coefficients"""
    n = len(a)
    out = [0] * n
    for i, v in enumerate(a):
        m = i * g % (2 * n)
        out[m % n] = -v if m >= n else v
    return out


@functools.lru_cache(maxsize=None)
def bitrevs(n):
    logn = n.bit_length() - 1
    k = np.arange(n, dtype=np.int64)
    r = np.zeros(n, dtype=np.int64)
    for b in range(logn):
        r |= ((k >> b) & 1) << (logn - 1 - b)
    return r


def eval_perm(n, g):
    """pi_g: the evaluation form of sigma_g is out = x[..., pi_g] (entry k = a(psi^(2 br(k) + 1)))"""
    br = bitrevs(n)
    return br[((g * (2 * br + 1)) % (2 * n) - 1) // 2]


def odd_elements(n):
    return list(range(1, 2 * n, 2))


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("n", (4, 8, 16, 32, 64))
def test_coefficient_oracle_is_the_definition(n):
    rng = random.Random(n)
    for q in (PRIMES[50][0], PRIMES[62][1]):
        a = [rng.randrange(q) for _ in range(n)]
        for i in rng.sample(range(n), n // 4):
            a[i] = 0                                                     # zeros: -0 stays 0
        a[0] = q - 1
        x = np.array(a, dtype=np.uint64).reshape(1, n)
        for g in odd_elements(n):
            assert [int(v) for v in automorph_coeff(x, g, [q])[0]] == automorph_bigint(a, g, q), (n, q, g)


@pytest.mark.parametrize("n", (4, 8, 16, 32, 64))
def test_evaluation_index_map_against_textbook(n):
    """textbook_fwd(sigma_g(x)) = textbook_fwd(x)[pi_g] with the minimal and a non-minimal root"""
    rng = random.Random(100 + n)
    q = PRIMES[60][0]
    x = np.array([rng.randrange(q) for _ in range(n)], dtype=np.uint64)
    gs = sorted({1, 3, 5, 2 * n - 1, pow(5, 3, 2 * n), rng.randrange(1, 2 * n, 2)})
    for psi in (O.min_psi(n, q), O.primitive_roots_2n(n, q, 2)[1]):
        X = O.textbook_fwd(x, q, psi)
        for g in gs:
            want = O.textbook_fwd(automorph_coeff(x.reshape(1, n), g, [q])[0], q, psi)
            assert (X[eval_perm(n, g)] == want).all(), (n, psi, g)


@pytest.mark.parametrize("n", (4, 64, 1024, 32768))
def test_evaluation_index_map_blocks(n):
    """What the evaluation-form kernel relies on: pi_g maps every aligned block of 2^m entries onto one aligned block,
    pi_g(j + 1) = pi_g(j) ^ 1 for even j, and pi_{g^-1} is the inverse permutation of pi_g."""
    rng = random.Random(n)
    gs = {1, 2 * n - 1, galois_element(n, 1), galois_element(n, -5), rng.randrange(1, 2 * n, 2)}
    for g in gs:
        p = eval_perm(n, g)
        assert (np.sort(p) == np.arange(n)).all()
        assert (p[1::2] == p[0::2] ^ 1).all()
        for m in range(n.bit_length()):
            blocks = (p >> m).reshape(-1, 1 << m)
            assert (blocks == blocks[:, :1]).all(), (g, m)
        pinv = eval_perm(n, pow(g, -1, 2 * n))
        assert (p[pinv] == np.arange(n)).all() and (pinv[p] == np.arange(n)).all()


@pytest.mark.parametrize("n", (4, 16, 64))
def test_group_laws(n):
    rng = random.Random(7 * n)
    primes = MIXED[:2]
    x = np.array([[rng.randrange(q) for _ in range(n)] for q in primes], dtype=np.uint64)
    x[:, ::5] = 0
    for g in odd_elements(n):
        sg = automorph_coeff(x, g, primes)
        gi = pow(g, -1, 2 * n)
        assert (automorph_coeff(sg, gi, primes) == x).all()
        for h in rng.sample(odd_elements(n), min(n, 8)):
            assert (automorph_coeff(sg, h, primes) == automorph_coeff(x, g * h % (2 * n), primes)).all()
    for a in range(-6, 7):
        for b in range(-6, 7):
            assert galois_element(n, a + b) == galois_element(n, a) * galois_element(n, b) % (2 * n)
    assert galois_element(n, 0) == 1 and galois_element(n, 1) == 5 % (2 * n)


def _cuobjdump(*args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import agilex_ntt_b200 as A
    return subprocess.run([exe, *args, A.build.build_lib()], capture_output=True, text=True, check=True).stdout


def test_automorph_kernels_use_no_local_memory():
    """Every automorphism kernel of the library's sm_100a code runs without local memory or stack, and every expected
    instantiation is there."""
    usage = _cuobjdump("--dump-resource-usage")
    found = re.findall(r"Function (\S*automorph\S*):\s*\n\s*REG:(\d+) STACK:(\d+) \S+ LOCAL:(\d+)", usage)
    names = {n for n, *_ in found}
    assert len([n for n in names if "automorph64_coeff_cluster_kernel" in n]) == 1      # CL = 2 (n = 32768)
    for k in ("automorph64_ntt_kernel", "automorph64_coeff_kernel"):
        assert any(k in n for n in names), k
    for name, reg, stack, local in found:
        assert int(local) == 0 and int(stack) == 0, name
        assert int(reg) <= 40, name                                      # three 512-thread CTAs per SM


@pytest.mark.parametrize("cl", (2,))
def test_cluster_kernels_have_their_attribute_and_barriers(cl):
    """n = 32768 gathers through distributed shared memory: the kernel must be a cl-CTA cluster, and its last
    cluster barrier must come after its last remote load, so that no CTA exits while a partner still reads it."""
    name = f"_ZN3agx32automorph64_coeff_cluster_kernelILi{cl}EEEvPmPKmPKNS_9RnsLimb64ENS_15AutomorphCall64E"
    elf = _cuobjdump("-elf")
    info = elf[re.search(r"^\.nv\.info\." + name + "$", elf, flags=re.M).end():]
    info = info[:info.index("\n.")]
    assert "EIATTR_EXPLICIT_CLUSTER" in info
    assert re.search(r"EIATTR_CTA_PER_CLUSTER\s+Format:\s+\S+\s+Value:\s+0x%x 0x1 0x1" % cl, info)
    sass = _cuobjdump("-sass")
    body = sass[sass.index("Function : " + name):]
    body = body[:body.index("Function :", 20)] if "Function :" in body[20:] else body
    ops = [m.group(1) for m in re.finditer(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\w+\s+)?([A-Z_0-9.]+)", body)]
    arrives = [i for i, op in enumerate(ops) if op.startswith("UCGABAR_ARV")]
    waits = [i for i, op in enumerate(ops) if op.startswith("UCGABAR_WAIT")]
    loads = [i for i, op in enumerate(ops) if op.split(".")[0] in ("LD", "LDS")]
    assert len(arrives) >= 2 and len(waits) >= 2 and loads
    assert arrives[0] < min(loads) and max(loads) < arrives[-1] < waits[-1]


# ------------------------------------------------------------------------------------------ on a GPU

def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(np.uint64)


def data(B, primes, N, seed, zeros=True):
    """[B][L][N] words, limb l uniform below q_l, with zeros and q_l - 1 sprinkled in"""
    mods = np.array(primes, dtype=np.uint64).reshape(1, len(primes), 1)
    x = O.synthetic_u64(B * len(primes) * N, seed, (1 << 64) - 1).reshape(B, len(primes), N) % mods
    if zeros:
        x[:, :, ::7] = 0
        x[:, :, 3::11] = (mods - np.uint64(1))[:, :, 0:1]
    return x


@pytest.fixture(scope="module")
def orc(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "native", "u64_inverse_oracle.c")
    so = str(tmp_path_factory.mktemp("u64_automorph_oracle") / "libu64oracle.so")
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


def empty(*shape):
    import torch
    return torch.empty(shape, dtype=torch.int64, device="cuda")


@gpu
@pytest.mark.parametrize("name", SETS)
@pytest.mark.parametrize("N", SIZES)
def test_coefficient_form_vs_oracle(ctx, N, name):
    """G = 1 for g = 1, 5 and 2N - 1, and G = 8, against the oracle; d_in unchanged"""
    primes = SETS[name]
    c = ctx(N, primes)
    x = data(3, primes, N, 101 + N)
    d_in = dev(x)
    for g in (1, galois_element(N, 1), 2 * N - 1):
        out = empty(3, len(primes), N)
        c.automorph(out, d_in, g, ntt_form=False)
        assert (host(out) == automorph_coeff(x, g, primes)).all(), g
    gs = eight_elements(N)
    out = empty(8, 3, len(primes), N)
    c.automorph(out, d_in, gs, ntt_form=False)
    got = host(out)
    for t, g in enumerate(gs):
        assert (got[t] == automorph_coeff(x, g, primes)).all(), (t, g)
    assert (host(d_in) == x).all()


@gpu
@pytest.mark.parametrize("roots", ("minimal", "caller"))
@pytest.mark.parametrize("N", SIZES)
def test_evaluation_form(orc, ctx, N, roots):
    """automorph(ntt_form=1)(x_hat) = fwd(automorph(ntt_form=0)(inv(x_hat))) through the public calls, and = the oracle's
    forward of the oracle's sigma_g of the oracle's inverse."""
    import torch
    primes = MIXED
    psis = caller_roots(N, primes) if roots == "caller" else None
    c = ctx(N, primes, psis)
    gs = eight_elements(N)
    x_hat = data(2, primes, N, 211 + N)
    d_in = dev(x_hat)
    got = empty(8, 2, len(primes), N)
    c.automorph(got, d_in, gs, ntt_form=True)
    t = d_in.clone()
    c.inv(t)
    want = empty(8, 2, len(primes), N)
    c.automorph(want, t, gs, ntt_form=False)
    c.fwd(want)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert (host(d_in) == x_hat).all()
    X = rns_inv(orc, x_hat, primes, psis)
    g_h = host(got)
    for k, g in enumerate(gs):
        assert (g_h[k] == rns_fwd(automorph_coeff(X, g, primes), primes, psis)).all(), g
        assert (g_h[k] == x_hat[..., eval_perm(N, g)]).all(), g


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (4, 1024, 16384, 32768))
def test_composition_and_round_trip(ctx, N, form):
    import torch
    c = ctx(N, DESC)
    L = len(DESC)
    d = dev(data(2, DESC, N, 31 + N))
    g, h = galois_element(N, 3), 2 * N - 1
    y, z, w = empty(2, L, N), empty(2, L, N), empty(2, L, N)
    c.automorph(y, d, h, ntt_form=form)
    c.automorph(z, y, g, ntt_form=form)
    c.automorph(w, d, g * h % (2 * N), ntt_form=form)
    torch.cuda.synchronize()
    assert torch.equal(z, w)
    back = empty(2, L, N)
    c.automorph(y, d, g, ntt_form=form)
    c.automorph(back, y, pow(g, -1, 2 * N), ntt_form=form)
    torch.cuda.synchronize()
    assert torch.equal(back, d)


@gpu
@pytest.mark.parametrize("form", (False, True))
@pytest.mark.parametrize("N", (32, 2048, 16384, 32768))
def test_one_call_equals_single_calls(ctx, N, form):
    import torch
    c = ctx(N, ASC)
    L = len(ASC)
    d = dev(data(2, ASC, N, 41 + N))
    gs = eight_elements(N)
    many = empty(8, 2, L, N)
    c.automorph(many, d, gs, ntt_form=form)
    for t, g in enumerate(gs):
        one = empty(2, L, N)
        c.automorph(one, d, g, ntt_form=form)
        torch.cuda.synchronize()
        assert torch.equal(many[t], one), g


@gpu
@pytest.mark.parametrize("N", (512, 8192, 16384, 32768))
def test_batches_above_two_waves(ctx, N):
    """More than two waves of CTAs in every coefficient-form geometry (16 rows per CTA at N = 512, one 64 KB row per CTA
    at 8192, one 128 KB row per CTA at 16384, a cluster of two 128 KB CTAs per row at 32768), and a grid-stride
    evaluation form over the same batch; both against the oracle on every word."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    primes = MIXED
    L = len(primes)
    rows_per_cta = {512: 16, 8192: 1, 16384: 0.5, 32768: 0.25}[N]
    B = -(-int(7 * sms * rows_per_cta) // L) + 1
    x = data(B, primes, N, 307 + N)
    c = ctx(N, primes)
    d_in = dev(x)
    gs = [galois_element(N, -1), 2 * N - 1]
    out = empty(2, B, L, N)
    for form in (False, True):
        c.automorph(out, d_in, gs, ntt_form=form)
        got = host(out)
        for t, g in enumerate(gs):
            want = x[..., eval_perm(N, g)] if form else automorph_coeff(x, g, primes)
            assert (got[t] == want).all(), (form, g)


def ternary(rng, N):
    return [rng.choice((-1, 0, 1)) for _ in range(N)]


def small(rng, N, bound):
    return [rng.randint(-bound, bound) for _ in range(N)]


def rns_of(coeffs, primes):
    """[1][L][N] residues of a list of integer coefficients"""
    return np.array([[v % q for v in coeffs] for q in primes], dtype=np.uint64).reshape(1, len(primes), len(coeffs))


def p_broadcast(primes, Pbig, B, N):
    """[B][L][N] words: P mod q_i everywhere (an element-wise factor P in either form)"""
    return dev(np.broadcast_to(np.array([Pbig % q for q in primes], dtype=np.uint64).reshape(1, -1, 1),
                               (B, len(primes), N)))


@gpu
@pytest.mark.parametrize("N", (1024, 8192))
def test_rotation_end_to_end(ctx, N):
    """A rotation from public calls only.  Q = 2 primes, P = 3 special primes (P > Q), s ternary, c = (-a*s + m + e, a)
    over Q.  The rotation key for g is (-a'*s + e' + P*sigma_g(s), a') over QP, with sigma_g(s) from automorph.
    Plain: (sigma_g(c0), 0) + moddown(modup(sigma_g(c1)) * key).  Decryption c0' + c1'*s gives sigma_g(m + e) plus the
    key switch's error, whose centred coefficients are at most N * (Q/2) * |e'|_inf / P + (N + 1) / 2 (as in the key-switch
    test of the basis conversions).  Hoisted: modup(c1) once in evaluation form, one automorph call with all three
    elements, a product with each key, moddown: the same ciphertexts bit for bit."""
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
    s, m, e = ternary(rng, N), small(rng, N, 1000), small(rng, N, ebound)
    gs = [galois_element(N, 1), galois_element(N, -3), 2 * N - 1]
    # the ciphertext over Q
    d_a = dev(data(1, Qp, N, 71, zeros=False))
    as_ = empty(1, 2, N)
    cq.polymul(as_, d_a, dev(rns_of(s, Qp)))
    c0 = empty(1, 2, N)
    cq.elementwise("add", c0, dev(rns_of(m, Qp)), dev(rns_of(e, Qp)))
    cq.elementwise("sub", c0, c0, as_)
    c1 = d_a
    # the rotation keys: sigma_g(s) over QP from the library
    d_s = dev(rns_of(s, QP))
    sig_s = empty(3, 1, L, N)
    cqp.automorph(sig_s, d_s, gs, ntt_form=False)
    keys = []
    for t in range(3):
        a2 = dev(data(1, QP, N, 80 + t, zeros=False))
        e2 = dev(rns_of(small(rng, N, ebound), QP))
        k0 = empty(1, L, N)
        cqp.polymul(k0, a2, d_s)
        cqp.elementwise("sub", k0, e2, k0)
        ps = empty(1, L, N)
        cqp.elementwise("mul", ps, sig_s[t], p_broadcast(QP, P, 1, N))
        cqp.elementwise("add", k0, k0, ps)
        keys.append((k0, a2))
    # plain: sigma_g on (c0, c1), then key-switch sigma_g(c1), all in coefficient form
    plain = []
    for t, g in enumerate(gs):
        r0, r1 = empty(1, 2, N), empty(1, 2, N)
        cq.automorph(r0, c0, g, ntt_form=False)
        cq.automorph(r1, c1, g, ntt_form=False)
        D = empty(1, L, N)
        cqp.modup(D, r1, 0, 2, ntt_form=False)
        t0, t1 = empty(1, L, N), empty(1, L, N)
        cqp.polymul(t0, D, keys[t][0])
        cqp.polymul(t1, D, keys[t][1])
        o0, o1 = empty(1, 2, N), empty(1, 2, N)
        cqp.moddown(o0, t0, k, ntt_form=False)
        cqp.moddown(o1, t1, k, ntt_form=False)
        cq.elementwise("add", o0, o0, r0)
        plain.append((o0, o1))
    # hoisted: ModUp once in evaluation form, one automorph call over QP with all three elements, MAC, ModDown
    c1_hat = c1.clone()
    cq.fwd(c1_hat)
    D_hat = empty(1, L, N)
    cqp.modup(D_hat, c1_hat, 0, 2, ntt_form=True)
    rot = empty(3, 1, L, N)
    cqp.automorph(rot, D_hat, gs, ntt_form=True)
    c0_hat = c0.clone()
    cq.fwd(c0_hat)
    rot0 = empty(3, 1, 2, N)
    cq.automorph(rot0, c0_hat, gs, ntt_form=True)
    for t in range(3):
        k0, k1 = keys[t][0].clone(), keys[t][1].clone()
        cqp.fwd(k0)
        cqp.fwd(k1)
        cqp.elementwise("mul", k0, rot[t], k0)
        cqp.elementwise("mul", k1, rot[t], k1)
        h0, h1 = empty(1, 2, N), empty(1, 2, N)
        cqp.moddown(h0, k0, k, ntt_form=True)
        cqp.moddown(h1, k1, k, ntt_form=True)
        cq.elementwise("add", h0, h0, rot0[t])
        cq.inv(h0)
        cq.inv(h1)
        torch.cuda.synchronize()
        assert torch.equal(h0, plain[t][0]) and torch.equal(h1, plain[t][1]), gs[t]
    # decryption
    sq = dev(rns_of(s, Qp))
    bound = N * (Q // 2) * ebound // P + (N + 1) // 2 + 1 + ebound
    assert bound < Q >> 60
    for t, g in enumerate(gs):
        r = empty(1, 2, N)
        cq.polymul(r, plain[t][1], sq)
        cq.elementwise("add", r, r, plain[t][0])
        cq.elementwise("sub", r, r, dev(rns_of(automorph_ints(m, g), Qp)))
        rh = host(r)[0]
        vals = [(int(rh[0, j]) * Qp[1] * pow(Qp[1], -1, Qp[0]) + int(rh[1, j]) * Qp[0] * pow(Qp[0], -1, Qp[1])) % Q
                for j in range(N)]
        worst = max(min(v, Q - v) for v in vals)
        assert worst <= bound, (g, worst, bound)


def garr(*gs):
    return (C.c_uint32 * max(len(gs), 1))(*gs)


@gpu
def test_refusals_and_empty_calls(A, ctx):
    import torch
    N = 1024
    lib = A.lib()
    c = ctx(N, MIXED)
    L = len(MIXED)
    x = dev(data(2, MIXED, N, 3))
    snap = x.clone()
    o = torch.full((3, 2, L, N), 7, dtype=torch.int64, device="cuda")
    osnap = o.clone()
    pin, pout = x.data_ptr(), o.data_ptr()
    big = torch.zeros(8 * L * N + 2, dtype=torch.int64, device="cuda")
    bp = big.data_ptr()
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    torch.cuda.synchronize()
    ok = garr(3, 5)
    try:
        for form in (0, 1):
            bad = [
                (c32._h, pout, pin, 2, ok, 2),                                   # u32 context
                (c._h, None, pin, 2, ok, 2), (c._h, pout, None, 2, ok, 2),       # null with B > 0
                (c._h, pout, pin, 2, None, 2),                                   # null galois with G > 0
                (c._h, pout + 8, pin, 1, ok, 2), (c._h, pout, pin + 8, 1, ok, 2),   # 8-byte aligned
                (c._h, pout, pin, 0x7fffffff // (2 * L) + 1, ok, 2),             # G * B * L > 2^31 - 1
                (c._h, pout, pin, 2, garr(2), 1), (c._h, pout, pin, 2, garr(0), 1),   # even, 0
                (c._h, pout, pin, 2, garr(2 * N), 1), (c._h, pout, pin, 2, garr(2 * N + 1), 1),   # >= 2n
                (c._h, pout, pin, 2, garr(0xffffffff), 1), (c._h, pout, pin, 2, garr(3, 5, 4), 3),
                (c._h, pin, pin, 2, ok, 1),                                      # in place
                (c._h, bp + 8 * L * N, bp, 2, ok, 2),                            # out starts inside in
                (c._h, bp, bp + 8 * 3 * L * N, 2, ok, 2),                        # in starts inside out
                (c._h, bp + 8 * (2 * L * N - 2), bp, 2, ok, 1),                  # last 16 bytes of in are out's first
            ]
            for h, po, pi, B, gp, G in bad:
                l0 = [c.launch_count(), c32.launch_count()]
                assert lib.agx_automorph64(h, po, pi, B, gp, G, form, None) == -1, (form, po, pi, B, G)
                assert [c.launch_count(), c32.launch_count()] == l0
            l0 = c.launch_count()
            assert lib.agx_automorph64(c._h, pout, pin, 2, garr(*([3] * 65)), 65, form, None) == -2
            for po, pi in ((None, None), (pout, pin), (bp, bp + 16)):            # B == 0
                assert lib.agx_automorph64(c._h, po, pi, 0, ok, 2, form, None) == 0
            assert lib.agx_automorph64(c._h, pout, pin, 2, None, 0, form, None) == 0      # G == 0
            assert lib.agx_automorph64(c._h, pin, pin, 2, None, 0, form, None) == 0
            assert c.launch_count() == l0
            torch.cuda.synchronize()
            assert torch.equal(o, osnap)
            # adjacent, not overlapping: allowed (one launch)
            assert lib.agx_automorph64(c._h, bp + 8 * 2 * L * N, bp, 2, ok, 2, form, None) == 0
            assert c.launch_count() == l0 + 1
        with pytest.raises(ValueError):
            c.automorph(empty(2, L, N), x, [3, 5])
        with pytest.raises(ValueError):
            c.automorph(empty(1, 2, L, N), x, 3)
        with pytest.raises(ValueError):
            c.automorph(empty(2, L, N), x[:, :2], 3)
        for g in (2**32 + 5, -1):                                        # not a 32-bit element: never wrapped
            with pytest.raises(ValueError):
                c.automorph(empty(2, L, N), x, g)
        with pytest.raises(ValueError):
            c.automorph(empty(2, 2, L, N), x, [5, 2**32 + 5])
        with pytest.raises(A.AgxError) as e:
            c.automorph(empty(2, L, N), x, 4)
        assert e.value.code == -1
        torch.cuda.synchronize()
        assert torch.equal(x, snap)
    finally:
        c32.close()


@gpu
@pytest.mark.parametrize("N", (32, 1024, 16384, 32768))
def test_launch_counts(ctx, N):
    import torch
    c = ctx(N, MIXED)
    L = len(MIXED)
    d_in = dev(data(2, MIXED, N, 5))
    for form in (False, True):
        for gs in (galois_element(N, 1), eight_elements(N)):
            out = empty(2, L, N) if isinstance(gs, int) else empty(8, 2, L, N)
            l0 = c.launch_count()
            c.automorph(out, d_in, gs, ntt_form=form)
            torch.cuda.synchronize()
            assert c.launch_count() - l0 == 1, (form, gs)


@gpu
@pytest.mark.parametrize("form", (False, True))
def test_side_stream(ctx, form):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 16384
    primes = MIXED
    L = len(primes)
    c = ctx(N, primes)
    gs = eight_elements(N)
    x = data(4, primes, N, 9)
    want = np.stack([x[..., eval_perm(N, g)] if form else automorph_coeff(x, g, primes) for g in gs])
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_x = dev(x)                                                    # the copy is ordered on s
        d_in = torch.empty_like(d_x)
        d_in.copy_(d_x)                                                 # torch work the call must follow
        d_out = empty(8, 4, L, N)
    c.automorph(d_out, d_in, gs, ntt_form=form, stream=s)
    s.synchronize()
    assert (d_out.cpu().numpy().view(np.uint64) == want).all()
