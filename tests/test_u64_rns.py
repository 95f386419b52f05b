"""u64 RNS batches (agx_create64 / Context64): [B][L][N] forward, inverse, products and element-wise arithmetic over L
primes of 50-62 bits, with the tables built on the device.

The CPU tests pin the per-limb oracle composed here (the C restatement of the forward, the C oracle of the inverse in
tests/native/u64_inverse_oracle.c) against the big-int definitions.  The GPU tests compare the library with that oracle
bit for bit, and every limb's slice of a batched call with the single-modulus call (agx_ref_*_dev) on it."""
import ctypes as C
import os
import re
import shutil
import subprocess

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
MIXED = [PRIMES[50][0], PRIMES[60][0], PRIMES[62][0]]                  # L = 3, one of each width
FOUR = [PRIMES[62][1], PRIMES[50][1], PRIMES[60][1], PRIMES[62][2]]    # L = 4


@pytest.fixture(scope="module")
def orc(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "native", "u64_inverse_oracle.c")
    so = str(tmp_path_factory.mktemp("u64_rns_oracle") / "libu64oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc") or "cc"
    base = [cc, "-O2", "-std=c11", "-fPIC", "-shared", "-o", so, src]
    if subprocess.run(base + ["-fopenmp"], capture_output=True).returncode != 0:
        subprocess.run(base + ["-Wno-unknown-pragmas"], check=True)
    L = C.CDLL(so)
    L.orc_inv_u64.argtypes = [C.c_uint32, _u64p, C.c_uint64, _u64p, C.c_size_t, C.c_int]
    L.orc_polymul_schoolbook_u64.argtypes = [C.c_uint32, C.c_uint64, _u64p, _u64p, _u64p]
    return L


def _p(a):
    assert a.dtype == np.uint64 and a.flags.c_contiguous
    return a.ctypes.data_as(_u64p)


_TABLES = {}


def tables(N, q, psi=None):
    key = (N, q, psi)
    if key not in _TABLES:
        _TABLES[key] = O.tables_u64(N, q, psi) + O.tables_u64(N, q, psi, inverse=True)
    return _TABLES[key]


def data(B, primes, N, seed, lazy=1):
    """[B][L][N] words, limb l uniform below lazy * q_l."""
    L = len(primes)
    mods = np.array([lazy * q for q in primes], dtype=np.uint64).reshape(1, L, 1)
    return O.synthetic_u64(B * L * N, seed, (1 << 64) - 1).reshape(B, L, N) % mods


# ---- the RNS oracle: per limb, from the single-modulus oracles
def rns_map(fn, x, primes):
    out = np.empty_like(x)
    for l, q in enumerate(primes):
        out[:, l, :] = fn(np.ascontiguousarray(x[:, l, :]), q, l).reshape(x.shape[0], -1)
    return out


def rns_fwd(x, primes, psis=None):
    N = x.shape[-1]

    def one(v, q, l):
        tw, pre, _, _ = tables(N, q, psis[l] if psis else None)
        return O.ref_fwd_u64(v, v, q, tw, pre, v.shape[0])
    return rns_map(one, x, primes)


def rns_inv(orc, X, primes):
    N = X.shape[-1]

    def one(v, q, l):
        y = np.ascontiguousarray(v, dtype=np.uint64).copy()
        orc.orc_inv_u64(N, _p(y), q, _p(tables(N, q)[2]), y.size // N, max(1, min(O.max_threads(), 16)))
        return y
    return rns_map(one, X, primes)


def rns_pointwise(x, y, primes):
    out = np.empty_like(x)
    for l, q in enumerate(primes):
        out[:, l, :] = np.array([int(u) * int(v) % q for u, v in zip(x[:, l, :].ravel(), y[:, l, :].ravel())],
                                dtype=np.uint64).reshape(x.shape[0], -1)
    return out


def rns_polymul(orc, a, b, primes):
    return rns_inv(orc, rns_pointwise(rns_fwd(a, primes), rns_fwd(b, primes), primes), primes)


# ------------------------------------------------------------------------------------------ on the CPU

@pytest.mark.parametrize("bits", (50, 60, 62))
def test_prime_finder(bits):
    ps = PRIMES[bits]
    assert len(set(ps)) == 3
    for q in ps:
        assert q.bit_length() == bits and q % (1 << 16) == 1 and O.is_prime(q)
    assert O.U64_PRIMES[bits] % (1 << 16) == 1 and O.U64_PRIMES[bits].bit_length() == bits


@pytest.mark.parametrize("N", [4, 16, 32])
def test_rns_oracle_is_the_definition(orc, N):
    B = 2
    x = data(B, MIXED, N, 3 + N, lazy=4)
    X = rns_fwd(x, MIXED)
    a, b = data(B, MIXED, N, 5 + N), data(B, MIXED, N, 7 + N)
    Xl = data(B, MIXED, N, 9 + N, lazy=2)
    Y, C_ = rns_inv(orc, Xl, MIXED), rns_polymul(orc, a, b, MIXED)
    for l, q in enumerate(MIXED):
        psi = O.min_psi(N, q)
        for f in range(B):
            assert (X[f, l] == O.textbook_fwd(x[f, l] % np.uint64(q), q, psi)).all()
            assert (Y[f, l] == O.textbook_inv(Xl[f, l], q, psi)).all()
            assert (C_[f, l] == O.textbook_polymul(a[f, l], b[f, l], q)).all()


def _cuobjdump(*args):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import agilex_ntt_b200 as A
    return subprocess.run([exe, *args, A.build.build_lib()], capture_output=True, text=True, check=True).stdout


PAIR_KERNEL = "_ZN3agx29ref_u64_rns_frame_pair_kernelEPKmPmS1_S1_PKNS_9RnsLimb64Ej"


def test_pair_kernel_is_a_cluster_with_its_barrier():
    """The in-place forward at N = 32768 is safe only because both CTAs of a frame form a 2-CTA cluster and each waits
    on the cluster barrier before any global store: checked on the sm_100a code of the library."""
    elf = _cuobjdump("-elf")
    info = elf[re.search(r"^\.nv\.info\." + PAIR_KERNEL + "$", elf, flags=re.M).end():]   # the section's body
    info = info[:info.index("\n.")]
    assert "EIATTR_EXPLICIT_CLUSTER" in info
    assert re.search(r"EIATTR_CTA_PER_CLUSTER\s+Format:\s+\S+\s+Value:\s+0x2 0x1 0x1", info)
    sass = _cuobjdump("-sass")
    body = sass[sass.index("Function : " + PAIR_KERNEL):]
    body = body[:body.index("Function :", 20)] if "Function :" in body[20:] else body
    ops = [m.group(1) for m in re.finditer(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\w+\s+)?([A-Z_0-9.]+)", body)]
    arrive, wait = ops.index("UCGABAR_ARV"), ops.index("UCGABAR_WAIT")
    stores = [i for i, op in enumerate(ops) if op.startswith("STG")]
    assert arrive < wait and stores and min(stores) > wait


# ------------------------------------------------------------------------------------------ on a GPU

def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(np.uint64)


@pytest.fixture(scope="module")
def A():
    import agilex_ntt_b200 as A
    return A


@pytest.fixture(scope="module")
def P(A):
    p = A.RefPipeline()
    yield p
    p.close()


_CTX = {}


@pytest.fixture(scope="module")
def ctx(A):
    """Context64 per (N, primes), kept for the module."""
    def get(N, primes):
        key = (N, tuple(primes))
        if key not in _CTX:
            _CTX[key] = A.Context64(N, primes)
        return _CTX[key]
    yield get
    for c in _CTX.values():
        c.close()
    _CTX.clear()


@gpu
@pytest.mark.parametrize("N", [4, 1024, 32768])
def test_tables(A, ctx, N):
    c = ctx(N, MIXED)
    for l, q in enumerate(MIXED):
        assert c.psi(l) == O.min_psi(N, q)
        for inverse in (False, True):
            r, p = c.tables(l, inverse)
            want_r, want_p = O.tables_u64(N, q, inverse=inverse)
            assert (r == want_r).all() and (p == want_p).all(), (l, inverse)
    psis = [O.primitive_roots_2n(N, q, 2)[1] for q in MIXED]              # non-minimal roots
    c2 = A.Context64(N, MIXED, psi=psis)
    try:
        for l, q in enumerate(MIXED):
            assert c2.psi(l) == psis[l]
            for inverse in (False, True):
                r, p = c2.tables(l, inverse)
                want_r, want_p = O.tables_u64(N, q, psis[l], inverse=inverse)
                assert (r == want_r).all() and (p == want_p).all(), (l, inverse)
    finally:
        c2.close()


@gpu
def test_refusals(A, ctx):
    import torch
    N, q = 1024, PRIMES[60][0]
    composite = next(k * (1 << 16) + 1 for k in range(3, 1000) if not O.is_prime(k * (1 << 16) + 1))
    bad_parms = [
        (N, [q, composite]),                     # not prime (= 1 mod 2n)
        (N, [q + 1]),                            # even
        (N, [O.U64_PRIMES[63]]),                 # prime, >= 2^62
        (N, [7681]),                             # prime, not 1 mod 2n
        (2, [q]), (65536, [q]),                  # n out of range
        (N, []), (N, [q] * 65),                  # nlimbs 0 and 65
    ]
    assert O.is_prime(7681) and (7681 - 1) % (2 * N) != 0
    for n, primes in bad_parms:
        with pytest.raises(A.AgxError) as e:
            A.Context64(n, primes)
        assert e.value.code == -1, (n, primes)
    psi = O.min_psi(N, q)
    for bad_psi in (psi * psi % q, 0, q + psi, 1):                    # psi^n != -1 (or not a residue)
        with pytest.raises(A.AgxError) as e:
            A.Context64(N, [q], psi=[bad_psi])
        assert e.value.code == -1
    c = ctx(N, [q])
    t = dev(data(2, [q], N, 1))
    for call in (lambda: A.lib().agx_ntt64_fwd(c._h, t.data_ptr() + 8, 1, None),           # 8-byte aligned
                 lambda: A.lib().agx_ntt64_inv(c._h, t.data_ptr() + 8, 1, None),
                 lambda: A.lib().agx_polymul64(c._h, t.data_ptr(), t.data_ptr() + 8, t.data_ptr(), 1, None),
                 lambda: A.lib().agx_polymul64_by_spectrum(c._h, t.data_ptr(), t.data_ptr(), t.data_ptr() + 8, 1, None),
                 lambda: A.lib().agx_elementwise64(c._h, 0, t.data_ptr() + 8, t.data_ptr(), t.data_ptr(), 1, None),
                 lambda: A.lib().agx_elementwise64(c._h, 4, t.data_ptr(), t.data_ptr(), t.data_ptr(), 1, None)):
        assert call() == -1
    # u32 calls on a u64 context, u64 calls on a u32 context
    t32 = torch.zeros(N, dtype=torch.int32, device="cuda")
    for call in (lambda: A.lib().agx_ntt_fwd(c._h, t32.data_ptr(), 1, None),
                 lambda: A.lib().agx_ntt_inv(c._h, t32.data_ptr(), 1, None),
                 lambda: A.lib().agx_polymul(c._h, t32.data_ptr(), t32.data_ptr(), t32.data_ptr(), 1, None),
                 lambda: A.lib().agx_elementwise(c._h, 0, t32.data_ptr(), t32.data_ptr(), t32.data_ptr(), 1, None),
                 lambda: A.lib().agx_get_psi(c._h, 0, C.byref(C.c_uint32()))):
        assert call() == -1
    c32 = A.Context(N, [O.SEAL_PRIMES_30[0]])
    try:
        for call in (lambda: A.lib().agx_ntt64_fwd(c32._h, t.data_ptr(), 1, None),
                     lambda: A.lib().agx_ntt64_inv(c32._h, t.data_ptr(), 1, None),
                     lambda: A.lib().agx_polymul64(c32._h, t.data_ptr(), t.data_ptr(), t.data_ptr(), 1, None),
                     lambda: A.lib().agx_polymul64_by_spectrum(c32._h, t.data_ptr(), t.data_ptr(), t.data_ptr(), 1, None),
                     lambda: A.lib().agx_elementwise64(c32._h, 0, t.data_ptr(), t.data_ptr(), t.data_ptr(), 1, None),
                     lambda: A.lib().agx_get_psi64(c32._h, 0, C.byref(C.c_uint64()))):
            assert call() == -1
    finally:
        c32.close()
    x = data(2, [q], N, 2)
    t = dev(x)
    c.fwd(t)
    c.inv(t)
    assert (host(t) == x).all()                                     # the context still computes


@gpu
@pytest.mark.parametrize("N", SIZES)
def test_fwd_inv_vs_oracle(orc, ctx, N):
    """L = 3 of mixed widths, 2 polynomials; lazy inputs (< 4q forward, < 2q inverse); round trip."""
    c = ctx(N, MIXED)
    x = data(2, MIXED, N, 11 + N, lazy=4)
    t = dev(x)
    c.fwd(t)
    X = host(t).reshape(x.shape)
    assert (X == rns_fwd(x, MIXED)).all()
    c.inv(t)
    assert (host(t).reshape(x.shape) == x % np.array(MIXED, dtype=np.uint64).reshape(1, 3, 1)).all()
    Xl = data(2, MIXED, N, 13 + N, lazy=2)
    t = dev(Xl)
    c.inv(t)
    assert (host(t).reshape(Xl.shape) == rns_inv(orc, Xl, MIXED)).all()


def _ref_tables(c, l):
    return [dev(a) for a in c.tables(l) + c.tables(l, True)]


@gpu
@pytest.mark.parametrize("op", ("fwd", "inv", "polymul", "by_spectrum"))
@pytest.mark.parametrize("N", [1024, 16384, 32768])
def test_equals_single_modulus_calls(P, ctx, N, op):
    """L = 4, B * L frames of more than two waves of CTAs: every limb's slice equals the agx_ref_*_dev call on it."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    per_sm = max(1, 512 // (N // 32)) if N <= 16384 else 1
    frames = 2 * sms * per_sm + 5
    B = -(-frames // 4)
    c = ctx(N, FOUR)
    lazy = {"fwd": 4, "inv": 2}.get(op, 1)
    a = dev(data(B, FOUR, N, 17 + N, lazy=lazy))
    b = dev(data(B, FOUR, N, 19 + N))
    if op == "by_spectrum":
        c.fwd(b)
    a3, b3 = a.view(B, 4, N), b.view(B, 4, N)
    want = []
    for l, q in enumerate(FOUR):
        tw, pre, itw, ipre = _ref_tables(c, l)
        al, bl = a3[:, l, :].contiguous(), b3[:, l, :].contiguous()
        out = torch.empty_like(al)
        if op == "fwd":
            P.fwd_dev(N, al, al, out, q, tw, pre, B)
        elif op == "inv":
            P.inv_dev(N, al, out, q, itw, ipre, B)
        elif op == "polymul":
            P.polymul_dev(N, out, al, bl, q, tw, pre, itw, ipre, B)
        else:
            P.polymul_by_spectrum_dev(N, out, al, bl, q, tw, pre, itw, ipre, B)
        want.append(out)
    if op == "fwd":
        c.fwd(a)
        got = a
    elif op == "inv":
        c.inv(a)
        got = a
    else:
        got = torch.empty_like(a)
        (c.polymul if op == "polymul" else c.polymul_by_spectrum)(got, a, b)
    torch.cuda.synchronize()
    g3 = got.view(B, 4, N)
    for l in range(4):
        assert torch.equal(g3[:, l, :], want[l]), l


@gpu
def test_in_place_fwd_32768_is_one_launch(P, ctx):
    """Result and launch count of the in-place forward at N = 32768.  This cannot show a missing cluster barrier: the two
    CTAs of a cluster are co-scheduled, so the write-after-read race it prevents would almost never fire here.  The
    barrier is pinned by test_pair_kernel_is_a_cluster_with_its_barrier, on the compiled code."""
    import torch
    N = 32768
    c = ctx(N, MIXED)
    x = data(3, MIXED, N, 23, lazy=4)
    t = dev(x)
    l0 = c.launch_count()
    c.fwd(t)
    torch.cuda.synchronize()
    assert c.launch_count() - l0 == 1
    got = host(t).reshape(x.shape)
    for l, q in enumerate(MIXED):
        tw, pre, _, _ = _ref_tables(c, l)
        src = dev(np.ascontiguousarray(x[:, l, :]))
        out = torch.empty_like(src)
        P.fwd_dev(N, src, src, out, q, tw, pre, 3)
        assert (host(out).reshape(3, N) == got[:, l, :]).all(), l


ALIASES = ("disjoint", "c=a", "c=b", "a=b", "c=a=b")


def _operands(alias, a, b):
    import torch
    da = dev(a)
    if alias == "disjoint":
        return torch.empty_like(da), da, dev(b), a, b
    if alias == "c=a":
        return da, da, dev(b), a, b
    if alias == "c=b":
        db = dev(b)
        return db, da, db, a, b
    if alias == "a=b":
        return torch.empty_like(da), da, da, a, a
    return da, da, da, a, a


@gpu
@pytest.mark.parametrize("N", [4, 32, 64])
def test_polymul_vs_schoolbook(orc, ctx, N):
    c = ctx(N, MIXED)
    a, b = data(3, MIXED, N, 29 + N), data(3, MIXED, N, 31 + N)
    for l, q in enumerate(MIXED):
        a[0, l, 0] = b[0, l, N - 1] = q - 1
    d_c = dev(np.zeros_like(a))
    c.polymul(d_c, dev(a), dev(b))
    got = host(d_c).reshape(a.shape)
    for f in range(3):
        for l, q in enumerate(MIXED):
            want = np.empty(N, dtype=np.uint64)
            orc.orc_polymul_schoolbook_u64(N, q, _p(np.ascontiguousarray(a[f, l])), _p(np.ascontiguousarray(b[f, l])),
                                           _p(want))
            assert (got[f, l] == want).all()


@gpu
@pytest.mark.parametrize("alias", ALIASES)
@pytest.mark.parametrize("N", [4, 1024, 8192, 32768])
def test_polymul_aliasing_vs_oracle(orc, ctx, N, alias):
    c = ctx(N, MIXED)
    a, b = data(1, MIXED, N, 37 + N), data(1, MIXED, N, 41 + N)
    d_c, d_a, d_b, ha, hb = _operands(alias, a, b)
    c.polymul(d_c, d_a, d_b)
    assert (host(d_c).reshape(a.shape) == rns_polymul(orc, ha, hb, MIXED)).all()


@gpu
@pytest.mark.parametrize("alias", ("disjoint", "c=a", "c=b_hat", "a=b_hat", "c=a=b_hat"))
@pytest.mark.parametrize("N", [4, 1024, 8192, 32768])
def test_polymul_by_spectrum_equals_polymul(ctx, N, alias):
    import torch
    c = ctx(N, MIXED)
    a, b = data(2, MIXED, N, 43 + N), data(2, MIXED, N, 47 + N)
    d_a, d_b = dev(a), dev(b)
    b_hat = d_b.clone()
    c.fwd(b_hat)
    if alias in ("a=b_hat", "c=a=b_hat"):                                # a is the buffer holding b_hat
        a, d_a = host(b_hat), b_hat
    want = torch.empty_like(d_b)
    c.polymul(want, dev(a), d_b)
    d_c = {"disjoint": torch.empty_like(d_b), "c=a": d_a, "c=b_hat": b_hat, "a=b_hat": torch.empty_like(d_b),
           "c=a=b_hat": b_hat}[alias]
    c.polymul_by_spectrum(d_c, d_a, b_hat)
    assert torch.equal(d_c, want)


@gpu
@pytest.mark.parametrize("alias", ("disjoint", "c=a", "c=b", "a=b"))
@pytest.mark.parametrize("op", ("add", "sub", "mul", "mac"))
def test_elementwise_vs_bigint(ctx, op, alias):
    N = 32
    c = ctx(N, MIXED)
    a, b, c0 = data(2, MIXED, N, 53), data(2, MIXED, N, 59), data(2, MIXED, N, 61)
    for l, q in enumerate(MIXED):                                       # extreme operands
        a[0, l, :4] = [q - 1, q - 1, 0, 0]
        b[0, l, :4] = [q - 1, 0, q - 1, 0]
        c0[0, l, :4] = [q - 1, 0, q - 1, 0]
    if alias == "a=b":
        b = a
    da = dev(a)
    db = da if alias == "a=b" else dev(b)
    dc = {"disjoint": dev(c0), "c=a": da, "c=b": db, "a=b": dev(c0)}[alias]
    cv = {"disjoint": c0, "c=a": a, "c=b": b, "a=b": c0}[alias]
    want = np.empty_like(a)
    for f in range(2):
        for l, q in enumerate(MIXED):
            for i in range(N):
                x, y, z = int(a[f, l, i]), int(b[f, l, i]), int(cv[f, l, i])
                want[f, l, i] = {"add": x + y, "sub": x - y, "mul": x * y, "mac": z + x * y}[op] % q
    c.elementwise(op, dc, da, db)
    assert (host(dc).reshape(a.shape) == want).all()


@gpu
@pytest.mark.parametrize("N", [32, 1024, 16384, 32768])
def test_launch_counts(ctx, N):
    import torch
    c = ctx(N, MIXED)
    x = data(2, MIXED, N, 67)
    d_a, d_b, d_c = dev(x), dev(x[::-1].copy()), dev(np.zeros_like(x))
    split = 1 if N == 32768 else 0

    def launches(fn):
        l0 = c.launch_count()
        fn()
        torch.cuda.synchronize()
        return c.launch_count() - l0

    assert launches(lambda: c.fwd(d_c)) == 1
    assert launches(lambda: c.inv(d_c)) == 1 + split
    assert launches(lambda: c.polymul_by_spectrum(d_c, d_a, d_b)) == 2 + split
    assert launches(lambda: c.polymul(d_c, d_a, d_b)) == 3 + split
    assert launches(lambda: c.elementwise("mac", d_c, d_a, d_b)) == 1
    empty = d_a[:0]
    for fn in (lambda: c.fwd(empty), lambda: c.inv(empty), lambda: c.polymul(empty, empty, empty),
               lambda: c.polymul_by_spectrum(empty, empty, empty), lambda: c.elementwise("add", empty, empty, empty)):
        assert launches(fn) == 0


@gpu
def test_side_stream(orc, ctx):
    """Issued on a non-default stream right after torch work on that stream, synchronised on that stream only."""
    import torch
    N = 8192
    c = ctx(N, MIXED)
    a, b = data(2, MIXED, N, 71), data(2, MIXED, N, 73)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_a, d_b = dev(a), dev(b)                                       # the copies are ordered on s
        d_c = torch.empty_like(d_a)
        d_c.copy_(d_a)                                                  # torch work the product must follow
    c.polymul(d_c, d_c, d_b, stream=s)
    s.synchronize()
    assert (d_c.cpu().numpy().view(np.uint64).reshape(a.shape) == rns_polymul(orc, a, b, MIXED)).all()
