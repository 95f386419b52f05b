"""The u64 inverse transform and negacyclic product on device pointers (agx_ref_inv_dev, agx_ref_polymul_dev,
agx_ref_polymul_by_spectrum_dev) on 50-, 60- and 62-bit NTT primes.

The CPU oracle of these operations (tests/native/u64_inverse_oracle.c) is built into a temporary directory and pinned
here against the big-int definitions of oracle/oracle.py (the non-GPU tests); the GPU tests compare the library with it
bit for bit."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
BITS = (50, 60, 62)
SIZES = (4, 32, 512, 1024, 2048, 4096, 8192, 16384, 32768)
_u64p = C.POINTER(C.c_uint64)


@pytest.fixture(scope="module")
def orc(tmp_path_factory):
    src = os.path.join(ROOT, "tests", "native", "u64_inverse_oracle.c")
    so = str(tmp_path_factory.mktemp("u64_oracle") / "libu64oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc") or "cc"
    base = [cc, "-O2", "-std=c11", "-fPIC", "-shared", "-o", so, src]
    if subprocess.run(base + ["-fopenmp"], capture_output=True).returncode != 0:
        subprocess.run(base + ["-Wno-unknown-pragmas"], check=True)       # single-threaded oracle without OpenMP
    L = C.CDLL(so)
    L.orc_inv_u64.argtypes = [C.c_uint32, _u64p, C.c_uint64, _u64p, C.c_size_t, C.c_int]
    L.orc_polymul_schoolbook_u64.argtypes = [C.c_uint32, C.c_uint64, _u64p, _u64p, _u64p]
    return L


def _p(a):
    assert a.dtype == np.uint64 and a.flags.c_contiguous
    return a.ctypes.data_as(_u64p)


def inv_u64(orc, X, q, iroots):
    """Oracle inverse of every N-word frame of X (bit-reversed in, natural out, [0,q)); returns a new array."""
    N = len(iroots)
    y = np.ascontiguousarray(X, dtype=np.uint64).copy()
    orc.orc_inv_u64(N, _p(y), q, _p(np.ascontiguousarray(iroots, dtype=np.uint64)), y.size // N,
                    max(1, min(O.max_threads(), 16)))
    return y


def schoolbook_u64(orc, a, b, q, N):
    a, b = np.ascontiguousarray(a, dtype=np.uint64), np.ascontiguousarray(b, dtype=np.uint64)
    c = np.empty_like(a)
    for f in range(a.size // N):
        s = slice(f * N, (f + 1) * N)
        orc.orc_polymul_schoolbook_u64(N, q, _p(a[s]), _p(b[s]), _p(c[s]))
    return c


def fwd_u64(X, q, tw, pre):
    N = len(tw)
    return O.ref_fwd_u64(X, X, q, tw, pre, X.size // N)


def pointwise(x, y, q):
    return np.array([int(u) * int(v) % q for u, v in zip(x, y)], dtype=np.uint64)


def product_oracle(orc, a, b, q, tabs):
    """INTT(NTT(a) .* NTT(b)) through the oracle: forward of the C restatement, exact pointwise product, oracle inverse."""
    tw, pre, itw, _ = tabs
    return inv_u64(orc, pointwise(fwd_u64(a, q, tw, pre), fwd_u64(b, q, tw, pre), q), q, itw)


_TABLES = {}


def tables(N, q, psi=None):
    key = (N, q, psi)
    if key not in _TABLES:
        _TABLES[key] = O.tables_u64(N, q, psi) + O.tables_u64(N, q, psi, inverse=True)
    return _TABLES[key]


# ------------------------------------------------------------------------------------------ the oracle, on the CPU

@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("N", [8, 32, 64])
def test_oracle_inverse_is_the_definition(orc, N, bits):
    q = O.U64_PRIMES[bits]
    X = O.synthetic_u64(N, 11 + bits, 2 * q)                             # lazy [0,2q), as the library accepts
    want = O.textbook_inv(X, q, O.min_psi(N, q))
    assert (inv_u64(orc, X, q, tables(N, q)[2]) == want).all()


@pytest.mark.parametrize("N", [1 << k for k in range(2, 16)])
def test_oracle_inverse_undoes_the_forward(orc, N):
    for bits in BITS:
        q = O.U64_PRIMES[bits]
        tw, pre, itw, _ = tables(N, q)
        x = O.synthetic_u64(2 * N, N + bits, 4 * q)                      # the forward's lazy input range [0,4q)
        assert (inv_u64(orc, fwd_u64(x, q, tw, pre), q, itw) == x % np.uint64(q)).all()


@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("N", [32, 64])
def test_oracle_schoolbook_is_the_definition(orc, N, bits):
    q = O.U64_PRIMES[bits]
    a, b = O.synthetic_u64(N, 1 + bits, q), O.synthetic_u64(N, 2 + bits, q)
    a[0] = b[N - 1] = q - 1                                              # (q-1)^2 terms
    assert (schoolbook_u64(orc, a, b, q, N) == O.textbook_polymul(a, b, q)).all()


# --------------------------------------------------------------------------------------------- the library, on a GPU

@pytest.fixture(scope="module")
def P():
    import agilex_ntt_b200 as A
    p = A.RefPipeline()
    yield p
    p.close()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(np.uint64)


def dev_tables(N, q, psi=None):
    return [dev(t) for t in tables(N, q, psi)]


@gpu
@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("N", SIZES)
def test_inverse_vs_oracle(orc, P, N, bits):
    """5 frames of lazy [0,2q) spectra: out of place (the input left untouched) and in place."""
    q = O.U64_PRIMES[bits]
    X = O.synthetic_u64(5 * N, 3 * N + bits, 2 * q)
    want = inv_u64(orc, X, q, tables(N, q)[2])
    _, _, d_itw, d_ipre = dev_tables(N, q)
    d_in = dev(X)
    d_out = dev(np.zeros_like(X))
    P.inv_dev(N, d_in, d_out, q, d_itw, d_ipre, 5)
    assert (host(d_out) == want).all()
    assert (host(d_in) == X).all()
    P.inv_dev(N, d_in, d_in, q, d_itw, d_ipre, 5)
    assert (host(d_in) == want).all()


@gpu
@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("N", SIZES)
def test_round_trip(P, N, bits):
    """inv_dev(fwd_dev(x)) == x mod q, from the forward's lazy [0,4q) inputs."""
    q = O.U64_PRIMES[bits]
    x = O.synthetic_u64(3 * N, 5 * N + bits, 4 * q)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    d_x = dev(x)
    d_y = dev(np.zeros_like(x))
    P.fwd_dev(N, d_x, d_x, d_y, q, d_tw, d_pre, 3)
    P.inv_dev(N, d_y, d_y, q, d_itw, d_ipre, 3)
    assert (host(d_y) == x % np.uint64(q)).all()


@gpu
@pytest.mark.parametrize("N", [32, 1024, 16384, 32768])
def test_round_trip_non_minimal_root(orc, P, N):
    """Tables of another primitive 2N-th root: the inverse depends only on the caller's tables."""
    q = O.U64_PRIMES[60]
    psi = O.primitive_roots_2n(N, q, 1)[0]
    x = O.synthetic_u64(2 * N, 7 * N, q)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q, psi)
    d_x = dev(x)
    d_y = dev(np.zeros_like(x))
    P.fwd_dev(N, d_x, d_x, d_y, q, d_tw, d_pre, 2)
    spectrum = host(d_y)
    P.inv_dev(N, d_y, d_y, q, d_itw, d_ipre, 2)
    assert (host(d_y) == x).all()
    assert (inv_u64(orc, spectrum, q, tables(N, q, psi)[2]) == x).all()


@gpu
@pytest.mark.parametrize("N", [16384, 32768])
def test_large_batch_vs_oracle(orc, P, N):
    """More than two waves of CTAs (2 x SMs + 3 frames), lazy inputs, against the oracle."""
    import torch
    frames = 2 * torch.cuda.get_device_properties(0).multi_processor_count + 3
    q = O.U64_PRIMES[62]
    X = O.synthetic_u64(frames * N, 9 * N, 2 * q)
    _, _, d_itw, d_ipre = dev_tables(N, q)
    d_in = dev(X)
    d_out = torch.empty_like(d_in)
    P.inv_dev(N, d_in, d_out, q, d_itw, d_ipre, frames)
    assert (host(d_out) == inv_u64(orc, X, q, tables(N, q)[2])).all()


ALIASES = ("disjoint", "c=a", "c=b", "a=b", "c=a=b")


def _operands(alias, a, b):
    """Device buffers (c, a, b) for one aliasing case, and the host operands the product is of."""
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
@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("N", [4, 32, 256, 1024])
def test_polymul_vs_schoolbook(orc, P, N, bits):
    q = O.U64_PRIMES[bits]
    a, b = O.synthetic_u64(3 * N, 13 + N, q), O.synthetic_u64(3 * N, 17 + N, q)
    a[0] = b[1] = q - 1
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    d_a, d_b = dev(a), dev(b)
    d_c = dev(np.zeros_like(a))
    P.polymul_dev(N, d_c, d_a, d_b, q, d_tw, d_pre, d_itw, d_ipre, 3)
    assert (host(d_c) == schoolbook_u64(orc, a, b, q, N)).all()
    assert (host(d_a) == a).all() and (host(d_b) == b).all()


@gpu
@pytest.mark.parametrize("alias", ALIASES)
@pytest.mark.parametrize("N", SIZES)
def test_polymul_aliasing_vs_oracle(orc, P, N, alias):
    q = O.U64_PRIMES[BITS[N.bit_length() % 3]]
    a, b = O.synthetic_u64(3 * N, 21 + N, q), O.synthetic_u64(3 * N, 23 + N, q)
    d_c, d_a, d_b, ha, hb = _operands(alias, a, b)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    P.polymul_dev(N, d_c, d_a, d_b, q, d_tw, d_pre, d_itw, d_ipre, 3)
    assert (host(d_c) == product_oracle(orc, ha, hb, q, tables(N, q))).all()


@gpu
@pytest.mark.parametrize("alias", ("disjoint", "c=a", "c=b_hat", "a=b_hat", "c=a=b_hat"))
@pytest.mark.parametrize("N", SIZES)
def test_polymul_by_spectrum_equals_polymul(P, N, alias):
    import torch
    q = O.U64_PRIMES[BITS[N.bit_length() % 3]]
    a, b = O.synthetic_u64(3 * N, 31 + N, q), O.synthetic_u64(3 * N, 37 + N, q)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    d_a, d_b = dev(a), dev(b)
    b_hat = torch.empty_like(d_b)
    P.fwd_dev(N, d_b, d_b, b_hat, q, d_tw, d_pre, 3)
    if alias in ("a=b_hat", "c=a=b_hat"):                                # a is the buffer holding b_hat (reduced words)
        a, d_a = host(b_hat), b_hat
    want_c = torch.empty_like(d_b)
    P.polymul_dev(N, want_c, dev(a), d_b, q, d_tw, d_pre, d_itw, d_ipre, 3)
    want = host(want_c)
    d_c = {"disjoint": torch.empty_like(d_b), "c=a": d_a, "c=b_hat": b_hat, "a=b_hat": torch.empty_like(d_b),
           "c=a=b_hat": b_hat}[alias]
    P.polymul_by_spectrum_dev(N, d_c, d_a, b_hat, q, d_tw, d_pre, d_itw, d_ipre, 3)
    assert (host(d_c) == want).all()


@gpu
def test_refusals_leave_the_context_usable(P):
    import agilex_ntt_b200 as A
    N, q = 1024, O.U64_PRIMES[60]
    x = O.synthetic_u64(N, 1, q)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    d_a, d_b, d_c = dev(x), dev(x), dev(np.zeros_like(x))
    calls = {
        "inv": lambda n, mod, p: P.inv_dev(n, p, d_c, mod, d_itw, d_ipre, 1),
        "polymul": lambda n, mod, p: P.polymul_dev(n, d_c, p, d_b, mod, d_tw, d_pre, d_itw, d_ipre, 1),
        "by_spectrum": lambda n, mod, p: P.polymul_by_spectrum_dev(n, d_c, p, d_b, mod, d_tw, d_pre, d_itw, d_ipre, 1),
    }
    bad = [(N, q + 1, d_a),                          # even modulus
           (N, O.U64_PRIMES[63], d_a),               # q >= 2^62
           (N, 1, d_a),                              # no Barrett constants for q = 1
           (3 * 256, q, d_a), (2, q, d_a), (65536, q, d_a), (0, q, d_a),
           (N, q, d_a.data_ptr() + 8),               # 8-byte aligned
           (N, q, 0)]                                # null
    for name, call in calls.items():
        for n, mod, ptr in bad:
            with pytest.raises(A.AgxError) as e:
                call(n, mod, ptr)
            assert e.value.code == -1, (name, n, mod)
    P.inv_dev(N, d_a, d_c, q, d_itw, d_ipre, 1)
    P.fwd_dev(N, d_c, d_c, d_b, q, d_tw, d_pre, 1)
    assert (host(d_b) == x).all()                    # fwd(inv(x)) == x: the context still computes


@gpu
@pytest.mark.parametrize("N", [32, 1024, 16384, 32768])
def test_launch_counts(P, N):
    import torch
    q = O.U64_PRIMES[50]
    x = O.synthetic_u64(2 * N, 5, q)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    d_a, d_b, d_c = dev(x), dev(x[::-1].copy()), dev(np.zeros_like(x))
    split = 1 if N == 32768 else 0

    def launches(fn):
        l0 = P.launch_count()
        fn()
        torch.cuda.synchronize()
        return P.launch_count() - l0

    assert launches(lambda: P.inv_dev(N, d_a, d_c, q, d_itw, d_ipre, 2)) == 1 + split
    assert launches(lambda: P.polymul_by_spectrum_dev(N, d_c, d_a, d_b, q, d_tw, d_pre, d_itw, d_ipre, 2)) == 2 + split
    assert launches(lambda: P.polymul_dev(N, d_c, d_a, d_b, q, d_tw, d_pre, d_itw, d_ipre, 2)) == 3 + split
    assert launches(lambda: P.inv_dev(N, d_a, d_c, q, d_itw, d_ipre, 0)) == 0          # empty batch
    assert launches(lambda: P.polymul_dev(N, d_c, d_a, d_b, q, d_tw, d_pre, d_itw, d_ipre, 0)) == 0


@gpu
def test_side_stream(orc, P):
    """Issued on a non-default stream (the scratch buffer of the product is ordered on it), synchronised on that stream."""
    import torch
    N, q = 8192, O.U64_PRIMES[62]
    a, b = O.synthetic_u64(4 * N, 41, q), O.synthetic_u64(4 * N, 43, q)
    d_tw, d_pre, d_itw, d_ipre = dev_tables(N, q)
    d_a, d_b = dev(a), dev(b)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_c = torch.empty_like(d_a)
        d_x = torch.empty_like(d_a)
    P.polymul_dev(N, d_c, d_a, d_b, q, d_tw, d_pre, d_itw, d_ipre, 4, stream=s)
    P.inv_dev(N, d_c, d_x, q, d_itw, d_ipre, 4, stream=s)
    s.synchronize()
    c = d_c.cpu().numpy().view(np.uint64)
    assert (c == product_oracle(orc, a, b, q, tables(N, q))).all()
    assert (d_x.cpu().numpy().view(np.uint64) == inv_u64(orc, c, q, tables(N, q)[2])).all()
