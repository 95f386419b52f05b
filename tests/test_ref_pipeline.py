"""The reference-shaped u64 forward pipeline (agx_ref_input / agx_ref_fwd / agx_ref_output / agx_wait), driven
with main.cpp's call sequence (src/main.cpp:60-74), against the C restatement of ntt.cpp and the golden outputs
recorded from the reference's own code.  Bit-exact, including wrap-around mod 2^64 on main.cpp's dummy data."""
import hashlib

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A():
    import agilex_ntt_b200 as pkg
    return pkg


def run_pipeline(A, in1, in2, modulus, tw, pre, frames, order=("input", "fwd", "output")):
    p = A.RefPipeline()
    out = np.zeros(len(tw) * frames, dtype=np.uint64)
    for step in order:
        if step == "input":
            p.ntt_input_kernel(in1, in2, np.array([modulus], dtype=np.uint64), tw, pre, frames)
        elif step == "fwd":
            p.fwd_ntt_kernel(0)
        else:
            p.ntt_output_kernel(out, frames)
    p.wait()
    n_launch = p.launch_count()
    p.close()
    return out, n_launch


def test_main_cpp_dummy_data(A, golden):
    """main.cpp:49-55: in[i]=i, in2[i]=i+1, twiddle[i]=i+2, precon[i]=i+3, modulus 65537, N=16384, 1 frame."""
    g, meta = golden
    N = 16384
    i = np.arange(N, dtype=np.uint64)
    out, launches = run_pipeline(A, i, i + 1, 65537, i + 2, i + 3, 1)
    assert launches == 1          # N = 16384: one launch, the frame resident in one CTA's shared memory
    assert (out == g["main_dummy_u64"]).all()
    assert hashlib.sha256(out.tobytes()).hexdigest() == meta["main_dummy_sha256_le64"][0]
    txt = "".join("%d\n" % int(v) for v in out)      # what main.cpp:82 prints
    assert hashlib.sha256(txt.encode()).hexdigest() == \
        "68db50a07a87d4e18387a721d88b42291198aba2f9e9138e2e52d45ad6537c5c"


@pytest.mark.parametrize("N", [32, 512, 1024, 2048, 4096, 8192, 16384, 32768])
def test_reference_sizes_vs_restatement(A, N):
    q = O.SEAL_PRIMES_30[1]
    tw, pre = O.tables_u64(N, q)
    frames = 3 if N <= 8192 else 2
    x = np.array([O.splitmix64(1000 + i) % (4 * q) for i in range(N * frames)], dtype=np.uint64)   # lazy [0,4q)
    x2 = np.array([O.splitmix64(5000 + i) % q for i in range(N * frames)], dtype=np.uint64)
    out, _ = run_pipeline(A, x, x2, q, tw, pre, frames)
    assert (out == O.ref_fwd_u64(x, x2, q, tw, pre, frames)).all()
    assert (out < q).all()


def test_golden_lazy_and_multiframe(A, golden):
    g, meta = golden
    for name in ("n1024_lazy", "n1024_sm_f4", "n32_sm_f3", "n8192_sm"):
        m = meta[name]
        N, q, psi, kind, frames, seed = int(m[0]), int(m[1]), int(m[2]), m[3], int(m[4]), int(m[5])
        mod = 4 * q if kind == "lazy4q" else q
        x = np.array([O.splitmix64(seed + i) % mod for i in range(N * frames)], dtype=np.uint64)
        tw, pre = O.tables_u64(N, q, psi)
        out, _ = run_pipeline(A, x, x, q, tw, pre, frames)
        assert (out == g[name]).all(), name


def test_golden_u64_large_primes(A, golden_u64):
    """50-, 60-, 62-bit NTT primes (the moduli the reference's 64-bit datapath exists for) and a 63-bit one whose lazy
    range wraps mod 2^64: lazy inputs, several frames, in2 != in, N = 1024 ... 32768, against the outputs of the
    reference's own code (stored for N <= 8192, SHA-256 for N >= 16384)."""
    g, cases = golden_u64
    for name, c in cases.items():
        mod = 4 * c["q"] if c["lazy"] else c["q"]
        n = c["N"] * c["frames"]
        x, x2 = O.synthetic_u64(n, c["seed_in"], mod), O.synthetic_u64(n, c["seed_in2"], mod)
        tw, pre = O.tables_u64(c["N"], c["q"], c["psi"])
        out, _ = run_pipeline(A, x, x2, c["q"], tw, pre, c["frames"])
        assert hashlib.sha256(out.tobytes()).hexdigest() == c["sha256"], name
        if name in g.files:
            assert (out == g[name]).all(), name


@pytest.mark.parametrize("bits", [50, 60, 63])
@pytest.mark.parametrize("N", [512, 2048, 16384, 32768])
def test_large_primes_vs_restatement(A, N, bits):
    """Sizes between the golden ones, against the C restatement (itself pinned on the same primes by the golden file)."""
    q = O.U64_PRIMES[bits]
    tw, pre = O.tables_u64(N, q)
    frames = 3
    mod = 4 * q if bits < 62 else q
    x, x2 = O.synthetic_u64(N * frames, 5 + bits, mod), O.synthetic_u64(N * frames, 6 + bits, mod)
    out, _ = run_pipeline(A, x, x2, q, tw, pre, frames)
    assert (out == O.ref_fwd_u64(x, x2, q, tw, pre, frames)).all()


def test_call_order_is_free_like_the_reference(A):
    """The reference's three kernels run concurrently and meet through pipes; submission order does not matter."""
    N, q = 1024, O.SEAL_PRIMES_30[0]
    tw, pre = O.tables_u64(N, q)
    x = np.arange(N, dtype=np.uint64)
    want = O.ref_fwd_u64(x, x, q, tw, pre, 1)
    for order in (("output", "input", "fwd"), ("fwd", "output", "input"), ("input", "output", "fwd")):
        out, _ = run_pipeline(A, x, x, q, tw, pre, 1, order)
        assert (out == want).all()


def test_protocol_errors(A):
    p = A.RefPipeline()
    N, q = 32, O.SEAL_PRIMES_30[0]
    tw, pre = O.tables_u64(N, q)
    x = np.arange(N, dtype=np.uint64)
    p.ntt_input_kernel(x, x, np.array([q], dtype=np.uint64), tw, pre, 1)
    with pytest.raises(A.AgxError):            # a second input before the round completed
        p.ntt_input_kernel(x, x, np.array([q], dtype=np.uint64), tw, pre, 1)
    with pytest.raises(A.AgxError):            # waiting on a round that can never complete
        p.wait()
    with pytest.raises(A.AgxError):            # only compute unit 0 exists (ntt.cpp:648)
        p.fwd_ntt_kernel(1)
    # frame-count mismatch between loader and drain
    out = np.zeros(N * 2, dtype=np.uint64)
    p.ntt_input_kernel(x, x, np.array([q], dtype=np.uint64), tw, pre, 1)
    p.fwd_ntt_kernel(0)
    with pytest.raises(A.AgxError):
        p.ntt_output_kernel(out, 2)
    p.close()


def _run_driver(name, *args):
    import os
    import subprocess
    import agilex_ntt_b200 as pkg
    exe = os.path.join(os.path.dirname(pkg.build.LIB), "..", "bin", name)
    if not os.path.exists(exe):
        pytest.skip(f"{name} not built (agx_ref_main needs the reference tree at build time)")
    r = subprocess.run([exe, *args], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-500:]
    return [l for l in r.stdout.splitlines() if l.strip().isdigit()]


def test_reference_main_cpp_unmodified_runs_on_the_gpu():
    """The reference's own src/main.cpp, compiled unmodified against agilex-ntt_b200/host/, prints the known answer."""
    lines = _run_driver("agx_ref_main")
    assert len(lines) == 16384
    txt = "".join(l + "\n" for l in lines)
    assert hashlib.sha256(txt.encode()).hexdigest() == "68db50a07a87d4e18387a721d88b42291198aba2f9e9138e2e52d45ad6537c5c"


def test_compat_driver_real_ntt_instance():
    """Our main.cpp-shaped driver on a real instance: q = 1053818881, N = 1024, ramp input, 2 frames."""
    N, q, frames = 1024, O.SEAL_PRIMES_30[0], 2
    lines = _run_driver("agx_main_compat", "--seal", str(N), str(frames))
    got = np.array([int(l) for l in lines], dtype=np.uint64)
    tw, pre = O.tables_u64(N, q)
    x = np.arange(N * frames, dtype=np.uint64) % np.uint64(q)
    assert (got == O.ref_fwd_u64(x, x, q, tw, pre, frames)).all()
    dummy = _run_driver("agx_main_compat")          # main.cpp's dummy data by default
    assert len(dummy) == 16384 and int(dummy[0]) == 15752083817248508221
    # what the reference's main.cpp prints for the same data (the known answer of the unmodified-main.cpp test above)
    assert hashlib.sha256("".join(l + "\n" for l in dummy).encode()).hexdigest() == \
        "68db50a07a87d4e18387a721d88b42291198aba2f9e9138e2e52d45ad6537c5c"


def test_c_abi_from_plain_c():
    """host/c_example.c (C99, no CUDA headers): round trip and X^(n-1) * X = -1 through the host-pointer entry points."""
    import os
    import subprocess
    import agilex_ntt_b200 as pkg
    exe = os.path.join(os.path.dirname(pkg.build.LIB), "..", "bin", "agx_c_example")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "c_example ok" in r.stdout, r.stderr[-500:]


def _pinned_u64(a: np.ndarray) -> np.ndarray:
    import torch
    t = torch.empty(a.size, dtype=torch.int64).pin_memory()
    v = t.numpy().view(np.uint64)
    v[:] = a
    v_holder.append(t)             # keep the page-locked allocation alive for the duration of the test
    return v


v_holder = []


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("same", [True, False])
def test_chunked_pipeline_many_frames(A, pinned, same, monkeypatch):
    """More frames than one pipeline chunk holds (3 slots; chunk pinned to 16 MiB here, the library's own choice is whole
    waves of frame CTAs): H2D / kernel / D2H overlap across slots; the high halves come from in2 (ntt.cpp:582-591), by
    pitched copies when the caller's buffers are page-locked."""
    monkeypatch.setenv("AGX_REF_CHUNK_KB", "16384")
    N, q = 8192, O.SEAL_PRIMES_30[2]
    frames = 4 * (16 << 20) // (N * 8) + 5          # 4 full chunks and a ragged one
    tw, pre = O.tables_u64(N, q)
    rng = np.random.default_rng(7)
    x = rng.integers(0, 4 * q, size=N * frames, dtype=np.uint64)
    x2 = x if same else rng.integers(0, q, size=N * frames, dtype=np.uint64)
    want = O.ref_fwd_u64(x, x2, q, tw, pre, frames)
    if pinned:
        px = _pinned_u64(x)
        px2 = px if same else _pinned_u64(x2)
        p = A.RefPipeline()
        out = _pinned_u64(np.zeros(N * frames, dtype=np.uint64))
        p.ntt_input_kernel(px, px2, np.array([q], dtype=np.uint64), tw, pre, frames)
        p.fwd_ntt_kernel(0)
        p.ntt_output_kernel(out, frames)
        p.wait()
        assert p.launch_count() == 5              # 5 chunks, one launch each
        p.close()
    else:
        out, launches = run_pipeline(A, x, x2, q, tw, pre, frames)
        assert launches == 5
    assert (out == want).all()
    v_holder.clear()


def test_default_chunks_are_whole_waves(A):
    """The pipeline's own chunking: SMs x 128 KiB of frames per chunk (one wave of frame CTAs), ragged last chunk, results
    as the restatement's."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N, q = 16384, O.U64_PRIMES[60]
    frames = 2 * sms + 9
    tw, pre = O.tables_u64(N, q)
    rng = np.random.default_rng(11)
    x = rng.integers(0, 4 * q, size=N * frames, dtype=np.uint64)
    out, launches = run_pipeline(A, x, x, q, tw, pre, frames)
    assert launches == 3
    assert (out == O.batch_ref_fwd_u64(N, x.copy(), q, tw, pre, threads=O.max_threads())).all()


@pytest.mark.parametrize("N,bits", [(1024, 60), (8192, 50), (16384, 60), (32768, 50), (64, 60)])
def test_device_pointer_entry_point(A, N, bits):
    """agx_ref_fwd_dev: the same transform on device buffers (what the pipeline runs per chunk), in2 != in, separate
    output and fully in place, against the restatement."""
    import torch
    q = O.U64_PRIMES[bits]
    tw, pre = O.tables_u64(N, q)
    frames = 5
    x, x2 = O.synthetic_u64(N * frames, 3, 4 * q), O.synthetic_u64(N * frames, 4, 4 * q)
    want = O.ref_fwd_u64(x, x2, q, tw, pre, frames)
    dev = lambda a: torch.from_numpy(a.view(np.int64)).cuda()
    d_in, d_in2, d_tw, d_pre = dev(x), dev(x2), dev(tw), dev(pre)
    d_out = torch.zeros_like(d_in)
    p = A.RefPipeline()
    p.fwd_dev(N, d_in, d_in2, d_out, q, d_tw, d_pre, frames)
    torch.cuda.synchronize()
    assert (d_out.cpu().numpy().view(np.uint64) == want).all()
    assert (d_in.cpu().numpy().view(np.uint64) == x).all()            # inputs untouched
    same = O.ref_fwd_u64(x, x, q, tw, pre, frames)
    p.fwd_dev(N, d_in, d_in, d_in, q, d_tw, d_pre, frames)            # in place
    torch.cuda.synchronize()
    assert (d_in.cpu().numpy().view(np.uint64) == same).all()
    with pytest.raises(A.AgxError):                                   # output overlapping only one of the inputs
        p.fwd_dev(N, d_in, d_in2, d_in, q, d_tw, d_pre, frames)
    with pytest.raises(A.AgxError):
        p.fwd_dev(N + 1, d_in, d_in2, d_out, q, d_tw, d_pre, frames)
    # frames and tables are read by 16-byte accesses: a pointer that is only 8-byte aligned is refused, not faulted on
    pad = torch.zeros(N + 1, dtype=torch.int64, device="cuda")
    pad[1:] = d_tw
    with pytest.raises(A.AgxError):
        p.fwd_dev(N, d_in, d_in2, d_out, q, pad[1:], d_pre, frames)
    with pytest.raises(A.AgxError):
        p.fwd_dev(N, d_in, d_in2, d_out, q, d_tw, pad[1:], frames)
    p.fwd_dev(N, d_in, d_in2, d_out, q, d_tw, d_pre, frames)          # the context still works after the refusals
    torch.cuda.synchronize()
    p.close()


def test_device_pointer_entry_point_large_batch_two_ctas_per_frame(A):
    """N = 16384 with at least two waves of frames and a separate output runs two CTAs per frame (each an 8192-point half
    after its own copy of stage 0, as N = 32768 always does); in place it must keep one CTA per frame.  Both against the
    restatement, lazy inputs, in2 != in."""
    import torch
    N, q = 16384, O.U64_PRIMES[60]
    tw, pre = O.tables_u64(N, q)
    frames = 2 * torch.cuda.get_device_properties(0).multi_processor_count + 5
    x, x2 = O.synthetic_u64(N * frames, 5, 4 * q), O.synthetic_u64(N * frames, 6, 4 * q)
    want = O.batch_ref_fwd_u64(N, np.concatenate([a for f in range(frames) for a in
                                                   (x[f * N: f * N + N // 2], x2[f * N + N // 2: (f + 1) * N])]),
                               q, tw, pre, threads=O.max_threads())
    dev = lambda a: torch.from_numpy(a.view(np.int64)).cuda()
    d_in, d_in2, d_tw, d_pre = dev(x), dev(x2), dev(tw), dev(pre)
    d_out = torch.zeros_like(d_in)
    p = A.RefPipeline()
    p.fwd_dev(N, d_in, d_in2, d_out, q, d_tw, d_pre, frames)
    torch.cuda.synchronize()
    assert (d_out.cpu().numpy().view(np.uint64) == want).all()
    assert (d_in.cpu().numpy().view(np.uint64) == x).all() and (d_in2.cpu().numpy().view(np.uint64) == x2).all()
    same = O.batch_ref_fwd_u64(N, x.copy(), q, tw, pre, threads=O.max_threads())
    p.fwd_dev(N, d_in, d_in, d_in, q, d_tw, d_pre, frames)            # in place: one CTA per frame
    torch.cuda.synchronize()
    assert (d_in.cpu().numpy().view(np.uint64) == same).all()
    p.close()


def test_buffer_size_contract_is_checked(A):
    """ADVICE r1: agx_ref_* take bare pointers, so the mirrors of ntt_input_kernel / ntt_output_kernel check that the
    buffers describe numFrames x N (main.cpp:26-37) before anything is handed to the DMA engines."""
    N, q = 64, O.SEAL_PRIMES_30[0]
    tw, pre = O.tables_u64(N, q)
    x = np.arange(N * 2, dtype=np.uint64)
    mod = np.array([q], dtype=np.uint64)
    p = A.RefPipeline()
    with pytest.raises(ValueError):
        p.ntt_input_kernel(x, x, mod, tw, pre, 3)                     # inputs hold 2 frames, 3 requested
    with pytest.raises(ValueError):
        p.ntt_input_kernel(x, x, mod, tw, pre[:-1], 2)
    p.ntt_input_kernel(x, x, mod, tw, pre, 2)
    p.fwd_ntt_kernel(0)
    with pytest.raises(ValueError):
        p.ntt_output_kernel(np.zeros(N * 2 - 1, dtype=np.uint64), 2)  # too small for 2 frames
    out = np.zeros(N * 2, dtype=np.uint64)
    p.ntt_output_kernel(out, 2)
    p.wait()
    assert (out == O.ref_fwd_u64(x, x, q, tw, pre, 2)).all()
    p.close()
