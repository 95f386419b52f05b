"""ctypes binding of include/agxntt.h -- the Python host side over the C ABI.

The CUDA library is REQUIRED: importing this module without lib/libagxntt.so raises, and every call goes to the
GPU kernels.  There is no CPU fallback anywhere in this package (oracle/ is test infrastructure and is never
imported from here).
"""
from __future__ import annotations

import ctypes as C
import numbers
import os

import numpy as np

from . import build as _build

_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


class AgxError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"{what}: {error_string(code)} (code {code})")
        self.code = code


class _Parms(C.Structure):
    _fields_ = [("n", C.c_uint32), ("logn", C.c_uint32), ("nlimbs", C.c_uint32), ("q", _u32p)]


class _Parms64(C.Structure):
    _fields_ = [("n", C.c_uint32), ("logn", C.c_uint32), ("nlimbs", C.c_uint32), ("q", _u64p)]


def _load() -> C.CDLL:
    path = os.environ.get("AGX_LIB", _build.LIB)   # AGX_LIB: experiment builds of the same ABI (kernel variants)
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the CUDA extension is mandatory; there is no CPU fallback)")
    if "AGX_LIB" not in os.environ and _build.recorded_hash() not in (None, _build.source_hash()):
        import warnings
        warnings.warn(f"{path} was built from other sources than the ones in csrc/: rebuild with "
                      "`python -c 'import __graft_entry__ as g; g.build()'`", RuntimeWarning, stacklevel=3)
    L = C.CDLL(path)
    vp = C.c_void_p
    sigs = {
        "agx_create": [C.POINTER(vp), C.POINTER(_Parms), C.c_int],
        "agx_create_tables": [C.POINTER(vp), C.POINTER(_Parms), _u32p, C.c_int],
        "agx_set_tables": [vp, C.c_uint32, C.c_int, _u32p, _u32p],
        "agx_destroy": [vp],
        "agx_get_psi": [vp, C.c_uint32, _u32p],
        "agx_get_tables": [vp, C.c_uint32, C.c_int, _u32p, _u32p],
        "agx_ntt_fwd": [vp, vp, C.c_size_t, vp],
        "agx_ntt_inv": [vp, vp, C.c_size_t, vp],
        "agx_polymul": [vp, vp, vp, vp, C.c_size_t, vp],
        "agx_polymul_by_spectrum": [vp, vp, vp, vp, C.c_size_t, vp],
        "agx_elementwise": [vp, C.c_int, vp, vp, vp, C.c_size_t, vp],
        "agx_bitrev": [vp, vp, C.c_size_t, vp],
        "agx_ntt_fwd_host": [vp, vp, vp, C.c_size_t],
        "agx_ntt_inv_host": [vp, vp, vp, C.c_size_t],
        "agx_polymul_host": [vp, vp, vp, vp, C.c_size_t],
        "agx_polymul_by_spectrum_host": [vp, vp, vp, vp, C.c_size_t],
        "agx_host_alloc": [C.POINTER(vp), C.c_size_t],
        "agx_host_free": [vp],
        "agx_fill_synthetic": [vp, vp, C.c_size_t, C.c_uint64, C.c_size_t, vp],
        "agx_checksum": [vp, vp, C.c_size_t, C.c_size_t, _u64p, vp],
        "agx_ref_input": [vp, C.c_uint32, _u64p, _u64p, _u64p, _u64p, _u64p, C.c_uint32],
        "agx_ref_fwd": [vp, C.c_uint32],
        "agx_ref_output": [vp, _u64p, C.c_int32],
        "agx_wait": [vp],
        "agx_ref_fwd_dev": [vp, C.c_uint32, vp, vp, vp, C.c_uint64, vp, vp, C.c_uint32, vp],
        "agx_ref_inv_dev": [vp, C.c_uint32, vp, vp, C.c_uint64, vp, vp, C.c_uint32, vp],
        "agx_ref_polymul_dev": [vp, C.c_uint32, vp, vp, vp, C.c_uint64, vp, vp, vp, vp, C.c_uint32, vp],
        "agx_ref_polymul_by_spectrum_dev": [vp, C.c_uint32, vp, vp, vp, C.c_uint64, vp, vp, vp, vp, C.c_uint32, vp],
        "agx_create64": [C.POINTER(vp), C.POINTER(_Parms64), _u64p, C.c_int],
        "agx_get_psi64": [vp, C.c_uint32, _u64p],
        "agx_get_tables64": [vp, C.c_uint32, C.c_int, _u64p, _u64p],
        "agx_ntt64_fwd": [vp, vp, C.c_size_t, vp],
        "agx_ntt64_inv": [vp, vp, C.c_size_t, vp],
        "agx_polymul64": [vp, vp, vp, vp, C.c_size_t, vp],
        "agx_polymul64_by_spectrum": [vp, vp, vp, vp, C.c_size_t, vp],
        "agx_elementwise64": [vp, C.c_int, vp, vp, vp, C.c_size_t, vp],
        "agx_rescale64": [vp, vp, vp, C.c_size_t, C.c_int, vp],
        "agx_moddown64": [vp, vp, vp, C.c_size_t, C.c_uint32, C.c_int, vp],
        "agx_modup64": [vp, vp, vp, C.c_size_t, C.c_uint32, C.c_uint32, C.c_int, vp],
        "agx_automorph64": [vp, vp, vp, C.c_size_t, _u32p, C.c_uint32, C.c_int, vp],
        "agx_keyswitch64": [vp, vp, vp, C.c_size_t, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, vp],
        "agx_rotate64": [vp, vp, vp, C.c_size_t, _u32p, C.c_uint32, C.POINTER(vp), C.c_uint32, C.c_uint32, C.c_uint32,
                         C.c_int, vp],
        "agx_lintrans64": [vp, vp, vp, C.c_size_t, _u32p, C.c_uint32, C.POINTER(vp), C.c_uint32, C.POINTER(vp),
                           C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, vp],
        "agx_mulrelin64": [vp, vp, vp, vp, C.c_size_t, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_int, vp],
        "agx_encode64": [vp, vp, vp, C.c_size_t, C.c_double, C.c_uint32, C.c_int, vp],
        "agx_decode64": [vp, vp, vp, C.c_size_t, C.c_double, C.c_uint32, C.c_int, vp],
        "agx_measure_butterfly_peak": [vp, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)],
        "agx_launch_count": [vp, _u64p],
        "agx_variant": [vp, C.c_char_p, C.c_size_t],
    }
    for name, args in sigs.items():
        fn = getattr(L, name)          # AttributeError here = header/library mismatch: fail loudly
        fn.argtypes = args
        fn.restype = C.c_int
    L.agx_error_string.argtypes = [C.c_int]
    L.agx_error_string.restype = C.c_char_p
    return L


EXPORTS = ("agx_create agx_create_tables agx_set_tables agx_ref_fwd_dev agx_ref_inv_dev agx_ref_polymul_dev "
           "agx_ref_polymul_by_spectrum_dev agx_measure_butterfly_peak agx_destroy agx_get_psi agx_get_tables agx_ntt_fwd agx_ntt_inv agx_polymul agx_polymul_by_spectrum agx_polymul_by_spectrum_host agx_elementwise agx_bitrev "
           "agx_ntt_fwd_host agx_ntt_inv_host agx_polymul_host agx_host_alloc agx_host_free agx_fill_synthetic "
           "agx_checksum agx_ref_input agx_ref_fwd agx_ref_output agx_wait agx_error_string agx_launch_count "
           "agx_variant agx_create64 agx_get_psi64 agx_get_tables64 agx_ntt64_fwd agx_ntt64_inv agx_polymul64 "
           "agx_polymul64_by_spectrum agx_elementwise64 agx_rescale64 agx_moddown64 agx_modup64 "
           "agx_automorph64 agx_keyswitch64 agx_rotate64 agx_lintrans64 agx_mulrelin64 agx_encode64 agx_decode64").split()

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


def error_string(code: int) -> str:
    return lib().agx_error_string(code).decode()


def _ck(code: int, what: str) -> None:
    if code != 0:
        raise AgxError(code, what)


def _dev_ptr(t) -> int:
    """Device pointer of a torch CUDA tensor (any 4-byte integer dtype) or a raw int address."""
    if isinstance(t, int):
        return t
    if not t.is_cuda or not t.is_contiguous() or t.element_size() != 4:
        raise ValueError("need a contiguous CUDA tensor of a 4-byte integer dtype")
    return t.data_ptr()


def _dev_ptr8(t) -> int:
    """Device pointer of a torch CUDA tensor of an 8-byte integer dtype (int64, uint64) or a raw int address."""
    if isinstance(t, int):
        return t
    if not t.is_cuda or not t.is_contiguous() or t.element_size() != 8 or t.is_floating_point() or t.is_complex():
        raise ValueError("need a contiguous CUDA tensor of an 8-byte integer dtype")
    return t.data_ptr()


def _complex128():
    import torch
    return torch.complex128


def _stream_ptr(stream) -> int:
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    return stream if isinstance(stream, int) else stream.cuda_stream


class Context:
    """One (n, primes) parameter set bound to one GPU: owns the device twiddle tables and the host pipeline."""

    def __init__(self, n: int, primes, device: int = 0, psi=None):
        """psi: the caller's primitive 2n-th root per limb (agx_create_tables); None = the minimal root (agx_create)."""
        self._h = C.c_void_p()
        self.n = int(n)
        self.logn = self.n.bit_length() - 1
        self.primes = [int(q) for q in primes]
        self.L = len(self.primes)
        self.device = device
        self._q = (C.c_uint32 * self.L)(*self.primes)
        p = _Parms(self.n, self.logn, self.L, C.cast(self._q, _u32p))
        if psi is None:
            _ck(lib().agx_create(C.byref(self._h), C.byref(p), device), "agx_create")
        else:
            psi = [int(v) for v in psi]
            if len(psi) != self.L:
                raise ValueError("need one psi per limb")
            arr = (C.c_uint32 * self.L)(*psi)
            _ck(lib().agx_create_tables(C.byref(self._h), C.byref(p), C.cast(arr, _u32p), device), "agx_create_tables")

    def set_tables(self, limb: int, roots, precons=None, inverse: bool = False):
        """Replace one limb's forward / inverse table by the caller's, in the reference's order (ntt.cpp:298-300)."""
        r = np.ascontiguousarray(roots, dtype=np.uint32)
        if r.size != self.n:
            raise ValueError("need n table entries")
        pp = None
        if precons is not None:
            pc = np.ascontiguousarray(precons, dtype=np.uint32)
            if pc.size != self.n:
                raise ValueError("need n table entries")
            pp = pc.ctypes.data_as(_u32p)
        _ck(lib().agx_set_tables(self._h, limb, int(inverse), r.ctypes.data_as(_u32p), pp), "agx_set_tables")

    def measure_butterfly_peak(self, kind: int = 0, threads_per_sm: int = 1024):
        """(butterflies per clock per SM, implied SM MHz) of the butterfly instruction stream alone on this GPU."""
        v, mhz = C.c_double(), C.c_double()
        _ck(lib().agx_measure_butterfly_peak(self._h, kind, threads_per_sm, C.byref(v), C.byref(mhz)),
            "agx_measure_butterfly_peak")
        return v.value, mhz.value

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().agx_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    # ---- introspection
    def psi(self, limb: int = 0) -> int:
        v = C.c_uint32()
        _ck(lib().agx_get_psi(self._h, limb, C.byref(v)), "agx_get_psi")
        return v.value

    def tables(self, limb: int = 0, inverse: bool = False):
        r = np.empty(self.n, dtype=np.uint32)
        p = np.empty(self.n, dtype=np.uint32)
        _ck(lib().agx_get_tables(self._h, limb, int(inverse), r.ctypes.data_as(_u32p), p.ctypes.data_as(_u32p)),
            "agx_get_tables")
        return r, p

    def variant(self) -> str:
        b = C.create_string_buffer(64)
        _ck(lib().agx_variant(self._h, b, 64), "agx_variant")
        return b.value.decode()

    def launch_count(self) -> int:
        v = C.c_uint64()
        _ck(lib().agx_launch_count(self._h, C.byref(v)), "agx_launch_count")
        return v.value

    def _batch(self, t) -> int:
        words = t.numel()
        if words % (self.L * self.n):
            raise ValueError("tensor is not a whole number of [L][n] polynomials")
        return words // (self.L * self.n)

    # ---- device-pointer entry points (torch CUDA tensors, in place)
    def fwd(self, t, stream=None):
        _ck(lib().agx_ntt_fwd(self._h, _dev_ptr(t), self._batch(t), _stream_ptr(stream)), "agx_ntt_fwd")
        return t

    def inv(self, t, stream=None):
        _ck(lib().agx_ntt_inv(self._h, _dev_ptr(t), self._batch(t), _stream_ptr(stream)), "agx_ntt_inv")
        return t

    def polymul(self, c, a, b, stream=None):
        B = self._batch(a)
        if self._batch(b) != B or self._batch(c) != B:
            raise ValueError("shape mismatch")
        _ck(lib().agx_polymul(self._h, _dev_ptr(c), _dev_ptr(a), _dev_ptr(b), B, _stream_ptr(stream)), "agx_polymul")
        return c

    def polymul_by_spectrum(self, c, a, b_hat, stream=None):
        """c = INTT(NTT(a) .* b_hat) with b_hat = fwd(b): the product when one operand is kept in evaluation form."""
        B = self._batch(a)
        if self._batch(b_hat) != B or self._batch(c) != B:
            raise ValueError("shape mismatch")
        _ck(lib().agx_polymul_by_spectrum(self._h, _dev_ptr(c), _dev_ptr(a), _dev_ptr(b_hat), B, _stream_ptr(stream)),
            "agx_polymul_by_spectrum")
        return c

    EW = {"add": 0, "sub": 1, "mul": 2, "mac": 3}

    def elementwise(self, op: str, c, a, b, stream=None):
        """c = a + b | a - b | a * b | c + a * b, modulo each limb's prime (operands reduced, device tensors)."""
        B = self._batch(a)
        if self._batch(b) != B or self._batch(c) != B:
            raise ValueError("shape mismatch")
        _ck(lib().agx_elementwise(self._h, self.EW[op], _dev_ptr(c), _dev_ptr(a), _dev_ptr(b), B, _stream_ptr(stream)),
            "agx_elementwise")
        return c

    def bitrev(self, t, stream=None):
        """Permute every polynomial of t by bit reversal, in place (natural <-> bit-reversed coefficient order)."""
        _ck(lib().agx_bitrev(self._h, _dev_ptr(t), self._batch(t), _stream_ptr(stream)), "agx_bitrev")
        return t

    def fill_synthetic(self, t, seed: int = 42, first_poly: int = 0, stream=None):
        _ck(lib().agx_fill_synthetic(self._h, _dev_ptr(t), self._batch(t), seed, first_poly, _stream_ptr(stream)),
            "agx_fill_synthetic")
        return t

    def checksum(self, t, first_index: int = 0, stream=None) -> int:
        v = C.c_uint64()
        _ck(lib().agx_checksum(self._h, _dev_ptr(t), t.numel(), first_index, C.byref(v), _stream_ptr(stream)),
            "agx_checksum")
        return v.value

    # ---- host-pointer entry points (numpy uint32 arrays or raw addresses)
    @staticmethod
    def _host_ptr(a) -> int:
        if isinstance(a, int):
            return a
        if isinstance(a, np.ndarray):
            if a.dtype != np.uint32 or not a.flags.c_contiguous:
                raise ValueError("need a C-contiguous uint32 array")
            return a.ctypes.data
        if hasattr(a, "data_ptr"):   # pinned torch CPU tensor
            if a.is_cuda or not a.is_contiguous() or a.element_size() != 4:
                raise ValueError("need a contiguous 4-byte CPU tensor")
            return a.data_ptr()
        raise TypeError(type(a))

    def _host_batch(self, a, B):
        if B is not None:
            return B
        words = a.size if isinstance(a, np.ndarray) else a.numel()
        if words % (self.L * self.n):
            raise ValueError("array is not a whole number of [L][n] polynomials")
        return words // (self.L * self.n)

    def fwd_host(self, src, dst=None, B=None):
        dst = src if dst is None else dst
        _ck(lib().agx_ntt_fwd_host(self._h, self._host_ptr(src), self._host_ptr(dst), self._host_batch(src, B)),
            "agx_ntt_fwd_host")
        return dst

    def inv_host(self, src, dst=None, B=None):
        dst = src if dst is None else dst
        _ck(lib().agx_ntt_inv_host(self._h, self._host_ptr(src), self._host_ptr(dst), self._host_batch(src, B)),
            "agx_ntt_inv_host")
        return dst

    def polymul_host(self, c, a, b, B=None):
        _ck(lib().agx_polymul_host(self._h, self._host_ptr(c), self._host_ptr(a), self._host_ptr(b),
                                   self._host_batch(a, B)), "agx_polymul_host")
        return c

    def polymul_by_spectrum_host(self, c, a, b_hat, B=None):
        _ck(lib().agx_polymul_by_spectrum_host(self._h, self._host_ptr(c), self._host_ptr(a), self._host_ptr(b_hat),
                                               self._host_batch(a, B)), "agx_polymul_by_spectrum_host")
        return c


class Context64:
    """One (n, primes) u64 parameter set bound to one GPU: L primes of up to 62 bits (q = 1 mod 2n), the device tables,
    and batched [B][L][n] transforms and products over them (agx_create64).  Data are contiguous CUDA tensors of int64 or
    uint64 words; every call works in place on them, on the current torch stream unless `stream` is given."""

    EW = Context.EW

    def __init__(self, n: int, primes, device: int = 0, psi=None):
        """psi: the caller's primitive 2n-th root per limb; None = the minimal root of each prime."""
        self._h = C.c_void_p()
        self.n = int(n)
        self.logn = self.n.bit_length() - 1
        self.primes = [int(q) for q in primes]
        self.L = len(self.primes)
        self.device = device
        self._q = (C.c_uint64 * max(self.L, 1))(*self.primes)
        p = _Parms64(self.n, self.logn, self.L, C.cast(self._q, _u64p))
        arr = None
        if psi is not None:
            psi = [int(v) for v in psi]
            if len(psi) != self.L:
                raise ValueError("need one psi per limb")
            arr = C.cast((C.c_uint64 * self.L)(*psi), _u64p)
        _ck(lib().agx_create64(C.byref(self._h), C.byref(p), arr, device), "agx_create64")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().agx_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def psi(self, limb: int = 0) -> int:
        v = C.c_uint64()
        _ck(lib().agx_get_psi64(self._h, limb, C.byref(v)), "agx_get_psi64")
        return v.value

    def tables(self, limb: int = 0, inverse: bool = False):
        """(roots, precons) of one limb as uint64 arrays in the reference's order: what agx_ref_fwd_dev / inv_dev take."""
        r = np.empty(self.n, dtype=np.uint64)
        p = np.empty(self.n, dtype=np.uint64)
        _ck(lib().agx_get_tables64(self._h, limb, int(inverse), r.ctypes.data_as(_u64p), p.ctypes.data_as(_u64p)),
            "agx_get_tables64")
        return r, p

    def launch_count(self) -> int:
        v = C.c_uint64()
        _ck(lib().agx_launch_count(self._h, C.byref(v)), "agx_launch_count")
        return v.value

    def _batch(self, t) -> int:
        words = t.numel()
        if words % (self.L * self.n):
            raise ValueError("tensor is not a whole number of [L][n] polynomials")
        return words // (self.L * self.n)

    def _batch3(self, c, a, b) -> int:
        B = self._batch(a)
        if self._batch(b) != B or self._batch(c) != B:
            raise ValueError("shape mismatch")
        return B

    def fwd(self, t, stream=None):
        """Forward NTT of every limb (inputs < 4q), natural in, bit-reversed out, results in [0,q)."""
        _ck(lib().agx_ntt64_fwd(self._h, _dev_ptr8(t), self._batch(t), _stream_ptr(stream)), "agx_ntt64_fwd")
        return t

    def inv(self, t, stream=None):
        """Inverse NTT of every limb (inputs < 2q), bit-reversed in, natural out, n^-1 folded in."""
        _ck(lib().agx_ntt64_inv(self._h, _dev_ptr8(t), self._batch(t), _stream_ptr(stream)), "agx_ntt64_inv")
        return t

    def polymul(self, c, a, b, stream=None):
        """c = a * b mod (X^n + 1, q_limb) for every limb (reduced operands; c may alias a and/or b)."""
        B = self._batch3(c, a, b)
        _ck(lib().agx_polymul64(self._h, _dev_ptr8(c), _dev_ptr8(a), _dev_ptr8(b), B, _stream_ptr(stream)),
            "agx_polymul64")
        return c

    def polymul_by_spectrum(self, c, a, b_hat, stream=None):
        """c = INTT(NTT(a) .* b_hat) with b_hat = fwd(b): the product when one operand is kept in evaluation form."""
        B = self._batch3(c, a, b_hat)
        _ck(lib().agx_polymul64_by_spectrum(self._h, _dev_ptr8(c), _dev_ptr8(a), _dev_ptr8(b_hat), B,
                                            _stream_ptr(stream)), "agx_polymul64_by_spectrum")
        return c

    def elementwise(self, op: str, c, a, b, stream=None):
        """c = a + b | a - b | a * b | c + a * b, modulo each limb's prime (operands reduced)."""
        B = self._batch3(c, a, b)
        _ck(lib().agx_elementwise64(self._h, self.EW[op], _dev_ptr8(c), _dev_ptr8(a), _dev_ptr8(b), B,
                                    _stream_ptr(stream)), "agx_elementwise64")
        return c

    def rescale(self, out, inp, ntt_form=True, stream=None):
        """Divide by the last prime and round (agx_rescale64): inp (B, L, n) -> out (B, L - 1, n), the residues of
        floor((X + h) / q_{L-1}) with h = floor(q_{L-1} / 2) over the first L - 1 primes.  ntt_form: both in evaluation
        form as fwd leaves them (else both in coefficient form).  Reduced inputs; out must not overlap inp.  The result
        belongs to a context over primes[:-1] (same roots), whose tables are this context's first L - 1 limbs."""
        for t in (out, inp):
            if not t.is_cuda or t.device.index != self.device:
                raise ValueError(f"need CUDA tensors on device {self.device}")
        if inp.dim() != 3 or tuple(inp.shape[1:]) != (self.L, self.n):
            raise ValueError(f"inp must have shape (B, {self.L}, {self.n})")
        B = inp.shape[0]
        if tuple(out.shape) != (B, self.L - 1, self.n):
            raise ValueError(f"out must have shape ({B}, {self.L - 1}, {self.n})")
        _ck(lib().agx_rescale64(self._h, _dev_ptr8(out), _dev_ptr8(inp), B, int(bool(ntt_form)), _stream_ptr(stream)),
            "agx_rescale64")
        return out

    def _check_dev(self, *ts):
        for t in ts:
            if not t.is_cuda or t.device.index != self.device:
                raise ValueError(f"need CUDA tensors on device {self.device}")

    def moddown(self, out, inp, k, ntt_form=True, stream=None):
        """Divide by P = q_{L-k} ... q_{L-1}, the last k primes, and round (agx_moddown64): inp (B, L, n) ->
        out (B, L - k, n), the residues of floor((X + (P - 1) / 2) / P) over the first L - k primes.  ntt_form: both in
        evaluation form as fwd leaves them (else both in coefficient form).  k = 1 is rescale.  Reduced inputs; out must
        not overlap inp.  The result belongs to a context over primes[:L - k] (same roots)."""
        self._check_dev(out, inp)
        if inp.dim() != 3 or tuple(inp.shape[1:]) != (self.L, self.n):
            raise ValueError(f"inp must have shape (B, {self.L}, {self.n})")
        B = inp.shape[0]
        if not 0 < k < self.L:
            raise ValueError(f"k must be in [1, {self.L - 1}]")
        if tuple(out.shape) != (B, self.L - k, self.n):
            raise ValueError(f"out must have shape ({B}, {self.L - k}, {self.n})")
        _ck(lib().agx_moddown64(self._h, _dev_ptr8(out), _dev_ptr8(inp), B, k, int(bool(ntt_form)), _stream_ptr(stream)),
            "agx_moddown64")
        return out

    def modup(self, out, inp, first, count, ntt_form=True, stream=None):
        """Extend from the primes q_first .. q_{first+count-1} (product S) to all L primes (agx_modup64): inp
        (B, count, n) -> out (B, L, n), every limb the residue of the centred lift ((X + h) mod S) - h, h = (S - 1) / 2;
        out's limbs first .. first + count - 1 equal inp.  ntt_form: both in evaluation form (else both in coefficient
        form).  Reduced inputs; out must not overlap inp."""
        self._check_dev(out, inp)
        if not (0 < count < self.L and 0 <= first <= self.L - count):
            raise ValueError(f"need 0 < count < {self.L} and 0 <= first <= {self.L} - count")
        if inp.dim() != 3 or tuple(inp.shape[1:]) != (count, self.n):
            raise ValueError(f"inp must have shape (B, {count}, {self.n})")
        B = inp.shape[0]
        if tuple(out.shape) != (B, self.L, self.n):
            raise ValueError(f"out must have shape ({B}, {self.L}, {self.n})")
        _ck(lib().agx_modup64(self._h, _dev_ptr8(out), _dev_ptr8(inp), B, first, count, int(bool(ntt_form)),
                              _stream_ptr(stream)), "agx_modup64")
        return out

    def automorph(self, out, inp, galois, ntt_form=True, stream=None):
        """Galois automorphism sigma_g: a(X) -> a(X^g) mod X^n + 1 on every limb (agx_automorph64), g odd in [1, 2n).
        galois: one int, with inp and out of shape (B, L, n), or a sequence of G ints (at most 64), with out of shape
        (G, B, L, n), out[t] = sigma_{galois[t]}(inp): the input is read once for all G.  galois_element(n, r) rotates the
        slots by r steps; 2n - 1 is the conjugation.  ntt_form: both in evaluation form as fwd leaves them, where sigma_g
        is a permutation (else both in coefficient form, where it also negates).  Reduced inputs; out must not overlap
        inp."""
        self._check_dev(out, inp)
        if inp.dim() != 3 or tuple(inp.shape[1:]) != (self.L, self.n):
            raise ValueError(f"inp must have shape (B, {self.L}, {self.n})")
        B = inp.shape[0]
        single = isinstance(galois, numbers.Integral)
        gs = [int(galois)] if single else [int(g) for g in galois]
        want = (B, self.L, self.n) if single else (len(gs), B, self.L, self.n)
        if tuple(out.shape) != want:
            raise ValueError(f"out must have shape {want}")
        if any(not 0 <= g < 1 << 32 for g in gs):
            raise ValueError("Galois elements must be 32-bit unsigned integers (odd, below 2n)")
        arr = (C.c_uint32 * max(len(gs), 1))(*gs)
        _ck(lib().agx_automorph64(self._h, _dev_ptr8(out), _dev_ptr8(inp), B, C.cast(arr, _u32p), len(gs),
                                  int(bool(ntt_form)), _stream_ptr(stream)), "agx_automorph64")
        return out

    def keyswitch(self, out, inp, ksk, alpha, k, ntt_form=True, stream=None):
        """Hybrid key switching in one call (agx_keyswitch64), this context being Q_l u P with the k special primes last:
        inp (B, L - k, n) over Q_l -> out (2, B, L - k, n), out[c] = ModDown_P(sum_j ModUp_j(digit_j) * ksk[j][c]).
        Digit j is limbs j*alpha .. (j+1)*alpha - 1 of inp (the last one may be shorter; alpha >= L - k is one digit).
        ksk (D, 2, key_limbs, n), D >= the number of digits, in evaluation form as fwd leaves it; key_limbs >= L: limb
        i < L - k reads key row i, special prime t reads row key_limbs - k + t, so one key over Q_top u P serves every
        level.  ntt_form: inp and out in evaluation form (else both in coefficient form; the key is in evaluation form
        either way).  Reduced inputs; out must not overlap inp or ksk.  The result belongs to a context over
        primes[:L - k]."""
        self._check_dev(out, inp, ksk)
        if not 0 < int(k) < self.L:
            raise ValueError(f"k must be in [1, {self.L - 1}]")
        alpha, k = int(alpha), int(k)
        if not 1 <= alpha < 1 << 32:
            raise ValueError("alpha must be a 32-bit unsigned integer, at least 1")
        ell1 = self.L - k
        if inp.dim() != 3 or tuple(inp.shape[1:]) != (ell1, self.n):
            raise ValueError(f"inp must have shape (B, {ell1}, {self.n})")
        B = inp.shape[0]
        if tuple(out.shape) != (2, B, ell1, self.n):
            raise ValueError(f"out must have shape (2, {B}, {ell1}, {self.n})")
        dnum = -(-ell1 // min(alpha, ell1))
        if ksk.dim() != 4 or ksk.shape[0] < dnum or ksk.shape[1] != 2 or ksk.shape[2] < self.L or ksk.shape[3] != self.n:
            raise ValueError(f"ksk must have shape (D >= {dnum}, 2, key_limbs >= {self.L}, {self.n})")
        _ck(lib().agx_keyswitch64(self._h, _dev_ptr8(out), _dev_ptr8(inp), B, _dev_ptr8(ksk), ksk.shape[2], alpha, k,
                                  int(bool(ntt_form)), _stream_ptr(stream)), "agx_keyswitch64")
        return out

    def rotate(self, out, ct, galois, rks, alpha, k, ntt_form=True, stream=None):
        """Hoisted rotations in one call (agx_rotate64), this context being Q_l u P with the k special primes last:
        ct (2, B, L - k, n), ciphertexts (c0, c1) over Q_l.  galois: one int with out of shape (2, B, L - k, n), or a
        sequence of G ints (at most 64) with out of shape (G, 2, B, L - k, n); rks: a sequence of G keys (D, 2, key_limbs,
        n) with one key_limbs, key t switching sigma_{galois[t]}(s) to s, laid out as for keyswitch (the same tensor may
        serve several elements).  out[t] = (sigma_t(c0) + KS_t(sigma_t(c1))[0], KS_t(sigma_t(c1))[1]), bit for bit what
        automorph, keyswitch with rks[t] and an elementwise add give, with one ModUp of c1 for all G.  ntt_form: ct and
        out in evaluation form (else both in coefficient form; the keys are in evaluation form either way).  out must
        not overlap ct or the keys.  The result belongs to a context over primes[:L - k]."""
        single = isinstance(galois, numbers.Integral)
        gs = [int(galois)] if single else [int(g) for g in galois]
        rks = list(rks)
        self._check_dev(out, ct, *rks)
        if not 0 < int(k) < self.L:
            raise ValueError(f"k must be in [1, {self.L - 1}]")
        alpha, k = int(alpha), int(k)
        if not 1 <= alpha < 1 << 32:
            raise ValueError("alpha must be a 32-bit unsigned integer, at least 1")
        ell1 = self.L - k
        if ct.dim() != 4 or ct.shape[0] != 2 or tuple(ct.shape[2:]) != (ell1, self.n):
            raise ValueError(f"ct must have shape (2, B, {ell1}, {self.n})")
        B = ct.shape[1]
        want = (2, B, ell1, self.n) if single else (len(gs), 2, B, ell1, self.n)
        if tuple(out.shape) != want:
            raise ValueError(f"out must have shape {want}")
        if any(not 0 <= g < 1 << 32 for g in gs):
            raise ValueError("Galois elements must be 32-bit unsigned integers (odd, below 2n)")
        if len(rks) != len(gs):
            raise ValueError(f"rks must hold one key per Galois element ({len(gs)})")
        dnum = -(-ell1 // min(alpha, ell1))
        key_limbs = rks[0].shape[2] if rks and rks[0].dim() == 4 else 0
        for rk in rks:
            if rk.dim() != 4 or rk.shape[0] < dnum or rk.shape[1] != 2 or rk.shape[2] != key_limbs or \
                    key_limbs < self.L or rk.shape[3] != self.n:
                raise ValueError(f"every key must have shape (D >= {dnum}, 2, key_limbs >= {self.L}, {self.n}), "
                                 "with one key_limbs for all")
        arr = (C.c_uint32 * max(len(gs), 1))(*gs)
        ptrs = (C.c_void_p * max(len(rks), 1))(*[_dev_ptr8(rk) for rk in rks])
        _ck(lib().agx_rotate64(self._h, _dev_ptr8(out), _dev_ptr8(ct), B, C.cast(arr, _u32p), len(gs), ptrs, key_limbs,
                               alpha, k, int(bool(ntt_form)), _stream_ptr(stream)), "agx_rotate64")
        return out

    def lintrans(self, out, ct, galois, rks, diags, alpha, k, ntt_form=True, stream=None):
        """Hoisted linear transform in one call (agx_lintrans64), this context being Q_l u P with the k special primes
        last: ct (2, B, L - k, n), ciphertexts (c0, c1) over Q_l; galois a sequence of G ints (at most 64); rks G keys
        laid out as for rotate, or None where the element is 1 (the identity term, with no key switch); diags M
        sequences (at most 16, M * G <= 256) of G entries, each an (L, n) tensor over all L primes in evaluation form, or
        None for a zero diagonal.  out (M, 2, B, L - k, n): out[m] = ModDown_P(sum_t diags[m][t] * A_t), A_t rotate's
        inner product for element t before its ModDown, so out[m] is sum_t d_{m,t} rot_t(ct) with one ModUp for all G
        and one rounding per output (not bit-equal to summing rotate's outputs, which rounds G times).  ntt_form: ct and
        out in evaluation form (else both in coefficient form; keys and diagonals are in evaluation form either way).
        out must not overlap ct, the keys or the diagonals.  The result belongs to a context over primes[:L - k]."""
        gs = [int(g) for g in galois]
        rks = list(rks)
        diags = [list(row) for row in diags]
        keys = [rk for rk in rks if rk is not None]
        dlist = [d for row in diags for d in row if d is not None]
        self._check_dev(out, ct, *keys, *dlist)
        if not 0 < int(k) < self.L:
            raise ValueError(f"k must be in [1, {self.L - 1}]")
        alpha, k = int(alpha), int(k)
        if not 1 <= alpha < 1 << 32:
            raise ValueError("alpha must be a 32-bit unsigned integer, at least 1")
        ell1 = self.L - k
        if ct.dim() != 4 or ct.shape[0] != 2 or tuple(ct.shape[2:]) != (ell1, self.n):
            raise ValueError(f"ct must have shape (2, B, {ell1}, {self.n})")
        B, G, M = ct.shape[1], len(gs), len(diags)
        if tuple(out.shape) != (M, 2, B, ell1, self.n):
            raise ValueError(f"out must have shape {(M, 2, B, ell1, self.n)}")
        if any(not 0 <= g < 1 << 32 for g in gs):
            raise ValueError("Galois elements must be 32-bit unsigned integers (odd, below 2n)")
        if len(rks) != G:
            raise ValueError(f"rks must hold one key (or None for the element 1) per Galois element ({G})")
        if any(rk is None and g != 1 for rk, g in zip(rks, gs)):
            raise ValueError("only the element 1 may go without a key")
        if any(len(row) != G for row in diags):
            raise ValueError(f"every row of diags must hold one entry (or None) per Galois element ({G})")
        dnum = -(-ell1 // min(alpha, ell1))
        key_limbs = keys[0].shape[2] if keys and keys[0].dim() == 4 else self.L
        for rk in keys:
            if rk.dim() != 4 or rk.shape[0] < dnum or rk.shape[1] != 2 or rk.shape[2] != key_limbs or \
                    key_limbs < self.L or rk.shape[3] != self.n:
                raise ValueError(f"every key must have shape (D >= {dnum}, 2, key_limbs >= {self.L}, {self.n}), "
                                 "with one key_limbs for all")
        for d in dlist:
            if tuple(d.shape) != (self.L, self.n):
                raise ValueError(f"every diagonal must have shape ({self.L}, {self.n})")
        arr = (C.c_uint32 * max(G, 1))(*gs)
        kp = (C.c_void_p * max(G, 1))(*[None if rk is None else _dev_ptr8(rk) for rk in rks])
        dp = (C.c_void_p * max(M * G, 1))(*[None if d is None else _dev_ptr8(d) for row in diags for d in row])
        _ck(lib().agx_lintrans64(self._h, _dev_ptr8(out), _dev_ptr8(ct), B, C.cast(arr, _u32p), G, kp, key_limbs, dp, M,
                                 alpha, k, int(bool(ntt_form)), _stream_ptr(stream)), "agx_lintrans64")
        return out

    def mulrelin(self, out, a, b, rlk, alpha, k, rescale=False, ntt_form=True, stream=None):
        """Ciphertext multiplication in one call (agx_mulrelin64), this context being Q_l u P with the k special primes
        last: a and b (2, B, L - k, n), ciphertexts over Q_l (the same tensor squares); rlk the relinearisation key (the
        key-switch key for s^2), laid out as for keyswitch.  With D_0 = a0 b0, D_1 = a0 b1 + a1 b0, D_2 = a1 b1 and
        A_c = sum_j ModUp_j(digit_j(D_2)) * rlk[j][c] + P D_c over Q_l u P:
        rescale False: out (2, B, L - k, n), out[c] = ModDown_P(A_c) = D_c + keyswitch(D_2)[c], bit for bit;
        rescale True: out (2, B, L - k - 1, n), A_c divided by q_l P (the last k + 1 primes) and rounded once, i.e.
        moddown with k + 1, which equals rescale of the unrescaled result bit for bit (the roundings compose); it
        belongs to a context over primes[:L - k - 1].  ntt_form: a, b and out in evaluation form (else all in coefficient form; the key is in
        evaluation form either way).  out must not overlap a, b or rlk."""
        self._check_dev(out, a, b, rlk)
        if not 0 < int(k) < self.L:
            raise ValueError(f"k must be in [1, {self.L - 1}]")
        alpha, k = int(alpha), int(k)
        if not 1 <= alpha < 1 << 32:
            raise ValueError("alpha must be a 32-bit unsigned integer, at least 1")
        ell1 = self.L - k
        for t in (a, b):
            if t.dim() != 4 or t.shape[0] != 2 or tuple(t.shape[2:]) != (ell1, self.n):
                raise ValueError(f"a and b must have shape (2, B, {ell1}, {self.n})")
        B = a.shape[1]
        if b.shape[1] != B:
            raise ValueError("a and b must hold the same number of ciphertexts")
        if rescale and ell1 < 2:
            raise ValueError("rescale needs at least two primes in Q_l")
        want = (2, B, ell1 - 1 if rescale else ell1, self.n)
        if tuple(out.shape) != want:
            raise ValueError(f"out must have shape {want}")
        dnum = -(-ell1 // min(alpha, ell1))
        if rlk.dim() != 4 or rlk.shape[0] < dnum or rlk.shape[1] != 2 or rlk.shape[2] < self.L or rlk.shape[3] != self.n:
            raise ValueError(f"rlk must have shape (D >= {dnum}, 2, key_limbs >= {self.L}, {self.n})")
        _ck(lib().agx_mulrelin64(self._h, _dev_ptr8(out), _dev_ptr8(a), _dev_ptr8(b), B, _dev_ptr8(rlk), rlk.shape[2],
                                 alpha, k, int(bool(rescale)), int(bool(ntt_form)), _stream_ptr(stream)),
            "agx_mulrelin64")
        return out

    def _slots_and_residues(self, z, res):
        self._check_dev(z, res)
        if z.dtype != _complex128() or z.dim() != 2 or z.shape[1] != self.n // 2 or not z.is_contiguous():
            raise ValueError(f"slots must be a contiguous complex128 tensor of shape (B, {self.n // 2})")
        B = z.shape[0]
        if res.dim() != 3 or res.shape[0] != B or not 1 <= res.shape[1] <= self.L or res.shape[2] != self.n:
            raise ValueError(f"residues must have shape ({B}, limbs, {self.n}) with 1 <= limbs <= {self.L}")
        return B, res.shape[1]

    def encode(self, out, z, scale, ntt_form=True, stream=None):
        """CKKS encoding (agx_encode64): slots z (B, n/2) complex128 -> out (B, limbs, n) int64 or uint64 over the first
        limbs primes (limbs from out's shape): c_i = rint(scale * m_i), m the real polynomial with m(zeta^(5^j)) = z_j,
        zeta = exp(i pi / n), reduced mod each prime exactly at any magnitude.  ntt_form: out in evaluation form as fwd
        leaves it (else coefficient form).  With limbs = L, out[b] is a diagonal as lintrans takes it."""
        B, limbs = self._slots_and_residues(z, out)
        _ck(lib().agx_encode64(self._h, _dev_ptr8(out), z.data_ptr(), B, float(scale), limbs, int(bool(ntt_form)),
                               _stream_ptr(stream)), "agx_encode64")
        return out

    def decode(self, z, inp, scale, ntt_form=True, stream=None):
        """CKKS decoding (agx_decode64): inp (B, limbs, n) over the first limbs primes -> slots z (B, n/2) complex128:
        the centred CRT value of each coefficient over q_0 ... q_(limbs-1), divided by scale, then evaluated at
        zeta^(5^j).  ntt_form: inp in evaluation form (else coefficient form); inp is not modified."""
        B, limbs = self._slots_and_residues(z, inp)
        _ck(lib().agx_decode64(self._h, z.data_ptr(), _dev_ptr8(inp), B, float(scale), limbs, int(bool(ntt_form)),
                               _stream_ptr(stream)), "agx_decode64")
        return z


def galois_element(n: int, step: int) -> int:
    """The Galois element of a slot rotation by `step` on X^n + 1: 5^step mod 2n, a negative step taking the inverse of
    5 (mod 2n).  The conjugation is 2n - 1, which no power of 5 reaches."""
    return pow(5, int(step), 2 * int(n))


class RefPipeline:
    """Reference-shaped u64 forward pipeline: ntt_input_kernel / fwd_ntt_kernel<0> / ntt_output_kernel / q.wait()
    (include/kernel/ntt.h:32-45, src/main.cpp:60-74) over agx_ref_*."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _ck(lib().agx_create(C.byref(self._h), None, device), "agx_create")
        self._keep = []

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().agx_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    @staticmethod
    def _p(a):
        assert a.dtype == np.uint64 and a.flags.c_contiguous
        return a.ctypes.data_as(_u64p)

    def ntt_input_kernel(self, in1, in2, modulus, twiddles, precons, num_frames: int):
        N = len(twiddles)
        arrs = [np.ascontiguousarray(x, dtype=np.uint64) for x in (in1, in2, modulus, twiddles, precons)]
        # agx_ref_input takes bare pointers: the buffer-size contract of ntt_input_kernel (main.cpp:26-37) is checked here
        if len(arrs[4]) != N or len(arrs[2]) < 1 or len(arrs[0]) < N * num_frames or len(arrs[1]) < N * num_frames:
            raise ValueError("buffer sizes do not describe numFrames x N")
        self._n = N
        self._check_out()
        self._keep += arrs
        _ck(lib().agx_ref_input(self._h, N, *[self._p(a) for a in arrs], num_frames), "agx_ref_input")

    def fwd_ntt_kernel(self, compute_unit: int = 0):
        _ck(lib().agx_ref_fwd(self._h, compute_unit), "agx_ref_fwd")

    def _check_out(self):
        if getattr(self, "_n", 0) and getattr(self, "_out", None) is not None:
            if self._out[0] < self._out[1] * self._n:
                self._out = None
                raise ValueError("out is smaller than numFrames x N")

    def ntt_output_kernel(self, out: np.ndarray, num_frames: int):
        if num_frames < 0:
            raise ValueError("negative numFrames")
        self._out = (out.size, num_frames)
        self._check_out()
        self._keep.append(out)
        _ck(lib().agx_ref_output(self._h, self._p(out), num_frames), "agx_ref_output")

    def wait(self):
        try:
            _ck(lib().agx_wait(self._h), "agx_wait")
        finally:
            self._keep.clear()
            self._n, self._out = 0, None

    @staticmethod
    def _ptr(t) -> int:
        return t if isinstance(t, int) else t.data_ptr()

    def fwd_dev(self, N: int, d_in, d_in2, d_out, modulus: int, d_tw, d_pre, frames: int, stream=None):
        """agx_ref_fwd_dev on torch CUDA int64 tensors (or raw device addresses)."""
        ptr = self._ptr
        _ck(lib().agx_ref_fwd_dev(self._h, N, ptr(d_in), ptr(d_in2), ptr(d_out), modulus, ptr(d_tw), ptr(d_pre), frames,
                                  _stream_ptr(stream)), "agx_ref_fwd_dev")

    def inv_dev(self, N: int, d_in, d_out, modulus: int, d_itw, d_ipre, frames: int, stream=None):
        """agx_ref_inv_dev: the inverse of fwd_dev (bit-reversed in, natural out); d_itw / d_ipre from psi^-1."""
        ptr = self._ptr
        _ck(lib().agx_ref_inv_dev(self._h, N, ptr(d_in), ptr(d_out), modulus, ptr(d_itw), ptr(d_ipre), frames,
                                  _stream_ptr(stream)), "agx_ref_inv_dev")

    def polymul_dev(self, N: int, d_c, d_a, d_b, modulus: int, d_tw, d_pre, d_itw, d_ipre, frames: int, stream=None):
        """agx_ref_polymul_dev: c = a * b mod (X^N + 1, q) per frame (reduced operands; c may alias a and/or b)."""
        ptr = self._ptr
        _ck(lib().agx_ref_polymul_dev(self._h, N, ptr(d_c), ptr(d_a), ptr(d_b), modulus, ptr(d_tw), ptr(d_pre), ptr(d_itw),
                                      ptr(d_ipre), frames, _stream_ptr(stream)), "agx_ref_polymul_dev")

    def polymul_by_spectrum_dev(self, N: int, d_c, d_a, d_b_hat, modulus: int, d_tw, d_pre, d_itw, d_ipre, frames: int,
                                stream=None):
        """agx_ref_polymul_by_spectrum_dev: c = INTT(NTT(a) .* b_hat), b_hat = fwd_dev(b)."""
        ptr = self._ptr
        _ck(lib().agx_ref_polymul_by_spectrum_dev(self._h, N, ptr(d_c), ptr(d_a), ptr(d_b_hat), modulus, ptr(d_tw),
                                                  ptr(d_pre), ptr(d_itw), ptr(d_ipre), frames, _stream_ptr(stream)),
            "agx_ref_polymul_by_spectrum_dev")

    def launch_count(self) -> int:
        v = C.c_uint64()
        _ck(lib().agx_launch_count(self._h, C.byref(v)), "agx_launch_count")
        return v.value
