"""Kernel rates of the u64 inverse transform and negacyclic product on device-resident frames (agx_ref_inv_dev,
agx_ref_polymul_dev, agx_ref_polymul_by_spectrum_dev) beside the forward (agx_ref_fwd_dev) of the same call: frames/s
and products/s, launches per call, fractions of the HBM copy rate and of the u64 butterfly rate both MEASURED in this run
(a 1 GiB device-to-device copy; agx_measure_butterfly_peak kind 1).  60-bit NTT prime, 16 MiB (L2-resident) and 1 GiB
batches; forward and inverse are timed alternately with CUDA events after a warm-up.  Every line carries a parity spot
check of its first two frames against the CPU oracle (tests/native/u64_inverse_oracle.c, built into a temporary directory).
Usage (GPU box): python profiles/bench_u64_inv.py > <log>.jsonl"""
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import agilex_ntt_b200 as A
from oracle import oracle as O      # inputs / tables / spot checks only (this is a measurement script, not the product)

_u64p = C.POINTER(C.c_uint64)


def load_oracle(tmp):
    so = os.path.join(tmp, "libu64oracle.so")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc") or "cc"
    base = [cc, "-O2", "-std=c11", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "tests", "native", "u64_inverse_oracle.c")]
    if subprocess.run(base + ["-fopenmp"], capture_output=True).returncode != 0:
        subprocess.run(base + ["-Wno-unknown-pragmas"], check=True)
    L = C.CDLL(so)
    L.orc_inv_u64.argtypes = [C.c_uint32, _u64p, C.c_uint64, _u64p, C.c_size_t, C.c_int]
    return L


def u64(t):
    return t.cpu().numpy().view(np.uint64)


def timed_pair(f, g, iters, rounds=3):
    """ms per call of f and of g, alternated: `rounds` windows of `iters` calls each, after a warm-up of both."""
    for _ in range(2):
        f(); g()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tf = tg = 0.0
    for _ in range(rounds):
        ev[0].record()
        for _ in range(iters):
            f()
        ev[1].record()
        for _ in range(iters):
            g()
        ev[2].record()
        torch.cuda.synchronize()
        tf += ev[0].elapsed_time(ev[1])
        tg += ev[1].elapsed_time(ev[2])
    return tf / (rounds * iters), tg / (rounds * iters)


def main():
    tmp = tempfile.mkdtemp(prefix="bench_u64_inv_")
    orc = load_oracle(tmp)
    q = O.U64_PRIMES[60]
    p = A.RefPipeline()
    ctx = A.Context(1024, [1053818881])
    peak64, mhz = ctx.measure_butterfly_peak(1, 1024)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    src = torch.empty(1 << 27, dtype=torch.int64, device="cuda")
    dst = torch.empty_like(src)
    ms_copy, _ = timed_pair(lambda: dst.copy_(src), lambda: None, 10)
    copy_gbs = 2 * src.numel() * 8 / (ms_copy * 1e-3) / 1e9
    del src, dst
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "power_limit": power, "sms": sms,
                      "u64_butterflies_per_clk_per_sm": peak64, "implied_sm_mhz": mhz,
                      "hbm_copy_GBps_measured": copy_gbs}), flush=True)

    def rates(N, frames, ms, mults):
        per_s = frames / (ms * 1e-3)
        bfly = per_s * mults / (sms * mhz * 1e6)
        return per_s, bfly / peak64

    for N in (1024, 8192, 16384, 32768):
        logn = N.bit_length() - 1
        tw, pre, itw, ipre = O.tables_u64(N, q) + O.tables_u64(N, q, inverse=True)
        d_tw, d_pre, d_itw, d_ipre = (torch.from_numpy(t.view(np.int64)).cuda() for t in (tw, pre, itw, ipre))
        for chunk_mib in (16, 1024):
            frames = (chunk_mib << 20) // (N * 8)
            rep = min(frames, 64)
            x, y = O.synthetic_u64(N * rep, 7, q), O.synthetic_u64(N * rep, 8, q)
            d_x = torch.from_numpy(np.tile(x, frames // rep).view(np.int64)).cuda()
            d_y = torch.from_numpy(np.tile(y, frames // rep).view(np.int64)).cuda()
            d_spec, d_inv, d_c, d_c2, d_yhat = (torch.empty_like(d_x) for _ in range(5))
            iters = 20 if chunk_mib == 16 else 4

            def fwd():
                p.fwd_dev(N, d_x, d_x, d_spec, q, d_tw, d_pre, frames)

            def inv():
                p.inv_dev(N, d_spec, d_inv, q, d_itw, d_ipre, frames)

            def mul():
                p.polymul_dev(N, d_c, d_x, d_y, q, d_tw, d_pre, d_itw, d_ipre, frames)

            def mulspec():
                p.polymul_by_spectrum_dev(N, d_c2, d_x, d_yhat, q, d_tw, d_pre, d_itw, d_ipre, frames)

            p.fwd_dev(N, d_y, d_y, d_yhat, q, d_tw, d_pre, frames)
            launches = {}
            for name, fn in (("fwd", fwd), ("inv", inv), ("polymul", mul), ("polymul_by_spectrum", mulspec)):
                l0 = p.launch_count()
                fn()
                launches[name] = p.launch_count() - l0
            torch.cuda.synchronize()
            # parity on the first two frames: forward vs the C restatement, inverse vs the oracle (and == x), products vs
            # the oracle's INTT(NTT(x) .* NTT(y)), by-spectrum == polymul
            spec = u64(d_spec[: 2 * N])
            ok_fwd = (spec == O.ref_fwd_u64(x[: 2 * N], x[: 2 * N], q, tw, pre, 2)).all()
            want_inv = spec.copy()
            orc.orc_inv_u64(N, want_inv.ctypes.data_as(_u64p), q, itw.ctypes.data_as(_u64p), 2, 1)
            ok_inv = (u64(d_inv[: 2 * N]) == want_inv).all() and (want_inv == x[: 2 * N]).all()
            yspec = O.ref_fwd_u64(y[: 2 * N], y[: 2 * N], q, tw, pre, 2)
            prod = np.array([int(a) * int(b) % q for a, b in zip(spec, yspec)], dtype=np.uint64)
            orc.orc_inv_u64(N, prod.ctypes.data_as(_u64p), q, itw.ctypes.data_as(_u64p), 2, 1)
            ok_mul = (u64(d_c[: 2 * N]) == prod).all() and (u64(d_c2[: 2 * N]) == prod).all()

            ms_f, ms_i = timed_pair(fwd, inv, iters)
            ms_m, ms_s = timed_pair(mul, mulspec, iters)
            nb = (N // 2) * logn
            fps_f, frac_f = rates(N, frames, ms_f, nb)
            fps_i, frac_i = rates(N, frames, ms_i, nb + N // 2)
            pps_m, frac_m = rates(N, frames, ms_m, 3 * nb + N // 2 + N)          # 2 forwards, pointwise, inverse
            pps_s, frac_s = rates(N, frames, ms_s, 2 * nb + N // 2 + N)
            line = {"N": N, "chunk_MiB": chunk_mib, "frames": frames, "launches": launches,
                    "fwd_ms": ms_f, "fwd_frames_per_s": fps_f, "inv_ms": ms_i, "inv_frames_per_s": fps_i,
                    "inv_over_fwd_time": ms_i / ms_f,
                    "fwd_frac_of_measured_hbm_copy": fps_f * 2 * N * 8 / 1e9 / copy_gbs,
                    "inv_frac_of_measured_hbm_copy": fps_i * 2 * N * 8 / 1e9 / copy_gbs,
                    "fwd_frac_of_measured_u64_bfly_peak": frac_f, "inv_frac_of_measured_u64_bfly_peak": frac_i,
                    "polymul_ms": ms_m, "polymul_products_per_s": pps_m, "polymul_frac_of_measured_u64_bfly_peak": frac_m,
                    "by_spectrum_ms": ms_s, "by_spectrum_products_per_s": pps_s,
                    "by_spectrum_frac_of_measured_u64_bfly_peak": frac_s,
                    "parity": "ok" if (ok_fwd and ok_inv and ok_mul) else
                    "FAILED fwd=%s inv=%s products=%s" % (ok_fwd, ok_inv, ok_mul)}
            print(json.dumps(line), flush=True)
            del d_x, d_y, d_spec, d_inv, d_c, d_c2, d_yhat
            torch.cuda.empty_cache()
    p.close()
    ctx.close()
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
