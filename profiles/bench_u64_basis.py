"""RNS basis conversion (Context64.moddown / modup, agx_moddown64 / agx_modup64) in both forms, beside what bounds each of
them, in the same process.

- Coefficient forms: one pass.  ModDown reads B*L*n words and writes B*(L-k)*n; ModUp reads B*m*n and writes B*L*n.
  Two yardsticks: the HBM copy rate measured here (a device-to-device copy of a [B][L][n] batch) applied to their bytes,
  (2L - k)*n*8 and (m + L)*n*8 per polynomial; and their modular products per coefficient against the u64 butterfly
  rate of agx_measure_butterfly_peak kind 1 (one u64 butterfly is about one Shoup product: an approximation).
  ModDown: k(k-1)/2 for the digits, k per target limb for Horner and its reduction, 1 per target for the finish;
  ModUp: m(m-1)/2 + m per target limb.  `coeff_fraction_of_bound` is the time of the larger bound over the call's time.
- Evaluation forms: compared with the transforms they cannot avoid, timed with the existing calls.  ModDown: the
  inverse over B*k frames (a context over the last k primes) plus the forward over B*(L-k) frames (the first L - k).
  ModUp: the inverse over B*m frames (a context over the source primes) plus the forward over B*(L-m) frames.

Workload: L = 12 primes of 60 bits (q = 1 mod 2^16); ModDown with k = 2 and 4; ModUp of m = 4 source primes at first = 0
and first = 4; N = 8192, 16384, 32768; B such that a [B][L][N] batch is 1 GiB (the ModDown input, the ModUp output),
well above the 126 MB of L2.  The timed calls are alternated in 5 windows timed with CUDA events after a warm-up
(median and spread).  Each line first checks that the evaluation form equals the existing calls composed around the
coefficient form on the same input, and records launch counts; the header line carries the GPU name and power limit
read in the same run.
Usage (GPU box): python profiles/bench_u64_basis.py [--out profiles/r06_u64_basis.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import agilex_ntt_b200 as A
from oracle import oracle as O      # prime search only (this is a measurement script, not the product)


def primes60(count):
    out, q = [], (1 << 60) - (1 << 16) + 1
    while len(out) < count:
        if O.is_prime(q):
            out.append(q)
        q -= 1 << 16
    return out


def timed(fns, iters, rounds=5):
    """ms per call of each fn, alternated: `rounds` windows of `iters` calls of each, after a warm-up of all.
    Returns (median, min, max) per fn."""
    for _ in range(2):
        for f in fns:
            f()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(fns) + 1)]
    t = [[] for _ in fns]
    for _ in range(rounds):
        ev[0].record()
        for k, f in enumerate(fns):
            for _ in range(iters):
                f()
            ev[k + 1].record()
        torch.cuda.synchronize()
        for k in range(len(fns)):
            t[k].append(ev[k].elapsed_time(ev[k + 1]) / iters)
    return [(float(np.median(v)), min(v), max(v)) for v in t]


def launches_of(ctx, fn):
    l0 = ctx.launch_count()
    fn()
    torch.cuda.synchronize()
    return ctx.launch_count() - l0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_u64_basis.jsonl"))
    ap.add_argument("--gib", type=float, default=1.0)
    args = ap.parse_args()
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    L = 12
    primes = primes60(L)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pc = A.Context(1024, [1053818881])
    bfly_per_clk_sm, mhz = pc.measure_butterfly_peak(1, 1024)
    pc.close()
    mul_rate = bfly_per_clk_sm * sms * mhz * 1e6                  # u64 Shoup products per second (approximation)
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power, "sms": sms, "primes": primes, "L": L,
              "data_GiB": args.gib, "u64_butterflies_per_clk_per_sm": bfly_per_clk_sm, "implied_sm_mhz": mhz}]
    print(json.dumps(lines[0]), flush=True)
    qs = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, L, 1)
    configs = [("moddown", 2, None), ("moddown", 4, None), ("modup", 4, 0), ("modup", 4, 4)]
    for N in (8192, 16384, 32768):
        B = int(args.gib * (1 << 30)) // (L * N * 8)
        full = A.Context64(N, primes)
        g = torch.Generator(device="cuda").manual_seed(N)
        x = torch.randint(0, 1 << 62, (B, L, N), dtype=torch.int64, device="cuda", generator=g) % qs
        copy_dst = torch.empty_like(x)
        for op, m, first in configs:
            if op == "moddown":
                src_primes, tgt_primes = primes[-m:], primes[:-m]
                inp = x
                out = torch.empty((B, L - m, N), dtype=torch.int64, device="cuda")
                call = lambda form: full.moddown(out, inp, m, ntt_form=form)
                lower = A.Context64(N, tgt_primes)
                inv_buf = x[:, L - m:, :].contiguous()
                fwd_buf = x[:, :L - m, :].contiguous()
            else:
                src_primes = primes[first:first + m]
                tgt_primes = primes[:first] + primes[first + m:]
                inp = x[:, first:first + m, :].contiguous()
                out = torch.empty_like(x)
                call = lambda form: full.modup(out, inp, first, m, ntt_form=form)
                lower = A.Context64(N, tgt_primes)
                inv_buf = inp.clone()
                fwd_buf = torch.cat([x[:, :first, :], x[:, first + m:, :]], dim=1).contiguous()
            srcctx = A.Context64(N, src_primes)

            # same words: op(eval)(x) = fwd(op(coeff)(inv(x))) through the existing calls
            call(True)
            got = out.clone()
            t = inp.clone()
            (full if op == "moddown" else srcctx).inv(t)
            if op == "moddown":
                full.moddown(out, t, m, ntt_form=False)
                lower.fwd(out)
            else:
                full.modup(out, t, first, m, ntt_form=False)
                full.fwd(out)
            torch.cuda.synchronize()
            same = bool(torch.equal(got, out))
            del t, got
            torch.cuda.empty_cache()
            launches = {"coeff": launches_of(full, lambda: call(False)), "eval": launches_of(full, lambda: call(True))}

            def transforms():
                srcctx.inv(inv_buf)
                lower.fwd(fwd_buf)

            fns = [lambda: call(False), lambda: call(True), transforms, lambda: copy_dst.copy_(x)]
            (coeff, ev, tr, cp) = timed(fns, 3)
            ntgt = L - m
            if op == "moddown":
                words = 2 * L - m
                muls = m * (m - 1) // 2 + ntgt * (m + 1)
            else:
                words = m + L
                muls = m * (m - 1) // 2 + ntgt * m
            coeff_bytes = words * N * 8 * B
            copy_GBps = 2 * x.numel() * 8 / (cp[0] * 1e-3) / 1e9
            coeff_GBps = coeff_bytes / (coeff[0] * 1e-3) / 1e9
            t_hbm = coeff_bytes / (copy_GBps * 1e9)
            t_mul = muls * N * B / mul_rate
            bound = "hbm_copy_rate" if t_hbm >= t_mul else "u64_multiply_rate"
            line = {"op": op, "m": m, "first": first, "L": L, "N": N, "B": B, "same_output": same,
                    "launches": launches, "coeff_ms": coeff[0], "coeff_spread_ms": coeff[1:], "coeff_GBps": coeff_GBps,
                    "copy_ms": cp[0], "copy_GBps": copy_GBps, "coeff_over_copy_rate": coeff_GBps / copy_GBps,
                    "products_per_coeff": muls, "coeff_products_per_s": muls * N * B / (coeff[0] * 1e-3),
                    "coeff_over_multiply_rate": (muls * N * B / (coeff[0] * 1e-3)) / mul_rate,
                    "coeff_bound": bound, "coeff_fraction_of_bound": max(t_hbm, t_mul) * 1e3 / coeff[0],
                    "eval_ms": ev[0], "eval_spread_ms": ev[1:], "transforms_ms": tr[0], "transforms_spread_ms": tr[1:],
                    "eval_over_transforms_time": ev[0] / tr[0], "eval_polys_per_s": B / (ev[0] * 1e-3)}
            print(json.dumps(line), flush=True)
            lines.append(line)
            for c in (lower, srcctx):
                c.close()
            del out, inv_buf, fwd_buf, inp
            torch.cuda.empty_cache()
        full.close()
        del x, copy_dst
        torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
