"""RNS rescale (Context64.rescale, agx_rescale64) in both forms, beside what bounds each of them, in the same process.

- Coefficient form: one pass that reads B*L*n words and writes B*(L-1)*n.  Its yardstick is the HBM copy rate measured
  here (a device-to-device copy of the same input), applied to its (2L - 1)*n*8*B bytes.
- Evaluation form: the inverse of the last limb into a scratch row, then a forward of every other limb with the rescale
  fused into its load and its store.  Its yardstick is the transform work it cannot avoid, timed with the existing calls:
  agx_ntt64_inv over B frames on a 1-limb context of q_{L-1}, plus agx_ntt64_fwd over B*(L-1) frames on the context of
  the first L - 1 primes.

Workload: 1 GiB of input, L = 4 and 8 primes of 60 bits (q = 1 mod 2^16), N = 8192, 16384 and 32768.  The timed calls are
alternated in windows timed with CUDA events after a warm-up; 1 GiB is well above the 126 MB of L2, so every call streams
from HBM.  Each line first checks that the evaluation form equals the existing calls composed around the coefficient
form on the same input; the header line carries the GPU name and power limit read in the same run.
Usage (GPU box): python profiles/bench_u64_rescale.py [--out profiles/r05_u64_rescale.jsonl]"""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_u64_rescale.jsonl"))
    ap.add_argument("--gib", type=float, default=1.0)
    args = ap.parse_args()
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    all_primes = primes60(8)
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "primes": all_primes,
              "data_GiB": args.gib}]
    print(json.dumps(lines[0]), flush=True)
    for L in (4, 8):
        primes = all_primes[:L]
        qs = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, L, 1)
        for N in (8192, 16384, 32768):
            B = int(args.gib * (1 << 30)) // (L * N * 8)
            full, lower, last = A.Context64(N, primes), A.Context64(N, primes[:-1]), A.Context64(N, primes[-1:])
            g = torch.Generator(device="cuda").manual_seed(N + L)
            x = torch.randint(0, 1 << 62, (B, L, N), dtype=torch.int64, device="cuda", generator=g) % qs
            out = torch.empty((B, L - 1, N), dtype=torch.int64, device="cuda")
            inv_buf = x[:, L - 1:, :].contiguous()                     # B frames of q_{L-1}
            fwd_buf = x[:, :L - 1, :].contiguous()                     # B * (L-1) frames of the first L - 1 primes
            copy_dst = torch.empty_like(x)

            # same words: rescale(eval)(x) = fwd_{L-1}(rescale(coeff)(inv_L(x)))
            full.rescale(out, x, ntt_form=True)
            t = x.clone()
            full.inv(t)
            want = torch.empty_like(out)
            full.rescale(want, t, ntt_form=False)
            lower.fwd(want)
            torch.cuda.synchronize()
            same = bool(torch.equal(out, want))
            del t, want
            torch.cuda.empty_cache()

            launches = {}
            for form in (False, True):
                l0 = full.launch_count()
                full.rescale(out, x, ntt_form=form)
                torch.cuda.synchronize()
                launches["eval" if form else "coeff"] = full.launch_count() - l0

            def transforms():
                last.inv(inv_buf)
                lower.fwd(fwd_buf)

            fns = [lambda: full.rescale(out, x, ntt_form=False), lambda: full.rescale(out, x, ntt_form=True),
                   transforms, lambda: copy_dst.copy_(x)]
            (coeff, ev, tr, cp) = timed(fns, 3)
            coeff_bytes = (2 * L - 1) * N * 8 * B
            copy_GBps = 2 * x.numel() * 8 / (cp[0] * 1e-3) / 1e9
            coeff_GBps = coeff_bytes / (coeff[0] * 1e-3) / 1e9
            line = {"L": L, "N": N, "B": B, "same_output": same, "launches": launches,
                    "coeff_ms": coeff[0], "coeff_spread_ms": coeff[1:], "coeff_GBps": coeff_GBps,
                    "copy_ms": cp[0], "copy_GBps": copy_GBps, "coeff_over_copy_rate": coeff_GBps / copy_GBps,
                    "eval_ms": ev[0], "eval_spread_ms": ev[1:], "transforms_ms": tr[0], "transforms_spread_ms": tr[1:],
                    "eval_over_transforms_time": ev[0] / tr[0],
                    "eval_polys_per_s": B / (ev[0] * 1e-3), "coeff_polys_per_s": B / (coeff[0] * 1e-3)}
            print(json.dumps(line), flush=True)
            lines.append(line)
            for c in (full, lower, last):
                c.close()
            del x, out, inv_buf, fwd_buf, copy_dst
            torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
