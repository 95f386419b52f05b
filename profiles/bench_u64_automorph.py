"""Galois automorphisms (Context64.automorph, agx_automorph64) in both forms, beside the HBM copy rate, in the same process.

Both forms are one streaming pass: a call with G elements reads the B*L*n input words once and writes G*B*L*n.  The
yardstick is the device-to-device copy rate of the same input measured here, applied to the call's (1 + G)*B*L*n*8
bytes.  G = 8 (rotations by 1, -1, 2, -2, 4, -4, 8 and the conjugation, as a hoisted key switch issues them) is also timed
against 8 calls with one element each over the same outputs; the byte model predicts (1 + 8) / 16 of their time.

Workload: 1 GiB of input, L = 8 primes of 60 bits (q = 1 mod 2^16), N = 8192, 16384 and 32768.  The timed calls are
alternated in windows timed with CUDA events after a warm-up; 1 GiB is well above the 126 MB of L2, so every call streams
from HBM.  Each line first checks that the evaluation form equals fwd(sigma(inv(x))) composed from the public calls on
the same input, and counts each form's launches; the header line carries the GPU name and power limit read in the same
run.  Usage (GPU box): python profiles/bench_u64_automorph.py [--out profiles/r07_u64_automorph.jsonl]"""
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_u64_automorph.jsonl"))
    ap.add_argument("--gib", type=float, default=1.0)
    args = ap.parse_args()
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    L = 8
    primes = primes60(L)
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "primes": primes,
              "data_GiB": args.gib}]
    print(json.dumps(lines[0]), flush=True)
    qs = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, L, 1)
    for N in (8192, 16384, 32768):
        B = int(args.gib * (1 << 30)) // (L * N * 8)
        c = A.Context64(N, primes)
        gen = torch.Generator(device="cuda").manual_seed(N)
        x = torch.randint(0, 1 << 62, (B, L, N), dtype=torch.int64, device="cuda", generator=gen) % qs
        copy_dst = torch.empty_like(x)
        eight = [A.galois_element(N, r) for r in (1, -1, 2, -2, 4, -4, 8)] + [2 * N - 1]
        for gs in ([A.galois_element(N, 1)], eight):
            G = len(gs)
            out = torch.empty((G, B, L, N), dtype=torch.int64, device="cuda")

            # same words: automorph(eval)(x) = fwd(automorph(coeff)(inv(x)))
            c.automorph(out, x, gs, ntt_form=True)
            t = x.clone()
            c.inv(t)
            want = torch.empty_like(out)
            c.automorph(want, t, gs, ntt_form=False)
            c.fwd(want)
            torch.cuda.synchronize()
            same = bool(torch.equal(out, want))
            del t, want
            torch.cuda.empty_cache()

            launches = {}
            for form in (False, True):
                l0 = c.launch_count()
                c.automorph(out, x, gs, ntt_form=form)
                torch.cuda.synchronize()
                launches["eval" if form else "coeff"] = c.launch_count() - l0

            def singles(form):
                def run():
                    for k, g in enumerate(gs):
                        c.automorph(out[k], x, g, ntt_form=form)
                return run

            fns = [lambda: c.automorph(out, x, gs, ntt_form=False), lambda: c.automorph(out, x, gs, ntt_form=True),
                   lambda: copy_dst.copy_(x)]
            if G > 1:
                fns += [singles(False), singles(True)]
            res = timed(fns, 3)
            coeff, ev, cp = res[:3]
            nbytes = (1 + G) * B * L * N * 8
            copy_GBps = 2 * x.numel() * 8 / (cp[0] * 1e-3) / 1e9
            line = {"L": L, "N": N, "B": B, "G": G, "galois": gs, "same_output": same, "launches": launches,
                    "bytes": nbytes, "copy_ms": cp[0], "copy_GBps": copy_GBps}
            for name, r in (("coeff", coeff), ("eval", ev)):
                GBps = nbytes / (r[0] * 1e-3) / 1e9
                line.update({f"{name}_ms": r[0], f"{name}_spread_ms": r[1:], f"{name}_GBps": GBps,
                             f"{name}_over_copy_rate": GBps / copy_GBps})
            if G > 1:
                for name, r, one in (("coeff", res[3], coeff), ("eval", res[4], ev)):
                    line.update({f"{name}_singles_ms": r[0], f"{name}_singles_spread_ms": r[1:],
                                 f"{name}_hoisted_over_singles_time": one[0] / r[0]})
                line["predicted_hoisted_over_singles_time"] = (1 + G) / (2 * G)
            print(json.dumps(line), flush=True)
            lines.append(line)
            del out
            torch.cuda.empty_cache()
        c.close()
        del x, copy_dst
        torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
