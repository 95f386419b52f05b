"""Batched u64 RNS transforms (Context64: agx_ntt64_fwd, agx_ntt64_inv, agx_polymul64_by_spectrum) against what a caller
does without them: a loop of L single-modulus calls (agx_ref_fwd_dev, agx_ref_inv_dev, agx_ref_polymul_by_spectrum_dev),
in place, over the same bytes held limb-major ([L][B][N] instead of [B][L][N]).

Workload: 1 GiB of data, L = 4 primes of 60 bits (q = 1 mod 2^16), N = 8192, 16384 and 32768, everything in place.  Both
forms run in the same process, alternated in windows timed with CUDA events after a warm-up; 1 GiB is well above the
126 MB of L2, so every call streams from HBM.  Each line first checks that both forms give the same words from the same
input (forward, inverse and by-spectrum product), and the header line carries the GPU name and power limit read in the
same run.  Usage (GPU box): python profiles/bench_u64_rns.py [--out profiles/r04_u64_rns.jsonl]"""
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

L = 4


def primes60(count):
    out, q = [], (1 << 60) - (1 << 16) + 1
    while len(out) < count:
        if O.is_prime(q):
            out.append(q)
        q -= 1 << 16
    return out


def timed_pair(f, g, iters, rounds=5):
    """ms per call of f and of g, alternated: `rounds` windows of `iters` calls each, after a warm-up of both."""
    for _ in range(2):
        f(); g()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tf, tg = [], []
    for _ in range(rounds):
        ev[0].record()
        for _ in range(iters):
            f()
        ev[1].record()
        for _ in range(iters):
            g()
        ev[2].record()
        torch.cuda.synchronize()
        tf.append(ev[0].elapsed_time(ev[1]) / iters)
        tg.append(ev[1].elapsed_time(ev[2]) / iters)
    return float(np.median(tf)), float(np.median(tg)), (min(tf), max(tf)), (min(tg), max(tg))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_u64_rns.jsonl"))
    ap.add_argument("--gib", type=float, default=1.0)
    args = ap.parse_args()
    primes = primes60(L)
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "primes": primes, "L": L,
              "data_GiB": args.gib, "in_place": True}]
    print(json.dumps(lines[0]), flush=True)
    P = A.RefPipeline()
    qs = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, L, 1)
    for N in (8192, 16384, 32768):
        B = int(args.gib * (1 << 30)) // (L * N * 8)
        ctx = A.Context64(N, primes)
        tabs = [[torch.from_numpy(t.view(np.int64)).cuda() for t in ctx.tables(l) + ctx.tables(l, True)] for l in range(L)]
        g = torch.Generator(device="cuda").manual_seed(N)
        x = torch.randint(0, 1 << 62, (B, L, N), dtype=torch.int64, device="cuda", generator=g) % qs
        y = torch.randint(0, 1 << 62, (B, L, N), dtype=torch.int64, device="cuda", generator=g) % qs
        x_lm = x.permute(1, 0, 2).contiguous()               # the same words, limb-major: [L][B][N]
        y_hat = y.clone()
        ctx.fwd(y_hat)
        y_hat_lm = y_hat.permute(1, 0, 2).contiguous()
        del y

        def loop(fn):
            def run():
                for l in range(L):
                    fn(l, x_lm[l])
            return run

        rns = {"fwd": lambda: ctx.fwd(x), "inv": lambda: ctx.inv(x),
               "by_spectrum": lambda: ctx.polymul_by_spectrum(x, x, y_hat)}
        per_limb = {
            "fwd": loop(lambda l, s: P.fwd_dev(N, s, s, s, primes[l], tabs[l][0], tabs[l][1], B)),
            "inv": loop(lambda l, s: P.inv_dev(N, s, s, primes[l], tabs[l][2], tabs[l][3], B)),
            "by_spectrum": loop(lambda l, s: P.polymul_by_spectrum_dev(N, s, s, y_hat_lm[l], primes[l], *tabs[l], B)),
        }
        same = {}
        for op in ("fwd", "inv", "by_spectrum"):             # one call of each form on the same words, then compare
            rns[op]()
            per_limb[op]()
            torch.cuda.synchronize()
            same[op] = bool(torch.equal(x.permute(1, 0, 2), x_lm))
        launches = {}
        for op in rns:
            l0 = ctx.launch_count()
            rns[op]()
            torch.cuda.synchronize()
            launches[op] = ctx.launch_count() - l0
        line = {"N": N, "B": B, "frames": B * L, "same_output": same, "rns_launches": launches}
        for op in ("fwd", "inv", "by_spectrum"):
            ms_r, ms_l, spread_r, spread_l = timed_pair(rns[op], per_limb[op], 3)
            line[op] = {"rns_ms": ms_r, "per_limb_loop_ms": ms_l, "rns_spread_ms": spread_r,
                        "per_limb_spread_ms": spread_l, "rns_frames_per_s": B * L / (ms_r * 1e-3),
                        "per_limb_frames_per_s": B * L / (ms_l * 1e-3), "rns_over_loop_time": ms_r / ms_l}
        print(json.dumps(line), flush=True)
        lines.append(line)
        ctx.close()
        del x, x_lm, y_hat, y_hat_lm, tabs
        torch.cuda.empty_cache()
    P.close()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
