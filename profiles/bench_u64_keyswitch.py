"""Hybrid key switching in one call (Context64.keyswitch, agx_keyswitch64) against the same key switch composed from
public calls with the key rows sliced and replicated over the batch, in the same process.

Workloads: N = 16384 and 32768, 60-bit primes (q = 1 mod 2^16); (l + 1, alpha, k) = (12, 4, 4), (12, 12, 12) and
(24, 8, 8), i.e. dnum = 3, 1 and 3; and one line with a top-level key over 16 + 4 primes (key_limbs = 20) used at
l + 1 = 8 (alpha = 4, k = 4).  B is chosen so that the input is about 1 GiB, far above the 126 MB of L2.

Each line first checks both forms of the call against the composed recipe on the same input, bit for bit, then times
the evaluation forms of both, alternated in 5 windows with CUDA events, beside the device-to-device copy rate of the
input measured in the same run.  The inner-product kernel's time comes from a separate torch.profiler run (CUDA
activities), by kernel name, and is set against the copy rate over its bytes: dnum * B * L * n words of extended digits
read, 2 * B * L * n written, and the key (dnum * 2 * L * n words) read once.  The recipe's inner phase (dnum element-wise
mul / mac pairs over replicated keys) moves (8 * dnum - 2) * B * L * n words.  The header line carries the GPU name and
power limit read in the same run.
Usage (GPU box): python profiles/bench_u64_keyswitch.py [--out profiles/r08_u64_keyswitch.jsonl]"""
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


def digits_of(ell1, alpha):
    m = min(alpha, ell1)
    return [(f, min(m, ell1 - f)) for f in range(0, ell1, m)]


def make_recipe(c, x, ksk, alpha, k):
    """The composed key switch over prepared buffers: the replicated key rows are built once, outside the timing (a
    caller of the recipe keeps its keys that way); each call cuts its digits out, extends them, and accumulates."""
    L, N, B = c.L, c.n, x.shape[0]
    ell1 = L - k
    kr = torch.cat([ksk[:, :, :ell1], ksk[:, :, ksk.shape[2] - k:]], dim=2)
    digits = digits_of(ell1, alpha)
    reps = [[kr[j, cc].expand(B, L, N).contiguous() for cc in (0, 1)] for j in range(len(digits))]
    U = torch.empty((B, L, N), dtype=torch.int64, device="cuda")
    tmp = torch.empty((B, L, N), dtype=torch.int64, device="cuda")
    acc = [torch.empty((B, L, N), dtype=torch.int64, device="cuda") for _ in (0, 1)]
    cut = {cnt: torch.empty((B, cnt, N), dtype=torch.int64, device="cuda") for _, cnt in digits}

    def run(out, form):
        for j, (f, cnt) in enumerate(digits):
            src = x
            if len(digits) > 1:
                cut[cnt].copy_(x[:, f:f + cnt])
                src = cut[cnt]
            c.modup(U, src, f, cnt, ntt_form=form)
            for cc in (0, 1):
                if form:
                    c.elementwise("mul" if j == 0 else "mac", acc[cc], U, reps[j][cc])
                elif j == 0:
                    c.polymul_by_spectrum(acc[cc], U, reps[j][cc])
                else:
                    c.polymul_by_spectrum(tmp, U, reps[j][cc])
                    c.elementwise("add", acc[cc], acc[cc], tmp)
        for cc in (0, 1):
            c.moddown(out[cc], acc[cc], k, ntt_form=form)
    return run


def inner_kernel_ms(fn, reps=3):
    """mean device time of the inner-product kernel over `reps` calls, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for e in prof.key_averages():
        if "keyswitch64_inner_kernel" in e.key:
            us += e.device_time * e.count
            n += e.count
    return (us / n) / 1e3 if n else None, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_u64_keyswitch.jsonl"))
    ap.add_argument("--gib", type=float, default=1.0)
    args = ap.parse_args()
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    allp = primes60(40)
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "bits": 60, "data_GiB": args.gib}]
    print(json.dumps(lines[0]), flush=True)
    # (N, l + 1, alpha, k, primes of the key's Q_top)
    cases = [(N, e, a, k, e) for N in (16384, 32768) for e, a, k in ((12, 4, 4), (12, 12, 12), (24, 8, 8))]
    cases.append((16384, 8, 4, 4, 16))
    for N, ell1, alpha, k, top in cases:
        qtop, ps = allp[:top], allp[top:top + k]
        primes = qtop[:ell1] + ps
        L = len(primes)
        key_primes = qtop + ps
        dnum = len(digits_of(ell1, alpha))
        B = int(args.gib * (1 << 30)) // (ell1 * N * 8)
        c = A.Context64(N, primes)
        gen = torch.Generator(device="cuda").manual_seed(N + ell1)
        qv = torch.tensor(primes[:ell1], dtype=torch.int64, device="cuda").view(1, ell1, 1)
        kq = torch.tensor(key_primes, dtype=torch.int64, device="cuda").view(1, 1, len(key_primes), 1)
        x = torch.randint(0, 1 << 62, (B, ell1, N), dtype=torch.int64, device="cuda", generator=gen) % qv
        ksk = torch.randint(0, 1 << 62, (dnum, 2, len(key_primes), N), dtype=torch.int64, device="cuda",
                            generator=gen) % kq
        out = torch.empty((2, B, ell1, N), dtype=torch.int64, device="cuda")
        want = torch.empty_like(out)
        recipe = make_recipe(c, x, ksk, alpha, k)
        same = {}
        for form in (False, True):
            c.keyswitch(out, x, ksk, alpha, k, ntt_form=form)
            recipe(want, form)
            torch.cuda.synchronize()
            same["eval" if form else "coeff"] = bool(torch.equal(out, want))
        launches = {}
        for name, fn in (("call_eval", lambda: c.keyswitch(out, x, ksk, alpha, k, ntt_form=True)),
                         ("call_coeff", lambda: c.keyswitch(out, x, ksk, alpha, k, ntt_form=False)),
                         ("recipe_eval", lambda: recipe(want, True))):
            l0 = c.launch_count()
            fn()
            torch.cuda.synchronize()
            launches[name] = c.launch_count() - l0
        copy_dst = torch.empty_like(x)
        res = timed([lambda: c.keyswitch(out, x, ksk, alpha, k, ntt_form=True), lambda: recipe(want, True),
                     lambda: copy_dst.copy_(x)], 2)
        call, rec, cp = res
        copy_GBps = 2 * x.numel() * 8 / (cp[0] * 1e-3) / 1e9
        inner_ms, inner_n = inner_kernel_ms(lambda: c.keyswitch(out, x, ksk, alpha, k, ntt_form=True))
        inner_bytes = (dnum * B * L + 2 * B * L + dnum * 2 * L) * N * 8
        line = {"N": N, "l+1": ell1, "alpha": alpha, "k": k, "L": L, "dnum": dnum, "key_limbs": len(key_primes),
                "B": B, "input_bytes": x.numel() * 8, "same_output": same, "launches": launches,
                "call_ms": call[0], "call_spread_ms": call[1:], "recipe_ms": rec[0], "recipe_spread_ms": rec[1:],
                "call_over_recipe_time": call[0] / rec[0], "copy_ms": cp[0], "copy_GBps": copy_GBps,
                "inner_ms": inner_ms, "inner_launches_profiled": inner_n, "inner_bytes": inner_bytes,
                "inner_GBps": inner_bytes / (inner_ms * 1e-3) / 1e9 if inner_ms else None,
                "inner_share_of_time": inner_ms / call[0] if inner_ms else None,
                "inner_words_per_coeff_model": f"{dnum}L + 2L (+ key {2 * dnum}L/B)",
                "recipe_inner_words_per_coeff_model": f"{8 * dnum - 2}L"}
        if inner_ms:
            line["inner_over_copy_rate"] = line["inner_GBps"] / copy_GBps
        print(json.dumps(line), flush=True)
        lines.append(line)
        del x, ksk, out, want, recipe, copy_dst
        c.close()
        torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
