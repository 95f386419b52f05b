"""Hoisted rotations in one call (Context64.rotate, agx_rotate64) against the plain recipe of public calls (for each
element: automorph of (c0, c1), keyswitch of sigma(c1) with its key, add sigma(c0)), in the same process.

Workloads, 60-bit primes (q = 1 mod 2^16):
- batch: N = 16384 and 32768, (l + 1, alpha, k) = (12, 4, 4) (dnum = 3), G = 1, 8 and 16, B chosen so that one
  ciphertext component is 256 MiB (far above the 126 MB of L2; the G * 2 outputs are then G * 512 MiB);
- one digit: N = 16384, (12, 12, 4), G = 8, where the hoisted composition of public calls also applies (modup of c1
  once, one automorph call over all G elements for the extended digit and one for c0, per element two element-wise
  products with keys replicated over the batch, two moddowns and an add);
- bootstrapping: B = 1, N = 32768, (24, 8, 8), G = 16: small and launch-bound.

Each line first checks both forms of the call against the plain recipe on the same input, bit for bit (and the hoisted
composition, where it applies, in evaluation form), then times the evaluation forms, alternated in 5 windows with CUDA
events, beside a device-to-device copy of the ciphertexts.  The inner kernel's time comes from a separate torch.profiler
run (CUDA activities), by kernel name, against the copy rate over its byte model: dnum * B * L words of extended digits
and B * (l + 1) of c0 read once (the G re-reads served from L2), the keys (2 * G * dnum * L words) once per slice of the
batch, and 2 * G * B * L words written, per coefficient.  The header line carries the GPU name and power limit read in
the same run.
Usage (GPU box): python profiles/bench_u64_rotate.py [--out profiles/r09_u64_rotate.jsonl]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import torch
import agilex_ntt_b200 as A
from bench_u64_keyswitch import digits_of, primes60, timed


def make_plain(c, cq, ct, gs, rks, alpha, k):
    B, ell1, N = ct.shape[1], ct.shape[2], ct.shape[3]
    r = torch.empty((2, B, ell1, N), dtype=torch.int64, device="cuda")

    def run(out, form):
        for t, g in enumerate(gs):
            cq.automorph(r.view(2 * B, ell1, N), ct.view(2 * B, ell1, N), g, ntt_form=form)
            c.keyswitch(out[t], r[1], rks[t], alpha, k, ntt_form=form)
            cq.elementwise("add", out[t, 0], out[t, 0], r[0])
    return run


def make_hoisted(c, cq, ct, gs, rks, k):
    """One digit, evaluation form: modup of c1 once, automorph of the extended digit and of c0 for all G, then per
    element two products with the replicated key rows (built outside the timing), two moddowns and the add of sigma(c0)."""
    L, N, B, G = c.L, c.n, ct.shape[1], len(gs)
    ell1 = L - k
    D = torch.empty((B, L, N), dtype=torch.int64, device="cuda")
    rot = torch.empty((G, B, L, N), dtype=torch.int64, device="cuda")
    rot0 = torch.empty((G, B, ell1, N), dtype=torch.int64, device="cuda")
    prod = [torch.empty((B, L, N), dtype=torch.int64, device="cuda") for _ in (0, 1)]
    reps = [[torch.cat([rk[0, cc, :ell1], rk[0, cc, rk.shape[2] - k:]]).expand(B, L, N).contiguous() for cc in (0, 1)]
            for rk in rks]

    def run(out):
        c.modup(D, ct[1], 0, ell1, ntt_form=True)
        c.automorph(rot, D, gs, ntt_form=True)
        cq.automorph(rot0, ct[0], gs, ntt_form=True)
        for t in range(G):
            for cc in (0, 1):
                c.elementwise("mul", prod[cc], rot[t], reps[t][cc])
                c.moddown(out[t, cc], prod[cc], k, ntt_form=True)
            cq.elementwise("add", out[t, 0], out[t, 0], rot0[t])
    return run


def inner_kernel_ms(fn, reps=3):
    """mean device time of the rotations' inner-product kernel over `reps` calls, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for e in prof.key_averages():
        if "rotate64_inner_kernel" in e.key:
            us += e.device_time * e.count
            n += e.count
    return (us / n) / 1e3 if n else None, n


def slices(B, G, L, N, sms):
    """agx_rotate64's slices of the batch (ks_slice): each reads every key once"""
    per_slice, want = G * L * N // 2, sms * 1024
    S = min(B, max(1, -(-want // per_slice)))
    slice_ = -(-B // S)
    return -(-B // slice_)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_u64_rotate.jsonl"))
    ap.add_argument("--mib", type=float, default=256.0, help="MiB of one ciphertext component (batch workloads)")
    args = ap.parse_args()
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    allp = primes60(40)
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power, "sms": sms, "bits": 60,
              "component_MiB": args.mib}]
    print(json.dumps(lines[0]), flush=True)
    # (workload, N, l + 1, alpha, k, G, B or None for the batch size)
    cases = [("batch", N, 12, 4, 4, G, None) for N in (16384, 32768) for G in (1, 8, 16)]
    cases += [("one_digit", 16384, 12, 12, 4, 8, None), ("bootstrapping", 32768, 24, 8, 8, 16, 1)]
    for name, N, ell1, alpha, k, G, B in cases:
        primes = allp[:ell1] + allp[ell1:ell1 + k]
        L = len(primes)
        dnum = len(digits_of(ell1, alpha))
        B = B or int(args.mib * (1 << 20)) // (ell1 * N * 8)
        c, cq = A.Context64(N, primes), A.Context64(N, primes[:ell1])
        gen = torch.Generator(device="cuda").manual_seed(N + ell1 + G)
        qv = torch.tensor(primes[:ell1], dtype=torch.int64, device="cuda").view(1, 1, ell1, 1)
        kq = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, 1, L, 1)
        ct = torch.randint(0, 1 << 62, (2, B, ell1, N), dtype=torch.int64, device="cuda", generator=gen) % qv
        gs = [A.galois_element(N, r) for r in range(1, G)] + [2 * N - 1] if G > 1 else [A.galois_element(N, 1)]
        rks = [torch.randint(0, 1 << 62, (dnum, 2, L, N), dtype=torch.int64, device="cuda", generator=gen) % kq
               for _ in gs]
        out = torch.empty((G, 2, B, ell1, N), dtype=torch.int64, device="cuda")
        want = torch.empty_like(out)
        plain = make_plain(c, cq, ct, gs, rks, alpha, k)
        hoisted = make_hoisted(c, cq, ct, gs, rks, k) if dnum == 1 else None
        same = {}
        for form in (False, True):
            c.rotate(out, ct, gs, rks, alpha, k, ntt_form=form)
            plain(want, form)
            torch.cuda.synchronize()
            same["eval" if form else "coeff"] = bool(torch.equal(out, want))
        if hoisted:
            hoisted(want)
            torch.cuda.synchronize()
            same["hoisted_eval"] = bool(torch.equal(out, want))
        fns = {"call_eval": lambda: c.rotate(out, ct, gs, rks, alpha, k, ntt_form=True),
               "call_coeff": lambda: c.rotate(out, ct, gs, rks, alpha, k, ntt_form=False),
               "plain_eval": lambda: plain(want, True)}
        if hoisted:
            fns["hoisted_eval"] = lambda: hoisted(want)
        launches = {}
        for key, fn in fns.items():
            l0, l1 = c.launch_count(), cq.launch_count()
            fn()
            torch.cuda.synchronize()
            launches[key] = c.launch_count() - l0 + cq.launch_count() - l1
        copy_dst = torch.empty_like(ct)
        timed_fns = [fns["call_eval"], fns["plain_eval"]] + ([fns["hoisted_eval"]] if hoisted else [])
        res = timed(timed_fns + [lambda: copy_dst.copy_(ct)], 20 if B == 1 else 2)
        call, pl, cp = res[0], res[1], res[-1]
        copy_GBps = 2 * ct.numel() * 8 / (cp[0] * 1e-3) / 1e9
        inner_ms, inner_n = inner_kernel_ms(fns["call_eval"])
        S = slices(B, G, L, N, sms)
        inner_bytes = (dnum * B * L + B * ell1 + 2 * G * dnum * L * S + 2 * G * B * L) * N * 8
        line = {"workload": name, "N": N, "l+1": ell1, "alpha": alpha, "k": k, "L": L, "dnum": dnum, "G": G, "B": B,
                "component_bytes": ct[0].numel() * 8, "same_output": same, "launches": launches,
                "call_ms": call[0], "call_spread_ms": call[1:], "plain_ms": pl[0], "plain_spread_ms": pl[1:],
                "call_over_plain_time": call[0] / pl[0], "copy_ms": cp[0], "copy_GBps": copy_GBps,
                "inner_ms": inner_ms, "inner_launches_profiled": inner_n, "inner_bytes": inner_bytes, "slices": S,
                "inner_GBps": inner_bytes / (inner_ms * 1e-3) / 1e9 if inner_ms else None,
                "inner_share_of_time": inner_ms / call[0] if inner_ms else None}
        if hoisted:
            line.update(hoisted_ms=res[2][0], hoisted_spread_ms=res[2][1:], call_over_hoisted_time=call[0] / res[2][0])
        if inner_ms:
            line["inner_over_copy_rate"] = line["inner_GBps"] / copy_GBps
        print(json.dumps(line), flush=True)
        lines.append(line)
        del ct, rks, out, want, plain, hoisted, copy_dst
        c.close()
        cq.close()
        torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
