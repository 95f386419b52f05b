"""Ciphertext multiplication in one call (Context64.mulrelin, agx_mulrelin64) against today's route: the tensor from
four element-wise products over Q_l, agx_keyswitch64 of D_2 with the relinearisation key, two element-wise adds, and in
the rescale line agx_rescale64 of both components.  Same process, alternated timed windows.

Workloads, 60-bit primes (q = 1 mod 2^16):
- batch: N = 16384, (l + 1, alpha, k) = (12, 4, 4), B chosen so that one ciphertext component is 256 MiB (far above
  the 126 MB of L2);
- deep: B = 1, N = 32768, (24, 8, 8).

Each workload first checks both forms of the call, with and without rescale, bit for bit against the recipe composed
from public calls (the tensor, modup of each digit of D_2, element-wise products with the key rows and the sum plus
(P mod q_i) D_c over Q_l u P, one moddown of 2 B by k or k + 1 primes; not timed), and against today's route.  Then it
times the evaluation forms of the call and of the route, alternated in 5 windows with CUDA events, beside a
device-to-device copy of one ciphertext batch.  Launches are counted per call, and the inner kernel's time comes from a
separate torch.profiler run (CUDA activities), by kernel name.

Byte model, in words of n per polynomial (x 8 B N per workload), every launch's reads and writes counted once (re-reads
of the same rows by other CTAs assumed to hit L2): an element-wise MUL 3 (l + 1), MAC 4 (l + 1), ADD 3 (l + 1); the
evaluation-form ModUp of a digit of c primes 2c (the gather, with dnum > 1) + 2c (the source spectra copied) + 2c (the
inverse) + 2c (the digits, c >= 2) + c + (L - c) (the fused forward); the key inner product dnum L read + 2 L written,
the call's also 4 (l + 1) of the inputs read; a ModDown over kd primes, per polynomial, 2 kd + 2 kd + kd + 2 (L - kd)
(inverse, digits, fused forward reading and writing the L - kd others; no digits kernel for kd = 1); agx_rescale64 is
that with kd = 1 over the l + 1 limbs.  The model's time ratio call / route is its bytes' ratio."""
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


def empty(*shape):
    return torch.empty(shape, dtype=torch.int64, device="cuda")


def moddown_words(L, kd):
    return 2 * kd + (2 * kd if kd >= 2 else 0) + kd + 2 * (L - kd)


def model_words(ell1, alpha, k):
    """(call, route) words per B N for rescale False and True (module docstring)"""
    L = ell1 + k
    digits = digits_of(ell1, alpha)
    dnum = len(digits)
    modup = sum((2 * c if dnum > 1 else 0) + 2 * c + 2 * c + (2 * c if c >= 2 else 0) + c + (L - c) for _, c in digits)
    call = 3 * ell1 + modup + dnum * L + 4 * ell1 + 2 * L
    route = 13 * ell1 + modup + dnum * L + 2 * L + 2 * moddown_words(L, k) + 6 * ell1
    return {False: (call + 2 * moddown_words(L, k), route),
            True: (call + 2 * moddown_words(L, k + 1), route + 2 * moddown_words(ell1, 1))}


def inner_words(ell1, alpha, k):
    L = ell1 + k
    return len(digits_of(ell1, alpha)) * L + 4 * ell1 + 2 * L


def make_route(c, cq, a, b, rlk, alpha, k, rescale):
    """today's route in evaluation form: tensor, keyswitch of D_2, two adds, and rescale of both components"""
    B, ell1, N = a.shape[1], a.shape[2], a.shape[3]
    D = empty(3, B, ell1, N)
    ks = empty(2, B, ell1, N)

    def run(out):
        cq.elementwise("mul", D[0], a[0], b[0])
        cq.elementwise("mul", D[1], a[0], b[1])
        cq.elementwise("mac", D[1], a[1], b[0])
        cq.elementwise("mul", D[2], a[1], b[1])
        c.keyswitch(ks, D[2], rlk, alpha, k, ntt_form=True)
        dst = ks if rescale else out
        for cc in (0, 1):
            cq.elementwise("add", dst[cc], ks[cc], D[cc])
        if rescale:
            cq.rescale(out.view(2 * B, ell1 - 1, N), ks.view(2 * B, ell1, N), ntt_form=True)
    return run


def recipe(c, cq, a, b, rlk, alpha, k, rescale):
    """the definition from public calls in evaluation form, ending in one moddown of 2 B by k or k + 1 primes"""
    L, N, B = c.L, c.n, a.shape[1]
    ell1 = L - k
    D = empty(3, B, ell1, N)
    cq.elementwise("mul", D[0], a[0], b[0])
    cq.elementwise("mul", D[1], a[0], b[1])
    cq.elementwise("mac", D[1], a[1], b[0])
    cq.elementwise("mul", D[2], a[1], b[1])
    kr = torch.cat([rlk[:, :, :ell1], rlk[:, :, rlk.shape[2] - k:]], dim=2)
    P = 1
    for q in c.primes[ell1:]:
        P *= q
    pm = torch.tensor([P % q if i < ell1 else 0 for i, q in enumerate(c.primes)], dtype=torch.int64,
                      device="cuda").view(1, L, 1).expand(B, L, N).contiguous()
    acc = empty(2, B, L, N)
    U = empty(B, L, N)
    for j, (f, cnt) in enumerate(digits_of(ell1, alpha)):
        c.modup(U, D[2, :, f:f + cnt].contiguous(), f, cnt, ntt_form=True)
        for cc in (0, 1):
            c.elementwise("mul" if j == 0 else "mac", acc[cc], U, kr[j, cc].expand(B, L, N).contiguous())
    del U
    for cc in (0, 1):
        padded = torch.cat([D[cc], torch.zeros(B, k, N, dtype=D.dtype, device=D.device)], 1)
        c.elementwise("mac", acc[cc], padded, pm)
        del padded
    del D
    kd = k + 1 if rescale else k
    out = empty(2, B, L - kd, N)
    c.moddown(out.view(2 * B, L - kd, N), acc.view(2 * B, L, N), kd)
    return out


def inner_kernel_ms(fn, reps=3):
    """mean device time of the multiplication's inner kernel over `reps` calls, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for e in prof.key_averages():
        if "mulrelin64_inner_kernel" in e.key:
            us += e.device_time * e.count
            n += e.count
    return (us / n) / 1e3 if n else None, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_u64_mulrelin.jsonl"))
    ap.add_argument("--mib", type=float, default=256.0, help="MiB of one ciphertext component (batch workload)")
    ap.add_argument("--dry", action="store_true", help="print the workloads' byte models and exit (no GPU needed)")
    args = ap.parse_args()
    # (workload, N, l + 1, alpha, k, B or None for the batch size)
    cases = [("batch", 16384, 12, 4, 4, None), ("deep", 32768, 24, 8, 8, 1)]
    if args.dry:
        for name, N, ell1, alpha, k, B in cases:
            B = B or int(args.mib * (1 << 20)) // (ell1 * N * 8)
            mw = model_words(ell1, alpha, k)
            print(json.dumps({"workload": name, "N": N, "B": B, "model_words_per_BN": {str(r): mw[r] for r in mw},
                              "model_call_over_route": {str(r): mw[r][0] / mw[r][1] for r in mw}}))
        return
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
    for name, N, ell1, alpha, k, B in cases:
        primes = allp[:ell1] + allp[ell1:ell1 + k]
        L = len(primes)
        dnum = len(digits_of(ell1, alpha))
        B = B or int(args.mib * (1 << 20)) // (ell1 * N * 8)
        c, cq, cr = A.Context64(N, primes), A.Context64(N, primes[:ell1]), A.Context64(N, primes[:ell1 - 1])
        gen = torch.Generator(device="cuda").manual_seed(N + ell1)
        qv = torch.tensor(primes[:ell1], dtype=torch.int64, device="cuda").view(1, 1, ell1, 1)
        kq = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, 1, L, 1)
        a = torch.randint(0, 1 << 62, (2, B, ell1, N), dtype=torch.int64, device="cuda", generator=gen) % qv
        b = torch.randint(0, 1 << 62, (2, B, ell1, N), dtype=torch.int64, device="cuda", generator=gen) % qv
        rlk = torch.randint(0, 1 << 62, (dnum, 2, L, N), dtype=torch.int64, device="cuda", generator=gen) % kq
        same = {}
        outs = {r: empty(2, B, ell1 - 1 if r else ell1, N) for r in (False, True)}
        for r in (False, True):
            want = recipe(c, cq, a, b, rlk, alpha, k, r)
            torch.cuda.synchronize()
            c.mulrelin(outs[r], a, b, rlk, alpha, k, rescale=r, ntt_form=True)
            torch.cuda.synchronize()
            same[f"eval_rescale{int(r)}"] = bool(torch.equal(outs[r], want))
            route = make_route(c, cq, a, b, rlk, alpha, k, r)
            route(outs[r])
            torch.cuda.synchronize()
            same[f"route_rescale{int(r)}"] = bool(torch.equal(outs[r], want))
            del route
            torch.cuda.empty_cache()
            ac, bc = a.clone(), b.clone()                    # coefficient form: inv of the result on fwd of the inputs
            cq.inv(ac.view(2 * B, ell1, N))
            cq.inv(bc.view(2 * B, ell1, N))
            c.mulrelin(outs[r], ac, bc, rlk, alpha, k, rescale=r, ntt_form=False)
            del ac, bc
            (cr if r else cq).inv(want.view(2 * B, -1, N))
            torch.cuda.synchronize()
            same[f"coeff_rescale{int(r)}"] = bool(torch.equal(outs[r], want))
            del want
            torch.cuda.empty_cache()
        routes = {r: make_route(c, cq, a, b, rlk, alpha, k, r) for r in (False, True)}
        fns = {}
        for r in (False, True):
            fns[f"call_rescale{int(r)}"] = (lambda r=r: c.mulrelin(outs[r], a, b, rlk, alpha, k, rescale=r))
            fns[f"route_rescale{int(r)}"] = (lambda r=r: routes[r](outs[r]))
        launches = {}
        for key, fn in fns.items():
            l0 = c.launch_count() + cq.launch_count()
            fn()
            torch.cuda.synchronize()
            launches[key] = c.launch_count() + cq.launch_count() - l0
        copy_dst = torch.empty_like(a)
        keys = list(fns)
        res = timed([fns[x] for x in keys] + [lambda: copy_dst.copy_(a)], 20 if B == 1 else 2)
        ms = dict(zip(keys + ["copy"], res))
        copy_GBps = 2 * a.numel() * 8 / (ms["copy"][0] * 1e-3) / 1e9
        inner_ms, inner_n = inner_kernel_ms(fns["call_rescale0"])
        mw = model_words(ell1, alpha, k)
        unit = B * N * 8
        line = {"workload": name, "N": N, "l+1": ell1, "alpha": alpha, "k": k, "L": L, "dnum": dnum, "B": B,
                "component_bytes": a[0].numel() * 8, "same_output": same, "launches": launches,
                "copy_ms": ms["copy"][0], "copy_GBps": copy_GBps}
        for r in (False, True):
            call, route = ms[f"call_rescale{int(r)}"], ms[f"route_rescale{int(r)}"]
            line[f"rescale{int(r)}"] = {
                "call_ms": call[0], "call_spread_ms": call[1:], "route_ms": route[0], "route_spread_ms": route[1:],
                "call_over_route_time": call[0] / route[0], "model_call_bytes": mw[r][0] * unit,
                "model_route_bytes": mw[r][1] * unit, "model_call_over_route": mw[r][0] / mw[r][1],
                "call_GBps_over_model": mw[r][0] * unit / (call[0] * 1e-3) / 1e9,
                "route_GBps_over_model": mw[r][1] * unit / (route[0] * 1e-3) / 1e9}
        nbytes = inner_words(ell1, alpha, k) * unit
        line.update({"inner_ms": inner_ms, "inner_launches_profiled": inner_n, "inner_bytes": nbytes,
                     "inner_GBps": nbytes / (inner_ms * 1e-3) / 1e9 if inner_ms else None,
                     "inner_share_of_call": inner_ms / ms["call_rescale0"][0] if inner_ms else None})
        if inner_ms:
            line["inner_over_copy_rate"] = line["inner_GBps"] / copy_GBps
        print(json.dumps(line), flush=True)
        lines.append(line)
        del a, b, rlk, outs, routes, copy_dst, fns
        for x in (c, cq, cr):
            x.close()
        torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
