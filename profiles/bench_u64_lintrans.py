"""Hoisted linear transforms in one call (Context64.lintrans, agx_lintrans64) against route (a), today's way: the G
rotations from agx_rotate64, then the M * G element-wise products and sums with the diagonals over Q_l.  Same process,
alternated timed windows.

Workloads, 60-bit primes (q = 1 mod 2^16):
- bootstrapping: B = 1, N = 32768, (l + 1, alpha, k) = (24, 8, 8), G = 16 with baby step 0 (g = 1) keyless, M = 4
  dense: the baby steps of a CoeffToSlot-sized BSGS level.  Route (a) rotates by the 15 keyed elements and uses the
  input itself for g = 1;
- batch: N = 16384, (12, 4, 4), G = 8 (g = 1 keyed, rotations by 1..6 and the conjugation), M = 2, B chosen so that
  one ciphertext component is 256 MiB (far above the 126 MB of L2).

Each line first checks both forms of the call bit for bit against the recipe composed from public calls (modup of the
digits, automorph, element-wise products and sums over Q_l u P, one moddown of 2 M B; not timed), then times the
evaluation forms of the call and of route (a), alternated in 5 windows with CUDA events, beside a device-to-device copy
of the ciphertexts.  Route (a) is not bit-equal to the call (it rounds G times), so only the call is checked.  The
inner kernel's time comes from a separate torch.profiler run (CUDA activities), by kernel name, against the copy rate
over its byte model, per coefficient: dnum * B * L words of extended digits and B * (l + 1) of c0 (and as much of c1
when a term is keyless) read once (the G re-reads served from L2), the keys (2 * dnum * L words per keyed term) and
diagonals (L words per non-NULL one) once per call (once per polynomial from L2), and 2 * M * B * L words written.
The header line carries the GPU name and power limit read in the same run.
Usage (GPU box): python profiles/bench_u64_lintrans.py [--out profiles/r10_u64_lintrans.jsonl]"""
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


def make_recipe(c, cq, ct, gs, rks, diags, alpha, k):
    """The definition composed from public calls in evaluation form (tests/test_u64_lintrans.py's recipe)."""
    L, N, B = c.L, c.n, ct.shape[1]
    ell1 = L - k
    P = 1
    for q in c.primes[ell1:]:
        P *= q
    pm = torch.tensor([P % q if i < ell1 else 0 for i, q in enumerate(c.primes)], dtype=torch.int64,
                      device="cuda").view(1, L, 1).expand(B, L, N).contiguous()
    pad = lambda x: torch.cat([x, torch.zeros(B, k, N, dtype=x.dtype, device=x.device)], 1)

    def run(out):
        Us = []
        for f, cnt in digits_of(ell1, alpha):
            U = empty(B, L, N)
            c.modup(U, ct[1, :, f:f + cnt].contiguous(), f, cnt, ntt_form=True)
            Us.append(U)
        M = len(diags)
        acc = torch.zeros(M, 2, B, L, N, dtype=torch.int64, device="cuda")
        At, sU = [empty(B, L, N), empty(B, L, N)], empty(B, L, N)
        for t, (g, rk) in enumerate(zip(gs, rks)):
            if rk is None:
                for cc in (0, 1):
                    c.elementwise("mul", At[cc], pad(ct[cc]), pm)
            else:
                kr = torch.cat([rk[:, :, :ell1], rk[:, :, rk.shape[2] - k:]], dim=2)
                for j, U in enumerate(Us):
                    c.automorph(sU, U, g)
                    for cc in (0, 1):
                        c.elementwise("mul" if j == 0 else "mac", At[cc], sU, kr[j, cc].expand(B, L, N).contiguous())
                s0 = empty(B, ell1, N)
                cq.automorph(s0, ct[0], g)
                c.elementwise("mac", At[0], pad(s0), pm)
            for m, row in enumerate(diags):
                if row[t] is not None:
                    dd = row[t].expand(B, L, N).contiguous()
                    for cc in (0, 1):
                        c.elementwise("mac", acc[m, cc], At[cc], dd)
        c.moddown(out.view(2 * M * B, ell1, N), acc.view(2 * M * B, L, N), k)
    return run


def make_route_a(c, cq, ct, gs, rks, diags, alpha, k):
    """agx_rotate64 over the keyed elements, then per (m, t) one element-wise product or MAC over Q_l with the
    diagonal's first l + 1 rows replicated over the 2 B polynomials of a ciphertext (built outside the timing); a
    keyless g = 1 term multiplies the input itself."""
    B, ell1, N = ct.shape[1], ct.shape[2], ct.shape[3]
    keyed = [t for t, rk in enumerate(rks) if rk is not None]
    rot = empty(len(keyed), 2, B, ell1, N)
    reps = [[None if d is None else d[:ell1].expand(2 * B, ell1, N).contiguous() for d in row] for row in diags]

    def run(out):
        c.rotate(rot, ct, [gs[t] for t in keyed], [rks[t] for t in keyed], alpha, k, ntt_form=True)
        for m, row in enumerate(reps):
            o = out[m].view(2 * B, ell1, N)
            first = True
            for t, d in enumerate(row):
                if d is None:
                    continue
                src = rot[keyed.index(t)] if rks[t] is not None else ct
                cq.elementwise("mul" if first else "mac", o, src.view(2 * B, ell1, N), d)
                first = False
    return run


def inner_kernel_ms(fn, reps=3):
    """mean device time of the linear transform's inner kernel over `reps` calls, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us, n = 0.0, 0
    for e in prof.key_averages():
        if "lintrans64_inner_kernel" in e.key:
            us += e.device_time * e.count
            n += e.count
    return (us / n) / 1e3 if n else None, n


def inner_bytes(B, L, ell1, dnum, rks, diags, N):
    """the inner kernel's byte model (see the module docstring)"""
    M = len(diags)
    kept = [t for t in range(len(rks)) if any(row[t] is not None for row in diags)]
    keyed = sum(rks[t] is not None for t in kept)
    keyless = any(rks[t] is None for t in kept)
    nd = sum(row[t] is not None for row in diags for t in kept)
    words = dnum * B * L + B * ell1 * (2 if keyless else 1) + 2 * dnum * L * keyed + L * nd + 2 * M * B * L
    return words * N * 8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_u64_lintrans.jsonl"))
    ap.add_argument("--mib", type=float, default=256.0, help="MiB of one ciphertext component (batch workload)")
    ap.add_argument("--dry", action="store_true", help="print the workloads' byte models and exit (no GPU needed)")
    args = ap.parse_args()
    # (workload, N, l + 1, alpha, k, G, M, B or None for the batch size, keyless baby step 0)
    cases = [("bootstrapping", 32768, 24, 8, 8, 16, 4, 1, True), ("batch", 16384, 12, 4, 4, 8, 2, None, False)]
    if args.dry:
        for name, N, ell1, alpha, k, G, M, B, keyless in cases:
            B = B or int(args.mib * (1 << 20)) // (ell1 * N * 8)
            rks = [None if keyless and t == 0 else 1 for t in range(G)]
            diags = [[1] * G for _ in range(M)]
            L, dnum = ell1 + k, len(digits_of(ell1, alpha))
            print(json.dumps({"workload": name, "N": N, "B": B, "L": L, "dnum": dnum, "G": G, "M": M,
                              "inner_bytes": inner_bytes(B, L, ell1, dnum, rks, diags, N)}))
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
    for name, N, ell1, alpha, k, G, M, B, keyless in cases:
        primes = allp[:ell1] + allp[ell1:ell1 + k]
        L = len(primes)
        dnum = len(digits_of(ell1, alpha))
        B = B or int(args.mib * (1 << 20)) // (ell1 * N * 8)
        c, cq = A.Context64(N, primes), A.Context64(N, primes[:ell1])
        gen = torch.Generator(device="cuda").manual_seed(N + ell1 + G)
        qv = torch.tensor(primes[:ell1], dtype=torch.int64, device="cuda").view(1, 1, ell1, 1)
        kq = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, 1, L, 1)
        ct = torch.randint(0, 1 << 62, (2, B, ell1, N), dtype=torch.int64, device="cuda", generator=gen) % qv
        if keyless:
            gs = [A.galois_element(N, r) for r in range(G)]
        else:
            gs = [1] + [A.galois_element(N, r) for r in range(1, G - 1)] + [2 * N - 1]
        rks = [None if keyless and g == 1 else
               torch.randint(0, 1 << 62, (dnum, 2, L, N), dtype=torch.int64, device="cuda", generator=gen) % kq
               for g in gs]
        diags = [[torch.randint(0, 1 << 62, (1, L, N), dtype=torch.int64, device="cuda", generator=gen).view(L, N) %
                  kq.view(L, 1) for _ in gs] for _ in range(M)]
        out = empty(M, 2, B, ell1, N)
        want = torch.empty_like(out)
        recipe = make_recipe(c, cq, ct, gs, rks, diags, alpha, k)
        same = {}
        recipe(want)
        for form in (True, False):
            if form:
                c.lintrans(out, ct, gs, rks, diags, alpha, k, ntt_form=True)
                torch.cuda.synchronize()
                same["eval"] = bool(torch.equal(out, want))
            else:                                            # coefficient form: inv of the result on fwd of the input
                cth = ct.clone()
                cq.inv(cth.view(2 * B, ell1, N))              # cth's spectrum is ct
                c.lintrans(out, cth, gs, rks, diags, alpha, k, ntt_form=False)
                w2 = want.clone()
                cq.inv(w2.view(2 * M * B, ell1, N))
                torch.cuda.synchronize()
                same["coeff"] = bool(torch.equal(out, w2))
                del cth, w2
        del recipe
        torch.cuda.empty_cache()
        route_a = make_route_a(c, cq, ct, gs, rks, diags, alpha, k)
        fns = {"call_eval": lambda: c.lintrans(out, ct, gs, rks, diags, alpha, k, ntt_form=True),
               "call_coeff": lambda: c.lintrans(out, ct, gs, rks, diags, alpha, k, ntt_form=False),
               "route_a_eval": lambda: route_a(want)}
        launches = {}
        for key, fn in fns.items():
            l0, l1 = c.launch_count(), cq.launch_count()
            fn()
            torch.cuda.synchronize()
            launches[key] = c.launch_count() - l0 + cq.launch_count() - l1
        copy_dst = torch.empty_like(ct)
        res = timed([fns["call_eval"], fns["route_a_eval"], lambda: copy_dst.copy_(ct)], 20 if B == 1 else 2)
        call, ra, cp = res
        copy_GBps = 2 * ct.numel() * 8 / (cp[0] * 1e-3) / 1e9
        inner_ms, inner_n = inner_kernel_ms(fns["call_eval"])
        nbytes = inner_bytes(B, L, ell1, dnum, rks, diags, N)
        line = {"workload": name, "N": N, "l+1": ell1, "alpha": alpha, "k": k, "L": L, "dnum": dnum, "G": G, "M": M,
                "B": B, "keyless_identity": keyless, "component_bytes": ct[0].numel() * 8, "same_output": same,
                "launches": launches, "call_ms": call[0], "call_spread_ms": call[1:], "route_a_ms": ra[0],
                "route_a_spread_ms": ra[1:], "call_over_route_a_time": call[0] / ra[0], "copy_ms": cp[0],
                "copy_GBps": copy_GBps, "inner_ms": inner_ms, "inner_launches_profiled": inner_n,
                "inner_bytes": nbytes, "inner_GBps": nbytes / (inner_ms * 1e-3) / 1e9 if inner_ms else None,
                "inner_share_of_time": inner_ms / call[0] if inner_ms else None}
        if inner_ms:
            line["inner_over_copy_rate"] = line["inner_GBps"] / copy_GBps
        print(json.dumps(line), flush=True)
        lines.append(line)
        del ct, rks, diags, out, want, route_a, copy_dst, fns
        c.close()
        cq.close()
        torch.cuda.empty_cache()
    with open(args.out, "w") as fh:
        for ln in lines:
            fh.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
