"""CKKS encoding and decoding (Context64.encode / decode, agx_encode64 / agx_decode64) against a torch route and the
byte model.  Same process, alternated timed windows (CUDA events), the card's name and power limit read in the same run.

Workloads, 60-bit primes (q = 1 mod 2^16): N = 16384 and 32768, limbs in {1, 12, 24}, both forms, B chosen so that the
residues are at least 256 MiB (far above the 126 MB of L2).

Byte model per polynomial: encode reads 8 n (the S complex slots) and writes 8 limbs n; the evaluation form adds the
forward's read and write of the 8 limbs n.  Decode reads 8 limbs n and writes 8 n (the doubles m), then the FFT reads
8 n and writes 8 n; the evaluation form adds the inverse's 16 limbs n.  `frac_copy` is the model's bytes over the call's
time, over the device-to-device copy rate measured in the same run (bytes read + written per second).

Torch route (valid where |scale m| < 2^63): encode = torch.fft on the GPU (the oracle's formula on the odd indices of a
length-2n array), rint, int64 remainder per prime; its residues are compared with the call's at limb 0 (count of
differing coefficients, largest difference, and how many of the route's scaled coefficients lie within 1e-3 of a .5
boundary, where two FP64 FFTs that round differently can round to different integers); decode at one limb = centre
the residues, divide by the scale, torch.fft.ifft.  Not compared at 12 and 24 limbs (the route has no exact CRT).
Usage (GPU box): python profiles/bench_u64_encode.py [--out profiles/r12_u64_encode.jsonl]"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import torch
import agilex_ntt_b200 as A
from bench_u64_keyswitch import primes60, timed


class TorchRoute:
    def __init__(self, n, primes):
        self.n, self.S = n, n // 2
        g = torch.tensor([pow(5, j, 2 * n) for j in range(n // 2)], dtype=torch.int64, device="cuda")
        self.g, self.gc = g, (-g) % (2 * n)
        i = torch.arange(n, device="cuda", dtype=torch.float64)
        self.tw = torch.exp(-1j * math.pi * i / n)
        self.itw = torch.exp(1j * math.pi * i / n)
        self.q = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, -1, 1)
        self.sel = (g - 1) // 2

    def encode(self, z, scale, limbs):
        w = torch.zeros(z.shape[0], 2 * self.n, dtype=torch.complex128, device="cuda")
        w[:, self.g] = z
        w[:, self.gc] = z.conj()
        m = (self.tw * torch.fft.fft(w[:, 1::2], dim=-1) / self.n).real
        self.m = m
        c = torch.round(m * scale).to(torch.int64).unsqueeze(1)
        return torch.remainder(c, self.q[:, :limbs])

    def decode1(self, res, scale):
        q = self.q[0, 0, 0]
        x = res[:, 0]
        x = torch.where(x > q // 2, x - q, x).to(torch.float64) / scale
        return (self.n * torch.fft.ifft(x * self.itw, dim=-1))[:, self.sel]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_u64_encode.jsonl"))
    ap.add_argument("--mib", type=int, default=256)
    args = ap.parse_args()
    try:                                                     # read-only query of the card's power limit
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception:
        power = "unknown"
    primes = primes60(24)
    lines = [{"gpu": torch.cuda.get_device_name(0), "power_limit": power,
              "sms": torch.cuda.get_device_properties(0).multi_processor_count, "bits": 60, "residue_MiB": args.mib}]
    print(json.dumps(lines[0]), flush=True)
    scale = 2.0 ** 40
    for N in (16384, 32768):
        c = A.Context64(N, primes)
        route = TorchRoute(N, primes)
        for limbs in (1, 12, 24):
            B = max(1, (args.mib << 20) // (8 * limbs * N))
            g = torch.Generator(device="cuda").manual_seed(N + limbs)
            z = torch.complex(torch.rand(B, N // 2, generator=g, device="cuda", dtype=torch.float64) * 2 - 1,
                              torch.rand(B, N // 2, generator=g, device="cuda", dtype=torch.float64) * 2 - 1)
            res = torch.empty(B, limbs, N, dtype=torch.int64, device="cuda")
            zo = torch.empty_like(z)
            cp_src = torch.empty(B * limbs * N, dtype=torch.int64, device="cuda")
            cp_dst = torch.empty_like(cp_src)
            # correctness on this workload: the call against the route (coefficient form), and the round trip
            c.encode(res, z, scale, ntt_form=False)
            rr = route.encode(z, scale, limbs)
            q0 = int(primes[0])
            diff = torch.remainder(res[:, 0] - rr[:, 0], q0)            # limb 0, centred: c_call - c_route
            diff = torch.where(diff > q0 // 2, diff - q0, diff)
            mism, maxdiff = int((diff != 0).sum().item()), int(diff.abs().max().item())
            near_half = int(((torch.remainder(route.m * scale, 1.0) - 0.5).abs() < 1e-3).sum().item())
            del rr, diff
            c.decode(zo, res, scale, ntt_form=False)
            rt_err = (zo - z).abs().max().item()
            dec_route_err = (route.decode1(res, scale) - zo).abs().max().item() if limbs == 1 else None
            for form in (False, True):
                fns = [lambda: c.encode(res, z, scale, ntt_form=form),
                       lambda: c.decode(zo, res, scale, ntt_form=form),
                       lambda: cp_dst.copy_(cp_src)]
                if not form:
                    fns.append(lambda: route.encode(z, scale, limbs))
                    if limbs == 1:
                        fns.append(lambda: route.decode1(res, scale))
                t = timed(fns, iters=5)
                copy_rate = 2 * cp_src.numel() * 8 / (t[2][0] * 1e-3)
                enc_bytes = B * N * 8 * (1 + limbs + (2 * limbs if form else 0))
                dec_bytes = B * N * 8 * (limbs + 3 + (2 * limbs if form else 0))
                line = {"N": N, "limbs": limbs, "B": B, "form": "eval" if form else "coeff",
                        "encode_ms": t[0][0], "encode_ms_min_max": t[0][1:], "decode_ms": t[1][0],
                        "decode_ms_min_max": t[1][1:], "copy_GBps": copy_rate / 1e9,
                        "encode_model_GBps": enc_bytes / (t[0][0] * 1e-3) / 1e9,
                        "decode_model_GBps": dec_bytes / (t[1][0] * 1e-3) / 1e9,
                        "encode_frac_copy": enc_bytes / (t[0][0] * 1e-3) / copy_rate,
                        "decode_frac_copy": dec_bytes / (t[1][0] * 1e-3) / copy_rate,
                        "encode_vs_route_mismatches": mism, "encode_vs_route_max_diff": maxdiff,
                        "coefficients": B * N, "route_fractions_within_1e-3_of_half": near_half,
                        "round_trip_max_err": rt_err}
                if not form:
                    line["route_encode_ms"] = t[3][0]
                    if limbs == 1:
                        line["route_decode_ms"] = t[4][0]
                        line["decode_vs_route_max_diff"] = dec_route_err
                lines.append(line)
                print(json.dumps(line), flush=True)
            del z, res, zo, cp_src, cp_dst
            torch.cuda.empty_cache()
        c.close()
    with open(args.out, "w") as fh:
        for l in lines:
            fh.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
