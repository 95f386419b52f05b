"""One rotation (G = 1) at the first batch shape of bench_u64_rotate.py (N = 16384, (l + 1, alpha, k) = (12, 4, 4),
256 MiB per ciphertext component): agx_rotate64, the plain recipe and agx_keyswitch64 alone, alternated with CUDA events
(4 calls per window, median / min / max of 5 windows, ms), then each one's kernels from torch.profiler over 3 calls.
Usage (GPU box): python profiles/prof_u64_rotate_g1.py > profiles/r09_u64_rotate_g1_profile.txt"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "profiles"))
import torch
import agilex_ntt_b200 as A
from bench_u64_keyswitch import primes60, timed
from bench_u64_rotate import make_plain
from torch.profiler import ProfilerActivity, profile

N, ell1, alpha, k, G = 16384, 12, 4, 4, 1
allp = primes60(20)
primes = allp[:ell1] + allp[ell1:ell1 + k]
L = len(primes)
B = (256 << 20) // (ell1 * N * 8)
c, cq = A.Context64(N, primes), A.Context64(N, primes[:ell1])
gen = torch.Generator(device="cuda").manual_seed(1)
qv = torch.tensor(primes[:ell1], dtype=torch.int64, device="cuda").view(1, 1, ell1, 1)
kq = torch.tensor(primes, dtype=torch.int64, device="cuda").view(1, 1, L, 1)
ct = torch.randint(0, 1 << 62, (2, B, ell1, N), dtype=torch.int64, device="cuda", generator=gen) % qv
gs = [A.galois_element(N, 1)]
rks = [torch.randint(0, 1 << 62, (3, 2, L, N), dtype=torch.int64, device="cuda", generator=gen) % kq]
out = torch.empty((G, 2, B, ell1, N), dtype=torch.int64, device="cuda")
want = torch.empty_like(out)
ks_out = torch.empty((2, B, ell1, N), dtype=torch.int64, device="cuda")
plain = make_plain(c, cq, ct, gs, rks, alpha, k)
fns = {"call": lambda: c.rotate(out, ct, gs, rks, alpha, k), "plain": lambda: plain(want, True),
       "keyswitch": lambda: c.keyswitch(ks_out, ct[1], rks[0], alpha, k)}
res = timed(list(fns.values()), 4)
for n_, r in zip(fns, res):
    print(n_, r)
for n_, f in fns.items():
    f(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            f()
        torch.cuda.synchronize()
    print("=====", n_)
    print(prof.key_averages().table(sort_by="device_time_total", row_limit=14, max_name_column_width=70))
